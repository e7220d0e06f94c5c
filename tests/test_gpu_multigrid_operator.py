"""GPU: the multigrid preconditioner of csrc/mg.cu stage by stage against its fp64 restatement (tests/mg_reference.py).

Outer CG absorbs preconditioner errors — a wrong transfer weight or Chebyshev coefficient costs iterations, not the
answer — so the stages are compared one by one through the test hook fi_field_mg_stage, on the hierarchy the solve
itself uses (fi_field::get_mg):

* level operators A_l, restriction P^T, prolongation P and the dense coarse solve: to fp32 rounding;
* the Chebyshev bound: lambda_max(D^-1 A_l) <= lmax_l <= 1.1 lambda_max (1 + 1e-3) on every smoothed level;
* the smoother and the whole cycle (V, W over 1 / 2 / 3 coarse levels with 6 coarse steps, the single-kernel tail):
  relative L2 difference from the fp64 restatement;
* on lattices small enough to form B: B symmetric to fp32 rounding, the eigenvalues of B A real and positive (V and W);
* fp64 CG preconditioned by the restatement and the library's FI_F64 MG-PCG take the same iterations (+-1);
* the process-wide kernel switches (FI_B200_DATA_TERM, FI_B200_STENCIL_TY), read once per process, in child processes.

Tolerances of the smoother and cycle checks (relative L2 against fp64): ten times the worst fp32-vs-fp64 difference
measured on a B200 (1000 W) over every case and cycle configuration of this file with the default kernel switches
(scripts/mg_operator_spread.py, profiles/mg_operator_spread_b200.jsonl): smoother 1.15e-6, whole cycle 8.3e-7."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg as sla
import scipy.sparse.linalg as spla

import mg_reference as R
from conftest import ROOT
from field_interpolation_b200 import workloads as W
from field_interpolation_b200 import _lib as L

pytestmark = pytest.mark.gpu

EPS32 = float(np.finfo(np.float32).eps)
TOL_SMOOTH = 1.2e-5  # relative L2, SMOOTH against the fp64 Chebyshev steps (10 x 1.15e-6 measured)
TOL_CYCLE = 8.5e-6   # relative L2, CYCLE against the fp64 cycle (10 x 8.3e-7 measured)

ALL_ON = dict(model_0=0.1, model_1=0.2, model_2=0.5, model_3=0.3, model_4=0.25, gradient_smoothness=0.15)

# sizes, points, weights, caller rows on level 0, FI_B200_MG_COARSEST.  Odd sizes 2n - 1 coarsen 2:1 exactly, even ones
# do not; x sizes that are multiples of 4 take prolong_add4_kernel, the others the scalar kernel; x % 4 == 0 and x >= 32
# (with y >= 8 in 3D) takes the TMA stencil kernels in epilogue mode (fused smoother steps) wherever a level has no
# caller rows.
CASES = {
    "small_1d_odd": dict(sizes=[65], npts=40, wkw={}, coarsest=8),
    "small_1d_even": dict(sizes=[96], npts=40, wkw=dict(model_1=0.3, gradient_kernel=0), coarsest=8),
    "small_2d_odd": dict(sizes=[33, 29], npts=300, wkw=dict(model_1=0.2, gradient_smoothness=0.3, gradient_kernel=0), coarsest=16),
    "small_2d_rows": dict(sizes=[64, 36], npts=400, wkw=dict(gradient_kernel=2), rows=True, coarsest=30),
    "small_2d_tma": dict(sizes=[96, 40], npts=500, wkw=dict(model_2=0.0, model_3=0.4), coarsest=30),
    "small_3d_odd": dict(sizes=[21, 18, 17], npts=600, wkw=dict(model_0=0.1, model_3=0.2), coarsest=40),
    "small_3d_tma": dict(sizes=[32, 16, 16], npts=700, wkw=dict(ALL_ON, gradient_kernel=2), coarsest=130),
    "small_3d_flat": dict(sizes=[24, 1, 22], npts=200, wkw=dict(value_kernel=0), coarsest=20),
}
# lattices on which B is formed explicitly (n <= ~2000)
EXPLICIT = ["small_1d_odd", "small_1d_even", "small_2d_odd", "small_3d_flat"]

CYCLES = {
    "V": {},
    "W1": dict(FI_B200_MG_GAMMA="2", FI_B200_MG_WLEVELS="1", FI_B200_MG_NU_COARSE="6"),
    "W2": dict(FI_B200_MG_GAMMA="2", FI_B200_MG_WLEVELS="2", FI_B200_MG_NU_COARSE="6"),
    "W3": dict(FI_B200_MG_GAMMA="2", FI_B200_MG_WLEVELS="3", FI_B200_MG_NU_COARSE="6"),
    "tail": dict(FI_B200_MG_TAIL_CELLS="4096"),
}
MG_ENV = ("FI_B200_MG_COARSEST", "FI_B200_MG_GAMMA", "FI_B200_MG_WLEVELS", "FI_B200_MG_NU_COARSE", "FI_B200_MG_TAIL_CELLS",
          "FI_B200_MG_DENSE_APPLY")


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


@pytest.fixture(scope="module")
def fi():
    import field_interpolation_b200 as m
    return m


def problem(name):
    c = CASES[name]
    sizes, D = c["sizes"], len(c["sizes"])
    if D == 1:
        rng = np.random.default_rng(sizes[0])
        pos = rng.uniform(0.3, sizes[0] - 1.3, (c["npts"], 1)).astype(np.float32)
        nrm = np.where(rng.uniform(size=(c["npts"], 1)) < 0.5, -1.0, 1.0).astype(np.float32)
    else:
        pos, nrm = W.random_cloud(D, c["npts"], sizes, seed=int(np.prod(sizes)))
    n = int(np.prod(sizes))
    rows = [(0.7, 1.5, [0, n - 1, n // 2], [1.0, -2.0, 0.5]), (0.3, -1.0, [n // 3], [2.0])] if c.get("rows") else []
    return R.Problem(list(sizes), dict(c["wkw"]), pos, nrm, None, rows)


def make_field(fi, prob):
    f = fi.sdf_from_points(prob.sizes, fi.Weights(**prob.weights), prob.pos, prob.nrm)
    for weight, rhs, cols, vals in prob.rows:
        fi.add_equation(f, weight, rhs, list(zip(cols, vals)))
    return f


def set_env(monkeypatch, name, cycle="V"):
    for k in MG_ENV:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("FI_B200_MG_COARSEST", str(CASES[name]["coarsest"]))
    for k, v in CYCLES[cycle].items():
        monkeypatch.setenv(k, v)


def mg_opts(fi, **kw):
    return fi.solve_options(fi.FI_F32, 0, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID, **kw)


_FIELDS, _REFS = {}, {}


def field_and_reference(fi, port, name, monkeypatch, cycle="V"):
    """The library's field (hierarchy built under the case's environment) and the restatement of the hierarchy it
    reports.  Level operators are cached per case: they do not depend on the cycle."""
    set_env(monkeypatch, name, cycle)
    if name not in _FIELDS:
        _FIELDS[name] = (problem(name), None)
        _FIELDS[name] = (_FIELDS[name][0], make_field(fi, _FIELDS[name][0]))
    prob, f = _FIELDS[name]
    info = f.mg_info(mg_opts(fi))
    key = name
    if key not in _REFS:
        _REFS[key] = R.Hierarchy(port, prob, info)
    H = _REFS[key]
    H.info, H.lmax = info, list(info["lmax"])
    return prob, f, info, H


# ---- 1. level operators, hierarchy shape --------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_level_operators(fi, port, name, monkeypatch):
    """OPERATOR on every level against A_l of the coarsening rule (bound of test_operator_matches_reference_normal_equations);
    the level sizes against the rule in mg.cu."""
    prob, f, info, H = field_and_reference(fi, port, name, monkeypatch)
    D = prob.D
    assert [s[:D] for s in info["sizes"]] == R.level_sizes(prob.sizes, CASES[name]["coarsest"])
    assert info["levels"] >= 3, info
    rng = np.random.default_rng(1)
    for l in range(info["levels"]):
        A = H.A[l]
        x = rng.normal(size=(2, A.shape[0]))
        got = f.mg_stage(L.FI_MG_OPERATOR, l, x, options=mg_opts(fi))
        for k in range(2):
            scale = abs(A).max() * np.abs(x[k]).max() * 30
            np.testing.assert_allclose(got[k], A @ x[k], rtol=0, atol=2e-6 * scale, err_msg=f"level {l}")


# ---- 2. transfers -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_transfers(fi, port, name, monkeypatch):
    """RESTRICT = P^T and PROLONG_ADD = e + P e_c on every level pair, to fp32 rounding."""
    prob, f, info, H = field_and_reference(fi, port, name, monkeypatch)
    rng = np.random.default_rng(2)
    for l in range(info["levels"] - 1):
        P = H.P[l]
        nf, nc = P.shape
        xf = rng.normal(size=(2, nf))
        got = f.mg_stage(L.FI_MG_RESTRICT, l, xf, options=mg_opts(fi))
        for k in range(2):
            np.testing.assert_allclose(got[k], P.T @ xf[k], rtol=0, atol=8 * EPS32 * 16 * np.abs(xf[k]).max(), err_msg=f"restrict {l}")
        xc, e = rng.normal(size=(2, nc)), rng.normal(size=(2, nf))
        got = f.mg_stage(L.FI_MG_PROLONG_ADD, l, xc, e, options=mg_opts(fi))
        got0 = f.mg_stage(L.FI_MG_PROLONG_ADD, l, xc, None, options=mg_opts(fi))
        for k in range(2):
            atol = 8 * EPS32 * (np.abs(xc[k]).max() + np.abs(e[k]).max())
            np.testing.assert_allclose(got[k], e[k] + P @ xc[k], rtol=0, atol=atol, err_msg=f"prolong {l}")
            np.testing.assert_allclose(got0[k], P @ xc[k], rtol=0, atol=atol, err_msg=f"prolong from zero {l}")


# ---- 3. coarse solve ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dense_apply", ["0", "1"])
@pytest.mark.parametrize("name", ["small_1d_odd", "small_2d_rows", "small_3d_tma", "small_3d_flat"])
def test_coarse_solve(fi, port, name, dense_apply, monkeypatch):
    """COARSE against inv(A_L) of the restatement, with the coarsest matrix written directly and column by column
    (FI_B200_MG_DENSE_APPLY=1): the fp32-assembled matrix inverted in fp64 differs by cond(A_L) times fp32 rounding."""
    set_env(monkeypatch, name)
    monkeypatch.setenv("FI_B200_MG_DENSE_APPLY", dense_apply)
    prob = problem(name)
    f = make_field(fi, prob)  # the switch is read when the hierarchy is built: a fresh field
    info = f.mg_info(mg_opts(fi))
    Lc = info["levels"] - 1
    Ac = R.level_operator(port, prob, info["sizes"][Lc][:prob.D], Lc).toarray()
    cond = np.linalg.cond(Ac)
    r = np.random.default_rng(3).normal(size=(3, Ac.shape[0]))
    got = f.mg_stage(L.FI_MG_COARSE, Lc, r, options=mg_opts(fi))
    f.close()
    for k in range(3):
        want = np.linalg.solve(Ac, r[k])
        assert rel(got[k], want) <= 30 * EPS32 * cond, (rel(got[k], want), cond)


# ---- 4. Chebyshev bound -------------------------------------------------------------------------------------------
def lambda_max(A):
    d = 1.0 / np.sqrt(A.diagonal())
    S = A.multiply(d[:, None]).multiply(d[None, :]).tocsr()
    if S.shape[0] <= 3000:
        return float(sla.eigvalsh(S.toarray()).max())
    return float(spla.eigsh(S, k=1, which="LA", tol=1e-10)[0][0])


@pytest.mark.parametrize("name", list(CASES))
def test_chebyshev_bound(fi, port, name, monkeypatch):
    """Every smoothed level: lambda_max(D^-1 A_l) <= lmax_l <= 1.1 lambda_max (1 + 1e-3).  Below lambda_max the smoother
    amplifies the top modes instead of damping them."""
    prob, f, info, H = field_and_reference(fi, port, name, monkeypatch)
    ratios = []
    for l in range(info["levels"] - 1):
        lam = lambda_max(H.A[l])
        ratios.append(info["lmax"][l] / lam)
    assert all(1.0 <= q <= 1.1 * (1 + 1e-3) for q in ratios), [f"level {l}: lmax / lambda_max = {q:.5f}" for l, q in enumerate(ratios)]


# ---- 5. smoother --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_smoother(fi, port, name, monkeypatch):
    """SMOOTH (the cycle's Chebyshev steps, fused with the TMA epilogue where the cycle fuses them) from zero and from a
    given e, on every smoothed level, against the fp64 recurrence with the library's lmax."""
    prob, f, info, H = field_and_reference(fi, port, name, monkeypatch)
    rng = np.random.default_rng(5)
    for l in range(info["levels"] - 1):
        n = H.A[l].shape[0]
        r, e = rng.normal(size=(2, n)), rng.normal(size=(2, n))
        z0 = f.mg_stage(L.FI_MG_SMOOTH, l, r, None, options=mg_opts(fi))
        z1 = f.mg_stage(L.FI_MG_SMOOTH, l, r, e, options=mg_opts(fi))
        for k in range(2):
            assert rel(z0[k], H.smooth(l, r[k])) <= TOL_SMOOTH, (l, rel(z0[k], H.smooth(l, r[k])))
            assert rel(z1[k], H.smooth(l, r[k], e[k])) <= TOL_SMOOTH, (l, rel(z1[k], H.smooth(l, r[k], e[k])))


# ---- 6. whole cycle -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cycle", list(CYCLES))
@pytest.mark.parametrize("name", list(CASES))
def test_cycle_matches_reference(fi, port, name, cycle, monkeypatch):
    """CYCLE (the captured graph the solve launches) against the fp64 cycle: V, W with the second coarse correction on
    levels 1 .. 1 / 2 / 3 and 6 coarse steps, and the last levels walked by mg_tail_kernel."""
    prob, f, info, H = field_and_reference(fi, port, name, monkeypatch, cycle)
    if cycle.startswith("W"):
        assert info["gamma"] == 2 and info["nu_coarse"] == 6 and info["w_levels"] == int(cycle[1])
    if cycle == "tail" and name in ("small_1d_odd", "small_2d_odd", "small_3d_odd"):  # (generic rows keep a level off the tail)
        assert info["tail_from"] > 0, info
    r = np.random.default_rng(6).normal(size=(3, prob.n))
    z = f.mg_stage(L.FI_MG_CYCLE, 0, r, options=mg_opts(fi))
    for k in range(3):
        want = H.cycle(r[k])
        assert rel(z[k], want) <= TOL_CYCLE, rel(z[k], want)


# ---- 7. properties of B that need no reference ----------------------------------------------------------------------
@pytest.mark.parametrize("cycle", ["V", "W3"])
@pytest.mark.parametrize("name", EXPLICIT)
def test_cycle_is_symmetric_positive_definite(fi, port, name, cycle, monkeypatch):
    """B formed column by column: symmetric to fp32 rounding, and the eigenvalues of B A real and positive (B A is similar
    to A^1/2 B A^1/2).  A W-cycle is positive definite only while the V-cycle it repeats converges."""
    prob, f, info, H = field_and_reference(fi, port, name, monkeypatch, cycle)
    n = prob.n
    B = f.mg_stage(L.FI_MG_CYCLE, 0, np.eye(n), options=mg_opts(fi)).astype(np.float64).T  # column k = B e_k
    asym = np.abs(B - B.T).max() / np.abs(B).max()
    assert asym <= 200 * EPS32, asym
    A = H.A[0].toarray()
    C = np.linalg.cholesky(A)
    lam = sla.eigvalsh(C.T @ (0.5 * (B + B.T)) @ C)
    assert lam.min() > 0, f"{cycle}: lambda(BA) in [{lam.min():.4g}, {lam.max():.4g}]"
    # the same spectrum from the unsymmetrised product: real
    ev = np.linalg.eigvals(B @ A)
    assert np.abs(ev.imag).max() <= 1e-3 * np.abs(ev.real).max() and ev.real.min() > 0, \
        f"{cycle}: lambda(BA) in [{lam.min():.4g}, {lam.max():.4g}], max |imag| {np.abs(ev.imag).max():.3g}"


# ---- 8. consequence for the solve -----------------------------------------------------------------------------------
@pytest.mark.parametrize("cycle", ["V", "W2"])
@pytest.mark.parametrize("name", ["small_1d_odd", "small_2d_odd", "small_2d_rows", "small_3d_odd", "small_3d_tma"])
def test_pcg_iterations_match_reference(fi, port, name, cycle, monkeypatch):
    """fp64 CG preconditioned by the fp64 cycle and the library's FI_F64 MG-PCG, both to 1e-8: the same iteration count
    (+-1) — the preconditioner is the intended one, not merely a working one."""
    prob, f, info, H = field_and_reference(fi, port, name, monkeypatch, cycle)
    _, atb = O_normal(port, prob)
    _, it_ref = R.pcg(H.A[0], atb, H.cycle, 1e-8)
    _, st = f.solve(fi.solve_options(fi.FI_F64, 0, 1e-8, preconditioner=fi.FI_PRECOND_MULTIGRID))
    assert st["converged"] and abs(st["iterations"] - it_ref) <= 1, (st["iterations"], it_ref)


def O_normal(port, prob):
    from oracle import oracle as O
    return O.normal_equations_f64(R.level_system(port, prob, prob.sizes, 0), prob.n)


def test_solve_after_hook_calls(fi, port, monkeypatch):
    """The hook captures the cycle's graph on its own vectors; a solve afterwards re-captures on its own and is the
    same solve as before."""
    name = "small_2d_tma"
    set_env(monkeypatch, name)
    f = make_field(fi, problem(name))
    opt = fi.solve_options(fi.FI_F32, 0, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID)
    x0, s0 = f.solve(opt)
    r = np.random.default_rng(8).normal(size=(2, f.num_unknowns))
    f.mg_stage(L.FI_MG_CYCLE, 0, r, options=opt)
    f.mg_stage(L.FI_MG_SMOOTH, 0, r, None, options=opt)
    x1, s1 = f.solve(opt)
    assert s0["converged"] and s1["converged"] and abs(s0["iterations"] - s1["iterations"]) <= 1, (s0, s1)
    assert rel(x1, x0) <= 1e-5
    f.close()


# ---- 9. process-wide switches ---------------------------------------------------------------------------------------
SWITCH_BODIES = ("test_level_operators or test_smoother or test_cycle_matches_reference or "
                 "test_fast_stencil_matches_generic_and_oracle or test_fused_pcg_matches_unfused")


@pytest.mark.parametrize("env", ["FI_B200_DATA_TERM=node", "FI_B200_DATA_TERM=split", "FI_B200_STENCIL_TY=8", "FI_B200_STENCIL_TY=7"])
def test_process_wide_switches(env):
    """Kernel switches read once per process (apply_nodes_epilogue_kernel is reached only with FI_B200_DATA_TERM=node; the
    8-row TMA tiles of small lattices only with FI_B200_STENCIL_TY=8): the operator, smoother and cycle checks above and
    the stencil / fused-PCG parity tests of test_gpu_solve.py in a child pytest per setting."""
    k, v = env.split("=")
    child = dict(os.environ, **{k: v})
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_multigrid_operator.py"),
                        os.path.join(ROOT, "tests", "test_gpu_solve.py"), "-m", "gpu", "-q", "-k", SWITCH_BODIES,
                        "-p", "no:cacheprovider"], env=child, capture_output=True, text=True, timeout=1800, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-1000:]
    assert " passed" in r.stdout and " failed" not in r.stdout
