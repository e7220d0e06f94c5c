"""GPU: the fused Jacobi-PCG keeps a ring of m search directions and adds their terms to x once per m iterations
(solver.cu, FI_B200_X_RING).  The r, p, q, alpha, beta recurrence is the same for every m, so the iteration counts are
identical and x differs only by the order in which it sums the same alpha_k p_k terms.

Tolerances on x against m = 2 (relative L2), 10x the spread of two m = 2 runs, measured on a B200 over every lattice,
precision and iteration count of test_x_ring_same_iterates_every_pending_count (scripts/x_ring_spread.py,
profiles/x_ring_b200.jsonl):
  fp32: two m = 2 runs differ by up to 2.03e-7 (the data term's atomics), m = 4 / 8 from m = 2 by up to 2.64e-7 -> 2.0e-6;
  fp64: the field is returned in fp32, and after that rounding two m = 2 runs and m = 4 / 8 against m = 2 were identical
        in every case -> 0 (identical fields)."""
import numpy as np
import pytest

from field_interpolation_b200 import workloads as W

pytestmark = pytest.mark.gpu

TOL = {"f32": 2.0e-6, "f64": 0.0}
ITERS = list(range(1, 18)) + [40, 41]


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


@pytest.fixture(scope="module")
def fi():
    import field_interpolation_b200 as m
    return m


def lattice_3d(fi):
    """The 3D lattice of test_fused_pcg_matches_unfused."""
    sizes = [64, 40, 24]
    cloud = W.sphere_torus_3d(3000, seed=9)
    return fi.sdf_from_points(sizes, fi.Weights(), W.to_lattice(cloud["unit_pos"], sizes), cloud["normals"])


def lattice_2d(fi):
    sizes = [96, 70]
    cloud = W.circles_2d(600, seed=4)
    return fi.sdf_from_points(sizes, fi.Weights(model_1=0.1, model_2=1.0, gradient_smoothness=0.3),
                              W.to_lattice(cloud["unit_pos"], sizes), cloud["normals"])


def set_ring(monkeypatch, ring):
    if ring is None:
        monkeypatch.delenv("FI_B200_X_RING", raising=False)
    else:
        monkeypatch.setenv("FI_B200_X_RING", str(ring))


def solve(fi, f, monkeypatch, ring, prec, its, tol=1e-30, check_every=8):
    set_ring(monkeypatch, ring)
    P = fi.FI_F32 if prec == "f32" else fi.FI_F64
    return f.solve(fi.solve_options(P, its, tol, check_every=check_every))


@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("make", [lattice_3d, lattice_2d], ids=["3d", "2d"])
def test_x_ring_same_iterates_every_pending_count(fi, monkeypatch, make, prec):
    """Iteration counts 1..17, 40 and 41 leave every number of directions pending at the end (0 .. m-1 for m = 2, 4, 8):
    same iteration counts as m = 2, x within TOL of it."""
    f = make(fi)
    for its in ITERS:
        x2, s2 = solve(fi, f, monkeypatch, 2, prec, its)
        assert s2["iterations"] == its
        for ring in (4, 8, None):
            x, s = solve(fi, f, monkeypatch, ring, prec, its)
            assert s["iterations"] == its, (ring, its)
            assert rel(x, x2) <= TOL[prec], (ring, its, rel(x, x2))


@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_x_ring_check_every_not_a_multiple(fi, monkeypatch, prec):
    """check_every is rounded up to whole rings (graph slot i is ring position i mod m): 3, 5 and 6 iterations per
    convergence poll give what 8 gives."""
    f = lattice_3d(fi)
    for its in (13, 40):
        x2, _ = solve(fi, f, monkeypatch, 2, prec, its)
        for ring in (4, 8):
            for ce in (3, 5, 6):
                x, s = solve(fi, f, monkeypatch, ring, prec, its, check_every=ce)
                assert s["iterations"] == its, (ring, ce)
                assert rel(x, x2) <= TOL[prec], (ring, ce, rel(x, x2))


@pytest.mark.parametrize("prec", ["f32", "f64"])
@pytest.mark.parametrize("make", [lattice_3d, lattice_2d], ids=["3d", "2d"])
def test_x_ring_tolerance_stop(fi, monkeypatch, make, prec):
    """A solve stopped by the tolerance (mid-graph, any ring position) converges as with m = 2: the same iteration count
    and the same true-residual guarantee as test_fused_pcg_matches_unfused asks of the fused iteration."""
    f = make(fi)
    x2, s2 = solve(fi, f, monkeypatch, 2, prec, 0, tol=1e-5, check_every=32)
    for ring in (4, 8):
        x, s = solve(fi, f, monkeypatch, ring, prec, 0, tol=1e-5, check_every=32)
        assert s["iterations"] == s2["iterations"], (ring, s, s2)
        assert s["relative_residual"] <= 1e-5, s
        assert s["true_residual"] <= (1e-4 if prec == "f32" else 1.25e-5), s
        assert prec == "f32" or s["converged"]
        assert rel(x, x2) <= 1e-3


def test_x_ring_policy_and_override(fi, monkeypatch):
    """The default keeps m = 2 where the two-direction working set is L2-resident (the 2D lattice: six vectors of 27 KB);
    FI_B200_X_RING overrides it; x_ring reports the ring the solve ran with."""
    f = lattice_2d(fi)
    opt = fi.solve_options(fi.FI_F32, 0, 1e-6)
    set_ring(monkeypatch, None)
    t = f.time_iterations(8, opt)
    assert t["fused"] and t["x_ring"] == 2
    for ring in (2, 4, 8):
        set_ring(monkeypatch, ring)
        assert f.time_iterations(8, opt)["x_ring"] == ring
    set_ring(monkeypatch, 3)
    with pytest.raises(Exception):
        f.time_iterations(8, opt)
    # the unfused iteration updates x every iteration, whatever the switch says
    set_ring(monkeypatch, 8)
    t = f.time_iterations(8, fi.solve_options(fi.FI_F32, 0, 1e-6, use_fast_stencil=False))
    assert not t["fused"] and t["x_ring"] == 1
