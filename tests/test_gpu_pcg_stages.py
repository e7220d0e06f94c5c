"""GPU: the Jacobi-PCG iteration of csrc/solver.cu kernel by kernel against its fp64 restatement (tests/pcg_reference.py).

The outer CG absorbs small errors in these kernels — a wrong halo row, a dropped cross term on one chunk boundary or a
wrong parity in beta costs a few iterations and still converges — so each stage runs alone through the test hook
fi_field_pcg_stage (the solve's operator, work buffers and launch helpers) on given vectors and a given scalar state:

* the fused direction+stencil kernel (3D TMA, tiled 3D, 2D TMA; R = 1 / 2 / 4, gradient smoothness on and off, 7- and
  8-row tiles, one and several z chunks), at iteration 0 and with a non-trivial beta of both parities;
* the data term (cell blocks, node-major, split, CSR rows);
* the update of every ring position for m = 2 / 4 / 8, the pending flush, and the unfused pair;
* the scalar edges (done on entry, breakdown, the three stopping rules) and bitwise repeatability;
* whole fp64 solves of k iterations against the restated loop.

Every stage reports the instantiation it launched; each test asserts the one it means to cover (the 3D TMA tile rows
and z chunks against a restatement of launch_gs / plan_chunks), so a dispatch change fails instead of quietly testing
something else.

Bounds are per entry and derived from the rounding of each operation (u = 2^-24 or 2^-53); each is written beside its
assertion.  scripts/pcg_stage_spread.py records the worst error / bound per stage and case on the B200.  With
FI_B200_TEST_EMU=1 the small cases run on the CPU emulator (tests/emu/)."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import pcg_reference as PR
from conftest import ROOT
from field_interpolation_b200 import _lib as L
from field_interpolation_b200 import workloads as W

pytestmark = pytest.mark.gpu

EMU = os.environ.get("FI_B200_TEST_EMU") == "1"
F32, F64 = L.FI_F32, L.FI_F64
U = {F32: 2.0 ** -24, F64: 2.0 ** -53}
DT = {F32: np.float32, F64: np.float64}
U64 = 2.0 ** -53
ALL_ON = dict(model_0=0.1, model_1=0.2, model_2=0.5, model_3=0.3, model_4=0.25)


@pytest.fixture(scope="module")
def fi():
    import field_interpolation_b200 as m
    return m


def sm_count():
    if EMU:
        return 4  # the emulator's "GPU" (tests/emu/cuda_emu.cpp)
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def env_int(name):
    v = os.environ.get(name)
    return int(v) if v else 0


def data_kind():
    v = os.environ.get("FI_B200_DATA_TERM", "")
    return L.FI_PCG_DATA_NODES if v.startswith("n") else L.FI_PCG_DATA_SPLIT if v.startswith("s") else L.FI_PCG_DATA_CELLS


# ---- problems -----------------------------------------------------------------------------------------------------
class Case:
    """A field built as add_model calls, add_points, caller rows / border rows; its restated operator."""

    def __init__(self, fi, sizes, models, vk=1, gk=1, npts=None, rows=False, border=False, cloud=None, seed=0):
        self.sizes, self.models, self.D = list(sizes), models, len(sizes)
        self.n = int(np.prod(sizes))
        f = fi.LatticeField(sizes)
        for w in models:
            fi.add_field_constraints(f, fi.Weights(**w))
        nmodel, _ = f.counts()
        if cloud is None:
            pos, nrm = W.random_cloud(self.D, npts or max(8, self.n // 20), sizes, seed=seed + self.n)
        else:
            pos, nrm = cloud
        fi.add_points(f, 1.0, vk, 0.7, gk, pos, nrm)
        if rows:
            fi.add_equation(f, 0.7, 1.5, [(0, 1.0), (self.n - 1, -2.0), (self.n // 2, 0.5)])
            fi.add_equation(f, 0.3, -1.0, [(self.n // 3, 2.0)])
        if border:
            fi.add_border_distance_constraints(f, 0.3, pos[:64])
        nr, nt = f.counts()
        trips = np.empty(0, dtype=[("row", np.int32), ("col", np.int32), ("value", np.float32)])
        if nr > nmodel:
            # triplets of the rows from nmodel on: the difference of two counts
            g = fi.LatticeField(sizes)
            for w in models:
                fi.add_field_constraints(g, fi.Weights(**w))
            _, tm = g.counts()
            g.close()
            trips = np.empty(nt - tm, dtype=trips.dtype)
            rhs = np.empty(nr - nmodel, np.float32)
            L.check(L.lib().fi_field_export_rows(f._h, nmodel, C.c_void_p(trips.ctypes.data), C.c_void_p(rhs.ctypes.data)))
        self.f = f
        self.A_pts = PR.rows_matrix(trips, nmodel, nr - nmodel, self.n)
        self.op = PR.Operator(sizes, models, self.A_pts)
        self.has_rows = rows or border or (gk == 2 and self.D >= 2)
        # most rows that touch one node: the blocks and the atomics into q add at most that many terms
        self.K = int(np.diff(self.A_pts.tocsc().indptr).max()) if self.A_pts.nnz else 0
        self._minv = {}

    def minv(self, prec):
        """M^-1 exactly as the device holds it: 1 / diag in the operator's precision, 1 where diag is 0."""
        if prec not in self._minv:
            d = self.f.diagonal(prec)
            one = DT[prec](1)
            self._minv[prec] = np.where(d != 0, one / np.where(d != 0, d, one), one).astype(DT[prec])
        return self._minv[prec]

    @property
    def gs(self):
        return self.op.S.gs2 > 0

    @property
    def R(self):
        r = self.op.S.radius
        return 1 if r <= 1 else (2 if r == 2 else 4)


_CASES = {}


def case(fi, key, **kw):
    if key not in _CASES:
        _CASES[key] = Case(fi, **kw)
    return _CASES[key]


def opts(fi, prec, mode=1, **kw):
    return fi.solve_options(prec, kw.pop("max_iterations", 0), kw.pop("tolerance", 1e-30), use_fast_stencil=mode, **kw)


# ---- which kernel the dispatch should pick: restated from stencil_tma.cu / stencil_fast.cu / stencil_2d.cu ----------
def tma_plan(sizes, R, prec, sm):
    """(tile rows, z chunks) of launch_gs / plan_chunks."""
    nx, ny, nz = sizes
    V = 4 if prec == F32 else 2
    S, MINB = {1: (3, 2), 2: (3, 2), 4: (2, 1)}[R]
    txc = 32 * V

    def plan(ty):
        tiles = math.ceil(nx / txc) * math.ceil(ny / ty)
        resident = sm * MINB
        best, chunks = 1e300, 1
        for c in range(1, min(max(1, nz // (2 * R + 1)), 256) + 1):
            zc = math.ceil(nz / c)
            cc = math.ceil(nz / zc)
            waves = math.ceil(tiles * cc / resident)
            cost = max(waves - 0.5, tiles * cc / resident) * (zc + 2 * R + S + 1)
            if cost < best - 1e-9:
                best, chunks = cost, cc
        return chunks

    c8 = plan(8)
    if R <= 2:
        forced = env_int("FI_B200_STENCIL_TY")
        c7 = plan(7)

        def busiest(ty, ch):
            blocks = math.ceil(nx / txc) * math.ceil(ny / ty) * ch
            return math.ceil(blocks / (sm * MINB)) * (math.ceil(nz / ch) + 2 * R + S + 1) * ty
        if forced == 7 or (forced != 8 and busiest(7, c7) < 0.97 * busiest(8, c8)):
            return 7, c7
    return 8, c8


def expected_stencil(c, prec, mode):
    """(kind, R, gs, tile rows, z chunks) the fused step should launch, or kind NONE."""
    V = 4 if prec == F32 else 2
    s = c.sizes
    if c.op.S.radius < 1:
        return (L.FI_PCG_KERNEL_NONE,)
    if c.D == 2 and mode == 1 and s[0] % V == 0 and s[0] >= 32 and s[1] >= 8:
        return (L.FI_PCG_KERNEL_TMA_2D, c.R, int(c.gs), 16, 1)
    if c.D == 3 and s[0] % V == 0 and s[0] >= 32 and s[1] >= 8 and s[2] >= 8:
        if mode == 1:
            return (L.FI_PCG_KERNEL_TMA_3D, c.R, int(c.gs)) + tma_plan(s, c.R, prec, sm_count())
        if mode == 2 and not c.gs:
            tiles = math.ceil(s[0] / (32 * V)) * math.ceil(s[1] / 8)
            ch = min(max(1, sm_count() * 3 * 8 // tiles), max(1, s[2] // 8))
            ch = math.ceil(s[2] / math.ceil(s[2] / ch))
            return (L.FI_PCG_KERNEL_TILED_3D, c.R, 0, 8, ch)
    return (L.FI_PCG_KERNEL_NONE,)


def check(name, got, want, bound, ratios):
    """|got - want| <= bound entry by entry; records the worst ratio."""
    got, want, bound = np.asarray(got, np.float64), np.asarray(want, np.float64), np.asarray(bound, np.float64)
    err = np.abs(got - want)
    ratio = float(np.max(err / np.maximum(bound, 1e-300))) if err.size else 0.0
    ratios[name] = max(ratios.get(name, 0.0), ratio)
    if not ratio <= 1.0:
        k = int(np.argmax(err / np.maximum(bound, 1e-300)))
        raise AssertionError(f"{name}: entry {k} off by {err.flat[k]:.3g}, bound {bound.flat[k]:.3g} (ratio {ratio:.3g})")


def axpy_bound(u, y, t):
    """y + t in T with t = a v, a rounded to T: u |y| + 3u |t| to first order, (1 + 4u) for the second; plus the fp64
    reference's own product and sum (2 u64 (|y| + |t|), which matters when T is fp64)."""
    return (u * np.abs(y) + 3 * u * np.abs(t)) * (1 + 4 * u) + 2 * U64 * (np.abs(y) + np.abs(t))


def sum_terms(n, blocks, per_thread):
    """Longest chain of fp64 additions of a reduction: per_thread sequential terms, the block's shuffle tree (8), the
    blocks added in order by the last one, and numpy's pairwise sum of the reference (log2 n)."""
    return per_thread + 8 + blocks + math.ceil(math.log2(max(n, 2)))


def vec_sum_terms(n):
    """sum_terms of the vector kernels' grid-stride walk (vec_grid: at most 8 blocks of 256 threads per SM)."""
    grid = max(1, min(math.ceil(n / 256), sm_count() * 8))
    return sum_terms(n, grid, math.ceil(n / (grid * 256)))


def as64(a):
    return np.asarray(a.cpu().numpy() if hasattr(a, "cpu") else a, np.float64)


# ---- 1. fused direction + stencil ----------------------------------------------------------------------------------
def stencil_terms(c):
    """Terms the kernel sums per entry: 2R + 1 taps per axis, the cross terms' 20 (with GS), two coefficient roundings."""
    return c.D * (2 * c.R + 1) + (20 if c.gs else 0) + 2


def run_stencil(fi, c, prec, mode, par, iters, seed=0, device=False):
    """One STENCIL stage; returns the error / bound ratios.  Also checks the report and that r and p_old are untouched."""
    T, u, n = DT[prec], U[prec], c.n
    rng = np.random.default_rng(seed)
    r, p_old = rng.normal(size=n).astype(T), rng.normal(size=n).astype(T)
    rho = [1.3, 0.7] if par == 0 else [0.45, 1.9]
    st_in = dict(rho=rho, iters=iters, max_iters=1 << 40, bb=1.0)
    dirs = [None, None]
    dirs[par], dirs[par ^ 1] = p_old, np.full(n, 7.0, T)
    vec = dict(r=r, q=np.full(n, -3.0, T), dir=dirs)
    if device:
        import torch
        tt = torch.float32 if prec == F32 else torch.float64
        vec = dict(r=torch.from_numpy(r).cuda(), q=torch.full((n,), -3.0, dtype=tt, device="cuda"),
                   dir=[torch.from_numpy(d).to(dtype=tt).cuda() for d in dirs])
    out, st, rep = c.f.pcg_stage(L.FI_PCG_STENCIL, vec, st_in, par=par, pos=par, ring=2, options=opts(fi, prec, mode))
    want = expected_stencil(c, prec, mode)
    got = (rep["stencil"], rep["radius"], rep["gs"], rep["tile_rows"], rep["z_chunks"])[:len(want)]
    assert got == want, (got, want)
    ratios = {}
    if want[0] == L.FI_PCG_KERNEL_NONE:
        return ratios
    p, q = as64(out["dir"][par ^ 1]), as64(out["q"])
    assert np.array_equal(as64(out["r"]), r) and np.array_equal(as64(out["dir"][par]), p_old)
    beta = 0.0 if iters == 0 else rho[par] / rho[par ^ 1]
    m = c.minv(prec).astype(np.float64)
    mr, bp = m * r.astype(np.float64), beta * p_old.astype(np.float64)
    # p = M r + beta p_old: two products, one sum, beta rounded to T
    check("p", p, mr + bp, 3 * u * (np.abs(mr) + np.abs(bp)) + 2 * U64 * (np.abs(mr) + np.abs(bp)), ratios)
    # q = S p of the kernel's own p: each term and the coefficients rounded once per term summed
    Sabs = c.op.S.apply(p, absolute=True)
    # (the fp64 reference rounds each of its terms too)
    check("q", q, c.op.S.apply(p), stencil_terms(c) * (u + U64) * Sabs, ratios)
    V = 4 if prec == F32 else 2
    pq_abs = float(np.abs(p) @ np.abs(q))
    # pq: V products per pack summed in T, then fp64 sums over the block's planes, the block and the blocks of the grid
    ty, chunks = (want[3], want[4]) if len(want) > 4 else (8, 1)
    nz = c.sizes[2] if c.D == 3 else 1
    blocks = math.ceil(c.sizes[0] / (32 * V)) * math.ceil(c.sizes[1] / ty) * chunks
    b_self = (V + 1) * u * pq_abs + sum_terms(c.n, blocks, math.ceil(nz / chunks)) * U64 * pq_abs
    check("pq_self", st["pq"], float(p @ q), b_self, ratios)
    check("pq_ref", st["pq"], float(p @ c.op.S.apply(p)), b_self + stencil_terms(c) * u * float(np.abs(p) @ Sabs), ratios)
    assert st["iters"] == iters and st["done"] == 0 and st["rho"] == rho
    return ratios


def sc(sizes, models, **kw):
    return dict(sizes=sizes, models=models, **kw)


# (case key, case, precisions, modes): the shapes where tiles go ragged
STENCIL_CASES = {
    # 3D TMA, R = 1 / 2 / 4 (model_3 alone has radius 3: the R = 4 kernel), GS off and on
    "3d_m1_32x9x8": (sc([32, 9, 8], [dict(model_1=0.3, model_2=0.0)]), (F32, F64)),
    "3d_m1gs_36x8x13": (sc([36, 8, 13], [dict(model_1=0.3, model_2=0.0, gradient_smoothness=0.2)]), (F32, F64)),
    "3d_m2_132x10x9": (sc([132, 10, 9], [dict()]), (F32, F64)),
    "3d_m2gs_32x15x40": (sc([32, 15, 40], [dict(gradient_smoothness=0.25)]), (F32, F64)),
    "3d_m3_32x8x8": (sc([32, 8, 8], [dict(model_2=0.0, model_3=0.4)]), (F32, F64)),
    "3d_m4gs_36x9x8": (sc([36, 9, 8], [dict(model_2=0.0, model_4=0.2, gradient_smoothness=0.3)]), (F32, F64)),
    "3d_all_gs_260x8x17": (sc([260, 8, 17], [dict(ALL_ON, gradient_smoothness=0.15)], rows=True), (F32, F64)),
    "3d_all_32x23x12": (sc([32, 23, 12], [ALL_ON], gk=2), (F32, F64)),
    # eligible for the fp64 TMA kernel only (x a multiple of 2, not of 4)
    "3d_m2_34x8x9": (sc([34, 8, 9], [dict(gradient_smoothness=0.1)]), (F64,)),
    "3d_m1_66x9x10": (sc([66, 9, 10], [dict(model_1=0.2)]), (F64,)),
    # tall z: many chunks, chunk boundaries next to the GS ring
    "3d_m1gs_32x8x64": (sc([32, 8, 64], [dict(model_1=0.3, model_2=0.0, gradient_smoothness=0.2)]), (F32, F64)),
    "3d_m2gs_32x16x57": (sc([32, 16, 57], [dict(gradient_smoothness=0.3)], border=True), (F32,)),
    # 2D TMA, R = 1 / 2 / 4 x GS
    "2d_m1_32x9": (sc([32, 9], [dict(model_1=0.3, model_2=0.0)]), (F32, F64)),
    "2d_m1gs_36x20": (sc([36, 20], [dict(model_1=0.3, model_2=0.0, gradient_smoothness=0.2)]), (F32, F64)),
    "2d_m2_132x8": (sc([132, 8], [dict()], rows=True), (F32, F64)),
    "2d_m2gs_260x17": (sc([260, 17], [dict(gradient_smoothness=0.3)]), (F32, F64)),
    "2d_m3_32x23": (sc([32, 23], [dict(model_2=0.0, model_3=0.3)], gk=2), (F32, F64)),
    "2d_m4gs_34x12": (sc([34, 12], [dict(ALL_ON, gradient_smoothness=0.2)]), (F64,)),
}


@pytest.mark.parametrize("iters,par", [(0, 0), (3, 0), (4, 1)])
@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("name", list(STENCIL_CASES))
def test_fused_stencil(fi, name, prec, iters, par):
    kw, precs = STENCIL_CASES[name]
    if prec not in precs:
        pytest.skip("x size not eligible for the fp32 TMA kernel")
    c = case(fi, name, **kw)
    run_stencil(fi, c, prec, 1, par, iters, seed=iters)


@pytest.mark.parametrize("name", ["3d_m1_32x9x8", "3d_m2_132x10x9", "3d_m3_32x8x8", "3d_all_32x23x12", "3d_m1gs_32x8x64"])
def test_tiled_stencil(fi, name):
    """use_fast_stencil = 2: the tiled kernel's fused form, R = 1 / 2 / 4; with GS it has none (NONE reported, nothing
    ran: the solve runs the unfused pair there)."""
    kw, _ = STENCIL_CASES[name]
    c = case(fi, name, **kw)
    for prec in (F32, F64):
        run_stencil(fi, c, prec, 2, 1, 5, seed=7)


def test_bench_launch_shape(fi):
    """512 x 512 x 16, fp32, default weights: launch_gs picks 7-row tiles and one z chunk on a 148-SM B200 (the bench's
    tile rule; the planes are the bench's)."""
    if EMU or sm_count() != 148:
        pytest.skip("the rule is stated for a 148-SM B200")
    if env_int("FI_B200_STENCIL_TY"):
        pytest.skip("tile rows forced")
    assert tma_plan([512, 512, 16], 2, F32, 148) == (7, 1)
    c = case(fi, "bench_planes", sizes=[512, 512, 16], models=[dict()], npts=20000)
    run_stencil(fi, c, F32, 1, 1, 2)


# ---- 2. data term ------------------------------------------------------------------------------------------------
DATA_CASES = {
    "1d_points": sc([301], [dict(model_1=0.2)], npts=200),
    "1d_rows": sc([64], [dict()], rows=True, gk=0),
    "2d_points": sc([40, 33], [dict()], npts=300),
    "2d_linear_grad": sc([36, 20], [dict()], gk=2, npts=200),
    "2d_rows_border": sc([33, 17], [dict()], rows=True, border=True, npts=150),
    "3d_points": sc([20, 17, 9], [dict()], npts=400, vk=0, gk=0),
    "3d_linear_grad": sc([16, 12, 10], [dict()], gk=2, npts=300),
    "3d_rows_border": sc([12, 11, 9], [dict()], rows=True, border=True, npts=250),
}


def run_data(fi, c, prec, seed=0):
    T, u, n = DT[prec], U[prec], c.n
    rng = np.random.default_rng(seed)
    p, q_in = rng.normal(size=n).astype(T), rng.normal(size=n).astype(T)
    out, st, rep = c.f.pcg_stage(L.FI_PCG_DATA, dict(q=q_in, dir=[np.zeros(n, T), p]), dict(pq=2.5, max_iters=10),
                                 par=0, pos=0, ring=2, options=opts(fi, prec))
    want_bits = data_kind() | (L.FI_PCG_DATA_ROWS if c.has_rows else 0)
    assert rep["data_term"] == want_bits, (rep, want_bits)
    ratios = {}
    p64 = p.astype(np.float64)
    Pp, Pabs = c.op.data(p64), c.op.data(p64, absolute=True)
    C_ = 2 ** c.D
    # blocks: D + 1 products per row and up to K rows folded per entry; apply: C terms per cell; atomics into q: up to C
    # cells and K rows per node, plus q itself
    cd = (c.D + 1 + c.K) + C_ + (C_ + c.K + 1)
    check("data_q", out["q"], q_in.astype(np.float64) + Pp, cd * (u + U64) * (Pabs + np.abs(q_in)), ratios)
    check("data_pq", st["pq"], 2.5 + float(p64 @ Pp), cd * (u + U64) * float(np.abs(p64) @ Pabs) + 2.5 * U64 * 4, ratios)
    assert np.array_equal(out["dir"][1], p)
    return ratios


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("name", list(DATA_CASES))
def test_data_term(fi, name, prec):
    run_data(fi, case(fi, "data_" + name, **DATA_CASES[name]), prec)


# ---- 3. ring update, pending flush, unfused pair ----------------------------------------------------------------------
def update_inputs(c, prec, m, seed):
    T, n = DT[prec], c.n
    rng = np.random.default_rng(seed)
    vec = dict(x=rng.normal(size=n).astype(T), r=rng.normal(size=n).astype(T), q=rng.normal(size=n).astype(T),
               dir=[rng.normal(size=n).astype(T) for _ in range(m)])
    alpha = list(rng.uniform(0.2, 1.5, size=7))
    return vec, alpha


def run_update(fi, c, prec, m, pos, seed=0):
    T, u, n = DT[prec], U[prec], c.n
    par = pos & 1
    vec, alpha = update_inputs(c, prec, m, seed + 10 * m + pos)
    st_in = dict(rho=[0.8, 1.1], pq=1.7, iters=11, max_iters=1000, tol2bb=1e-30, bb=1.0, alpha=alpha)
    out, st, _ = c.f.pcg_stage(L.FI_PCG_UPDATE, vec, st_in, par=par, pos=pos, ring=m, options=opts(fi, prec))
    ratios = {}
    a = st_in["rho"][par] / st_in["pq"]
    x, r, q = (vec[k].astype(np.float64) for k in ("x", "r", "q"))
    # r -= a q: a rounded to T, one product (2u |a q|), one difference (u |r - a q|)
    check("update_r", out["r"], r - a * q, axpy_bound(u, r, a * q), ratios)
    rk = as64(out["r"])
    m_ = c.minv(prec).astype(np.float64)
    rho_abs = float(np.abs(rk) @ np.abs(m_ * rk))
    # r.M^-1 r of the kernel's r: M^-1 r rounded to T, fp64 sums
    check("update_rho", st["rho"][par ^ 1], float(rk @ (m_ * rk)), (u + vec_sum_terms(n) * U64) * rho_abs, ratios)
    check("update_rr", st["rr"], float(rk @ rk), vec_sum_terms(n) * U64 * float(rk @ rk), ratios)
    assert st["rho"][par] == st_in["rho"][par] and st["iters"] == 12 and st["done"] == 0
    if pos < m - 1:  # skip form: a parked, x untouched
        assert np.array_equal(out["x"], vec["x"])
        assert st["alpha"][pos] == a
        assert [st["alpha"][j] for j in range(7) if j != pos] == [alpha[j] for j in range(7) if j != pos]
    else:  # flush form: x += a_0 d_1 + ... + a_m-2 d_m-1 + a d_0 (p_k-m+1 .. p_k), oldest first
        terms = [alpha[j] * vec["dir"][(j + 1) % m].astype(np.float64) for j in range(m - 1)] + [a * vec["dir"][0].astype(np.float64)]
        s = np.sum(terms, axis=0)
        absum = np.sum(np.abs(terms), axis=0)
        # m coefficients rounded to T, m products, m - 1 sums, one add to x
        check("flush_x", out["x"], x + s, (m + 2) * (u + U64) * (np.abs(x) + absum), ratios)
        assert st["alpha"] == alpha
    for j in range(m):
        assert np.array_equal(out["dir"][j], vec["dir"][j])
    return ratios


UPDATE_CASE = sc([36, 9, 10], [dict(gradient_smoothness=0.1)], npts=150)


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("m", [2, 4, 8])
def test_ring_update(fi, m, prec):
    c = case(fi, "update", **UPDATE_CASE)
    for pos in range(m):
        run_update(fi, c, prec, m, pos)


def run_flush(fi, c, prec, m, count, seed=0):
    T, u = DT[prec], U[prec]
    vec, alpha = update_inputs(c, prec, m, seed + 100 + count)
    st_in = dict(rho=[0.8, 1.1], pq=1.7, iters=11, max_iters=12, done=1, alpha=alpha)  # runs after the loop: done set
    out, st, _ = c.f.pcg_stage(L.FI_PCG_FLUSH, vec, st_in, ring=m, count=count, options=opts(fi, prec))
    ratios = {}
    terms = [alpha[i] * vec["dir"][i + 1].astype(np.float64) for i in range(count)]
    x = vec["x"].astype(np.float64)
    check("pending_x", out["x"], x + np.sum(terms, axis=0), (count + 2) * (u + U64) * (np.abs(x) + np.sum(np.abs(terms), axis=0)), ratios)
    assert np.array_equal(out["r"], vec["r"]) and np.array_equal(out["q"], vec["q"])
    assert st["iters"] == 11 and st["alpha"] == alpha
    return ratios


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("m", [2, 4, 8])
def test_pending_flush(fi, m, prec):
    c = case(fi, "update", **UPDATE_CASE)
    for count in range(1, m):
        run_flush(fi, c, prec, m, count)


def run_unfused(fi, c, prec, par, seed=0):
    T, u = DT[prec], U[prec]
    vec, _ = update_inputs(c, prec, 1, seed + par)
    st_in = dict(rho=[0.8, 1.1], pq=1.7, iters=5, max_iters=1000, tol2bb=1e-30, bb=1.0)
    out, st, _ = c.f.pcg_stage(L.FI_PCG_UNFUSED, vec, st_in, par=par, ring=2, options=opts(fi, prec))
    ratios = {}
    a = st_in["rho"][par] / st_in["pq"]
    x, r, q = (vec[k].astype(np.float64) for k in ("x", "r", "q"))
    p = vec["dir"][0].astype(np.float64)
    check("unfused_x", out["x"], x + a * p, axpy_bound(u, x, a * p), ratios)
    check("unfused_r", out["r"], r - a * q, axpy_bound(u, r, a * q), ratios)
    rk, m_ = as64(out["r"]), c.minv(prec).astype(np.float64)
    rho_new = float(rk @ (m_ * rk))
    check("unfused_rho", st["rho"][par ^ 1], rho_new, (u + vec_sum_terms(c.n) * U64) * float(np.abs(rk) @ np.abs(m_ * rk)), ratios)
    # p = M r + beta p, beta = rho_new / rho_old from the state
    beta = st["rho"][par ^ 1] / st_in["rho"][par]
    mr, bp = m_ * rk, beta * p
    check("unfused_p", out["dir"][0], mr + bp, (3 * u + 2 * U64) * (np.abs(mr) + np.abs(bp)), ratios)
    assert st["iters"] == 6 and st["done"] == 0
    return ratios


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("name,kw", [("1d", sc([257], [dict(model_1=0.2)], npts=100)),
                                     ("3d_x33", sc([33, 9, 8], [dict()], npts=150))])
def test_unfused_pair(fi, name, kw, prec):
    """The pair 1D lattices and lattices no fused kernel takes (x = 33) run; the fused step reports NONE there."""
    c = case(fi, "unfused_" + name, **kw)
    for par in (0, 1):
        run_unfused(fi, c, prec, par)
    assert expected_stencil(c, prec, 1) == (L.FI_PCG_KERNEL_NONE,)
    run_stencil(fi, c, prec, 1, 0, 0)


# ---- 4. init --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("guess", [False, True])
def test_init(fi, prec, guess):
    c = case(fi, "3d_m1gs_36x8x13", **STENCIL_CASES["3d_m1gs_36x8x13"][0])
    T, u, n = DT[prec], U[prec], c.n
    rng = np.random.default_rng(5)
    b = rng.normal(size=n).astype(T)
    vec = dict(b=b, r=np.zeros(n, T), q=np.zeros(n, T), dir=[np.zeros(n, T), np.zeros(n, T)])
    if guess:
        vec["x"] = (0.1 * rng.normal(size=n)).astype(T)
    out, st, _ = c.f.pcg_stage(L.FI_PCG_INIT, vec, {}, options=opts(fi, prec, tolerance=1e-3, max_iterations=77))
    ratios = {}
    b64 = b.astype(np.float64)
    if guess:
        x = vec["x"].astype(np.float64)
        Ax, Aabs = c.op.apply(x), c.op.apply(x, absolute=True)
        cd = (c.D + 1 + c.K) + 2 * 2 ** c.D + c.K + 1
        # r = b - A x: A x by the unfused stencil and the data term, one difference
        check("init_r", out["r"], b64 - Ax, u * np.abs(b64) + (stencil_terms(c) + cd + 1) * u * Aabs, ratios)
    else:
        assert np.array_equal(out["r"], b)
    r = as64(out["r"])
    m_ = c.minv(prec).astype(np.float64)
    check("init_p", out["dir"][0], m_ * r, u * np.abs(m_ * r), ratios)
    z = as64(out["dir"][0])
    assert st["rho"][0] == pytest.approx(float(r @ z), rel=1e-12) and st["rho"][1] == 0.0
    assert st["rr"] == pytest.approx(float(r @ r), rel=1e-12) and st["rr0"] == st["rr"]
    assert st["bb"] == pytest.approx(float(b64 @ b64), rel=1e-12) and st["tol2bb"] == 1e-6 * st["bb"]
    assert st["iters"] == 0 and st["max_iters"] == 77 and st["done"] == 0 and st["breakdown"] == 0 and st["pq"] == 0.0


# ---- 5. scalar edges and repeatability ---------------------------------------------------------------------------------
EDGE = "3d_m2gs_32x15x40"


def edge_case(fi):
    return case(fi, EDGE, **STENCIL_CASES[EDGE][0])


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("stage,pos", [(L.FI_PCG_STENCIL, 0), (L.FI_PCG_DATA, 1), (L.FI_PCG_UPDATE, 0), (L.FI_PCG_UPDATE, 3),
                                       (L.FI_PCG_UNFUSED, 0)])
def test_done_on_entry_changes_nothing(fi, prec, stage, pos):
    c = edge_case(fi)
    vec, alpha = update_inputs(c, prec, 4, 3)
    st_in = dict(rho=[0.8, 1.1], pq=1.7, iters=9, max_iters=1000, tol2bb=1e-30, bb=1.0, done=1, alpha=alpha)
    out, st, _ = c.f.pcg_stage(stage, vec, st_in, par=pos & 1, pos=pos, ring=4, options=opts(fi, prec))
    for k in ("x", "r", "q"):
        assert np.array_equal(out[k], vec[k]), k
    for j in range(4):
        assert np.array_equal(out["dir"][j], vec["dir"][j]), j
    for k, v in st_in.items():
        assert st[k] == v, k
    assert st["breakdown"] == 0


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("pq", [0.0, -1.0, float("nan")])
@pytest.mark.parametrize("stage,pos", [(L.FI_PCG_UPDATE, 0), (L.FI_PCG_UPDATE, 3), (L.FI_PCG_UNFUSED, 0)])
def test_breakdown(fi, prec, pq, stage, pos):
    """pq <= 0 or NaN: breakdown = 1, done = 1, no vector touched, nothing parked, iters unchanged."""
    c = edge_case(fi)
    vec, alpha = update_inputs(c, prec, 4, 4)
    st_in = dict(rho=[0.8, 1.1], pq=pq, iters=9, max_iters=1000, tol2bb=1e-30, bb=1.0, alpha=alpha)
    out, st, _ = c.f.pcg_stage(stage, vec, st_in, par=pos & 1, pos=pos, ring=4, options=opts(fi, prec))
    assert st["breakdown"] == 1 and st["done"] == 1 and st["iters"] == 9 and st["rho"] == st_in["rho"] and st["alpha"] == alpha
    for k in ("x", "r", "q"):
        assert np.array_equal(out[k], vec[k]), k
    for j in range(4):
        assert np.array_equal(out["dir"][j], vec["dir"][j]), j


@pytest.mark.parametrize("prec", [F32, F64])
@pytest.mark.parametrize("stage", [L.FI_PCG_UPDATE, L.FI_PCG_UNFUSED])
def test_stopping_rules(fi, prec, stage):
    """done is set exactly when rr <= tol2bb, iters + 1 = max_iters or rho <= 0, and not otherwise."""
    c = edge_case(fi)
    T = DT[prec]
    vec, alpha = update_inputs(c, prec, 2, 5)

    def run(**kw):
        st_in = dict(dict(rho=[0.8, 1.1], pq=1.7, iters=9, max_iters=1000, tol2bb=1e-30, bb=1.0, alpha=alpha), **kw)
        v = dict(vec, q=kw.pop("q", vec["q"])) if "q" in kw else vec
        st_in.pop("q", None)
        return c.f.pcg_stage(stage, v, st_in, par=0, pos=0, ring=2, options=opts(fi, prec))[1]

    st = run()
    assert st["done"] == 0 and st["iters"] == 10
    st = run(tol2bb=1e300)
    assert st["done"] == 1 and st["breakdown"] == 0 and st["iters"] == 10
    assert run(max_iters=10)["done"] == 1 and run(max_iters=11)["done"] == 0
    # q = r and pq = rho: a = 1 and r becomes exactly zero, so rho = rr = 0; with tol2bb < 0 only rho <= 0 stops it
    st = run(q=vec["r"].copy(), pq=0.8, tol2bb=-1.0)
    assert st["rr"] == 0.0 and st["rho"][1] == 0.0 and st["done"] == 1 and st["breakdown"] == 0


@pytest.mark.parametrize("prec", [F32, F64])
def test_repeat_launches_are_bit_identical(fi, prec):
    """Stencil and update dot products repeat bit for bit (DESIGN.md §4: fixed-order grid sums); the second launch also
    shows that the grid-sum tickets re-armed."""
    c = edge_case(fi)
    vec, alpha = update_inputs(c, prec, 2, 6)
    st_in = dict(rho=[0.8, 1.1], pq=1.7, iters=3, max_iters=1000, tol2bb=1e-30, bb=1.0, alpha=alpha)
    for stage in (L.FI_PCG_STENCIL, L.FI_PCG_UPDATE, L.FI_PCG_UNFUSED):
        a = c.f.pcg_stage(stage, vec, st_in, par=1, pos=1, ring=2, options=opts(fi, prec))
        b = c.f.pcg_stage(stage, vec, st_in, par=1, pos=1, ring=2, options=opts(fi, prec))
        assert a[1] == b[1], (stage, a[1], b[1])
        for k in ("x", "r", "q"):
            assert np.array_equal(a[0][k], b[0][k])
        for j in range(2):
            assert np.array_equal(a[0]["dir"][j], b[0]["dir"][j])


# ---- 6. whole loop ------------------------------------------------------------------------------------------------
LOOP_CASES = {
    "3d_r1_gs": sc([32, 8, 12], [dict(model_1=0.3, model_2=0.0, gradient_smoothness=0.2)], npts=120),
    "2d_r4": sc([36, 20], [dict(model_2=0.0, model_4=0.2)], npts=90, rows=True),
}


@pytest.mark.parametrize("ring,check_every", [(2, 3), (4, 5), (8, 7), (8, 32)])
@pytest.mark.parametrize("name", list(LOOP_CASES))
def test_k_iterations_match_reference(fi, name, ring, check_every, monkeypatch):
    """fp64 solves of exactly k iterations (tolerance 1e-30) against the restated fp64 PCG from the device's A^T b and
    M^-1: x after its narrowing to fp32 and relative_residual = sqrt(rr / bb)."""
    monkeypatch.setenv("FI_B200_X_RING", str(ring))
    c = case(fi, "loop_" + name, **LOOP_CASES[name])
    atb = c.f.rhs(F64)
    minv = c.minv(F64).astype(np.float64)

    class Op:
        n = c.n
        apply = staticmethod(c.op.apply)

        @staticmethod
        def minv():
            return minv
    ks = list(range(1, 18)) + [40, 41]
    for k in ks:
        x, st = c.f.solve(opts(fi, F64, max_iterations=k, tolerance=1e-30, check_every=check_every))
        xr, rr, _, sr = PR.pcg(Op, atb, k)
        assert st["iterations"] == k and sr["iters"] == k
        # fp32 narrowing (half an ulp each side) plus the fp64 loops' difference, far below it
        tol = 2.0 ** -23 * np.abs(xr) + 1e-9 * np.abs(xr).max()
        assert np.all(np.abs(x - xr) <= tol), (k, float(np.max(np.abs(x - xr) / tol)))
        assert st["relative_residual"] == pytest.approx(math.sqrt(sr["rr"] / sr["bb"]), rel=1e-7), k


# ---- 7. full size ---------------------------------------------------------------------------------------------------
@pytest.mark.skipif(EMU, reason="full-size lattices")
def test_full_size_512_f32(fi):
    """512^3 fp32 with the bench's cloud (1 M points of sphere_torus_3d, seed 0), vectors on the device: one fused
    stencil stage, the data term and a flush-form update against the slab-wise reference."""
    sizes = [512, 512, 512]
    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    c = case(fi, "full_512", sizes=sizes, models=[dict()], cloud=(W.to_lattice(cloud["unit_pos"], sizes), cloud["normals"]))
    run_stencil(fi, c, F32, 1, 1, 3, device=True)
    run_data(fi, c, F32)
    run_update(fi, c, F32, 2, 1)


@pytest.mark.skipif(EMU, reason="full-size lattices")
def test_full_size_2048sq_f32(fi):
    """C3: 2048^2 fp32 with 200k circle samples, the 2D kernel."""
    cl = W.circles_2d(200_000, seed=0)
    sizes = [2048, 2048]
    c = case(fi, "full_2048", sizes=sizes, models=[dict()], cloud=(W.to_lattice(cl["unit_pos"], sizes), cl["normals"]))
    run_stencil(fi, c, F32, 1, 0, 2)
    run_data(fi, c, F32)


@pytest.mark.skipif(EMU, reason="full-size lattices")
def test_full_size_256_f64(fi):
    sizes = [256, 256, 256]
    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    c = case(fi, "full_256", sizes=sizes, models=[dict()], cloud=(W.to_lattice(cloud["unit_pos"], sizes), cloud["normals"]))
    run_stencil(fi, c, F64, 1, 1, 3)
    run_data(fi, c, F64)


# ---- 8. process-wide switches -----------------------------------------------------------------------------------------
@pytest.mark.skipif(EMU, reason="child processes of the GPU build")
@pytest.mark.parametrize("env", ["FI_B200_DATA_TERM=node", "FI_B200_DATA_TERM=split", "FI_B200_STENCIL_TY=8", "FI_B200_STENCIL_TY=7"])
def test_process_wide_switches(env):
    """Kernel switches read once per process: the stencil and data-term checks above in a child pytest per setting (the
    expected report follows the setting)."""
    k, v = env.split("=")
    child = dict(os.environ, **{k: v})
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-k",
                        "test_fused_stencil or test_data_term or test_tiled_stencil", "-p", "no:cacheprovider"],
                       env=child, capture_output=True, text=True, timeout=1800, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-1000:]
    assert " passed" in r.stdout and " failed" not in r.stdout
