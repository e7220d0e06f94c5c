"""GPU: fi_sample_field (csrc/sample_field.cuh) — values and gradients of lattice fields at arbitrary points.

Bar: values bit-identical to fi_upscale_field where the upscale formula puts its points; everything bit-identical to
the numpy port (tests/sample_port.py), which tests/test_sample_port.py ties to the reference's rows; the rows' own
measure on the GPU output; linear fields reproduced; marching-cubes vertices sample to iso; grid_sample agrees in the
interior; a solved cloud sampled at its own points; locations, edge cases, errors and the C++ drop-in."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import sample_port as S
from conftest import ROOT, bits
from sample_port import reference_measures, same_values

pytestmark = pytest.mark.gpu
F = np.float32


@pytest.fixture(scope="module")
def fi():
    import field_interpolation_b200 as m
    return m


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def _same_bits(got, want):
    got, want = _host(got), _host(want)
    assert got.shape == want.shape
    assert np.array_equal(bits(got), bits(want))


def _grid(shape):
    """(x, y, z) float64 coordinates of an (nz, ny, nx) lattice, centred."""
    nz, ny, nx = shape
    z, y, x = np.meshgrid(np.arange(nz, dtype=np.float64), np.arange(ny, dtype=np.float64), np.arange(nx, dtype=np.float64), indexing="ij")
    return x - (nx - 1) / 2, y - (ny - 1) / 2, z - (nz - 1) / 2


def sphere_sdf(n, r):
    x, y, z = _grid((n, n, n))
    return (np.sqrt(x * x + y * y + z * z) - r).astype(F)


def torus_sdf(n, R, r):
    x, y, z = _grid((n, n, n))
    q = np.sqrt(x * x + y * y) - R
    return (np.sqrt(q * q + z * z) - r).astype(F)


# ---- 1. values equal fi_upscale_field ----------------------------------------------------------------------------------
@pytest.mark.parametrize("small,large", [([12], [37]), ([5], [5]), ([1], [4]), ([9, 13], [17, 25]), ([4, 3], [11, 3]),
                                         ([7, 9, 11], [13, 17, 21]), ([8, 8, 8], [15, 15, 15]), ([2, 3, 2], [5, 5, 5])])
def test_values_equal_upscale(fi, small, large):
    rng = np.random.default_rng(sum(small) + sum(large))
    f = rng.standard_normal(int(np.prod(small))).astype(F)
    want = fi.upscale_field(f, small, large)
    # the upscale formula's positions (:462): (float)coord * (small - 1.0f) / (large - 1.0f), left to right in fp32
    axes = []
    for s, l in zip(small, large):
        c = np.arange(l, dtype=F)
        axes.append((c * (F(s) - F(1))) / (F(l) - F(1)))
    mesh = np.meshgrid(*axes[::-1], indexing="ij")[::-1]  # x fastest
    pos = np.stack([m.ravel() for m in mesh], axis=1).astype(F)
    got = fi.sample_field(f.reshape(small[::-1]), pos)
    _same_bits(got, want)


# ---- 2. bit-identical to the numpy port ------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(13,), (1,), (2,), (17, 23), (1, 9), (2, 2), (11, 7, 5), (3, 1, 4), (2, 2, 2), (33, 20, 9)])
@pytest.mark.parametrize("kernel", [None, 0, 1, 2])
def test_vs_port(fi, shape, kernel):
    rng = np.random.default_rng(sum(shape) + len(shape))
    f = rng.standard_normal(shape).astype(F)
    sizes = shape[::-1]
    pts = S.positions_of_every_kind(sizes, 3000, seed=len(shape))
    got = fi.sample_field(f, pts, kernel)
    want = S.sample(sizes, f, pts, kernel)
    if kernel is None:
        _same_bits(got, want)
    else:
        _same_bits(got[0], want[0])
        _same_bits(got[1], want[1])


def test_vs_port_512(fi):
    """A 512^3 field (larger than L2) and 1M points of every kind, on the device, all kernels."""
    import torch
    n = 512
    rng = np.random.default_rng(512)
    f = rng.standard_normal((n, n, n), dtype=F)
    pts = S.positions_of_every_kind([n] * 3, 1_000_000, seed=5)
    df, dp = torch.from_numpy(f).cuda(), torch.from_numpy(pts).cuda()
    want_v = S.sample([n] * 3, f, pts)
    _same_bits(fi.sample_field(df, dp), want_v)
    for k in (0, 1, 2):
        v, g = fi.sample_field(df, dp, k)
        _same_bits(v, want_v)
        _same_bits(g, S.sample([n] * 3, f, pts, k)[1])


# ---- 3. against the reference-pinned rows ----------------------------------------------------------------------------------
@pytest.mark.parametrize("sizes", [[9], [6, 5], [4, 3, 5], [3, 1, 4]])
@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_vs_reference_rows(fi, port, sizes, kernel):
    rng = np.random.default_rng(11 * sum(sizes) + kernel)
    x = rng.standard_normal(int(np.prod(sizes))).astype(F)
    pts = S.positions_of_every_kind(sizes, 80, seed=kernel + 3 * sum(sizes))
    v, g = fi.sample_field(x.reshape(sizes[::-1]), pts, kernel)
    want_v, want_g = zip(*(reference_measures(port, sizes, x, p, kernel) for p in pts))
    same_values(v, np.array(want_v, F))
    same_values(g, np.array(want_g, F))


# ---- 4. linear fields ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(31,), (19, 23), (13, 17, 21)])
def test_linear_fields(fi, shape):
    """f = a x + b y + c z + d with dyadic coefficients, so every lattice value is exact in fp32.  Interior values
    match the plane to fp32 rounding; all three kernels return (a, b, c): kernels 0 and 1 exactly (every term is
    exact), kernel 2 to the rounding of its weighted sum."""
    D = len(shape)
    coef = np.array([0.5, -2.0, 0.25][:D])
    d0 = 3.0
    axes = np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij")[::-1]  # x, y, z
    f = (sum(c * a for c, a in zip(coef, axes)) + d0).astype(F)
    scale = np.abs(f).max()
    rng = np.random.default_rng(D)
    pts = rng.uniform(0, np.array(shape[::-1]) - 1, (20_000, D)).astype(F)
    exact = pts.astype(np.float64) @ coef + d0
    for k in (0, 1, 2):
        v, g = fi.sample_field(f, pts, k)
        assert np.abs(v - exact).max() <= 8 * np.finfo(F).eps * scale
        if k < 2:
            assert np.array_equal(g, np.broadcast_to(coef.astype(F), g.shape))
        else:
            assert np.isfinite(g).all() and np.abs(g - coef).max() <= 16 * np.finfo(F).eps * scale


# ---- 5. marching-cubes vertices sample to iso -------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["sphere", "torus"])
@pytest.mark.parametrize("iso", [0.0, 1.25])
def test_marching_cubes_vertices_sample_to_iso(fi, which, iso):
    """Each vertex lies on a lattice edge (lower end a = f - iso, upper end b) at coord + a / (a - b).  Rounding the
    coordinate moves the point by at most ulp(coordinate) (half an ulp for a / (a - b) < 1, half for the sum), which
    changes the linear interpolant by |b - a| per unit; evaluating (1 - t) f_lo + t f_hi over wsum adds a few fp32
    roundings of max(|f_lo|, |f_hi|).  So |sample - iso| <= ulp(coord) |b - a| + 4 eps (|f_lo| + |f_hi|)."""
    n = 64
    f = sphere_sdf(n, 20.0) if which == "sphere" else torus_sdf(n, 18.0, 8.0)
    v, _ = fi.marching_cubes(f, iso)
    assert len(v) > 1000
    s = fi.sample_field(f, v).astype(np.float64)
    flat = f.ravel().astype(np.float64)
    eps = float(np.finfo(F).eps)
    lo = np.floor(v).astype(np.int64)
    frac = v - lo
    assert (frac != 0).sum(axis=1).max() <= 1
    on_edge = (frac != 0).any(axis=1)
    axis = np.argmax(frac != 0, axis=1)
    strides = np.array([1, n, n * n])
    i_lo = lo @ strides
    f_lo, f_hi = flat[i_lo], flat[i_lo + np.where(on_edge, strides[axis], 0)]
    coord = np.abs(v[np.arange(len(v)), axis]).astype(F)
    bound = np.spacing(coord) * np.abs(f_hi - f_lo) + 4 * eps * (np.abs(f_lo) + np.abs(f_hi))
    # a vertex whose a / (a - b) rounded onto a node: the edge is unknown, |b - a| is at most the largest edge step
    step = max(np.abs(np.diff(f, axis=a)).max() for a in range(3))
    at_node = np.spacing(np.abs(v).max(axis=1)) * step + 8 * eps * np.abs(f_lo)
    bound = np.where(on_edge, bound, at_node)
    err = np.abs(s - iso)
    assert (err <= bound).all(), float((err / bound).max())


# ---- 6. grid_sample -----------------------------------------------------------------------------------------------------------
def test_vs_grid_sample(fi):
    """torch's trilinear grid_sample (align_corners=True) on interior points agrees within 1e-6 of the field's
    magnitude; grid_sample's normalised coordinates round the position, which is all that separates the two."""
    import torch
    shape = (40, 48, 56)
    x, y, z = _grid(shape)
    f = (np.sqrt(x * x + y * y + z * z) - 15.0).astype(F)
    rng = np.random.default_rng(6)
    pts = rng.uniform(0, np.array(shape[::-1]) - 1, (200_000, 3))
    norm = (2 * pts / (np.array(shape[::-1]) - 1) - 1).astype(F)
    df = torch.from_numpy(f).cuda()
    gs = torch.nn.functional.grid_sample(df.view(1, 1, *shape), torch.from_numpy(norm).cuda().view(1, 1, 1, -1, 3),
                                         mode="bilinear", padding_mode="border", align_corners=True).view(-1)
    v = fi.sample_field(df, torch.from_numpy(pts.astype(F)).cuda())
    assert v.is_cuda
    assert float((v - gs).abs().max()) <= 1e-6 * float(df.abs().max())


# ---- 7. a solved cloud sampled at its own points ---------------------------------------------------------------------------
def test_solved_cloud_at_its_points(fi):
    """The use case: a C4-style cloud (sphere and torus, position noise 0.005 = 0.6 cells at 128^3) solved on the
    device, then sampled at its own points with the cell-edge gradient.  The solve fits both shapes, including the
    parts of each inside the other, where the field has to compromise.  Measured on a B200 (200k points, seed 4):
    median |f| 0.274 cells, p95 0.801, p99 1.04; grad . n > 0 for 99.06 % of the points, median grad . n 0.694.  The
    bounds (median < 0.5, p95 < 1.5, share > 95 %, median grad . n > 0.5) leave about 2x on |f| and 4 points of
    share: a regression that moves the zero set by half a cell or flips the gradient's sign at more than 5 % of the
    points fails, while the cloud's own noise (0.64 cells) does not."""
    import torch
    from field_interpolation_b200 import workloads as W
    n = 128
    sizes = [n, n, n]
    cloud = W.sphere_torus_3d(200_000, seed=4)
    pos = W.to_lattice(cloud["unit_pos"], sizes)
    field = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
    out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
    _, st = field.solve(fi.solve_options(fi.FI_F32, 200, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID), out=out)
    assert st["converged"]
    v, g = fi.sample_field(out.view(n, n, n), torch.from_numpy(np.ascontiguousarray(pos, F)).cuda(), fi.GradientKernel.kCellEdges)
    v, g = v.cpu().numpy(), g.cpu().numpy()
    assert np.isfinite(v).all() and np.isfinite(g).all()
    a = np.abs(v)
    dot = np.einsum("ij,ij->i", g, cloud["normals"])
    q = {"median|f|": float(np.median(a)), "p95|f|": float(np.quantile(a, 0.95)), "p99|f|": float(np.quantile(a, 0.99)),
         "share grad.n>0": float((dot > 0).mean()), "median grad.n": float(np.median(dot))}
    print("solved cloud:", q)
    assert q["median|f|"] < 0.5 and q["p95|f|"] < 1.5, q
    assert q["share grad.n>0"] > 0.95 and q["median grad.n"] > 0.5, q


# ---- 8. locations and edge cases ------------------------------------------------------------------------------------------------
def test_host_and_device_identical(fi):
    import torch
    from field_interpolation_b200 import _lib as L
    f = np.random.default_rng(8).standard_normal((9, 10, 11)).astype(F)
    pts = S.positions_of_every_kind([11, 10, 9], 2000, seed=8)
    for k in (None, 0, 1, 2):
        h = fi.sample_field(f, pts, k)
        d = fi.sample_field(torch.from_numpy(f).cuda(), torch.from_numpy(pts).cuda(), k)
        if k is None:
            assert isinstance(h, np.ndarray) and d.is_cuda
            _same_bits(d, h)
        else:
            assert isinstance(h[1], np.ndarray) and d[0].is_cuda and d[1].is_cuda
            _same_bits(d[0], h[0])
            _same_bits(d[1], h[1])
    # values only / gradients only through the ABI, on the device
    df, dp = torch.from_numpy(f).cuda(), torch.from_numpy(pts).cuda()
    dg = torch.full((len(pts), 3), 7.0, device="cuda")
    sizes = (C.c_int32 * 3)(11, 10, 9)
    assert L.lib().fi_sample_field(3, sizes, df.data_ptr(), len(pts), dp.data_ptr(), 2, L.FI_DEVICE, None, dg.data_ptr()) == L.FI_OK
    _same_bits(dg, S.sample([11, 10, 9], f, pts, 2)[1])


def test_non_contiguous_tensors_and_empty(fi):
    import torch
    f = torch.randn(12, 13, 14, device="cuda")
    p = torch.rand(3, 500, device="cuda") * 12
    v = fi.sample_field(f, p.t())  # a transposed view is made contiguous
    _same_bits(v, S.sample([14, 13, 12], f.cpu().numpy(), p.t().cpu().numpy()))
    v, g = fi.sample_field(f, torch.empty(0, 3, device="cuda"), 1)
    assert v.shape == (0,) and g.shape == (0, 3) and v.is_cuda
    assert fi.sample_field(f.cpu().numpy(), np.zeros((0, 3), F)).shape == (0,)


def test_non_finite_and_far_positions(fi):
    import torch
    f = torch.randn(6, 7, 8, device="cuda")
    bad = [np.nan, np.inf, -np.inf, 1e30, -1e30, 3e9, -3e9, 2147483520.0, -2147483648.0, 1e38]
    pts = np.full((len(bad) * 3, 3), 3.5, F)
    for i, b in enumerate(bad):
        for d in range(3):
            pts[3 * i + d, d] = b
    dp = torch.from_numpy(pts).cuda()
    for k in (0, 1, 2):
        v, g = fi.sample_field(f, dp, k)
        assert bool(torch.isnan(v).all()) and bool(torch.isnan(g).all())
    torch.cuda.synchronize()
    assert np.isfinite(_host(fi.sample_field(f, torch.full((4, 3), 2.5, device="cuda")))).all()


def test_errors(fi):
    import torch
    from field_interpolation_b200 import _lib as L
    dll = L.lib()
    f = np.random.default_rng(1).standard_normal((3, 4)).astype(F)
    pts = np.array([[1.5, 1.5]], F)
    v, g = np.zeros(1, F), np.zeros((1, 2), F)
    sizes = (C.c_int32 * 2)(4, 3)
    names = ["ndim", "sizes", "field", "n", "pos", "kernel", "loc", "values", "gradients"]
    ok = dict(zip(names, (2, sizes, f.ctypes.data, 1, pts.ctypes.data, 0, L.FI_HOST, v.ctypes.data, g.ctypes.data)))

    def call(**kw):
        a = dict(ok, **kw)
        return dll.fi_sample_field(*[a[k] for k in names])

    assert call() == L.FI_OK
    for bad in [dict(ndim=0), dict(ndim=4), dict(sizes=None), dict(field=None), dict(pos=None), dict(sizes=(C.c_int32 * 2)(0, 3)),
                dict(loc=7), dict(n=-1), dict(kernel=3), dict(kernel=-1)]:
        assert call(**bad) == L.FI_ERR_INVALID, bad
        assert dll.fi_last_error()
    assert call(kernel=3, gradients=None) == L.FI_OK
    assert call(n=0, sizes=None, field=None, pos=None) == L.FI_OK
    with pytest.raises(ValueError):
        fi.sample_field(torch.from_numpy(f).cuda(), pts)
    with pytest.raises(ValueError):
        fi.sample_field(f, torch.from_numpy(pts).cuda())
    with pytest.raises(ValueError):
        fi.sample_field(f, np.zeros((1, 3), F))
    with pytest.raises(fi.FiError):
        fi.sample_field(f, pts, 5)


# ---- 9. the C++ drop-in ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", [-1, 0, 2])
def test_cpp_sample_driver(fi, tmp_path, kernel):
    from field_interpolation_b200 import build as B
    B.build()
    exe = B.build_cpp_driver(os.path.join(ROOT, "tests", "cpp", "sample_driver.cpp"), os.path.join(ROOT, "tests", "cpp", "sample_driver"))
    shape = (7, 9, 11)
    f = np.random.default_rng(9).standard_normal(shape).astype(F)
    pts = S.positions_of_every_kind(shape[::-1], 500, seed=9)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as h:
        h.write(struct.pack("<iiiiiq", 3, 11, 9, 7, kernel, len(pts)))
        h.write(f.tobytes())
        h.write(pts.tobytes())
    r = subprocess.run([exe, str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    raw = np.fromfile(outp, F)
    if kernel < 0:
        _same_bits(raw, fi.sample_field(f, pts))
    else:
        v, g = fi.sample_field(f, pts, kernel)
        _same_bits(raw[:len(pts)], v)
        _same_bits(raw[len(pts):].reshape(-1, 3), g)
