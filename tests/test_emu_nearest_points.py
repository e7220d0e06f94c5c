"""CPU: the kernels of csrc/nearest_points.cuh on the functional emulator of tests/emu/, bit for bit against the numpy
port of the reference caller's brute-force loop (tests/nearest_port.py): distances and indices in 1D, 2D and 3D, one
point and clouds of many leaves, duplicates and clouds with a single Morton key, exact ties, points on box faces, the
underflow case the absolute slack exists for, non-finite points and queries, far-away points; the border rows on axes
of 1, 2, 3 and 5 nodes, every kind of weight, interleaved with model, point and caller rows and clones against the
oracle port's system; the error codes; the C++ drop-in.  Not parity evidence for the CUDA build
(test_gpu_zz_nearest_points.py is); they catch ordering, indexing and pruning errors."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import nearest_port as P
from conftest import ROOT, bits
from oracle import oracle as O

F = np.float32


def _check(emu, points, queries):
    points, queries = np.asarray(points, F), np.asarray(queries, F)
    d, k = emu.nearest_point_distance(points, queries, want_index=True)
    wd, wk = P.nearest(points, queries)
    assert d.dtype == F and k.dtype == np.int64
    assert np.array_equal(bits(d), bits(wd))
    assert np.array_equal(k, wk)
    return d, k


@pytest.mark.parametrize("D", [1, 2, 3])
@pytest.mark.parametrize("n", [1, 7, 33, 900])
def test_random_clouds_vs_port(emu, D, n):
    """900 points: 29 leaves and three levels of boxes above them."""
    rng = np.random.default_rng(10 * D + n)
    pts = rng.uniform(-2, 12, (n, D)).astype(F)
    qs = np.concatenate([rng.uniform(-5, 15, (150, D)), pts[:20] + rng.normal(0, 0.01, (min(n, 20), D))]).astype(F)
    _check(emu, pts, qs)


@pytest.mark.parametrize("D", [1, 2, 3])
def test_duplicates_and_a_single_morton_key(emu, D):
    rng = np.random.default_rng(D)
    base = rng.uniform(0, 8, (40, D)).astype(F)
    dup = base[rng.integers(0, 40, 600)]  # every point many times, in scrambled order
    qs = np.concatenate([rng.uniform(-1, 9, (100, D)), base[:10]]).astype(F)
    _check(emu, dup, qs)
    same = np.full((300, D), 3.25, F)  # one point, 300 times: the box has no extent
    _check(emu, same, qs)
    ulp = (np.float32(3.25) + (rng.integers(0, 3, (300, D)) * np.spacing(F(3.25)))).astype(F)  # a few ulps apart
    _check(emu, ulp, np.concatenate([qs, ulp[:5]]).astype(F))


@pytest.mark.parametrize("D", [2, 3])
def test_exact_ties_at_different_indices(emu, D):
    """Points placed symmetrically around lattice queries, lattice-aligned so that many of them sit exactly on the
    faces of leaf boxes: every query has ties, and nearest must be the lowest tied index."""
    rng = np.random.default_rng(7 + D)
    offs = np.array([o for o in np.ndindex(*([3] * D))], F) - 1  # the 3^D neighbourhood
    centres = rng.integers(0, 10, (30, D)).astype(F)
    pts = (centres[:, None, :] + offs[None, :, :]).reshape(-1, D)
    pts = pts[rng.permutation(len(pts))]
    qs = np.concatenate([centres, centres + F(0.5), rng.integers(-1, 11, (60, D)).astype(F)]).astype(F)
    d, k = _check(emu, pts, qs)
    assert (d[:30] == 0).all()


def test_absolute_slack_underflow(emu):
    """A point 1e-25 from border node (0, 0), at index 0, and a point exactly on it at a higher index: both have fp32
    d2 == 0 (1e-50 underflows), so nearest is 0.  The other points of the cloud also lie within 1e-24 of the node, so
    every d2 there is 0 and the search finds a 0 in another leaf before it reaches index 0's; a bound without the
    absolute slack would then skip that leaf (its real squared distance is > 0)."""
    rng = np.random.default_rng(3)
    pts = rng.uniform(-1e-24, 1e-24, (2000, 2)).astype(F)
    pts[0] = (1e-25, 0.0)
    pts[1500] = (0.0, 0.0)
    q = np.array([[0.0, 0.0], [1e-25, 0.0], [1.0, 0.0]], F)
    d, k = _check(emu, pts, q)
    assert d[0] == 0 and k[0] == 0
    f = emu.LatticeField([3, 3])
    assert emu.add_border_distance_constraints(f, 1.0, pts) == 8
    assert f.eq.rhs[0] == 0 and np.array_equal(bits(f.eq.rhs), bits(P.border_rows([3, 3], 1.0, pts)[2]))


@pytest.mark.parametrize("D", [1, 2, 3])
def test_non_finite_and_far_points(emu, D):
    rng = np.random.default_rng(20 + D)
    pts = rng.uniform(0, 6, (200, D)).astype(F)
    pts[rng.integers(0, 200, 30), rng.integers(0, D, 30)] = np.nan
    pts[rng.integers(0, 200, 10), rng.integers(0, D, 10)] = np.inf
    pts[rng.integers(0, 200, 10), rng.integers(0, D, 10)] = -np.inf
    pts[:5] = F(1e19)  # d2 ~ 1e38: finite
    pts[5:10] = F(-3e38)  # d2 overflows to +inf
    qs = rng.uniform(-2, 8, (80, D)).astype(F)
    qs[0, 0], qs[1, -1], qs[2, 0] = np.nan, np.inf, -np.inf
    qs[3] = F(1e19)
    d, k = _check(emu, pts, qs)
    assert np.isinf(d[:3]).all() and (k[:3] == -1).all()
    _check(emu, np.full((50, D), np.nan, F), qs)  # no finite point: +inf, -1
    far = np.full((40, D), F(3e38), F)  # every d2 overflows
    d, k = _check(emu, far, qs[4:])
    assert np.isinf(d).all() and (k == -1).all()
    d, k = emu.nearest_point_distance(np.zeros((0, D), F), qs, want_index=True)  # no point at all
    assert np.isinf(d).all() and (k == -1).all()


@pytest.mark.parametrize("sizes", [[1], [2], [5], [1, 3], [2, 5], [3, 3], [5, 3], [7, 6], [1, 1, 2], [2, 3, 5], [3, 2, 2],
                                   [5, 1, 3], [5, 5, 5], [6, 5, 4]], ids=lambda s: "x".join(map(str, s)))
def test_border_rows_vs_port(emu, sizes):
    D = len(sizes)
    rng = np.random.default_rng(sum(sizes))
    pts = np.concatenate([rng.uniform(-1, np.array(sizes), (150, D)), rng.integers(0, sizes, (20, D))]).astype(F)
    f = emu.LatticeField(sizes)
    nodes, _ = P.border_nodes(sizes)
    assert emu.add_border_distance_constraints(f, 0.5, pts) == nodes.size
    cols, vals, rhs = P.border_rows(sizes, 0.5, pts)
    eq = f.eq
    assert np.array_equal(eq.rows, np.arange(nodes.size)) and np.array_equal(eq.cols, cols)
    assert np.array_equal(bits(eq.vals), bits(vals)) and np.array_equal(bits(eq.rhs), bits(rhs))
    d, _ = P.nearest(pts, np.stack(np.unravel_index(nodes, sizes[::-1])[::-1], axis=1).astype(F))
    assert np.array_equal(bits(rhs), bits((d * F(0.5)).astype(F)))


def test_weights_zero_negative_nan(emu):
    rng = np.random.default_rng(4)
    pts = rng.uniform(0, 5, (60, 2)).astype(F)
    for w in (0.0, -0.0):
        f = emu.LatticeField([5, 4])
        assert emu.add_border_distance_constraints(f, w, pts) == 0 and f.counts() == (0, 0)
    for w in (-1.5, np.nan, 1e-30, 3.0):
        f = emu.LatticeField([5, 4])
        assert emu.add_border_distance_constraints(f, w, pts) == 14
        cols, vals, rhs = P.border_rows([5, 4], w, pts)
        assert np.array_equal(bits(f.eq.vals), bits(vals)) and np.array_equal(bits(f.eq.rhs), bits(rhs))


def test_all_nan_cloud_gives_infinite_rhs(emu):
    f = emu.LatticeField([4, 3])
    assert emu.add_border_distance_constraints(f, 2.0, np.full((5, 2), np.nan, F)) == 10
    assert np.isposinf(f.eq.rhs).all()


def _port_border(pf, sizes, w, pts):
    cols, vals, rhs = P.border_rows(sizes, w, pts)
    _, _, dist = P.border_rows(sizes, 1.0, pts)
    for c, d in zip(cols, dist):
        pf.add_equation(w, float(d), [int(c)], [1.0])
    return len(cols)


@pytest.mark.parametrize("sizes", [[9], [7, 6], [4, 3, 5]], ids=lambda s: "x".join(map(str, s)))
def test_interleaved_with_other_rows_and_clones(emu, port, sizes):
    """model, points, border, a caller row, border (another cloud and weight), points; then a clone that grows on its
    own.  Every system equals the oracle port's built with the caller's loop, bit for bit."""
    from conftest import assert_system_bit_exact
    import error_map_cases as E
    D = len(sizes)
    rng = np.random.default_rng(len(sizes))
    p1, n1 = rng.uniform(-1, np.array(sizes), (25, D)).astype(F), rng.normal(size=(25, D)).astype(F)
    p2 = rng.uniform(0, np.array(sizes) - 1, (40, D)).astype(F)
    p3 = rng.uniform(-3, np.array(sizes) + 2, (30, D)).astype(F)
    wm = dict(model_1=0.7, model_2=0.5, gradient_smoothness=0.4)
    f, pf = emu.LatticeField(sizes), port.field(sizes)
    emu.add_field_constraints(f, emu.Weights(**wm))
    pf.add_field_constraints(O.make_weights(**wm))
    emu.add_points(f, 1.0, 1, 0.8, 2, p1, n1)
    pf.add_points(1.0, 1, 0.8, 2, p1, n1)
    emu.add_border_distance_constraints(f, 0.5, p2)
    _port_border(pf, sizes, 0.5, p2)
    emu.add_rows(f, np.zeros(2, np.int32), np.array([1, 3], np.int32), np.array([0.5, -2.0], F), np.array([0.25], F))
    pf.add_equation(1.0, 0.25, [1, 3], [0.5, -2.0])
    emu.add_border_distance_constraints(f, -1.25, p3)
    _port_border(pf, sizes, -1.25, p3)
    emu.add_points(f, 0.7, 0, 1.3, 1, p1[:10], n1[:10])
    pf.add_points(0.7, 0, 1.3, 1, p1[:10], n1[:10])
    want = pf.system()
    assert_system_bit_exact(f.eq, want.rows, want.cols, want.vals, want.rhs)
    g = E.clone(emu, f)
    assert_system_bit_exact(g.eq, want.rows, want.cols, want.vals, want.rhs)
    emu.add_border_distance_constraints(g, 2.0, p1)
    _port_border(pf, sizes, 2.0, p1)
    want2 = pf.system()
    assert_system_bit_exact(g.eq, want2.rows, want2.cols, want2.vals, want2.rhs)
    assert_system_bit_exact(f.eq, want.rows, want.cols, want.vals, want.rhs)  # the source did not change
    r0 = want.num_rows
    tr = np.empty(want2.num_triplets - want.num_triplets, dtype=[("row", np.int32), ("col", np.int32), ("value", F)])
    rhs = np.empty(want2.num_rows - r0, F)
    from field_interpolation_b200 import _lib as L
    L.check(L.lib().fi_field_export_rows(g._h, r0, C.c_void_p(tr.ctypes.data), C.c_void_p(rhs.ctypes.data)))
    assert np.array_equal(tr["row"], want2.rows[want.num_triplets:]) and np.array_equal(bits(rhs), bits(want2.rhs[r0:]))


def test_device_location(emu):
    """loc = FI_DEVICE through the ABI (emulated device memory is host memory) equals the host path."""
    from field_interpolation_b200 import _lib as L
    dll = L.lib()
    rng = np.random.default_rng(5)
    pts, qs = rng.uniform(0, 6, (100, 3)).astype(F), rng.uniform(-1, 7, (50, 3)).astype(F)
    want_d, want_k = P.nearest(pts, qs)
    for loc in (L.FI_HOST, L.FI_DEVICE):
        d, k = np.empty(50, F), np.empty(50, np.int64)
        assert dll.fi_nearest_point_distance(3, 100, pts.ctypes.data, 50, qs.ctypes.data, loc, d.ctypes.data, k.ctypes.data) == L.FI_OK
        assert np.array_equal(bits(d), bits(want_d)) and np.array_equal(k, want_k)
        d2 = np.empty(50, F)
        assert dll.fi_nearest_point_distance(3, 100, pts.ctypes.data, 50, qs.ctypes.data, loc, d2.ctypes.data, None) == L.FI_OK
        k2 = np.empty(50, np.int64)
        assert dll.fi_nearest_point_distance(3, 100, pts.ctypes.data, 50, qs.ctypes.data, loc, None, k2.ctypes.data) == L.FI_OK
        assert np.array_equal(bits(d2), bits(want_d)) and np.array_equal(k2, want_k)
        f = emu.LatticeField([4, 5, 3])
        n = C.c_int64(-1)
        assert dll.fi_field_add_border_distance(f._h, 0.5, 100, pts.ctypes.data, loc, C.byref(n)) == L.FI_OK
        cols, vals, rhs = P.border_rows([4, 5, 3], 0.5, pts)
        assert n.value == cols.size and np.array_equal(bits(f.eq.rhs), bits(rhs))


def test_error_codes(emu):
    from field_interpolation_b200 import _lib as L
    dll = L.lib()
    pts, qs, d, k = np.zeros((4, 2), F), np.zeros((3, 2), F), np.zeros(3, F), np.zeros(3, np.int64)
    call = dll.fi_nearest_point_distance
    assert call(2, 4, pts.ctypes.data, 3, qs.ctypes.data, L.FI_HOST, d.ctypes.data, k.ctypes.data) == L.FI_OK
    assert call(0, 4, pts.ctypes.data, 3, qs.ctypes.data, L.FI_HOST, d.ctypes.data, None) == L.FI_ERR_INVALID
    assert call(4, 4, pts.ctypes.data, 3, qs.ctypes.data, L.FI_HOST, d.ctypes.data, None) == L.FI_ERR_INVALID
    assert call(2, -1, pts.ctypes.data, 3, qs.ctypes.data, L.FI_HOST, d.ctypes.data, None) == L.FI_ERR_INVALID
    assert call(2, 4, pts.ctypes.data, -3, qs.ctypes.data, L.FI_HOST, d.ctypes.data, None) == L.FI_ERR_INVALID
    assert call(2, 4, None, 3, qs.ctypes.data, L.FI_HOST, d.ctypes.data, None) == L.FI_ERR_INVALID
    assert call(2, 4, pts.ctypes.data, 3, None, L.FI_HOST, d.ctypes.data, None) == L.FI_ERR_INVALID
    assert call(2, 4, pts.ctypes.data, 3, qs.ctypes.data, 2, d.ctypes.data, None) == L.FI_ERR_INVALID
    assert call(2, 1 << 32, pts.ctypes.data, 3, qs.ctypes.data, L.FI_HOST, d.ctypes.data, None) == L.FI_ERR_RANGE
    d[:] = 7
    assert call(2, 4, pts.ctypes.data, 3, qs.ctypes.data, L.FI_HOST, None, None) == L.FI_OK  # nothing to write
    assert call(2, 4, pts.ctypes.data, 0, None, L.FI_HOST, d.ctypes.data, None) == L.FI_OK and (d == 7).all()
    f = emu.LatticeField([4, 4])
    add = dll.fi_field_add_border_distance
    assert add(None, 1.0, 4, pts.ctypes.data, L.FI_HOST, None) == L.FI_ERR_INVALID
    assert add(f._h, 1.0, 0, pts.ctypes.data, L.FI_HOST, None) == L.FI_ERR_INVALID
    assert add(f._h, 1.0, -2, pts.ctypes.data, L.FI_HOST, None) == L.FI_ERR_INVALID
    assert add(f._h, 1.0, 4, None, L.FI_HOST, None) == L.FI_ERR_INVALID
    assert add(f._h, 1.0, 4, pts.ctypes.data, 5, None) == L.FI_ERR_INVALID
    assert add(f._h, 1.0, 1 << 32, pts.ctypes.data, L.FI_HOST, None) == L.FI_ERR_RANGE
    assert f.counts() == (0, 0)  # refused calls append nothing
    big = emu.LatticeField([2048, 1024, 1025])  # columns do not fit int32 (checked before anything is read)
    assert add(big._h, 1.0, 4, pts.ctypes.data, L.FI_HOST, None) == L.FI_ERR_RANGE
    with pytest.raises(ValueError):
        emu.nearest_point_distance(np.zeros((4, 2), F), np.zeros((3, 3), F))
    for bad in (np.zeros((4, 3), F), np.zeros(8, F), np.zeros((4, 1), F)):  # not (n, D) for this 2D field
        with pytest.raises(ValueError):
            emu.add_border_distance_constraints(f, 1.0, bad)
    assert f.counts() == (0, 0)


def test_cpp_drop_in_on_the_emulator(tmp_path):
    """tests/cpp/border_driver.cpp (b200::add_border_distance_constraints against the demo's hand loop in the same
    process) with libfi_b200.so resolved to the emulator build."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    os.symlink(build_emu.build(), tmp_path / "libfi_b200.so")
    env = dict(os.environ, FI_B200_TEST_EMU="1", LD_LIBRARY_PATH=str(tmp_path) + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_zz_nearest_points.py"), "-m", "gpu", "-q", "-x",
                        "-k", "cpp_border_driver", "-p", "no:cacheprovider"], env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    assert " passed" in r.stdout and " failed" not in r.stdout
