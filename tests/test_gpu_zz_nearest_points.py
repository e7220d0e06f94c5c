"""GPU: fi_nearest_point_distance and fi_field_add_border_distance on a B200, bit for bit against the reference caller's
brute-force loop: the numpy port (tests/nearest_port.py) on small cases, its chunked torch restatement on large ones.
The demo's 2D field; every border node of 128^3 with 100k points; 512^3 with the bench cloud; 1M uniform queries and
the marching-cubes vertices of a solved 256^3 C4 field against a 1M-point cloud; the error map and an MG-PCG solve of a
256^3 field with border rows; host and device inputs; errors; the C++ drop-in."""
import os
import struct
import subprocess

import numpy as np
import pytest

import nearest_port as P
from conftest import ROOT, assert_system_bit_exact, bits
from oracle import oracle as O

pytestmark = pytest.mark.gpu
F = np.float32


@pytest.fixture(scope="module")
def fi():
    import field_interpolation_b200 as m
    return m


def _border_coords(sizes, b):
    """Lattice coordinates (float32, x y z) of linear node indices b."""
    return np.stack(np.unravel_index(b, sizes[::-1])[::-1], axis=1).astype(F)


# ---- 1. the demo's 2D field --------------------------------------------------------------------------------------------
def test_demo_2d_field_matches_oracle(fi, port):
    """The field of tests/test_cpp_api.py::test_sdf_2d_caller_with_border_rows_and_coarse_to_fine (same cloud and sizes,
    full and coarse level), built with the new call, exports bit-identical to that test's oracle_field."""
    from field_interpolation_b200 import workloads as W
    width, height, bw, factor, npts = 44, 37, 0.5, 2, 600
    cloud = W.circles_2d(npts, seed=5)
    for w, h in ((width, height), ((width + factor - 1) // factor, (height + factor - 1) // factor)):
        pos = (cloud["unit_pos"] * np.array([np.float32(w) - np.float32(1), np.float32(h) - np.float32(1)], np.float32)[None, :]).astype(np.float32)
        pf = port.sdf_from_points([w, h], O.make_weights(), pos, cloud["normals"])
        for y in range(h):
            for x in range(w):
                if x in (0, w - 1) or y in (0, h - 1):
                    dx, dy = pos[:, 0] - np.float32(x), pos[:, 1] - np.float32(y)
                    d2 = (dx * dx + dy * dy).astype(np.float32).min()
                    pf.add_equation(bw, float(np.sqrt(np.float32(d2))), [y * w + x], [1.0])
        want = pf.system()
        f = fi.sdf_from_points([w, h], fi.Weights(), pos, cloud["normals"])
        assert fi.add_border_distance_constraints(f, bw, pos) == 2 * (w + h) - 4
        assert_system_bit_exact(f.eq, want.rows, want.cols, want.vals, want.rhs)


# ---- 2. every border node of 128^3 -----------------------------------------------------------------------------------------
def test_border_128_sphere_torus_all_nodes(fi):
    import torch
    from field_interpolation_b200 import workloads as W
    sizes = [128, 128, 128]
    pos = W.to_lattice(W.sphere_torus_3d(100_000, seed=1)["unit_pos"], sizes)
    f = fi.LatticeField(sizes)
    nodes, q = P.border_nodes(sizes)
    assert fi.add_border_distance_constraints(f, 1.0, pos) == nodes.size == 6 * 128 * 128 - 12 * 128 + 8
    eq = f.eq
    assert np.array_equal(eq.cols, nodes) and (eq.vals == 1.0).all()
    dp, dq = torch.from_numpy(pos).cuda(), torch.from_numpy(q).cuda()
    wd, wk = P.torch_nearest(dp, dq)
    assert np.array_equal(bits(eq.rhs), bits(wd.cpu().numpy()))
    d, k = fi.nearest_point_distance(dp, dq, want_index=True)
    assert np.array_equal(bits(d.cpu().numpy()), bits(eq.rhs)) and torch.equal(k, wk)


# ---- 3. 512^3 with the bench cloud -----------------------------------------------------------------------------------------
def test_border_512_bench_cloud(fi):
    import torch
    from field_interpolation_b200 import workloads as W
    n = 512
    sizes = [n, n, n]
    pos = W.to_lattice(W.sphere_torus_3d(1_000_000, seed=0)["unit_pos"], sizes)
    f = fi.LatticeField(sizes)
    nb = 6 * n * n - 12 * n + 8
    assert fi.add_border_distance_constraints(f, 1.0, torch.from_numpy(pos).cuda()) == nb
    assert f.counts() == (nb, nb)
    eq = f.eq
    rng = np.random.default_rng(0)
    pick = rng.choice(nb, 65536, replace=False).astype(np.int64)
    corners = np.array([x + n * (y + n * z) for z in (0, n - 1) for y in (0, n - 1) for x in (0, n - 1)], np.int64)
    pos_of = {int(c): i for i, c in enumerate(eq.cols)}
    pick = np.concatenate([pick, [pos_of[int(c)] for c in corners]]).astype(np.int64)
    q = _border_coords(sizes, eq.cols[pick].astype(np.int64))
    wd, _ = P.torch_nearest(torch.from_numpy(pos).cuda(), torch.from_numpy(q).cuda())
    assert np.array_equal(bits(eq.rhs[pick]), bits(wd.cpu().numpy()))
    assert np.isfinite(eq.rhs).all() and (eq.rhs > 0).all()


# ---- 4. arbitrary queries against 1M points ---------------------------------------------------------------------------------
def test_arbitrary_queries_uniform_and_mesh_vertices(fi):
    import torch
    from field_interpolation_b200 import workloads as W
    n = 256
    sizes = [n, n, n]
    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    pos = W.to_lattice(cloud["unit_pos"], sizes)
    dp = torch.from_numpy(pos).cuda()
    g = torch.Generator(device="cuda").manual_seed(0)
    uni = torch.rand((1_000_000, 3), generator=g, device="cuda") * (n - 1)
    f = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
    out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
    _, st = f.solve(fi.solve_options(fi.FI_F32, 200, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID), out=out)
    assert st["converged"]
    verts, _ = fi.marching_cubes(out.view(n, n, n), 0.0)
    assert verts.shape[0] > 100_000
    for qs in (uni, verts.contiguous()):
        d, k = fi.nearest_point_distance(dp, qs, want_index=True)
        assert d.shape == (qs.shape[0],) and k.dtype == torch.int64
        pick = torch.randperm(qs.shape[0], generator=torch.Generator().manual_seed(1))[:65536].cuda()
        wd, wk = P.torch_nearest(dp, qs[pick])
        assert np.array_equal(bits(d[pick].cpu().numpy()), bits(wd.cpu().numpy()))
        assert torch.equal(k[pick], wk)
    dv = fi.nearest_point_distance(dp, verts.contiguous())
    print(f"mesh -> cloud distance at 256^3: median {float(dv.median()):.3f}, max {float(dv.max()):.3f} cells")


# ---- 5. error map and MG-PCG solve of a 256^3 field with border rows --------------------------------------------------------
def test_error_map_and_solve_with_border_rows_256(fi):
    """Model, point and border rows (weight 0.5).  The heat map equals that of the same field whose border rows were
    computed by the torch brute force and appended as caller rows (whose error map the error-map tests tie to the
    port bit for bit).  MG-PCG does not reach 1e-6 on this field: the coarse levels do not see caller rows, and on one
    B200 it stalled at a true residual of 0.047 after 300 iterations (DESIGN.md §3g, §8).  The solve must report that
    honestly: `converged` is decided by the true residual."""
    import torch
    from field_interpolation_b200 import workloads as W
    n = 256
    sizes = [n, n, n]
    cloud = W.sphere_torus_3d(100_000, seed=2)
    pos = W.to_lattice(cloud["unit_pos"], sizes)
    f = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
    nb = fi.add_border_distance_constraints(f, 0.5, pos)
    g = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
    nodes, q = P.border_nodes(sizes)
    wd, _ = P.torch_nearest(torch.from_numpy(pos).cuda(), torch.from_numpy(q).cuda())
    rhs = (wd.cpu().numpy() * F(0.5)).astype(F)
    fi.add_rows(g, np.arange(nb, dtype=np.int32), nodes.astype(np.int32), np.full(nb, F(1.0) * F(0.5), F), rhs)
    assert f.counts() == g.counts()
    x = torch.from_numpy(np.random.default_rng(3).normal(size=n ** 3).astype(F)).cuda()
    a, sa = fi.generate_error_map(f, x, want_sums=True)
    b, sb = fi.generate_error_map(g, x, want_sums=True)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)) and np.array_equal(sa, sb) and sa[2] > 0
    out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
    _, st = f.solve(fi.solve_options(fi.FI_F32, 300, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID), out=out)
    print(f"256^3 with border rows: {st}")
    assert bool(st["converged"]) == (st["true_residual"] <= 1e-6)
    assert st["true_residual"] < 0.1 and bool(torch.isfinite(out).all())


# ---- 6. host and device inputs, errors ------------------------------------------------------------------------------------
def test_host_and_device_identical_and_errors(fi):
    import torch
    from field_interpolation_b200 import _lib as L
    rng = np.random.default_rng(6)
    pts = rng.uniform(0, 40, (50_000, 3)).astype(F)
    pts[::97, 1] = np.nan
    qs = rng.uniform(-5, 45, (20_000, 3)).astype(F)
    hd, hk = fi.nearest_point_distance(pts, qs, want_index=True)
    dd, dk = fi.nearest_point_distance(torch.from_numpy(pts).cuda(), torch.from_numpy(qs).cuda(), want_index=True)
    assert isinstance(hd, np.ndarray) and dd.is_cuda
    assert np.array_equal(bits(hd), bits(dd.cpu().numpy())) and np.array_equal(hk, dk.cpu().numpy())
    wd, wk = P.nearest(pts, qs[:300])
    assert np.array_equal(bits(hd[:300]), bits(wd)) and np.array_equal(hk[:300], wk)
    f1, f2 = fi.LatticeField([40, 30, 20]), fi.LatticeField([40, 30, 20])
    assert fi.add_border_distance_constraints(f1, 0.5, pts) == fi.add_border_distance_constraints(f2, 0.5, torch.from_numpy(pts).cuda())
    e1, e2 = f1.eq, f2.eq
    assert np.array_equal(bits(e1.rhs), bits(e2.rhs)) and np.array_equal(e1.cols, e2.cols)
    dll = L.lib()
    dp = torch.from_numpy(pts).cuda()
    d = torch.empty(4, dtype=torch.float32, device="cuda")
    assert dll.fi_nearest_point_distance(3, 10, dp.data_ptr(), 4, None, L.FI_DEVICE, d.data_ptr(), None) == L.FI_ERR_INVALID
    assert dll.fi_nearest_point_distance(5, 10, dp.data_ptr(), 4, dp.data_ptr(), L.FI_DEVICE, d.data_ptr(), None) == L.FI_ERR_INVALID
    assert dll.fi_field_add_border_distance(f1._h, 1.0, 0, dp.data_ptr(), L.FI_DEVICE, None) == L.FI_ERR_INVALID
    big = fi.LatticeField([2048, 1024, 1025])
    assert dll.fi_field_add_border_distance(big._h, 1.0, 10, dp.data_ptr(), L.FI_DEVICE, None) == L.FI_ERR_RANGE


# ---- 7. the C++ drop-in ------------------------------------------------------------------------------------------------------
def test_cpp_border_driver(fi, port, tmp_path):
    """tests/cpp/border_driver.cpp: b200::add_border_distance_constraints against the demo's hand loop in one process
    (also deferred), and its field against the oracle's."""
    from field_interpolation_b200 import build as B
    from field_interpolation_b200 import workloads as W
    B.build()
    exe = B.build_cpp_driver(os.path.join(ROOT, "tests", "cpp", "border_driver.cpp"), os.path.join(ROOT, "tests", "cpp", "border_driver"))
    w, h, bw = 44, 37, 0.5
    cloud = W.circles_2d(600, seed=5)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as fh:
        fh.write(struct.pack("<iifq", w, h, bw, 600))
        fh.write(np.ascontiguousarray(cloud["unit_pos"], F).tobytes())
        fh.write(np.ascontiguousarray(cloud["normals"], F).tobytes())
    r = subprocess.run([exe, str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    raw = open(outp, "rb").read()
    nr, nt = struct.unpack("<qq", raw[:16])
    tr = np.frombuffer(raw[16:16 + 12 * nt], dtype=[("row", np.int32), ("col", np.int32), ("value", F)])
    rhs = np.frombuffer(raw[16 + 12 * nt:], F)
    pos = (cloud["unit_pos"] * np.array([np.float32(w) - np.float32(1), np.float32(h) - np.float32(1)], np.float32)[None, :]).astype(np.float32)
    pf = port.sdf_from_points([w, h], O.make_weights(), pos, cloud["normals"])
    pf.add_equation(2.0, 0.5, [1, 3], [1.0, -0.5])
    cols, _, _ = P.border_rows([w, h], bw, pos)
    _, _, dist = P.border_rows([w, h], 1.0, pos)
    for c, d in zip(cols, dist):
        pf.add_equation(bw, float(d), [int(c)], [1.0])
    want = pf.system()
    assert nr == want.num_rows and np.array_equal(tr["row"], want.rows) and np.array_equal(tr["col"], want.cols)
    assert np.array_equal(bits(tr["value"]), bits(want.vals)) and np.array_equal(bits(rhs), bits(want.rhs))
