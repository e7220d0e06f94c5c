"""GPU: fi_marching_cubes (csrc/marching_cubes.cuh) — triangle meshes of solved 3D fields on the device.

Bar: vertices, normals and indices bit-identical to the sequential CPU port (tests/mc_port.cpp); meshes closed and
consistently wound; on every lattice face the mesh's border equals the reference-pinned 2D contour of
fi_marching_squares bit for bit; analytic volume, area, Euler characteristic and normals on a sphere and a torus."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import mesh_checks as M
from conftest import ROOT, bits
from mc_port import port as mc_port

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fi():
    import field_interpolation_b200 as m
    return m


def _host(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else a


def same_mesh(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        g = _host(g)
        assert g.shape == w.shape
        assert np.array_equal(bits(g) if g.dtype == np.float32 else g, bits(w) if w.dtype == np.float32 else w)


def _grid(n):
    c = (n - 1) / 2
    z, y, x = np.meshgrid(*[np.arange(n, dtype=np.float64)] * 3, indexing="ij")
    return x - c, y - c, z - c


def sphere_sdf(n, r):
    x, y, z = _grid(n)
    return (np.sqrt(x * x + y * y + z * z) - r).astype(np.float32)


def torus_sdf(n, R, r):
    x, y, z = _grid(n)
    q = np.sqrt(x * x + y * y) - R
    return (np.sqrt(q * q + z * z) - r).astype(np.float32)


def random_field(shape, seed):
    rng = np.random.default_rng(seed)
    f = rng.standard_normal(shape).astype(np.float32)
    f[rng.random(shape) < 0.10] = 0.0
    f[rng.random(shape) < 0.05] = -0.0
    return f


# ---- 1. parity with the port --------------------------------------------------------------------------------------
def test_all_256_configurations(fi):
    import torch
    for cfg in range(256):
        f = np.array([1.0 if (cfg >> c) & 1 else -1.0 for c in range(8)], np.float32).reshape(2, 2, 2)
        f *= np.linspace(0.5, 1.5, 8, dtype=np.float32).reshape(2, 2, 2)
        want = mc_port().marching_cubes(f, 0.0, want_normals=True)
        same_mesh(fi.marching_cubes(f, 0.0, want_normals=True), want)
        same_mesh(fi.marching_cubes(torch.from_numpy(f).cuda(), 0.0, want_normals=True), want)


@pytest.mark.parametrize("shape", [(5, 5, 1), (2, 2, 2), (2, 7, 3), (9, 20, 33), (257, 3, 130), (257, 257, 257)])
@pytest.mark.parametrize("iso", [0.0, 0.3])
def test_random_fields_vs_port(fi, shape, iso):
    """Shapes are (nz, ny, nx): 1x5x5 (empty), 2x2x2, 3x7x2, 33x20x9, 130x3x257 and 257^3, whose 1024-node tiles span
    rows and planes; host arrays and CUDA tensors."""
    import torch
    f = random_field(shape, sum(shape))
    want = mc_port().marching_cubes(f, iso, want_normals=True)
    if min(shape) < 2:
        assert len(want[0]) == 0 and len(want[1]) == 0
    same_mesh(fi.marching_cubes(f, iso, want_normals=True), want)
    got = fi.marching_cubes(torch.from_numpy(f).cuda(), iso, want_normals=True)
    assert all(a.is_cuda for a in got)
    same_mesh(got, want)
    same_mesh(fi.marching_cubes(f, iso), want[:2])


# ---- 2. closed and consistently oriented ------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(3))
def test_closed_on_padded_smooth_fields(fi, seed):
    f = M.smooth_field((40 + seed, 57, 66), seed)
    v, t = fi.marching_cubes(f, 0.0)
    assert len(t) > 100
    M.assert_closed(t, len(v))
    assert M.volume(v, t) > 0  # the inside is enclosed; winding toward the outside makes its volume positive


# ---- 3. the reference-pinned 2D contour on every lattice face -----------------------------------------------------------
@pytest.mark.parametrize("seed", range(3))
@pytest.mark.parametrize("iso", [0.0, 0.3])
def test_faces_equal_marching_squares(fi, seed, iso):
    """The unpaired half-edges on each lattice face equal fi_marching_squares of that plane bit for bit, in the same
    direction on the x = 0, y = ny-1 and z = 0 faces and reversed on the other three (M.FACE_DIRECTION); all other
    half-edges have twins."""
    f = random_field((11 + seed, 14, 17), 100 + seed)
    v, t = fi.marching_cubes(f, iso)
    total = 0
    for axis, n in ((0, f.shape[2]), (1, f.shape[1]), (2, f.shape[0])):
        for which, coord in (("min", 0), ("max", n - 1)):
            got = M.face_contour(v, t, f, iso, axis, coord)
            want = fi.iso_surface(M.face_plane(f, axis, coord), iso)
            assert len(want) > 0
            if M.FACE_DIRECTION[(axis, which)] == "reversed":
                want = M.reversed_segments(want)
            assert M.same_segments(got, want), (axis, which)
            total += len(got)
    # every unpaired half-edge was found on some face (one along a box edge is counted on both of its faces)
    assert M.unpaired_half_edges(t, len(v)).shape[0] <= total


# ---- 4. analytic shapes -------------------------------------------------------------------------------------------------
def test_sphere(fi):
    n, r = 128, 40.0
    v, t, nrm = fi.marching_cubes(sphere_sdf(n, r), 0.0, want_normals=True)
    M.assert_closed(t, len(v))
    assert M.euler_characteristic(t, len(v)) == 2
    assert abs(M.volume(v, t) / (4 / 3 * np.pi * r ** 3) - 1) < 1e-3
    assert abs(M.area(v, t) / (4 * np.pi * r * r) - 1) < 1e-2
    radial = v - (n - 1) / 2
    radial /= np.linalg.norm(radial, axis=1, keepdims=True)
    assert (np.einsum("ij,ij->i", radial, nrm) > 0.99).all()
    fn = M.face_normals(v, t)
    big = np.linalg.norm(fn, axis=1) > 1e-6
    vn = nrm[t].sum(axis=1)
    assert (np.einsum("ij,ij->i", fn[big], vn[big]) > 0).all()


def test_torus(fi):
    n, R, r = 128, 36.0, 16.0
    v, t, nrm = fi.marching_cubes(torus_sdf(n, R, r), 0.0, want_normals=True)
    M.assert_closed(t, len(v))
    assert M.euler_characteristic(t, len(v)) == 0
    assert abs(M.volume(v, t) / (2 * np.pi ** 2 * R * r * r) - 1) < 1e-3
    assert abs(M.area(v, t) / (4 * np.pi ** 2 * R * r) - 1) < 1e-2
    fn = M.face_normals(v, t)
    big = np.linalg.norm(fn, axis=1) > 1e-6
    assert (np.einsum("ij,ij->i", fn[big], nrm[t].sum(axis=1)[big]) > 0).all()


# ---- 5. end to end on the device ------------------------------------------------------------------------------------------
def test_solved_field_on_device(fi):
    """A C4-style cloud solved into a CUDA tensor and meshed there.  The cloud samples the whole sphere and the whole
    torus, including the parts inside each other, so the solved field also has zero crossings that belong to neither
    shape; the check is that the mesh is closed and passes within 1.5 cells of every point of the union's outer
    boundary (analytic points on either shape at least 2 cells outside the other)."""
    import torch
    from scipy.spatial import cKDTree
    from field_interpolation_b200 import workloads as W
    n = 128
    sizes = [n, n, n]
    cloud = W.sphere_torus_3d(200_000, seed=4)
    field = fi.sdf_from_points(sizes, fi.Weights(), W.to_lattice(cloud["unit_pos"], sizes), cloud["normals"])
    out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
    _, st = field.solve(fi.solve_options(fi.FI_F32, 200, 1e-6, preconditioner=fi.FI_PRECOND_MULTIGRID), out=out)
    assert st["converged"]
    v, t = fi.marching_cubes(out.view(n, n, n), 0.0)
    assert v.is_cuda and t.is_cuda and len(t) > 1000
    v, t = v.cpu().numpy().astype(np.float64), t.cpu().numpy()
    M.assert_closed(t, len(v))

    rng = np.random.default_rng(0)
    d = rng.normal(size=(20_000, 3))
    sphere = 0.5 + 0.3 * d / np.linalg.norm(d, axis=1, keepdims=True)
    u, w = rng.random(20_000) * 2 * np.pi, rng.random(20_000) * 2 * np.pi
    ring = np.stack([np.cos(u), np.sin(u), np.zeros_like(u)], axis=1)
    torus = 0.5 + 0.25 * ring + 0.10 * (ring * np.cos(w)[:, None] + np.array([0.0, 0.0, 1.0]) * np.sin(w)[:, None])

    def sd_sphere(p):
        return np.linalg.norm(p - 0.5, axis=1) - 0.3

    def sd_torus(p):
        c = p - 0.5
        return np.sqrt((np.sqrt(c[:, 0] ** 2 + c[:, 1] ** 2) - 0.25) ** 2 + c[:, 2] ** 2) - 0.10

    margin = 2.0 / (n - 1)
    outer = np.concatenate([sphere[sd_torus(sphere) > margin], torus[sd_sphere(torus) > margin]])
    assert len(outer) > 10_000
    dist, _ = cKDTree(v / (n - 1)).query(outer)
    assert (dist * (n - 1)).max() < 1.5


# ---- 6. full size -------------------------------------------------------------------------------------------------------
def _device_sphere(n, r):
    import torch
    a = torch.arange(n, device="cuda", dtype=torch.float32) - (n - 1) / 2
    z, y, x = a.view(n, 1, 1), a.view(1, n, 1), a.view(1, 1, n)
    return torch.sqrt(x * x + y * y + z * z) - r


def test_full_size_1024(fi):
    import torch
    n, r = 1024, 400.0
    f = _device_sphere(n, r).contiguous()
    v, t = fi.marching_cubes(f, 0.0)
    del f
    assert abs(len(v) / (1.5 * 4 * np.pi * r * r) - 1) < 0.01
    # closed: every directed edge has exactly one twin (sort keys on the device)
    e = torch.cat([t[:, [0, 1]], t[:, [1, 2]], t[:, [2, 0]]]).long()
    key = torch.sort(e[:, 0] * len(v) + e[:, 1]).values
    assert bool((key[1:] != key[:-1]).all())
    twin = e[:, 1] * len(v) + e[:, 0]
    pos = torch.searchsorted(key, twin)
    assert bool((key[pos.clamp(max=len(key) - 1)] == twin).all())
    assert int(torch.unique(t).numel()) == len(v)


def test_parity_512(fi):
    import torch
    n = 512
    f = sphere_sdf(n, 200.0) + 0.25 * torus_sdf(n, 120.0, 50.0)
    want = mc_port().marching_cubes(f, 0.0, want_normals=True)
    same_mesh(fi.marching_cubes(torch.from_numpy(f).cuda(), 0.0, want_normals=True), want)


# ---- 7. errors ----------------------------------------------------------------------------------------------------------
def test_capacity_count_only_and_invalid(fi):
    from field_interpolation_b200 import _lib as L
    f = M.smooth_field((21, 22, 23), 1)
    v, t = mc_port().marching_cubes(f, 0.0)
    sizes = (C.c_int32 * 3)(23, 22, 21)
    nv, nt = C.c_int64(-1), C.c_int64(-1)
    dll = L.lib()
    a = np.ascontiguousarray(f)
    assert dll.fi_marching_cubes(sizes, a.ctypes.data, 0.0, L.FI_HOST, None, None, 0, None, 0, C.byref(nv), C.byref(nt)) == L.FI_OK
    assert (nv.value, nt.value) == (len(v), len(t))
    for cap_v, cap_t in ((len(v) - 1, len(t)), (len(v), len(t) - 1)):
        out, nrm = np.full((len(v), 3), 7.0, np.float32), np.full((len(v), 3), 7.0, np.float32)
        tri = np.full((len(t), 3), 7, np.int32)
        nv.value = nt.value = -1
        st = dll.fi_marching_cubes(sizes, a.ctypes.data, 0.0, L.FI_HOST, out.ctypes.data, nrm.ctypes.data, cap_v, tri.ctypes.data, cap_t,
                                   C.byref(nv), C.byref(nt))
        assert st == L.FI_ERR_RANGE and (nv.value, nt.value) == (len(v), len(t))
        assert (out == 7.0).all() and (nrm == 7.0).all() and (tri == 7).all()
    # device outputs: only 4-byte alignment is required
    import torch
    d = torch.from_numpy(f).cuda()
    buf = torch.zeros(3 * len(v) + 1, dtype=torch.float32, device="cuda")
    tri = torch.zeros(3 * len(t) + 1, dtype=torch.int32, device="cuda")
    st = dll.fi_marching_cubes(sizes, C.c_void_p(d.data_ptr()), 0.0, L.FI_DEVICE, C.c_void_p(buf.data_ptr() + 4), None, len(v),
                               C.c_void_p(tri.data_ptr() + 4), len(t), C.byref(nv), C.byref(nt))
    assert st == L.FI_OK
    assert np.array_equal(bits(buf[1:].cpu().numpy().reshape(-1, 3)), bits(v)) and np.array_equal(tri[1:].cpu().numpy().reshape(-1, 3), t)
    # bad arguments
    good = dict(sizes=sizes, values=a.ctypes.data)
    assert dll.fi_marching_cubes(None, good["values"], 0.0, L.FI_HOST, None, None, 0, None, 0, C.byref(nv), C.byref(nt)) == L.FI_ERR_INVALID
    assert dll.fi_marching_cubes(sizes, None, 0.0, L.FI_HOST, None, None, 0, None, 0, C.byref(nv), C.byref(nt)) == L.FI_ERR_INVALID
    assert dll.fi_marching_cubes(sizes, good["values"], 0.0, L.FI_HOST, None, None, 0, None, 0, None, C.byref(nt)) == L.FI_ERR_INVALID
    assert dll.fi_marching_cubes((C.c_int32 * 3)(23, 0, 21), good["values"], 0.0, L.FI_HOST, None, None, 0, None, 0, C.byref(nv),
                                 C.byref(nt)) == L.FI_ERR_INVALID
    assert dll.fi_marching_cubes(sizes, good["values"], 0.0, L.FI_HOST, out.ctypes.data, None, -1, None, 0, C.byref(nv),
                                 C.byref(nt)) == L.FI_ERR_INVALID
    assert dll.fi_marching_cubes((C.c_int32 * 3)(2048, 1024, 1024), good["values"], 0.0, L.FI_DEVICE, None, None, 0, None, 0, C.byref(nv),
                                 C.byref(nt)) == L.FI_ERR_RANGE
    with pytest.raises(ValueError):
        fi.marching_cubes(np.zeros((4, 4), np.float32))


# ---- 8. the C++ drop-in ---------------------------------------------------------------------------------------------------
def test_cpp_mesh_driver(fi, tmp_path):
    from field_interpolation_b200 import build as B
    B.build()
    exe = B.build_cpp_driver(os.path.join(ROOT, "tests", "cpp", "mesh_driver.cpp"), os.path.join(ROOT, "tests", "cpp", "mesh_driver"))
    f = random_field((13, 17, 19), 9)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as h:
        h.write(struct.pack("<iiifi", 19, 17, 13, 0.3, 1))
        h.write(f.tobytes())
    r = subprocess.run([exe, str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    raw = open(outp, "rb").read()
    nv, nt = struct.unpack("<qq", raw[:16])
    body = np.frombuffer(raw[16:], np.uint8)
    pos = body[: 12 * nv].view(np.float32).reshape(-1, 3)
    nrm = body[12 * nv: 24 * nv].view(np.float32).reshape(-1, 3)
    tri = body[24 * nv:].view(np.int32).reshape(-1, 3)
    assert len(tri) == nt
    same_mesh((pos, tri, nrm), fi.marching_cubes(f, 0.3, want_normals=True))
