"""CPU: the kernels of csrc/marching_cubes.cuh (count -> scan -> emit -> triangles) on the functional emulator of
tests/emu/, bit for bit against the CPU port (tests/mc_port.cpp) on lattices the emulator finishes in seconds.  Not
parity evidence for the CUDA build (test_gpu_zz_marching_cubes.py is); they catch indexing and protocol errors."""
import numpy as np
import pytest

import mesh_checks as M
from conftest import bits
from mc_port import port as mc_port


def same_mesh(got, want):
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.shape == w.shape
        assert np.array_equal(bits(g) if g.dtype == np.float32 else g, bits(w) if w.dtype == np.float32 else w)


def test_all_256_configurations_of_one_cell(emu):
    for cfg in range(256):
        f = np.array([1.0 if (cfg >> c) & 1 else -1.0 for c in range(8)], np.float32).reshape(2, 2, 2)
        f *= np.linspace(0.5, 1.5, 8, dtype=np.float32).reshape(2, 2, 2)
        same_mesh(emu.marching_cubes(f, 0.0, want_normals=True), mc_port().marching_cubes(f, 0.0, want_normals=True))


@pytest.mark.parametrize("shape", [(1, 5, 5), (2, 2, 2), (3, 7, 2), (33, 20, 9), (5, 3, 130)])
@pytest.mark.parametrize("iso", [0.0, 0.3])
def test_random_fields_vs_port(emu, shape, iso):
    rng = np.random.default_rng(sum(shape))
    f = rng.standard_normal(shape).astype(np.float32)
    f[rng.random(shape) < 0.10] = 0.0
    f[rng.random(shape) < 0.05] = -0.0
    got = emu.marching_cubes(f, iso, want_normals=True)
    same_mesh(got, mc_port().marching_cubes(f, iso, want_normals=True))
    same_mesh(emu.marching_cubes(f, iso), got[:2])
    if min(shape) >= 2:
        assert len(got[0]) > 0 and np.array_equal(bits(got[0]), bits(M.contract_vertices(f, iso)))


def test_smooth_field_closed(emu):
    f = M.smooth_field((17, 19, 23), 7)
    v, t = emu.marching_cubes(f, 0.0)
    same_mesh((v, t), mc_port().marching_cubes(f, 0.0))
    M.assert_closed(t, len(v))


def test_capacity_and_count_only(emu):
    import ctypes as C
    from field_interpolation_b200 import _lib as L
    f = M.smooth_field((9, 10, 11), 2)
    v, t = mc_port().marching_cubes(f, 0.0)
    sizes = (C.c_int32 * 3)(11, 10, 9)
    nv, nt = C.c_int64(-1), C.c_int64(-1)
    a = np.ascontiguousarray(f)
    dll = L.lib()
    assert dll.fi_marching_cubes(sizes, a.ctypes.data, 0.0, L.FI_HOST, None, None, 0, None, 0, C.byref(nv), C.byref(nt)) == L.FI_OK
    assert (nv.value, nt.value) == (len(v), len(t))
    out = np.full((len(v), 3), 7.0, np.float32)
    tri = np.full((len(t), 3), 7, np.int32)
    st = dll.fi_marching_cubes(sizes, a.ctypes.data, 0.0, L.FI_HOST, out.ctypes.data, None, len(v), tri.ctypes.data, len(t) - 1,
                               C.byref(nv), C.byref(nt))
    assert st == L.FI_ERR_RANGE and (nv.value, nt.value) == (len(v), len(t))
    assert (out == 7.0).all() and (tri == 7).all()
