"""CPU: the kernels of csrc/sample_field.cuh on the functional emulator of tests/emu/, bit for bit against the numpy
port (tests/sample_port.py) on small lattices, through the host and the "device" path of fi_sample_field, plus its
error codes.  Not parity evidence for the CUDA build (test_gpu_zz_sample_field.py is); they catch indexing and
protocol errors."""
import ctypes as C

import numpy as np
import pytest

import sample_port as S
from conftest import bits

F = np.float32
SHAPES = [(9,), (1,), (5, 7), (1, 3), (4, 3, 6), (2, 2, 2), (3, 1, 5)]


def _field(shape, seed):
    return np.random.default_rng(seed).standard_normal(shape).astype(F)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("kernel", [None, 0, 1, 2])
def test_host_path_vs_port(emu, shape, kernel):
    f = _field(shape, sum(shape))
    sizes = shape[::-1]
    pts = S.positions_of_every_kind(sizes, 200, seed=len(shape))
    got = emu.sample_field(f, pts, kernel)
    want = S.sample(sizes, f, pts, kernel)
    if kernel is None:
        assert got.shape == (len(pts),) and np.array_equal(bits(got), bits(want))
    else:
        assert got[1].shape == (len(pts), len(shape))
        assert np.array_equal(bits(got[0]), bits(want[0])) and np.array_equal(bits(got[1]), bits(want[1]))


@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_device_path_and_gradients_only(emu, kernel):
    """loc = FI_DEVICE (emulated device memory is host memory), and values = null with gradients requested."""
    from field_interpolation_b200 import _lib as L
    shape = (4, 5, 6)
    f = _field(shape, 3)
    pts = S.positions_of_every_kind(shape[::-1], 100, seed=4)
    want_v, want_g = S.sample(shape[::-1], f, pts, kernel)
    sizes = (C.c_int32 * 3)(*shape[::-1])
    v = np.full(len(pts), 7, F)
    g = np.full((len(pts), 3), 7, F)
    dll = L.lib()
    assert dll.fi_sample_field(3, sizes, f.ctypes.data, len(pts), pts.ctypes.data, kernel, L.FI_DEVICE, v.ctypes.data, g.ctypes.data) == L.FI_OK
    assert np.array_equal(bits(v), bits(want_v)) and np.array_equal(bits(g), bits(want_g))
    g[:] = 7
    assert dll.fi_sample_field(3, sizes, f.ctypes.data, len(pts), pts.ctypes.data, kernel, L.FI_HOST, None, g.ctypes.data) == L.FI_OK
    assert np.array_equal(bits(g), bits(want_g))


def test_error_codes(emu):
    from field_interpolation_b200 import _lib as L
    dll = L.lib()
    f = _field((3, 4), 0)
    pts = np.array([[1.5, 1.5]], F)
    v, g = np.zeros(1, F), np.zeros((1, 2), F)
    sizes = (C.c_int32 * 2)(4, 3)
    ok = (2, sizes, f.ctypes.data, 1, pts.ctypes.data, 0, L.FI_HOST, v.ctypes.data, g.ctypes.data)

    def call(**kw):
        names = ["ndim", "sizes", "field", "n", "pos", "kernel", "loc", "values", "gradients"]
        a = dict(zip(names, ok))
        a.update(kw)
        return dll.fi_sample_field(*[a[k] for k in names])

    assert call() == L.FI_OK
    assert call(ndim=0) == L.FI_ERR_INVALID and call(ndim=4) == L.FI_ERR_INVALID
    assert call(sizes=None) == L.FI_ERR_INVALID and call(field=None) == L.FI_ERR_INVALID and call(pos=None) == L.FI_ERR_INVALID
    assert call(sizes=(C.c_int32 * 2)(4, 0)) == L.FI_ERR_INVALID
    assert call(loc=2) == L.FI_ERR_INVALID and call(n=-1) == L.FI_ERR_INVALID
    assert call(kernel=3) == L.FI_ERR_INVALID and call(kernel=-1) == L.FI_ERR_INVALID
    assert call(kernel=3, gradients=None) == L.FI_OK          # the kernel is only read when gradients are asked for
    assert call(n=0, sizes=None, field=None, pos=None) == L.FI_OK  # no points: a no-op
    assert call(values=None, gradients=None) == L.FI_OK


def test_python_shapes_and_empty(emu):
    f = _field((3, 4), 1)
    with pytest.raises(ValueError):
        emu.sample_field(f, np.zeros((2, 3), F))
    with pytest.raises(ValueError):
        emu.sample_field(np.zeros((2, 2, 2, 2), F), np.zeros((2, 4), F))
    v, g = emu.sample_field(f, np.zeros((0, 2), F), 1)
    assert v.shape == (0,) and g.shape == (0, 2)
