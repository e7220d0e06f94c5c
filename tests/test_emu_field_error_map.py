"""CPU: the kernels of csrc/field_error_map.cuh on the functional emulator of tests/emu/, bit for bit against the
oracle port's generate_error_map on the exported system, in 1D, 2D and 3D (axes of 1, 2, 3 and 5 nodes included),
with every model weight, every value and gradient kernel, caller rows between model calls, clones, chunked point and
caller rows, both locations, and the error codes.  Not parity evidence for the CUDA build
(test_gpu_zz_field_error_map.py is); they catch ordering, indexing and protocol errors."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import error_map_cases as E
from conftest import ROOT, bits

F = np.float32
SIZES = [[1], [2], [3], [5], [9], [5, 1], [1, 3], [2, 5], [3, 3], [7, 6], [2, 3, 5], [5, 1, 3], [1, 1, 2], [3, 2, 2], [6, 5, 4]]
RECIPE = ["model", "points0", "rows", "model2", "points1", "points2", "rows", "points3", "points4"]


def _x(f, seed):
    return np.random.default_rng(seed).normal(size=f.num_unknowns).astype(F)


def _check(emu, port, f, kinds, x):
    heat, sums = emu.generate_error_map(f, x, want_sums=True)
    eq = f.eq
    want = port.generate_error_map(eq, x)
    assert heat.dtype == F and heat.shape == (f.num_unknowns,)
    assert np.array_equal(bits(heat), bits(want))
    np.testing.assert_allclose(sums, E.kind_sums(eq, x, kinds), rtol=1e-12, atol=0)
    return heat, sums


@pytest.mark.parametrize("sizes", SIZES, ids=lambda s: "x".join(map(str, s)))
def test_mixed_recipe_vs_port(emu, port, sizes):
    f, kinds = E.build(emu, sizes, RECIPE, n_points=30, seed=len(sizes) * 10 + sizes[0])
    assert set(kinds) == {0, 1, 2}
    _check(emu, port, f, kinds, _x(f, 1))


@pytest.mark.parametrize("recipe", [["model"], ["model2"], ["points1"], ["rows"], ["rows", "model", "rows", "model"],
                                    ["points0", "model", "points0"]], ids="-".join)
def test_single_kinds_and_orders(emu, port, recipe):
    for sizes in ([6], [4, 5], [3, 5, 2]):
        f, kinds = E.build(emu, sizes, recipe, n_points=25, seed=3)
        _check(emu, port, f, kinds, _x(f, 2))


def test_each_model_order_alone(emu, port):
    for key in ["model_0", "model_1", "model_2", "model_3", "model_4", "gradient_smoothness"]:
        for sizes in ([5], [5, 3], [5, 2, 3]):
            w = dict(model_0=0.0, model_1=0.0, model_2=0.0, model_3=0.0, model_4=0.0, gradient_smoothness=0.0)
            w[key] = 0.8
            f = emu.LatticeField(sizes)
            emu.add_field_constraints(f, emu.Weights(**w))
            x = _x(f, 4)
            assert np.array_equal(bits(emu.generate_error_map(f, x)), bits(port.generate_error_map(f.eq, x)))


def test_clone_and_repeat(emu, port):
    f, kinds = E.build(emu, [4, 3, 5], RECIPE, n_points=30, seed=7)
    x = _x(f, 5)
    a, sa = _check(emu, port, f, kinds, x)
    g = E.clone(emu, f)
    b, sb = emu.generate_error_map(g, x, want_sums=True)
    c, sc = emu.generate_error_map(f, x, want_sums=True)
    assert np.array_equal(bits(a), bits(b)) and np.array_equal(bits(a), bits(c))
    assert np.array_equal(sa, sb) and np.array_equal(sa, sc)
    emu.add_rows(g, *E.caller_rows(g.num_unknowns, 5, np.random.default_rng(1)))  # the clone grows on its own
    _check(emu, port, g, np.concatenate([kinds, np.full(5, 2)]), x)


def test_chunked_point_and_caller_rows(emu, port, monkeypatch):
    """Chunk caps of 60 and 7 triplets: many point chunks of one or two points, caller-row chunks of single rows and
    rows longer than the cap.  The result does not depend on the chunking."""
    f, kinds = E.build(emu, [5, 4, 3], RECIPE, n_points=30, seed=9)
    x = _x(f, 6)
    whole, sums = _check(emu, port, f, kinds, x)
    for cap in ("60", "7"):
        monkeypatch.setenv("FI_B200_ERROR_MAP_CHUNK", cap)
        h, s = emu.generate_error_map(f, x, want_sums=True)
        assert np.array_equal(bits(h), bits(whole))
        np.testing.assert_allclose(s, sums, rtol=1e-12, atol=0)


def test_device_location_nan_and_empty(emu, port):
    """loc = FI_DEVICE through the ABI (emulated device memory is host memory); NaN in the solution propagates as the
    reference's arithmetic does; a field without rows gives zeros."""
    from field_interpolation_b200 import _lib as L
    dll = L.lib()
    f, kinds = E.build(emu, [5, 6], RECIPE, n_points=30, seed=11)
    x = _x(f, 7)
    x[[3, 17]] = np.nan
    want = port.generate_error_map(f.eq, x)
    assert np.isnan(want).any()
    heat = np.full(f.num_unknowns, 7, F)
    sums = (C.c_double * 3)()
    assert dll.fi_field_error_map(f._h, x.ctypes.data, L.FI_DEVICE, heat.ctypes.data, sums) == L.FI_OK
    assert np.array_equal(bits(heat), bits(want))
    assert np.isnan(sums[0]) and np.isnan(sums[1])
    assert dll.fi_field_error_map(f._h, x.ctypes.data, L.FI_HOST, heat.ctypes.data, None) == L.FI_OK
    assert np.array_equal(bits(heat), bits(want))
    empty = emu.LatticeField([4, 3])
    h, s = emu.generate_error_map(empty, np.ones(12, F), want_sums=True)
    assert np.array_equal(bits(h), bits(np.zeros(12, F))) and np.array_equal(s, np.zeros(3))


def test_error_codes(emu):
    from field_interpolation_b200 import _lib as L
    dll = L.lib()
    f, _ = E.build(emu, [4, 4], ["model", "points0"], n_points=5)
    x, heat = np.zeros(16, F), np.zeros(16, F)
    assert dll.fi_field_error_map(f._h, x.ctypes.data, L.FI_HOST, heat.ctypes.data, None) == L.FI_OK
    assert dll.fi_field_error_map(None, x.ctypes.data, L.FI_HOST, heat.ctypes.data, None) == L.FI_ERR_INVALID
    assert dll.fi_field_error_map(f._h, None, L.FI_HOST, heat.ctypes.data, None) == L.FI_ERR_INVALID
    assert dll.fi_field_error_map(f._h, x.ctypes.data, L.FI_HOST, None, None) == L.FI_ERR_INVALID
    assert dll.fi_field_error_map(f._h, x.ctypes.data, 2, heat.ctypes.data, None) == L.FI_ERR_INVALID
    with pytest.raises(ValueError):
        emu.generate_error_map(f, np.zeros(15, F))
    # point rows on more than 2^31 - 1 nodes: their columns do not fit int32 (checked before anything is read)
    big = emu.LatticeField([2048, 1024, 1025])
    emu.add_points(big, 1.0, 1, 0.0, 1, np.array([[3.5, 4.5, 5.5]], F))
    assert dll.fi_field_error_map(big._h, x.ctypes.data, L.FI_HOST, heat.ctypes.data, None) == L.FI_ERR_RANGE


def test_cpp_drop_in_on_the_emulator(tmp_path):
    """tests/cpp/error_map_driver.cpp (b200::generate_error_map on a deferred LatticeField with a hand-written row) with
    libfi_b200.so resolved to the emulator build, against the same field built through the ABI."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    os.symlink(build_emu.build(), tmp_path / "libfi_b200.so")
    env = dict(os.environ, FI_B200_TEST_EMU="1", LD_LIBRARY_PATH=str(tmp_path) + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_zz_field_error_map.py"), "-m", "gpu", "-q", "-x",
                        "-k", "cpp_error_map_driver", "-p", "no:cacheprovider"], env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    assert " passed" in r.stdout and " failed" not in r.stdout
