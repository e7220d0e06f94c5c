import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
WKEYS = ["data_pos", "data_gradient", "model_0", "model_1", "model_2", "model_3", "model_4", "gradient_smoothness",
         "value_kernel", "gradient_kernel"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    if os.environ.get("FI_B200_TEST_EMU") == "1":
        # Developer switch for the GPU-less build container, never set by the driver: run `-m gpu` tests against the CPU
        # functional emulator build of the library (tests/emu/) to debug kernel LOGIC before a GPU box is available.
        # Passing this way is not parity evidence; only a run on the B200 is.
        use_emulated_library()


def use_emulated_library():
    """Swaps field_interpolation_b200._lib's handle for tests/emu/_build/libfi_emu.so in this process; returns a
    function that undoes it."""
    import ctypes
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import build_emu
    from field_interpolation_b200 import _lib
    dll = ctypes.CDLL(build_emu.build())
    assert dll.fi_emu_marker() == 1
    for name, (res, args) in _lib.SIGNATURES.items():
        fn = getattr(dll, name)
        fn.restype, fn.argtypes = res, args
    before = _lib._dll
    _lib._dll = dll

    def undo():
        _lib._dll = before
    return undo


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def golden_names(prefix):
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.startswith(prefix) and f.endswith(".npz"))


def weights_kwargs(vec):
    kw = {k: float(v) for k, v in zip(WKEYS, vec)}
    kw["value_kernel"] = int(kw["value_kernel"])
    kw["gradient_kernel"] = int(kw["gradient_kernel"])
    return kw


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_system_bit_exact(got, want_rows, want_cols, want_vals, want_rhs):
    assert got.num_rows == len(want_rhs) and got.num_triplets == len(want_vals)
    assert np.array_equal(got.rows, want_rows)
    assert np.array_equal(got.cols, want_cols)
    assert np.array_equal(bits(got.vals), bits(want_vals))
    assert np.array_equal(bits(got.rhs), bits(want_rhs))


@pytest.fixture(scope="session")
def port():
    from oracle import oracle as O
    return O.port()


@pytest.fixture
def emu():
    """The package bound to the CPU functional emulator build of the library (tests/emu/) for one test."""
    undo = use_emulated_library()
    import field_interpolation_b200 as m
    try:
        yield m
    finally:
        undo()
