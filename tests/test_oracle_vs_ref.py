"""CPU: the oracle port against the reference's own code, bit for bit, on randomised inputs that hit every skip rule.

What the reference returns on these inputs is stored in tests/golden/vs_ref.npz (written by tests/golden/make_golden.py),
so the comparison runs on every checkout.  Small outputs are stored whole; larger ones as the SHA-256 of their dtype,
shape and bytes.  Where oracle/_ref has been built from the reference's source tree (oracle/Makefile), the port is also
compared with it live."""
import hashlib

import numpy as np
import pytest

from conftest import load_golden
from field_interpolation_b200 import workloads as W
from oracle import oracle as O

SDF_SIZES = [[13], [2], [9, 7], [1, 5], [6, 5, 7], [3, 3, 3], [2, 9, 2]]
STORE_WHOLE_UP_TO = 1024  # bytes; a larger output is stored as its digest


def digest(a):
    a = np.ascontiguousarray(a)
    return np.frombuffer(hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).digest(), np.uint8)


def stored_form(outputs):
    """The arrays make_golden.py writes for `outputs` (name -> array)."""
    return {(k if a.nbytes <= STORE_WHOLE_UP_TO else k + ".sha256"): (a if a.nbytes <= STORE_WHOLE_UP_TO else digest(a))
            for k, a in ((k, np.ascontiguousarray(v)) for k, v in outputs.items())}


def _system(prefix, s):
    return {f"{prefix}.rows": s.rows, f"{prefix}.cols": s.cols, f"{prefix}.vals": s.vals, f"{prefix}.rhs": s.rhs}


def sdf_from_points_outputs(lib, sizes, vk, gk):
    D = len(sizes)
    seed = 1000 * D + 10 * vk + gk + sum(sizes)
    pos, nrm = W.random_cloud(D, 300, sizes, seed)
    pw = np.random.default_rng(seed).uniform(0, 2, 300).astype(np.float32)
    pw[::5] = 0
    w = O.make_weights(model_0=0.3 * (seed % 2), model_1=0.2, model_2=0.5, model_3=0.1 * (seed % 3 == 0),
                       model_4=0.05, gradient_smoothness=0.2 * (seed % 2 == 0), value_kernel=vk, gradient_kernel=gk)
    out = {}
    for tag, weights_arr in (("unweighted", None), ("weighted", pw)):
        out.update(_system(f"sdf.{'x'.join(map(str, sizes))}.v{vk}g{gk}.{tag}", lib.sdf_from_points(sizes, w, pos, nrm, weights_arr).system()))
    return out


def single_point_builder_outputs(lib):
    rng = np.random.default_rng(5)
    out = {}
    for sizes in ([10], [6, 7], [4, 5, 6]):
        D = len(sizes)
        f = lib.field(sizes)
        pos, nrm = W.random_cloud(D, 200, sizes, 77)
        ret = []
        for p, g in zip(pos, nrm):
            v, w = float(rng.normal()), float(rng.choice([0.0, 0.5, 1.0, 2.0]))
            k = int(rng.integers(0, 3))
            ret.append([f.add_value_constraint(p, v, w), f.add_value_constraint_nearest_neighbor(p, g, v, w),
                        f.add_gradient_constraint(p, g, w, k)])
        name = "single." + "x".join(map(str, sizes))
        out[name + ".returns"] = np.array(ret, dtype=bool)
        out.update(_system(name, f.system()))
    return out


def upscale_and_error_map_outputs(lib):
    rng = np.random.default_rng(9)
    out = {}
    for small, large in (([3], [10]), ([5, 3], [11, 8]), ([4, 3, 5], [9, 8, 13]), ([8, 8, 8], [16, 16, 16])):
        src = rng.normal(size=int(np.prod(small))).astype(np.float32)
        out["upscale." + "x".join(map(str, large))] = lib.upscale_field(src, small, large)
    s = lib.sdf_from_points([8, 9], O.make_weights(), *W.random_cloud(2, 100, [8, 9], 3)).system()
    sol = rng.normal(size=72).astype(np.float32)
    out.update(_system("error_map.8x9", s))
    out["error_map.8x9.heat"] = lib.generate_error_map(s, sol)
    return out


def iso_surface_outputs(lib):
    """Randomised: fields with exact zeros, negative zeros, saddles and 1-wide shapes."""
    rng = np.random.default_rng(21)
    out = {}
    for h, w in ((2, 2), (5, 7), (33, 20), (1, 5), (6, 1), (64, 64), (3, 200)):
        a = rng.standard_normal((h, w)).astype(np.float32)
        a[rng.random((h, w)) < 0.1] = 0.0
        a[rng.random((h, w)) < 0.05] = np.float32(-0.0)
        name = f"iso.{h}x{w}"
        for iso in (0.0, 0.3, -1.5):
            lines = lib.iso_surface(a, iso)
            out[f"{name}.iso{iso}.lines"] = lines
            out[f"{name}.iso{iso}.area"] = np.float32(lib.calc_area(lines))
        out[f"{name}.marching_squares"] = lib.marching_squares(a)
        for up in (2, 3, 7):
            out[f"{name}.bicubic{up}"] = lib.bicubic_upsample(a, up)
    return out


@pytest.fixture(scope="module")
def stored():
    return load_golden("vs_ref")


def check(make_outputs, port, stored):
    """The port's outputs equal what the reference returned (stored), and the live reference's where it is built."""
    got = stored_form(make_outputs(port))
    for k, a in got.items():
        assert k in stored.files, f"{k}: not in tests/golden/vs_ref.npz"
        want = stored[k]
        assert a.dtype == want.dtype and a.shape == want.shape and a.tobytes() == want.tobytes(), k
    ref = O.reference()
    if ref is not None:
        want = stored_form(make_outputs(ref))
        assert got.keys() == want.keys()
        for k in got:
            assert got[k].tobytes() == want[k].tobytes(), k


@pytest.mark.parametrize("sizes", SDF_SIZES)
@pytest.mark.parametrize("vk", [0, 1])
@pytest.mark.parametrize("gk", [0, 1, 2])
def test_sdf_from_points_matches_reference(port, stored, sizes, vk, gk):
    check(lambda lib: sdf_from_points_outputs(lib, sizes, vk, gk), port, stored)


def test_single_point_builders_match_reference(port, stored):
    check(single_point_builder_outputs, port, stored)


def test_upscale_and_error_map_match_reference(port, stored):
    check(upscale_and_error_map_outputs, port, stored)


def test_iso_surface_helpers_match_reference(port, stored):
    check(iso_surface_outputs, port, stored)
