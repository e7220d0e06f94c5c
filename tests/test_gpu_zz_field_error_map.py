"""GPU: fi_field_error_map (csrc/field_error_map.cuh) — generate_error_map of a field's own system on the device.

Bar: bit-identical to the oracle port's generate_error_map on the exported triplets for randomised systems (every
model weight, both value kernels, all gradient kernels, caller rows between model calls) up to 128^3 with 100k points
and 2048^2 with 200k points; repeat calls and clones give the same bits; the row error sums agree with the heat map;
an analytic model_2 check at 512^3 with no oracle; a deferred 1024^3 field whose export is impossible; the solved
C4-style cloud at 512^3, device-resident in and out; the C++ drop-in on a deferred field."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import error_map_cases as E
from conftest import ROOT, bits

pytestmark = pytest.mark.gpu
F = np.float32


@pytest.fixture(scope="module")
def fi():
    import field_interpolation_b200 as m
    return m


def _x(n, seed):
    return np.random.default_rng(seed).normal(size=n).astype(F)


def _heat_sum_matches(heat, sums):
    """sum(heat) spreads each row's fp32 err^2 over its columns (terms rounded to fp32, heat summed in fp32): it agrees
    with the fp64 row sums to fp32 summation rounding."""
    h = float(heat.double().sum()) if hasattr(heat, "is_cuda") else float(np.asarray(heat, np.float64).sum())
    assert abs(h - sums.sum()) <= 1e-4 * sums.sum(), (h, sums)


# ---- 1. bit-identical to the port on the exported system ---------------------------------------------------------------
@pytest.mark.parametrize("sizes,n_points,recipe", [
    ([1000], 3000, ["model", "points0", "rows", "model2", "points1", "points2", "rows"]),
    ([97, 131], 20_000, ["model", "points0", "rows", "model2", "points1", "points3", "points4", "rows"]),
    ([2048, 2048], 200_000, ["model", "points0"]),
    ([48, 37, 29], 30_000, ["model", "points0", "rows", "model2", "points1", "points2", "points3", "points4", "rows"]),
    ([96, 96, 96], 100_000, ["model", "points1", "rows", "model2", "points0"]),
    ([128, 128, 128], 100_000, ["model2", "points0", "points1", "rows"]),
], ids=["1d", "2d", "2048sq_200k", "3d_ragged", "96cube_all_weights", "128cube_100k"])
def test_bit_identical_to_port(fi, port, sizes, n_points, recipe):
    f, kinds = E.build(fi, sizes, recipe, n_points=n_points, seed=sum(sizes))
    x = _x(f.num_unknowns, len(sizes))
    heat, sums = fi.generate_error_map(f, x, want_sums=True)
    eq = f.eq
    want = port.generate_error_map(eq, x)
    assert np.array_equal(bits(heat), bits(want))
    np.testing.assert_allclose(sums, E.kind_sums(eq, x, kinds), rtol=1e-9, atol=0)


# ---- 2. reproducible; sums agree with the heat ----------------------------------------------------------------------------
def test_repeat_and_clone_identical(fi):
    import torch
    f, _ = E.build(fi, [160, 150, 140], ["model", "points0", "model2", "points2"], n_points=200_000, seed=5)
    x = torch.from_numpy(_x(f.num_unknowns, 3)).cuda()
    a, sa = fi.generate_error_map(f, x, want_sums=True)
    b, sb = fi.generate_error_map(f, x, want_sums=True)
    c, sc = fi.generate_error_map(E.clone(fi, f), x, want_sums=True)
    assert a.is_cuda and torch.equal(a.view(torch.int32), b.view(torch.int32)) and torch.equal(a.view(torch.int32), c.view(torch.int32))
    assert np.array_equal(sa, sb) and np.array_equal(sa, sc)
    _heat_sum_matches(a, sa)  # no caller rows: every row has sq != 0


# ---- 3. analytic: model_2 rows of an integer quadratic --------------------------------------------------------------------
def test_quadratic_model2_closed_form_512(fi):
    """x = cx^2 + 2 cy^2 + 3 cz^2 (integers below 2^24: exact in fp32) has second difference 2 a_d along axis d, so
    every model_2 row (coefficients w, -2w, w) has err = -2 a_d w, exactly.  The heat map must equal an fp64 computation
    of err^2 spread over each row's taps by c^2 / sum c^2, to 1e-5 relative."""
    import torch
    n, w = 512, 0.5
    f = fi.LatticeField([n, n, n])
    fi.add_field_constraints(f, fi.Weights(model_2=w))
    c = torch.arange(n, device="cuda", dtype=torch.float64)
    x64 = c.view(1, 1, n) ** 2 + 2 * c.view(1, n, 1) ** 2 + 3 * c.view(n, 1, 1) ** 2
    x = x64.to(torch.float32).reshape(-1)
    heat, sums = fi.generate_error_map(f, x, want_sums=True)
    want = torch.zeros((n, n, n), dtype=torch.float64, device="cuda")
    coef = torch.tensor([w, -2 * w, w], dtype=torch.float64)
    share = (coef * coef / (coef * coef).sum()).tolist()
    total = 0.0
    for d in range(3):  # axis d of the (z, y, x) tensor is lattice axis 2 - d
        xd = x64.movedim(2 - d, 0)
        err = -(w * xd[:-2] - 2 * w * xd[1:-1] + w * xd[2:])  # = -2 a_d w
        e2 = err * err
        total += float(e2.sum())
        wd = want.movedim(2 - d, 0)
        for m in range(3):
            wd[m:n - 2 + m] += share[m] * e2
    rel = (heat.view(n, n, n).double() - want).abs().max() / want.abs().max()
    assert float(rel) <= 1e-5, float(rel)
    assert abs(sums[0] - total) <= 1e-12 * total and sums[1] == 0 and sums[2] == 0


# ---- 4. a deferred 1024^3 field: no triplet view exists ------------------------------------------------------------------
def test_deferred_1024_beyond_export(fi):
    import torch
    from field_interpolation_b200 import _lib as L
    from field_interpolation_b200 import workloads as W
    n = 1024
    sizes = [n, n, n]
    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    pos = W.to_lattice(cloud["unit_pos"], sizes)
    f = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
    assert L.lib().fi_field_export(f._h, None, None) == L.FI_ERR_RANGE
    # an analytic field: distance to the sphere of the cloud (centre 0.5, radius 0.3 in unit coordinates)
    c = (torch.arange(n, device="cuda", dtype=torch.float32) / (n - 1) - 0.5)
    x = (torch.sqrt(c.view(1, 1, n) ** 2 + c.view(1, n, 1) ** 2 + c.view(n, 1, 1) ** 2) - 0.3) * (n - 1)
    x = x.reshape(-1).contiguous()
    L.check(L.lib().fi_trim_memory())
    heat, sums = fi.generate_error_map(f, x, want_sums=True)
    cached = int(L.lib().fi_cached_bytes())
    cap = 1 << 26
    print(f"1024^3 error map: library device memory {cached / 2**30:.2f} GiB, sums {sums}")
    assert cached <= 64 * cap + (1 << 28), cached  # chunk scratch (~40 B per triplet), model partials
    assert heat.is_cuda and bool(torch.isfinite(heat).all()) and sums[2] == 0 and sums[0] > 0 and sums[1] > 0
    _heat_sum_matches(heat, sums)


# ---- 5. the solved C4-style cloud at 512^3, device-resident --------------------------------------------------------------
def test_solved_cloud_512_device_resident(fi):
    import torch
    from field_interpolation_b200 import workloads as W
    n = 512
    sizes = [n, n, n]
    cloud = W.sphere_torus_3d(1_000_000, seed=0)
    pos = W.to_lattice(cloud["unit_pos"], sizes)
    f = fi.sdf_from_points(sizes, fi.Weights(), pos, cloud["normals"])
    out = torch.zeros(n ** 3, dtype=torch.float32, device="cuda")
    _, st = f.solve(fi.solve_options(fi.FI_F32, 200, 1e-5, preconditioner=fi.FI_PRECOND_MULTIGRID), out=out)
    heat, sums = fi.generate_error_map(f, out, want_sums=True)
    assert heat.is_cuda and heat.shape == (n ** 3,) and bool(torch.isfinite(heat).all())
    assert bool((heat >= 0).all())  # every term is c^2 / sum c^2 * err^2
    _heat_sum_matches(heat, sums)
    # CG from a zero guess lowers the objective below that of the zero field (whose error is the gradient rows' rhs)
    zero, zsums = fi.generate_error_map(f, torch.zeros_like(out), want_sums=True)
    print(f"solved 512^3 cloud: objective {sums.sum():.4g} (model {sums[0]:.4g}, points {sums[1]:.4g}) vs zero field {zsums.sum():.4g}; solve {st}")
    assert sums.sum() < zsums.sum()


# ---- 6. host / device, errors ------------------------------------------------------------------------------------------------
def test_host_and_device_identical_and_errors(fi):
    import torch
    from field_interpolation_b200 import _lib as L
    f, _ = E.build(fi, [33, 20, 17], ["model", "points1", "rows", "points2"], n_points=5000, seed=2)
    x = _x(f.num_unknowns, 9)
    h, hs = fi.generate_error_map(f, x, want_sums=True)
    d, ds = fi.generate_error_map(f, torch.from_numpy(x).cuda(), want_sums=True)
    assert isinstance(h, np.ndarray) and d.is_cuda and np.array_equal(bits(d.cpu().numpy()), bits(h)) and np.array_equal(hs, ds)
    dll = L.lib()
    heat = torch.empty_like(d)
    xd = torch.from_numpy(x).cuda()
    assert dll.fi_field_error_map(None, xd.data_ptr(), L.FI_DEVICE, heat.data_ptr(), None) == L.FI_ERR_INVALID
    assert dll.fi_field_error_map(f._h, None, L.FI_DEVICE, heat.data_ptr(), None) == L.FI_ERR_INVALID
    assert dll.fi_field_error_map(f._h, xd.data_ptr(), L.FI_DEVICE, None, None) == L.FI_ERR_INVALID
    assert dll.fi_field_error_map(f._h, xd.data_ptr(), 5, heat.data_ptr(), None) == L.FI_ERR_INVALID
    big = fi.LatticeField([2048, 1024, 1025])
    fi.add_points(big, 1.0, 1, 0.0, 1, np.array([[3.5, 4.5, 5.5]], F))
    assert dll.fi_field_error_map(big._h, xd.data_ptr(), L.FI_DEVICE, heat.data_ptr(), None) == L.FI_ERR_RANGE


# ---- 7. the C++ drop-in on a deferred field -------------------------------------------------------------------------------
def test_cpp_error_map_driver(fi, tmp_path):
    from field_interpolation_b200 import build as B
    from field_interpolation_b200 import workloads as W
    B.build()
    exe = B.build_cpp_driver(os.path.join(ROOT, "tests", "cpp", "error_map_driver.cpp"), os.path.join(ROOT, "tests", "cpp", "error_map_driver"))
    sizes = [40, 33, 27]
    cloud = W.sphere_torus_3d(20_000, seed=6)
    pos = np.ascontiguousarray(W.to_lattice(cloud["unit_pos"], sizes), F)
    nrm = np.ascontiguousarray(cloud["normals"], F)
    x = _x(int(np.prod(sizes)), 6)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as h:
        h.write(struct.pack("<iiiiq", 3, *sizes, len(pos)))
        h.write(pos.tobytes())
        h.write(nrm.tobytes())
        h.write(x.tobytes())
    r = subprocess.run([exe, str(inp), str(outp)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    raw = open(outp, "rb").read()
    heat = np.frombuffer(raw[:4 * x.size], F)
    sums = np.frombuffer(raw[4 * x.size:], np.float64)
    f = fi.LatticeField(sizes)
    w = fi.Weights()
    fi.add_field_constraints(f, w)
    fi.add_points(f, w.data_pos, w.value_kernel, w.data_gradient, w.gradient_kernel, pos, nrm)
    fi.add_equation(f, 2.0, 0.5, [(1, 1.0), (3, -0.5)])
    want, wsums = fi.generate_error_map(f, x, want_sums=True)
    assert np.array_equal(bits(heat), bits(want)) and np.array_equal(sums, wsums) and sums[2] > 0
