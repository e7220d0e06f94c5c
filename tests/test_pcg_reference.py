"""CPU: the fp64 restatement of the Jacobi-PCG iteration (tests/pcg_reference.py) against the oracle.

* S + P formed matrix-free from the model definition and the point / caller rows equals the normal equations of the
  reference-assembled system (O.normal_equations_f64) to 1e-13 relative, on 1D / 2D / 3D lattices with every model
  order, gradient smoothness on and off, axes of 1, 2, 3 and 5 nodes, all value and gradient kernels and caller rows;
  the z-slab evaluation equals the whole-lattice one;
* the restated k-step PCG equals a dense fp64 preconditioned CG on small systems.
"""
import numpy as np
import pytest

import pcg_reference as PR
from oracle import oracle as O

ALL_ON = dict(model_0=0.1, model_1=0.2, model_2=0.5, model_3=0.3, model_4=0.25)

# sizes, model weights (a list: one dict per add_model call), value / gradient kernels, caller rows
CASES = {
    "1d_all": ([13], [ALL_ON], 1, 1, True),
    "1d_5": ([5], [dict(model_1=0.3, model_4=0.2)], 0, 0, False),
    "1d_3_m3": ([3], [dict(model_2=0.0, model_3=0.4)], 1, 2, True),
    "2d_gs": ([9, 7], [dict(ALL_ON, gradient_smoothness=0.3)], 1, 2, True),
    "2d_axis1": ([11, 1], [dict(model_1=0.2, gradient_smoothness=0.2)], 1, 1, False),
    "2d_axis2": ([2, 6], [dict(model_3=0.3, gradient_smoothness=0.1)], 0, 1, False),
    "2d_two_calls": ([8, 5], [dict(model_1=0.2), dict(model_2=0.3, gradient_smoothness=0.25)], 1, 0, True),
    "3d_gs": ([6, 5, 7], [dict(model_1=0.2, model_2=0.5, gradient_smoothness=0.15)], 1, 1, True),
    "3d_all": ([5, 3, 9], [dict(ALL_ON, gradient_smoothness=0.2)], 1, 2, False),
    "3d_flat": ([7, 1, 6], [dict(model_4=0.2, gradient_smoothness=0.3)], 0, 2, True),
    "3d_thin": ([2, 3, 5], [dict(model_0=0.3, model_2=0.4)], 1, 0, False),
}


def build_case(port, sizes, models, vk, gk, rows, npts=None, seed=0):
    """The port's field: the add_model calls, then add_points (kernels vk / gk), then caller rows.  Returns the whole
    system, the number of model rows and the point-row matrix A_pts."""
    D, n = len(sizes), int(np.prod(sizes))
    f = port.field(sizes)
    for w in models:
        f.add_field_constraints(O.make_weights(**w))
    nmodel = f.system().num_rows
    rng = np.random.default_rng(seed + n)
    npts = npts or max(4, n // 3)
    pos = (rng.uniform(0, 1, (npts, D)) * (np.array(sizes) - 1 + 0.6) - 0.3).astype(np.float32)
    nrm = rng.normal(size=(npts, D)).astype(np.float32)
    f.add_points(1.0, vk, 0.7, gk, pos, nrm)
    if rows:
        f.add_equation(0.7, 1.5, [0, n - 1, n // 2], [1.0, -2.0, 0.5])
        f.add_equation(0.3, -1.0, [n // 3], [2.0])
    sys_ = f.system()
    trips = np.zeros(sys_.num_triplets, dtype=[("row", np.int32), ("col", np.int32), ("value", np.float32)])
    trips["row"], trips["col"], trips["value"] = sys_.rows, sys_.cols, sys_.vals
    keep = trips["row"] >= nmodel
    A_pts = PR.rows_matrix(trips[keep], nmodel, sys_.num_rows - nmodel, n)
    return sys_, nmodel, A_pts


@pytest.mark.parametrize("name", list(CASES))
def test_operator_matches_normal_equations(port, name):
    sizes, models, vk, gk, rows = CASES[name]
    sys_, _, A_pts = build_case(port, sizes, models, vk, gk, rows)
    n = int(np.prod(sizes))
    A, _ = O.normal_equations_f64(sys_, n)
    op = PR.Operator(sizes, models, A_pts)
    M = op.matrix().toarray()
    ref = A.toarray()
    scale = np.abs(ref).max()
    assert np.abs(M - ref).max() <= 1e-13 * scale, np.abs(M - ref).max() / scale
    np.testing.assert_allclose(op.diagonal(), ref.diagonal(), rtol=0, atol=1e-13 * scale)
    # |S| |p| and |P| |p| bound |(S + P) p| entry by entry
    p = np.random.default_rng(1).normal(size=n)
    assert np.all(np.abs(ref @ p) <= op.apply(p, absolute=True) * (1 + 1e-12) + 1e-300)


@pytest.mark.parametrize("sizes,models", [([40, 9, 37], [dict(model_4=0.2, gradient_smoothness=0.3)]),
                                          ([16, 12, 23], [dict(model_1=0.3)])])
def test_slab_evaluation_matches_whole_lattice(sizes, models):
    """The z-slab walk (R halo planes) against one window over the whole lattice, S p and |S| |p|."""
    S = PR.Smoothness(sizes, models)
    p = np.random.default_rng(2).normal(size=int(np.prod(sizes)))
    whole = S._window(p.reshape(sizes[::-1]), 0, False).ravel()
    for slab in (1, 4, 16):
        np.testing.assert_allclose(S.apply(p, slab=slab), whole, rtol=1e-14, atol=1e-14 * np.abs(whole).max())
    whole_abs = S._window(np.abs(p).reshape(sizes[::-1]), 0, True).ravel()
    np.testing.assert_allclose(S.apply(p, absolute=True, slab=3), whole_abs, rtol=1e-14)


def dense_pcg(A, b, minv, k):
    """Textbook preconditioned CG, k steps from zero, dense fp64."""
    x = np.zeros_like(b)
    r = b.copy()
    z = minv * r
    p = z.copy()
    rz = r @ z
    for _ in range(k):
        q = A @ p
        a = rz / (p @ q)
        x += a * p
        r -= a * q
        z = minv * r
        rz_new = r @ z
        p = z + rz_new / rz * p
        rz = rz_new
    return x, r


@pytest.mark.parametrize("name", ["1d_all", "2d_gs", "3d_gs", "3d_flat"])
@pytest.mark.parametrize("k", [1, 2, 5, 9])
def test_short_loop_matches_dense_cg(port, name, k):
    sizes, models, vk, gk, rows = CASES[name]
    sys_, _, A_pts = build_case(port, sizes, models, vk, gk, rows)
    n = int(np.prod(sizes))
    A, atb = O.normal_equations_f64(sys_, n)
    op = PR.Operator(sizes, models, A_pts)
    x, r, _, st = PR.pcg(op, atb, k)
    xd, rd = dense_pcg(A.toarray(), atb, op.minv(), k)
    assert st["iters"] == k and st["done"] == 1 and st["breakdown"] == 0
    np.testing.assert_allclose(x, xd, rtol=0, atol=1e-10 * np.abs(xd).max())
    np.testing.assert_allclose(r, rd, rtol=0, atol=1e-10 * np.abs(atb).max())
    assert abs(st["rr"] - rd @ rd) <= 1e-9 * (atb @ atb)


def test_recurrence_stops_where_the_solver_stops():
    """done once rr <= tol2bb, at max_iters, or when rho stops being positive; breakdown on pq <= 0 / NaN."""
    st = PR.init_state(np.array([1.0, 0.0]), np.array([1.0, 0.0]), np.array([2.0, 0.0]), 0.25, 3)
    assert st["done"] == 0 and st["tol2bb"] == 0.25 and st["rho"] == [1.0, 0.0] and PR.beta(st, 0) == 0.0
    PR.finish(st, 0, 0.5, 2.0)
    assert st["done"] == 0 and st["iters"] == 1 and st["rho"] == [1.0, 0.5] and PR.beta(st, 1) == 0.5
    PR.finish(st, 1, 0.25, 0.25)
    assert st["done"] == 1  # rr <= tol2bb
    st = PR.init_state(np.ones(2), np.ones(2), np.ones(2), 1e-3, 1)
    PR.finish(st, 0, 1.0, 1.0)
    assert st["done"] == 1  # max_iters
    st = PR.init_state(np.ones(2), np.ones(2), np.ones(2), 1e-3, 9)
    PR.finish(st, 0, 0.0, 1.0)
    assert st["done"] == 1  # rho <= 0
