"""CPU: the fp64 restatement of the multigrid preconditioner (tests/mg_reference.py) that the GPU tests of
test_gpu_multigrid_operator.py compare the library's cycle with — checked here on its own terms."""
import numpy as np
import pytest
import scipy.linalg as sla

import mg_reference as R
from field_interpolation_b200 import workloads as W


def _problem(sizes, npts=60, seed=3, **wkw):
    D = len(sizes)
    if D == 1:
        rng = np.random.default_rng(seed)
        pos = rng.uniform(0.5, sizes[0] - 1.5, (npts, 1)).astype(np.float32)
        nrm = np.where(rng.uniform(size=(npts, 1)) < 0.5, -1.0, 1.0).astype(np.float32)
    else:
        pos, nrm = W.random_cloud(D, npts, sizes, seed=seed)
    return R.Problem(list(sizes), dict(wkw), pos, nrm)


def _info(port, prob, coarsest, nu=2, nu_coarse=4, gamma=1, w_levels=3, ratio=12.0, margin=1.1):
    sizes = R.level_sizes(prob.sizes, coarsest)
    lmax = []
    for l, s in enumerate(sizes[:-1]):
        A = R.level_operator(port, prob, s, l).toarray()
        d = 1.0 / np.sqrt(A.diagonal())
        lmax.append(margin * sla.eigvalsh(d[:, None] * A * d[None, :]).max())
    return {"levels": len(sizes), "sizes": [s + [1] * (3 - len(s)) for s in sizes], "lmax": lmax + [0.0], "nu": nu,
            "nu_coarse": nu_coarse, "gamma": gamma, "w_levels": w_levels, "cheb_ratio": ratio}


@pytest.mark.parametrize("small,large", [([5], [9]), ([5], [10]), ([4], [7]), ([7, 4], [13, 8]), ([3, 4, 5], [5, 8, 9]),
                                         ([4, 3], [7, 6]), ([5, 5], [9, 10])])
def test_prolongation_is_the_ports_upscale(port, small, large):
    rng = np.random.default_rng(len(small) * 10 + large[0])
    v = rng.normal(size=int(np.prod(small))).astype(np.float32)
    want = port.upscale_field(v, small, large)
    got = R.prolongation(large, small) @ v.astype(np.float64)
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-6 * np.abs(v).max())
    # a coarse node is touched by at most 4 fine nodes per axis (the transfer kernels' fan), every fine row sums to one
    P = R.prolongation(large, small)
    np.testing.assert_allclose(np.asarray(P.sum(axis=1)).ravel(), 1.0, rtol=0, atol=1e-15)
    assert np.asarray((P != 0).sum(axis=0)).max() <= 4 ** len(small)


def test_prolongation_size_one_axis():
    """A size-1 axis (which upscale_field does not define) carries the one plane over unchanged."""
    assert (R.prolongation([7, 1, 6], [4, 1, 3]) != R.prolongation([7, 6], [4, 3])).nnz == 0


def test_level_sizes_follow_the_coarsening_rule():
    assert R.level_sizes([33, 17], 20) == [[33, 17], [17, 9], [9, 5]]  # next would have an axis of 3 < 4
    assert R.level_sizes([64], 10) == [[64], [32], [16], [8]]          # 8 <= 10
    assert R.level_sizes([20, 1, 20], 10) == [[20, 1, 20], [10, 1, 10], [5, 1, 5]]  # size-1 axes never stop coarsening
    assert R.level_sizes([9, 9], 600) == [[9, 9]]


@pytest.mark.parametrize("gamma", [1, 2])
@pytest.mark.parametrize("sizes,coarsest,wkw", [([80], 12, {}), ([25, 24], 60, dict(model_1=0.2, gradient_smoothness=0.3)),
                                                ([9, 8, 7], 100, dict(model_0=0.1, model_3=0.2))])
def test_reference_cycle_is_symmetric(port, sizes, coarsest, wkw, gamma):
    prob = _problem(sizes, **wkw)
    H = R.Hierarchy(port, prob, _info(port, prob, coarsest=coarsest, gamma=gamma, w_levels=2))
    assert H.L >= (3 if len(sizes) < 3 else 2)
    B = H.matrix()
    assert np.abs(B - B.T).max() <= 1e-12 * np.abs(B).max()


def test_two_level_cycle_tends_to_the_inverse(port):
    """With Chebyshev smoothing over the whole spectrum and many steps, pre-smoothing alone solves the level: the cycle
    is A^-1 whatever the coarse correction does."""
    prob = _problem([24], npts=30)
    info = _info(port, prob, coarsest=12)
    assert info["levels"] == 2
    A = R.level_operator(port, prob, [24], 0).toarray()
    d = 1.0 / np.sqrt(A.diagonal())
    ev = sla.eigvalsh(d[:, None] * A * d[None, :])
    info.update(lmax=[ev.max(), 0.0], cheb_ratio=ev.max() / ev.min() * 1.001)
    Ainv = np.linalg.inv(A)
    errs = []
    for nu in (2, 20, 400):
        info.update(nu=nu, nu_coarse=nu)
        B = R.Hierarchy(port, prob, info).matrix()
        errs.append(np.abs(B - Ainv).max() / np.abs(Ainv).max())
    assert errs[0] > errs[1] > errs[2] and errs[2] <= 1e-9, errs


def test_reference_pcg_with_exact_preconditioner_takes_one_step(port):
    prob = _problem([30])
    A = R.level_operator(port, prob, [30], 0)
    b = np.random.default_rng(1).normal(size=30)
    x, it = R.pcg(A, b, lambda r: np.linalg.solve(A.toarray(), r), 1e-10)
    assert it == 1 and np.allclose(A @ x, b)
