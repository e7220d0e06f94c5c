"""CPU: the numpy restatement of fi_sample_field (tests/sample_port.py) against the rows the CPU oracle port emits for
add_value_constraint(p, 1, 1) and add_gradient_constraint(p, (1, ..., 1), 1, K); test_oracle_golden pins those rows
to the reference's own code.  Each row's sequential fp32 dot with the field, divided by its rhs (the sum of its
weights), must equal the port's value or gradient component.  They are compared as values (+0 == -0), since the row
of kernel 0 reads x[cell + s_d] + (-x[cell]) where the port subtracts.  Where the oracle emits no row, or a row whose
rhs is 0, the port must give NaN."""
import numpy as np
import pytest

import sample_port as S
from sample_port import reference_measures, same_values

F = np.float32


@pytest.mark.parametrize("sizes", [[7], [1], [2], [6, 5], [1, 4], [4, 3, 5], [2, 2, 2], [3, 1, 4]])
@pytest.mark.parametrize("kernel", [0, 1, 2])
def test_port_matches_reference_rows(port, sizes, kernel):
    rng = np.random.default_rng(len(sizes) * 31 + sum(sizes) + kernel)
    x = rng.standard_normal(int(np.prod(sizes))).astype(F)
    pts = S.positions_of_every_kind(sizes, 60, seed=kernel + 7 * sum(sizes))
    values, grads = S.sample(sizes, x, pts, kernel)
    want_v, want_g = zip(*(reference_measures(port, sizes, x, p, kernel) for p in pts))
    same_values(values, np.array(want_v, F))
    same_values(grads, np.array(want_g, F))
    assert np.isfinite(values).sum() > len(pts) // 3


def test_values_only_equals_values_with_gradients():
    sizes = [5, 4, 3]
    x = np.random.default_rng(0).standard_normal(60).astype(F)
    pts = S.positions_of_every_kind(sizes, 50, seed=1)
    v = S.sample(sizes, x, pts)
    for k in (0, 1, 2):
        assert np.array_equal(S.sample(sizes, x, pts, k)[0].view(np.uint32), v.view(np.uint32))


def test_non_finite_and_far_points_are_nan():
    sizes = [4, 4]
    x = np.arange(16, dtype=F)
    pts = np.array([[np.nan, 1], [1, np.inf], [-np.inf, 1], [1e30, 1], [1, -3e9], [-1, 1], [4, 1], [1, -1.5]], F)
    for k in (0, 1, 2):
        v, g = S.sample(sizes, x, pts, k)
        assert np.isnan(v).all() and np.isnan(g).all()
