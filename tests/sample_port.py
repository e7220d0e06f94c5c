"""TEST INFRASTRUCTURE.  A vectorised numpy float32 restatement of fi_sample_field (include/fi_b200.h,
csrc/sample_field.cuh): the value of upscale_field's expression at each point and the gradient that each of the three
gradient rows of the reference measures.  Every fp32 operation is one numpy step in the order of the CUDA code, one
corner at a time; numpy never fuses a multiply and an add, so the result is bit-exact against the -fmad=false build."""
import numpy as np

F = np.float32
NAN = F(np.nan)
LIMIT = F(2.0 ** 31)  # |p| below this: floor(p) + 2 fits int32; every point outside the lattice is NaN anyway


def _strides(sizes):
    s, out = 1, []
    for n in sizes:
        out.append(s)
        s *= int(n)
    return out


def _corners(sizes, strides, p, margin):
    """(ok, index, weight) per corner of cell floor(p), in ascending corner order (corner_weights of assembly.cu)."""
    D = len(sizes)
    base = np.floor(p).astype(np.int64)
    frac = (p - base.astype(F)).astype(F)
    for corner in range(1 << D):
        index = np.zeros(len(p), np.int64)
        w = np.ones(len(p), F)
        ok = np.ones(len(p), bool)
        for d in range(D):
            bit = (corner >> d) & 1
            c = base[:, d] + bit
            index += strides[d] * c
            w = w * (frac[:, d] if bit else F(1) - frac[:, d])
            ok &= (0 <= c) & (c + margin < sizes[d])
        yield ok, index, w


def sample(sizes, field, positions, gradient_kernel=None):
    """sizes: (nx[, ny[, nz]]); field: x-fastest values; positions: (N, D).  Returns values, or (values, gradients)."""
    sizes = [int(n) for n in sizes]
    D = len(sizes)
    x = np.ascontiguousarray(field, F).ravel()
    p = np.ascontiguousarray(positions, F).reshape(-1, D)
    strides = _strides(sizes)
    finite = (np.abs(p) < LIMIT).all(axis=1)
    p = np.where(finite[:, None], p, F(0))
    take = lambda ok, idx: x[np.where(ok, idx, 0)]  # noqa: E731

    wsum, fsum = np.zeros(len(p), F), np.zeros(len(p), F)
    for ok, idx, k in _corners(sizes, strides, p, 0):
        xi = take(ok, idx)
        wsum = np.where(ok, wsum + k, wsum)
        fsum = np.where(ok, fsum + k * xi, fsum)
    with np.errstate(divide="ignore", invalid="ignore"):
        values = np.where(finite & (wsum != 0), fsum / wsum, NAN).astype(F)
    if gradient_kernel is None:
        return values

    grad = np.full((len(p), D), NAN, F)
    if gradient_kernel in (0, 1):
        base = np.floor(p).astype(np.int64)
        inside = finite & ((0 <= base) & (base + 1 < np.array(sizes))).all(axis=1)
        cell = np.where(inside, (base * np.array(strides)).sum(axis=1), 0)
        if gradient_kernel == 0:
            for d in range(D):
                grad[:, d] = np.where(inside, take(inside, cell + strides[d]) - take(inside, cell), NAN)
        else:
            term = F(2) / F(1 << D)
            acc = np.zeros((len(p), D), F)
            for c in range(1 << D):
                node = cell + sum(strides[a] for a in range(D) if (c >> a) & 1)
                v = take(inside, node)
                for d in range(D):
                    acc[:, d] = acc[:, d] + (term if (c >> d) & 1 else -term) * v
            grad = np.where(inside[:, None], acc, NAN).astype(F)
    elif gradient_kernel == 2:
        shifted = p - F(0.5)
        acc = np.zeros((len(p), D), F)
        ksum = np.zeros(len(p), F)
        for ok, idx, k in _corners(sizes, strides, shifted, 1):
            ksum = np.where(ok, ksum + k, ksum)
            v = take(ok, idx)
            for d in range(D):
                acc[:, d] = np.where(ok, acc[:, d] + (-k) * v, acc[:, d])
                acc[:, d] = np.where(ok, acc[:, d] + k * take(ok, idx + strides[d]), acc[:, d])
        with np.errstate(divide="ignore", invalid="ignore"):
            grad = np.where((finite & (ksum != 0))[:, None], acc / ksum[:, None], NAN).astype(F)
    else:
        raise ValueError("gradient_kernel must be 0, 1 or 2")
    return values, grad


def row_measure(system, x):
    """Sequential fp32 dot / rhs of every row, in row order."""
    out = []
    for r in range(system.num_rows):
        sel = system.rows == r
        acc = F(0)
        for c, v in zip(system.cols[sel], system.vals[sel]):
            acc = F(acc + F(v * x[c]))
        rhs = system.rhs[r]
        out.append(F(np.nan) if rhs == 0 else F(acc / rhs))
    return np.array(out, F)


def same_values(got, want):
    """Equal as fp32 values, NaN where the other is NaN."""
    got, want = np.asarray(got, F), np.asarray(want, F)
    assert got.shape == want.shape
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), (got, want)
    assert np.array_equal(got[~nan], want[~nan]), (got, want)


def reference_measures(port, sizes, x, p, kernel):
    """Value and gradient that the CPU oracle port's rows for p measure on x: NaN where no row, or a row with rhs 0."""
    D = len(sizes)
    f = port.field(sizes)
    emitted_value = f.add_value_constraint(p, 1.0, 1.0)
    nv = f.system().num_rows
    emitted_grad = f.add_gradient_constraint(p, np.ones(D, F), 1.0, kernel)
    m = row_measure(f.system(), x)
    value = m[0] if emitted_value else F(np.nan)
    grad = m[nv:nv + D] if emitted_grad else np.full(D, np.nan, F)
    assert len(m) == nv + (D if emitted_grad else 0)
    return value, grad


def positions_of_every_kind(sizes, n, seed):
    """Points inside, on integer coordinates, in the outer half-cells, just outside, far outside and non-finite,
    shuffled; (N, D) float32 with columns x y z."""
    rng = np.random.default_rng(seed)
    sizes = np.array(sizes, np.float64)
    D = len(sizes)
    parts = [
        rng.uniform(0, sizes - 1, (n, D)),                                    # inside
        np.floor(rng.uniform(0, sizes, (n // 4 + 1, D))),                     # lattice nodes
        rng.uniform(-0.5, sizes - 0.5, (n // 4 + 1, D)),                      # inside plus the outer half-cells
        rng.uniform(-1.0, sizes, (n // 4 + 1, D)),                            # the whole domain of the value
        rng.uniform(-3.0, sizes + 2, (n // 4 + 1, D)),                        # around and outside
    ]
    pts = np.concatenate(parts).astype(F)
    # integer and half-integer coordinates on single axes (the kernel-2 cell boundaries), and the border planes
    m = len(pts)
    sel = rng.random((m, D))
    pts = np.where(sel < 0.08, np.round(pts), pts)
    pts = np.where((sel >= 0.08) & (sel < 0.14), np.round(pts) + F(0.5), pts)
    pts = np.where((sel >= 0.14) & (sel < 0.17), F(-1), pts)
    pts = np.where((sel >= 0.17) & (sel < 0.20), sizes.astype(F) - F(1), pts)
    special = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30, 3e9, -3e9, 2147483520.0, -0.0, -1e-7], F)
    extra = np.tile(rng.uniform(0, sizes - 1, (1, D)).astype(F), (len(special) * D, 1))
    for i, s in enumerate(special):
        for d in range(D):
            extra[i * D + d, d] = s
    pts = np.concatenate([pts, extra]).astype(F)
    return pts[rng.permutation(len(pts))]
