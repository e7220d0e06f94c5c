"""Systems for the tests of fi_field_error_map: fields built from a recipe of builder calls (every model weight, every
value and gradient kernel, point weights and values, caller rows between model calls), and the fp64 row error sums of
an exported system computed with numpy from the reference's fp32 row errors."""
import ctypes as C

import numpy as np

F = np.float32
ALL_MODEL = dict(model_0=0.3, model_1=0.7, model_2=0.5, model_3=0.2, model_4=0.1, gradient_smoothness=0.4)
OTHER_MODEL = dict(model_0=0.0, model_1=0.25, model_2=0.0, model_3=0.6, model_4=0.0, gradient_smoothness=0.9)

# (value weight, value kernel, gradient weight, gradient kernel): both value kernels, all three gradient kernels
POINT_CALLS = [(1.0, 1, 0.8, 1), (0.7, 0, 1.3, 2), (1.1, 1, 0.5, 0), (0.0, 1, 1.0, 2), (0.9, 0, 0.0, 1)]


def points(sizes, n, rng):
    """Positions over [-1, size] per axis (some fall outside the lattice), unit-ish normals, weights, values."""
    D = len(sizes)
    pos = np.stack([rng.uniform(-1.0, s, n) for s in sizes], axis=1).astype(F)
    nrm = rng.normal(size=(n, D)).astype(F)
    return pos, nrm, rng.uniform(0.2, 1.5, n).astype(F), rng.normal(size=n).astype(F)


def caller_rows(N, nrows, rng):
    """COO rows of 0..4 taps each, duplicate columns included (a row with no tap adds only its rhs)."""
    r, c, v = [], [], []
    for row in range(nrows):
        for _ in range(int(rng.integers(0, 5))):
            r.append(row)
            c.append(int(rng.integers(0, N)))
            v.append(rng.normal())
    return np.asarray(r, np.int32), np.asarray(c, np.int32), np.asarray(v, F), rng.normal(size=nrows).astype(F)


def build(m, sizes, recipe, n_points=40, seed=0):
    """A field of module `m` (the package, or its emulator binding) from a recipe of "model", "model2", "points<k>"
    (k indexes POINT_CALLS) and "rows" steps.  Returns the field and the kind of each of its rows (0 model, 1 point,
    2 caller), read from the row counts between calls."""
    rng = np.random.default_rng(seed)
    f = m.LatticeField(sizes)
    N = f.num_unknowns
    kinds, before = [], 0
    for step in recipe:
        if step in ("model", "model2"):
            m.add_field_constraints(f, m.Weights(**(ALL_MODEL if step == "model" else OTHER_MODEL)))
            kind = 0
        elif step.startswith("points"):
            vw, vk, gw, gk = POINT_CALLS[int(step[6:])]
            pos, nrm, pw, val = points(sizes, n_points, rng)
            m.add_points(f, vw, vk, gw, gk, pos, nrm, pw, val)
            kind = 1
        elif step == "rows":
            m.add_rows(f, *caller_rows(N, 7, rng))
            kind = 2
        else:
            raise KeyError(step)
        now = f.counts()[0]
        kinds += [kind] * (now - before)
        before = now
    return f, np.asarray(kinds, np.int64)


def clone(m, f):
    from field_interpolation_b200 import _lib as L
    h = C.c_void_p()
    L.check(L.lib().fi_field_clone(f._h, C.byref(h)))
    return m.LatticeField(f.sizes, _handle=h)


def row_errors(eq, x):
    """The reference's fp32 row errors: err = rhs; err -= x[col] * v in triplet order (np.subtract.at is sequential)."""
    err = np.array(eq.rhs, F, copy=True)
    np.subtract.at(err, eq.rows, (np.asarray(x, F)[eq.cols] * eq.vals).astype(F))
    return err


def kind_sums(eq, x, row_kinds):
    """sum of float64(err)^2 over the rows of each kind (0 model, 1 point, 2 caller); row_kinds: one per row."""
    e = row_errors(eq, x).astype(np.float64) ** 2
    return np.array([e[row_kinds == k].sum() for k in range(3)])
