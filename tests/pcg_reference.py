"""TEST INFRASTRUCTURE — fp64 restatement of one Jacobi-PCG iteration of csrc/solver.cu, matrix-free.

Written from the model definition and the recurrence the solver's header comment states, not from the kernels:

* smoothness part S: per add_model call and axis d, sum over active orders k of D_k^T D_k, D_k the order-k difference
  rows (field_interpolation.cpp:243-316: rows j = 0 .. n-k-1 touch nodes j .. j+k; rows that would stick out of the
  lattice do not exist) with the coefficients the reference stores, float32(binomial * w_k) (DESIGN.md §4), plus the
  gradient-smoothness cross terms 2 w_gs^2 sum over axis pairs d < o of (D_1^T D_1)_d (x) (D_1^T D_1)_o (:303-315).
  Applied axis by axis, z slab by z slab (R halo planes), so that 512^3 fits in host memory.  |S| |p| is formed the
  same way from |D_k|^T |D_k| (an upper bound of the true |S| |p|, which is what a rounding bound needs);
* data term P = A_pts^T A_pts, A_pts the point and caller rows of the field exported by fi_field_export_rows from the
  row count after add_model (bit-exact, pinned to the reference by the oracle tests);
* the Jacobi preconditioner: 1 / diag(S + P), 1 where the diagonal is 0;
* the scalar recurrence init -> beta -> p -> q -> alpha -> r -> rho, rr -> done / breakdown / iters of pcg_init_kernel,
  the fused kernels and the update kernels, as plain Python.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

BINOM = [[1], [-1, 1], [1, -2, 1], [1, -3, 3, -1], [1, -4, 6, -4, 1]]
WDEF = dict(model_0=0.0, model_1=0.0, model_2=0.5, model_3=0.0, model_4=0.0, gradient_smoothness=0.0)


def _diff_rows(n, k, coef):
    """(n-k) x n order-k difference rows with coefficients `coef` (k + 1 values)."""
    m = n - k
    if m <= 0:
        return sp.csr_matrix((0, n))
    rows = np.repeat(np.arange(m), k + 1)
    cols = (np.arange(m)[:, None] + np.arange(k + 1)[None, :]).ravel()
    vals = np.tile(np.asarray(coef, np.float64), m)
    return sp.csr_matrix((vals, (rows, cols)), shape=(m, n))


def _diagonals(M, n, R):
    """{o: v} with v[i] = M[i, i + o] (0 where i + o is outside), |o| <= R."""
    M = M.tocsr()
    out = {}
    for o in range(-R, R + 1):
        d = M.diagonal(o)
        v = np.zeros(n)
        if o >= 0:
            v[:len(d)] = d
        else:
            v[-o:-o + len(d)] = d
        if np.any(v != 0):
            out[o] = v
    return out


def _apply_axis(P, ax, diags, start=0):
    """out[i] = sum_o diags[o][start + i] * P[i + o] along array axis `ax` (reads outside P are dropped)."""
    out = np.zeros_like(P)
    m = P.shape[ax]
    for o, c in diags.items():
        lo, hi = max(0, -o), min(m, m - o)
        if hi <= lo:
            continue
        shape = [1] * P.ndim
        shape[ax] = hi - lo
        so = [slice(None)] * P.ndim
        si = [slice(None)] * P.ndim
        so[ax], si[ax] = slice(lo, hi), slice(lo + o, hi + o)
        out[tuple(so)] += c[start + lo:start + hi].reshape(shape) * P[tuple(si)]
    return out


class Smoothness:
    """S of the add_model calls `models` (list of weight dicts) on a lattice of `sizes` (x first)."""

    def __init__(self, sizes, models):
        self.sizes, self.D = list(sizes), len(sizes)
        self.orders = sorted({k for w in models for k in range(5) if float(w.get(f"model_{k}", WDEF[f"model_{k}"])) > 0})
        self.gs2 = 2.0 * sum(float(np.float32(w.get("gradient_smoothness", 0.0))) ** 2 for w in models
                             if float(w.get("gradient_smoothness", 0.0)) > 0)
        self.radius = max(self.orders, default=0)
        if self.D > 1 and self.gs2 > 0:
            self.radius = max(self.radius, 1)
        R = max(self.radius, 1)
        self.T, self.Tabs, self.L, self.Labs = [], [], [], []
        for n in self.sizes:
            T = sp.csr_matrix((n, n))
            Tabs = sp.csr_matrix((n, n))
            for w in models:
                for k in range(5):
                    wk = np.float32(w.get(f"model_{k}", WDEF[f"model_{k}"]))
                    if not wk > 0:
                        continue
                    c = [float(np.float32(np.float32(b) * wk)) for b in BINOM[k]]  # fp32, as stored in the triplets
                    Dk = _diff_rows(n, k, c)
                    T = T + Dk.T @ Dk
                    Tabs = Tabs + abs(Dk).T @ abs(Dk)
            D1 = _diff_rows(n, 1, [-1.0, 1.0])
            L = D1.T @ D1
            self.T.append(_diagonals(T, n, R))
            self.Tabs.append(_diagonals(Tabs, n, R))
            self.L.append(_diagonals(L, n, 1))
            self.Labs.append(_diagonals(abs(L), n, 1))

    def diagonal(self):
        D = self.D
        diag = np.zeros(self.sizes[::-1])
        for d in range(D):
            shape = [1] * D
            shape[D - 1 - d] = self.sizes[d]
            diag = diag + self.T[d].get(0, np.zeros(self.sizes[d])).reshape(shape)
        if self.gs2 > 0:
            for d in range(D):
                for o in range(d + 1, D):
                    sd, so_ = [1] * D, [1] * D
                    sd[D - 1 - d], so_[D - 1 - o] = self.sizes[d], self.sizes[o]
                    ld = self.L[d].get(0, np.zeros(self.sizes[d]))
                    lo_ = self.L[o].get(0, np.zeros(self.sizes[o]))
                    diag = diag + self.gs2 * ld.reshape(sd) * lo_.reshape(so_)
        return diag.ravel()

    def _window(self, W, z0, absolute):
        D = self.D
        T, Lm = (self.Tabs, self.Labs) if absolute else (self.T, self.L)
        out = np.zeros_like(W)
        for d in range(D):
            out += _apply_axis(W, D - 1 - d, T[d], z0 if d == D - 1 else 0)
        if self.gs2 > 0:
            for d in range(D):
                for o in range(d + 1, D):
                    a = _apply_axis(W, D - 1 - d, Lm[d], z0 if d == D - 1 else 0)
                    out += self.gs2 * _apply_axis(a, D - 1 - o, Lm[o], z0 if o == D - 1 else 0)
        return out

    def apply(self, p, absolute=False, slab=16):
        """S p (absolute: |S| |p|) in fp64, z slab by z slab."""
        P = np.abs(np.asarray(p, np.float64)) if absolute else np.asarray(p, np.float64)
        P = P.reshape(self.sizes[::-1])
        nz, R = P.shape[0], max(self.radius, 1)
        if self.D < 3 or nz <= slab:
            return self._window(P, 0, absolute).ravel()
        out = np.empty_like(P)
        for z0 in range(0, nz, slab):
            z1 = min(nz, z0 + slab)
            lo, hi = max(0, z0 - R), min(nz, z1 + R)
            out[z0:z1] = self._window(P[lo:hi], lo, absolute)[z0 - lo:z1 - lo]
        return out.ravel()


def rows_matrix(trips, row_begin, num_rows, n):
    """A_pts (num_rows x n, fp64) from exported triplets (fields row / col / value) numbered from row_begin."""
    return sp.csr_matrix((trips["value"].astype(np.float64), (trips["row"].astype(np.int64) - row_begin, trips["col"].astype(np.int64))),
                         shape=(num_rows, n))


class Operator:
    """S + P with the Jacobi preconditioner; A_pts: scipy sparse rows of the point and caller rows."""

    def __init__(self, sizes, models, A_pts):
        self.S = Smoothness(sizes, models)
        self.A = A_pts.tocsr()
        self.Aabs = abs(self.A)
        self.n = int(np.prod(sizes))

    def data(self, p, absolute=False):
        if absolute:
            return self.Aabs.T @ (self.Aabs @ np.abs(np.asarray(p, np.float64)))
        return self.A.T @ (self.A @ np.asarray(p, np.float64))

    def apply(self, p, absolute=False):
        return self.S.apply(p, absolute) + self.data(p, absolute)

    def diagonal(self):
        return self.S.diagonal() + np.asarray(self.A.multiply(self.A).sum(axis=0)).ravel()

    def minv(self):
        d = self.diagonal()
        return np.where(d != 0, 1.0 / np.where(d != 0, d, 1.0), 1.0)

    def matrix(self):
        """S + P explicitly (small lattices): the operator applied to the unit vectors."""
        return sp.csr_matrix(np.column_stack([self.apply(np.eye(self.n)[:, k]) for k in range(self.n)]))


# ---- the scalar recurrence --------------------------------------------------------------------------------------------
def init_state(r, z, b, tol, max_iters):
    """pcg_init_kernel's state from r, z = M^-1 r and b."""
    rho, rr, bb = float(r @ z), float(r @ r), float(b @ b)
    return dict(rho=[rho, 0.0], pq=0.0, rr=rr, rr0=rr, bb=bb, tol2bb=tol * tol * bb, iters=0, max_iters=max_iters, breakdown=0,
                done=int(bb == 0.0 or rr <= tol * tol * bb or max_iters <= 0))


def beta(st, par):
    """beta of the fused direction update of an iteration of parity par (0 in iteration 0)."""
    return 0.0 if st["iters"] == 0 else st["rho"][par] / st["rho"][par ^ 1]


def finish(st, par, rho_new, rr_new):
    """The update kernels' end of an iteration (the state after r -= alpha q), in place."""
    st["rho"][par ^ 1] = rho_new
    st["rr"] = rr_new
    st["iters"] += 1
    if rr_new <= st["tol2bb"] or st["iters"] >= st["max_iters"] or not rho_new > 0.0:
        st["done"] = 1


def pcg(op, b, k, tol=1e-30, max_iters=None, x0=None):
    """k iterations (at most) of the fused iteration in fp64 from x0 (None: zero): returns x, r, p, state."""
    minv = op.minv()
    x = np.zeros(op.n) if x0 is None else np.array(x0, np.float64)
    r = b - op.apply(x) if x0 is not None else np.array(b, np.float64)
    p = minv * r
    st = init_state(r, p, b, tol, k if max_iters is None else max_iters)
    p_old = p
    for it in range(k):
        if st["done"]:
            break
        par = it & 1
        p = minv * r + beta(st, par) * p_old
        q = op.apply(p)
        st["pq"] = float(p @ q)
        if not st["pq"] > 0.0:
            st["breakdown"], st["done"] = 1, 1
            break
        alpha = st["rho"][par] / st["pq"]
        x = x + alpha * p
        r = r - alpha * q
        finish(st, par, float(r @ (minv * r)), float(r @ r))
        p_old = p
    return x, r, p_old, st
