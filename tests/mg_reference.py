"""TEST INFRASTRUCTURE — fp64 restatement of the multigrid preconditioner of csrc/mg.cu (numpy / scipy plus the port).

Written from the rules the mg.cu header comment and level_inputs() state, not from the kernels:

* levels: every axis halved with ceil until a level has at most `coarsest_cells` nodes, nothing shrinks any more, or
  the next level would have an axis (of more than one node) shorter than 4; at most 20 levels;
* A_0: the normal equations of the reference-assembled system of the field, caller rows included;
  A_l (l >= 1): the same points re-assembled by the port on the coarse lattice — positions scaled by
  float32((n_l - 1) / (n_0 - 1)) in float32, value weight unchanged, gradient weight * 0.5^l, model_k * 2^((D - 2k) l / 2),
  gradient_smoothness * 2^((D - 4) l / 2) — and no caller rows;
* P_l: upscale_field's align-corners multilinear interpolation, t = i (n_c - 1) / (n_f - 1) in double; restriction P_l^T;
* smoother: Chebyshev on D^-1 A over [lmax / cheb_ratio, lmax] with the recurrence of smooth();
* cycle: vcycle_level()'s recursion — pre-smoothing from zero, restriction of the residual, the coarse correction (a
  second one on the residual of the first for the coarse problems of levels 1 .. w_levels when gamma = 2),
  prolongation, post-smoothing; inv((A_L + A_L^T) / 2) on the coarsest level.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
import scipy.sparse as sp

from oracle import oracle as O

MAX_LEVELS = 20


@dataclass
class Problem:
    """What a field was built from: sdf_from_points(sizes, weights, pos, nrm, pw) plus caller rows add_equation(weight,
    rhs, cols, vals) on level 0."""
    sizes: List[int]
    weights: dict
    pos: np.ndarray
    nrm: Optional[np.ndarray] = None
    pw: Optional[np.ndarray] = None
    rows: list = field(default_factory=list)

    @property
    def D(self):
        return len(self.sizes)

    @property
    def n(self):
        return int(np.prod(self.sizes))


def level_sizes(sizes, coarsest_cells):
    out = [list(sizes)]
    while len(out) < MAX_LEVELS:
        f = out[-1]
        c = [(s + 1) // 2 for s in f]
        shrunk = any(a < b for a, b in zip(c, f))
        smallest = min([cc for cc, ff in zip(c, f) if ff > 1], default=1 << 30)
        if int(np.prod(f)) <= coarsest_cells or not shrunk or smallest < 4:
            break
        out.append(c)
    return out


def _weights(prob: Problem, level: int):
    w = dict(prob.weights)
    D = prob.D
    if level > 0:
        for k in range(5):
            key = f"model_{k}"
            w[key] = float(w.get(key, 0.5 if k == 2 else 0.0)) * 2.0 ** ((D - 2 * k) * level / 2.0)
        w["gradient_smoothness"] = float(w.get("gradient_smoothness", 0.0)) * 2.0 ** ((D - 4) * level / 2.0)
        w["data_gradient"] = float(w.get("data_gradient", 1.0)) * 0.5 ** level
    return O.make_weights(**w)


def level_system(port, prob: Problem, sizes_l, level: int):
    """The reference-assembled rows of level `level` (the port's triplets)."""
    pos = np.ascontiguousarray(prob.pos, np.float32).reshape(-1, prob.D)
    if level > 0:
        sc = np.array([np.float32((nl - 1) / (n0 - 1)) if n0 > 1 else np.float32(0.0) for nl, n0 in zip(sizes_l, prob.sizes)],
                      np.float32)
        pos = (pos * sc).astype(np.float32)
    f = port.sdf_from_points(sizes_l, _weights(prob, level), pos, prob.nrm, prob.pw)
    if level == 0:
        for weight, rhs, cols, vals in prob.rows:
            f.add_equation(weight, rhs, cols, vals)
    return f.system()


def level_operator(port, prob: Problem, sizes_l, level: int):
    sys_ = level_system(port, prob, sizes_l, level)
    A, _ = O.normal_equations_f64(sys_, int(np.prod(sizes_l)))
    return A.tocsr()


def axis_interpolation(nf: int, nc: int):
    """(nf x nc) align-corners linear interpolation of one axis."""
    sc = (nc - 1) / (nf - 1) if nf > 1 else 0.0
    rows, cols, vals = [], [], []
    for i in range(nf):
        t = i * sc
        b = min(int(t), nc - 1)
        fr = t - b
        rows.append(i), cols.append(b), vals.append(1.0 - fr)
        if fr != 0.0 and b + 1 < nc:
            rows.append(i), cols.append(b + 1), vals.append(fr)
    return sp.csr_matrix((vals, (rows, cols)), shape=(nf, nc))


def prolongation(fine_sizes, coarse_sizes):
    """P (N_f x N_c) on lattices stored x fastest."""
    P = sp.identity(1, format="csr")
    for nf, nc in zip(fine_sizes, coarse_sizes):  # x first: it ends up as the fastest (rightmost) kron factor
        P = sp.kron(axis_interpolation(nf, nc), P, format="csr")
    return P


class Hierarchy:
    """The hierarchy of one problem with the parameters the library reports (LatticeField.mg_info)."""

    def __init__(self, port, prob: Problem, info: dict):
        self.info = info
        self.sizes = [list(s[:prob.D]) for s in info["sizes"]]
        self.L = info["levels"]
        self.A = [level_operator(port, prob, self.sizes[l], l) for l in range(self.L)]
        self.P = [prolongation(self.sizes[l], self.sizes[l + 1]) for l in range(self.L - 1)]
        self.dinv = [1.0 / A.diagonal() for A in self.A]
        Ac = self.A[-1].toarray()
        self.coarse_inv = np.linalg.inv(0.5 * (Ac + Ac.T))
        self.lmax = list(info["lmax"])

    def nu(self, l):
        nc = self.info["nu_coarse"]
        return nc if (l > 0 and nc > 0) else self.info["nu"]

    def smooth(self, l, r, e=None, lmax=None):
        """e after nu(l) Chebyshev steps on A_l e = r from e (None: zero); also the residual r - A_l e."""
        A, dinv = self.A[l], self.dinv[l]
        lmax = self.lmax[l] if lmax is None else lmax
        lmin = lmax / self.info["cheb_ratio"]
        theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
        sigma = theta / delta
        if e is None:
            res = np.array(r, np.float64)
            e = np.zeros_like(res)
        else:
            e = np.array(e, np.float64)
            res = r - A @ e
        d = dinv * res / theta
        e = e + d
        rho = 1.0 / sigma
        for _ in range(1, self.nu(l)):
            rho_new = 1.0 / (2.0 * sigma - rho)
            res = res - A @ d
            d = rho_new * rho * d + 2.0 * rho_new / delta * dinv * res
            e = e + d
            rho = rho_new
        return e

    def cycle(self, r, l=0):
        if l == self.L - 1:
            return self.coarse_inv @ r
        e = self.smooth(l, r)
        rc = self.P[l].T @ (r - self.A[l] @ e)
        ec = self.cycle(rc, l + 1)
        if self.info["gamma"] > 1 and l + 1 < self.L - 1 and l + 1 <= self.info["w_levels"]:
            ec = ec + self.cycle(rc - self.A[l + 1] @ ec, l + 1)
        e = e + self.P[l] @ ec
        return self.smooth(l, r, e)

    def matrix(self):
        """B explicitly (N_0 x N_0): the cycle applied to the unit vectors."""
        n = self.A[0].shape[0]
        return np.column_stack([self.cycle(np.eye(n)[:, k]) for k in range(n)])


def pcg(A, b, precond, tol, max_iter=10000):
    """fp64 CG on A x = b from zero preconditioned by `precond`; stops once |r| <= tol |b| (the library's rule).
    Returns (x, iterations)."""
    x = np.zeros_like(b)
    r = b.copy()
    bb = float(b @ b)
    if bb == 0.0:
        return x, 0
    z = precond(r)
    p = z.copy()
    rz = float(r @ z)
    for it in range(1, max_iter + 1):
        q = A @ p
        alpha = rz / float(p @ q)
        x += alpha * p
        r -= alpha * q
        if float(r @ r) <= tol * tol * bb:
            return x, it
        z = precond(r)
        rz_new = float(r @ z)
        p = z + (rz_new / rz) * p
        rz = rz_new
    return x, max_iter
