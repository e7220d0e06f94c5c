"""Python host layer over the C ABI, mirroring the reference's C++ API name for name
(field_interpolation/field_interpolation.hpp:44-183, field_interpolation/sparse_linear.hpp:8-80 of the
reference tree) so parity tests read like calls into the reference.  All compute happens in libfi_b200.so on
the GPU; inputs may be numpy arrays (host) or torch CUDA tensors (device pointers are passed through).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field as dc_field
from typing import Optional, Sequence

import numpy as np

from . import _lib as L
from ._lib import (FI_DEVICE, FI_F32, FI_F64, FI_HOST, FI_MIXED, FI_PRECOND_JACOBI, FI_PRECOND_MULTIGRID,  # noqa: F401
                   FiError)


class ValueKernel:  # field_interpolation.hpp:47-51
    kNearestNeighbor = 0
    kLinearInterpolation = 1


class GradientKernel:  # field_interpolation.hpp:54-59
    kNearestNeighbor = 0
    kCellEdges = 1
    kLinearInterpolation = 2


@dataclass
class Weights:  # field_interpolation.hpp:75-95, same defaults
    data_pos: float = 1.0
    data_gradient: float = 1.0
    model_0: float = 0.0
    model_1: float = 0.0
    model_2: float = 0.5
    model_3: float = 0.0
    model_4: float = 0.0
    gradient_smoothness: float = 0.0
    value_kernel: int = ValueKernel.kLinearInterpolation
    gradient_kernel: int = GradientKernel.kCellEdges

    def c(self) -> L.fi_weights:
        return L.fi_weights(self.data_pos, self.data_gradient, self.model_0, self.model_1, self.model_2, self.model_3,
                            self.model_4, self.gradient_smoothness, int(self.value_kernel), int(self.gradient_kernel))


@dataclass
class SolveOptions:  # sparse_linear.hpp:66-73
    tile: bool = False
    tile_size: int = 16
    cg: bool = True
    max_iterations: int = 0
    error_tolerance: float = 1e-3


@dataclass
class LinearEquation:  # sparse_linear.hpp:18-22, as arrays
    rows: np.ndarray
    cols: np.ndarray
    vals: np.ndarray
    rhs: np.ndarray

    @property
    def num_rows(self):
        return int(self.rhs.shape[0])

    @property
    def num_triplets(self):
        return int(self.vals.shape[0])


def _is_device(a) -> bool:
    return hasattr(a, "data_ptr") and bool(getattr(a, "is_cuda", False))


def _f32_host(a):
    return np.ascontiguousarray(a, dtype=np.float32)


class _Buf:
    """Pointer + location of a caller array; keeps the backing object alive for the call."""

    def __init__(self, a, n_expected: Optional[int] = None):
        self.keep, self.ptr, self.loc = None, None, None
        if a is None:
            return
        if _is_device(a):
            import torch
            assert a.dtype == torch.float32 and a.is_contiguous(), "device inputs must be contiguous float32"
            self.keep, self.ptr, self.loc, n = a, C.c_void_p(a.data_ptr()), FI_DEVICE, a.numel()
        else:
            h = _f32_host(a)
            self.keep, self.ptr, self.loc, n = h, C.c_void_p(h.ctypes.data), FI_HOST, h.size
        if n_expected is not None and n != n_expected:
            raise ValueError(f"expected {n_expected} floats, got {n}")


def _common_loc(bufs):
    locs = {b.loc for b in bufs if b.loc is not None}
    if len(locs) > 1:
        raise ValueError("all point arrays must live in the same place (all host or all device)")
    return locs.pop() if locs else FI_HOST


def solve_options(precision=FI_F32, max_iterations=0, tolerance=1e-3, check_every=32, use_fast_stencil=True,
                  refine_max_outer=20, refine_inner_tolerance=1e-3, preconditioner=FI_PRECOND_JACOBI, mg_smoothing_steps=0,
                  mg_cheb_ratio=12.0) -> L.fi_solve_options:
    return L.fi_solve_options(int(precision), int(max_iterations), float(tolerance), int(check_every),
                              int(use_fast_stencil), int(refine_max_outer), float(refine_inner_tolerance), int(preconditioner),
                              int(mg_smoothing_steps), float(mg_cheb_ratio))


class LatticeField:
    """field_interpolation.hpp:97-114.  `eq` is materialised on demand from the device (bit-identical to the
    reference's triplets); the solver itself never needs it."""

    def __init__(self, sizes: Sequence[int], _handle=None):
        self.sizes = [int(s) for s in sizes]
        self.strides = []
        s = 1
        for n in self.sizes:
            self.strides.append(s)
            s *= n
        self.num_unknowns = s
        if _handle is None:
            h = C.c_void_p()
            sz = (C.c_int32 * len(self.sizes))(*self.sizes)
            L.check(L.lib().fi_field_create(len(self.sizes), sz, C.byref(h)))
            _handle = h
        self._h = _handle

    def num_dim(self):
        return len(self.sizes)

    def close(self):
        if getattr(self, "_h", None):
            L.lib().fi_field_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- triplet view -------------------------------------------------------------------------
    def counts(self):
        r, t = C.c_int64(0), C.c_int64(0)
        L.check(L.lib().fi_field_counts(self._h, C.byref(r), C.byref(t)))
        return int(r.value), int(t.value)

    @property
    def eq(self) -> LinearEquation:
        nr, nt = self.counts()
        trips = np.empty(nt, dtype=np.dtype([("row", np.int32), ("col", np.int32), ("value", np.float32)]))
        rhs = np.empty(nr, np.float32)
        L.check(L.lib().fi_field_export(self._h, C.c_void_p(trips.ctypes.data), C.c_void_p(rhs.ctypes.data)))
        return LinearEquation(trips["row"].copy(), trips["col"].copy(), trips["value"].copy(), rhs)

    # ---- normal equations ---------------------------------------------------------------------
    def _vec(self, fn, precision):
        out = np.empty(self.num_unknowns, np.float32 if precision == FI_F32 else np.float64)
        L.check(fn(self._h, precision, C.c_void_p(out.ctypes.data)))
        return out

    def rhs(self, precision=FI_F64):
        return self._vec(L.lib().fi_field_rhs, precision)

    def diagonal(self, precision=FI_F64):
        return self._vec(L.lib().fi_field_diagonal, precision)

    def use_fast_stencil(self, mode):
        """0/False generic kernel, 1/True best specialised kernel (TMA-staged), 2 tiled kernel without TMA."""
        L.check(L.lib().fi_field_use_fast_stencil(self._h, int(mode)))

    def apply(self, x, precision=FI_F64):
        dt = np.float32 if precision == FI_F32 else np.float64
        xi = np.ascontiguousarray(x, dtype=dt)
        assert xi.size == self.num_unknowns
        y = np.empty_like(xi)
        L.check(L.lib().fi_field_apply(self._h, precision, C.c_void_p(xi.ctypes.data), C.c_void_p(y.ctypes.data)))
        return y

    # ---- solve ---------------------------------------------------------------------------------
    def solve(self, options: Optional[L.fi_solve_options] = None, guess=None, out=None):
        """Returns (solution, stats dict).  guess/out: numpy (host) or torch CUDA tensors (device)."""
        opt = options if options is not None else solve_options()
        g = _Buf(guess, self.num_unknowns)
        if out is None:
            if g.loc == FI_DEVICE:
                import torch
                out = torch.empty(self.num_unknowns, dtype=torch.float32, device=guess.device)
            else:
                out = np.empty(self.num_unknowns, np.float32)
        o = _Buf(out, self.num_unknowns)
        if g.loc is not None and g.loc != o.loc:
            raise ValueError("guess and out must live in the same place")
        st = L.fi_solve_stats()
        L.check(L.lib().fi_field_solve(self._h, C.byref(opt), g.ptr, o.ptr, o.loc, C.byref(st)))
        return (out if _is_device(out) else o.keep), st.as_dict()

    def time_iterations(self, iterations: int, options: Optional[L.fi_solve_options] = None):
        """Device ms (totals over `iterations` launches): whole iterations, apply kernels, update, direction; fused?"""
        opt = options if options is not None else solve_options()
        ms = (C.c_double * 8)()
        L.check(L.lib().fi_field_time_iterations(self._h, C.byref(opt), int(iterations), ms))
        return {"iteration_ms": ms[0], "apply_ms": ms[1], "update_ms": ms[2], "direction_ms": ms[3], "fused": bool(ms[4]),
                "stencil_ms": ms[5], "data_term_ms": ms[6]}


# ---- builders (field_interpolation.hpp:116-173) ------------------------------------------------------

def add_field_constraints(field: LatticeField, weights: Weights) -> None:
    w = weights.c()
    L.check(L.lib().fi_field_add_model(field._h, C.byref(w)))


def add_points(field: LatticeField, value_weight: float, value_kernel: int, gradient_weight: float, gradient_kernel: int,
               positions, normals=None, point_weights=None, values=None) -> int:
    """add_points (field_interpolation.cpp:343-371).  Returns the number of equations appended."""
    D = field.num_dim()
    p = _Buf(positions)
    n = (p.keep.numel() if p.loc == FI_DEVICE else p.keep.size) // D if p.keep is not None else 0
    nr, pw, va = _Buf(normals, n * D if normals is not None else None), _Buf(point_weights, n if point_weights is not None else None), _Buf(values, n if values is not None else None)
    loc = _common_loc([p, nr, pw, va])
    added = C.c_int64(0)
    L.check(L.lib().fi_field_add_points(field._h, float(value_weight), int(value_kernel), float(gradient_weight),
                                        int(gradient_kernel), n, p.ptr, nr.ptr, pw.ptr, va.ptr, loc, C.byref(added)))
    return int(added.value)


def add_value_constraint(field: LatticeField, pos, value: float, weight: float) -> bool:
    """field_interpolation.cpp:57-80: false when the weight is zero or no corner of the cell is inside."""
    return add_points(field, weight, ValueKernel.kLinearInterpolation, 0.0, GradientKernel.kCellEdges,
                      np.asarray(pos, np.float32).reshape(1, -1), None, None, np.asarray([value], np.float32)) > 0


def _round_half_away(x: float) -> int:
    return int(math.floor(abs(x) + 0.5) * (1 if x >= 0 else -1))


def add_value_constraint_nearest_neighbor(field: LatticeField, pos, gradient, value: float, weight: float) -> bool:
    """field_interpolation.cpp:82-107: false iff the nearest lattice point is outside (a zero weight still
    returns true there, the row is merely dropped by add_equation)."""
    p = np.asarray(pos, np.float32).reshape(-1)
    inside = all(0 <= _round_half_away(float(p[d])) < field.sizes[d] for d in range(field.num_dim()))
    if not inside:
        return False
    add_points(field, weight, ValueKernel.kNearestNeighbor, 0.0, GradientKernel.kCellEdges, p.reshape(1, -1),
               np.asarray(gradient, np.float32).reshape(1, -1), None, np.asarray([value], np.float32))
    return True


def add_gradient_constraint(field: LatticeField, pos, gradient, weight: float, kernel: int) -> bool:
    """field_interpolation.cpp:123-240."""
    if kernel not in (0, 1, 2):
        raise FiError(L.FI_ERR_INVALID, f"Unknown gradient kernel: {kernel}")  # the reference ABORTs (:238)
    return add_points(field, 0.0, ValueKernel.kLinearInterpolation, weight, kernel,
                      np.asarray(pos, np.float32).reshape(1, -1), np.asarray(gradient, np.float32).reshape(1, -1)) > 0


def add_equation(field: LatticeField, weight: float, rhs: float, pairs) -> None:
    """add_equation (sparse_linear.cpp:34-50) on field.eq: pairs = [(column, value), ...]."""
    w = np.float32(weight)
    if w == 0:
        return
    cols = [int(c) for c, v in pairs if np.float32(v) != 0]
    vals = np.array([np.float32(v) * w for c, v in pairs if np.float32(v) != 0], np.float32)
    if not cols:
        return
    r = np.zeros(len(cols), np.int32)
    c = np.asarray(cols, np.int32)
    b = np.array([np.float32(rhs) * w], np.float32)
    L.check(L.lib().fi_field_add_rows(field._h, 1, len(cols), r.ctypes.data_as(L._pi32), c.ctypes.data_as(L._pi32),
                                      vals.ctypes.data_as(L._pf), b.ctypes.data_as(L._pf)))


def add_rows(field: LatticeField, trip_row, trip_col, trip_val, rhs) -> None:
    """Bulk form of add_equation: already-weighted COO rows."""
    r, c = np.ascontiguousarray(trip_row, np.int32), np.ascontiguousarray(trip_col, np.int32)
    v, b = _f32_host(trip_val), _f32_host(rhs)
    L.check(L.lib().fi_field_add_rows(field._h, b.size, v.size, r.ctypes.data_as(L._pi32), c.ctypes.data_as(L._pi32),
                                      v.ctypes.data_as(L._pf), b.ctypes.data_as(L._pf)))


def sdf_from_points(sizes: Sequence[int], weights: Weights, positions, normals=None, point_weights=None) -> LatticeField:
    """field_interpolation.cpp:373-400."""
    D = len(sizes)
    p = _Buf(positions)
    if p.keep is None:
        raise FiError(L.FI_ERR_INVALID, "positions is null")  # CHECK_NOTNULL_F (:382)
    n = (p.keep.numel() if p.loc == FI_DEVICE else p.keep.size) // D
    nr, pw = _Buf(normals, n * D if normals is not None else None), _Buf(point_weights, n if point_weights is not None else None)
    loc = _common_loc([p, nr, pw])
    h = C.c_void_p()
    sz = (C.c_int32 * D)(*[int(s) for s in sizes])
    w = weights.c()
    L.check(L.lib().fi_sdf_from_points(D, sz, C.byref(w), n, p.ptr, nr.ptr, pw.ptr, loc, C.byref(h)))
    return LatticeField(sizes, _handle=h)


def upscale_field(small_field, small_sizes: Sequence[int], large_sizes: Sequence[int]):
    """field_interpolation.cpp:431-485."""
    D = len(small_sizes)
    ss, ls = (C.c_int32 * D)(*map(int, small_sizes)), (C.c_int32 * D)(*map(int, large_sizes))
    src = _Buf(small_field, int(np.prod(small_sizes, dtype=np.int64)))
    nl = int(np.prod(large_sizes, dtype=np.int64))
    if src.loc == FI_DEVICE:
        import torch
        out = torch.empty(nl, dtype=torch.float32, device=small_field.device)
        dst = C.c_void_p(out.data_ptr())
    else:
        out = np.empty(nl, np.float32)
        dst = C.c_void_p(out.ctypes.data)
    L.check(L.lib().fi_upscale_field(D, ss, ls, src.ptr, dst, src.loc))
    return out


# ---- iso-surface helpers of the callers (emilib/marching_squares.cpp, src/sdf_field.cpp:555-614) -------------------
def _field_2d(values):
    """(height, width) field as a _Buf; row-major like the reference's `width * height` arrays."""
    shape = tuple(values.shape)
    if len(shape) != 2:
        raise ValueError("a 2D (height, width) field is expected")
    if _is_device(values):
        values = values.contiguous()
    return _Buf(values, shape[0] * shape[1]), int(shape[0]), int(shape[1])


def iso_surface(values, iso: float = 0.0, want_area: bool = False):
    """iso_surface, src/sdf_field.cpp:605-614 = emilib::marching_squares (marching_squares.cpp:11-134) of `values - iso`.
    values: (height, width) numpy array or CUDA tensor.  Returns the (num_segments, 4) segments x0 y0 x1 y1 in the
    reference's order, living where `values` lives; with want_area also emilib::calc_area of them (:136-150)."""
    buf, h, w = _field_2d(values)
    n = C.c_int64(0)
    L.check(L.lib().fi_marching_squares(w, h, buf.ptr, float(iso), buf.loc, None, 0, C.byref(n), None))
    ns = int(n.value)
    area = C.c_float(0.0)
    if buf.loc == FI_DEVICE:
        import torch
        out = torch.empty((ns, 4), dtype=torch.float32, device=values.device)
        dst = C.c_void_p(out.data_ptr()) if ns else None
    else:
        out = np.empty((ns, 4), np.float32)
        dst = C.c_void_p(out.ctypes.data) if ns else None
    if ns:
        L.check(L.lib().fi_marching_squares(w, h, buf.ptr, float(iso), buf.loc, dst, ns, C.byref(n), C.byref(area) if want_area else None))
    return (out, float(area.value)) if want_area else out


def marching_squares(iso_field):
    """emilib::marching_squares, third_party/emilib/emilib/marching_squares.cpp:11-134: the contour at 0."""
    return iso_surface(iso_field, 0.0)


def calc_area(lines) -> float:
    """emilib::calc_area, marching_squares.cpp:136-150."""
    if _is_device(lines):
        lines = lines.contiguous()
    buf = _Buf(lines)
    n = (buf.keep.numel() if buf.loc == FI_DEVICE else buf.keep.size) // 4 if buf.keep is not None else 0
    area = C.c_float(0.0)
    L.check(L.lib().fi_calc_area(n, buf.ptr if n else None, buf.loc if buf.loc is not None else FI_HOST, C.byref(area)))
    return float(area.value)


def bicubic_upsample(values, upsample: int):
    """bicubic_upsample, src/sdf_field.cpp:555-603: (height, width) -> (upsample*height - upsample + 1, upsample*width - upsample + 1)."""
    buf, h, w = _field_2d(values)
    lh, lw = upsample * h - upsample + 1, upsample * w - upsample + 1
    if buf.loc == FI_DEVICE:
        import torch
        out = torch.empty((lh, lw), dtype=torch.float32, device=values.device)
        dst = C.c_void_p(out.data_ptr())
    else:
        out = np.empty((lh, lw), np.float32)
        dst = C.c_void_p(out.ctypes.data)
    L.check(L.lib().fi_bicubic_upsample(w, h, buf.ptr, int(upsample), dst, buf.loc))
    return out


def marching_cubes(values, iso: float = 0.0, want_normals: bool = False):
    """Triangle mesh of the surface `values == iso` of a 3D field (fi_marching_cubes, include/fi_b200.h).
    values: (nz, ny, nx) numpy array or contiguous CUDA tensor, e.g. the `out` of LatticeField.solve.  Returns
    (vertices (V, 3) float32 in lattice coordinates x y z, triangles (T, 3) int32[, normals (V, 3) float32]), living
    where `values` lives; triangles are wound so that (P1 - P0) x (P2 - P0) points toward values >= iso."""
    shape = tuple(values.shape)
    if len(shape) != 3:
        raise ValueError("a 3D (nz, ny, nx) field is expected")
    sizes = (C.c_int32 * 3)(int(shape[2]), int(shape[1]), int(shape[0]))
    buf = _Buf(values, shape[0] * shape[1] * shape[2])
    nv, nt = C.c_int64(0), C.c_int64(0)
    fn = L.lib().fi_marching_cubes
    L.check(fn(sizes, buf.ptr, float(iso), buf.loc, None, None, 0, None, 0, C.byref(nv), C.byref(nt)))
    V, T = int(nv.value), int(nt.value)
    if buf.loc == FI_DEVICE:
        import torch
        verts = torch.empty((V, 3), dtype=torch.float32, device=values.device)
        tris = torch.empty((T, 3), dtype=torch.int32, device=values.device)
        nrms = torch.empty((V, 3), dtype=torch.float32, device=values.device) if want_normals else None
        ptr = lambda a: C.c_void_p(a.data_ptr())  # noqa: E731
    else:
        verts, tris = np.empty((V, 3), np.float32), np.empty((T, 3), np.int32)
        nrms = np.empty((V, 3), np.float32) if want_normals else None
        ptr = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    if V:
        L.check(fn(sizes, buf.ptr, float(iso), buf.loc, ptr(verts), ptr(nrms) if want_normals else None, V, ptr(tris), T,
                   C.byref(nv), C.byref(nt)))
    return (verts, tris, nrms) if want_normals else (verts, tris)


def sample_field(field, positions, gradient_kernel=None):
    """Value (and gradient) of a lattice field at arbitrary points (fi_sample_field, include/fi_b200.h).
    field: (n,), (ny, nx) or (nz, ny, nx), numpy array or CUDA tensor; positions: (N, D) lattice coordinates, columns
    x y z, living where `field` lives.  gradient_kernel: None (values only) or a GradientKernel.  Returns values (N,)
    float32, or (values, gradients (N, D)) when a kernel is given, living where the inputs live.  Points where the
    reference would emit no row (outside the lattice, non-finite) read NaN."""
    shape = tuple(field.shape)
    D = len(shape)
    if D not in (1, 2, 3):
        raise ValueError("a (n,), (ny, nx) or (nz, ny, nx) field is expected")
    pshape = tuple(positions.shape)
    if len(pshape) != 2 or pshape[1] != D:
        raise ValueError(f"positions must be (N, {D})")
    if _is_device(field) != _is_device(positions):
        raise ValueError("field and positions must live in the same place (both host or both device)")
    if _is_device(field):
        field, positions = field.contiguous(), positions.contiguous()
    N = int(pshape[0])
    sizes = (C.c_int32 * D)(*[int(s) for s in reversed(shape)])
    fb = _Buf(field, int(np.prod(shape, dtype=np.int64)))
    pb = _Buf(positions, N * D)
    want = gradient_kernel is not None
    if fb.loc == FI_DEVICE:
        import torch
        vals = torch.empty(N, dtype=torch.float32, device=field.device)
        grads = torch.empty((N, D), dtype=torch.float32, device=field.device) if want else None
        ptr = lambda a: C.c_void_p(a.data_ptr())  # noqa: E731
    else:
        vals = np.empty(N, np.float32)
        grads = np.empty((N, D), np.float32) if want else None
        ptr = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    if N:
        L.check(L.lib().fi_sample_field(D, sizes, fb.ptr, N, pb.ptr, int(gradient_kernel) if want else 0, fb.loc, ptr(vals),
                                        ptr(grads) if want else None))
    return (vals, grads) if want else vals


def generate_error_map(field: LatticeField, solution, want_sums: bool = False):
    """generate_error_map (field_interpolation.cpp:402-429) of the field's own system (fi_field_error_map,
    include/fi_b200.h): bit-identical to the reference's function on field.eq, computed on the device without the
    triplet list.  Like the solvers, it takes the field where the reference takes field.eq.  solution: N floats,
    numpy array or CUDA tensor.  Returns the heat map (N,) float32, living where `solution` lives; with want_sums
    also the fp64 sums of err^2 over model, point and caller rows (a (3,) float64 numpy array)."""
    if _is_device(solution):
        solution = solution.contiguous()
    N = field.num_unknowns
    sol = _Buf(solution, N)
    if sol.loc == FI_DEVICE:
        import torch
        heat = torch.empty(N, dtype=torch.float32, device=solution.device)
        dst = C.c_void_p(heat.data_ptr())
    else:
        heat = np.empty(N, np.float32)
        dst = C.c_void_p(heat.ctypes.data)
    sums = (C.c_double * 3)()
    L.check(L.lib().fi_field_error_map(field._h, sol.ptr, sol.loc, dst, sums))
    return (heat, np.array(sums[:], np.float64)) if want_sums else heat


# ---- solvers (sparse_linear.hpp:44-80), on a LatticeField ---------------------------------------------
# The reference passes field.eq; here the field itself carries the structure (a bare triplet list has lost the
# lattice).  A failed solve returns an empty array like the reference returns {}.

def _solve(field, opt, guess=None):
    try:
        x, st = field.solve(opt, guess)
        return x, st
    except FiError:
        return np.zeros(0, np.float32), {}


def solve_sparse_linear_exact(field: LatticeField, num_columns: Optional[int] = None, tolerance: float = 1e-12):
    """sparse_linear.cpp:154-184 (double Cholesky) -> fp64 PCG driven to `tolerance`."""
    return _solve(field, solve_options(FI_F64, 0, tolerance))[0]


def solve_sparse_linear_fast(field: LatticeField, num_columns: Optional[int] = None):
    """sparse_linear.cpp:115-152 (float Cholesky).  A direct float factorisation has no iterative analogue that
    is both cheaper and as robust on these ill-conditioned systems (cond ~ n^4), so this is the fp64 PCG at a
    float-level tolerance."""
    return _solve(field, solve_options(FI_F64, 0, 1e-9))[0]


def solve_sparse_linear_with_guess(field: LatticeField, guess, max_iterations: int = 0, error_tolerance: float = 0.0):
    """sparse_linear.cpp:186-212 (float BiCGSTAB, diagonal preconditioner) -> fp32 PCG, same stopping rule."""
    return _solve(field, solve_options(FI_F32, max_iterations, error_tolerance), guess)[0]


def solve_tiled_with_guess(field: LatticeField, guess, sizes=None, options: Optional[SolveOptions] = None, precision=FI_F32,
                           return_stats: bool = False):
    """sparse_linear.cpp:392-443: optional tile phase (tile_solver_square :246-390), then the optional CG phase."""
    o = options or SolveOptions()
    g = np.ascontiguousarray(guess, np.float32).ravel()
    if g.size != field.num_unknowns:
        return np.zeros(0, np.float32)  # "Incomplete guess." (:402-405)
    out = np.empty_like(g)
    st, tst = L.fi_solve_stats(), L.fi_solve_stats()
    opt = solve_options(precision, o.max_iterations, o.error_tolerance)
    L.check(L.lib().fi_field_solve_tiled(field._h, C.byref(opt), int(bool(o.tile)), int(o.tile_size), int(bool(o.cg)),
                                         C.c_void_p(g.ctypes.data), C.c_void_p(out.ctypes.data), FI_HOST, C.byref(st), C.byref(tst)))
    return (out, st.as_dict(), tst.as_dict()) if return_stats else out


def jacobi_iterations(field: LatticeField, guess, num_iterations: int, weight: float):
    """sparse_linear.cpp:214-241."""
    g = _f32_host(guess)
    out = np.empty_like(g)
    L.check(L.lib().fi_field_jacobi(field._h, g.ctypes.data_as(L._pf), int(num_iterations), float(weight),
                                    out.ctypes.data_as(L._pf)))
    return out


def sdf_solve_cascade(sizes: Sequence[int], weights: Weights, unit_positions, normals=None, point_weights=None,
                      options: Optional[L.fi_solve_options] = None, factor: int = 2, coarsest_size: int = 16,
                      coarse_tolerance: float = 0.0, max_levels: int = 0, out=None):
    """Coarse-to-fine solve (reference recipe src/sdf_field.cpp:251-304, applied recursively)."""
    D = len(sizes)
    p = _Buf(unit_positions)
    n = (p.keep.numel() if p.loc == FI_DEVICE else p.keep.size) // D if p.keep is not None else 0
    nr, pw = _Buf(normals, n * D if normals is not None else None), _Buf(point_weights, n if point_weights is not None else None)
    loc = _common_loc([p, nr, pw])
    N = int(np.prod(sizes, dtype=np.int64))
    if out is None:
        if loc == FI_DEVICE:
            import torch
            out = torch.empty(N, dtype=torch.float32, device=unit_positions.device)
        else:
            out = np.empty(N, np.float32)
    o = _Buf(out, N)
    if o.loc != loc:
        raise ValueError("out must live where the inputs live")
    copt = L.fi_cascade_options(options if options is not None else solve_options(), int(factor), int(coarsest_size),
                                float(coarse_tolerance), int(max_levels))
    st = L.fi_cascade_stats()
    sz = (C.c_int32 * D)(*[int(s) for s in sizes])
    w = weights.c()
    L.check(L.lib().fi_sdf_solve_cascade(D, sz, C.byref(w), n, p.ptr, nr.ptr, pw.ptr, C.byref(copt), o.ptr, loc, C.byref(st)))
    return (out if _is_device(out) else o.keep), st.as_dict()


def kernel_launches() -> int:
    return int(L.lib().fi_kernel_launches())


def kernel_launches_reset() -> None:
    L.lib().fi_kernel_launches_reset()
