"""ctypes view of libfi_b200.so (include/fi_b200.h).  There is no fallback: if the shared object is missing or
a call fails, an exception is raised."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libfi_b200.so")

FI_OK, FI_ERR_INVALID, FI_ERR_CUDA, FI_ERR_RANGE, FI_ERR_UNSUPPORTED, FI_ERR_COMM = range(6)
FI_HOST, FI_DEVICE = 0, 1
FI_F32, FI_F64, FI_MIXED = 0, 1, 2
FI_PRECOND_JACOBI, FI_PRECOND_MULTIGRID = 0, 1


class FiError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"libfi_b200 status {code}: {text}")
        self.code = code


class fi_weights(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("data_pos", "data_gradient", "model_0", "model_1", "model_2", "model_3",
                                         "model_4", "gradient_smoothness")] + [("value_kernel", C.c_int32),
                                                                               ("gradient_kernel", C.c_int32)]


class fi_triplet(C.Structure):
    _fields_ = [("row", C.c_int32), ("col", C.c_int32), ("value", C.c_float)]


class fi_solve_options(C.Structure):
    _fields_ = [("precision", C.c_int32), ("max_iterations", C.c_int32), ("tolerance", C.c_double),
                ("check_every", C.c_int32), ("use_fast_stencil", C.c_int32), ("refine_max_outer", C.c_int32),
                ("refine_inner_tolerance", C.c_double), ("preconditioner", C.c_int32), ("mg_smoothing_steps", C.c_int32),
                ("mg_cheb_ratio", C.c_double)]


class fi_solve_stats(C.Structure):
    _fields_ = [("iterations", C.c_int64), ("relative_residual", C.c_double), ("true_residual", C.c_double),
                ("initial_residual", C.c_double), ("setup_ms", C.c_double), ("solve_ms", C.c_double),
                ("converged", C.c_int32), ("outer_sweeps", C.c_int32), ("occupied_cells", C.c_int64),
                ("generic_rows", C.c_int64), ("widened_after", C.c_int64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class fi_cascade_options(C.Structure):
    _fields_ = [("fine", fi_solve_options), ("factor", C.c_int32), ("coarsest_size", C.c_int32),
                ("coarse_tolerance", C.c_double), ("max_levels", C.c_int32)]


class fi_cascade_stats(C.Structure):
    _fields_ = [("levels", C.c_int32), ("level_cells", C.c_int64 * 16), ("level_iterations", C.c_int64 * 16),
                ("level_ms", C.c_double * 16), ("level_initial_residual", C.c_double * 16), ("total_ms", C.c_double),
                ("cell_iterations", C.c_int64), ("finest", fi_solve_stats)]

    def as_dict(self):
        L = self.levels
        return {"levels": L, "level_cells": list(self.level_cells[:L]), "level_iterations": list(self.level_iterations[:L]),
                "level_ms": list(self.level_ms[:L]), "level_initial_residual": list(self.level_initial_residual[:L]),
                "total_ms": self.total_ms, "cell_iterations": self.cell_iterations, "finest": self.finest.as_dict()}


FI_MG_MAX_LEVELS = 20
FI_MG_CYCLE, FI_MG_OPERATOR, FI_MG_RESTRICT, FI_MG_PROLONG_ADD, FI_MG_SMOOTH, FI_MG_COARSE = range(6)


class fi_mg_info(C.Structure):
    _fields_ = [("levels", C.c_int32), ("sizes", (C.c_int32 * 3) * FI_MG_MAX_LEVELS), ("lmax", C.c_double * FI_MG_MAX_LEVELS),
                ("nu", C.c_int32), ("nu_coarse", C.c_int32), ("gamma", C.c_int32), ("w_levels", C.c_int32),
                ("cheb_ratio", C.c_double), ("tail_from", C.c_int32), ("coarsest", C.c_int32)]

    def as_dict(self):
        L = self.levels
        return {"levels": L, "sizes": [list(self.sizes[l]) for l in range(L)], "lmax": list(self.lmax[:L]), "nu": self.nu,
                "nu_coarse": self.nu_coarse, "gamma": self.gamma, "w_levels": self.w_levels, "cheb_ratio": self.cheb_ratio,
                "tail_from": self.tail_from, "coarsest": self.coarsest}


_p = C.POINTER
_vp, _i32, _i64, _f, _d = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double
_pf, _pi32, _pi64, _pd = _p(C.c_float), _p(C.c_int32), _p(C.c_int64), _p(C.c_double)

# name -> (restype, argtypes); every symbol include/fi_b200.h declares
SIGNATURES = {
    "fi_abi_version": (C.c_int, []),
    "fi_last_error": (C.c_char_p, []),
    "fi_device_count": (C.c_int, [_pi32]),
    "fi_set_device": (C.c_int, [_i32]),
    "fi_weights_default": (None, [_p(fi_weights)]),
    "fi_solve_options_default": (None, [_p(fi_solve_options)]),
    "fi_field_create": (C.c_int, [_i32, _pi32, _p(_vp)]),
    "fi_field_destroy": (C.c_int, [_vp]),
    "fi_field_clone": (C.c_int, [_vp, _p(_vp)]),
    "fi_field_add_model": (C.c_int, [_vp, _p(fi_weights)]),
    "fi_field_add_points": (C.c_int, [_vp, _f, _i32, _f, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _pi64]),
    "fi_field_add_border_distance": (C.c_int, [_vp, _f, _i64, _vp, _i32, _pi64]),
    "fi_field_add_rows": (C.c_int, [_vp, _i64, _i64, _pi32, _pi32, _pf, _pf]),
    "fi_sdf_from_points": (C.c_int, [_i32, _pi32, _p(fi_weights), _i64, _vp, _vp, _vp, _i32, _p(_vp)]),
    "fi_field_counts": (C.c_int, [_vp, _pi64, _pi64]),
    "fi_field_export": (C.c_int, [_vp, _vp, _vp]),
    "fi_field_export_rows": (C.c_int, [_vp, _i64, _vp, _vp]),
    "fi_field_apply": (C.c_int, [_vp, _i32, _vp, _vp]),
    "fi_field_use_fast_stencil": (C.c_int, [_vp, _i32]),
    "fi_field_rhs": (C.c_int, [_vp, _i32, _vp]),
    "fi_field_diagonal": (C.c_int, [_vp, _i32, _vp]),
    "fi_field_solve": (C.c_int, [_vp, _p(fi_solve_options), _vp, _vp, _i32, _p(fi_solve_stats)]),
    "fi_field_solve_tiled": (C.c_int, [_vp, _p(fi_solve_options), _i32, _i32, _i32, _vp, _vp, _i32, _p(fi_solve_stats), _p(fi_solve_stats)]),
    "fi_field_jacobi": (C.c_int, [_vp, _pf, _i32, _f, _pf]),
    "fi_upscale_field": (C.c_int, [_i32, _pi32, _pi32, _vp, _vp, _i32]),
    "fi_error_map": (C.c_int, [_i64, _vp, _i64, _pf, _i64, _pf, _pf]),
    "fi_field_error_map": (C.c_int, [_vp, _vp, _i32, _vp, _pd]),
    "fi_marching_squares": (C.c_int, [_i32, _i32, _vp, _f, _i32, _vp, _i64, _pi64, _pf]),
    "fi_calc_area": (C.c_int, [_i64, _vp, _i32, _pf]),
    "fi_bicubic_upsample": (C.c_int, [_i32, _i32, _vp, _i32, _vp, _i32]),
    "fi_marching_cubes": (C.c_int, [_pi32, _vp, _f, _i32, _vp, _vp, _i64, _vp, _i64, _pi64, _pi64]),
    "fi_sample_field": (C.c_int, [_i32, _pi32, _vp, _i64, _vp, _i32, _i32, _vp, _vp]),
    "fi_nearest_point_distance": (C.c_int, [_i32, _i64, _vp, _i64, _vp, _i32, _vp, _vp]),
    "fi_sdf_solve_cascade": (C.c_int, [_i32, _pi32, _p(fi_weights), _i64, _vp, _vp, _vp, _p(fi_cascade_options), _vp, _i32,
                                       _p(fi_cascade_stats)]),
    "fi_comm_unique_id": (C.c_int, [_vp, _i64]),
    "fi_comm_create": (C.c_int, [_i32, _i32, _vp, _p(_vp)]),
    "fi_comm_destroy": (C.c_int, [_vp]),
    "fi_slab_balanced_cuts": (C.c_int, [_pi32, _i32, _i64, _vp, _i32, _d, _i32, _pi32]),
    "fi_comm_set_slab_cuts": (C.c_int, [_vp, _i32, _pi32]),
    "fi_slab_range": (C.c_int, [_i32, _i32, _i32, _pi32, _pi32]),
    "fi_slab_mg_plan": (C.c_int, [_pi32, _i32, _i32, _i64, _pi32, _pi32, _pi32, _pi32]),
    "fi_slab_sdf_solve": (C.c_int, [_vp, _pi32, _p(fi_weights), _i64, _vp, _vp, _vp, _i32, _p(fi_solve_options), _vp, _vp, _i32,
                                    _p(fi_solve_stats)]),
    "fi_trim_memory": (C.c_int, []),
    "fi_cached_bytes": (_i64, []),
    "fi_kernel_launches": (_i64, []),
    "fi_kernel_launches_reset": (None, []),
    "fi_field_time_iterations": (C.c_int, [_vp, _p(fi_solve_options), _i32, _pd]),
    "fi_field_mg_info": (C.c_int, [_vp, _p(fi_solve_options), _p(fi_mg_info)]),
    "fi_field_mg_stage": (C.c_int, [_vp, _p(fi_solve_options), _i32, _i32, _i64, _vp, _vp, _vp]),
}

_dll = None


def lib():
    """Loads libfi_b200.so (once).  Raises if it has not been built — there is no CPU path to fall back to."""
    global _dll
    if _dll is None:
        if not os.path.exists(LIB_PATH):
            raise FiError(FI_ERR_CUDA, f"{LIB_PATH} not built; run python -m field_interpolation_b200.build "
                                       "(or __graft_entry__.build())")
        dll = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(dll, name)
            fn.restype, fn.argtypes = res, args
        _dll = dll
    return _dll


def check(status):
    if status != FI_OK:
        raise FiError(status, lib().fi_last_error().decode("utf-8", "replace"))
