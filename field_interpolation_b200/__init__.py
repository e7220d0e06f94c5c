"""field_interpolation_b200 — B200 (sm_100a) implementation of the hot path of emilk/field_interpolation:
assembling and solving the sparse least-squares system that fits a LatticeField (1D/2D/3D) to value and
gradient data under the finite-difference smoothness model.

The product is the C-ABI library ``libfi_b200.so`` (include/fi_b200.h; CUDA sources in csrc/).  This package
is its Python host layer, mirroring the reference's C++ API name for name (see api.py).  There is no CPU
fallback: importing is cheap, but every call needs the built library and a CUDA device.
"""
from .api import (FI_DEVICE, FI_F32, FI_F64, FI_HOST, FI_MIXED, FI_PRECOND_JACOBI, FI_PRECOND_MULTIGRID, FiError, GradientKernel, LatticeField, LinearEquation,
                  SolveOptions, ValueKernel, Weights, add_equation, add_field_constraints, add_gradient_constraint,
                  add_points, add_rows, add_value_constraint, add_value_constraint_nearest_neighbor, jacobi_iterations,
                  kernel_launches, kernel_launches_reset, sdf_from_points, sdf_solve_cascade, solve_options,
                  solve_sparse_linear_exact, solve_sparse_linear_fast, solve_sparse_linear_with_guess,
                  solve_tiled_with_guess, upscale_field, bicubic_upsample, calc_area, iso_surface, marching_squares,
                  marching_cubes, sample_field, generate_error_map)

__all__ = [n for n in dir() if not n.startswith("_")]
