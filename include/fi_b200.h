/* fi_b200.h — C ABI of libfi_b200.so, the B200 (sm_100a) implementation of the hot path of
 * emilk/field_interpolation: assembling and solving the sparse least-squares system that fits a
 * LatticeField to value / gradient data under the finite-difference smoothness model.
 *
 * The reference has no FFI layer; its drop-in surface is the C++ API of
 *   field_interpolation/field_interpolation.hpp:44-183  and  field_interpolation/sparse_linear.hpp:8-80
 * (paths relative to the reference tree).  The C++ mirror of those two headers shipped in
 * include/field_interpolation/ is a thin host layer over the entry points below; each entry point cites
 * the reference interface it stands in for.  Plain pointers and sizes only, 64-bit counts, every function
 * returns an int status and never throws.  There is no CPU fallback: without a CUDA device every compute
 * entry point returns FI_ERR_CUDA.
 *
 * Conventions
 *   - lattice: x fastest, index = sum coord[d]*stride[d], stride[0] = 1 (field_interpolation.hpp:104-111)
 *   - positions / normals: interleaved fp32, D floats per point (field_interpolation.hpp:160)
 *   - `loc` arguments say where caller buffers live: FI_HOST (borrowed for the call) or FI_DEVICE
 *   - rows are numbered in call order exactly as the reference numbers them (running eq.rhs.size())
 */
#ifndef FI_B200_H
#define FI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 2: + fi_marching_squares, fi_calc_area, fi_bicubic_upsample, fi_slab_balanced_cuts, fi_comm_set_slab_cuts (additions only) */
/* 4: + fi_marching_cubes (additions only) */
/* 5: + fi_sample_field (additions only) */
/* 6: + fi_field_error_map (additions only) */
#define FI_B200_ABI_VERSION 6

#if defined(__GNUC__)
#define FI_API __attribute__((visibility("default")))
#else
#define FI_API
#endif

enum fi_status {
	FI_OK              = 0,
	FI_ERR_INVALID     = 1, /* bad argument (null pointer, ndim outside 1..3, size < 1, unknown kernel enum) */
	FI_ERR_CUDA        = 2, /* CUDA runtime failure or no device; fi_last_error() has the text */
	FI_ERR_RANGE       = 3, /* result does not fit the reference's int32 Triplet view (sparse_linear.hpp:10) */
	FI_ERR_UNSUPPORTED = 4, /* feature outside the built scope (see DESIGN.md) */
	FI_ERR_COMM        = 5  /* multi-GPU communicator failure */
};

enum fi_location { FI_HOST = 0, FI_DEVICE = 1 };

/* ValueKernel / GradientKernel, field_interpolation.hpp:47-59 (same numeric values) */
enum fi_value_kernel { FI_VALUE_NEAREST_NEIGHBOR = 0, FI_VALUE_LINEAR_INTERPOLATION = 1 };
enum fi_gradient_kernel { FI_GRADIENT_NEAREST_NEIGHBOR = 0, FI_GRADIENT_CELL_EDGES = 1, FI_GRADIENT_LINEAR_INTERPOLATION = 2 };

/* Arithmetic of the solve.  FI_F32 mirrors the reference's float path (sparse_linear.cpp:186-212,392-443),
 * FI_F64 its double path (:154-184).  FI_MIXED = fp32 PCG inside fp64 iterative refinement. */
enum fi_precision { FI_F32 = 0, FI_F64 = 1, FI_MIXED = 2 };

/* Preconditioner of the CG solve.  FI_PRECOND_JACOBI = 1/diag(AtA), Eigen's DiagonalPreconditioner (what the
 * reference's BiCGSTAB uses).  FI_PRECOND_MULTIGRID = one geometric-multigrid V-cycle per iteration: the reference's
 * coarse-to-fine idea (the same problem re-assembled on coarser lattices, src/sdf_field.cpp:251-304) applied to the
 * error on every level; iteration counts stop growing with the lattice size.  The V-cycle runs in fp32; with FI_F64
 * (or FI_MIXED, the same thing here) the outer CG and its residual are fp64.  One GPU through fi_field_solve, z-slab
 * sharded through fi_slab_sdf_solve. */
enum fi_preconditioner { FI_PRECOND_JACOBI = 0, FI_PRECOND_MULTIGRID = 1 };

/* Weights, field_interpolation.hpp:75-95 (same field order and defaults; see fi_weights_default) */
typedef struct fi_weights {
	float   data_pos, data_gradient;
	float   model_0, model_1, model_2, model_3, model_4;
	float   gradient_smoothness;
	int32_t value_kernel, gradient_kernel;
} fi_weights;

/* Triplet, sparse_linear.hpp:8-15: 12 bytes, layout-identical */
typedef struct fi_triplet {
	int32_t row, col;
	float   value;
} fi_triplet;

/* SolveOptions (sparse_linear.hpp:66-73) plus what the iterative GPU path needs. */
typedef struct fi_solve_options {
	int32_t precision;      /* fi_precision */
	int32_t max_iterations; /* <= 0: 2*N, Eigen's default for its iterative solvers */
	double  tolerance;      /* stop when |r| <= tolerance*|Atb| (Eigen's rule); <= 0: epsilon of the precision */
	int32_t check_every;    /* iterations per CUDA-graph launch between convergence polls; <= 0: 32 */
	int32_t use_fast_stencil; /* 0: generic kernel only (debug / parity), 1: best specialised kernel (TMA-staged 3D kernel
	                           * when applicable, else the tiled one), 2: tiled 3D kernel without TMA */
	int32_t refine_max_outer; /* FI_MIXED: max fp64 refinement sweeps; <= 0: 20 */
	double  refine_inner_tolerance; /* FI_MIXED: relative tolerance of each inner fp32 solve; <= 0: 1e-3 */
	int32_t preconditioner;   /* fi_preconditioner.  FI_PRECOND_JACOBI is what the reference's Eigen solvers use */
	int32_t mg_smoothing_steps; /* FI_PRECOND_MULTIGRID: Chebyshev steps on the finest level before and after each coarse correction;
	                             * <= 0: by the smoothness model and the lattice — 2 on the finest level and 4 (6 inside the W-cycles
	                             * that 3D lattices from 50 M cells get on one GPU) on the coarse ones, or 5 everywhere when
	                             * model_3 / model_4 rows (6th / 8th-order stencils) are present */
	double  mg_cheb_ratio;    /* ... smoothed part of the spectrum is [lambda_max / ratio, lambda_max]; <= 0: 12 */
} fi_solve_options;

typedef struct fi_solve_stats {
	int64_t iterations;        /* CG iterations at this lattice (all refinement sweeps summed) */
	double  relative_residual; /* recurrence |r|/|Atb| at exit (what Eigen reports as error()) */
	double  true_residual;     /* |Atb - AtA x|/|Atb| recomputed from x at exit */
	double  initial_residual;  /* |Atb - AtA guess|/|Atb| */
	double  setup_ms;          /* operator build: sort, scatter, diagonal (device time) */
	double  solve_ms;          /* iteration loop (device time) */
	int32_t converged;         /* 1 if the stopping rule was met by the TRUE residual (recomputed from x), not merely by the
	                            * recurrence: an fp32 solve that stalls at its rounding floor reports 0 */
	int32_t outer_sweeps;      /* FI_MIXED: fp64 refinement sweeps.  FI_PRECOND_MULTIGRID: coarse corrections per level the solve ended
	                            * with — 1 V-cycle, 2 W-cycle (a W-cycle on which CG breaks down is demoted to V mid-solve) */
	int64_t occupied_cells;    /* cells holding at least one data row */
	int64_t generic_rows;      /* rows applied through the COO fallback */
	int64_t widened_after;     /* -1: the solve ran in the requested arithmetic throughout.  k >= 0: an FI_F32 multigrid solve
	                            * reached the fp32 rounding floor of this system (or broke down) after k iterations and was
	                            * continued from that iterate with the fp64 outer CG (FI_MIXED); `iterations` counts both */
} fi_solve_stats;

typedef struct fi_field fi_field; /* opaque: one LatticeField (field_interpolation.hpp:97-114) on one GPU */

/* ---- library -------------------------------------------------------------------------------- */
FI_API int         fi_abi_version(void);
FI_API const char* fi_last_error(void);        /* thread-local text of the last failure */
FI_API int         fi_device_count(int32_t* count);
FI_API int         fi_set_device(int32_t device);
FI_API void        fi_weights_default(fi_weights* w); /* data_pos=1, data_gradient=1, model_2=0.5, linear value, cell edges */
FI_API void        fi_solve_options_default(fi_solve_options* o);

/* ---- LatticeField lifetime ------------------------------------------------------------------ */
/* LatticeField{sizes}, field_interpolation.hpp:104-111.  1 <= ndim <= 3 (MAX_DIM, :44). */
FI_API int fi_field_create(int32_t ndim, const int32_t* sizes, fi_field** out);
FI_API int fi_field_destroy(fi_field* f);
/* Deep copy of everything a field holds (model calls, point records, caller rows).  The reference's LatticeField is a
 * plain value type (field_interpolation.hpp:97-114: `b = a` copies the triplet list); the C++ host layer clones the
 * device description the first time a copied LatticeField / LinearEquation is appended to, so the copies stay
 * independent. */
FI_API int fi_field_clone(const fi_field* f, fi_field** out);

/* ---- builders (each call appends rows after all earlier ones, like the reference) ---------- */
/* add_field_constraints, field_interpolation.cpp:326-341 (+ add_model_constraint :243-316). */
FI_API int fi_field_add_model(fi_field* f, const fi_weights* w);

/* add_points, field_interpolation.cpp:343-371.  `values` (nullable) is the per-point f(pos) of
 * add_value_constraint (:57-80); add_points itself always uses 0.  normals / point_weights / values may be
 * null.  rows_added (nullable) receives the number of equations appended.  A single-point batch is
 * add_value_constraint / add_value_constraint_nearest_neighbor (:82-107) / add_gradient_constraint
 * (:123-240): pass value_weight or gradient_weight = 0 to leave that part out. */
FI_API int fi_field_add_points(fi_field* f, float value_weight, int32_t value_kernel, float gradient_weight,
                        int32_t gradient_kernel, int64_t num_points, const float* positions, const float* normals,
                        const float* point_weights, const float* values, int32_t loc, int64_t* rows_added);

/* Rows appended by the caller with add_equation (sparse_linear.cpp:34-50), already weighted, as COO:
 * trip_row in [0,num_rows) non-decreasing, trip_col in [0,N).  Host buffers. */
FI_API int fi_field_add_rows(fi_field* f, int64_t num_rows, int64_t num_triplets, const int32_t* trip_row,
                      const int32_t* trip_col, const float* trip_val, const float* rhs);

/* sdf_from_points, field_interpolation.cpp:373-400 = create + add_model + add_points. */
FI_API int fi_sdf_from_points(int32_t ndim, const int32_t* sizes, const fi_weights* w, int64_t num_points,
                       const float* positions, const float* normals, const float* point_weights, int32_t loc,
                       fi_field** out);

/* ---- the triplet view (LinearEquation, sparse_linear.hpp:18-22) ------------------------------ */
FI_API int fi_field_counts(fi_field* f, int64_t* num_rows, int64_t* num_triplets);
/* Writes eq.triplets / eq.rhs bit-identical to the reference's.  Host buffers sized by fi_field_counts.
 * FI_ERR_RANGE when rows or triplets exceed INT32_MAX (the reference's int row overflows there). */
FI_API int fi_field_export(fi_field* f, fi_triplet* triplets, float* rhs);
/* The same for the rows numbered >= row_begin only (row numbers stay absolute), so that a host mirror of
 * LatticeField::eq can append what one builder call added.  row_begin must be the row count before some
 * builder call.  Buffers sized by the difference of two fi_field_counts results. */
FI_API int fi_field_export_rows(fi_field* f, int64_t row_begin, fi_triplet* triplets, float* rhs);

/* ---- normal equations, matrix-free ----------------------------------------------------------- */
/* y = (AtA) x, Atb and diag(AtA) of everything added so far; make_square / Atb, sparse_linear.cpp:105-113,
 * :120.  x, y: N elements of float (FI_F32) or double (FI_F64), host buffers. */
FI_API int fi_field_apply(fi_field* f, int32_t precision, const void* x, void* y);
/* Selects the kernel fi_field_apply uses for the smoothness part: 1 (default) best specialised kernel where
 * applicable (TMA-staged), 2 the tiled kernel without TMA, 0 the generic reference-shaped kernel.
 * fi_field_solve takes the same switch in its options. */
FI_API int fi_field_use_fast_stencil(fi_field* f, int32_t enable);
FI_API int fi_field_rhs(fi_field* f, int32_t precision, void* atb);
FI_API int fi_field_diagonal(fi_field* f, int32_t precision, void* diag);

/* ---- solvers ---------------------------------------------------------------------------------- */
/* Jacobi-preconditioned CG on the normal equations with Eigen's stopping rule.  Stands in for
 * solve_sparse_linear_exact / _fast (sparse_linear.cpp:115-184: pass FI_F64 and a tight tolerance),
 * solve_sparse_linear_with_guess (:186-212) and the CG phase of solve_tiled_with_guess (:392-443).
 * guess: N floats or null (zeros).  solution: N floats; with loc = FI_DEVICE both must be 16-byte aligned (the kernels
 * access them in 16-byte packs; FI_ERR_INVALID otherwise).  Non-convergence is not an error (Eigen returns the last
 * iterate too); stats->converged says which. */
FI_API int fi_field_solve(fi_field* f, const fi_solve_options* opt, const float* guess, float* solution, int32_t loc,
                   fi_solve_stats* stats);

/* solve_tiled_with_guess, sparse_linear.cpp:392-443, with the fields of SolveOptions (sparse_linear.hpp:66-73) as
 * arguments: when tile != 0 the guess is first replaced by the tile-by-tile solution of tile_solver_square (:246-390
 * — tile_size^D tiles; couplings between tiles moved to the right-hand side with the guess, applied twice as the
 * reference does; 1e-6 diagonal regularisation; tiles without any entry keep the guess), then, when cg != 0, the CG
 * phase runs from there with opt's max_iterations / tolerance (fi_field_solve).  The tile systems are solved by
 * Jacobi-PCG on the block-diagonal matrix, all tiles at once, to a relative residual of 1e-6 (FI_F32) or 1e-12
 * (FI_F64 / FI_MIXED) in place of the reference's per-tile Cholesky.  guess is required (the reference returns an
 * empty vector for an incomplete guess); stats (CG phase) and tile_stats (tile phase) are nullable. */
FI_API int fi_field_solve_tiled(fi_field* f, const fi_solve_options* opt, int32_t tile, int32_t tile_size, int32_t cg,
                         const float* guess, float* solution, int32_t loc, fi_solve_stats* stats, fi_solve_stats* tile_stats);

/* jacobi_iterations, sparse_linear.cpp:214-241: x <- w*(Atb - R x)/D + (1-w)*x, fp32. Host buffers. */
FI_API int fi_field_jacobi(fi_field* f, const float* guess, int32_t num_iterations, float weight, float* solution);

/* upscale_field, field_interpolation.cpp:431-485 (bit-identical fp32 arithmetic). */
FI_API int fi_upscale_field(int32_t ndim, const int32_t* small_sizes, const int32_t* large_sizes, const float* small_field,
                     float* large_field, int32_t loc);

/* generate_error_map, field_interpolation.cpp:402-429: (A x - b)^2 per row, distributed over the row's columns
 * by squared coefficient.  Any triplet list (rows need not be grouped).  Host buffers; heatmap: num_columns floats. */
FI_API int fi_error_map(int64_t num_triplets, const fi_triplet* triplets, int64_t num_columns, const float* solution,
                 int64_t num_rows, const float* rhs, float* heatmap);

/* generate_error_map of the field's own system, computed on the device from what the field holds (no triplet list,
 * no O(rows) host buffer; deferred fields and systems beyond fi_field_export's int32 limits included).
 * heatmap (N floats) is bit-identical to generate_error_map (field_interpolation.cpp:402-429) applied to the triplets
 * and rhs fi_field_export would write for f, for every mix and order of builder calls and for clones:
 *   per row, err = rhs; err -= x[col] * v and sq += v * v in triplet order; then err *= err;
 *   then out[col] += (v * v) / sq * err in global triplet order, skipped where sq == 0
 * (fp32, no FMA contraction; NaN in the solution propagates as that arithmetic propagates it).
 * row_error_sums (nullable, 3 doubles) receives sum over rows of err^2 — err the fp32 row error above, squared and
 * summed in fp64 — split into [0] model rows, [1] point rows, [2] caller rows: the least-squares objective the solve
 * minimises, by term.  The sums are reduced in a fixed order and repeat bit for bit from run to run.
 * solution and heatmap live where `loc` says; device buffers need 4-byte alignment only.  A field without rows gives
 * zeros.  FI_ERR_INVALID: null f, solution or heatmap, an unknown loc.  FI_ERR_RANGE: point or caller rows on a
 * lattice of more than 2^31 - 1 nodes (their columns are int32, as in the triplet view). */
FI_API int fi_field_error_map(fi_field* f, const float* solution /* N */, int32_t loc, float* heatmap /* N */,
                              double* row_error_sums /* nullable, 3 */);

/* ---- iso-surface helpers of the callers (SURVEY.md 8f rank 4): what the demo runs on every solved 2D field -------- */
/* emilib::marching_squares (third_party/emilib/emilib/marching_squares.cpp:11-134) of `values - iso` — iso_surface,
 * src/sdf_field.cpp:605-614; iso = 0 is marching_squares itself.  values: row-major width x height floats, >= 0 means
 * "outside".  Segments come out in the reference's order (cells y-major, one or two directed segments x0 y0 x1 y1 per
 * crossed cell) and are bit-identical to the reference's.  *num_segments always receives the count.  lines (nullable:
 * count only) must hold capacity_segments * 4 floats; when the count exceeds the capacity nothing is written and the
 * call returns FI_ERR_RANGE.  area (nullable) receives emilib::calc_area of the segments (:136-150).  values and lines
 * live where `loc` says (a device `lines` buffer must be 16-byte aligned). */
FI_API int fi_marching_squares(int32_t width, int32_t height, const float* values, float iso, int32_t loc, float* lines,
                        int64_t capacity_segments, int64_t* num_segments, float* area);
/* emilib::calc_area, marching_squares.cpp:136-150: half the shoelace sum over the segments (double accumulation). */
FI_API int fi_calc_area(int64_t num_segments, const float* lines, int32_t loc, float* area);
/* bicubic_upsample, src/sdf_field.cpp:555-603: Catmull-Rom upsampling of a width x height field to
 * (upsample * width - upsample + 1) x (upsample * height - upsample + 1), clamped reads at the border; upsample >= 2
 * (the reference CHECKs > 1).  Bit-identical fp32 arithmetic. */
FI_API int fi_bicubic_upsample(int32_t width, int32_t height, const float* values, int32_t upsample, float* large, int32_t loc);
/* Triangle mesh of the surface values == iso of a 3D lattice (x fastest), in lattice coordinates.
 * sizes: nx, ny, nz.  A node is outside when value - iso >= 0 (-0.0 and exact zeros included), as in marching squares.
 * Vertices: one per lattice edge whose two end nodes lie on different sides, numbered by (lower end node's linear index,
 * then axis x < y < z); the coordinate along the edge is float(coord_lo) + a / (a - b) with a, b = the lower and upper
 * end's value - iso, the other two are the node's.  Normals (optional): the central-difference gradient of the values
 * (one-sided at the border) at both ends, interpolated with t = a / (a - b) and normalised (zero stays zero); they
 * point toward increasing values.  Triangles: three int32 vertex indices each, in cell order (cell = its lowest node)
 * and case-table order within a cell, wound so that (P1 - P0) x (P2 - P0) points to the outside side.  Each cell
 * face is resolved from its own four corners the way fi_marching_squares resolves a saddle, so the mesh is crack-free
 * and its cross-section on every lattice face is that plane's marching-squares contour.  Deterministic.
 * *num_vertices and *num_triangles always receive the counts.  vertices / normals (3 floats per vertex) and triangles
 * are nullable (all null: count only); when a count exceeds its capacity nothing is written and the call returns
 * FI_ERR_RANGE.  values and all outputs live where `loc` says (device outputs need 4-byte alignment only).  Any size
 * < 2 gives an empty mesh; more than 2^31 - 1 nodes or vertices: FI_ERR_RANGE. */
FI_API int fi_marching_cubes(const int32_t* sizes /* 3 */, const float* values, float iso, int32_t loc,
                             float* vertices /* 3 per vertex, nullable */, float* normals /* 3 per vertex, nullable */,
                             int64_t capacity_vertices, int32_t* triangles /* 3 per triangle, nullable */,
                             int64_t capacity_triangles, int64_t* num_vertices, int64_t* num_triangles);
/* Value and, optionally, gradient of a lattice field (x fastest) at arbitrary points, as the reference's constraint
 * rows measure them (field_interpolation.cpp:57-80, :123-240).  positions: D interleaved floats per point in lattice
 * coordinates, as fi_field_add_points takes them.  Outputs are in caller order, each the fp32 expression below with no
 * FMA contraction:
 *   value      upscale_field's expression (:431-485) at p: over the in-lattice corners of cell floor(p), in ascending
 *              corner order, wsum = sum k and fsum = sum k * x sequentially, then fsum / wsum.  This is what a
 *              linear-interpolation value row sees (coefficients k * w, rhs w * sum k * value); it is defined on
 *              (-1, n_d) per axis, partly outside cells use the normalised partial sum, and where wsum == 0 (no row)
 *              the value is NaN, not the 0 that fi_upscale_field writes.
 *   gradient   (gradients != null) what an add_gradient_constraint(p, ., weight 1, gradient_kernel) row measures:
 *              FI_GRADIENT_NEAREST_NEIGHBOR      x[cell + s_d] - x[cell], cell = floor(p);
 *              FI_GRADIENT_CELL_EDGES            acc = acc + (+-2 / 2^D) * x[corner] over the cell's corners in
 *                                                order, + where corner bit d is set;
 *              FI_GRADIENT_LINEAR_INTERPOLATION  the corners of floor(p - 0.5) with c + 1 < n_d, weights k:
 *                                                acc = acc + (-k) * x[i], acc = acc + k * x[i + s_d] per corner in
 *                                                order, then acc / sum k.
 *              NaN in every component where the reference emits no row: kernels 0 and 1 when the cell is not
 *              entirely inside, kernel 2 when no corner is kept or the kept weights sum to 0.
 * NaN or infinite positions, and positions outside the lattice (however far), give NaN outputs.  The
 * nearest-neighbour value kernel (:82-107) is not offered: its prediction depends on each point's normal.
 * field, positions, values (nullable) and gradients (D per point, nullable) live where `loc` says; device buffers need
 * 4-byte alignment only.  num_points == 0 is a no-op.  FI_ERR_INVALID: ndim outside 1..3, a size < 1, an unknown loc,
 * a negative count, null sizes / field / positions with points present, an unknown gradient_kernel with gradients
 * != null. */
FI_API int fi_sample_field(int32_t ndim, const int32_t* sizes, const float* field, int64_t num_points,
                           const float* positions /* D per point, lattice coordinates */, int32_t gradient_kernel,
                           int32_t loc, float* values /* nullable */, float* gradients /* D per point, nullable */);

/* Coarse-to-fine solve mirroring the demo's recipe (src/sdf_field.cpp:251-304) applied recursively:
 * positions are in UNIT coordinates and are scaled per level by (size-1) as on_lattice does (:198-210);
 * each level re-assembles sdf_from_points with the same weights and unscaled normals, the coarser solution
 * is upscaled (upscale_field) and multiplied by the size ratio (:284-288), then refined by PCG.
 * Levels: sizes, ceil(sizes/factor), ... while every axis stays >= coarsest_size. */
typedef struct fi_cascade_options {
	fi_solve_options fine;     /* solve options of the finest level */
	int32_t factor;            /* downscale_factor between levels (>= 2); 0/1: no cascade (zero guess) */
	int32_t coarsest_size;     /* stop coarsening below this size; <= 0: 16 */
	double  coarse_tolerance;  /* tolerance of every level but the finest; <= 0: same as fine.tolerance */
	int32_t max_levels;        /* <= 0: unlimited */
} fi_cascade_options;

typedef struct fi_cascade_stats {
	int32_t levels;
	int64_t level_cells[16];
	int64_t level_iterations[16];
	double  level_ms[16];           /* assemble + solve per level (device time) */
	double  level_initial_residual[16];
	double  total_ms;
	int64_t cell_iterations;        /* sum over levels of cells * iterations */
	fi_solve_stats finest;
} fi_cascade_stats;

FI_API int fi_sdf_solve_cascade(int32_t ndim, const int32_t* sizes, const fi_weights* w, int64_t num_points,
                         const float* unit_positions, const float* normals, const float* point_weights,
                         const fi_cascade_options* opt, float* solution, int32_t loc, fi_cascade_stats* stats);

/* ---- multi-GPU: one process per GPU, z-slab partition of a 3D lattice (SURVEY.md 8e) ---------------------- */
/* The reference is single-process; this is the scale-out of the same solve.  Ranks share an NCCL communicator
 * created from a 128-byte id that rank 0 obtains and the caller distributes (MPI, torch.distributed, a file).
 * NCCL is loaded at run time; FI_ERR_COMM when it is missing or a collective fails. */
typedef struct fi_comm fi_comm;
FI_API int fi_comm_unique_id(void* id, int64_t capacity /* >= 128 */);
FI_API int fi_comm_create(int32_t rank, int32_t world, const void* id, fi_comm** out); /* binds the current device */
FI_API int fi_comm_destroy(fi_comm* c);
/* Planes [z0, z1) of an nz-plane lattice owned by `rank` (contiguous, balanced to one plane).  Pure host code. */
FI_API int fi_slab_range(int32_t nz, int32_t world, int32_t rank, int32_t* z0, int32_t* z1);
/* A non-uniform partition for this communicator: cuts[0] = 0 < cuts[1] < ... < cuts[world] = nz, rank k owns planes
 * [cuts[k], cuts[k+1]) of every later fi_slab_sdf_solve on an nz-plane lattice (collective in effect: every rank must set
 * the same cuts).  cuts = null: back to fi_slab_range.  The data term makes slabs unequal in cost — the occupied cells of an
 * SDF cloud cluster in a few slabs, and the slowest rank sets the pace of every iteration.  An iteration is two phases,
 * each ended by an exchange all ranks wait in: A = stencil + data term, B = the update kernel.  fi_slab_balanced_cuts
 * minimises  max_rank A + max_rank B  with  A = sum over the slab's planes of (nx ny + point_weight * points whose cell starts
 * in the plane)  and  B = 1.22 nx ny planes  (bisection over a greedy fill for every cap on the planes of a slab).
 * point_weight = the cost of one data point in lattice cells of stencil work (<= 0: 30, measured on 8 B200s:
 * profiles/r2e_trace_n8.txt), min_planes = thinnest slab allowed (>= the stencil radius; 2 x radius for multigrid).
 * Pure function of its arguments (one histogram kernel over the points): every rank computes the same cuts. */
FI_API int fi_slab_balanced_cuts(const int32_t* sizes /* 3 */, int32_t world, int64_t num_points, const float* positions, int32_t loc,
                          double point_weight, int32_t min_planes, int32_t* cuts /* world + 1 */);
FI_API int fi_comm_set_slab_cuts(fi_comm* c, int32_t nz, const int32_t* cuts /* world + 1, or null */);
/* How a FI_PRECOND_MULTIGRID slab solve shards its V-cycle over `world` ranks (pure host code, the same on every
 * rank): levels 0 .. *sharded_levels - 1 are z-slab sharded, level *sharded_levels and everything below it is
 * replicated (its restricted residual is all-gathered).  stencil_radius = highest active model order (1..4);
 * gather_cells: levels with at most this many cells are replicated (<= 0: 3,000,000).  Outputs for levels
 * l = 0 .. *sharded_levels: level_sizes[3 l + d] (room for 27 ints) and plane_ranges[2 (l world + rank) + {0, 1}] = the
 * planes [z0, z1) of level l that `rank` owns / restricts into (room for 18 * world ints).  *halo = planes stored
 * per side.  FI_ERR_UNSUPPORTED when the lattice cannot be sharded this way. */
FI_API int fi_slab_mg_plan(const int32_t* sizes /* 3 */, int32_t world, int32_t stencil_radius, int64_t gather_cells, int32_t* sharded_levels,
                    int32_t* halo, int32_t* level_sizes, int32_t* plane_ranges);
/* sdf_from_points + PCG on the slab of this rank: every rank passes the whole point cloud (positions in lattice
 * coordinates of the full lattice) and receives its owned planes ([z0, z1) of fi_slab_range, or of the cuts set with
 * fi_comm_set_slab_cuts), (z1 - z0) * nx * ny floats, in solution_own.
 * Collective: all ranks of the communicator call it together with the same arguments except the buffers.
 * guess_own (nullable) is this rank's part of the starting guess.  FI_F32 or FI_F64; star-shaped smoothness
 * (gradient_smoothness = 0), nearest / cell-edge gradient kernels.  opt->preconditioner = FI_PRECOND_MULTIGRID runs
 * the V-cycle sharded the way fi_slab_mg_plan says (halo planes by ncclSend/ncclRecv before every operator
 * application of the smoother, one all-gather of the restricted residual per V-cycle). */
FI_API int fi_slab_sdf_solve(fi_comm* c, const int32_t* sizes /* 3 */, const fi_weights* w, int64_t num_points,
                      const float* positions, const float* normals, const float* point_weights, int32_t loc,
                      const fi_solve_options* opt, const float* guess_own, float* solution_own, int32_t solution_loc,
                      fi_solve_stats* stats);

/* ---- device memory ------------------------------------------------------------------------------------------ */
/* Freed lattice-sized device blocks are cached per process for reuse (FI_B200_POOL_GB caps the cache, default 96).
 * fi_trim_memory returns the cache to the driver; fi_cached_bytes reports its size. */
FI_API int     fi_trim_memory(void);
FI_API int64_t fi_cached_bytes(void);

/* ---- instrumentation -------------------------------------------------------------------------- */
/* Number of kernels this library has launched on the calling thread's device since load (bench.py's
 * gpu_launches), and a reset. */
FI_API int64_t fi_kernel_launches(void);
FI_API void    fi_kernel_launches_reset(void);

/* Times the CG kernels of the already-built operator with CUDA events on the solver stream (device
 * milliseconds, totals over `iterations` launches), for the roofline figures:
 *   ms[0] `iterations` whole PCG iterations as fi_field_solve runs them (CUDA graph, no convergence stop)
 *   ms[1] the operator-apply kernels alone, back to back: the fused direction+stencil kernel when the solve
 *         uses it, else the stencil kernel (plus the data-term kernels)
 *   ms[2] the update kernel alone (x += a p, r -= a q, r.Mr, r.r)
 *   ms[3] the direction kernel alone (0 when it is fused into the stencil)
 *   ms[4] 1 if the fused kernel is in use, else 0
 *   ms[5] the lattice-sized stencil kernel of ms[1] alone (the dominant kernel of the roofline figure)
 *   ms[6] the data-term kernels of ms[1] alone (occupied-cell blocks + generic rows)
 * `ms` must hold 8 doubles (ms[7] is reserved, written as 0). */
FI_API int fi_field_time_iterations(fi_field* f, const fi_solve_options* opt, int32_t iterations, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* FI_B200_H */
