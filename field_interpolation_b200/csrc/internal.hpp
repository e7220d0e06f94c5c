// Internal interfaces between the translation units of libfi_b200 (not installed).
#pragma once

#include <memory>

#include "common.cuh"

namespace fi {

struct Geom  // LatticeField geometry, reference field_interpolation.hpp:97-114 (x fastest)
{
	int     ndim = 0;
	int     size[kMaxDim]   = {1, 1, 1};   // the whole lattice (also when this process holds one z slab of it)
	int64_t stride[kMaxDim] = {1, 1, 1};
	int64_t N = 1;                         // cells stored locally = nx * ny * nzl
	// z-slab window (multi-GPU, dist.cu).  Local plane l holds lattice plane l + zoff; planes whose lattice z
	// falls outside [0, size[2]) exist in memory but stay zero.  Unsharded: zoff = 0, nzl = size[2].
	int     zoff = 0;
	int     nzl = 1;                       // planes stored locally
	int     zown0 = 0, zown1 = 1;          // local planes this process owns (computes rows for): [zown0, zown1)
	int64_t shift = 0;                     // = -stride[2] * zoff: local index = sum coord[d] * stride[d] + shift
	// Tile mode (tile_solver_square, reference sparse_linear.cpp:246-390): with tile >= 2 the operator kernels drop
	// every entry (i, j) of A^T A whose nodes lie in different tile^D tiles and add tile_reg to the diagonal
	// (:306-309), i.e. they apply the block-diagonal matrix the reference factorises tile by tile.  Unsharded only.
	int     tile = 0;
	float   tile_reg = 0.0f;

	__host__ __device__ bool sharded() const { return zown0 != 0 || zown1 != nzl; }
	__host__ __device__ int64_t own_offset() const { return static_cast<int64_t>(zown0) * (ndim == 3 ? stride[2] : 0); }
	__host__ __device__ int64_t own_cells() const { return ndim == 3 ? static_cast<int64_t>(zown1 - zown0) * stride[2] : N; }
};

// Linear tile number of unsharded lattice node `index` (x fastest over ceil(size / tile) tiles per axis).
__host__ __device__ inline int64_t tile_of_node(const Geom& g, int64_t index)
{
	int64_t t = 0, ts = 1;
	for (int d = 0; d < g.ndim; ++d) {
		const int c = static_cast<int>(index % g.size[d]);
		index /= g.size[d];
		t += static_cast<int64_t>(c / g.tile) * ts;
		ts *= (g.size[d] + g.tile - 1) / g.tile;
	}
	return t;
}

inline Geom make_geom(int ndim, const int32_t* sizes)
{
	Geom g;
	g.ndim    = ndim;
	int64_t s = 1;
	for (int d = 0; d < ndim; ++d) {
		g.size[d]   = sizes[d];
		g.stride[d] = s;
		s *= sizes[d];
	}
	g.N = s;
	g.nzl   = ndim == 3 ? sizes[2] : 1;
	g.zown1 = g.nzl;
	return g;
}

// The slab of lattice planes [z0, z1) with `halo` planes stored on either side (3D only).
inline Geom make_slab_geom(const int32_t* sizes, int z0, int z1, int halo)
{
	Geom g  = make_geom(3, sizes);
	g.zoff  = z0 - halo;
	g.nzl   = (z1 - z0) + 2 * halo;
	g.zown0 = halo;
	g.zown1 = halo + (z1 - z0);
	g.shift = -g.stride[2] * g.zoff;
	g.N     = g.stride[2] * g.nzl;
	return g;
}

// Canonical per-point records, appended by every add_points call (struct of arrays on the device).
// kind: bit0 value kernel (0 nearest, 1 linear), bits1-2 gradient kernel, bit3 has-gradient.
struct PointStore
{
	DevBuf<float>   pos, grad;        // D floats per point, interleaved
	DevBuf<float>   value, vw, gw;    // f(pos), weight*value_weight, weight*gradient_weight (add_points :357-368)
	DevBuf<uint8_t> kind;
	int64_t         count = 0;
};

struct PointView
{
	const float *  pos, *grad, *value, *vw, *gw;
	const uint8_t* kind;
};

inline PointView view(const PointStore& s)
{
	return PointView{s.pos.data(), s.grad.data(), s.value.data(), s.vw.data(), s.gw.data(), s.kind.data()};
}

// ---- sort_scan.cu ------------------------------------------------------------------------------------
// Exclusive prefix sum over n uint64 values (in may alias out).  Returns nothing; total = out[n-1]+in[n-1]
// is written to *total_dev (device, nullable).
void exclusive_scan_u64(const uint64_t* in, uint64_t* out, int64_t n, uint64_t* total_dev, cudaStream_t s);
// Stable LSD radix sort of (key, value) pairs on the low `bits` bits of the key.  Sorted data ends in
// keys/vals (scratch buffers are swapped internally and results copied back if needed).
void radix_sort_pairs(DevBuf<uint64_t>& keys, DevBuf<uint32_t>& vals, int64_t n, int bits, cudaStream_t s);

// ---- assembly.cu (compiled with -fmad=false: bit-exact restatement of the reference's fp32 arithmetic) ----
void canonicalise_points(const Geom& g, PointStore& store, float value_weight, int value_kernel, float gradient_weight,
                         int gradient_kernel, int64_t n, const float* d_pos, const float* d_nrm, const float* d_pw,
                         const float* d_val, cudaStream_t s);
// rows / triplets contributed by points [p0,p1) (exclusive prefix per point into out_rows/out_trips, totals to host)
void count_point_rows(const Geom& g, PointView pv, int64_t p0, int64_t p1, uint64_t* d_rowoff, uint64_t* d_tripoff,
                      uint64_t* h_rows, uint64_t* h_trips, cudaStream_t s);
void emit_point_rows(const Geom& g, PointView pv, int64_t p0, int64_t p1, const uint64_t* d_rowoff,
                     const uint64_t* d_tripoff, int64_t row_base, int64_t trip_base, fi_triplet* d_trips, float* d_rhs,
                     cudaStream_t s);
void count_model_rows(const Geom& g, const fi_weights& w, uint64_t* d_rowoff, uint64_t* d_tripoff, uint64_t* h_rows,
                      uint64_t* h_trips, cudaStream_t s);
void emit_model_rows(const Geom& g, const fi_weights& w, const uint64_t* d_rowoff, const uint64_t* d_tripoff,
                     int64_t row_base, int64_t trip_base, fi_triplet* d_trips, float* d_rhs, cudaStream_t s);
void upscale_device(const Geom& small, const Geom& large, const float* d_small, float* d_large, float post_scale,
                    cudaStream_t s);
// sample_field.cuh (included by assembly.cu): value (d_values, nullable) and gradient (d_gradients, D per point,
// nullable; gradient_kernel 0..2) of the unsharded lattice field at n interleaved positions; fi_sample_field states
// the contract.
void sample_field_device(const Geom& g, int64_t n, const float* d_positions, const float* d_field, int gradient_kernel,
                         float* d_values, float* d_gradients, cudaStream_t s);

// Data term of the normal equations in compact form: per occupied cell a symmetric 2^D x 2^D block
// (upper triangle, struct-of-arrays [tri][cell]) plus the rows that do not fit a cell (linear-interpolation
// gradient rows) as CSR.
template <typename T>
struct DataTerm
{
	int64_t            nocc = 0;
	DevBuf<uint64_t>   cell_key;  // per occupied cell: sum (base_d + 1) * kstride_d, sorted ascending
	DevBuf<int64_t>    cell_base; // local index of the cell's corner 0 (may lie outside the lattice: see cell_mask)
	DevBuf<uint32_t>   cell_mask; // bits 0..7: corner is a lattice node; bits 8..15: ... whose row this process owns
	DevBuf<T>          blocks;    // [tri(2^D)][nocc]
	// The same matrix P = sum of the cell blocks, node-major (built only with FI_B200_DATA_TERM=node, assembly.cu): for
	// every lattice node that is a corner of an occupied cell (and whose row this process owns) the 3^D coefficients of its
	// row, so that q += P p is a gather with one writer per node — no atomics, bit-reproducible.
	int64_t            nnode = 0;
	DevBuf<int64_t>    node_index; // [nnode] local index of the node, ascending
	DevBuf<T>          node_coef;  // [3^D][nnode]; slot = sum_d (delta_d + 1) 3^d for the neighbour at offset delta in {-1,0,1}^D
	int64_t            nrows = 0; // generic rows (derived + caller-appended)
	DevBuf<uint64_t>   row_ptr;   // nrows + 1
	DevBuf<int32_t>    col;
	DevBuf<float>      val;
	DevBuf<double>     partial;   // reduction scratch of the two apply kernels
	DevBuf<unsigned>   ticket;
};

struct HostRows  // caller-appended rows (add_equation), already weighted
{
	std::vector<uint64_t> ptr{0};
	std::vector<int32_t>  col;
	std::vector<float>    val, rhs;
	int64_t rows() const { return static_cast<int64_t>(rhs.size()); }
};

// Builds the data term, and accumulates Atb and diag(AtA) of all data rows into d_atb / d_diag (pre-zeroed or
// pre-filled by the caller).
template <typename T>
void build_data_term(const Geom& g, const PointStore& pts, const HostRows& user_rows, DataTerm<T>& out, T* d_atb,
                     T* d_diag, cudaStream_t s);

// q += P p over the compact data term; p.(P p) is *added* to d_dot_accum[0] (nullable).
// pub (multi-GPU peer path, nullable): the block that completes the sum also publishes d_dot_accum[0] to every rank's
// mailbox (peer.cuh) — returns true when it did, false when the caller has to (no occupied cells here, generic rows).
struct PeerPublish;
template <typename T>
bool apply_data_term(const Geom& g, const DataTerm<T>& dt, const T* p, T* q, double* d_dot_accum, const int* d_done,
                     cudaStream_t s, const PeerPublish* pub = nullptr);

// The data term's share of the epilogue-mode stencil step (stencil_tma_3d_epilogue): with u = P in,
// res_out -= u and, when d_new is given, d_new -= b minv u, e -= b minv u — by atomics over the occupied cells.
// Cell blocks only: false (nothing done) when the data term has generic rows.
template <typename T>
bool apply_data_term_epilogue(const Geom& g, const DataTerm<T>& dt, const T* in, T* res_out, const T* minv, T* e, T* d_new, T b,
                              cudaStream_t s);

// ---- field_error_map.cuh (included by assembly.cu, compiled with -fmad=false) ---------------------------------
// generate_error_map of the rows one builder call added, from the field's own description; fi_field_error_map states
// the contract.  Each adds the segment's terms to d_heat (device, N floats) in the segment's triplet order and the
// fp64 sum of its rows' err^2 to *d_sum (device).  Point and caller rows go through scratch of at most
// error_map_chunk_triplets() triplets at a time (2^26; FI_B200_ERROR_MAP_CHUNK overrides it).
struct ErrorMapScratch
{
	DevBuf<uint64_t>   rowoff, tripoff, row_ptr, key;
	DevBuf<uint32_t>   idx;
	DevBuf<fi_triplet> trips;
	DevBuf<int32_t>    col;
	DevBuf<float>      val, rhs, term;
	DevBuf<double>     partial;
};
int64_t error_map_chunk_triplets();
void    model_error_map(const Geom& g, const fi_weights& w, const float* d_x, float* d_heat, double* d_sum, ErrorMapScratch& sc, cudaStream_t s);
void    point_error_map(const Geom& g, PointView pv, int64_t p0, int64_t p1, const float* d_x, float* d_heat, double* d_sum, ErrorMapScratch& sc,
                        cudaStream_t s);
void    caller_rows_error_map(const Geom& g, const HostRows& rows, int64_t r0, int64_t r1, const float* d_x, float* d_heat, double* d_sum,
                              ErrorMapScratch& sc, cudaStream_t s);

// ---- errormap.cu ------------------------------------------------------------------------------------------
void error_map(int64_t nt, const fi_triplet* h_trips, int64_t n, const float* h_x, int64_t nrows, const float* h_rhs, float* h_out);

// ---- isosurface.cu (compiled with -fmad=false) ----------------------------------------------------------------
int64_t marching_squares_device(int width, int height, const float* d_values, float iso, float* d_lines, int64_t capacity, cudaStream_t s);
double  area_twice_device(int64_t nseg, const float* d_lines, cudaStream_t s);
void    bicubic_upsample_device(int width, int height, const float* d_values, int upsample, float* d_large, cudaStream_t s);

// ---- marching_cubes.cuh (included by isosurface.cu, compiled with -fmad=false) --------------------------------------
// Mesh of `values == iso` of a sizes[0] x sizes[1] x sizes[2] lattice (x fastest) on the device; the contract is in
// include/fi_b200.h (fi_marching_cubes).  Always returns the counts.  Vertices / normals (3 floats each, nullable) and
// triangles (3 int32 each, nullable) are written only when every requested buffer holds its count; all outputs
// nullptr: count only.
struct McCounts
{
	int64_t vertices = 0, triangles = 0;
};
McCounts marching_cubes_device(const int32_t* sizes, const float* d_values, float iso, float* d_vertices, float* d_normals,
                               int64_t capacity_vertices, int32_t* d_triangles, int64_t capacity_triangles, cudaStream_t s);

// ---- stencil.cu ------------------------------------------------------------------------------------------
// Per-axis banded operator T_d = sum_k w_k^2 D_k^T D_k (rows that stick out dropped), 9 row classes x 9 taps,
// plus the tri-diagonal D_1^T D_1 used by the gradient-smoothness cross terms.  See DESIGN.md §3.
struct StencilTables
{
	double band[kMaxDim][9][9];  // [axis][row class][tap t = offset + 4]
	double gs2;                  // 2 * sum of gradient_smoothness^2
	int    radius;               // highest active order (taps beyond are zero)
	bool   any;                  // any smoothness at all
};

// Sum over add_model calls of the products of row coefficients.  The reference stores each coefficient as the
// fp32 product binomial * w_k (add_equation, sparse_linear.cpp:43) before anything is squared, so the products
// are formed from those rounded values: cc[k][a][b] = sum_calls double(c_ka) * double(c_kb).
struct ModelAccum
{
	double cc[5][5][5] = {};
	bool   on[5]       = {false, false, false, false, false};
	double gs_sq       = 0;  // sum of double(1.0f * w_gs)^2
};

StencilTables make_tables(const Geom& g, const ModelAccum& m);

// d_diag += diag(S); with d_minv also the Jacobi preconditioner of the finished diagonal: 1 / diag (1 where diag == 0)
template <typename T>
void stencil_diagonal(const Geom& g, const StencilTables& t, T* d_diag /* += */, T* d_minv /* nullable */, cudaStream_t s);

// q = S p (overwrites q).  When d_dot_out is non-null, p.q is reduced deterministically (per-block partials in
// d_partial, summed in block order by the last block to arrive) and *stored* to d_dot_out[0].  d_done
// (nullable) is the solver's device-side convergence flag: the kernel returns at once when it is set.
// mode selects the kernel: generic (reference-shaped, any dimension / weights), auto (TMA-staged 3D kernel when
// applicable, else the tiled one, else generic), tiled (register-pipeline 3D kernel without TMA, else generic).
enum StencilMode { kStencilGeneric = 0, kStencilAuto = 1, kStencilTiled = 2 };
template <typename T>
void stencil_apply(const Geom& g, const StencilTables& t, const T* p, T* q, double* d_dot_out, double* d_partial,
                   unsigned* d_ticket, const int* d_done, int mode, cudaStream_t s);
int stencil_partial_slots(const Geom& g);  // upper bound of blocks any stencil launch uses (size of d_partial)

// ---- dist.cu ------------------------------------------------------------------------------------------------
void     slab_range(int nz, int world, int rank, int* z0, int* z1);
// Planes [z0, z1) of `rank` on this communicator: its custom cuts when they were set for an nz-plane lattice, else slab_range.
void     comm_slab_range(const fi_comm* c, int nz, int rank, int* z0, int* z1);
const int* comm_cuts(const fi_comm* c, int nz);  // world + 1 plane numbers, or nullptr (uniform partition)
void     comm_set_cuts(fi_comm* c, int nz, const int32_t* cuts);
// Cuts that balance  planes * nx * ny + point_weight * (points whose cell starts in the plane)  over the ranks, every slab at
// least min_planes thick.  Deterministic: every rank computes the same cuts from the same cloud.
void     balanced_cuts(const int32_t* sizes, int world, int64_t num_points, const float* positions, int loc, double point_weight, int min_planes,
                       int32_t* cuts);
void     comm_unique_id(void* id, int64_t capacity);
fi_comm* comm_create(int rank, int world, const void* id);
void     comm_destroy(fi_comm* c);
void     slab_sdf_solve(fi_comm* c, const int32_t* sizes, const fi_weights& w, int64_t num_points, const float* positions, const float* normals,
                        const float* point_weights, int loc, const fi_solve_options& o, const float* guess_own, float* solution_own,
                        int sol_loc, fi_solve_stats* st);

}  // namespace fi
