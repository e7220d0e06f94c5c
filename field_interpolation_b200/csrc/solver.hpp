// Normal-equation operator and the preconditioned conjugate-gradient driver (solver.cu).
#pragma once

#include <utility>
#include <vector>

#include "internal.hpp"
#include "peer.cuh"

namespace fi {

// Multi-GPU plumbing of one z-slab solve (dist.cu); nullptr everywhere else.
struct DistHooks
{
	virtual ~DistHooks() = default;
	// Peer-memory path.  link() is null when it is unavailable (then the NCCL calls below carry the iteration).
	virtual const PeerLink* link() { return nullptr; }
	// A lattice vector of `bytes` that the neighbouring ranks can store into (collective; contents zeroed on
	// stream s).  lo / hi receive the neighbours' mappings of *their* vector (null at the ends).
	virtual void* shared_vector(size_t bytes, void** lo, void** hi, cudaStream_t s)
	{
		(void)bytes; (void)lo; (void)hi; (void)s;
		return nullptr;
	}
	virtual int64_t peer_own_cells(int peer) { (void)peer; return 0; }
	virtual unsigned long long next_seq() { return 0; }
	// in-place sum over ranks of `count` doubles in device memory, enqueued on s (capturable)
	virtual void allreduce(double* d_ptr, int count, cudaStream_t s) = 0;
	// fills the halo planes of a local lattice vector from the neighbouring slabs' owned planes
	virtual void exchange_halo(void* d_vec, size_t elem_size, cudaStream_t s) = 0;
	virtual int rank() const { return 0; }
	virtual int world() const { return 1; }
	// hooks on the same communicator for another slab geometry (a coarser multigrid level); NCCL path only
	virtual std::unique_ptr<DistHooks> for_geom(const Geom& g, int halo)
	{
		(void)g; (void)halo;
		return nullptr;
	}
	// `full` is a whole (unsharded) lattice vector of planes of `plane_cells` floats of which rank k has filled planes
	// [own[k].first, own[k].second); afterwards every rank holds every plane (all-gather with ragged counts)
	virtual void allgather_planes(float* full, int64_t plane_cells, const std::vector<std::pair<int, int>>& own, cudaStream_t s)
	{
		(void)full; (void)plane_cells; (void)own; (void)s;
	}
};

// Most search directions the fused PCG iteration keeps before it folds their terms into x (solver.cu, choose_x_ring).
constexpr int kMaxXRing = 8;

template <typename T>
struct PcgWork
{
	DevBuf<T>        r, q;
	// Search directions.  The fused direction+stencil iteration k reads dir[k mod m] and writes dir[(k+1) mod m] (m = the
	// x ring of the solve, 2 on slab-sharded lattices: the ping-pong pair dir[0] / dir[1]); the unfused iteration uses dir[0].
	DevBuf<T>        dir[kMaxXRing];
	int              dirs = 0;  // dir[0 .. dirs) are allocated (lattice-sized, zeroed when allocated)
	DevBuf<double>   alpha;     // step lengths of the iterations whose x update is still pending (kMaxXRing - 1)
	DevBuf<double>   partial;
	DevBuf<unsigned> ticket;
	DevBuf<PcgState> state;
};

// A^T A = S (matrix-free stencil) + P (cell blocks + generic rows), with A^T b and the Jacobi preconditioner.
template <typename T>
struct Operator
{
	Geom             g;
	StencilTables    tabs;
	DataTerm<T>      data;
	DevBuf<T>        atb, diag, minv;
	DevBuf<double>   partial;  // stencil reduction scratch
	DevBuf<unsigned> ticket;
	int              use_fast = kStencilAuto;  // StencilMode
	double           setup_ms = 0;
	PcgWork<T>       work;
	DistHooks*       dist = nullptr;  // set for a z-slab of a lattice shared with other ranks
	// Set by a caller that hands pcg_solve an all-zero guess: the initial residual is then b itself and the operator
	// application that would compute A x is skipped.  Consumed (reset) by the solve.
	bool             guess_is_zero = false;

	// q = (S + P) p; when d_dot is non-null it receives p.q (deterministic apart from the order of the data
	// term's atomics into q).
	void apply(const T* p, T* q, double* d_dot, const int* d_done, cudaStream_t s)
	{
		stencil_apply<T>(g, tabs, p, q, d_dot, partial.data(), ticket.data(), d_done, use_fast, s);
		apply_data_term<T>(g, data, p, q, d_dot, d_done, s);
	}
};

template <typename T>
std::unique_ptr<Operator<T>> build_operator(const Geom& g, const ModelAccum& m, const PointStore& pts, const HostRows& rows,
                                            cudaStream_t s);

struct PcgResult
{
	long long iterations = 0;
	double    rel_residual = 0, initial_residual = 0, true_residual = 0, solve_ms = 0;
	double    loop_ms = 0;  // graph launches only (no init, capture or instantiation)
	int       x_ring = 1;   // iterations per x update: the ring of directions the fused path kept (1: the unfused iteration)
	bool      converged = false, zero_rhs = false;
	// The iteration cannot get further in this arithmetic: CG broke down, or the residual recomputed from x stopped
	// following the recurrence (an fp32 solve at the rounding floor of an ill-conditioned system).  The caller may continue
	// from x in wider arithmetic.
	bool      stalled = false;
};

// `converged` means the TRUE residual met the stopping rule, with this much slack on |r| for the difference between the
// recurrence (which decided when to stop) and the residual recomputed from x.
constexpr double kConvergedSlack = 1.25;

// Solves A x = b from the guess in x (device, N elements of T).  b == nullptr: the operator's own A^T b.
// With op.dist set, x / b are local slab vectors (halo planes included) and every rank calls this together.
template <typename T>
PcgResult pcg_solve(Operator<T>& op, const T* b, T* x, double tol, long long max_iter, int check_every, bool want_true_residual,
                    cudaStream_t s);

// stencil_fast.cu: p_new = M r + beta p_old, q = S p_new, dot = p_new.q in one pass.  false: not applicable.
template <typename T>
bool stencil_fast_3d_fused(const Geom& g, const StencilTables& t, const T* r, const T* minv, const T* p_old, T* p_new, T* q,
                           const PcgState* st, int par, double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done,
                           cudaStream_t s);

// stencil_tma.cu: the same fused step with TMA-staged loads.  false: not applicable.
template <typename T>
bool stencil_tma_3d_fused(const Geom& g, const StencilTables& t, const T* r, const T* minv, const T* p_old, T* p_new, T* q,
                          const PcgState* st, int par, double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done,
                          cudaStream_t s);

// stencil_tma.cu, epilogue mode (multigrid smoother): res_out = res_in - S in; with d_new: d_new = a in + b minv res_out,
// e += d_new.  Nothing else is stored.  false: not applicable (then the caller uses apply + vector kernels).
template <typename T>
bool stencil_tma_3d_epilogue(const Geom& g, const StencilTables& t, const T* in, const T* res_in, T* res_out, const T* minv, T* e, T* d_new,
                             T a, T b, cudaStream_t s);

// stencil_2d.cu: the same three entry points for 2D lattices (any weights, gradient smoothness included).
template <typename T>
bool stencil_tma_2d_fused(const Geom& g, const StencilTables& t, const T* r, const T* minv, const T* p_old, T* p_new, T* q, const PcgState* st, int par,
                          double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s);
template <typename T>
bool stencil_tma_2d_epilogue(const Geom& g, const StencilTables& t, const T* in, const T* res_in, T* res_out, const T* minv, T* e, T* d_new, T a, T b,
                             cudaStream_t s);

// The fused direction+stencil step in the given StencilMode; false when no fused kernel applies.
template <typename T>
inline bool stencil_fused_step(int mode, const Geom& g, const StencilTables& t, const T* r, const T* minv, const T* p_old, T* p_new,
                               T* q, const PcgState* st, int par, double* d_dot_out, double* d_partial, unsigned* d_ticket,
                               const int* d_done, cudaStream_t s)
{
	if (g.tile) { return false; }  // tile mode: generic kernels only
	if (mode == kStencilAuto && g.ndim == 2) { return stencil_tma_2d_fused<T>(g, t, r, minv, p_old, p_new, q, st, par, d_dot_out, d_partial, d_ticket, d_done, s); }
	if (mode == kStencilAuto && stencil_tma_3d_fused<T>(g, t, r, minv, p_old, p_new, q, st, par, d_dot_out, d_partial, d_ticket, d_done, s)) { return true; }
	if (mode != kStencilGeneric && stencil_fast_3d_fused<T>(g, t, r, minv, p_old, p_new, q, st, par, d_dot_out, d_partial, d_ticket, d_done, s)) { return true; }
	return false;
}

// ---- mg.cu: geometric multigrid preconditioner ----------------------------------------------------------------
struct MgOptions
{
	int    nu               = 3;     // Chebyshev steps before and after the coarse-grid correction
	int    nu_coarse        = 0;     // ... on levels >= 1 (each costs 1/2^D of the level above); 0: the same as nu
	int    gamma            = 1;     // 1: V-cycle; 2: W-cycle (two coarse corrections per level, the second on the residual of the first)
	int    w_levels         = 3;     // gamma = 2 applies to the coarse problems of levels 1 .. w_levels only: below, the levels are tiny and a
	                                 // W-cycle would visit them 2^level times for no gain but launch latency
	double cheb_ratio       = 12.0;  // the smoother targets the eigenvalues of D^-1 A in [lambda_max / ratio, lambda_max]
	int    coarsest_cells   = 600;   // coarsen until a level has at most this many cells (dense solve there, inverse computed on the device)
	int    power_iterations = 20;    // for lambda_max, per level, at setup.  The top of the spectrum of D^-1 A is dense, so the estimate
	                                 // creeps up slowly: after 12 rounds it was 0.877 lambda_max on a 48 x 20 level, and 1.1 times that is
	                                 // below lambda_max (the smoother then amplifies the top modes); 20 rounds reach >= 0.93 on every level
	                                 // of tests/test_gpu_multigrid_operator.py
	int    tail_cells       = 0;     // > 0: coarse levels with at most this many nodes are walked by ONE kernel (mg_tail_kernel) instead of
	                                 // three launches per smoothing step (FI_B200_MG_TAIL_CELLS).  Off by default: measured slower — one SM
	                                 // retires the data term's reductions at 1.3 cycles per lane, 283 us per visit of a 16^3 level against
	                                 // ~130 us for the launches it replaces (profiles/r2p_time_to_tol_tail_kernel.jsonl)
};

// The hierarchy's parameters when the caller leaves them alone, from the B200 sweeps of round 2
// (profiles/r2d_mg_sweep.jsonl; fp64-outer MG-PCG to a 1e-6 true residual, default Weights):
//   * operators up to model_2: 2 Chebyshev steps on the finest level, 4 on the coarse ones (each level costs 1/2^D of
//     the one above) — 512^3: 27 iterations / 254 ms against 30 / 322 ms with 3 steps everywhere; 256^3: 48 against 59 ms;
//   * 3D lattices from 50 M cells on one GPU: W-cycles over the three largest coarse levels with 6 coarse steps — 512^3:
//     10 iterations / 169 ms.  Below that size the extra visits are launch latency, not work, and V wins; on z-slabs the
//     replicated tail would be visited four times per rank, so sharded solves stay with V;
//   * model_3 / model_4 rows (6th / 8th-order stencils) leave more high-frequency error per step: 5 steps everywhere, V
//     (model_3 alone, 32x16x24: 80 MG-PCG iterations reach 3e-7 with 5 steps, 2e-3 with 3; round 1).
// `user_nu` > 0 (fi_solve_options::mg_smoothing_steps) sets the finest level's steps; the coarse levels get at least as many.
inline MgOptions default_mg_options(const ModelAccum& m, const Geom& g, bool sharded, int user_nu, double user_ratio)
{
	MgOptions o;
	const bool high_order = m.on[3] || m.on[4];
	o.nu        = high_order ? 5 : 2;
	o.nu_coarse = high_order ? 0 : 4;
	const int64_t cells = static_cast<int64_t>(g.size[0]) * g.size[1] * g.size[2];
	if (g.ndim == 3 && !sharded && !high_order && cells >= 50000000) {
		o.gamma     = 2;
		o.nu_coarse = 6;
		o.w_levels  = 3;
	}
	if (user_nu > 0) {
		o.nu = user_nu;
		if (o.nu_coarse > 0 && o.nu_coarse < user_nu) { o.nu_coarse = user_nu; }
	}
	if (user_ratio > 1.0) { o.cheb_ratio = user_ratio; }
	return o;
}

// Tuning knobs of the hierarchy read from the environment (same on every rank): FI_B200_MG_COARSEST (cells of the dense
// coarsest level), FI_B200_MG_NU_COARSE, FI_B200_MG_GAMMA, FI_B200_MG_WLEVELS.
void mg_options_from_env(MgOptions& o);

struct Multigrid
{
	struct Level;
	MgOptions                           opt;
	std::vector<std::unique_ptr<Level>> levels;      // 0 = finest
	DevBuf<float>                       coarse_inv;  // dense inverse of the coarsest operator, row-major nc x nc
	int                                 nc = 0;
	int                                 base_level = 0;  // level of levels[0] in the hierarchy of the root lattice (> 0: the replicated tail of a slab V-cycle)
	DevBuf<unsigned char>               tail_plan;       // descriptors of levels tail_from .. (mg_tail_kernel); tail_from = 0: none
	int                                 tail_from = 0, tail_nlev = 0;
	cudaGraphExec_t                     exec = nullptr;  // the V-cycle for (graph_r -> graph_z)
	const float*                        graph_r = nullptr;
	float*                              graph_z = nullptr;
	int64_t                             graph_launches = 0;

	Multigrid();
	~Multigrid();
	// z = V-cycle(r): one application of the preconditioner (fp32, finest-level vectors of N floats)
	void vcycle(const float* r, float* z, cudaStream_t s);
	// A W-cycle is a symmetric preconditioner but positive definite only while the V-cycle it repeats converges as a
	// stationary iteration; when CG breaks down on it the solver falls back to V-cycles.  False: already V.
	bool demote_to_v_cycle();
};

// Builds the hierarchy under `fine` (which must outlive it): re-discretised coarse operators from the same points
// and the same smoothness model, Chebyshev bounds, dense coarsest inverse.  `model` / `pts` describe the ROOT lattice
// of the hierarchy (sizes root_size; null: fine.g.size) and `fine` is its level `fine_level` (0: the root itself) —
// the slab-sharded V-cycle hands the levels below its last sharded one to a hierarchy built this way, so that every
// level's operator is the one the single-GPU hierarchy would have.
std::unique_ptr<Multigrid> build_multigrid(Operator<float>& fine, const ModelAccum& model, const PointStore& pts, const MgOptions& opt, cudaStream_t s,
                                           const int* root_size = nullptr, int fine_level = 0);

// The hierarchy's shape and parameters (fi_field_mg_info), and one stage of its cycle applied to `count` host vectors
// (fi_field_mg_stage: stage FI_MG_*, the kernels vcycle() runs, on scratch vectors of its own).  For tests.
void mg_info(const Multigrid& mg, fi_mg_info* out);
void mg_stage(Multigrid& mg, int stage, int level, int64_t count, const float* in, const float* in2, float* out, cudaStream_t s);

// ---- mg.cu: the same V-cycle with the finest levels z-slab sharded over the ranks of a communicator -------------
// Levels 0 .. nd-1 are sharded (each rank smooths its slab; halo planes of the smoothed vector are exchanged before
// every operator application), level nd and everything below it is replicated: the restricted residual is
// all-gathered and every rank runs the rest of the V-cycle (a plain `Multigrid`, one CUDA graph) redundantly, then
// prolongs into its own planes.  Coarse plane C of a level pair belongs to the rank that owns the middle one of the
// fine planes restriction reads for it, so restriction needs at most `halo` (>= 2) planes from a neighbour.
constexpr int kMaxSlabLevels = 8;

struct SlabMgPlan  // pure host arithmetic, identical on every rank
{
	int nd   = 0;                    // sharded levels (>= 1)
	int halo = 2;                    // halo planes stored per side on every sharded level
	int world = 1;
	int size[kMaxSlabLevels + 1][kMaxDim] = {};             // lattice sizes of levels 0 .. nd
	std::vector<std::pair<int, int>> own[kMaxSlabLevels + 1];  // own[l][rank]: planes [z0, z1) of level l (for level nd: the planes the rank restricts into)
};

// Throws FI_ERR_UNSUPPORTED when level 0 cannot be sharded this way (slabs thinner than the halo, sizes the TMA stencil
// kernel does not take, a restriction that would reach beyond the halo).  gather_cells: levels with at most this many
// cells are replicated.
// cuts (nullable): world + 1 plane numbers of a non-uniform level-0 partition (fi_comm_set_slab_cuts); else slab_range.
SlabMgPlan plan_slab_multigrid(const int32_t* sizes, int world, int radius, int64_t gather_cells, const int* cuts = nullptr);

struct SlabMultigrid
{
	struct DLevel;
	MgOptions                             opt;
	SlabMgPlan                            plan;
	int                                   rank = 0;
	std::vector<std::unique_ptr<DLevel>>  dl;       // sharded levels, 0 = finest
	std::unique_ptr<Operator<float>>      tail_op;  // first replicated level (unsharded lattice)
	PointStore                            tail_pts;
	std::unique_ptr<Multigrid>            tail;
	DevBuf<float>                         tail_r, tail_e;

	SlabMultigrid();
	~SlabMultigrid();
	// z = V-cycle(r) on slab-local vectors of the finest level (owned planes are read / written)
	void vcycle(const float* r, float* z, cudaStream_t s);
	bool demote_to_v_cycle() { return false; }  // sharded levels run V-cycles only
};

// fine: this rank's slab operator of the finest level with fine.dist set (it must outlive the hierarchy); model / pts:
// the whole problem (every rank holds all points).
std::unique_ptr<SlabMultigrid> build_slab_multigrid(Operator<float>& fine, const ModelAccum& model, const PointStore& pts, const MgOptions& opt,
                                                    const SlabMgPlan& plan, cudaStream_t s);

// CG preconditioned by one V-cycle per iteration; same contract as pcg_solve.  guard_every > 0: every that many
// iterations the residual is recomputed from x, and the solve stops with `stalled` set once it is more than twice the
// recurrence residual (the floor of the arithmetic T has been reached; see PcgResult::stalled).
template <typename T>
PcgResult mgpcg_solve(Operator<T>& op, Multigrid& mg, const T* b, T* x, double tol, long long max_iter, cudaStream_t s, int guard_every = 0);
// The same on a slab (op.dist set; x / b are slab-local vectors, every rank calls this together).
template <typename T>
PcgResult slab_mgpcg_solve(Operator<T>& op, SlabMultigrid& mg, const T* b, T* x, double tol, long long max_iter, cudaStream_t s, int guard_every = 0);

// Tile phase of solve_tiled_with_guess (reference sparse_linear.cpp:246-390): x holds the guess on entry and the
// tile-by-tile solution on exit.  The returned statistics are those of the block-diagonal solve.
template <typename T>
PcgResult tile_phase(Operator<T>& op, int tile_size, T* x, double tol, long long max_iter, int check_every, cudaStream_t s);

template <typename T>
void jacobi_sweeps(Operator<T>& op, T* x, int iterations, T weight, cudaStream_t s);

// out[0..7]: see fi_field_time_iterations in include/fi_b200.h.
template <typename T>
void time_kernels(Operator<T>& op, int iterations, int check_every, double* out, cudaStream_t s);

// One stage of the unsharded Jacobi-PCG iteration (fi_field_pcg_stage, include/fi_b200.h).  For tests.
template <typename T>
void pcg_stage(Operator<T>& op, int stage, int par, int pos, int ring, int count, int loc, void* const* vecs, double tol, long long max_iters,
               fi_pcg_state* state, fi_pcg_report* report, cudaStream_t s);

// r = b - A x (device), returns |r|^2 and |b|^2.
template <typename T>
void residual(Operator<T>& op, const T* b, const T* x, T* r, double* rr, double* bb, cudaStream_t s);

void convert(const float* src, double* dst, int64_t n, cudaStream_t s);
void convert(const double* src, float* dst, int64_t n, cudaStream_t s);
void axpy_f32_into_f64(const float* e, double* x, int64_t n, cudaStream_t s);  // x += e

}  // namespace fi
