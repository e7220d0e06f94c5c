// C ABI of libfi_b200 (declared in include/fi_b200.h): the LatticeField handle, the constraint builders, the
// triplet view, the solvers and the coarse-to-fine driver.  Everything crosses the boundary as plain pointers
// and sizes; C++ exceptions stop here and become status codes.
#include <time.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <exception>
#include <map>
#include <mutex>
#include <new>

#include "solver.hpp"

namespace fi {

int64_t                   g_launches = 0;
LaunchNote                g_note;
static thread_local std::string t_last_error;

void set_last_error(const std::string& s) { t_last_error = s; }

int sm_count()
{
	static thread_local int cached_dev = -1, cached = 0;
	int dev = 0;
	if (cudaGetDevice(&dev) != cudaSuccess) { return 148; }
	if (dev != cached_dev) {
		cudaDeviceProp prop;
		if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) { cached = prop.multiProcessorCount; } else { cached = 148; }
		cached_dev = dev;
	}
	return cached;
}

// ---- tracing ---------------------------------------------------------------------------------------------
static double now_ms()
{
	timespec ts;
	clock_gettime(CLOCK_MONOTONIC, &ts);
	return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
bool trace_enabled()
{
	static const bool on = [] {
		const char* e = getenv("FI_B200_TRACE");
		return e && *e && *e != '0';
	}();
	return on;
}
static thread_local int t_trace_depth = 0;
TraceScope::TraceScope(const char* n) : name(n), t0(0)
{
	if (trace_enabled()) {
		t0 = now_ms();
		++t_trace_depth;
	}
}
TraceScope::~TraceScope()
{
	if (trace_enabled()) {
		--t_trace_depth;
		fprintf(stderr, "[fi_b200] %*s%s: %.3f ms\n", 2 * t_trace_depth, "", name, now_ms() - t0);
	}
}

// ---- device memory cache -----------------------------------------------------------------------------------
namespace {
struct Pool
{
	std::mutex                        mu;
	std::multimap<size_t, void*>      free_blocks;  // per device: keyed by (device, bytes) folded into one size_t below
	size_t                            cached = 0;
	bool                              dirty[16] = {};  // per device: blocks were released since its last synchronisation
	size_t                            limit  = 0;
};
Pool& pool()
{
	static Pool p;
	return p;
}
size_t round_block(size_t bytes) { return bytes >= (1u << 20) ? ((bytes + (2u << 20) - 1) >> 21) << 21 : ((bytes + 511) >> 9) << 9; }
int pool_device()
{
	int dev = 0;
	cudaGetDevice(&dev);
	return dev & 15;
}
size_t pool_key(size_t rounded, int dev)
{
	return rounded * 16 + static_cast<size_t>(dev);  // sizes are multiples of 512: the low bits are free for the device
}
}  // namespace

void* pool_alloc(size_t bytes)
{
	Pool&        P = pool();
	const int    dev = pool_device();
	const size_t rb = round_block(bytes), key = pool_key(rb, dev);
	{
		std::lock_guard<std::mutex> lock(P.mu);
		auto it = P.free_blocks.find(key);
		if (it != P.free_blocks.end()) {
			void* p = it->second;
			P.free_blocks.erase(it);
			P.cached -= rb;
			if (P.dirty[dev]) {  // whoever released it may still have had work in flight on some stream of this device
				cudaDeviceSynchronize();
				P.dirty[dev] = false;
			}
			return p;
		}
	}
	void*       p = nullptr;
	cudaError_t e = cudaMalloc(&p, rb);
	if (e != cudaSuccess) {  // give the cache back and retry once
		cudaGetLastError();
		pool_trim();
		e = cudaMalloc(&p, rb);
	}
	if (e != cudaSuccess) {
		throw Error{FI_ERR_CUDA, std::string("cudaMalloc of ") + std::to_string(rb) + " bytes: " + cudaGetErrorString(e)};
	}
	return p;
}

void pool_free(void* p, size_t bytes)
{
	if (!p) { return; }
	Pool&        P = pool();
	const size_t rb = round_block(bytes);
	std::lock_guard<std::mutex> lock(P.mu);
	if (P.limit == 0) {
		const char* e = getenv("FI_B200_POOL_GB");
		P.limit       = static_cast<size_t>((e ? atof(e) : 96.0) * 1073741824.0) + 1;
	}
	if (P.cached + rb > P.limit) {
		cudaFree(p);
		return;
	}
	const int dev = pool_device();
	P.free_blocks.emplace(pool_key(rb, dev), p);
	P.cached += rb;
	P.dirty[dev] = true;
}

void pool_trim()
{
	Pool& P = pool();
	std::lock_guard<std::mutex> lock(P.mu);
	for (auto& kv : P.free_blocks) { cudaFree(kv.second); }
	P.free_blocks.clear();
	P.cached = 0;
	for (bool& d : P.dirty) { d = false; }
}

size_t pool_cached_bytes()
{
	Pool& P = pool();
	std::lock_guard<std::mutex> lock(P.mu);
	return P.cached;
}

template <typename F>
int guarded(F&& f)
{
	try {
		f();
		return FI_OK;
	} catch (const Error& e) {
		set_last_error(e.what);
		return e.code;
	} catch (const std::bad_alloc&) {
		set_last_error("host allocation failed");
		return FI_ERR_INVALID;
	} catch (const std::exception& e) {
		set_last_error(e.what());
		return FI_ERR_INVALID;
	}
}

struct Segment
{
	enum Kind { kModel, kPoints, kRows } kind;
	fi_weights w{};          // kModel
	int64_t    p0 = 0, p1 = 0;  // kPoints: range in the point store
	int64_t    r0 = 0, r1 = 0;  // kRows: row range in the caller-row store
	int64_t    rows = -1, trips = -1;  // cached counts (-1: not computed yet)
};

}  // namespace fi

struct fi_field
{
	fi::Geom                               g;
	cudaStream_t                           stream = nullptr;
	std::vector<fi::Segment>               segs;
	fi::PointStore                         pts;
	fi::HostRows                           rows;
	fi::ModelAccum                         model;
	std::unique_ptr<fi::Operator<float>>   op32;
	std::unique_ptr<fi::Operator<double>>  op64;
	std::unique_ptr<fi::Multigrid>         mg;      // hierarchy under op32 (FI_PRECOND_MULTIGRID)
	fi::MgOptions                          mg_opt;
	int                                    fast = fi::kStencilAuto;  // kernel choice of fi_field_apply

	void invalidate()
	{
		mg.reset();
		op32.reset();
		op64.reset();
	}
	fi::Multigrid& get_mg(const fi_solve_options& o)
	{
		fi::MgOptions want = fi::default_mg_options(model, g, false, o.mg_smoothing_steps, o.mg_cheb_ratio);
		fi::mg_options_from_env(want);
		if (mg && (mg_opt.nu != want.nu || mg_opt.cheb_ratio != want.cheb_ratio || mg_opt.nu_coarse != want.nu_coarse || mg_opt.gamma != want.gamma ||
		           mg_opt.coarsest_cells != want.coarsest_cells || mg_opt.w_levels != want.w_levels || mg_opt.tail_cells != want.tail_cells)) {
			mg.reset();
		}
		if (!mg) {
			fi::Operator<float>& fine = get32();
			fine.use_fast             = fi::kStencilAuto;
			mg                        = fi::build_multigrid(fine, model, pts, want, stream);
			mg_opt                    = want;
		}
		return *mg;
	}
	fi::Operator<float>& get32()
	{
		if (!op32) { op32 = fi::build_operator<float>(g, model, pts, rows, stream); }
		return *op32;
	}
	fi::Operator<double>& get64()
	{
		if (!op64) { op64 = fi::build_operator<double>(g, model, pts, rows, stream); }
		return *op64;
	}
	~fi_field()
	{
		mg.reset();
		op32.reset();
		op64.reset();
		if (stream) { cudaStreamDestroy(stream); }
	}
};

namespace fi {

namespace {

// Stages a caller buffer on the device when it lives on the host.
template <typename T>
struct Staged
{
	DevBuf<T> own;
	const T*  ptr = nullptr;
	Staged(const T* src, size_t n, int loc, cudaStream_t s)
	{
		if (!src || n == 0) { return; }
		if (loc == FI_DEVICE) {
			ptr = src;
		} else {
			own.resize(n);
			FI_CUDA(cudaMemcpyAsync(own.data(), src, n * sizeof(T), cudaMemcpyHostToDevice, s));
			ptr = own.data();
		}
	}
};

void model_counts_closed_form(const Geom& g, const fi_weights& w, int64_t* rows, int64_t* trips)
{
	const float wk[5] = {w.model_0, w.model_1, w.model_2, w.model_3, w.model_4};
	int64_t     r = 0, t = 0;
	for (int d = 0; d < g.ndim; ++d) {
		const int64_t others = g.N / g.size[d];
		for (int k = 0; k <= 4; ++k) {
			if (wk[k] > 0 && g.size[d] > k) {
				r += (g.size[d] - k) * others;
				t += (g.size[d] - k) * others * (k + 1);
			}
		}
		if (w.gradient_smoothness > 0) {
			for (int o = 0; o < g.ndim; ++o) {
				if (o == d) { continue; }
				const int64_t n = static_cast<int64_t>(g.size[d] - 1) * (g.size[o] - 1) * (g.N / g.size[d] / g.size[o]);
				r += n;
				t += 4 * n;
			}
		}
	}
	*rows  = r;
	*trips = t;
}

void segment_counts(fi_field* f, Segment& sg)
{
	if (sg.rows >= 0) { return; }
	if (sg.kind == Segment::kModel) {
		model_counts_closed_form(f->g, sg.w, &sg.rows, &sg.trips);
	} else if (sg.kind == Segment::kPoints) {
		const int64_t    n = sg.p1 - sg.p0;
		DevBuf<uint64_t> ro(std::max<int64_t>(n, 1)), to(std::max<int64_t>(n, 1));
		uint64_t         hr = 0, ht = 0;
		count_point_rows(f->g, view(f->pts), sg.p0, sg.p1, ro.data(), to.data(), &hr, &ht, f->stream);
		sg.rows  = static_cast<int64_t>(hr);
		sg.trips = static_cast<int64_t>(ht);
	} else {
		sg.rows  = sg.r1 - sg.r0;
		sg.trips = static_cast<int64_t>(f->rows.ptr[sg.r1] - f->rows.ptr[sg.r0]);
	}
}

void check_weights(const fi_weights* w)
{
	FI_REQUIRE(w != nullptr, FI_ERR_INVALID, "weights is null");
	FI_REQUIRE(w->value_kernel == 0 || w->value_kernel == 1, FI_ERR_INVALID, "unknown value kernel");
	FI_REQUIRE(w->gradient_kernel >= 0 && w->gradient_kernel <= 2, FI_ERR_INVALID, "unknown gradient kernel");
}

}  // namespace

// Adds one add_field_constraints call to the accumulated smoothness operator (also used by dist.cu).
void accumulate_model(const fi_weights& w, ModelAccum& m)
{
	const float wk[5] = {w.model_0, w.model_1, w.model_2, w.model_3, w.model_4};
	static const float binom[5][5] = {{1, 0, 0, 0, 0}, {-1, 1, 0, 0, 0}, {1, -2, 1, 0, 0}, {1, -3, 3, -1, 0}, {1, -4, 6, -4, 1}};
	for (int k = 0; k <= 4; ++k) {
		if (!(wk[k] > 0)) { continue; }  // add_model_constraint emits order-k rows only for w_k > 0 (:257-292)
		m.on[k] = true;
		for (int a = 0; a <= k; ++a) {
			for (int b = 0; b <= k; ++b) {
				const volatile float ca = binom[k][a] * wk[k], cb = binom[k][b] * wk[k];  // fp32, as stored in the triplets
				m.cc[k][a][b] += static_cast<double>(ca) * static_cast<double>(cb);
			}
		}
	}
	if (w.gradient_smoothness > 0) {
		m.gs_sq += static_cast<double>(w.gradient_smoothness) * static_cast<double>(w.gradient_smoothness);
	}
}

namespace {

void add_model_impl(fi_field* f, const fi_weights* w)
{
	check_weights(w);
	Segment sg;
	sg.kind = Segment::kModel;
	sg.w    = *w;
	f->segs.push_back(sg);
	accumulate_model(*w, f->model);
	f->invalidate();
}

void add_points_impl(fi_field* f, float value_weight, int value_kernel, float gradient_weight, int gradient_kernel,
                     int64_t n, const float* pos, const float* nrm, const float* pw, const float* val, int loc,
                     int64_t* rows_added)
{
	TraceScope trace("add_points (stage + canonicalise)");
	FI_REQUIRE(n >= 0, FI_ERR_INVALID, "negative point count");
	FI_REQUIRE(value_kernel == 0 || value_kernel == 1, FI_ERR_INVALID, "unknown value kernel");
	FI_REQUIRE(gradient_kernel >= 0 && gradient_kernel <= 2, FI_ERR_INVALID, "unknown gradient kernel");
	FI_REQUIRE(n == 0 || pos != nullptr, FI_ERR_INVALID, "positions is null");
	// the reference CHECK-aborts when the nearest-neighbour value kernel is used without normals (:361)
	FI_REQUIRE(n == 0 || value_kernel != FI_VALUE_NEAREST_NEIGHBOR || nrm != nullptr, FI_ERR_INVALID,
	           "nearest-neighbour value kernel needs normals");
	FI_REQUIRE(f->pts.count + n < (1ll << 32), FI_ERR_RANGE, "more than 2^32 points in one field");
	if (rows_added) { *rows_added = 0; }
	if (n == 0) { return; }
	const int     D = f->g.ndim;
	Staged<float> dpos(pos, static_cast<size_t>(n) * D, loc, f->stream), dnrm(nrm, static_cast<size_t>(n) * D, loc, f->stream);
	Staged<float> dpw(pw, n, loc, f->stream), dval(val, n, loc, f->stream);
	Segment       sg;
	sg.kind = Segment::kPoints;
	sg.p0   = f->pts.count;
	canonicalise_points(f->g, f->pts, value_weight, value_kernel, gradient_weight, gradient_kernel, n, dpos.ptr, dnrm.ptr,
	                    dpw.ptr, dval.ptr, f->stream);
	sg.p1 = f->pts.count;
	FI_CUDA(cudaStreamSynchronize(f->stream));
	f->segs.push_back(sg);
	f->invalidate();
	if (rows_added) {
		segment_counts(f, f->segs.back());
		*rows_added = f->segs.back().rows;
	}
}

fi_field* create_impl(int32_t ndim, const int32_t* sizes)
{
	FI_REQUIRE(1 <= ndim && ndim <= kMaxDim, FI_ERR_INVALID, "ndim must be 1..3");
	FI_REQUIRE(sizes != nullptr, FI_ERR_INVALID, "sizes is null");
	int64_t n = 1;
	for (int d = 0; d < ndim; ++d) {
		FI_REQUIRE(sizes[d] >= 1, FI_ERR_INVALID, "lattice size must be >= 1");
		n *= sizes[d];
		FI_REQUIRE(n < (1ll << 40), FI_ERR_RANGE, "lattice too large");
	}
	int count = 0;
	FI_CUDA(cudaGetDeviceCount(&count));
	FI_REQUIRE(count > 0, FI_ERR_CUDA, "no CUDA device");
	auto f = std::make_unique<fi_field>();
	f->g   = make_geom(ndim, sizes);
	FI_CUDA(cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking));
	return f.release();
}

void fill_stats(fi_solve_stats* st, const PcgResult& r, double setup_ms, int64_t nocc, int64_t grows)
{
	if (!st) { return; }
	st->iterations        = r.iterations;
	st->relative_residual = r.rel_residual;
	st->true_residual     = r.true_residual;
	st->initial_residual  = r.initial_residual;
	st->setup_ms          = setup_ms;
	st->solve_ms          = r.solve_ms;
	st->converged         = r.converged ? 1 : 0;
	st->outer_sweeps      = 0;
	st->occupied_cells    = nocc;
	st->generic_rows      = grows;
	st->widened_after     = -1;
}

// Solves into d_out (device, N floats) from d_guess (device, nullable).
void solve_device(fi_field* f, const fi_solve_options& o, const float* d_guess, float* d_out, fi_solve_stats* st)
{
	const int64_t N = f->g.N;
	cudaStream_t  s = f->stream;
	const int     fast = o.use_fast_stencil;
	if (o.preconditioner == FI_PRECOND_MULTIGRID) {
		const bool fresh = !f->mg;
		CudaEvent  e0, e1;
		e0.record(s);
		Multigrid& mg = f->get_mg(o);
		PcgResult  r;
		long long  widened_after = -1;
		bool       start_wide = o.precision != FI_F32;
		if (o.precision == FI_F32) {
			Operator<float>& op = f->get32();
			op.use_fast         = fast;
			e1.record(s);
			if (d_guess) {
				if (d_guess != d_out) { FI_CUDA(cudaMemcpyAsync(d_out, d_guess, N * sizeof(float), cudaMemcpyDeviceToDevice, s)); }
			} else {
				FI_CUDA(cudaMemsetAsync(d_out, 0, N * sizeof(float), s));
			}
			// fp32 outer CG, watched: a fourth-order operator on a large lattice has cond ~ n^4, and fp32 vectors stop
			// describing the solution long before a tight tolerance is met (C3, 2048^2: breakdown after a handful of
			// iterations).  The solve then continues from the fp32 iterate with the fp64 outer CG (same fp32 V-cycle).
			r = mgpcg_solve<float>(op, mg, nullptr, d_out, o.tolerance, o.max_iterations, s, 4);
			const bool budget_left = o.max_iterations <= 0 || r.iterations < o.max_iterations;
			if (!r.converged && !r.zero_rhs && r.stalled && budget_left) {
				widened_after = r.iterations;
				start_wide    = true;
			}
		}
		if (start_wide) {  // FI_F64 and FI_MIXED (and a widened FI_F32): fp64 outer CG around the fp32 V-cycle
			Operator<double>& op = f->get64();
			op.use_fast          = fast;
			if (widened_after < 0) { e1.record(s); }
			DevBuf<double> x(N);
			const float*   from = widened_after >= 0 ? d_out : d_guess;
			if (from) { convert(from, x.data(), N, s); } else { x.zero(s); }
			const long long cap = o.max_iterations > 0 ? o.max_iterations - std::max<long long>(widened_after, 0) : 0;
			const PcgResult w   = mgpcg_solve<double>(op, mg, nullptr, x.data(), o.tolerance, cap, s);
			convert(x.data(), d_out, N, s);
			if (widened_after >= 0) {
				PcgResult tot        = w;
				tot.iterations       = r.iterations + w.iterations;
				tot.solve_ms         = r.solve_ms + w.solve_ms;
				tot.initial_residual = r.initial_residual;
				r                    = tot;
			} else {
				r = w;
			}
		}
		e1.sync();
		const double setup = e1.ms_since(e0);
		fill_stats(st, r, fresh ? setup : 0.0, f->op32 ? f->op32->data.nocc : 0, f->op32 ? f->op32->data.nrows : 0);
		if (st) {
			st->widened_after = widened_after;
			st->outer_sweeps  = mg.opt.gamma;  // the cycle the solve ended with: 1 V, 2 W (a W-cycle CG breaks down on is demoted)
		}
		FI_CUDA(cudaStreamSynchronize(s));
		return;
	}
	if (o.precision == FI_F32) {
		const bool fresh = !f->op32;
		Operator<float>& op = f->get32();
		op.use_fast = fast;
		if (d_guess) {
			if (d_guess != d_out) { FI_CUDA(cudaMemcpyAsync(d_out, d_guess, N * sizeof(float), cudaMemcpyDeviceToDevice, s)); }
		} else {
			FI_CUDA(cudaMemsetAsync(d_out, 0, N * sizeof(float), s));
		}
		op.guess_is_zero  = d_guess == nullptr;
		const PcgResult r = pcg_solve<float>(op, nullptr, d_out, o.tolerance, o.max_iterations, o.check_every, true, s);
		fill_stats(st, r, fresh ? op.setup_ms : 0.0, op.data.nocc, op.data.nrows);
	} else if (o.precision == FI_F64) {
		const bool fresh = !f->op64;
		Operator<double>& op = f->get64();
		op.use_fast = fast;
		DevBuf<double> x(N);
		if (d_guess) { convert(d_guess, x.data(), N, s); } else { x.zero(s); }
		op.guess_is_zero  = d_guess == nullptr;
		const PcgResult r = pcg_solve<double>(op, nullptr, x.data(), o.tolerance, o.max_iterations, o.check_every, true, s);
		convert(x.data(), d_out, N, s);
		fill_stats(st, r, fresh ? op.setup_ms : 0.0, op.data.nocc, op.data.nrows);
	} else if (o.precision == FI_MIXED) {
		// fp64 iterative refinement around fp32 PCG: x += solve32(b - A64 x)
		const bool fresh = !f->op64 || !f->op32;
		Operator<double>& op64 = f->get64();
		Operator<float>&  op32 = f->get32();
		op64.use_fast = op32.use_fast = fast;
		DevBuf<double> x(N), r64(N);
		DevBuf<float>  r32(N), e32(N);
		if (d_guess) { convert(d_guess, x.data(), N, s); } else { x.zero(s); }
		const double tol   = o.tolerance > 0 ? o.tolerance : 2.220446049250313e-16;
		const double itol  = o.refine_inner_tolerance > 0 ? o.refine_inner_tolerance : 1e-3;
		const int    outer = o.refine_max_outer > 0 ? o.refine_max_outer : 20;
		long long    max_it = o.max_iterations > 0 ? o.max_iterations : 2 * N;
		PcgResult    tot;
		cudaEvent_t  e0, e1;
		FI_CUDA(cudaEventCreate(&e0));
		FI_CUDA(cudaEventCreate(&e1));
		FI_CUDA(cudaEventRecord(e0, s));
		int sweeps = 0;
		for (;; ++sweeps) {
			double rr = 0, bb = 0;
			residual<double>(op64, nullptr, x.data(), r64.data(), &rr, &bb, s);
			const double rel = bb > 0 ? std::sqrt(rr / bb) : 0.0;
			if (sweeps == 0) { tot.initial_residual = rel; }
			tot.rel_residual = tot.true_residual = rel;
			if (bb == 0.0) { x.zero(s); tot.zero_rhs = tot.converged = true; break; }
			if (rel <= tol) { tot.converged = true; break; }
			if (sweeps >= outer || tot.iterations >= max_it) { break; }
			convert(r64.data(), r32.data(), N, s);
			e32.zero(s);
			// never ask the inner solve for more than the outer target needs
			const double    inner = std::max(itol, 0.5 * tol / rel);
			op32.guess_is_zero = true;
			const PcgResult r = pcg_solve<float>(op32, r32.data(), e32.data(), inner, max_it - tot.iterations, o.check_every, false, s);
			tot.iterations += r.iterations;
			axpy_f32_into_f64(e32.data(), x.data(), N, s);
			if (r.iterations == 0) { break; }
		}
		FI_CUDA(cudaEventRecord(e1, s));
		FI_CUDA(cudaEventSynchronize(e1));
		float ms = 0;
		FI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
		cudaEventDestroy(e0);
		cudaEventDestroy(e1);
		tot.solve_ms = ms;
		convert(x.data(), d_out, N, s);
		fill_stats(st, tot, fresh ? op64.setup_ms + op32.setup_ms : 0.0, op64.data.nocc, op64.data.nrows);
		if (st) { st->outer_sweeps = sweeps; }
	} else {
		throw Error{FI_ERR_INVALID, "unknown precision"};
	}
	FI_CUDA(cudaStreamSynchronize(s));
}

__global__ void scale_positions_kernel(int D, int64_t n, const float* __restrict__ unit, float* __restrict__ out, float sx, float sy, float sz)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n * D) { return; }
	const int   d = static_cast<int>(i % D);
	const float s = d == 0 ? sx : (d == 1 ? sy : sz);
	out[i]        = unit[i] * s;  // on_lattice, reference src/sdf_field.cpp:198-210: pos *= (resolution - 1.0f)
}

}  // namespace

}  // namespace fi

using namespace fi;

extern "C" {

int fi_abi_version(void) { return FI_B200_ABI_VERSION; }

const char* fi_last_error(void) { return t_last_error.c_str(); }

int fi_device_count(int32_t* count)
{
	return guarded([&] {
		FI_REQUIRE(count != nullptr, FI_ERR_INVALID, "count is null");
		int c = 0;
		FI_CUDA(cudaGetDeviceCount(&c));
		*count = c;
	});
}

int fi_set_device(int32_t device)
{
	return guarded([&] { FI_CUDA(cudaSetDevice(device)); });
}

void fi_weights_default(fi_weights* w)
{
	if (!w) { return; }
	*w = fi_weights{1.0f, 1.0f, 0.0f, 0.0f, 0.5f, 0.0f, 0.0f, 0.0f, FI_VALUE_LINEAR_INTERPOLATION, FI_GRADIENT_CELL_EDGES};
}

void fi_solve_options_default(fi_solve_options* o)
{
	if (!o) { return; }
	std::memset(o, 0, sizeof(*o));
	o->precision              = FI_F32;
	o->max_iterations         = 0;
	o->tolerance              = 1e-3;  // SolveOptions::error_tolerance, reference sparse_linear.hpp:72
	o->check_every            = 32;
	o->use_fast_stencil       = 1;
	o->refine_max_outer       = 20;
	o->refine_inner_tolerance = 1e-3;
	o->preconditioner         = FI_PRECOND_JACOBI;
	o->mg_smoothing_steps     = 0;  // by the smoothness model and the lattice: fi::default_mg_options
	o->mg_cheb_ratio          = 12.0;
}

int fi_field_create(int32_t ndim, const int32_t* sizes, fi_field** out)
{
	return guarded([&] {
		FI_REQUIRE(out != nullptr, FI_ERR_INVALID, "out is null");
		*out = nullptr;
		*out = create_impl(ndim, sizes);
	});
}

int fi_field_destroy(fi_field* f)
{
	return guarded([&] {
		TraceScope trace("fi_field_destroy");
		delete f;
	});
}

int fi_field_clone(const fi_field* f, fi_field** out)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr && out != nullptr, FI_ERR_INVALID, "null argument");
		*out = nullptr;
		std::unique_ptr<fi_field> c(create_impl(f->g.ndim, f->g.size));
		c->segs  = f->segs;
		c->rows  = f->rows;
		c->model = f->model;
		c->fast  = f->fast;
		cudaStream_t s = c->stream;
		FI_CUDA(cudaStreamSynchronize(f->stream));  // the source's point records are complete
		auto copy = [&](auto& dst, const auto& src) {
			dst.resize(src.size());
			if (src.size()) { FI_CUDA(cudaMemcpyAsync(dst.data(), src.data(), src.size() * sizeof(*src.data()), cudaMemcpyDeviceToDevice, s)); }
		};
		copy(c->pts.pos, f->pts.pos);
		copy(c->pts.grad, f->pts.grad);
		copy(c->pts.value, f->pts.value);
		copy(c->pts.vw, f->pts.vw);
		copy(c->pts.gw, f->pts.gw);
		copy(c->pts.kind, f->pts.kind);
		c->pts.count = f->pts.count;
		FI_CUDA(cudaStreamSynchronize(s));
		*out = c.release();
	});
}

int fi_field_add_model(fi_field* f, const fi_weights* w)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		add_model_impl(f, w);
	});
}

int fi_field_add_points(fi_field* f, float value_weight, int32_t value_kernel, float gradient_weight, int32_t gradient_kernel,
                        int64_t num_points, const float* positions, const float* normals, const float* point_weights,
                        const float* values, int32_t loc, int64_t* rows_added)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		add_points_impl(f, value_weight, value_kernel, gradient_weight, gradient_kernel, num_points, positions, normals,
		                point_weights, values, loc, rows_added);
	});
}

int fi_field_add_rows(fi_field* f, int64_t num_rows, int64_t num_triplets, const int32_t* trip_row, const int32_t* trip_col,
                      const float* trip_val, const float* rhs)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		FI_REQUIRE(num_rows >= 0 && num_triplets >= 0, FI_ERR_INVALID, "negative count");
		if (num_rows == 0) { return; }
		FI_REQUIRE(trip_row && trip_col && trip_val && rhs, FI_ERR_INVALID, "null row arrays");
		// validate everything before the first push: a call that fails leaves the row store exactly as it was
		for (int64_t k = 0; k < num_triplets; ++k) {
			FI_REQUIRE(0 <= trip_col[k] && trip_col[k] < f->g.N, FI_ERR_INVALID, "column out of range");
			FI_REQUIRE(0 <= trip_row[k] && trip_row[k] < num_rows && (k == 0 || trip_row[k - 1] <= trip_row[k]), FI_ERR_INVALID,
			           "trip_row must be non-decreasing and < num_rows");
		}
		HostRows& R  = f->rows;
		const int64_t r0 = R.rows();
		R.col.reserve(R.col.size() + static_cast<size_t>(num_triplets));
		R.val.reserve(R.val.size() + static_cast<size_t>(num_triplets));
		R.ptr.reserve(R.ptr.size() + static_cast<size_t>(num_rows));
		R.rhs.reserve(R.rhs.size() + static_cast<size_t>(num_rows));
		int64_t at = 0;
		for (int64_t r = 0; r < num_rows; ++r) {
			while (at < num_triplets && trip_row[at] == r) {
				R.col.push_back(trip_col[at]);
				R.val.push_back(trip_val[at]);
				++at;
			}
			R.ptr.push_back(R.col.size());
			R.rhs.push_back(rhs[r]);
		}
		Segment sg;
		sg.kind = Segment::kRows;
		sg.r0   = r0;
		sg.r1   = R.rows();
		f->segs.push_back(sg);
		f->invalidate();
	});
}

int fi_field_add_border_distance(fi_field* f, float weight, int64_t num_points, const float* positions, int32_t loc, int64_t* rows_added)
{
	return guarded([&] {
		TraceScope trace("fi_field_add_border_distance");
		if (rows_added) { *rows_added = 0; }
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		FI_REQUIRE(loc == FI_HOST || loc == FI_DEVICE, FI_ERR_INVALID, "add_border_distance: unknown loc");
		FI_REQUIRE(num_points >= 1, FI_ERR_INVALID, "add_border_distance: no points");
		FI_REQUIRE(positions != nullptr, FI_ERR_INVALID, "positions is null");
		FI_REQUIRE(num_points < (1ll << 32), FI_ERR_RANGE, "add_border_distance: 2^32 points or more");
		FI_REQUIRE(f->g.N <= INT32_MAX, FI_ERR_RANGE, "add_border_distance: more than 2^31 - 1 nodes (columns are int32)");
		if (weight == 0) { return; }  // add_equation drops the row
		Staged<float> p(positions, static_cast<size_t>(num_points) * f->g.ndim, loc, f->stream);
		HostRows&     R  = f->rows;
		const int64_t r0 = R.rows();
		append_border_rows(f->g, weight, num_points, p.ptr, R, f->stream);
		Segment sg;
		sg.kind = Segment::kRows;
		sg.r0   = r0;
		sg.r1   = R.rows();
		f->segs.push_back(sg);
		f->invalidate();
		if (rows_added) { *rows_added = sg.r1 - sg.r0; }
	});
}

int fi_sdf_from_points(int32_t ndim, const int32_t* sizes, const fi_weights* w, int64_t num_points, const float* positions,
                       const float* normals, const float* point_weights, int32_t loc, fi_field** out)
{
	return guarded([&] {
		FI_REQUIRE(out != nullptr, FI_ERR_INVALID, "out is null");
		*out = nullptr;
		check_weights(w);
		FI_REQUIRE(positions != nullptr || num_points == 0, FI_ERR_INVALID, "positions is null");  // CHECK_NOTNULL_F, :382
		std::unique_ptr<fi_field> f(create_impl(ndim, sizes));
		add_model_impl(f.get(), w);
		add_points_impl(f.get(), w->data_pos, w->value_kernel, w->data_gradient, w->gradient_kernel, num_points, positions,
		                normals, point_weights, nullptr, loc, nullptr);
		*out = f.release();
	});
}

int fi_field_counts(fi_field* f, int64_t* num_rows, int64_t* num_triplets)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		int64_t r = 0, t = 0;
		for (Segment& sg : f->segs) {
			segment_counts(f, sg);
			r += sg.rows;
			t += sg.trips;
		}
		if (num_rows) { *num_rows = r; }
		if (num_triplets) { *num_triplets = t; }
	});
}

// Exports the rows numbered >= row_begin (which must be where one builder call ended and the next began).
static void export_impl(fi_field* f, int64_t row_begin, fi_triplet* triplets, float* rhs)
{
	FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
	FI_REQUIRE(row_begin >= 0, FI_ERR_INVALID, "negative row_begin");
	int64_t R = 0, T = 0;
	for (Segment& sg : f->segs) {
		segment_counts(f, sg);
		R += sg.rows;
		T += sg.trips;
	}
	FI_REQUIRE(R <= INT32_MAX && T <= INT32_MAX && f->g.N <= INT32_MAX, FI_ERR_RANGE,
	           "system does not fit the reference's int32 triplet view");
	// first segment to export
	size_t  first = 0;
	int64_t row_base = 0, trip_base = 0;
	while (first < f->segs.size() && row_base < row_begin) {
		row_base += f->segs[first].rows;
		trip_base += f->segs[first].trips;
		++first;
	}
	// builder calls that appended nothing leave empty segments at the boundary: skipping them is harmless
	FI_REQUIRE(row_base == row_begin || (first == f->segs.size() && row_begin == R), FI_ERR_INVALID,
	           "row_begin is not a boundary between builder calls");
	const int64_t outR = R - row_base, outT = T - trip_base;
	if (outR == 0 && outT == 0) { return; }
	FI_REQUIRE((triplets || outT == 0) && (rhs || outR == 0), FI_ERR_INVALID, "output buffers are null");
	cudaStream_t       s = f->stream;
	DevBuf<fi_triplet> d_trips(std::max<int64_t>(outT, 1));
	DevBuf<float>      d_rhs(std::max<int64_t>(outR, 1));
	const int64_t      row0 = row_base, trip0 = trip_base;
	fi_triplet*        dt = d_trips.data() - trip0;  // indexed by absolute triplet number below
	float*             dr = d_rhs.data() - row0;
	for (size_t k = first; k < f->segs.size(); ++k) {
		Segment& sg = f->segs[k];
		if (sg.kind == Segment::kModel) {
			DevBuf<uint64_t> ro(f->g.N), to(f->g.N);
			uint64_t         hr = 0, ht = 0;
			count_model_rows(f->g, sg.w, ro.data(), to.data(), &hr, &ht, s);
			FI_REQUIRE(static_cast<int64_t>(hr) == sg.rows && static_cast<int64_t>(ht) == sg.trips, FI_ERR_INVALID,
			           "internal: model row count mismatch");
			emit_model_rows(f->g, sg.w, ro.data(), to.data(), row_base, trip_base, dt, dr, s);
			FI_CUDA(cudaStreamSynchronize(s));
		} else if (sg.kind == Segment::kPoints) {
			const int64_t    n = sg.p1 - sg.p0;
			DevBuf<uint64_t> ro(std::max<int64_t>(n, 1)), to(std::max<int64_t>(n, 1));
			uint64_t         hr = 0, ht = 0;
			count_point_rows(f->g, view(f->pts), sg.p0, sg.p1, ro.data(), to.data(), &hr, &ht, s);
			emit_point_rows(f->g, view(f->pts), sg.p0, sg.p1, ro.data(), to.data(), row_base, trip_base, dt, dr, s);
			FI_CUDA(cudaStreamSynchronize(s));
		} else {
			std::vector<fi_triplet> ht(static_cast<size_t>(sg.trips));
			size_t                  at = 0;
			for (int64_t r = sg.r0; r < sg.r1; ++r) {
				for (uint64_t kk = f->rows.ptr[r]; kk < f->rows.ptr[r + 1]; ++kk) {
					ht[at++] = fi_triplet{static_cast<int32_t>(row_base + (r - sg.r0)), f->rows.col[kk], f->rows.val[kk]};
				}
			}
			if (!ht.empty()) {
				FI_CUDA(cudaMemcpyAsync(dt + trip_base, ht.data(), ht.size() * sizeof(fi_triplet), cudaMemcpyHostToDevice, s));
			}
			if (sg.rows > 0) {
				FI_CUDA(cudaMemcpyAsync(dr + row_base, f->rows.rhs.data() + sg.r0, sg.rows * sizeof(float), cudaMemcpyHostToDevice, s));
			}
			FI_CUDA(cudaStreamSynchronize(s));
		}
		row_base += sg.rows;
		trip_base += sg.trips;
	}
	if (outT > 0) { FI_CUDA(cudaMemcpyAsync(triplets, d_trips.data(), outT * sizeof(fi_triplet), cudaMemcpyDeviceToHost, s)); }
	if (outR > 0) { FI_CUDA(cudaMemcpyAsync(rhs, d_rhs.data(), outR * sizeof(float), cudaMemcpyDeviceToHost, s)); }
	FI_CUDA(cudaStreamSynchronize(s));
}

int fi_field_export(fi_field* f, fi_triplet* triplets, float* rhs)
{
	return guarded([&] { export_impl(f, 0, triplets, rhs); });
}

int fi_field_export_rows(fi_field* f, int64_t row_begin, fi_triplet* triplets, float* rhs)
{
	return guarded([&] { export_impl(f, row_begin, triplets, rhs); });
}

int fi_field_use_fast_stencil(fi_field* f, int32_t enable)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		f->fast = enable;
	});
}

int fi_field_apply(fi_field* f, int32_t precision, const void* x, void* y)
{
	return guarded([&] {
		FI_REQUIRE(f && x && y, FI_ERR_INVALID, "null argument");
		const int64_t N = f->g.N;
		cudaStream_t  s = f->stream;
		if (precision == FI_F32) {
			Operator<float>& op = f->get32();
			op.use_fast = f->fast;
			DevBuf<float>    dx(N), dy(N);
			FI_CUDA(cudaMemcpyAsync(dx.data(), x, N * sizeof(float), cudaMemcpyHostToDevice, s));
			op.apply(dx.data(), dy.data(), nullptr, nullptr, s);
			FI_CUDA(cudaMemcpyAsync(y, dy.data(), N * sizeof(float), cudaMemcpyDeviceToHost, s));
		} else if (precision == FI_F64) {
			Operator<double>& op = f->get64();
			op.use_fast = f->fast;
			DevBuf<double>    dx(N), dy(N);
			FI_CUDA(cudaMemcpyAsync(dx.data(), x, N * sizeof(double), cudaMemcpyHostToDevice, s));
			op.apply(dx.data(), dy.data(), nullptr, nullptr, s);
			FI_CUDA(cudaMemcpyAsync(y, dy.data(), N * sizeof(double), cudaMemcpyDeviceToHost, s));
		} else {
			throw Error{FI_ERR_INVALID, "precision must be FI_F32 or FI_F64"};
		}
		FI_CUDA(cudaStreamSynchronize(s));
	});
}

static int copy_vector(fi_field* f, int32_t precision, void* out, int which)
{
	return guarded([&] {
		FI_REQUIRE(f && out, FI_ERR_INVALID, "null argument");
		const int64_t N = f->g.N;
		if (precision == FI_F32) {
			Operator<float>& op = f->get32();
			FI_CUDA(cudaMemcpy(out, which == 0 ? op.atb.data() : op.diag.data(), N * sizeof(float), cudaMemcpyDeviceToHost));
		} else if (precision == FI_F64) {
			Operator<double>& op = f->get64();
			FI_CUDA(cudaMemcpy(out, which == 0 ? op.atb.data() : op.diag.data(), N * sizeof(double), cudaMemcpyDeviceToHost));
		} else {
			throw Error{FI_ERR_INVALID, "precision must be FI_F32 or FI_F64"};
		}
	});
}

int fi_field_rhs(fi_field* f, int32_t precision, void* atb) { return copy_vector(f, precision, atb, 0); }
int fi_field_diagonal(fi_field* f, int32_t precision, void* diag) { return copy_vector(f, precision, diag, 1); }

int fi_field_solve(fi_field* f, const fi_solve_options* opt, const float* guess, float* solution, int32_t loc, fi_solve_stats* stats)
{
	return guarded([&] {
		TraceScope trace("fi_field_solve");
		FI_REQUIRE(f && solution, FI_ERR_INVALID, "null argument");
		fi_solve_options o;
		if (opt) { o = *opt; } else { fi_solve_options_default(&o); }
		const int64_t N = f->g.N;
		if (loc == FI_DEVICE) {
			// the update and stencil kernels access the solution (and the guess, when it is the same buffer) in 16-byte packs
			FI_REQUIRE((reinterpret_cast<uintptr_t>(solution) & 15u) == 0 && (reinterpret_cast<uintptr_t>(guess) & 15u) == 0, FI_ERR_INVALID,
			           "FI_DEVICE solution / guess buffers must be 16-byte aligned");
			solve_device(f, o, guess, solution, stats);
		} else {
			DevBuf<float> d(N);
			if (guess) { FI_CUDA(cudaMemcpyAsync(d.data(), guess, N * sizeof(float), cudaMemcpyHostToDevice, f->stream)); }
			solve_device(f, o, guess ? d.data() : nullptr, d.data(), stats);
			FI_CUDA(cudaMemcpyAsync(solution, d.data(), N * sizeof(float), cudaMemcpyDeviceToHost, f->stream));
			FI_CUDA(cudaStreamSynchronize(f->stream));
		}
	});
}

int fi_field_solve_tiled(fi_field* f, const fi_solve_options* opt, int32_t tile, int32_t tile_size, int32_t cg, const float* guess,
                         float* solution, int32_t loc, fi_solve_stats* stats, fi_solve_stats* tile_stats)
{
	return guarded([&] {
		TraceScope trace("fi_field_solve_tiled");
		FI_REQUIRE(f && solution, FI_ERR_INVALID, "null argument");
		FI_REQUIRE(guess != nullptr, FI_ERR_INVALID, "incomplete guess");  // sparse_linear.cpp:402-405
		fi_solve_options o;
		if (opt) { o = *opt; } else { fi_solve_options_default(&o); }
		FI_REQUIRE(o.precision == FI_F32 || o.precision == FI_F64 || o.precision == FI_MIXED, FI_ERR_INVALID, "unknown precision");
		const int64_t N = f->g.N;
		cudaStream_t  s = f->stream;
		DevBuf<float> staged;
		float*        d_x = solution;
		if (loc == FI_DEVICE) {
			FI_REQUIRE((reinterpret_cast<uintptr_t>(solution) & 15u) == 0, FI_ERR_INVALID, "FI_DEVICE solution buffer must be 16-byte aligned");
			if (guess != solution) { FI_CUDA(cudaMemcpyAsync(solution, guess, N * sizeof(float), cudaMemcpyDeviceToDevice, s)); }
		} else {
			staged.resize(N);
			d_x = staged.data();
			FI_CUDA(cudaMemcpyAsync(d_x, guess, N * sizeof(float), cudaMemcpyHostToDevice, s));
		}
		if (stats) { std::memset(stats, 0, sizeof(*stats)); }
		if (tile_stats) { std::memset(tile_stats, 0, sizeof(*tile_stats)); }
		if (tile) {  // sparse_linear.cpp:423-425
			if (o.precision == FI_F32) {
				const bool       fresh = !f->op32;
				Operator<float>& op    = f->get32();
				op.use_fast            = o.use_fast_stencil;
				const PcgResult r      = tile_phase<float>(op, tile_size, d_x, 1e-6, 0, o.check_every, s);
				fill_stats(tile_stats, r, fresh ? op.setup_ms : 0.0, op.data.nocc, op.data.nrows);
			} else {
				const bool        fresh = !f->op64;
				Operator<double>& op    = f->get64();
				op.use_fast             = o.use_fast_stencil;
				DevBuf<double> x(N);
				convert(d_x, x.data(), N, s);
				const PcgResult r = tile_phase<double>(op, tile_size, x.data(), 1e-12, 0, o.check_every, s);
				convert(x.data(), d_x, N, s);
				fill_stats(tile_stats, r, fresh ? op.setup_ms : 0.0, op.data.nocc, op.data.nrows);
			}
		}
		if (cg) { solve_device(f, o, d_x, d_x, stats); }  // :427-440
		if (loc != FI_DEVICE) { FI_CUDA(cudaMemcpyAsync(solution, d_x, N * sizeof(float), cudaMemcpyDeviceToHost, s)); }
		FI_CUDA(cudaStreamSynchronize(s));
	});
}

int fi_field_jacobi(fi_field* f, const float* guess, int32_t num_iterations, float weight, float* solution)
{
	return guarded([&] {
		FI_REQUIRE(f && guess && solution, FI_ERR_INVALID, "null argument");
		const int64_t N = f->g.N;
		if (num_iterations <= 0) {  // reference sparse_linear.cpp:220: returns the guess
			if (solution != guess) { std::memcpy(solution, guess, N * sizeof(float)); }
			return;
		}
		Operator<float>& op = f->get32();
		DevBuf<float>    x(N);
		FI_CUDA(cudaMemcpyAsync(x.data(), guess, N * sizeof(float), cudaMemcpyHostToDevice, f->stream));
		jacobi_sweeps<float>(op, x.data(), num_iterations, weight, f->stream);
		FI_CUDA(cudaMemcpyAsync(solution, x.data(), N * sizeof(float), cudaMemcpyDeviceToHost, f->stream));
		FI_CUDA(cudaStreamSynchronize(f->stream));
	});
}

int fi_upscale_field(int32_t ndim, const int32_t* small_sizes, const int32_t* large_sizes, const float* small_field,
                     float* large_field, int32_t loc)
{
	return guarded([&] {
		FI_REQUIRE(1 <= ndim && ndim <= kMaxDim, FI_ERR_INVALID, "ndim must be 1..3");
		FI_REQUIRE(small_sizes && large_sizes && small_field && large_field, FI_ERR_INVALID, "null argument");
		for (int d = 0; d < ndim; ++d) { FI_REQUIRE(small_sizes[d] >= 1 && large_sizes[d] >= 1, FI_ERR_INVALID, "size must be >= 1"); }
		const Geom gs = make_geom(ndim, small_sizes), gl = make_geom(ndim, large_sizes);
		if (loc == FI_DEVICE) {
			upscale_device(gs, gl, small_field, large_field, 1.0f, nullptr);
			FI_CUDA(cudaStreamSynchronize(nullptr));
		} else {
			DevBuf<float> a(gs.N), b(gl.N);
			FI_CUDA(cudaMemcpy(a.data(), small_field, gs.N * sizeof(float), cudaMemcpyHostToDevice));
			upscale_device(gs, gl, a.data(), b.data(), 1.0f, nullptr);
			FI_CUDA(cudaMemcpy(large_field, b.data(), gl.N * sizeof(float), cudaMemcpyDeviceToHost));
		}
	});
}

int fi_error_map(int64_t num_triplets, const fi_triplet* triplets, int64_t num_columns, const float* solution, int64_t num_rows,
                 const float* rhs, float* heatmap)
{
	return guarded([&] {
		FI_REQUIRE(num_triplets >= 0 && num_columns >= 0 && num_rows >= 0, FI_ERR_INVALID, "negative count");
		FI_REQUIRE((triplets || num_triplets == 0) && (solution || num_columns == 0) && (rhs || num_rows == 0) && (heatmap || num_columns == 0),
		           FI_ERR_INVALID, "null argument");
		error_map(num_triplets, triplets, num_columns, solution, num_rows, rhs, heatmap);
	});
}

int fi_field_error_map(fi_field* f, const float* solution, int32_t loc, float* heatmap, double* row_error_sums)
{
	return guarded([&] {
		TraceScope trace("fi_field_error_map");
		FI_REQUIRE(f && solution && heatmap, FI_ERR_INVALID, "field_error_map: null argument");
		FI_REQUIRE(loc == FI_HOST || loc == FI_DEVICE, FI_ERR_INVALID, "field_error_map: unknown loc");
		bool emitted_rows = false;  // point and caller rows go through int32 columns (the emitters' triplets)
		for (const Segment& sg : f->segs) {
			emitted_rows = emitted_rows || (sg.kind == Segment::kPoints && sg.p1 > sg.p0) || (sg.kind == Segment::kRows && sg.r1 > sg.r0);
		}
		FI_REQUIRE(!emitted_rows || f->g.N <= INT32_MAX, FI_ERR_RANGE, "field_error_map: point or caller rows on more than 2^31 - 1 nodes");
		const int64_t N = f->g.N;
		cudaStream_t  s = f->stream;
		Staged<float> x(solution, static_cast<size_t>(N), loc, s);
		DevBuf<float> own;
		float*        heat = heatmap;
		if (loc != FI_DEVICE) {
			own.resize(N);
			heat = own.data();
		}
		FI_CUDA(cudaMemsetAsync(heat, 0, N * sizeof(float), s));
		DevBuf<double> sums(3);
		sums.zero(s);
		ErrorMapScratch sc;
		for (const Segment& sg : f->segs) {  // in builder-call order: every column receives its terms in global triplet order
			if (sg.kind == Segment::kModel) {
				model_error_map(f->g, sg.w, x.ptr, heat, sums.data() + 0, sc, s);
			} else if (sg.kind == Segment::kPoints) {
				point_error_map(f->g, view(f->pts), sg.p0, sg.p1, x.ptr, heat, sums.data() + 1, sc, s);
			} else {
				caller_rows_error_map(f->g, f->rows, sg.r0, sg.r1, x.ptr, heat, sums.data() + 2, sc, s);
			}
		}
		double h[3];
		FI_CUDA(cudaMemcpyAsync(h, sums.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
		if (loc != FI_DEVICE) { FI_CUDA(cudaMemcpyAsync(heatmap, heat, N * sizeof(float), cudaMemcpyDeviceToHost, s)); }
		FI_CUDA(cudaStreamSynchronize(s));
		if (row_error_sums) { std::memcpy(row_error_sums, h, sizeof(h)); }
	});
}

int fi_marching_squares(int32_t width, int32_t height, const float* values, float iso, int32_t loc, float* lines, int64_t capacity_segments,
                        int64_t* num_segments, float* area)
{
	return guarded([&] {
		FI_REQUIRE(width >= 1 && height >= 1 && values && num_segments, FI_ERR_INVALID, "marching squares: bad argument");
		FI_REQUIRE(lines == nullptr || capacity_segments >= 0, FI_ERR_INVALID, "marching squares: negative capacity");
		*num_segments = 0;
		if (area) { *area = 0.0f; }
		cudaStream_t  s = nullptr;
		Staged<float> v(values, static_cast<size_t>(width) * height, loc, s);
		// the count decides how many segments exist; they are materialised on the device when the caller wants them or the area
		const int64_t n = marching_squares_device(width, height, v.ptr, iso, nullptr, 0, s);
		*num_segments   = n;
		FI_REQUIRE(lines == nullptr || n <= capacity_segments, FI_ERR_RANGE, "marching squares: segment buffer too small");
		if (n == 0 || (lines == nullptr && area == nullptr)) { return; }
		DevBuf<float> own;
		float*        d_lines = lines;
		if (lines == nullptr || loc != FI_DEVICE) {
			own.resize(static_cast<size_t>(n) * 4);
			d_lines = own.data();
		}
		marching_squares_device(width, height, v.ptr, iso, d_lines, n, s);
		if (area) { *area = static_cast<float>(area_twice_device(n, d_lines, s) / 2); }
		if (lines && loc != FI_DEVICE) { FI_CUDA(cudaMemcpy(lines, d_lines, static_cast<size_t>(n) * 4 * sizeof(float), cudaMemcpyDeviceToHost)); }
	});
}

int fi_calc_area(int64_t num_segments, const float* lines, int32_t loc, float* area)
{
	return guarded([&] {
		FI_REQUIRE(num_segments >= 0 && area && (lines || num_segments == 0), FI_ERR_INVALID, "calc_area: bad argument");
		cudaStream_t  s = nullptr;
		Staged<float> l(lines, static_cast<size_t>(num_segments) * 4, loc, s);
		*area = static_cast<float>(area_twice_device(num_segments, l.ptr, s) / 2);
	});
}

int fi_bicubic_upsample(int32_t width, int32_t height, const float* values, int32_t upsample, float* large, int32_t loc)
{
	return guarded([&] {
		FI_REQUIRE(width >= 1 && height >= 1 && values && large, FI_ERR_INVALID, "bicubic_upsample: bad argument");
		FI_REQUIRE(upsample > 1, FI_ERR_INVALID, "bicubic_upsample: upsample must be > 1 (src/sdf_field.cpp:557)");
		cudaStream_t  s = nullptr;
		const int64_t lw = static_cast<int64_t>(upsample) * width - upsample + 1, lh = static_cast<int64_t>(upsample) * height - upsample + 1;
		Staged<float> v(values, static_cast<size_t>(width) * height, loc, s);
		if (loc == FI_DEVICE) {
			bicubic_upsample_device(width, height, v.ptr, upsample, large, s);
			FI_CUDA(cudaStreamSynchronize(s));
		} else {
			DevBuf<float> out(static_cast<size_t>(lw * lh));
			bicubic_upsample_device(width, height, v.ptr, upsample, out.data(), s);
			FI_CUDA(cudaMemcpy(large, out.data(), static_cast<size_t>(lw * lh) * sizeof(float), cudaMemcpyDeviceToHost));
		}
	});
}

int fi_marching_cubes(const int32_t* sizes, const float* values, float iso, int32_t loc, float* vertices, float* normals, int64_t capacity_vertices,
                      int32_t* triangles, int64_t capacity_triangles, int64_t* num_vertices, int64_t* num_triangles)
{
	return guarded([&] {
		FI_REQUIRE(sizes && values && num_vertices && num_triangles, FI_ERR_INVALID, "marching cubes: null argument");
		FI_REQUIRE(sizes[0] >= 1 && sizes[1] >= 1 && sizes[2] >= 1, FI_ERR_INVALID, "marching cubes: size < 1");
		FI_REQUIRE(((vertices || normals) ? capacity_vertices >= 0 : true) && (triangles ? capacity_triangles >= 0 : true), FI_ERR_INVALID,
		           "marching cubes: negative capacity");
		*num_vertices  = 0;
		*num_triangles = 0;
		const int64_t nnodes = static_cast<int64_t>(sizes[0]) * sizes[1] * sizes[2];
		FI_REQUIRE(nnodes < (int64_t{1} << 31), FI_ERR_RANGE, "marching cubes: more than 2^31 - 1 nodes");
		cudaStream_t  s = nullptr;
		Staged<float> v(values, static_cast<size_t>(nnodes), loc, s);
		const bool    fill = vertices || normals || triangles;
		McCounts      n;
		if (loc == FI_DEVICE || !fill) {
			n = marching_cubes_device(sizes, v.ptr, iso, vertices, normals, capacity_vertices, triangles, capacity_triangles, s);
		} else {
			n = marching_cubes_device(sizes, v.ptr, iso, nullptr, nullptr, 0, nullptr, 0, s);
		}
		*num_vertices  = n.vertices;
		*num_triangles = n.triangles;
		FI_REQUIRE(!(vertices || normals) || n.vertices <= capacity_vertices, FI_ERR_RANGE, "marching cubes: vertex buffer too small");
		FI_REQUIRE(!triangles || n.triangles <= capacity_triangles, FI_ERR_RANGE, "marching cubes: triangle buffer too small");
		if (loc == FI_DEVICE || !fill || n.vertices == 0) { return; }
		const size_t  nv = static_cast<size_t>(n.vertices) * 3, nt = static_cast<size_t>(n.triangles) * 3;
		DevBuf<float> dv(vertices ? nv : 0), dn(normals ? nv : 0);
		DevBuf<int32_t> dt(triangles ? nt : 0);
		marching_cubes_device(sizes, v.ptr, iso, vertices ? dv.data() : nullptr, normals ? dn.data() : nullptr, n.vertices,
		                      triangles ? dt.data() : nullptr, n.triangles, s);
		if (vertices) { FI_CUDA(cudaMemcpy(vertices, dv.data(), nv * sizeof(float), cudaMemcpyDeviceToHost)); }
		if (normals) { FI_CUDA(cudaMemcpy(normals, dn.data(), nv * sizeof(float), cudaMemcpyDeviceToHost)); }
		if (triangles) { FI_CUDA(cudaMemcpy(triangles, dt.data(), nt * sizeof(int32_t), cudaMemcpyDeviceToHost)); }
	});
}

int fi_sample_field(int32_t ndim, const int32_t* sizes, const float* field, int64_t num_points, const float* positions,
                    int32_t gradient_kernel, int32_t loc, float* values, float* gradients)
{
	return guarded([&] {
		FI_REQUIRE(1 <= ndim && ndim <= kMaxDim, FI_ERR_INVALID, "sample_field: ndim must be 1..3");
		FI_REQUIRE(loc == FI_HOST || loc == FI_DEVICE, FI_ERR_INVALID, "sample_field: unknown loc");
		FI_REQUIRE(num_points >= 0, FI_ERR_INVALID, "sample_field: negative num_points");
		FI_REQUIRE(!gradients || (0 <= gradient_kernel && gradient_kernel <= 2), FI_ERR_INVALID, "sample_field: unknown gradient kernel");
		if (sizes) {
			for (int d = 0; d < ndim; ++d) { FI_REQUIRE(sizes[d] >= 1, FI_ERR_INVALID, "sample_field: size must be >= 1"); }
		}
		if (num_points == 0) { return; }
		FI_REQUIRE(sizes && field && positions, FI_ERR_INVALID, "sample_field: null argument");
		if (!values && !gradients) { return; }
		const Geom    g = make_geom(ndim, sizes);
		const size_t  np = static_cast<size_t>(num_points), nd = np * static_cast<size_t>(ndim);
		cudaStream_t  s = nullptr;
		Staged<float> x(field, static_cast<size_t>(g.N), loc, s), p(positions, nd, loc, s);
		if (loc == FI_DEVICE) {
			sample_field_device(g, num_points, p.ptr, x.ptr, gradient_kernel, values, gradients, s);
			FI_CUDA(cudaStreamSynchronize(s));
			return;
		}
		DevBuf<float> v(values ? np : 0), gr(gradients ? nd : 0);
		sample_field_device(g, num_points, p.ptr, x.ptr, gradient_kernel, values ? v.data() : nullptr, gradients ? gr.data() : nullptr, s);
		if (values) { FI_CUDA(cudaMemcpy(values, v.data(), np * sizeof(float), cudaMemcpyDeviceToHost)); }
		if (gradients) { FI_CUDA(cudaMemcpy(gradients, gr.data(), nd * sizeof(float), cudaMemcpyDeviceToHost)); }
	});
}

int fi_nearest_point_distance(int32_t ndim, int64_t num_points, const float* points, int64_t num_queries, const float* queries, int32_t loc,
                              float* distances, int64_t* nearest)
{
	return guarded([&] {
		TraceScope trace("fi_nearest_point_distance");
		FI_REQUIRE(1 <= ndim && ndim <= kMaxDim, FI_ERR_INVALID, "nearest_point_distance: ndim must be 1..3");
		FI_REQUIRE(loc == FI_HOST || loc == FI_DEVICE, FI_ERR_INVALID, "nearest_point_distance: unknown loc");
		FI_REQUIRE(num_points >= 0 && num_queries >= 0, FI_ERR_INVALID, "nearest_point_distance: negative count");
		FI_REQUIRE(num_points == 0 || points, FI_ERR_INVALID, "nearest_point_distance: points is null");
		FI_REQUIRE(num_queries == 0 || queries, FI_ERR_INVALID, "nearest_point_distance: queries is null");
		FI_REQUIRE(num_points < (1ll << 32), FI_ERR_RANGE, "nearest_point_distance: 2^32 points or more");
		if (num_queries == 0 || (!distances && !nearest)) { return; }
		const size_t  nq = static_cast<size_t>(num_queries);
		cudaStream_t  s  = nullptr;
		Staged<float> p(points, static_cast<size_t>(num_points) * ndim, loc, s), q(queries, nq * ndim, loc, s);
		if (loc == FI_DEVICE) {
			nearest_points_device(ndim, num_points, p.ptr, num_queries, q.ptr, distances, nearest, s);
			return;
		}
		DevBuf<float>   d(distances ? nq : 0);
		DevBuf<int64_t> k(nearest ? nq : 0);
		nearest_points_device(ndim, num_points, p.ptr, num_queries, q.ptr, distances ? d.data() : nullptr, nearest ? k.data() : nullptr, s);
		if (distances) { FI_CUDA(cudaMemcpyAsync(distances, d.data(), nq * sizeof(float), cudaMemcpyDeviceToHost, s)); }
		if (nearest) { FI_CUDA(cudaMemcpyAsync(nearest, k.data(), nq * sizeof(int64_t), cudaMemcpyDeviceToHost, s)); }
		FI_CUDA(cudaStreamSynchronize(s));
	});
}

int fi_sdf_solve_cascade(int32_t ndim, const int32_t* sizes, const fi_weights* w, int64_t num_points, const float* unit_positions,
                         const float* normals, const float* point_weights, const fi_cascade_options* opt, float* solution,
                         int32_t loc, fi_cascade_stats* stats)
{
	return guarded([&] {
		FI_REQUIRE(1 <= ndim && ndim <= kMaxDim, FI_ERR_INVALID, "ndim must be 1..3");
		FI_REQUIRE(sizes && opt && solution, FI_ERR_INVALID, "null argument");
		FI_REQUIRE(unit_positions != nullptr || num_points == 0, FI_ERR_INVALID, "positions is null");
		check_weights(w);
		const int factor   = opt->factor;
		const int coarsest = opt->coarsest_size > 0 ? opt->coarsest_size : 16;
		// level 0 = finest
		std::vector<std::vector<int32_t>> lv;
		lv.emplace_back(sizes, sizes + ndim);
		while (factor >= 2 && static_cast<int>(lv.size()) < 16 && (opt->max_levels <= 0 || static_cast<int>(lv.size()) < opt->max_levels)) {
			std::vector<int32_t> next(ndim);
			bool                 ok = true, shrunk = false;
			for (int d = 0; d < ndim; ++d) {
				next[d] = (lv.back()[d] + factor - 1) / factor;  // src/sdf_field.cpp:273
				ok      = ok && next[d] >= coarsest;
				shrunk  = shrunk || next[d] < lv.back()[d];
			}
			if (!ok || !shrunk) { break; }
			lv.push_back(next);
		}
		const int L = static_cast<int>(lv.size());
		if (stats) { std::memset(stats, 0, sizeof(*stats)); stats->levels = L; }

		cudaStream_t s0 = nullptr;  // staging on the default stream, then per-level field streams
		Staged<float> dunit(unit_positions, static_cast<size_t>(num_points) * ndim, loc, s0), dnrm(normals, static_cast<size_t>(num_points) * ndim, loc, s0);
		Staged<float> dpw(point_weights, num_points, loc, s0);
		FI_CUDA(cudaStreamSynchronize(s0));
		DevBuf<float> pos(std::max<int64_t>(num_points * ndim, 1));
		DevBuf<float> prev, cur;
		std::vector<int32_t> prev_sizes;
		cudaEvent_t e0, e1, t0;
		FI_CUDA(cudaEventCreate(&e0));
		FI_CUDA(cudaEventCreate(&e1));
		FI_CUDA(cudaEventCreate(&t0));
		FI_CUDA(cudaEventRecord(t0, s0));
		for (int l = L - 1; l >= 0; --l) {
			std::unique_ptr<fi_field> f(create_impl(ndim, lv[l].data()));
			cudaStream_t s = f->stream;
			FI_CUDA(cudaEventRecord(e0, s));
			if (num_points > 0) {
				const float sx = static_cast<float>(lv[l][0]) - 1.0f;
				const float sy = ndim > 1 ? static_cast<float>(lv[l][1]) - 1.0f : 0.0f;
				const float sz = ndim > 2 ? static_cast<float>(lv[l][2]) - 1.0f : 0.0f;
				FI_LAUNCH(scale_positions_kernel, div_up(num_points * ndim, 256), 256, 0, s, ndim, num_points, dunit.ptr, pos.data(), sx, sy, sz);
			}
			add_model_impl(f.get(), w);
			add_points_impl(f.get(), w->data_pos, w->value_kernel, w->data_gradient, w->gradient_kernel, num_points, pos.data(),
			                dnrm.ptr, dpw.ptr, nullptr, FI_DEVICE, nullptr);
			cur.resize(f->g.N);
			const float* guess = nullptr;
			if (l < L - 1) {
				const Geom gs = make_geom(ndim, prev_sizes.data());
				upscale_device(gs, f->g, prev.data(), cur.data(), static_cast<float>(factor), s);  // :284-288
				guess = cur.data();
			}
			fi_solve_options o = opt->fine;
			if (l > 0 && opt->coarse_tolerance > 0) { o.tolerance = opt->coarse_tolerance; }
			fi_solve_stats st{};
			solve_device(f.get(), o, guess, cur.data(), &st);
			FI_CUDA(cudaEventRecord(e1, s));
			FI_CUDA(cudaEventSynchronize(e1));
			float ms = 0;
			FI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
			if (stats) {
				stats->level_cells[l]            = f->g.N;
				stats->level_iterations[l]       = st.iterations;
				stats->level_ms[l]               = ms;
				stats->level_initial_residual[l] = st.initial_residual;
				stats->cell_iterations += f->g.N * st.iterations;
				stats->total_ms += ms;
				if (l == 0) { stats->finest = st; }
			}
			prev.swap(cur);
			prev_sizes = lv[l];
		}
		cudaEventDestroy(e0);
		cudaEventDestroy(e1);
		cudaEventDestroy(t0);
		const int64_t N = make_geom(ndim, sizes).N;
		FI_CUDA(cudaMemcpy(solution, prev.data(), N * sizeof(float), loc == FI_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost));
	});
}

int fi_comm_unique_id(void* id, int64_t capacity)
{
	return guarded([&] { comm_unique_id(id, capacity); });
}

int fi_comm_create(int32_t rank, int32_t world, const void* id, fi_comm** out)
{
	return guarded([&] {
		FI_REQUIRE(out != nullptr, FI_ERR_INVALID, "out is null");
		*out = nullptr;
		*out = comm_create(rank, world, id);
	});
}

int fi_comm_destroy(fi_comm* c)
{
	return guarded([&] { comm_destroy(c); });
}

int fi_slab_mg_plan(const int32_t* sizes, int32_t world, int32_t stencil_radius, int64_t gather_cells, int32_t* sharded_levels, int32_t* halo,
                    int32_t* level_sizes, int32_t* plane_ranges)
{
	return guarded([&] {
		FI_REQUIRE(sizes && sharded_levels && halo && level_sizes && plane_ranges && world >= 1 && world <= 64, FI_ERR_INVALID, "bad argument");
		const SlabMgPlan plan = plan_slab_multigrid(sizes, world, stencil_radius, gather_cells > 0 ? gather_cells : 3000000);
		*sharded_levels = plan.nd;
		*halo           = plan.halo;
		for (int l = 0; l <= plan.nd; ++l) {
			for (int d = 0; d < 3; ++d) { level_sizes[l * 3 + d] = plan.size[l][d]; }
			for (int k = 0; k < world; ++k) {
				plane_ranges[(l * world + k) * 2 + 0] = plan.own[l][k].first;
				plane_ranges[(l * world + k) * 2 + 1] = plan.own[l][k].second;
			}
		}
	});
}

int fi_slab_balanced_cuts(const int32_t* sizes, int32_t world, int64_t num_points, const float* positions, int32_t loc, double point_weight,
                          int32_t min_planes, int32_t* cuts)
{
	return guarded([&] {
		FI_REQUIRE(sizes && cuts && world >= 1 && world <= 64 && num_points >= 0 && (positions || num_points == 0), FI_ERR_INVALID, "bad argument");
		for (int d = 0; d < 3; ++d) { FI_REQUIRE(sizes[d] >= 1, FI_ERR_INVALID, "lattice size must be >= 1"); }
		balanced_cuts(sizes, world, num_points, positions, loc, point_weight > 0 ? point_weight : 30.0, min_planes, cuts);
	});
}

int fi_comm_set_slab_cuts(fi_comm* c, int32_t nz, const int32_t* cuts)
{
	return guarded([&] { comm_set_cuts(c, nz, cuts); });
}

int fi_slab_range(int32_t nz, int32_t world, int32_t rank, int32_t* z0, int32_t* z1)
{
	return guarded([&] {
		FI_REQUIRE(nz >= 1 && world >= 1 && rank >= 0 && rank < world && z0 && z1, FI_ERR_INVALID, "bad argument");
		int a = 0, b = 0;
		slab_range(nz, world, rank, &a, &b);
		*z0 = a;
		*z1 = b;
	});
}

int fi_slab_sdf_solve(fi_comm* c, const int32_t* sizes, const fi_weights* w, int64_t num_points, const float* positions, const float* normals,
                      const float* point_weights, int32_t loc, const fi_solve_options* opt, const float* guess_own, float* solution_own,
                      int32_t solution_loc, fi_solve_stats* stats)
{
	return guarded([&] {
		FI_REQUIRE(c && sizes && solution_own, FI_ERR_INVALID, "null argument");
		FI_REQUIRE(positions != nullptr || num_points == 0, FI_ERR_INVALID, "positions is null");
		check_weights(w);
		for (int d = 0; d < 3; ++d) { FI_REQUIRE(sizes[d] >= 1, FI_ERR_INVALID, "lattice size must be >= 1"); }
		fi_solve_options o;
		if (opt) { o = *opt; } else { fi_solve_options_default(&o); }
		slab_sdf_solve(c, sizes, *w, num_points, positions, normals, point_weights, loc, o, guess_own, solution_own, solution_loc, stats);
	});
}

int fi_trim_memory(void)
{
	return guarded([&] { pool_trim(); });
}

int64_t fi_cached_bytes(void) { return static_cast<int64_t>(pool_cached_bytes()); }

int64_t fi_kernel_launches(void) { return g_launches; }
void    fi_kernel_launches_reset(void) { g_launches = 0; }

int fi_field_time_iterations(fi_field* f, const fi_solve_options* opt, int32_t iterations, double* ms)
{
	return guarded([&] {
		FI_REQUIRE(f && ms && iterations > 0, FI_ERR_INVALID, "bad argument");
		fi_solve_options o;
		if (opt) { o = *opt; } else { fi_solve_options_default(&o); }
		if (o.precision == FI_F64) {
			Operator<double>& op = f->get64();
			op.use_fast = o.use_fast_stencil;
			time_kernels<double>(op, iterations, o.check_every, ms, f->stream);
		} else {
			Operator<float>& op = f->get32();
			op.use_fast = o.use_fast_stencil;
			time_kernels<float>(op, iterations, o.check_every, ms, f->stream);
		}
	});
}

int fi_field_mg_info(fi_field* f, const fi_solve_options* opt, fi_mg_info* out)
{
	return guarded([&] {
		FI_REQUIRE(f && out, FI_ERR_INVALID, "bad argument");
		fi_solve_options o;
		if (opt) { o = *opt; } else { fi_solve_options_default(&o); }
		mg_info(f->get_mg(o), out);
	});
}

int fi_field_mg_stage(fi_field* f, const fi_solve_options* opt, int32_t stage, int32_t level, int64_t count, const float* in, const float* in2, float* out)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		fi_solve_options o;
		if (opt) { o = *opt; } else { fi_solve_options_default(&o); }
		Multigrid& mg = f->get_mg(o);
		f->get32().use_fast = o.use_fast_stencil;  // the fine level's kernels as an FI_F32 solve with `o` picks them
		mg_stage(mg, stage, level, count, in, in2, out, f->stream);
	});
}

int fi_field_pcg_stage(fi_field* f, const fi_solve_options* opt, int32_t stage, int32_t par, int32_t pos, int32_t ring, int32_t count, int32_t loc,
                       void* const* vectors, fi_pcg_state* state, fi_pcg_report* report)
{
	return guarded([&] {
		FI_REQUIRE(f != nullptr, FI_ERR_INVALID, "field is null");
		fi_solve_options o;
		if (opt) { o = *opt; } else { fi_solve_options_default(&o); }
		if (o.precision == FI_F64) {
			Operator<double>& op = f->get64();
			op.use_fast = o.use_fast_stencil;
			pcg_stage<double>(op, stage, par, pos, ring, count, loc, vectors, o.tolerance, o.max_iterations, state, report, f->stream);
		} else {
			FI_REQUIRE(o.precision == FI_F32, FI_ERR_INVALID, "precision must be FI_F32 or FI_F64");
			Operator<float>& op = f->get32();
			op.use_fast = o.use_fast_stencil;
			pcg_stage<float>(op, stage, par, pos, ring, count, loc, vectors, o.tolerance, o.max_iterations, state, report, f->stream);
		}
	});
}

}  // extern "C"
