// Jacobi-preconditioned conjugate gradients on the normal equations — north-star item (c).
//
// Stands in for the reference's Eigen solves (sparse_linear.cpp:115-212, 392-443): same system A^T A x = A^T b,
// same diagonal preconditioner (Eigen's default DiagonalPreconditioner: 1/diag, 1 where diag == 0), same
// stopping rule |r| <= tol |A^T b|, same treatment of a zero right-hand side (x = 0) and of a failure to
// converge (the last iterate is returned).  A^T A is symmetric positive (semi-)definite, so CG replaces
// Eigen's BiCGSTAB at half the operator applications per iteration.
//
// x is not needed by the iteration itself, so the fused path keeps a ring of the last m directions (iteration k reads p_k-1
// from PcgWork::dir[k mod m] and writes p_k to dir[(k+1) mod m]) and updates x once per m iterations with all m terms.
// Iterations k mod m < m-1 are the *skip* form: they park a_k in PcgWork::alpha and move 16 B/cell (q, r, M read, r
// written).  Iteration k mod m = m-1 is the *flush* form: x += s with s = a_k-m+1 p_k-m+1, then s += a_j p_j for j up to k in
// increasing order, which moves (m+6) words per cell.  Averaged over m iterations that is 4 (5 + 2/m) bytes per fp32 cell:
// 24 at m = 2, 21 at m = 8, against 28 for x += a p every iteration.  The directions still pending when the loop stops are
// flushed by one launch after it.  m is chosen per solve by choose_x_ring.  Slab-sharded solves keep the two-direction
// scheme of the peer and NCCL update kernels (kXSkip / kXBoth below: a_k parked in PcgState::alpha_prev, both terms applied
// by the odd iteration).
// Per iteration three kernels touch the lattice vectors:
//   apply      q = (S+P) p, p.q                      read p, write q              8 B/cell (fp32)
//   update     x += a p, r -= a q, r.Mr, r.r         read x,p,q,r,M, write x,r   28 B/cell
//   direction  p = M r + b p                         read r,M,p, write p         16 B/cell
// All scalars (alpha, beta, norms, the convergence flag, the iteration counter) live in a PcgState on the
// device; dot products are reduced per block with warp shuffles and combined in a fixed order by the last
// block to finish, so a run is bit-reproducible up to the data term's atomics.  `check_every` iterations are
// captured into one CUDA graph; the host only polls the flag between graph launches.
#include "solver.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace fi {

namespace {

constexpr int kThreads = 256;

int vec_grid(int64_t n)
{
	const int64_t want = (n + kThreads - 1) / kThreads;
	return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(want, static_cast<int64_t>(sm_count()) * 8)));
}

template <typename T>
struct Pack;
template <>
struct Pack<float>
{
	using type = float4;
	static constexpr int V = 4;
};
template <>
struct Pack<double>
{
	using type = double2;
	static constexpr int V = 2;
};

// Applies f(i) to every element index, 16 bytes per thread per step where alignment allows.
template <typename T, typename F>
__device__ __forceinline__ void for_each_pack(int64_t n, F&& f)
{
	constexpr int V      = Pack<T>::V;
	const int64_t npacks = n / V;
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < npacks; k += stride) { f(k, true); }
	if (blockIdx.x == 0) {
		for (int64_t i = npacks * V + threadIdx.x; i < n; i += blockDim.x) { f(i, false); }
	}
}

// The same with a contiguous range of packs per block (coalesced inside the block) instead of a grid-stride walk: only the
// first and last few blocks touch the ends of the vector.  Returns the block's element range through first / last.
template <typename T, typename F>
__device__ __forceinline__ void for_each_pack_blocked(int64_t n, int64_t* first, int64_t* last, F&& f)
{
	constexpr int V      = Pack<T>::V;
	const int64_t npacks = n / V;
	const int64_t chunk  = (npacks + gridDim.x - 1) / gridDim.x;
	const int64_t k0 = static_cast<int64_t>(blockIdx.x) * chunk, k1 = min(k0 + chunk, npacks);
	for (int64_t k = k0 + threadIdx.x; k < k1; k += blockDim.x) { f(k, true); }
	*first = k0 * V;
	*last  = k1 * V;
	if (blockIdx.x == gridDim.x - 1) {
		for (int64_t i = npacks * V + threadIdx.x; i < n; i += blockDim.x) { f(i, false); }
		*last = n;
	}
}

// r = b - q, p = M r; rho = r.p, rr = r.r, bb = b.b
template <typename T>
__global__ void __launch_bounds__(kThreads) pcg_init_kernel(int64_t n, const T* __restrict__ b, const T* __restrict__ q,
                                                            const T* __restrict__ minv, T* __restrict__ r, T* __restrict__ p,
                                                            PcgState* st, double tol, long long max_iters, double* partial,
                                                            unsigned* ticket, int dist)
{
	__shared__ double red[32];
	double            acc[3] = {0, 0, 0};
	const int64_t     stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		const T bi = b[i], ri = q ? bi - q[i] : bi, zi = minv[i] * ri;  // q == nullptr: the guess is zero
		r[i] = ri;
		p[i] = zi;
		acc[0] += static_cast<double>(ri) * static_cast<double>(zi);
		acc[1] += static_cast<double>(ri) * static_cast<double>(ri);
		acc[2] += static_cast<double>(bi) * static_cast<double>(bi);
	}
	acc[0] = block_sum(acc[0], red);
	acc[1] = block_sum(acc[1], red);
	acc[2] = block_sum(acc[2], red);
	grid_sum<3>(acc, partial, ticket, red, [&](const double(&tot)[3]) {
		if (dist) {  // partial sums of this slab: all-reduced, then pcg_init_finish_kernel
			st->part[0] = tot[0];
			st->part[1] = tot[1];
			st->part[2] = tot[2];
			return;
		}
		st->rho[0]    = tot[0];
		st->rho[1]    = 0;
		st->pq        = 0;
		st->rr        = tot[1];
		st->rr0       = tot[1];
		st->bb        = tot[2];
		st->tol2bb    = tol * tol * tot[2];
		st->iters     = 0;
		st->max_iters = max_iters;
		st->breakdown = 0;
		st->done      = (tot[2] == 0.0 || tot[1] <= tol * tol * tot[2] || max_iters <= 0) ? 1 : 0;
	});
}

__global__ void peer_publish_kernel(PeerLink L, int which, int par, unsigned long long base, const PcgState* st, const double* src, int count,
                                    const int* done)
{
	if (blockIdx.x != 0 || threadIdx.x >= 32) { return; }
	const unsigned long long seq = seq_of(base, st, which);
	double v[2] = {0.0, 0.0};
	// a finished solve still publishes (zeros): the peers' kernels of this round are already waiting
	if (!(done && *done)) {
		for (int k = 0; k < count; ++k) { v[k] = src[k]; }
		if (threadIdx.x == 0) { L.local->stamp[0][st->iters & 511] = global_ns(); }
	}
	peer_publish_warp(L, which, par, seq, v, count);
}

// Ends an iteration on the peer-memory path: sums (r.Mr, r.r) over ranks and updates the shared CG state.
__global__ void pcg_update_finish_peer_kernel(PcgState* st, int par, PeerLink L, unsigned long long base)
{
	if (blockIdx.x != 0 || threadIdx.x >= 32) { return; }
	const unsigned long long seq = seq_of(base, st, 1);
	double tot[2];
	const bool ok = peer_collect_warp(L, 1, par, seq, tot, 2);
	if (threadIdx.x != 0 || st->done) { return; }
	if (!ok) {
		st->breakdown = 2;
		st->done      = 1;
		return;
	}
	L.local->stamp[2][st->iters & 511] = global_ns();
	st->rho[par ^ 1] = tot[0];
	st->rr           = tot[1];
	st->iters += 1;
	if (tot[1] <= st->tol2bb || st->iters >= st->max_iters || !(tot[0] > 0.0)) { st->done = 1; }
}

__global__ void pcg_init_finish_kernel(PcgState* st, double tol, long long max_iters)
{
	const double rho = st->part[0], rr = st->part[1], bb = st->part[2];
	st->rho[0]    = rho;
	st->rho[1]    = 0;
	st->pq        = 0;
	st->rr        = rr;
	st->rr0       = rr;
	st->bb        = bb;
	st->tol2bb    = tol * tol * bb;
	st->iters     = 0;
	st->max_iters = max_iters;
	st->breakdown = 0;
	st->done      = (bb == 0.0 || rr <= tol * tol * bb || max_iters <= 0) ? 1 : 0;
}

__global__ void pcg_update_finish_kernel(PcgState* st, int par)
{
	if (st->done) { return; }
	const double rho = st->part[0], rr = st->part[1];
	st->rho[par ^ 1] = rho;
	st->rr           = rr;
	st->iters += 1;
	if (rr <= st->tol2bb || st->iters >= st->max_iters || !(rho > 0.0)) { st->done = 1; }
}

// How an update kernel treats x (see the header comment): every iteration; not at all (even iteration of the deferred scheme:
// the step length is parked in PcgState::alpha_prev); or with this and the previous iteration's terms (odd iteration).
enum XMode { kXClassic = 0, kXSkip = 1, kXBoth = 2 };

// x, r of `count` consecutive elements starting at i: the element-wise part shared by the update kernels.
template <typename T, int XM, bool PACKED>
__device__ __forceinline__ void update_elements(int64_t k, T* __restrict__ x, T* __restrict__ r, const T* __restrict__ p, const T* __restrict__ p_prev,
                                                const T* __restrict__ q, const T* __restrict__ minv, T alpha, T alpha_prev, double (&acc)[2],
                                                typename Pack<T>::type* r_out)
{
	using P         = typename Pack<T>::type;
	constexpr int V = PACKED ? Pack<T>::V : 1;
	T xa[V], ra[V], pa[V], ppa[V], qa[V], ma[V];
	if (PACKED) {
		*reinterpret_cast<P*>(ra) = reinterpret_cast<const P*>(r)[k];
		*reinterpret_cast<P*>(qa) = reinterpret_cast<const P*>(q)[k];
		*reinterpret_cast<P*>(ma) = reinterpret_cast<const P*>(minv)[k];
		if (XM != kXSkip) {
			*reinterpret_cast<P*>(xa) = reinterpret_cast<const P*>(x)[k];
			*reinterpret_cast<P*>(pa) = reinterpret_cast<const P*>(p)[k];
		}
		if (XM == kXBoth) { *reinterpret_cast<P*>(ppa) = reinterpret_cast<const P*>(p_prev)[k]; }
	} else {
		ra[0] = r[k];
		qa[0] = q[k];
		ma[0] = minv[k];
		if (XM != kXSkip) {
			xa[0] = x[k];
			pa[0] = p[k];
		}
		if (XM == kXBoth) { ppa[0] = p_prev[k]; }
	}
#pragma unroll
	for (int j = 0; j < V; ++j) {
		if (XM == kXClassic) { xa[j] += alpha * pa[j]; }
		if (XM == kXBoth) { xa[j] += alpha_prev * ppa[j] + alpha * pa[j]; }
		ra[j] -= alpha * qa[j];
		const double rd = static_cast<double>(ra[j]);
		acc[0] += rd * static_cast<double>(ma[j] * ra[j]);
		acc[1] += rd * rd;
	}
	if (PACKED) {
		if (XM != kXSkip) { reinterpret_cast<P*>(x)[k] = *reinterpret_cast<const P*>(xa); }
		reinterpret_cast<P*>(r)[k] = *reinterpret_cast<const P*>(ra);
		if (r_out) { *r_out = *reinterpret_cast<const P*>(ra); }
	} else {
		if (XM != kXSkip) { x[k] = xa[0]; }
		r[k] = ra[0];
		if (r_out) { reinterpret_cast<T*>(r_out)[0] = ra[0]; }
	}
}

template <typename T, int XM>
__global__ void __launch_bounds__(kThreads) pcg_update_kernel(int64_t n, T* __restrict__ x, T* __restrict__ r,
                                                              const T* __restrict__ p, const T* __restrict__ p_prev, const T* __restrict__ q,
                                                              const T* __restrict__ minv, PcgState* st, int par,
                                                              double* partial, unsigned* ticket, int dist)
{
	__shared__ double red[32];
	if (st->done) { return; }
	const double pq = st->pq;
	if (!(pq > 0.0)) {  // breakdown (singular direction or NaN): keep the last iterate
		if (blockIdx.x == 0 && threadIdx.x == 0) {
			st->breakdown = 1;
			st->done      = 1;
		}
		return;
	}
	const double alpha_d = st->rho[par] / pq;
	const T      alpha = static_cast<T>(alpha_d), alpha_prev = XM == kXBoth ? static_cast<T>(st->alpha_prev) : T(0);
	double acc[2] = {0, 0};
	for_each_pack<T>(n, [&](int64_t k, bool packed) {
		if (packed) {
			update_elements<T, XM, true>(k, x, r, p, p_prev, q, minv, alpha, alpha_prev, acc, nullptr);
		} else {
			update_elements<T, XM, false>(k, x, r, p, p_prev, q, minv, alpha, alpha_prev, acc, nullptr);
		}
	});
	acc[0] = block_sum(acc[0], red);
	acc[1] = block_sum(acc[1], red);
	grid_sum<2>(acc, partial, ticket, red, [&](const double(&tot)[2]) {
		if (XM == kXSkip) { st->alpha_prev = alpha_d; }
		if (dist) {  // all-reduced, then pcg_update_finish_kernel
			st->part[0] = tot[0];
			st->part[1] = tot[1];
			return;
		}
		st->rho[par ^ 1] = tot[0];
		st->rr           = tot[1];
		st->iters += 1;
		if (tot[1] <= st->tol2bb || st->iters >= st->max_iters || !(tot[0] > 0.0)) { st->done = 1; }
	});
}

// Directions of a flush, oldest first (by value: a kernel argument).
template <typename T>
struct DirRing
{
	const T* p[kMaxXRing];
};

// r -= a q with the two dot products, and for M > 0 (flush form) also x += a[0] d_0 + ... + a[M-1] d_M-1, summed in that order
// into a temporary that is added to x last.
template <typename T, int M, bool PACKED>
__device__ __forceinline__ void ring_update_elements(int64_t k, T* __restrict__ x, T* __restrict__ r, const DirRing<T>& d, const T* __restrict__ q,
                                                     const T* __restrict__ minv, T alpha, const T (&a)[kMaxXRing], double (&acc)[2])
{
	using P         = typename Pack<T>::type;
	constexpr int V = PACKED ? Pack<T>::V : 1;
	constexpr int MD = M > 0 ? M : 1;
	T ra[V], qa[V], ma[V], xa[V], da[MD][V];
	if (PACKED) {
		*reinterpret_cast<P*>(ra) = reinterpret_cast<const P*>(r)[k];
		*reinterpret_cast<P*>(qa) = reinterpret_cast<const P*>(q)[k];
		*reinterpret_cast<P*>(ma) = reinterpret_cast<const P*>(minv)[k];
		if (M > 0) {
			*reinterpret_cast<P*>(xa) = reinterpret_cast<const P*>(x)[k];
#pragma unroll
			for (int j = 0; j < M; ++j) { *reinterpret_cast<P*>(da[j]) = reinterpret_cast<const P*>(d.p[j])[k]; }
		}
	} else {
		ra[0] = r[k];
		qa[0] = q[k];
		ma[0] = minv[k];
		if (M > 0) {
			xa[0] = x[k];
#pragma unroll
			for (int j = 0; j < M; ++j) { da[j][0] = d.p[j][k]; }
		}
	}
#pragma unroll
	for (int e = 0; e < V; ++e) {
		if (M > 0) {
			T s = a[0] * da[0][e];
#pragma unroll
			for (int j = 1; j < M; ++j) { s += a[j] * da[j][e]; }
			xa[e] += s;
		}
		ra[e] -= alpha * qa[e];
		const double rd = static_cast<double>(ra[e]);
		acc[0] += rd * static_cast<double>(ma[e] * ra[e]);
		acc[1] += rd * rd;
	}
	if (PACKED) {
		if (M > 0) { reinterpret_cast<P*>(x)[k] = *reinterpret_cast<const P*>(xa); }
		reinterpret_cast<P*>(r)[k] = *reinterpret_cast<const P*>(ra);
	} else {
		if (M > 0) { x[k] = xa[0]; }
		r[k] = ra[0];
	}
}

// The update kernel of the unsharded fused iteration with a ring of m directions (header comment).  M = 0: skip form, x is
// left alone and a_k is parked in alpha[pos] (pos = k mod m).  M = m: flush form, d holds p_k-m+1 .. p_k and alpha[0 .. m-2]
// the parked step lengths of the first m-1 of them.
template <typename T, int M>
__global__ void __launch_bounds__(kThreads) pcg_update_ring_kernel(int64_t n, T* __restrict__ x, T* __restrict__ r, DirRing<T> d,
                                                                   const T* __restrict__ q, const T* __restrict__ minv, PcgState* st, int par,
                                                                   double* __restrict__ alpha, int pos, double* partial, unsigned* ticket)
{
	__shared__ double red[32];
	if (st->done) { return; }
	const double pq = st->pq;
	if (!(pq > 0.0)) {  // breakdown (singular direction or NaN): keep the last iterate
		if (blockIdx.x == 0 && threadIdx.x == 0) {
			st->breakdown = 1;
			st->done      = 1;
		}
		return;
	}
	const double alpha_d = st->rho[par] / pq;
	T            a[kMaxXRing];
#pragma unroll
	for (int j = 0; j < kMaxXRing; ++j) { a[j] = j < M - 1 ? static_cast<T>(alpha[j]) : T(0); }
	if (M > 0) { a[M > 0 ? M - 1 : 0] = static_cast<T>(alpha_d); }
	double acc[2] = {0, 0};
	for_each_pack<T>(n, [&](int64_t k, bool packed) {
		if (packed) {
			ring_update_elements<T, M, true>(k, x, r, d, q, minv, static_cast<T>(alpha_d), a, acc);
		} else {
			ring_update_elements<T, M, false>(k, x, r, d, q, minv, static_cast<T>(alpha_d), a, acc);
		}
	});
	acc[0] = block_sum(acc[0], red);
	acc[1] = block_sum(acc[1], red);
	grid_sum<2>(acc, partial, ticket, red, [&](const double(&tot)[2]) {
		if (M == 0) { alpha[pos] = alpha_d; }
		st->rho[par ^ 1] = tot[0];
		st->rr           = tot[1];
		st->iters += 1;
		if (tot[1] <= st->tol2bb || st->iters >= st->max_iters || !(tot[0] > 0.0)) { st->done = 1; }
	});
}

// The update kernel of a slab on the peer-memory path: waits for the all-reduced p.Ap in its mailbox, updates x
// and r, stores the boundary planes of the new r straight into the neighbours' halo planes (NVLink peer stores),
// and the last block publishes this slab's (r.Mr, r.r) to every rank.
template <typename T, int XM>
__global__ void __launch_bounds__(kThreads) pcg_update_peer_kernel(int64_t n, T* __restrict__ x, T* __restrict__ r,
                                                                   const T* __restrict__ p, const T* __restrict__ p_prev, const T* __restrict__ q,
                                                                   const T* __restrict__ minv, PcgState* st, int par, double* partial,
                                                                   unsigned* ticket, PeerLink L, HaloPush<T> push, unsigned long long base, int fold,
                                                                   int blocked)
{
	__shared__ double red[32];
	__shared__ double s_pq, s_tot[2];
	__shared__ int    s_ok, s_pub;
	const bool was_done = st->done != 0;
	const unsigned long long seq_pq = seq_of(base, st, 0), seq_rr = seq_of(base, st, 1);
	// fold bit 0: this kernel also does the work of peer_publish_kernel (block 0, before anybody waits); bit 1: and of
	// pcg_update_finish_peer_kernel (the last block, after it has published) — a kernel boundary fewer per iteration each
	if ((fold & 1) && blockIdx.x == 0 && threadIdx.x < 32) {
		double mine[1] = {was_done ? 0.0 : st->pq};  // a finished solve still publishes: the peers' kernels are waiting
		if (threadIdx.x == 0 && !was_done) { L.local->stamp[0][st->iters & 511] = global_ns(); }
		peer_publish_warp(L, 0, par, seq_pq, mine, 1);
	}
	if (threadIdx.x < 32) {
		double     pq = 0.0;
		const bool ok = peer_collect_warp(L, 0, par, seq_pq, &pq, 1);
		if (threadIdx.x == 0) {
			s_ok  = ok ? 1 : 0;
			s_pq  = pq;
			s_pub = 0;
			if (blockIdx.x == 0 && !was_done) { L.local->stamp[1][st->iters & 511] = global_ns(); }
		}
	}
	__syncthreads();
	const double pq    = s_pq;
	const bool   bad   = !s_ok || !(pq > 0.0);  // lost peer, or breakdown (singular direction / NaN): keep the last iterate
	double       acc[2] = {0, 0};
	const double alpha_d = (!was_done && !bad) ? st->rho[par] / pq : 0.0;
	bool         pushed  = false;
	if (!was_done && !bad) {
		const T alpha = static_cast<T>(alpha_d), alpha_prev = XM == kXBoth ? static_cast<T>(st->alpha_prev) : T(0);
		using P       = typename Pack<T>::type;
		constexpr int V = Pack<T>::V;
		const int64_t hi_from = n - push.count;
		auto element = [&](int64_t k, bool packed) {
			if (packed) {
				P rv;
				update_elements<T, XM, true>(k, x, r, p, p_prev, q, minv, alpha, alpha_prev, acc, &rv);
				const int64_t i = k * V;  // halo extents are whole planes of a lattice whose x size is a multiple of V
				if (push.lo && i < push.count) { *reinterpret_cast<P*>(push.lo + i) = rv; }
				if (push.hi && i >= hi_from) { *reinterpret_cast<P*>(push.hi + (i - hi_from)) = rv; }
			} else {
				P rv;
				update_elements<T, XM, false>(k, x, r, p, p_prev, q, minv, alpha, alpha_prev, acc, &rv);
				const T ri = reinterpret_cast<const T*>(&rv)[0];
				if (push.lo && k < push.count) { push.lo[k] = ri; }
				if (push.hi && k >= hi_from) { push.hi[k - hi_from] = ri; }
			}
		};
		if (blocked) {
			// only the blocks at the two ends of the slab store into a neighbour's memory
			int64_t first = 0, last = 0;
			for_each_pack_blocked<T>(n, &first, &last, element);
			pushed = (push.lo && first < push.count) || (push.hi && last > hi_from);
		} else {
			for_each_pack<T>(n, element);
			pushed = push.lo != nullptr || push.hi != nullptr;  // a grid-stride walk takes most blocks through both ends
		}
	}
	acc[0] = block_sum(acc[0], red);
	acc[1] = block_sum(acc[1], red);
	// peer stores of every thread of this block are ordered before the ticket below (bar.sync above, fence here).  A
	// system-scope fence while the SM streams gigabytes of ordinary stores is expensive: only the blocks that pushed pay it
	// (block-contiguous ranges: the first and last few blocks), the others take grid_sum's device-scope fence.
	if (threadIdx.x == 0 && pushed) { __threadfence_system(); }
	grid_sum<2>(acc, partial, ticket, red, [&](const double(&tot)[2]) {
		if (!was_done && bad) {
			st->breakdown = s_ok ? 1 : 2;
			st->done      = 1;
		}
		if (XM == kXSkip && !was_done && !bad) { st->alpha_prev = alpha_d; }
		s_tot[0] = tot[0];
		s_tot[1] = tot[1];
		s_pub    = 1;
	});
	__syncthreads();
	// the last block to finish: its first warp publishes this slab's sums to every rank at once
	if (s_pub && threadIdx.x < 32) {
		const double tot[2] = {s_tot[0], s_tot[1]};
		peer_publish_warp(L, 1, par, seq_rr, tot, 2);
		if (fold & 2) {  // every other block of this kernel has finished: end the iteration here (pcg_update_finish_peer_kernel)
			double     all[2];
			const bool ok = peer_collect_warp(L, 1, par, seq_rr, all, 2);
			if (threadIdx.x == 0 && !st->done) {
				if (!ok) {
					st->breakdown = 2;
					st->done      = 1;
				} else {
					L.local->stamp[2][st->iters & 511] = global_ns();
					st->rho[par ^ 1] = all[0];
					st->rr           = all[1];
					st->iters += 1;
					if (all[1] <= st->tol2bb || st->iters >= st->max_iters || !(all[0] > 0.0)) { st->done = 1; }
				}
			}
		}
	}
}

template <typename T>
__global__ void __launch_bounds__(kThreads) pcg_direction_kernel(int64_t n, const T* __restrict__ r, const T* __restrict__ minv,
                                                                 T* __restrict__ p, const PcgState* st, int par)
{
	if (st->done) { return; }
	const T beta  = static_cast<T>(st->rho[par ^ 1] / st->rho[par]);
	using P       = typename Pack<T>::type;
	constexpr int V = Pack<T>::V;
	for_each_pack<T>(n, [&](int64_t k, bool packed) {
		if (packed) {
			const P  rv = reinterpret_cast<const P*>(r)[k], mv = reinterpret_cast<const P*>(minv)[k];
			P        pv = reinterpret_cast<P*>(p)[k];
			const T* ra = reinterpret_cast<const T*>(&rv);
			const T* ma = reinterpret_cast<const T*>(&mv);
			T*       pa = reinterpret_cast<T*>(&pv);
#pragma unroll
			for (int j = 0; j < V; ++j) { pa[j] = ma[j] * ra[j] + beta * pa[j]; }
			reinterpret_cast<P*>(p)[k] = pv;
		} else {
			p[k] = minv[k] * r[k] + beta * p[k];
		}
	});
}

// r = b - q; rr = r.r, bb = b.b (out[0], out[1])
template <typename T>
__global__ void __launch_bounds__(kThreads) residual_kernel(int64_t n, const T* __restrict__ b, const T* __restrict__ q, T* __restrict__ r,
                                                            double* out, double* partial, unsigned* ticket)
{
	__shared__ double red[32];
	double            acc[2] = {0, 0};
	const int64_t     stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		const T bi = b[i], ri = bi - q[i];
		if (r) { r[i] = ri; }
		acc[0] += static_cast<double>(ri) * static_cast<double>(ri);
		acc[1] += static_cast<double>(bi) * static_cast<double>(bi);
	}
	acc[0] = block_sum(acc[0], red);
	acc[1] = block_sum(acc[1], red);
	grid_sum<2>(acc, partial, ticket, red, [&](const double(&tot)[2]) {
		out[0] = tot[0];
		out[1] = tot[1];
	});
}

// jacobi_iterations, reference sparse_linear.cpp:232-239: temp = Atb - R x with R = AtA - D, then
// x = w*temp/D + (1-w)*x.  q holds AtA x.
template <typename T>
__global__ void jacobi_kernel(int64_t n, const T* __restrict__ atb, const T* __restrict__ q, const T* __restrict__ diag, T* __restrict__ x, T w)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		const T temp = atb[i] - (q[i] - diag[i] * x[i]);
		x[i]         = w * temp / diag[i] + (T(1) - w) * x[i];
	}
}

template <typename A, typename B>
__global__ void convert_kernel(int64_t n, const A* __restrict__ a, B* __restrict__ b)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) { b[i] = static_cast<B>(a[i]); }
}

__global__ void add_f32_f64_kernel(int64_t n, const float* __restrict__ e, double* __restrict__ x)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) { x[i] += static_cast<double>(e[i]); }
}

// x += alpha[0] d_0 + ... + alpha[count-1] d_count-1 (1 <= count < kMaxXRing), summed in the order of the flush form: the x
// update of the iterations still pending when the loop stopped
template <typename T>
__global__ void __launch_bounds__(kThreads) pcg_flush_x_kernel(int64_t n, T* __restrict__ x, DirRing<T> d, const double* alpha, int count)
{
	T a[kMaxXRing];
#pragma unroll
	for (int j = 0; j < kMaxXRing; ++j) { a[j] = j < count ? static_cast<T>(alpha[j]) : T(0); }
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		T s = a[0] * d.p[0][i];
#pragma unroll
		for (int j = 1; j < kMaxXRing; ++j) {
			if (j < count) { s += a[j] * d.p[j][i]; }
		}
		x[i] += s;
	}
}

// How many directions the fused iteration keeps before it updates x (header comment): FI_B200_X_RING=2|4|8 when set, else
// kDefaultXRing; 2 where the two-direction working set (x, r, q, M^-1 and two directions) fits the L2 cache — extra buffers
// there would push the vectors out of it for a few bytes per cell — or where no fused kernel runs; halved while the buffers
// not yet allocated would take more than half of the free device memory.  8 measured best on a B200 at 512^3 and 1024^3:
// 512^3 fp32 iteration 0.998 / 0.948 / 0.937 ms at m = 2 / 4 / 8 (DESIGN.md §3, profiles/x_ring_b200.jsonl).
constexpr int kDefaultXRing = 8;

template <typename T>
int choose_x_ring(const Operator<T>& op)
{
	const bool fusable = op.g.ndim >= 2 && !op.g.tile && op.use_fast != kStencilGeneric && op.dist == nullptr && !op.g.sharded();
	if (!fusable) { return 2; }
	const char* env = std::getenv("FI_B200_X_RING");
	int         m   = kDefaultXRing;
	const size_t vec = static_cast<size_t>(op.g.N) * sizeof(T);
	if (env && *env) {
		m = std::atoi(env);
		FI_REQUIRE(m == 2 || m == 4 || m == 8, FI_ERR_INVALID, "FI_B200_X_RING must be 2, 4 or 8");
	} else {
		int dev = 0, l2 = 0;
		FI_CUDA(cudaGetDevice(&dev));
		FI_CUDA(cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev));
		const size_t l2_bytes = l2 > 0 ? static_cast<size_t>(l2) : static_cast<size_t>(126) << 20;  // unreported: the B200's
		if (6 * vec <= l2_bytes) { return 2; }
	}
	size_t free_b = 0, total_b = 0;
	FI_CUDA(cudaMemGetInfo(&free_b, &total_b));
	while (m > 2 && static_cast<size_t>(std::max(0, m - op.work.dirs)) * vec > free_b / 2) { m /= 2; }
	return m;
}

// dir[0 .. m) allocated; the new ones zeroed (a flush timed on its own reads every slot)
template <typename T>
void ensure_ring(PcgWork<T>& w, size_t n, int m, cudaStream_t s)
{
	for (; w.dirs < m; ++w.dirs) {
		w.dir[w.dirs].resize(n);
		w.dir[w.dirs].zero(s);
	}
}

// Launches the update of ring position pos (= k mod m) of the unsharded fused iteration: the skip form, or at pos = m-1 the
// flush form over p_k-m+1 .. p_k, which sit in dir[1], ..., dir[m-1], dir[0].
template <typename T>
void launch_ring_update(PcgWork<T>& w, int m, int pos, int grid, int64_t n, T* x, const T* minv, int par, cudaStream_t s)
{
	DirRing<T> d = {};
	if (pos < m - 1) {
		auto ku = pcg_update_ring_kernel<T, 0>;
		FI_LAUNCH(ku, grid, kThreads, 0, s, n, x, w.r.data(), d, w.q.data(), minv, w.state.data(), par, w.alpha.data(), pos, w.partial.data(),
		          w.ticket.data());
		return;
	}
	for (int j = 0; j < m; ++j) { d.p[j] = w.dir[(j + 1) % m].data(); }
	auto ku = m == 8 ? pcg_update_ring_kernel<T, 8> : m == 4 ? pcg_update_ring_kernel<T, 4> : pcg_update_ring_kernel<T, 2>;
	FI_LAUNCH(ku, grid, kThreads, 0, s, n, x, w.r.data(), d, w.q.data(), minv, w.state.data(), par, w.alpha.data(), pos, w.partial.data(),
	          w.ticket.data());
}

template <typename T>
void ensure_work(Operator<T>& op, cudaStream_t s)
{
	PcgWork<T>& w = op.work;
	const size_t n = static_cast<size_t>(op.g.N);
	if (w.r.size() != n) {
		w.r.resize(n);
		w.q.resize(n);
		// the fused stencil kernel reads p_old before the first direction exists (times beta = 0): it must be finite.  On a slab
		// the halo planes and the planes beyond the lattice of r and q are read too; elsewhere every element of r and q is
		// written before it is read.  (On the solver's own stream: it is non-blocking, so work on the null stream is not
		// ordered with it.)  Directions beyond the first two are allocated by the solve that needs them (ensure_ring).
		for (int j = 2; j < kMaxXRing; ++j) { w.dir[j].release(); }
		w.dirs = 0;
		ensure_ring(w, n, 2, s);
		w.alpha.resize(kMaxXRing - 1);
		if (op.g.sharded()) {
			w.r.zero(s);
			w.q.zero(s);
		}
		w.partial.resize(static_cast<size_t>(3) * (static_cast<size_t>(sm_count()) * 8 + 8));
		w.ticket.resize(1);
		w.state.resize(1);
		w.ticket.zero(s);
	}
}

}  // namespace

void convert(const float* src, double* dst, int64_t n, cudaStream_t s)
{
	auto kern = convert_kernel<float, double>;
	FI_LAUNCH(kern, vec_grid(n), kThreads, 0, s, n, src, dst);
}
void convert(const double* src, float* dst, int64_t n, cudaStream_t s)
{
	auto kern = convert_kernel<double, float>;
	FI_LAUNCH(kern, vec_grid(n), kThreads, 0, s, n, src, dst);
}
void axpy_f32_into_f64(const float* e, double* x, int64_t n, cudaStream_t s)
{
	FI_LAUNCH(add_f32_f64_kernel, vec_grid(n), kThreads, 0, s, n, e, x);
}

template <typename T>
std::unique_ptr<Operator<T>> build_operator(const Geom& g, const ModelAccum& m, const PointStore& pts, const HostRows& rows,
                                            cudaStream_t s)
{
	TraceScope  trace("build_operator (data term, diagonal, preconditioner)");
	cudaEvent_t e0, e1;
	FI_CUDA(cudaEventCreate(&e0));
	FI_CUDA(cudaEventCreate(&e1));
	FI_CUDA(cudaEventRecord(e0, s));
	auto op  = std::make_unique<Operator<T>>();
	op->g    = g;
	op->tabs = make_tables(g, m);
	op->atb.resize(g.N);
	op->diag.resize(g.N);
	op->minv.resize(g.N);
	op->atb.zero(s);
	op->diag.zero(s);
	build_data_term<T>(g, pts, rows, op->data, op->atb.data(), op->diag.data(), s);
	stencil_diagonal<T>(g, op->tabs, op->diag.data(), op->minv.data(), s);  // + M^-1 = 1 / diag in the same pass
	op->partial.resize(static_cast<size_t>(stencil_partial_slots(g)));
	op->ticket.resize(1);
	op->ticket.zero(s);
	FI_CUDA(cudaEventRecord(e1, s));
	FI_CUDA(cudaEventSynchronize(e1));
	float ms = 0;
	FI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
	op->setup_ms = ms;
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
	return op;
}

template <typename T>
void residual(Operator<T>& op, const T* b, const T* x, T* r, double* rr, double* bb, cudaStream_t s)
{
	ensure_work(op, s);
	PcgWork<T>&   w   = op.work;
	const int64_t off = op.g.own_offset(), n = op.g.own_cells();
	if (op.dist) { op.dist->exchange_halo(const_cast<T*>(x), sizeof(T), s); }
	op.apply(x, w.q.data(), nullptr, nullptr, s);
	DevBuf<double> out(2);
	auto kern = residual_kernel<T>;
	FI_LAUNCH(kern, vec_grid(n), kThreads, 0, s, n, (b ? b : op.atb.data()) + off, w.q.data() + off, r ? r + off : nullptr, out.data(),
	          w.partial.data(), w.ticket.data());
	if (op.dist) { op.dist->allreduce(out.data(), 2, s); }
	double h[2];
	FI_CUDA(cudaMemcpyAsync(h, out.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	*rr = h[0];
	*bb = h[1];
}

template <typename T>
PcgResult pcg_solve(Operator<T>& op, const T* b, T* x, double tol, long long max_iter, int check_every, bool want_true_residual,
                    cudaStream_t s)
{
	TraceScope trace("pcg_solve");
	ensure_work(op, s);
	PcgWork<T>&   w = op.work;
	// vector kernels run over the planes this process owns (everything, unless the lattice is slab-sharded)
	const int64_t off = op.g.own_offset(), n = op.g.own_cells();
	DistHooks*    dist = op.dist;
	const T*      rhs = b ? b : op.atb.data();
	if (max_iter <= 0) {  // Eigen: maxIterations() = 2 * cols by default
		max_iter = 2 * static_cast<long long>(op.g.size[0]) * op.g.size[1] * op.g.size[2];
	}
	if (!(tol > 0)) { tol = std::is_same<T, float>::value ? 1.1920929e-07 : 2.220446049250313e-16; }
	// directions kept per x update of the fused iteration (2 on a slab: the peer and NCCL update kernels ping-pong)
	const int ring = choose_x_ring(op);
	ensure_ring(w, static_cast<size_t>(op.g.N), ring, s);
	// whole rings per graph: graph slot i is then always ring position i mod m (and parity i & 1)
	check_every = std::max(ring, check_every <= 0 ? 32 : check_every);
	check_every = (check_every + ring - 1) / ring * ring;

	cudaEvent_t e0, e1;
	FI_CUDA(cudaEventCreate(&e0));
	FI_CUDA(cudaEventCreate(&e1));
	FI_CUDA(cudaEventRecord(e0, s));

	const int grid = vec_grid(n);
	// r lives in peer-visible memory when the neighbours push their boundary planes into it
	const PeerLink* link = dist ? dist->link() : nullptr;
	T*              r_vec = w.r.data();
	HaloPush<T>     push;
	if (link) {
		void *lo = nullptr, *hi = nullptr;
		r_vec = static_cast<T*>(dist->shared_vector(static_cast<size_t>(op.g.N) * sizeof(T), &lo, &hi, s));
		const int64_t plane = op.g.stride[2], halo = op.g.zown0;
		push.count = halo * plane;
		// rank - 1 stores our first owned planes into its upper halo (behind its owned planes); rank + 1 into its lower halo (plane 0)
		if (lo) { push.lo = static_cast<T*>(lo) + halo * plane + dist->peer_own_cells(link->rank - 1); }
		if (hi) { push.hi = static_cast<T*>(hi); }
	}
	const bool zero_guess = op.guess_is_zero;
	op.guess_is_zero      = false;
	if (!zero_guess) {
		if (dist) { dist->exchange_halo(x, sizeof(T), s); }
		op.apply(x, w.q.data(), nullptr, nullptr, s);
	}
	{
		// p goes to dir[0]: the p_old of iteration 0 (read times beta = 0)
		auto kern = pcg_init_kernel<T>;
		FI_LAUNCH(kern, grid, kThreads, 0, s, n, rhs + off, zero_guess ? static_cast<const T*>(nullptr) : w.q.data() + off, op.minv.data() + off, r_vec + off, w.dir[0].data() + off,
		          w.state.data(), tol, max_iter, w.partial.data(), w.ticket.data(), dist ? 1 : 0);
		if (dist) {
			dist->allreduce(w.state.data()->part, 3, s);
			FI_LAUNCH(pcg_init_finish_kernel, 1, 1, 0, s, w.state.data(), tol, max_iter);
			dist->exchange_halo(r_vec, sizeof(T), s);
		}
	}
	PcgState h;
	FI_CUDA(cudaMemcpyAsync(&h, w.state.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));

	PcgResult res;
	res.zero_rhs         = (h.bb == 0.0);
	res.initial_residual = h.bb > 0 ? std::sqrt(h.rr0 / h.bb) : 0.0;
	if (res.zero_rhs) {
		FI_CUDA(cudaMemsetAsync(x + off, 0, n * sizeof(T), s));  // Eigen: rhs == 0 => x = 0
	} else if (!h.done) {
		const int* d_done = &w.state.data()->done;
		double*    d_pq   = &w.state.data()->pq;
		// check_every iterations per convergence poll
		// every solve gets its own block of mailbox sequence numbers (all ranks count solves alike)
		const unsigned long long seq_base = link ? (dist->next_seq() << 40) : 0ull;
		// Who publishes p.Ap and who ends the iteration on the peer-memory path (FI_B200_PEER_FOLD, the same on every rank):
		//   0  separate one-warp kernels for both (5 graph nodes per iteration)
		//   1  the update kernel publishes p.Ap (block 0) and ends the iteration (last block): 3 nodes
		//   2  the data-term kernel's last block publishes p.Ap, the update kernel ends the iteration: 3 nodes, and the
		//      publish travels while the update kernel is being launched (default)
		//   3  the data-term kernel publishes, a separate kernel ends the iteration: 4 nodes
		const char* fold_env  = std::getenv("FI_B200_PEER_FOLD");
		const int   fold_mode = !link ? 0 : (fold_env && *fold_env >= '0' && *fold_env <= '3' ? *fold_env - '0' : 2);
		const bool  data_publishes = fold_mode >= 2, update_finishes = fold_mode == 1 || fold_mode == 2;
		// Walk of the peer update kernel.  Block-contiguous ranges confine the halo stores — and the system-scope fence that must
		// follow them, expensive while the SM streams ordinary stores — to the few blocks at the ends of the slab: 8 GPUs, 512^3
		// (18 M elements per slab) 0.1913 -> 0.1852 ms per iteration (profiles/r2m_trace_n8.txt).  On large slabs 1,184 private
		// streams cost more DRAM locality than the fences save: 1024^3 on 8 GPUs (134 M elements per slab) 1.326 ms per iteration
		// with the grid-stride walk, 1.398 ms blocked (r2k / r2m).  FI_B200_PEER_UPDATE=blocked|stride overrides.
		const char* walk_env = std::getenv("FI_B200_PEER_UPDATE");
		const bool  peer_update_blocked = walk_env ? walk_env[0] == 'b' : n < (48ll << 20);
		bool deferred_x = false;  // the fused path updates x once per ring of directions
		auto enqueue_round = [&] {
			for (int it = 0; it < check_every; ++it) {
				const int par = it & 1, pos = it % ring;
				// fused form: direction update folded into the stencil's load stage (p_old = dir[pos], p_new = dir[pos + 1 mod m])
				T* const   p_old = w.dir[pos].data();
				T* const   p_new = w.dir[(pos + 1) % ring].data();
				const bool fused = stencil_fused_step<T>(op.use_fast, op.g, op.tabs, r_vec, op.minv.data(), p_old, p_new, w.q.data(),
				                                         w.state.data(), par, d_pq, op.partial.data(), op.ticket.data(), d_done, s);
				deferred_x = deferred_x || fused;
				if (fused && link) {
					// peer-memory path: no NCCL inside the iteration
					PeerPublish pub;
					pub.link  = *link;
					pub.which = 0;
					pub.par   = par;
					pub.base  = seq_base;
					pub.st    = w.state.data();
					const bool published = apply_data_term<T>(op.g, op.data, p_new, w.q.data(), d_pq, d_done, s, data_publishes ? &pub : nullptr);
					const bool in_update = fold_mode == 1;
					if (!published && !in_update) { FI_LAUNCH(peer_publish_kernel, 1, 32, 0, s, *link, 0, par, seq_base, w.state.data(), d_pq, 1, d_done); }
					auto ku = par == 0 ? pcg_update_peer_kernel<T, kXSkip> : pcg_update_peer_kernel<T, kXBoth>;
					FI_LAUNCH(ku, grid, kThreads, 0, s, n, x + off, r_vec + off, p_new + off, p_old + off, w.q.data() + off, op.minv.data() + off,
					          w.state.data(), par, w.partial.data(), w.ticket.data(), *link, push, seq_base, (in_update ? 1 : 0) | (update_finishes ? 2 : 0),
					          peer_update_blocked ? 1 : 0);
					if (!update_finishes) { FI_LAUNCH(pcg_update_finish_peer_kernel, 1, 32, 0, s, w.state.data(), par, *link, seq_base); }
				} else if (fused && !dist) {
					apply_data_term<T>(op.g, op.data, p_new, w.q.data(), d_pq, d_done, s);
					launch_ring_update<T>(w, ring, pos, grid, n, x, op.minv.data(), par, s);
				} else if (fused) {
					apply_data_term<T>(op.g, op.data, p_new, w.q.data(), d_pq, d_done, s);
					if (dist) { dist->allreduce(d_pq, 1, s); }
					auto ku = par == 0 ? pcg_update_kernel<T, kXSkip> : pcg_update_kernel<T, kXBoth>;
					FI_LAUNCH(ku, grid, kThreads, 0, s, n, x + off, r_vec + off, p_new + off, p_old + off, w.q.data() + off, op.minv.data() + off,
					          w.state.data(), par, w.partial.data(), w.ticket.data(), dist ? 1 : 0);
					if (dist) {
						dist->allreduce(w.state.data()->part, 2, s);
						FI_LAUNCH(pcg_update_finish_kernel, 1, 1, 0, s, w.state.data(), par);
						dist->exchange_halo(r_vec, sizeof(T), s);
					}
				} else {
					FI_REQUIRE(dist == nullptr, FI_ERR_UNSUPPORTED, "a slab-sharded solve needs the fused 3D stencil kernel");
					T* const p = w.dir[0].data();
					op.apply(p, w.q.data(), d_pq, d_done, s);
					auto ku = pcg_update_kernel<T, kXClassic>;
					FI_LAUNCH(ku, grid, kThreads, 0, s, n, x, w.r.data(), p, static_cast<const T*>(nullptr), w.q.data(), op.minv.data(), w.state.data(), par,
					          w.partial.data(), w.ticket.data(), 0);
					auto kd = pcg_direction_kernel<T>;
					FI_LAUNCH(kd, grid, kThreads, 0, s, n, w.r.data(), op.minv.data(), p, w.state.data(), par);
				}
			}
		};
		cudaEvent_t l0, l1;
		FI_CUDA(cudaEventCreate(&l0));
		FI_CUDA(cudaEventCreate(&l1));
		if (dist && !link) {
			// NCCL inside the iteration: launch directly.  Instantiating a graph that contains NCCL nodes costs tens of
			// milliseconds, and with ~7 launches per iteration of >= 0.1 ms the host stays ahead of the device anyway.
			TraceScope trl("iteration loop (direct launches)");
			FI_CUDA(cudaEventRecord(l0, s));
			while (true) {
				enqueue_round();
				FI_CUDA(cudaMemcpyAsync(&h, w.state.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
				FI_CUDA(cudaStreamSynchronize(s));
				if (h.done) { break; }
			}
		} else {
			// one CUDA graph = check_every iterations, replayed until the device-side flag says stop
			cudaGraph_t     graph = nullptr;
			cudaGraphExec_t exec  = nullptr;
			const int64_t   before = g_launches;
			FI_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
			try {
				enqueue_round();
			} catch (...) {
				cudaStreamEndCapture(s, &graph);
				if (graph) { cudaGraphDestroy(graph); }
				throw;
			}
			FI_CUDA(cudaStreamEndCapture(s, &graph));
			const int64_t per_graph = g_launches - before;
			g_launches              = before;
			{
				TraceScope tr("cudaGraphInstantiate");
				FI_CUDA(cudaGraphInstantiate(&exec, graph, 0));
			}
			TraceScope trl("iteration loop (graph launches)");
			FI_CUDA(cudaEventRecord(l0, s));
			while (true) {
				FI_CUDA(cudaGraphLaunch(exec, s));
				count_launch(static_cast<int>(per_graph));
				FI_CUDA(cudaMemcpyAsync(&h, w.state.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
				FI_CUDA(cudaStreamSynchronize(s));
				if (h.done) { break; }
			}
			cudaGraphExecDestroy(exec);
			cudaGraphDestroy(graph);
		}
		const int pending = deferred_x ? static_cast<int>(h.iters % ring) : 0;
		if (pending > 0) {
			// the last `pending` iterations (ring positions 0 .. pending-1, whichever way the loop stopped: convergence, the
			// iteration cap or a breakdown, which parks nothing) left their x update parked; p_j of position i is in dir[i + 1].
			// Their step lengths are in PcgWork::alpha, on a slab (m = 2) in PcgState::alpha_prev.
			DirRing<T> d = {};
			for (int i = 0; i < pending; ++i) { d.p[i] = w.dir[i + 1].data() + off; }
			const double* parked = dist ? &w.state.data()->alpha_prev : w.alpha.data();
			auto          kf     = pcg_flush_x_kernel<T>;
			FI_LAUNCH(kf, grid, kThreads, 0, s, n, x + off, d, parked, pending);
		}
		res.x_ring = deferred_x ? ring : 1;
		FI_CUDA(cudaEventRecord(l1, s));
		FI_CUDA(cudaEventSynchronize(l1));
		if (link && trace_enabled() && h.iters >= 8) {
			// phase durations on this rank from the device timestamps of the last iterations
			std::vector<unsigned long long> st3(3 * 512);
			FI_CUDA(cudaMemcpy(st3.data(), link->local->stamp, sizeof(unsigned long long) * 3 * 512, cudaMemcpyDeviceToHost));
			const long long last = h.iters - 1, first = std::max<long long>(1, h.iters - 400);
			double a = 0, b = 0, c = 0;
			for (long long k = first; k <= last; ++k) {
				a += static_cast<double>(st3[0 * 512 + (k & 511)] - st3[2 * 512 + ((k - 1) & 511)]);  // finish(k-1) -> publish(k)
				b += static_cast<double>(st3[1 * 512 + (k & 511)] - st3[0 * 512 + (k & 511)]);        // publish(k) -> update past wait
				c += static_cast<double>(st3[2 * 512 + (k & 511)] - st3[1 * 512 + (k & 511)]);        // update -> finish(k)
			}
			const double cnt = static_cast<double>(last - first + 1) * 1e3;
			fprintf(stderr, "[fi_b200] rank %d per-iteration us: stencil+data %.1f | wait p.Ap %.1f | update+wait r.r %.1f\n", link->rank, a / cnt,
			        b / cnt, c / cnt);
		}
		float lms = 0;
		FI_CUDA(cudaEventElapsedTime(&lms, l0, l1));
		res.loop_ms = lms;
		cudaEventDestroy(l0);
		cudaEventDestroy(l1);
	}
	FI_CUDA(cudaEventRecord(e1, s));
	FI_CUDA(cudaEventSynchronize(e1));
	float ms = 0;
	FI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);

	res.solve_ms     = ms;
	res.iterations   = h.iters;
	res.rel_residual = h.bb > 0 ? std::sqrt(h.rr / h.bb) : 0.0;
	res.converged    = res.zero_rhs || (h.rr <= h.tol2bb);
	res.true_residual = res.rel_residual;
	if (want_true_residual && !res.zero_rhs) {
		double rr = 0, bb = 0;
		residual<T>(op, rhs, x, nullptr, &rr, &bb, s);
		res.true_residual = bb > 0 ? std::sqrt(rr / bb) : 0.0;
		// the stopping rule must hold for the residual of x itself, not merely for the recurrence (fp32 on a large
		// lattice: the recurrence keeps falling after b - A x has reached its rounding floor)
		const bool recurrence_met = res.converged;
		res.converged             = res.true_residual <= kConvergedSlack * tol;
		res.stalled               = (recurrence_met && !res.converged) || h.breakdown != 0;
	}
	return res;
}

template <typename T>
void jacobi_sweeps(Operator<T>& op, T* x, int iterations, T weight, cudaStream_t s)
{
	ensure_work(op, s);
	PcgWork<T>& w = op.work;
	for (int it = 0; it < iterations; ++it) {
		op.apply(x, w.q.data(), nullptr, nullptr, s);
		auto kern = jacobi_kernel<T>;
		FI_LAUNCH(kern, vec_grid(op.g.N), kThreads, 0, s, op.g.N, op.atb.data(), w.q.data(), op.diag.data(), x, weight);
	}
	FI_CUDA(cudaStreamSynchronize(s));
}

// ---- tile phase of solve_tiled_with_guess (tile_solver_square, reference sparse_linear.cpp:246-390) ---------------
// rhs = Atb - 2 (A g - B g): every coupling between two tiles is moved to the right-hand side with the guess — twice,
// because the reference visits both stored triangles of the symmetric AtA and subtracts at both ends each time
// (:327-334).  minv = 1 / (diag + reg) (:306-309).  A tile counts as "regularisation only" (:345-348: skipped, the
// guess is kept) when none of its nodes has a diagonal entry.
template <typename T>
__global__ void tile_prepare_kernel(Geom g, const T* __restrict__ atb, const T* __restrict__ Ag, const T* __restrict__ Bg,
                                    const T* __restrict__ diag, T* __restrict__ rhs, T* __restrict__ minv, int* __restrict__ tile_active)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= g.N) { return; }
	rhs[i]  = atb[i] - T(2) * (Ag[i] - Bg[i]);
	minv[i] = T(1) / (diag[i] + static_cast<T>(g.tile_reg));
	if (diag[i] != T(0)) { tile_active[tile_of_node(g, i)] = 1; }
}

template <typename T>
__global__ void tile_merge_kernel(Geom g, const T* __restrict__ y, const int* __restrict__ tile_active, T* __restrict__ x)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= g.N) { return; }
	if (tile_active[tile_of_node(g, i)]) { x[i] = y[i]; }
}

// x: the guess on entry, the tile-wise solution on exit.  Every tile's system (A_tile + reg I) y = rhs_tile is
// solved by the same Jacobi-PCG as everything else, all tiles at once: the block-diagonal matrix is applied by the
// operator kernels in tile mode (Geom::tile), so the tiles never exchange information and the result is the
// per-tile exact solution up to `tol`.
template <typename T>
PcgResult tile_phase(Operator<T>& op, int tile_size, T* x, double tol, long long max_iter, int check_every, cudaStream_t s)
{
	TraceScope trace("tile_phase");
	FI_REQUIRE(tile_size >= 2, FI_ERR_INVALID, "tile_size must be >= 2");  // CHECK_GE_F(tile_size, 2), :255
	FI_REQUIRE(op.dist == nullptr && !op.g.sharded(), FI_ERR_UNSUPPORTED, "the tile phase runs on an unsharded lattice");
	const int64_t n = op.g.N;
	int64_t       tiles = 1;
	for (int d = 0; d < op.g.ndim; ++d) { tiles *= (op.g.size[d] + tile_size - 1) / tile_size; }
	DevBuf<T>   Ag(n), Bg(n), rhs(n), y(n), minv(n);
	DevBuf<int> active(static_cast<size_t>(tiles));
	active.zero(s);
	const int  old_fast = op.use_fast;
	const Geom old_g    = op.g;
	bool       swapped  = false;
	auto restore = [&] {
		op.g        = old_g;
		op.use_fast = old_fast;
		if (swapped) { op.minv.swap(minv); swapped = false; }
	};
	PcgResult r;
	try {
		op.apply(x, Ag.data(), nullptr, nullptr, s);
		op.g.tile     = tile_size;
		op.g.tile_reg = 0.0f;
		op.use_fast   = kStencilGeneric;
		op.apply(x, Bg.data(), nullptr, nullptr, s);
		op.g.tile_reg = 1e-6f;
		{
			auto kern = tile_prepare_kernel<T>;
			FI_LAUNCH(kern, div_up(n, kThreads), kThreads, 0, s, op.g, op.atb.data(), Ag.data(), Bg.data(), op.diag.data(), rhs.data(), minv.data(),
			          active.data());
		}
		op.minv.swap(minv);
		swapped = true;
		FI_CUDA(cudaMemcpyAsync(y.data(), x, n * sizeof(T), cudaMemcpyDeviceToDevice, s));
		r = pcg_solve<T>(op, rhs.data(), y.data(), tol, max_iter, check_every, false, s);
		auto kern = tile_merge_kernel<T>;
		FI_LAUNCH(kern, div_up(n, kThreads), kThreads, 0, s, op.g, y.data(), active.data(), x);
		FI_CUDA(cudaStreamSynchronize(s));
	} catch (...) {
		restore();
		throw;
	}
	restore();
	return r;
}

// Per-kernel device times for the roofline figures (fi_field_time_iterations).
template <typename T>
void time_kernels(Operator<T>& op, int iterations, int check_every, double* out, cudaStream_t s)
{
	ensure_work(op, s);
	PcgWork<T>&   w = op.work;
	const int64_t n = op.g.N;
	DevBuf<T>     x(n);
	x.zero(s);
	// a tolerance far below anything reachable: exactly `iterations` iterations run unless CG breaks down
	const PcgResult r = pcg_solve<T>(op, nullptr, x.data(), 1e-300, iterations, check_every, false, s);
	out[0] = r.loop_ms;
	// re-arm the state so the kernels do real work when launched on their own
	PcgState h;
	FI_CUDA(cudaMemcpyAsync(&h, w.state.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	h.done      = 0;
	h.max_iters = 1ll << 60;
	h.tol2bb    = 0;
	h.iters     = 1;
	h.alpha_prev = 0;
	if (!(h.rho[0] > 0)) { h.rho[0] = 1; }
	if (!(h.rho[1] > 0)) { h.rho[1] = 1; }
	if (!(h.pq > 0)) { h.pq = 1; }
	FI_CUDA(cudaMemcpyAsync(w.state.data(), &h, sizeof(h), cudaMemcpyHostToDevice, s));
	FI_CUDA(cudaStreamSynchronize(s));
	cudaEvent_t e0, e1;
	FI_CUDA(cudaEventCreate(&e0));
	FI_CUDA(cudaEventCreate(&e1));
	auto timed = [&](auto&& body) {
		FI_CUDA(cudaEventRecord(e0, s));
		for (int i = 0; i < iterations; ++i) { body(i); }
		FI_CUDA(cudaEventRecord(e1, s));
		FI_CUDA(cudaEventSynchronize(e1));
		float ms = 0;
		FI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
		return static_cast<double>(ms);
	};
	DevBuf<double> dot(1);
	// the directions as the solve cycles through them: ring position i mod m reads dir[i mod m] and writes the next one
	const int m     = std::max(2, r.x_ring);
	T*        p0    = w.dir[0].data();
	auto      p_old = [&](int i) { return w.dir[i % m].data(); };
	auto      p_new = [&](int i) { return w.dir[(i + 1) % m].data(); };
	bool      fused = false;
	out[1] = timed([&](int i) {
		const int par = i & 1;
		fused = stencil_fused_step<T>(op.use_fast, op.g, op.tabs, w.r.data(), op.minv.data(), p_old(i), p_new(i), w.q.data(),
		                              w.state.data(), par, dot.data(), op.partial.data(), op.ticket.data(), nullptr, s);
		if (fused) {
			apply_data_term<T>(op.g, op.data, p_new(i), w.q.data(), dot.data(), nullptr, s);
		} else {
			op.apply(p0, w.q.data(), dot.data(), nullptr, s);
		}
	});
	// alpha = rho/pq is recomputed from the (frozen) state each launch; a tiny alpha keeps the vectors finite
	h.pq = 1e30;
	FI_CUDA(cudaMemcpyAsync(w.state.data(), &h, sizeof(h), cudaMemcpyHostToDevice, s));
	FI_CUDA(cudaStreamSynchronize(s));
	out[2] = timed([&](int i) {
		// the fused path runs m-1 launches that leave x alone and one that applies m terms per ring of m iterations
		if (!fused) {
			auto ku = pcg_update_kernel<T, kXClassic>;
			FI_LAUNCH(ku, vec_grid(n), kThreads, 0, s, n, x.data(), w.r.data(), p0, static_cast<const T*>(nullptr), w.q.data(), op.minv.data(), w.state.data(), 0,
			          w.partial.data(), w.ticket.data(), 0);  // reads rho[0], pq (frozen); writes rho[1], rr, iters
		} else {
			launch_ring_update<T>(w, m, i % m, vec_grid(n), n, x.data(), op.minv.data(), 0, s);
		}
	});
	out[3] = 0.0;
	if (!fused) {
		out[3] = timed([&](int) {
			auto kd = pcg_direction_kernel<T>;
			FI_LAUNCH(kd, vec_grid(n), kThreads, 0, s, n, w.r.data(), op.minv.data(), p0, w.state.data(), 0);
		});
	}
	out[4] = fused ? 1.0 : 0.0;
	out[7] = fused ? m : 1;
	// the two halves of the apply on their own: the lattice-sized stencil kernel (the dominant kernel of the roofline
	// figure) and the data-term kernels over the occupied cells
	out[5] = timed([&](int i) {
		const int par = i & 1;
		if (fused) {
			stencil_fused_step<T>(op.use_fast, op.g, op.tabs, w.r.data(), op.minv.data(), p_old(i), p_new(i), w.q.data(), w.state.data(), par,
			                      dot.data(), op.partial.data(), op.ticket.data(), nullptr, s);
		} else {
			stencil_apply<T>(op.g, op.tabs, p0, w.q.data(), dot.data(), op.partial.data(), op.ticket.data(), nullptr, op.use_fast, s);
		}
	});
	out[6] = timed([&](int i) {
		apply_data_term<T>(op.g, op.data, fused ? p_new(i) : p0, w.q.data(), dot.data(), nullptr, s);
	});
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
}

template void time_kernels<float>(Operator<float>&, int, int, double*, cudaStream_t);
template void time_kernels<double>(Operator<double>&, int, int, double*, cudaStream_t);
template std::unique_ptr<Operator<float>> build_operator<float>(const Geom&, const ModelAccum&, const PointStore&, const HostRows&, cudaStream_t);
template std::unique_ptr<Operator<double>> build_operator<double>(const Geom&, const ModelAccum&, const PointStore&, const HostRows&, cudaStream_t);
template PcgResult pcg_solve<float>(Operator<float>&, const float*, float*, double, long long, int, bool, cudaStream_t);
template PcgResult pcg_solve<double>(Operator<double>&, const double*, double*, double, long long, int, bool, cudaStream_t);
template PcgResult tile_phase<float>(Operator<float>&, int, float*, double, long long, int, cudaStream_t);
template PcgResult tile_phase<double>(Operator<double>&, int, double*, double, long long, int, cudaStream_t);
template void jacobi_sweeps<float>(Operator<float>&, float*, int, float, cudaStream_t);
template void jacobi_sweeps<double>(Operator<double>&, double*, int, double, cudaStream_t);
template void residual<float>(Operator<float>&, const float*, const float*, float*, double*, double*, cudaStream_t);
template void residual<double>(Operator<double>&, const double*, const double*, double*, double*, double*, cudaStream_t);

}  // namespace fi
