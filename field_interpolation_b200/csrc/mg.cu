// Geometric multigrid preconditioner for the lattice normal equations, and the CG driver that uses it.
//
// Why: A^T A = S + P is a fourth-order operator for the default model_2 smoothness; Jacobi-preconditioned CG
// needs O(n^2) iterations on an n^D lattice (43,000 at 256^3 to reach 1e-6, measured).  The reference fights this
// with a coarse-to-fine initial guess (src/sdf_field.cpp:251-304): solve the same problem re-assembled on a
// coarser lattice and upscale.  A V-cycle applies that idea to the *error* on every level, every iteration:
//   * levels: sizes halved (ceil) until the lattice is tiny;
//   * coarse operators by re-discretisation, exactly the way the reference builds its coarse problem — the same
//     points in the coarse lattice's coordinates (positions * (n_c - 1) / (n_f - 1)) and the same smoothness
//     model — with the weights rescaled so that the coarse energy approximates the Galerkin energy P^T A P:
//     value rows unchanged, gradient rows / 2 per level, order-k smoothness rows * 2^((D - 2k) / 2) per level;
//   * prolongation = upscale_field's multilinear, align-corners interpolation (field_interpolation.cpp:431-485),
//     restriction = its transpose;
//   * smoother: Chebyshev polynomial in D^-1 A over [lambda_max / ratio, lambda_max] (symmetric, no dots);
//   * coarsest level: dense inverse, computed once on the host.
// The V-cycle runs in fp32 whatever the arithmetic of the outer CG (a fixed linear operator, symmetric up to
// rounding), and is captured in one CUDA graph.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "solver.hpp"

namespace fi {

namespace {

constexpr int kThreads = 256;

int vgrid(int64_t n) { return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + kThreads - 1) / kThreads, static_cast<int64_t>(sm_count()) * 8))); }

// ---- level construction ------------------------------------------------------------------------------------------
__global__ void coarsen_points_kernel(int D, int64_t n, const float* __restrict__ pos, const float* __restrict__ gw, float sx, float sy, float sz,
                                      float gscale, float* __restrict__ opos, float* __restrict__ ogw)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	for (int d = 0; d < D; ++d) { opos[i * D + d] = pos[i * D + d] * (d == 0 ? sx : (d == 1 ? sy : sz)); }
	ogw[i] = gw[i] * gscale;
}

// ---- smoother ----------------------------------------------------------------------------------------------------
// One Chebyshev step: res_out = res_in - q (when q is given), d = a d + b M^-1 res, e += d.  res_in / res_out may alias.
__global__ void __launch_bounds__(kThreads) cheb_step_kernel(int64_t n, const float* res_in, float* res_out, const float* __restrict__ q,
                                                             float* __restrict__ d, const float* __restrict__ minv, float* __restrict__ e, float a, float b,
                                                             int e_is_zero)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		float r = res_in[i];
		if (q) {
			r -= q[i];
			res_out[i] = r;
		}
		const float dn = (a != 0.0f ? a * d[i] : 0.0f) + b * minv[i] * r;
		d[i]           = dn;
		e[i]           = e_is_zero ? dn : e[i] + dn;
	}
}

// res = r - q
__global__ void __launch_bounds__(kThreads) residual_sub_kernel(int64_t n, const float* __restrict__ r, const float* __restrict__ q, float* __restrict__ res)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) { res[i] = r[i] - q[i]; }
}

// e += e2
__global__ void __launch_bounds__(kThreads) add_kernel(int64_t n, const float* __restrict__ e2, float* __restrict__ e)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) { e[i] += e2[i]; }
}

// ---- transfers -----------------------------------------------------------------------------------------------------
// Prolongation is upscale_field's multilinear, align-corners interpolation (field_interpolation.cpp:431-485): fine node
// i of an axis sits at coarse position t = i * (nc - 1) / (nf - 1), between coarse nodes floor(t) and floor(t) + 1.
// The per-axis tables are computed once on the host in double precision; both kernels read the same tables, so
// restriction is exactly the transpose of prolongation.
constexpr int kMaxFan = 6;  // fine nodes of one axis whose interpolation touches one coarse node (4 for a 2:1 ratio)

struct Xfer  // fine <-> coarse geometry of one level pair; unused axes have nf = nc = 1
{
	int          nf[kMaxDim], nc[kMaxDim];
	const int*   base[kMaxDim];   // [nf]  lower coarse node of fine node i
	const float* frac[kMaxDim];   // [nf]  weight of the upper coarse node (lower gets 1 - frac)
	const int*   first[kMaxDim];  // [nc]  first fine node with a non-zero weight on coarse node C
	const int*   count[kMaxDim];  // [nc]  how many consecutive fine nodes
	const float* weight[kMaxDim]; // [nc][kMaxFan]
};

// e_f += P e_c : every fine node gathers its 2^D coarse neighbours.  Block = 128 threads along x covering kXferRows
// consecutive y rows of one z plane (a block per row was 1 M blocks of 128 threads at 512^3: scheduling-bound, 1.6 TB/s);
// y and z come from the block index (no integer division per node).
constexpr int kXferRows = 4;

__global__ void __launch_bounds__(128) prolong_add_kernel(Xfer x, const float* __restrict__ ec, float* __restrict__ ef)
{
	const int ix = blockIdx.x * 128 + threadIdx.x, iy0 = blockIdx.y * kXferRows, iz = blockIdx.z;
	if (ix >= x.nf[0]) { return; }
	const int   bx = __ldg(x.base[0] + ix), bz = __ldg(x.base[2] + iz);
	const float fx = __ldg(x.frac[0] + ix), fz = __ldg(x.frac[2] + iz);
	// the upper neighbour of the last node does not exist; its weight is zero, the clamped read is harmless
	const int     bx1 = min(bx + 1, x.nc[0] - 1), bz1 = min(bz + 1, x.nc[2] - 1);
	const int64_t sy = x.nc[0], sz = static_cast<int64_t>(x.nc[0]) * x.nc[1];
	const float   gx = 1.0f - fx, gz = 1.0f - fz;
	float         acc[kXferRows], old[kXferRows];
#pragma unroll
	for (int r = 0; r < kXferRows; ++r) {
		const int iy = iy0 + r;
		acc[r]       = 0.0f;
		old[r]       = 0.0f;
		if (iy >= x.nf[1]) { continue; }
		const int    by  = __ldg(x.base[1] + iy);
		const float  fy  = __ldg(x.frac[1] + iy), gy = 1.0f - fy;
		const int    by1 = min(by + 1, x.nc[1] - 1);
		const float* p00 = ec + bz * sz + by * sy;
		const float* p01 = ec + bz * sz + by1 * sy;
		const float* p10 = ec + bz1 * sz + by * sy;
		const float* p11 = ec + bz1 * sz + by1 * sy;
		const float  v00 = gx * __ldg(p00 + bx) + fx * __ldg(p00 + bx1);
		const float  v01 = gx * __ldg(p01 + bx) + fx * __ldg(p01 + bx1);
		const float  v10 = gx * __ldg(p10 + bx) + fx * __ldg(p10 + bx1);
		const float  v11 = gx * __ldg(p11 + bx) + fx * __ldg(p11 + bx1);
		acc[r]           = gz * (gy * v00 + fy * v01) + fz * (gy * v10 + fy * v11);
		old[r]           = ef[(static_cast<int64_t>(iz) * x.nf[1] + iy) * x.nf[0] + ix];
	}
#pragma unroll
	for (int r = 0; r < kXferRows; ++r) {
		const int iy = iy0 + r;
		if (iy < x.nf[1]) { ef[(static_cast<int64_t>(iz) * x.nf[1] + iy) * x.nf[0] + ix] = old[r] + acc[r]; }
	}
}

// The same with four consecutive fine x nodes per thread (x size a multiple of 4): the four nodes interpolate from at most
// four consecutive coarse nodes, so a row costs 4 x 4 scalar loads and one 16-byte read-modify-write instead of 4 x 8 + 4 + 4 —
// the scalar kernel is bound by L1 load issue (1.9 TB/s of DRAM traffic at 512^3).
__device__ __forceinline__ float pick4(const float (&c)[4], int i) { return i == 0 ? c[0] : (i == 1 ? c[1] : (i == 2 ? c[2] : c[3])); }

__global__ void __launch_bounds__(128) prolong_add4_kernel(Xfer x, const float* __restrict__ ec, float* __restrict__ ef)
{
	const int ix0 = (blockIdx.x * 128 + threadIdx.x) * 4, iy0 = blockIdx.y * kXferRows, iz = blockIdx.z;
	if (ix0 >= x.nf[0]) { return; }
	const int4   b4 = *reinterpret_cast<const int4*>(x.base[0] + ix0);
	const float4 f4 = *reinterpret_cast<const float4*>(x.frac[0] + ix0);
	const int    bj[4] = {b4.x, b4.y, b4.z, b4.w};
	const float  fj[4] = {f4.x, f4.y, f4.z, f4.w};
	const int    b0 = b4.x, last = x.nc[0] - 1;
	int          lo[4], hi[4];
#pragma unroll
	for (int j = 0; j < 4; ++j) {
		lo[j] = bj[j] - b0;                  // 0 .. 2
		hi[j] = min(bj[j] + 1, last) - b0;   // 0 .. 3
	}
	const int     bz = __ldg(x.base[2] + iz), bz1 = min(bz + 1, x.nc[2] - 1);
	const float   fz = __ldg(x.frac[2] + iz), gz = 1.0f - fz;
	const int64_t sy = x.nc[0], sz = static_cast<int64_t>(x.nc[0]) * x.nc[1];
	const int     c0 = min(b0, last), c1 = min(b0 + 1, last), c2 = min(b0 + 2, last), c3 = min(b0 + 3, last);
#pragma unroll
	for (int r = 0; r < kXferRows; ++r) {
		const int iy = iy0 + r;
		if (iy >= x.nf[1]) { break; }
		const int   by  = __ldg(x.base[1] + iy), by1 = min(by + 1, x.nc[1] - 1);
		const float fy  = __ldg(x.frac[1] + iy), gy = 1.0f - fy;
		const float* rows[4] = {ec + bz * sz + by * sy, ec + bz * sz + by1 * sy, ec + bz1 * sz + by * sy, ec + bz1 * sz + by1 * sy};
		const float  wrow[4] = {gz * gy, gz * fy, fz * gy, fz * fy};
		float        c[4] = {0.0f, 0.0f, 0.0f, 0.0f};  // the four coarse columns, already combined over the (y, z) neighbours
#pragma unroll
		for (int q = 0; q < 4; ++q) {
			c[0] += wrow[q] * __ldg(rows[q] + c0);
			c[1] += wrow[q] * __ldg(rows[q] + c1);
			c[2] += wrow[q] * __ldg(rows[q] + c2);
			c[3] += wrow[q] * __ldg(rows[q] + c3);
		}
		float4* out = reinterpret_cast<float4*>(ef + (static_cast<int64_t>(iz) * x.nf[1] + iy) * x.nf[0] + ix0);
		float4  v   = *out;
		v.x += (1.0f - fj[0]) * pick4(c, lo[0]) + fj[0] * pick4(c, hi[0]);
		v.y += (1.0f - fj[1]) * pick4(c, lo[1]) + fj[1] * pick4(c, hi[1]);
		v.z += (1.0f - fj[2]) * pick4(c, lo[2]) + fj[2] * pick4(c, hi[2]);
		v.w += (1.0f - fj[3]) * pick4(c, lo[3]) + fj[3] * pick4(c, hi[3]);
		*out = v;
	}
}

// e_f += P e_c with the kernel that fits the lattice (e_f addressed from its first plane; 16-byte aligned rows when the x size
// is a multiple of 4)
void launch_prolong_add(const Xfer& x, int planes, const float* ec, float* ef, cudaStream_t s)
{
	if (x.nf[0] % 4 == 0 && (reinterpret_cast<uintptr_t>(ef) & 15u) == 0) {
		FI_LAUNCH(prolong_add4_kernel, dim3(div_up(x.nf[0] / 4, 128), div_up(x.nf[1], kXferRows), planes), 128, 0, s, x, ec, ef);
	} else {
		FI_LAUNCH(prolong_add_kernel, dim3(div_up(x.nf[0], 128), div_up(x.nf[1], kXferRows), planes), 128, 0, s, x, ec, ef);
	}
}

// r_c = P^T res_f : every coarse node gathers the fine nodes whose interpolation touches it; a block covers kXferRows
// coarse rows.  The hierarchy halves every axis (ceil), so a coarse node is touched by at most kFan = 4 consecutive fine
// nodes per axis: the 4 x 4 x 4 loads of a coarse node are issued branch-free (weights beyond the count are zero, indices
// clamped into the lattice) so that they are all in flight at once — the loop nest with run-time trip counts it replaces
// kept six loads in flight per thread and ran at 1.4 TB/s.
constexpr int kFan = 4;

__global__ void __launch_bounds__(128) restrict_kernel(Xfer x, const float* __restrict__ rf, float* __restrict__ rc)
{
	const int cx = blockIdx.x * 128 + threadIdx.x, cy0 = blockIdx.y * kXferRows, cz = blockIdx.z;
	if (cx >= x.nc[0]) { return; }
	const int    x0 = __ldg(x.first[0] + cx), z0 = __ldg(x.first[2] + cz);
	const int    nx = __ldg(x.count[0] + cx), nz = __ldg(x.count[2] + cz);
	const float* wx = x.weight[0] + static_cast<size_t>(cx) * kMaxFan;
	const float* wz = x.weight[2] + static_cast<size_t>(cz) * kMaxFan;
	float wxr[kFan], wzr[kFan];
	int   xi[kFan], zi[kFan];
#pragma unroll
	for (int i = 0; i < kFan; ++i) {
		wxr[i] = i < nx ? __ldg(wx + i) : 0.0f;
		wzr[i] = i < nz ? __ldg(wz + i) : 0.0f;
		xi[i]  = x0 + min(i, max(nx, 1) - 1);  // beyond the count: the last touched node again (weight zero) — always a valid,
		zi[i]  = z0 + min(i, max(nz, 1) - 1);  // stored address, also on a slab that holds only a window of the planes
	}
	const int64_t sy = x.nf[0], sz = static_cast<int64_t>(x.nf[0]) * x.nf[1];
	for (int r = 0; r < kXferRows; ++r) {
		const int cy = cy0 + r;
		if (cy >= x.nc[1]) { break; }
		const int    y0 = __ldg(x.first[1] + cy), ny = __ldg(x.count[1] + cy);
		const float* wy = x.weight[1] + static_cast<size_t>(cy) * kMaxFan;
		float        acc = 0.0f;
#pragma unroll
		for (int k = 0; k < kFan; ++k) {
			float plane = 0.0f;
#pragma unroll
			for (int j = 0; j < kFan; ++j) {
				const float  wj  = j < ny ? __ldg(wy + j) : 0.0f;
				const float* row = rf + zi[k] * sz + (y0 + min(j, max(ny, 1) - 1)) * sy;
				float        s   = 0.0f;
#pragma unroll
				for (int i = 0; i < kFan; ++i) { s += wxr[i] * __ldg(row + xi[i]); }
				plane += wj * s;
			}
			acc += wzr[k] * plane;
		}
		rc[(static_cast<int64_t>(cz) * x.nc[1] + cy) * x.nc[0] + cx] = acc;
	}
}

// ---- coarsest level: e = Ainv r (dense, one block per row) --------------------------------------------------------
__global__ void dense_matvec_kernel(int n, const float* __restrict__ A, const float* __restrict__ r, float* __restrict__ e)
{
	__shared__ double red[32];
	const int row = blockIdx.x;
	double    acc = 0.0;
	for (int j = threadIdx.x; j < n; j += blockDim.x) { acc += static_cast<double>(A[static_cast<size_t>(row) * n + j]) * static_cast<double>(r[j]); }
	acc = block_sum(acc, red);
	if (threadIdx.x == 0) { e[row] = static_cast<float>(acc); }
}

__global__ void unit_vector_kernel(int n, int k, float* v)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) { v[i] = i == k ? 1.0f : 0.0f; }
}

// ---- the tail of the cycle in one kernel (opt-in: MgOptions::tail_cells / FI_B200_MG_TAIL_CELLS) -----------------------
// Levels of a few thousand nodes are launch latency: a Chebyshev step on 16^3 nodes is three launches of a few
// microseconds each, and a W-cycle visits those levels eight times per iteration (profiles/r2j_mg_launches_512_f64outer_wcycle.md:
// ~500 of the ~985 launches of one iteration at 512^3).  One block of 1024 threads walks the whole tail instead —
// pre-smoothing, residual, restriction down to the dense level and back up — with __syncthreads() where the launches had
// their boundaries.  MEASURED (B200, round 2, profiles/r2p_*): correct, 1345 instead of 1969 launches per two iterations,
// and slower — 283 us per visit (the 16^3 level of the bench cloud has 3375 occupied cells: 27 k float reductions per
// operator application through ONE SM's 1.3 cycles per lane, 13 applications per visit), 512^3 solve 170.6 against
// 163.7 ms, 256^3 50.4 against 47.4 ms, 2D unchanged.  Hence off by default; what would make it pay is the data term
// accumulated in shared memory and a cluster of blocks instead of one.  The arithmetic is the one vcycle_level() launches
// (same Chebyshev recurrence, the generic kernels' operator application, the same transfer tables); sums are formed in
// a different order.  Vectors written inside the kernel are read with plain loads (never __ldg).
constexpr int kTailThreads   = 1024;
constexpr int kTailMaxLevels = 6;
constexpr int kTailMaxNu     = 16;

struct TailLevel
{
	int             ndim, n, nocc, radius, nu, any;
	int             size[kMaxDim], stride[kMaxDim];
	float           gs2, b0;
	float           ca[kTailMaxNu], cb[kTailMaxNu];  // Chebyshev step k = 1 .. nu-1: d = ca[k] d + cb[k] M^-1 res
	float           band[kMaxDim][9][9];
	const int64_t*  cell_base;
	const uint32_t* cell_mask;
	const float*    blocks;
	const float*    minv;
	float *         r, *e, *res, *d, *q;  // r / e: the level's own (the kernel arguments replace them on the first tail level)
	Xfer            x;                    // to the next tail level
};

__device__ __forceinline__ int tail_row_class(int i, int n) { return n <= 9 ? i : (i < 4 ? i : (i >= n - 4 ? i - n + 9 : 4)); }

__device__ __forceinline__ int tail_lap1(int i, int n, int o)
{
	if (o == 0) { return (i > 0 ? 1 : 0) + (i < n - 1 ? 1 : 0); }
	const int j = i + o;
	return (j >= 0 && j < n) ? -1 : 0;
}

// out = (S + P) in on level L; ends with a block barrier
template <int D>
__device__ void tail_apply(const TailLevel& L, const float* in, float* out)
{
	constexpr int C = 1 << D;
	for (int i = threadIdx.x; i < L.n; i += blockDim.x) {
		int c[kMaxDim] = {0, 0, 0};
		int rem        = i;
#pragma unroll
		for (int d = 0; d < D; ++d) {
			if (d == D - 1) {
				c[d] = rem;
			} else {
				c[d] = rem % L.size[d];
				rem /= L.size[d];
			}
		}
		float acc = 0.0f;
		if (L.any) {
			const int R = L.radius;
#pragma unroll
			for (int d = 0; d < D; ++d) {
				const float* row = L.band[d][tail_row_class(c[d], L.size[d])];
				for (int o = -R; o <= R; ++o) {
					const float coef = row[o + 4];
					if (coef != 0.0f) { acc += coef * in[i + o * L.stride[d]]; }  // taps beyond the lattice have zero coefficients
				}
			}
			if (L.gs2 != 0.0f) {
#pragma unroll
				for (int d = 0; d < D; ++d) {
#pragma unroll
					for (int o = d + 1; o < D; ++o) {
						for (int a = -1; a <= 1; ++a) {
							const int la = tail_lap1(c[d], L.size[d], a);
							if (la == 0) { continue; }
							for (int b = -1; b <= 1; ++b) {
								const int lb = tail_lap1(c[o], L.size[o], b);
								if (lb != 0) { acc += L.gs2 * static_cast<float>(la * lb) * in[i + a * L.stride[d] + b * L.stride[o]]; }
							}
						}
					}
				}
			}
		}
		out[i] = acc;
	}
	__syncthreads();
	for (int cell = threadIdx.x; cell < L.nocc; cell += blockDim.x) {
		const int      base = static_cast<int>(L.cell_base[cell]);
		const uint32_t mask = L.cell_mask[cell];
		float          pc[C], acc[C];
		int            off[C];
#pragma unroll
		for (int c = 0; c < C; ++c) {
			off[c] = 0;
#pragma unroll
			for (int d = 0; d < D; ++d) { off[c] += ((c >> d) & 1) ? L.stride[d] : 0; }
			pc[c]  = ((mask >> c) & 1u) ? in[base + off[c]] : 0.0f;
			acc[c] = 0.0f;
		}
		int tri = 0;
#pragma unroll
		for (int ci = 0; ci < C; ++ci) {
#pragma unroll
			for (int cj = ci; cj < C; ++cj) {
				const float v = __ldg(&L.blocks[static_cast<size_t>(tri) * L.nocc + cell]);
				acc[ci] += v * pc[cj];
				if (cj != ci) { acc[cj] += v * pc[ci]; }
				++tri;
			}
		}
#pragma unroll
		for (int c = 0; c < C; ++c) {
			if ((mask >> (8 + c)) & 1u) { atomicAdd(&out[base + off[c]], acc[c]); }
		}
	}
	__syncthreads();
}

// nu Chebyshev steps on A e = r (smooth() above); e_zero: e starts at zero.  Returns with the residual BEFORE the last
// correction in res_src (r itself after a single step from zero) and the last correction in L.d.
template <int D>
__device__ const float* tail_smooth(const TailLevel& L, const float* r, float* e, bool e_zero)
{
	const float* res_src = r;
	if (e_zero) {
		for (int i = threadIdx.x; i < L.n; i += blockDim.x) {
			const float dn = L.b0 * __ldg(&L.minv[i]) * r[i];
			L.d[i]         = dn;
			e[i]           = dn;
		}
		__syncthreads();
	} else {
		tail_apply<D>(L, e, L.q);
		for (int i = threadIdx.x; i < L.n; i += blockDim.x) {
			const float rr = r[i] - L.q[i];
			const float dn = L.b0 * __ldg(&L.minv[i]) * rr;
			L.res[i]       = rr;
			L.d[i]         = dn;
			e[i] += dn;
		}
		__syncthreads();
		res_src = L.res;
	}
	for (int k = 1; k < L.nu; ++k) {
		tail_apply<D>(L, L.d, L.q);
		const float a = L.ca[k], b = L.cb[k];
		for (int i = threadIdx.x; i < L.n; i += blockDim.x) {
			const float rr = res_src[i] - L.q[i];
			const float dn = a * L.d[i] + b * __ldg(&L.minv[i]) * rr;
			L.res[i]       = rr;
			L.d[i]         = dn;
			e[i] += dn;
		}
		__syncthreads();
		res_src = L.res;
	}
	return res_src;
}

template <int D>
__global__ void __launch_bounds__(kTailThreads, 1) mg_tail_kernel(const TailLevel* __restrict__ levels, int nlev, int nc, const float* __restrict__ coarse_inv,
                                                                   const float* r_top, float* e_top)
{
	__shared__ TailLevel L;
	__shared__ double    part[kTailThreads];
	auto load_level = [&](int l) {
		__syncthreads();
		const int* src = reinterpret_cast<const int*>(levels + l);
		int*       dst = reinterpret_cast<int*>(&L);
		for (int k = threadIdx.x; k < static_cast<int>(sizeof(TailLevel) / sizeof(int)); k += blockDim.x) { dst[k] = src[k]; }
		__syncthreads();
	};
	// down: pre-smooth from zero, residual after the last correction, restrict
	for (int l = 0; l + 1 < nlev; ++l) {
		load_level(l);
		const float* r   = l == 0 ? r_top : L.r;
		float*       e   = l == 0 ? e_top : L.e;
		const float* src = tail_smooth<D>(L, r, e, true);
		tail_apply<D>(L, L.d, L.q);
		for (int i = threadIdx.x; i < L.n; i += blockDim.x) { L.res[i] = src[i] - L.q[i]; }
		__syncthreads();
		const Xfer& x   = L.x;
		float*      rc  = levels[l + 1].r;
		const int   ncx = x.nc[0], ncy = x.nc[1], ncz = x.nc[2];
		for (int cn = threadIdx.x; cn < ncx * ncy * ncz; cn += blockDim.x) {
			const int    cx = cn % ncx, cy = (cn / ncx) % ncy, cz = cn / (ncx * ncy);
			const int    x0 = __ldg(x.first[0] + cx), y0 = __ldg(x.first[1] + cy), z0 = __ldg(x.first[2] + cz);
			const int    nx = __ldg(x.count[0] + cx), ny = __ldg(x.count[1] + cy), nz = __ldg(x.count[2] + cz);
			const float* wx = x.weight[0] + static_cast<size_t>(cx) * kMaxFan;
			const float* wy = x.weight[1] + static_cast<size_t>(cy) * kMaxFan;
			const float* wz = x.weight[2] + static_cast<size_t>(cz) * kMaxFan;
			float        acc = 0.0f;
			for (int k = 0; k < nz; ++k) {
				float plane = 0.0f;
				for (int j = 0; j < ny; ++j) {
					const float* row = L.res + (static_cast<size_t>(z0 + k) * x.nf[1] + (y0 + j)) * x.nf[0] + x0;
					float        s   = 0.0f;
					for (int i = 0; i < nx; ++i) { s += __ldg(wx + i) * row[i]; }
					plane += __ldg(wy + j) * s;
				}
				acc += __ldg(wz + k) * plane;
			}
			rc[cn] = acc;
		}
	}
	// coarsest level: e = Ainv r with the dense inverse (symmetric: column `row` is read, so that a warp reads consecutive
	// floats); nc <= blockDim.x / 2 splits a row over several threads
	{
		load_level(nlev - 1);
		const float* r     = nlev == 1 ? r_top : L.r;
		float*       e     = nlev == 1 ? e_top : L.e;
		const int    parts = nc < static_cast<int>(blockDim.x) ? static_cast<int>(blockDim.x) / nc : 1;
		if (parts == 1) {
			for (int row = threadIdx.x; row < nc; row += blockDim.x) {
				double acc = 0.0;
				for (int j = 0; j < nc; ++j) { acc += static_cast<double>(__ldg(&coarse_inv[static_cast<size_t>(j) * nc + row])) * static_cast<double>(r[j]); }
				e[row] = static_cast<float>(acc);
			}
		} else {
			const int row = threadIdx.x % nc, pt = threadIdx.x / nc;
			double    acc = 0.0;
			if (pt < parts) {
				for (int j = pt; j < nc; j += parts) { acc += static_cast<double>(__ldg(&coarse_inv[static_cast<size_t>(j) * nc + row])) * static_cast<double>(r[j]); }
			}
			part[threadIdx.x] = acc;
			__syncthreads();
			if (pt == 0) {
				for (int k = 1; k < parts; ++k) { acc += part[k * nc + row]; }
				e[row] = static_cast<float>(acc);
			}
		}
	}
	// up: add the prolonged correction, post-smooth
	for (int l = nlev - 2; l >= 0; --l) {
		load_level(l);
		const float* r  = l == 0 ? r_top : L.r;
		float*       e  = l == 0 ? e_top : L.e;
		const Xfer&  x  = L.x;
		const float* ec = levels[l + 1].e;
		const int    nfx = x.nf[0], nfy = x.nf[1];
		const int    sy = x.nc[0], sz = x.nc[0] * x.nc[1];
		for (int i = threadIdx.x; i < L.n; i += blockDim.x) {
			const int   ix = i % nfx, iy = (i / nfx) % nfy, iz = i / (nfx * nfy);
			const int   bx = __ldg(x.base[0] + ix), by = __ldg(x.base[1] + iy), bz = __ldg(x.base[2] + iz);
			const float fx = __ldg(x.frac[0] + ix), fy = __ldg(x.frac[1] + iy), fz = __ldg(x.frac[2] + iz);
			// the upper neighbour of the last node does not exist; its weight is zero, the clamped read is harmless
			const int   bx1 = min(bx + 1, x.nc[0] - 1), by1 = min(by + 1, x.nc[1] - 1), bz1 = min(bz + 1, x.nc[2] - 1);
			const float gx = 1.0f - fx, gy = 1.0f - fy, gz = 1.0f - fz;
			const float v00 = gx * ec[bz * sz + by * sy + bx] + fx * ec[bz * sz + by * sy + bx1];
			const float v01 = gx * ec[bz * sz + by1 * sy + bx] + fx * ec[bz * sz + by1 * sy + bx1];
			const float v10 = gx * ec[bz1 * sz + by * sy + bx] + fx * ec[bz1 * sz + by * sy + bx1];
			const float v11 = gx * ec[bz1 * sz + by1 * sy + bx] + fx * ec[bz1 * sz + by1 * sy + bx1];
			e[i] += gz * (gy * v00 + fy * v01) + fz * (gy * v10 + fy * v11);
		}
		__syncthreads();
		tail_smooth<D>(L, r, e, false);
	}
}

// ---- the coarsest operator as a dense matrix, written directly ---------------------------------------------------------
// cols[j * n + i] = A[i][j] for a level described by a TailLevel (no generic rows, no tile mask): the smoothness rows by one
// thread per node — only thread i writes entries of row i, plain read-modify-writes on the zeroed matrix — then the cell
// blocks by one thread per occupied cell with atomics.  Replaces n applications of the operator to unit vectors (3 launches
// each: 1536 launches, 6 ms of host launch time, for the 512 nodes under a 512^3 lattice).
template <int D>
__global__ void dense_stencil_kernel(TailLevel L, float* __restrict__ cols)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= L.n || !L.any) { return; }
	int c[kMaxDim] = {0, 0, 0};
	int rem        = i;
#pragma unroll
	for (int d = 0; d < D; ++d) {
		if (d == D - 1) {
			c[d] = rem;
		} else {
			c[d] = rem % L.size[d];
			rem /= L.size[d];
		}
	}
	const size_t n = static_cast<size_t>(L.n);
	const int    R = L.radius;
#pragma unroll
	for (int d = 0; d < D; ++d) {
		const float* row = L.band[d][tail_row_class(c[d], L.size[d])];
		for (int o = -R; o <= R; ++o) {
			const float coef = row[o + 4];
			if (coef != 0.0f) { cols[static_cast<size_t>(i + o * L.stride[d]) * n + i] += coef; }
		}
	}
	if (L.gs2 != 0.0f) {
#pragma unroll
		for (int d = 0; d < D; ++d) {
#pragma unroll
			for (int o = d + 1; o < D; ++o) {
				for (int a = -1; a <= 1; ++a) {
					const int la = tail_lap1(c[d], L.size[d], a);
					if (la == 0) { continue; }
					for (int b = -1; b <= 1; ++b) {
						const int lb = tail_lap1(c[o], L.size[o], b);
						if (lb != 0) { cols[static_cast<size_t>(i + a * L.stride[d] + b * L.stride[o]) * n + i] += L.gs2 * static_cast<float>(la * lb); }
					}
				}
			}
		}
	}
}

template <int D>
__global__ void dense_blocks_kernel(TailLevel L, float* __restrict__ cols)
{
	constexpr int C    = 1 << D;
	const int     cell = blockIdx.x * blockDim.x + threadIdx.x;
	if (cell >= L.nocc) { return; }
	const int      base = static_cast<int>(L.cell_base[cell]);
	const uint32_t mask = L.cell_mask[cell];
	const size_t   n    = static_cast<size_t>(L.n);
	int            node[C];
#pragma unroll
	for (int c = 0; c < C; ++c) {
		node[c] = base;
#pragma unroll
		for (int d = 0; d < D; ++d) { node[c] += ((c >> d) & 1) ? L.stride[d] : 0; }
	}
	int tri = 0;
#pragma unroll
	for (int ci = 0; ci < C; ++ci) {
#pragma unroll
		for (int cj = ci; cj < C; ++cj) {
			const float v = L.blocks[static_cast<size_t>(tri) * L.nocc + cell];
			// apply_blocks_kernel: out[ci] += v p[cj] when corner cj is a lattice node and the row of corner ci is owned
			if (((mask >> cj) & 1u) && ((mask >> (8 + ci)) & 1u)) { atomicAdd(&cols[static_cast<size_t>(node[cj]) * n + node[ci]], v); }
			if (cj != ci && ((mask >> ci) & 1u) && ((mask >> (8 + cj)) & 1u)) { atomicAdd(&cols[static_cast<size_t>(node[ci]) * n + node[cj]], v); }
			++tri;
		}
	}
}

// ---- power iteration helpers ----------------------------------------------------------------------------------------
// v[i] = pseudo-random in [-0.5, 0.5) from the lattice index i + first (a slab fills its planes with the values the
// unsharded vector has there)
__global__ void hash_fill_kernel(int64_t n, float* v, int64_t first)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		uint64_t h = static_cast<uint64_t>(i + first) * 0x9E3779B97F4A7C15ull + 0x7F4A7C15ull;
		h ^= h >> 31;
		h *= 0xBF58476D1CE4E5B9ull;
		h ^= h >> 29;
		v[i] = static_cast<float>(static_cast<double>(h >> 11) * (1.0 / 9007199254740992.0)) - 0.5f;
	}
}

// w = M^-1 q; out[0] = w.w, out[1] = v.w
__global__ void __launch_bounds__(kThreads) power_step_kernel(int64_t n, const float* __restrict__ v, const float* __restrict__ q,
                                                              const float* __restrict__ minv, float* __restrict__ w, double* out, double* partial,
                                                              unsigned* ticket)
{
	__shared__ double red[32];
	double            acc[2] = {0, 0};
	const int64_t     stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		const float wi = minv[i] * q[i];
		w[i]           = wi;
		acc[0] += static_cast<double>(wi) * wi;
		acc[1] += static_cast<double>(v[i]) * wi;
	}
	acc[0] = block_sum(acc[0], red);
	acc[1] = block_sum(acc[1], red);
	grid_sum<2>(acc, partial, ticket, red, [&](const double(&tot)[2]) {
		out[0] = tot[0];
		out[1] = tot[1];
	});
}

__global__ void scale_kernel(int64_t n, float* v, float a)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) { v[i] *= a; }
}

// ---- outer CG kernels -------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads) mg_residual_kernel(int64_t n, const T* __restrict__ b, const T* __restrict__ q, T* __restrict__ r, float* __restrict__ r32,
                                                               double* out, double* partial, unsigned* ticket)
{
	__shared__ double red[32];
	double            acc[2] = {0, 0};
	const int64_t     stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		const T bi = b[i], ri = bi - q[i];
		r[i]   = ri;
		r32[i] = static_cast<float>(ri);
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

// x += alpha p, r -= alpha q, r32 = float(r); out[0] = r.r
template <typename T>
__global__ void __launch_bounds__(kThreads) mg_update_kernel(int64_t n, T* __restrict__ x, T* __restrict__ r, const T* __restrict__ p, const T* __restrict__ q,
                                                             float* __restrict__ r32, T alpha, double* out, double* partial, unsigned* ticket)
{
	__shared__ double red[32];
	double            acc[1] = {0};
	const int64_t     stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		x[i] += alpha * p[i];
		const T ri = r[i] - alpha * q[i];
		r[i]   = ri;
		r32[i] = static_cast<float>(ri);
		acc[0] += static_cast<double>(ri) * static_cast<double>(ri);
	}
	acc[0] = block_sum(acc[0], red);
	grid_sum<1>(acc, partial, ticket, red, [&](const double(&tot)[1]) { out[0] = tot[0]; });
}

// out[0] = r.z
template <typename T>
__global__ void __launch_bounds__(kThreads) mg_dot_kernel(int64_t n, const T* __restrict__ r, const float* __restrict__ z, double* out, double* partial,
                                                          unsigned* ticket)
{
	__shared__ double red[32];
	double            acc[1] = {0};
	const int64_t     stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
		acc[0] += static_cast<double>(r[i]) * static_cast<double>(z[i]);
	}
	acc[0] = block_sum(acc[0], red);
	grid_sum<1>(acc, partial, ticket, red, [&](const double(&tot)[1]) { out[0] = tot[0]; });
}

// p = z + beta p
template <typename T>
__global__ void __launch_bounds__(kThreads) mg_direction_kernel(int64_t n, const float* __restrict__ z, T* __restrict__ p, T beta)
{
	const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) { p[i] = static_cast<T>(z[i]) + beta * p[i]; }
}

// ---- coarsest level setup: dense inverse on the device -------------------------------------------------------------
// M = (C + C^T) / 2 in fp64 (the applied operator is symmetric up to the fp32 rounding of the data term's atomics)
__global__ void symmetrise_kernel(int n, const float* __restrict__ cols, double* __restrict__ M)
{
	const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (t >= static_cast<int64_t>(n) * n) { return; }
	const int i = static_cast<int>(t / n), j = static_cast<int>(t % n);
	M[t] = 0.5 * (static_cast<double>(cols[static_cast<size_t>(i) * n + j]) + static_cast<double>(cols[static_cast<size_t>(j) * n + i]));
}

// Gauss-Jordan step c, out of place: row c <- the scaled pivot row (with the identity's column folded in); every other row
// r <- row r (column c cleared) - M[r][c] * pivot row.  Every thread reads the pivot, its pivot-row and pivot-column
// entries from `in` itself (L1 / L2 hits), so a step is one launch; in and out alternate.
__global__ void gj_step_kernel(int n, int c, const double* __restrict__ in, double* __restrict__ out, int* bad)
{
	const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (t >= static_cast<int64_t>(n) * n) { return; }
	const int    r = static_cast<int>(t / n), k = static_cast<int>(t % n);
	const double p = in[static_cast<size_t>(c) * n + c];
	if (t == 0 && !(p > 0.0)) { *bad = 1; }
	const double inv  = p != 0.0 ? 1.0 / p : 0.0;
	const double prow = (k == c ? 1.0 : in[static_cast<size_t>(c) * n + k]) * inv;
	const double pcol = in[static_cast<size_t>(r) * n + c];
	out[t] = r == c ? prow : (k == c ? 0.0 : in[t]) - pcol * prow;
}

__global__ void narrow_kernel(int64_t n, const double* __restrict__ in, float* __restrict__ out)
{
	const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (t < n) { out[t] = static_cast<float>(in[t]); }
}

}  // namespace

struct Multigrid::Level
{
	Geom                             g;
	Operator<float>*                 op = nullptr;   // level 0: the caller's operator; coarser: owned below
	std::unique_ptr<Operator<float>> owned;
	PointStore                       pts;
	DevBuf<float>                    r, e, res, d, d2, q;  // r / e of level 0 are the caller's vectors; d / d2 ping-pong
	DevBuf<float>                    r2, e2;               // W-cycle: residual after the first coarse correction and its correction
	double                           lmax = 0;
	Xfer                             to_coarser;     // this level (fine) -> next level (coarse)
	DevBuf<int>                      xfer_int;       // backing store of to_coarser's tables
	DevBuf<float>                    xfer_float;
};

namespace {

// Interpolation tables of one axis of a level pair (nf fine nodes, nc coarse nodes); the arithmetic is upscale_field's
// position rule (field_interpolation.cpp:462) evaluated in double.
struct AxisTables
{
	std::vector<int>   base, first, count;  // base[nf]; first[nc], count[nc]
	std::vector<float> frac, weight;        // frac[nf]; weight[nc][kMaxFan]
};

AxisTables axis_tables(int nf, int nc)
{
	AxisTables t;
	const double sc = nf > 1 ? static_cast<double>(nc - 1) / static_cast<double>(nf - 1) : 0.0;
	t.base.assign(nf, 0);
	t.first.assign(nc, 0);
	t.count.assign(nc, 0);
	t.frac.assign(nf, 0.0f);
	t.weight.assign(static_cast<size_t>(nc) * kMaxFan, 0.0f);
	for (int i = 0; i < nf; ++i) {
		const double x = i * sc;
		int          b = static_cast<int>(x);
		if (b > nc - 1) { b = nc - 1; }
		t.base[i] = b;
		t.frac[i] = static_cast<float>(x - b);
	}
	for (int i = 0; i < nf; ++i) {  // transpose: scatter every fine node's two weights to its coarse nodes
		const int   b = t.base[i];
		const float w[2] = {1.0f - t.frac[i], t.frac[i]};
		for (int k = 0; k < 2; ++k) {
			const int C = b + k;
			if (C >= nc || w[k] == 0.0f) { continue; }
			if (t.count[C] == 0) { t.first[C] = i; }
			const int at = i - t.first[C];
			FI_REQUIRE(at < 4, FI_ERR_UNSUPPORTED, "multigrid: coarsening ratio too large for the transfer kernels (more than 4 fine nodes per coarse node)");
			t.weight[static_cast<size_t>(C) * kMaxFan + at] = w[k];
			t.count[C] = at + 1;
		}
	}
	return t;
}

// Device copy of the tables of all axes of the pair (gf = fine, gc = coarse lattice sizes; unused axes have nf = nc = 1).
void build_xfer(Xfer& x, DevBuf<int>& xfer_int, DevBuf<float>& xfer_float, const Geom& gf, const Geom& gc, cudaStream_t s)
{
	std::vector<int>   hi;
	std::vector<float> hf;
	size_t off_base[kMaxDim], off_first[kMaxDim], off_count[kMaxDim], off_frac[kMaxDim], off_weight[kMaxDim];
	for (int d = 0; d < kMaxDim; ++d) {
		const int nf = d < gf.ndim ? gf.size[d] : 1, nc = d < gf.ndim ? gc.size[d] : 1;
		x.nf[d] = nf;
		x.nc[d] = nc;
		const AxisTables t = axis_tables(nf, nc);
		off_base[d]  = hi.size(); hi.insert(hi.end(), t.base.begin(), t.base.end());
		off_first[d] = hi.size(); hi.insert(hi.end(), t.first.begin(), t.first.end());
		off_count[d] = hi.size(); hi.insert(hi.end(), t.count.begin(), t.count.end());
		off_frac[d]   = hf.size(); hf.insert(hf.end(), t.frac.begin(), t.frac.end());
		off_weight[d] = hf.size(); hf.insert(hf.end(), t.weight.begin(), t.weight.end());
	}
	xfer_int.resize(hi.size());
	xfer_float.resize(hf.size());
	FI_CUDA(cudaMemcpyAsync(xfer_int.data(), hi.data(), hi.size() * sizeof(int), cudaMemcpyHostToDevice, s));
	FI_CUDA(cudaMemcpyAsync(xfer_float.data(), hf.data(), hf.size() * sizeof(float), cudaMemcpyHostToDevice, s));
	FI_CUDA(cudaStreamSynchronize(s));  // the host vectors go out of scope
	for (int d = 0; d < kMaxDim; ++d) {
		x.base[d]   = xfer_int.data() + off_base[d];
		x.first[d]  = xfer_int.data() + off_first[d];
		x.count[d]  = xfer_int.data() + off_count[d];
		x.frac[d]   = xfer_float.data() + off_frac[d];
		x.weight[d] = xfer_float.data() + off_weight[d];
	}
}

void build_xfer(Multigrid::Level& lv, const Geom& gc, cudaStream_t s) { build_xfer(lv.to_coarser, lv.xfer_int, lv.xfer_float, lv.g, gc, s); }

// Model and points of level `la` (>= 1) of the hierarchy whose level 0 is the lattice root_size with `model` and `pts`:
// the same points in the coarse lattice's coordinates, gradient rows / 2 per level, order-k smoothness rows scaled by
// 2^((D - 2k) / 2) per level (squared weights by 2^(D - 2k)).
void level_inputs(int D, const int* root_size, const ModelAccum& model, const PointStore& pts, const Geom& gl, int la, ModelAccum& m, PointStore& out,
                  cudaStream_t s)
{
	m = model;
	for (int k = 0; k <= 4; ++k) {
		const double f = std::pow(2.0, static_cast<double>(D - 2 * k) * la);
		for (int a = 0; a < 5; ++a) {
			for (int b = 0; b < 5; ++b) { m.cc[k][a][b] *= f; }
		}
	}
	m.gs_sq *= std::pow(2.0, static_cast<double>(D - 4) * la);
	const int64_t n = pts.count;
	if (n > 0) {
		out.pos.resize(static_cast<size_t>(n) * D);
		out.grad.resize(static_cast<size_t>(n) * D);
		out.value.resize(n);
		out.vw.resize(n);
		out.gw.resize(n);
		out.kind.resize(n);
		out.count = n;
		float sc[kMaxDim] = {1, 1, 1};
		for (int d = 0; d < D; ++d) {
			sc[d] = root_size[d] > 1 ? static_cast<float>(static_cast<double>(gl.size[d] - 1) / static_cast<double>(root_size[d] - 1)) : 0.0f;
		}
		FI_LAUNCH(coarsen_points_kernel, div_up(n, kThreads), kThreads, 0, s, D, n, pts.pos.data(), pts.gw.data(), sc[0], sc[1], sc[2],
		          static_cast<float>(std::pow(0.5, la)), out.pos.data(), out.gw.data());
		FI_CUDA(cudaMemcpyAsync(out.grad.data(), pts.grad.data(), static_cast<size_t>(n) * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
		FI_CUDA(cudaMemcpyAsync(out.value.data(), pts.value.data(), n * sizeof(float), cudaMemcpyDeviceToDevice, s));
		FI_CUDA(cudaMemcpyAsync(out.vw.data(), pts.vw.data(), n * sizeof(float), cudaMemcpyDeviceToDevice, s));
		FI_CUDA(cudaMemcpyAsync(out.kind.data(), pts.kind.data(), n * sizeof(uint8_t), cudaMemcpyDeviceToDevice, s));
	}
}

}  // namespace

void mg_options_from_env(MgOptions& o)
{
	auto geti = [](const char* name, int& v) {
		if (const char* e = getenv(name)) {
			if (atoi(e) > 0 || (e[0] == '0' && e[1] == 0 && std::string(name) == "FI_B200_MG_NU_COARSE")) { v = atoi(e); }
		}
	};
	geti("FI_B200_MG_COARSEST", o.coarsest_cells);
	geti("FI_B200_MG_NU_COARSE", o.nu_coarse);
	geti("FI_B200_MG_GAMMA", o.gamma);
	geti("FI_B200_MG_WLEVELS", o.w_levels);
	if (const char* e = getenv("FI_B200_MG_TAIL_CELLS")) { o.tail_cells = atoi(e); }  // 0: every level by its own launches
}

namespace {

// The operator of a small level as the single-kernel paths read it (mg_tail_kernel, dense_*_kernel).  false: it has generic
// rows, a tile mask or a slab window — those stay with the general kernels.
bool describe_operator(Operator<float>& op, TailLevel& t)
{
	std::memset(&t, 0, sizeof(t));
	if (op.data.nrows > 0 || op.g.tile != 0 || op.g.sharded() || op.dist != nullptr || op.g.N > (1 << 20)) { return false; }
	t.ndim   = op.g.ndim;
	t.n      = static_cast<int>(op.g.N);
	t.nocc   = static_cast<int>(op.data.nocc);
	t.radius = op.tabs.radius;
	t.any    = op.tabs.any ? 1 : 0;
	t.gs2    = static_cast<float>(op.tabs.gs2);
	for (int d = 0; d < kMaxDim; ++d) {
		t.size[d]   = op.g.size[d];
		t.stride[d] = static_cast<int>(op.g.stride[d]);
		for (int c = 0; c < 9; ++c) {
			for (int k = 0; k < 9; ++k) { t.band[d][c][k] = static_cast<float>(op.tabs.band[d][c][k]); }
		}
	}
	t.cell_base = op.data.cell_base.data();
	t.cell_mask = op.data.cell_mask.data();
	t.blocks    = op.data.blocks.data();
	t.minv      = op.minv.data();
	return true;
}

// Chooses the levels mg_tail_kernel walks (the last ones, from the first with at most opt.tail_cells nodes; level 0 is never
// one of them: it is the caller's operator and may carry generic rows or a tile mask) and writes their descriptors.
void build_tail(Multigrid& mg, cudaStream_t s)
{
	const int L = static_cast<int>(mg.levels.size());
	mg.tail_from = 0;
	mg.tail_nlev = 0;
	if (mg.opt.tail_cells <= 0 || L < 3) { return; }
	int from = L - 1;
	while (from - 1 >= 1 && mg.levels[from - 1]->g.N <= mg.opt.tail_cells && L - (from - 1) <= kTailMaxLevels) { --from; }
	if (from >= L - 1) { return; }  // only the dense level: one launch either way
	std::vector<TailLevel> h(static_cast<size_t>(L - from));
	for (int l = from; l < L; ++l) {
		Multigrid::Level& lv = *mg.levels[l];
		Operator<float>&  op = *lv.op;
		TailLevel&        t  = h[static_cast<size_t>(l - from)];
		if (!describe_operator(op, t)) { return; }
		t.r         = lv.r.data();
		t.e         = lv.e.data();
		if (l < L - 1) {
			// the coefficients smooth() passes to its kernels
			const int nu = (l + mg.base_level > 0 && mg.opt.nu_coarse > 0) ? mg.opt.nu_coarse : mg.opt.nu;
			if (nu < 1 || nu > kTailMaxNu) { return; }
			const double lmax = lv.lmax, lmin = lmax / mg.opt.cheb_ratio;
			const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sigma = theta / delta;
			t.nu  = nu;
			t.b0  = static_cast<float>(1.0 / theta);
			double rho = 1.0 / sigma;
			for (int k = 1; k < nu; ++k) {
				const double rho_new = 1.0 / (2.0 * sigma - rho);
				t.ca[k] = static_cast<float>(rho_new * rho);
				t.cb[k] = static_cast<float>(2.0 * rho_new / delta);
				rho     = rho_new;
			}
			t.res = lv.res.data();
			t.d   = lv.d.data();
			t.q   = lv.q.data();
			t.x   = lv.to_coarser;
		}
	}
	mg.tail_plan.resize(h.size() * sizeof(TailLevel));
	FI_CUDA(cudaMemcpyAsync(mg.tail_plan.data(), h.data(), h.size() * sizeof(TailLevel), cudaMemcpyHostToDevice, s));
	FI_CUDA(cudaStreamSynchronize(s));  // the host vector goes out of scope
	mg.tail_from = from;
	mg.tail_nlev = L - from;
}

}  // namespace

Multigrid::Multigrid()  = default;
Multigrid::~Multigrid()
{
	if (exec) { cudaGraphExecDestroy(exec); }
}

std::unique_ptr<Multigrid> build_multigrid(Operator<float>& fine, const ModelAccum& model, const PointStore& pts, const MgOptions& opt, cudaStream_t s,
                                           const int* root_size, int fine_level)
{
	TraceScope trace("build_multigrid");
	FI_REQUIRE(!fine.g.sharded(), FI_ERR_UNSUPPORTED, "build_multigrid takes an unsharded lattice (slabs: build_slab_multigrid)");
	if (!root_size) { root_size = fine.g.size; }
	auto mg     = std::make_unique<Multigrid>();
	mg->opt     = opt;
	mg->base_level = fine_level;
	const int D = fine.g.ndim;
	// levels
	{
		auto l0 = std::make_unique<Multigrid::Level>();
		l0->g   = fine.g;
		l0->op  = &fine;
		mg->levels.push_back(std::move(l0));
	}
	while (static_cast<int>(mg->levels.size()) < 20) {
		const Geom& gf = mg->levels.back()->g;
		int32_t     nc[kMaxDim] = {1, 1, 1};
		int64_t     cells = 1;
		bool        shrunk = false;
		int         smallest_next = 1 << 30;
		for (int d = 0; d < D; ++d) {
			nc[d] = (gf.size[d] + 1) / 2;
			shrunk = shrunk || nc[d] < gf.size[d];
			cells *= nc[d];
			if (gf.size[d] > 1) { smallest_next = std::min(smallest_next, nc[d]); }
		}
		// stop once the current level is small enough for the dense solve, or the next one would have fewer than 4 nodes
		// along an axis (too few for the higher-order difference rows to mean anything)
		if (gf.N <= opt.coarsest_cells || !shrunk || smallest_next < 4) { break; }
		auto lv = std::make_unique<Multigrid::Level>();
		lv->g   = make_geom(D, nc);
		mg->levels.push_back(std::move(lv));
	}
	const int L = static_cast<int>(mg->levels.size());
	FI_REQUIRE(mg->levels.back()->g.N <= 4096, FI_ERR_UNSUPPORTED, "multigrid: coarsest level too large for the dense solve");
	// coarse operators by re-discretisation
	for (int l = 1; l < L; ++l) {
		TraceScope tl("coarse level operator");
		Multigrid::Level& lv = *mg->levels[l];
		ModelAccum        m;
		level_inputs(D, root_size, model, pts, lv.g, fine_level + l, m, lv.pts, s);
		HostRows none;
		lv.owned = build_operator<float>(lv.g, m, lv.pts, none, s);
		lv.op    = lv.owned.get();
		lv.op->use_fast = kStencilAuto;
	}
	// work vectors and transfer geometry
	for (int l = 0; l < L; ++l) {
		Multigrid::Level& lv = *mg->levels[l];
		const size_t      n  = static_cast<size_t>(lv.g.N);
		if (l > 0) {
			lv.r.resize(n);
			lv.e.resize(n);
			if (opt.gamma > 1 && l < L - 1) {
				lv.r2.resize(n);
				lv.e2.resize(n);
			}
		}
		if (l < L - 1) {
			lv.res.resize(n);
			lv.d.resize(n);
			lv.d2.resize(n);
			lv.q.resize(n);
			build_xfer(lv, mg->levels[l + 1]->g, s);
		}
	}
	// largest eigenvalue of D^-1 A per smoothed level: power iteration
	{
		TraceScope tp("power iterations");
		// v_k = (D^-1 A)^k v_0 without normalising in between (|v| grows by lambda <= ~8 per round: 20 rounds stay far inside
		// fp32) — the squared norms of all rounds and levels are read back once, lambda = |v_K| / |v_K-1|.  Normalising every
		// round cost a kernel over the level and a host synchronisation each (16.6 ms at 512^3, profiles/r2p_trace_time_to_tol_512.txt).
		const int        K = std::max(2, opt.power_iterations);
		DevBuf<double>   out(static_cast<size_t>(2) * K * std::max(1, L - 1)), partial(static_cast<size_t>(2) * (static_cast<size_t>(sm_count()) * 8 + 8));
		DevBuf<unsigned> ticket(1);
		ticket.zero(s);
		for (int l = 0; l < L - 1; ++l) {
			Multigrid::Level& lv = *mg->levels[l];
			const int64_t     n  = lv.g.N;
			float *           v = lv.d.data(), *w = lv.res.data();
			FI_LAUNCH(hash_fill_kernel, vgrid(n), kThreads, 0, s, n, v, static_cast<int64_t>(0));
			for (int it = 0; it < K; ++it) {
				lv.op->apply(v, lv.q.data(), nullptr, nullptr, s);
				FI_LAUNCH(power_step_kernel, vgrid(n), kThreads, 0, s, n, v, lv.q.data(), lv.op->minv.data(), w, out.data() + 2 * (static_cast<size_t>(l) * K + it),
				          partial.data(), ticket.data());
				std::swap(v, w);
			}
		}
		if (L > 1) {
			std::vector<double> h(static_cast<size_t>(2) * K * (L - 1));
			FI_CUDA(cudaMemcpyAsync(h.data(), out.data(), h.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
			FI_CUDA(cudaStreamSynchronize(s));
			for (int l = 0; l < L - 1; ++l) {
				const double n1 = h[2 * (static_cast<size_t>(l) * K + K - 1)], n0 = h[2 * (static_cast<size_t>(l) * K + K - 2)];
				FI_REQUIRE(n0 > 0 && n1 > 0 && std::isfinite(n0) && std::isfinite(n1), FI_ERR_INVALID, "multigrid: power iteration broke down");
				mg->levels[l]->lmax = std::sqrt(n1 / n0) * 1.1;  // the power iteration approaches lambda_max from below
			}
		}
	}
	// dense inverse of the coarsest operator, computed on the device: the columns A e_k by n applies without a
	// host round trip, then an in-place Gauss-Jordan sweep in fp64 (no pivoting: the matrix is SPD)
	{
		TraceScope        td("dense inverse of the coarsest level");
		Multigrid::Level& lc = *mg->levels[L - 1];
		const int         n  = static_cast<int>(lc.g.N);
		mg->nc               = n;
		if (L == 1) { lc.r.resize(n); }  // scratch for the unit vectors (level 0 owns no vectors otherwise)
		const size_t   nn = static_cast<size_t>(n) * n;
		DevBuf<float>  cols(nn);
		DevBuf<double> M(nn), M2(nn);
		TailLevel      desc;
		const char*    by_apply = getenv("FI_B200_MG_DENSE_APPLY");  // test switch: the columns by n operator applications, as below
		if (!(by_apply && by_apply[0] == '1') && describe_operator(*lc.op, desc)) {  // the matrix written directly: two launches
			cols.zero(s);
			const int D = lc.g.ndim;
			auto ks = D == 3 ? dense_stencil_kernel<3> : (D == 2 ? dense_stencil_kernel<2> : dense_stencil_kernel<1>);
			auto kb = D == 3 ? dense_blocks_kernel<3> : (D == 2 ? dense_blocks_kernel<2> : dense_blocks_kernel<1>);
			FI_LAUNCH(ks, div_up(n, kThreads), kThreads, 0, s, desc, cols.data());
			if (desc.nocc > 0) { FI_LAUNCH(kb, div_up(desc.nocc, kThreads), kThreads, 0, s, desc, cols.data()); }
		} else {  // generic rows or a tile mask (a lattice small enough to be its own coarsest level): column k = A e_k
			for (int k = 0; k < n; ++k) {
				FI_LAUNCH(unit_vector_kernel, div_up(n, kThreads), kThreads, 0, s, n, k, lc.r.data());
				lc.op->apply(lc.r.data(), cols.data() + static_cast<size_t>(k) * n, nullptr, nullptr, s);
			}
		}
		const int g2 = static_cast<int>(div_up(static_cast<int64_t>(nn), kThreads));
		FI_LAUNCH(symmetrise_kernel, g2, kThreads, 0, s, n, cols.data(), M.data());
		DevBuf<int> bad(1);
		bad.zero(s);
		double *gin = M.data(), *gout = M2.data();
		for (int c = 0; c < n; ++c) {
			FI_LAUNCH(gj_step_kernel, g2, kThreads, 0, s, n, c, static_cast<const double*>(gin), gout, bad.data());
			std::swap(gin, gout);
		}
		mg->coarse_inv.resize(nn);
		FI_LAUNCH(narrow_kernel, g2, kThreads, 0, s, static_cast<int64_t>(nn), static_cast<const double*>(gin), mg->coarse_inv.data());
		int h_bad = 0;
		FI_CUDA(cudaMemcpyAsync(&h_bad, bad.data(), sizeof(int), cudaMemcpyDeviceToHost, s));
		FI_CUDA(cudaStreamSynchronize(s));
		FI_REQUIRE(h_bad == 0, FI_ERR_INVALID, "multigrid: the coarsest operator is singular");
	}
	build_tail(*mg, s);
	return mg;
}

namespace {

// res_out = res_in - A in and, with d_new, d_new = a in + b M^-1 res_out, e += d_new, in one pass over the level
// (TMA stencil kernel in epilogue mode + the data term's fix-up).  false: not applicable here, nothing was done.
bool fused_step(Multigrid::Level& lv, const float* in, const float* res_in, float* res_out, float* e, float* d_new, float a, float b, cudaStream_t s)
{
	Operator<float>& op = *lv.op;
	if (op.data.nrows > 0 || op.use_fast != kStencilAuto) { return false; }
	if (!(op.g.ndim == 2 ? stencil_tma_2d_epilogue<float>(op.g, op.tabs, in, res_in, res_out, op.minv.data(), e, d_new, a, b, s)
	                     : stencil_tma_3d_epilogue<float>(op.g, op.tabs, in, res_in, res_out, op.minv.data(), e, d_new, a, b, s))) {
		return false;
	}
	const bool ok = apply_data_term_epilogue<float>(op.g, op.data, in, res_out, op.minv.data(), e, d_new, b, s);
	FI_REQUIRE(ok, FI_ERR_UNSUPPORTED, "multigrid: data-term epilogue refused after the stencil epilogue ran");
	return true;
}

struct Smoothed
{
	const float* res;  // residual before the last correction: r - A e = res - A d
	float*       d;    // the last correction
};

// nu Chebyshev steps on A e = r at one level.  e_zero: e starts at zero (pre-smoothing).
Smoothed smooth(Multigrid::Level& lv, const MgOptions& opt, int nu, const float* r, float* e, bool e_zero, cudaStream_t s)
{
	const int64_t n     = lv.g.N;
	const double  lmax  = lv.lmax, lmin = lmax / opt.cheb_ratio;
	const double  theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sigma = theta / delta;
	float *       d = lv.d.data(), *d_other = lv.d2.data(), *res = lv.res.data();
	const float*  res_src = r;
	const float   b0 = static_cast<float>(1.0 / theta);
	if (e_zero) {  // res = r: d = b0 M^-1 r, e = d
		FI_LAUNCH(cheb_step_kernel, vgrid(n), kThreads, 0, s, n, r, res, static_cast<const float*>(nullptr), d, lv.op->minv.data(), e, 0.0f, b0, 1);
	} else if (fused_step(lv, e, r, res, nullptr, nullptr, 0.0f, 0.0f, s)) {  // res = r - A e, then the first step from it
		FI_LAUNCH(cheb_step_kernel, vgrid(n), kThreads, 0, s, n, res, res, static_cast<const float*>(nullptr), d, lv.op->minv.data(), e, 0.0f, b0, 0);
		res_src = res;
	} else {
		lv.op->apply(e, lv.q.data(), nullptr, nullptr, s);
		FI_LAUNCH(cheb_step_kernel, vgrid(n), kThreads, 0, s, n, r, res, static_cast<const float*>(lv.q.data()), d, lv.op->minv.data(), e, 0.0f, b0, 0);
		res_src = res;
	}
	double rho = 1.0 / sigma;
	for (int k = 1; k < nu; ++k) {
		const double rho_new = 1.0 / (2.0 * sigma - rho);
		const float  a = static_cast<float>(rho_new * rho), b = static_cast<float>(2.0 * rho_new / delta);
		if (fused_step(lv, d, res_src, res, e, d_other, a, b, s)) {
			std::swap(d, d_other);
		} else {
			lv.op->apply(d, lv.q.data(), nullptr, nullptr, s);
			FI_LAUNCH(cheb_step_kernel, vgrid(n), kThreads, 0, s, n, res_src, res, static_cast<const float*>(lv.q.data()), d, lv.op->minv.data(), e, a, b, 0);
		}
		res_src = res;
		rho     = rho_new;
	}
	return Smoothed{res_src, d};
}

void vcycle_level(Multigrid& mg, int l, const float* r, float* e, cudaStream_t s)
{
	const int L = static_cast<int>(mg.levels.size());
	Multigrid::Level& lv = *mg.levels[l];
	// the last levels in one kernel — unless a W-cycle would still recurse twice somewhere below this level
	if (mg.tail_from > 0 && l == mg.tail_from && (mg.opt.gamma <= 1 || l + 1 + mg.base_level > mg.opt.w_levels)) {
		const TailLevel* plan = reinterpret_cast<const TailLevel*>(mg.tail_plan.data());
		auto kern = lv.g.ndim == 3 ? mg_tail_kernel<3> : (lv.g.ndim == 2 ? mg_tail_kernel<2> : mg_tail_kernel<1>);
		FI_LAUNCH(kern, 1, kTailThreads, 0, s, plan, mg.tail_nlev, mg.nc, static_cast<const float*>(mg.coarse_inv.data()), r, e);
		return;
	}
	if (l == L - 1) {
		FI_LAUNCH(dense_matvec_kernel, mg.nc, 128, 0, s, mg.nc, mg.coarse_inv.data(), r, e);
		return;
	}
	Multigrid::Level& lc = *mg.levels[l + 1];
	const int         nu = (l + mg.base_level > 0 && mg.opt.nu_coarse > 0) ? mg.opt.nu_coarse : mg.opt.nu;
	const Smoothed    sm = smooth(lv, mg.opt, nu, r, e, true, s);
	// residual after the last correction, restricted
	if (!fused_step(lv, sm.d, sm.res, lv.res.data(), nullptr, nullptr, 0.0f, 0.0f, s)) {
		lv.op->apply(sm.d, lv.q.data(), nullptr, nullptr, s);
		FI_LAUNCH(residual_sub_kernel, vgrid(lv.g.N), kThreads, 0, s, lv.g.N, sm.res, lv.q.data(), lv.res.data());
	}
	{
		const Xfer& x = lv.to_coarser;
		FI_LAUNCH(restrict_kernel, dim3(div_up(x.nc[0], 128), div_up(x.nc[1], kXferRows), x.nc[2]), 128, 0, s, x, lv.res.data(), lc.r.data());
	}
	vcycle_level(mg, l + 1, lc.r.data(), lc.e.data(), s);
	if (mg.opt.gamma > 1 && l + 1 < L - 1 && l + 1 + mg.base_level <= mg.opt.w_levels) {  // W-cycle: a second coarse correction, on what the first one left
		lc.op->apply(lc.e.data(), lc.q.data(), nullptr, nullptr, s);
		FI_LAUNCH(residual_sub_kernel, vgrid(lc.g.N), kThreads, 0, s, lc.g.N, static_cast<const float*>(lc.r.data()), static_cast<const float*>(lc.q.data()), lc.r2.data());
		vcycle_level(mg, l + 1, lc.r2.data(), lc.e2.data(), s);
		FI_LAUNCH(add_kernel, vgrid(lc.g.N), kThreads, 0, s, lc.g.N, static_cast<const float*>(lc.e2.data()), lc.e.data());
	}
	{
		const Xfer& x = lv.to_coarser;
		launch_prolong_add(x, x.nf[2], lc.e.data(), e, s);
	}
	smooth(lv, mg.opt, nu, r, e, false, s);
}

}  // namespace

void Multigrid::vcycle(const float* r, float* z, cudaStream_t s)
{
	if (exec && graph_r == r && graph_z == z) {
		FI_CUDA(cudaGraphLaunch(exec, s));
		count_launch(static_cast<int>(graph_launches));
		return;
	}
	if (exec) {
		cudaGraphExecDestroy(exec);
		exec = nullptr;
	}
	cudaGraph_t   graph  = nullptr;
	const int64_t before = g_launches;
	FI_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
	try {
		vcycle_level(*this, 0, r, z, s);
	} catch (...) {
		cudaStreamEndCapture(s, &graph);
		if (graph) { cudaGraphDestroy(graph); }
		throw;
	}
	FI_CUDA(cudaStreamEndCapture(s, &graph));
	graph_launches = g_launches - before;
	g_launches     = before;
	FI_CUDA(cudaGraphInstantiate(&exec, graph, 0));
	cudaGraphDestroy(graph);
	graph_r = r;
	graph_z = z;
	FI_CUDA(cudaGraphLaunch(exec, s));
	count_launch(static_cast<int>(graph_launches));
}

bool Multigrid::demote_to_v_cycle()
{
	if (opt.gamma <= 1) { return false; }
	opt.gamma = 1;
	if (exec) {
		cudaGraphExecDestroy(exec);
		exec = nullptr;
	}
	return true;
}

// ---- test hook: the hierarchy and one stage of its cycle ---------------------------------------------------------------
void mg_info(const Multigrid& mg, fi_mg_info* out)
{
	const int L = static_cast<int>(mg.levels.size());
	FI_REQUIRE(L <= FI_MG_MAX_LEVELS, FI_ERR_RANGE, "multigrid: more levels than fi_mg_info holds");
	std::memset(out, 0, sizeof(*out));
	out->levels = L;
	for (int l = 0; l < L; ++l) {
		const Multigrid::Level& lv = *mg.levels[l];
		for (int d = 0; d < kMaxDim; ++d) { out->sizes[l][d] = d < lv.g.ndim ? lv.g.size[d] : 1; }
		out->lmax[l] = l + 1 < L ? lv.lmax : 0.0;
	}
	out->nu         = mg.opt.nu;
	out->nu_coarse  = mg.opt.nu_coarse;
	out->gamma      = mg.opt.gamma;
	out->w_levels   = mg.opt.w_levels;
	out->cheb_ratio = mg.opt.cheb_ratio;
	out->tail_from  = mg.tail_from;
	out->coarsest   = mg.nc;
}

void mg_stage(Multigrid& mg, int stage, int level, int64_t count, const float* in, const float* in2, float* out, cudaStream_t s)
{
	const int L = static_cast<int>(mg.levels.size());
	FI_REQUIRE(level >= 0 && level < L, FI_ERR_INVALID, "mg_stage: no such level");
	FI_REQUIRE(count >= 0 && (count == 0 || (in != nullptr && out != nullptr)), FI_ERR_INVALID, "mg_stage: in / out is null");
	Multigrid::Level& lv = *mg.levels[level];
	const bool        coarser = level + 1 < L;
	const int64_t     n = lv.g.N, nc = coarser ? mg.levels[level + 1]->g.N : 0;
	int64_t           n_in = n, n_out = n;
	bool              takes_in2 = false;
	switch (stage) {
	case FI_MG_CYCLE: FI_REQUIRE(level == 0, FI_ERR_INVALID, "mg_stage: the cycle starts at level 0"); break;
	case FI_MG_OPERATOR: break;
	case FI_MG_RESTRICT:
		FI_REQUIRE(coarser, FI_ERR_INVALID, "mg_stage: the coarsest level restricts nowhere");
		n_out = nc;
		break;
	case FI_MG_PROLONG_ADD:
		FI_REQUIRE(coarser, FI_ERR_INVALID, "mg_stage: nothing prolongs into the coarsest level");
		n_in      = nc;
		takes_in2 = true;
		break;
	case FI_MG_SMOOTH:
		FI_REQUIRE(coarser, FI_ERR_INVALID, "mg_stage: the coarsest level is solved, not smoothed");
		takes_in2 = true;
		break;
	case FI_MG_COARSE: FI_REQUIRE(level == L - 1, FI_ERR_INVALID, "mg_stage: the dense solve is on the coarsest level"); break;
	default: throw Error{FI_ERR_INVALID, "mg_stage: unknown stage"};
	}
	if (stage == FI_MG_CYCLE && mg.exec) {  // capture afresh: the caller may have changed the fine operator's kernel choice
		cudaGraphExecDestroy(mg.exec);
		mg.exec = nullptr;
	}
	DevBuf<float> din(static_cast<size_t>(n_in)), dout(static_cast<size_t>(n_out));
	const int     nu = (level + mg.base_level > 0 && mg.opt.nu_coarse > 0) ? mg.opt.nu_coarse : mg.opt.nu;
	for (int64_t k = 0; k < count; ++k) {
		FI_CUDA(cudaMemcpyAsync(din.data(), in + k * n_in, n_in * sizeof(float), cudaMemcpyHostToDevice, s));
		if (takes_in2) {
			if (in2) {
				FI_CUDA(cudaMemcpyAsync(dout.data(), in2 + k * n_out, n_out * sizeof(float), cudaMemcpyHostToDevice, s));
			} else {
				dout.zero(s);
			}
		}
		switch (stage) {
		case FI_MG_CYCLE: mg.vcycle(din.data(), dout.data(), s); break;
		case FI_MG_OPERATOR: lv.op->apply(din.data(), dout.data(), nullptr, nullptr, s); break;
		case FI_MG_RESTRICT: {
			const Xfer& x = lv.to_coarser;
			FI_LAUNCH(restrict_kernel, dim3(div_up(x.nc[0], 128), div_up(x.nc[1], kXferRows), x.nc[2]), 128, 0, s, x, din.data(), dout.data());
			break;
		}
		case FI_MG_PROLONG_ADD: launch_prolong_add(lv.to_coarser, lv.to_coarser.nf[2], din.data(), dout.data(), s); break;
		case FI_MG_SMOOTH: smooth(lv, mg.opt, nu, din.data(), dout.data(), in2 == nullptr, s); break;
		case FI_MG_COARSE: FI_LAUNCH(dense_matvec_kernel, mg.nc, 128, 0, s, mg.nc, mg.coarse_inv.data(), din.data(), dout.data()); break;
		}
		FI_CUDA(cudaMemcpyAsync(out + k * n_out, dout.data(), n_out * sizeof(float), cudaMemcpyDeviceToHost, s));
		FI_CUDA(cudaStreamSynchronize(s));
	}
}

// ---- the V-cycle with z-slab sharded fine levels ------------------------------------------------------------------------
struct SlabMultigrid::DLevel
{
	Geom                             g;             // this rank's slab of the level (halo planes either side)
	DistHooks*                       hooks = nullptr;  // level 0: the fine operator's; coarser: owned below
	std::unique_ptr<DistHooks>       owned_hooks;
	Operator<float>*                 op = nullptr;  // level 0: the caller's operator; coarser: owned below
	std::unique_ptr<Operator<float>> owned;
	PointStore                       pts;
	DevBuf<float>                    r, e, res, d, d2, q;  // slab-local; r / e of level 0 are the caller's vectors (d2: ping-pong partner of d)
	double                           lmax = 0;
	Xfer                             to_coarser;    // tables over the WHOLE axes of this level and the next
	DevBuf<int>                      xfer_int;
	DevBuf<float>                    xfer_float;
	int                              c0 = 0, c1 = 0;  // planes of the next level this rank restricts into
};

SlabMultigrid::SlabMultigrid()  = default;
SlabMultigrid::~SlabMultigrid() = default;

SlabMgPlan plan_slab_multigrid(const int32_t* sizes, int world, int radius, int64_t gather_cells, const int* cuts)
{
	FI_REQUIRE(sizes != nullptr && world >= 1 && radius >= 1 && radius <= 4, FI_ERR_INVALID, "bad slab multigrid request");
	SlabMgPlan plan;
	plan.world = world;
	plan.halo  = std::max(radius, 2);  // restriction reads up to two planes below the middle one
	auto tma_ok = [](const int* n) { return n[0] % 4 == 0 && n[0] >= 32 && n[1] >= 8; };  // stencil_tma.cu: eligible<float>()
	for (int d = 0; d < kMaxDim; ++d) { plan.size[0][d] = sizes[d]; }
	FI_REQUIRE(tma_ok(plan.size[0]), FI_ERR_UNSUPPORTED, "slab multigrid: the x size must be a multiple of 4 and >= 32, the y size >= 8");
	plan.own[0].resize(world);
	for (int k = 0; k < world; ++k) {
		if (cuts) {
			plan.own[0][k] = std::make_pair(cuts[k], cuts[k + 1]);
		} else {
			slab_range(sizes[2], world, k, &plan.own[0][k].first, &plan.own[0][k].second);
		}
		FI_REQUIRE(plan.own[0][k].second - plan.own[0][k].first >= plan.halo, FI_ERR_UNSUPPORTED, "slab multigrid: slabs thinner than the halo: use fewer ranks");
	}
	for (int l = 0;; ++l) {
		// the next level and who restricts into which of its planes
		int*       nc = plan.size[l + 1];
		const int* nf = plan.size[l];
		int        smallest = 1 << 30;
		int64_t    cells = 1;
		for (int d = 0; d < kMaxDim; ++d) {
			nc[d] = (nf[d] + 1) / 2;
			cells *= nc[d];
			smallest = std::min(smallest, nc[d]);
		}
		FI_REQUIRE(smallest >= 4, FI_ERR_UNSUPPORTED, "slab multigrid: the lattice is too small to coarsen");
		const AxisTables tz = axis_tables(nf[2], nc[2]);
		auto owner_of_fine = [&](int z) {
			for (int k = 0; k < world; ++k) {
				if (z >= plan.own[l][k].first && z < plan.own[l][k].second) { return k; }
			}
			return -1;
		};
		std::vector<std::pair<int, int>>& oc = plan.own[l + 1];
		oc.assign(world, std::make_pair(-1, -1));
		int last_owner = 0;
		for (int C = 0; C < nc[2]; ++C) {
			FI_REQUIRE(tz.count[C] >= 1, FI_ERR_UNSUPPORTED, "slab multigrid: a coarse plane without fine planes");
			const int mid = tz.first[C] + tz.count[C] / 2;  // the middle one of the fine planes restriction reads
			const int k   = owner_of_fine(std::min(mid, tz.first[C] + tz.count[C] - 1));
			FI_REQUIRE(k >= last_owner, FI_ERR_UNSUPPORTED, "slab multigrid: coarse plane owners are not monotone");
			last_owner = k;
			if (oc[k].first < 0) { oc[k].first = C; }
			oc[k].second = C + 1;
			// restriction of this plane stays inside the owner's stored window
			FI_REQUIRE(tz.first[C] >= plan.own[l][k].first - plan.halo && tz.first[C] + tz.count[C] <= plan.own[l][k].second + plan.halo, FI_ERR_UNSUPPORTED,
			           "slab multigrid: restriction reaches beyond the halo planes");
		}
		for (int k = 0; k < world; ++k) {
			FI_REQUIRE(oc[k].first >= 0, FI_ERR_UNSUPPORTED, "slab multigrid: a rank owns no plane of a coarse level: use fewer ranks");
			FI_REQUIRE(k == 0 ? oc[k].first == 0 : oc[k].first == oc[k - 1].second, FI_ERR_UNSUPPORTED, "slab multigrid: coarse planes are not partitioned");
		}
		FI_REQUIRE(oc[world - 1].second == nc[2], FI_ERR_UNSUPPORTED, "slab multigrid: coarse planes are not partitioned");
		plan.nd = l + 1;
		// is the next level sharded too?
		bool shard = cells > gather_cells && tma_ok(nc) && l + 2 <= kMaxSlabLevels && (nc[2] + 1) / 2 >= 4;
		for (int k = 0; shard && k < world; ++k) {
			shard = oc[k].second - oc[k].first >= plan.halo;
			// prolongation into this rank's planes of level l reads planes base, base + 1 of level l + 1: inside its window there
			for (int z = plan.own[l][k].first; shard && z < plan.own[l][k].second; ++z) {
				const int b0 = tz.base[z], b1 = std::min(tz.base[z] + 1, nc[2] - 1);
				shard = b0 >= oc[k].first - plan.halo && b1 < oc[k].second + plan.halo;
			}
		}
		if (!shard) { break; }
	}
	return plan;
}

std::unique_ptr<SlabMultigrid> build_slab_multigrid(Operator<float>& fine, const ModelAccum& model, const PointStore& pts, const MgOptions& opt,
                                                    const SlabMgPlan& plan, cudaStream_t s)
{
	TraceScope trace("build_slab_multigrid");
	FI_REQUIRE(fine.dist != nullptr && fine.g.ndim == 3, FI_ERR_INVALID, "build_slab_multigrid needs a 3D slab operator with its communicator hooks");
	DistHooks& hooks0 = *fine.dist;
	const int  rank = hooks0.rank(), world = hooks0.world();
	FI_REQUIRE(world == plan.world && plan.nd >= 1, FI_ERR_INVALID, "slab multigrid: the plan is for another communicator");
	FI_REQUIRE(opt.gamma <= 1, FI_ERR_UNSUPPORTED, "slab multigrid: the sharded levels run V-cycles only");
	FI_REQUIRE(fine.g.zown0 == plan.halo && fine.g.zoff == plan.own[0][rank].first - plan.halo && fine.g.zown1 - fine.g.zown0 == plan.own[0][rank].second - plan.own[0][rank].first,
	           FI_ERR_INVALID, "slab multigrid: the fine operator's slab is not the plan's");
	auto mg  = std::make_unique<SlabMultigrid>();
	mg->opt  = opt;
	mg->plan = plan;
	mg->rank = rank;
	const int D = 3;
	HostRows  none;
	// sharded levels
	for (int l = 0; l < plan.nd; ++l) {
		auto lv = std::make_unique<SlabMultigrid::DLevel>();
		if (l == 0) {
			lv->g     = fine.g;
			lv->op    = &fine;
			lv->hooks = &hooks0;
		} else {
			lv->g           = make_slab_geom(plan.size[l], plan.own[l][rank].first, plan.own[l][rank].second, plan.halo);
			lv->owned_hooks = hooks0.for_geom(lv->g, plan.halo);
			FI_REQUIRE(lv->owned_hooks != nullptr, FI_ERR_UNSUPPORTED, "slab multigrid: the communicator cannot serve another level");
			lv->hooks = lv->owned_hooks.get();
			ModelAccum m;
			level_inputs(D, plan.size[0], model, pts, lv->g, l, m, lv->pts, s);
			lv->owned       = build_operator<float>(lv->g, m, lv->pts, none, s);
			lv->op          = lv->owned.get();
			lv->op->dist    = lv->hooks;
			lv->op->use_fast = kStencilAuto;
		}
		lv->c0 = plan.own[l + 1][rank].first;
		lv->c1 = plan.own[l + 1][rank].second;
		const size_t n = static_cast<size_t>(lv->g.N);
		if (l > 0) {
			lv->r.resize(n);
			lv->e.resize(n);
			lv->r.zero(s);
			lv->e.zero(s);
		}
		lv->res.resize(n);
		lv->d.resize(n);
		lv->d2.resize(n);
		lv->q.resize(n);
		lv->res.zero(s);  // halo planes and planes beyond the lattice must be finite (zero) before anything reads them
		lv->d.zero(s);
		lv->d2.zero(s);
		lv->q.zero(s);
		const Geom gf = make_geom(D, plan.size[l]), gc = make_geom(D, plan.size[l + 1]);
		build_xfer(lv->to_coarser, lv->xfer_int, lv->xfer_float, gf, gc, s);
		mg->dl.push_back(std::move(lv));
	}
	// the first replicated level and everything below it
	{
		const Geom gt = make_geom(D, plan.size[plan.nd]);
		ModelAccum m;
		level_inputs(D, plan.size[0], model, pts, gt, plan.nd, m, mg->tail_pts, s);
		mg->tail_op           = build_operator<float>(gt, m, mg->tail_pts, none, s);
		mg->tail_op->use_fast = kStencilAuto;
		mg->tail              = build_multigrid(*mg->tail_op, model, pts, opt, s, plan.size[0], plan.nd);
		mg->tail_r.resize(static_cast<size_t>(gt.N));
		mg->tail_e.resize(static_cast<size_t>(gt.N));
		mg->tail_r.zero(s);
		mg->tail_e.zero(s);
	}
	// largest eigenvalue of D^-1 A per sharded level: power iteration from the start vector the unsharded hierarchy uses
	{
		DevBuf<double>   out(2), partial(static_cast<size_t>(2) * (static_cast<size_t>(sm_count()) * 8 + 8));
		DevBuf<unsigned> ticket(1);
		ticket.zero(s);
		for (int l = 0; l < plan.nd; ++l) {
			SlabMultigrid::DLevel& lv  = *mg->dl[l];
			const int64_t          off = lv.g.own_offset(), n = lv.g.own_cells();
			float *                v = lv.d.data(), *w = lv.res.data();
			FI_LAUNCH(hash_fill_kernel, vgrid(n), kThreads, 0, s, n, v + off, static_cast<int64_t>(plan.own[l][rank].first) * lv.g.stride[2]);
			double lam = 1.0;
			for (int it = 0; it < opt.power_iterations; ++it) {
				lv.hooks->exchange_halo(v, sizeof(float), s);
				lv.op->apply(v, lv.q.data(), nullptr, nullptr, s);
				FI_LAUNCH(power_step_kernel, vgrid(n), kThreads, 0, s, n, v + off, lv.q.data() + off, lv.op->minv.data() + off, w + off, out.data(), partial.data(),
				          ticket.data());
				lv.hooks->allreduce(out.data(), 2, s);
				double h[2];
				FI_CUDA(cudaMemcpyAsync(h, out.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
				FI_CUDA(cudaStreamSynchronize(s));
				const double nw = std::sqrt(h[0]);
				FI_REQUIRE(nw > 0 && std::isfinite(nw), FI_ERR_INVALID, "slab multigrid: power iteration broke down");
				lam = nw;
				FI_LAUNCH(scale_kernel, vgrid(n), kThreads, 0, s, n, w + off, static_cast<float>(1.0 / nw));
				std::swap(v, w);
			}
			lv.lmax = lam * 1.1;
			// the smoother expects clean work vectors: halo planes are refilled by exchanges, owned planes overwritten
		}
	}
	return mg;
}

namespace {

// One pass over the slab's owned planes after refreshing the halo planes of `in` from the neighbours:
//     res_out = res_in - A in   and, with d_new,   d_new = a in + b M^-1 res_out,   e += d_new
// — the TMA stencil kernel in epilogue mode plus the data term's fix-up when they apply (28 B/cell), else the plain
// operator and a vector kernel (8 + 32 B/cell).  Without d_new only the residual is formed.  d_new must not alias in.
void slab_step(SlabMultigrid::DLevel& lv, float* in, const float* res_in, float* res_out, float* e, float* d_new, float a, float b, cudaStream_t s)
{
	const int64_t    off = lv.g.own_offset(), n = lv.g.own_cells();
	Operator<float>& op  = *lv.op;
	lv.hooks->exchange_halo(in, sizeof(float), s);
	if (op.data.nrows == 0 && op.use_fast == kStencilAuto &&
	    stencil_tma_3d_epilogue<float>(op.g, op.tabs, in, res_in, res_out, op.minv.data(), e, d_new, a, b, s)) {
		const bool ok = apply_data_term_epilogue<float>(op.g, op.data, in, res_out, op.minv.data(), e, d_new, b, s);
		FI_REQUIRE(ok, FI_ERR_UNSUPPORTED, "slab multigrid: data-term epilogue refused after the stencil epilogue ran");
		return;
	}
	op.apply(in, lv.q.data(), nullptr, nullptr, s);
	if (d_new == nullptr) {
		FI_LAUNCH(residual_sub_kernel, vgrid(n), kThreads, 0, s, n, res_in + off, static_cast<const float*>(lv.q.data() + off), res_out + off);
		return;
	}
	// the vector kernel updates the direction in place: bring it to d_new first
	FI_CUDA(cudaMemcpyAsync(d_new + off, in + off, static_cast<size_t>(n) * sizeof(float), cudaMemcpyDeviceToDevice, s));
	FI_LAUNCH(cheb_step_kernel, vgrid(n), kThreads, 0, s, n, res_in + off, res_out + off, static_cast<const float*>(lv.q.data() + off), d_new + off,
	          op.minv.data() + off, e + off, a, b, 0);
}

// nu Chebyshev steps on A e = r over the slab's owned planes (smooth() on a slab).  Returns the residual before the last
// correction and the last correction, like smooth().
Smoothed slab_smooth(SlabMultigrid::DLevel& lv, const MgOptions& opt, int nu, const float* r, float* e, bool e_zero, cudaStream_t s)
{
	const int64_t off = lv.g.own_offset(), n = lv.g.own_cells();
	const double  lmax  = lv.lmax, lmin = lmax / opt.cheb_ratio;
	const double  theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin), sigma = theta / delta;
	float *       d = lv.d.data(), *d_other = lv.d2.data(), *res = lv.res.data();
	const float*  minv = lv.op->minv.data();
	const float*  res_src = r;
	const float   b0 = static_cast<float>(1.0 / theta);
	if (e_zero) {  // res = r: d = b0 M^-1 r, e = d
		FI_LAUNCH(cheb_step_kernel, vgrid(n), kThreads, 0, s, n, r + off, res + off, static_cast<const float*>(nullptr), d + off, minv + off, e + off, 0.0f, b0, 1);
	} else {  // res = r - A e, then the first step from it
		slab_step(lv, e, r, res, nullptr, nullptr, 0.0f, 0.0f, s);
		FI_LAUNCH(cheb_step_kernel, vgrid(n), kThreads, 0, s, n, res + off, res + off, static_cast<const float*>(nullptr), d + off, minv + off, e + off, 0.0f, b0, 0);
		res_src = res;
	}
	double rho = 1.0 / sigma;
	for (int k = 1; k < nu; ++k) {
		const double rho_new = 1.0 / (2.0 * sigma - rho);
		const float  a = static_cast<float>(rho_new * rho), b = static_cast<float>(2.0 * rho_new / delta);
		slab_step(lv, d, res_src, res, e, d_other, a, b, s);
		std::swap(d, d_other);
		res_src = res;
		rho     = rho_new;
	}
	return Smoothed{res_src, d};
}

void slab_vcycle_level(SlabMultigrid& mg, int l, const float* r, float* e, cudaStream_t s)
{
	SlabMultigrid::DLevel& lv  = *mg.dl[l];
	const int64_t          off = lv.g.own_offset(), n = lv.g.own_cells();
	const int              z0 = mg.plan.own[l][mg.rank].first, z1 = mg.plan.own[l][mg.rank].second;
	const bool             last = l + 1 == mg.plan.nd;
	const int              nu = (l > 0 && mg.opt.nu_coarse > 0) ? mg.opt.nu_coarse : mg.opt.nu;
	const Smoothed         sm = slab_smooth(lv, mg.opt, nu, r, e, true, s);
	// residual after the last correction
	slab_step(lv, sm.d, sm.res, lv.res.data(), nullptr, nullptr, 0.0f, 0.0f, s);
	lv.hooks->exchange_halo(lv.res.data(), sizeof(float), s);
	// restriction into the planes [c0, c1) of the next level: the kernel indexes fine planes by their lattice z, so the
	// slab pointer is moved back by the slab's first stored plane; the z tables start at c0
	const int64_t plane_f = lv.g.stride[2];
	const int64_t plane_c = static_cast<int64_t>(lv.to_coarser.nc[0]) * lv.to_coarser.nc[1];
	{
		Xfer x = lv.to_coarser;
		x.first[2] += lv.c0;
		x.count[2] += lv.c0;
		x.weight[2] += static_cast<size_t>(lv.c0) * kMaxFan;
		const float* rf = lv.res.data() - static_cast<int64_t>(lv.g.zoff) * plane_f;
		float*       rc = last ? mg.tail_r.data() + static_cast<int64_t>(lv.c0) * plane_c : mg.dl[l + 1]->r.data() + mg.dl[l + 1]->g.own_offset();
		FI_LAUNCH(restrict_kernel, dim3(div_up(x.nc[0], 128), div_up(x.nc[1], kXferRows), lv.c1 - lv.c0), 128, 0, s, x, rf, rc);
	}
	const float* ec = nullptr;  // the coarse correction, indexable by the lattice z of the next level
	if (last) {
		lv.hooks->allgather_planes(mg.tail_r.data(), plane_c, mg.plan.own[l + 1], s);
		mg.tail->vcycle(mg.tail_r.data(), mg.tail_e.data(), s);
		ec = mg.tail_e.data();
	} else {
		SlabMultigrid::DLevel& lc = *mg.dl[l + 1];
		slab_vcycle_level(mg, l + 1, lc.r.data(), lc.e.data(), s);
		lc.hooks->exchange_halo(lc.e.data(), sizeof(float), s);
		ec = lc.e.data() - static_cast<int64_t>(lc.g.zoff) * plane_c;
	}
	{
		Xfer x = lv.to_coarser;
		x.base[2] += z0;
		x.frac[2] += z0;
		launch_prolong_add(x, z1 - z0, ec, e + off, s);
	}
	slab_smooth(lv, mg.opt, nu, r, e, false, s);
}

}  // namespace

void SlabMultigrid::vcycle(const float* r, float* z, cudaStream_t s) { slab_vcycle_level(*this, 0, r, z, s); }

// CG on A x = b preconditioned by one V-cycle per iteration.  Scalars travel through the host (three small reads
// per iteration against several milliseconds of device work).  Same stopping rule as pcg_solve.  With op.dist set
// the vectors are slab-local: the vector kernels run over the owned planes, the halo planes of whatever the operator
// is applied to are exchanged first, and every sum is all-reduced before the host reads it.
namespace {

template <typename T, typename Precond>
PcgResult mgpcg_impl(Operator<T>& op, Precond& mg, const T* b, T* x, double tol, long long max_iter, cudaStream_t s, int guard_every)
{
	TraceScope    trace("mgpcg_solve");
	DistHooks*    dist = op.dist;
	const int64_t N = op.g.N, off = op.g.own_offset(), n = op.g.own_cells();
	const T*      rhs = b ? b : op.atb.data();
	if (max_iter <= 0) { max_iter = 2 * static_cast<long long>(op.g.size[0]) * op.g.size[1] * op.g.size[2]; }
	if (!(tol > 0)) { tol = std::is_same<T, float>::value ? 1.1920929e-07 : 2.220446049250313e-16; }
	DevBuf<T>        r(N), p(N), q(N);
	DevBuf<float>    r32(N), z(N);
	DevBuf<double>   out(2), partial(static_cast<size_t>(2) * (static_cast<size_t>(sm_count()) * 8 + 8));
	DevBuf<unsigned> ticket(1);
	ticket.zero(s);
	if (dist) {  // halo planes and planes beyond the lattice are read by the stencil kernels: start finite
		r.zero(s);
		q.zero(s);
		r32.zero(s);
		z.zero(s);
	}
	cudaEvent_t e0, e1;
	FI_CUDA(cudaEventCreate(&e0));
	FI_CUDA(cudaEventCreate(&e1));
	FI_CUDA(cudaEventRecord(e0, s));
	auto read = [&](double* h, int count) {
		if (dist) { dist->allreduce(out.data(), count, s); }
		FI_CUDA(cudaMemcpyAsync(h, out.data(), count * sizeof(double), cudaMemcpyDeviceToHost, s));
		FI_CUDA(cudaStreamSynchronize(s));
	};
	const int grid = vgrid(n);
	PcgResult res;
	double    h[2] = {0, 0};
	if (dist) { dist->exchange_halo(x, sizeof(T), s); }
	op.apply(x, q.data(), nullptr, nullptr, s);
	{
		auto k = mg_residual_kernel<T>;
		FI_LAUNCH(k, grid, kThreads, 0, s, n, rhs + off, q.data() + off, r.data() + off, r32.data() + off, out.data(), partial.data(), ticket.data());
	}
	read(h, 2);
	double       rr = h[0];
	const double bb = h[1];
	res.zero_rhs         = bb == 0.0;
	res.initial_residual = bb > 0 ? std::sqrt(rr / bb) : 0.0;
	const double target  = tol * tol * bb;
	long long    it      = 0;
	if (res.zero_rhs) {
		FI_CUDA(cudaMemsetAsync(x + off, 0, n * sizeof(T), s));
		rr = 0;
	} else if (rr > target) {
		double rz = 0;
		p.zero(s);
		bool fresh = true;  // no search direction yet (first iteration, or restarted after the preconditioner changed)
		// CG broke down on a W-cycle preconditioner: continue from x with V-cycles (r is the recurrence residual of x)
		auto demoted = [&] {
			if (!mg.demote_to_v_cycle()) { return false; }
			fresh = true;
			p.zero(s);  // beta = 0 next, but 0 * (a non-finite leftover) would not be
			return true;
		};
		while (it < max_iter) {
			mg.vcycle(r32.data(), z.data(), s);
			{
				auto k = mg_dot_kernel<T>;
				FI_LAUNCH(k, grid, kThreads, 0, s, n, r.data() + off, z.data() + off, out.data(), partial.data(), ticket.data());
			}
			read(h, 1);
			const double rz_new = h[0];
			if (!(rz_new > 0.0) || !std::isfinite(rz_new)) {  // breakdown: keep the last iterate
				if (demoted()) { continue; }
				res.stalled = true;
				break;
			}
			const double beta = fresh ? 0.0 : rz_new / rz;
			fresh             = false;
			rz                = rz_new;
			{
				auto k = mg_direction_kernel<T>;
				FI_LAUNCH(k, grid, kThreads, 0, s, n, z.data() + off, p.data() + off, static_cast<T>(beta));
			}
			if (dist) { dist->exchange_halo(p.data(), sizeof(T), s); }
			op.apply(p.data(), q.data(), out.data(), nullptr, s);
			read(h, 1);
			const double pq = h[0];
			if (!(pq > 0.0) || !std::isfinite(pq)) {
				if (demoted()) { continue; }
				res.stalled = true;
				break;
			}
			const double alpha = rz / pq;
			{
				auto k = mg_update_kernel<T>;
				FI_LAUNCH(k, grid, kThreads, 0, s, n, x + off, r.data() + off, p.data() + off, q.data() + off, r32.data() + off, static_cast<T>(alpha), out.data(),
				          partial.data(), ticket.data());
			}
			read(h, 1);
			rr = h[0];
			++it;
			if (rr <= target) { break; }
			if (!std::isfinite(rr)) {
				res.stalled = true;
				break;
			}
			if (guard_every > 0 && it % guard_every == 0) {
				// does the recurrence still describe x?  (q is free between iterations; the operator's own work vectors carry A x)
				double trr = 0, tbb = 0;
				residual<T>(op, rhs, x, nullptr, &trr, &tbb, s);
				if (!(trr <= 4.0 * rr)) {  // |b - A x| > 2 |r|: the floor of this arithmetic
					res.stalled = true;
					break;
				}
			}
		}
	}
	FI_CUDA(cudaEventRecord(e1, s));
	FI_CUDA(cudaEventSynchronize(e1));
	float ms = 0;
	FI_CUDA(cudaEventElapsedTime(&ms, e0, e1));
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
	res.solve_ms      = ms;
	res.loop_ms       = ms;
	res.iterations    = it;
	res.rel_residual  = bb > 0 ? std::sqrt(rr / bb) : 0.0;
	res.converged     = res.zero_rhs || rr <= target;
	res.true_residual = res.rel_residual;
	if (!res.zero_rhs) {
		double trr = 0, tbb = 0;
		residual<T>(op, rhs, x, nullptr, &trr, &tbb, s);
		res.true_residual = tbb > 0 ? std::sqrt(trr / tbb) : 0.0;
		// the stopping rule must hold for the residual of x itself, not merely for the recurrence
		const bool recurrence_met = res.converged;
		res.converged             = res.true_residual <= kConvergedSlack * tol;
		if (recurrence_met && !res.converged) { res.stalled = true; }
	}
	return res;
}

}  // namespace

template <typename T>
PcgResult mgpcg_solve(Operator<T>& op, Multigrid& mg, const T* b, T* x, double tol, long long max_iter, cudaStream_t s, int guard_every)
{
	FI_REQUIRE(op.dist == nullptr && !op.g.sharded(), FI_ERR_UNSUPPORTED, "mgpcg_solve takes an unsharded lattice (slabs: slab_mgpcg_solve)");
	return mgpcg_impl<T, Multigrid>(op, mg, b, x, tol, max_iter, s, guard_every);
}

template <typename T>
PcgResult slab_mgpcg_solve(Operator<T>& op, SlabMultigrid& mg, const T* b, T* x, double tol, long long max_iter, cudaStream_t s, int guard_every)
{
	FI_REQUIRE(op.dist != nullptr, FI_ERR_INVALID, "slab_mgpcg_solve needs the slab's communicator hooks");
	return mgpcg_impl<T, SlabMultigrid>(op, mg, b, x, tol, max_iter, s, guard_every);
}

template PcgResult mgpcg_solve<float>(Operator<float>&, Multigrid&, const float*, float*, double, long long, cudaStream_t, int);
template PcgResult mgpcg_solve<double>(Operator<double>&, Multigrid&, const double*, double*, double, long long, cudaStream_t, int);
template PcgResult slab_mgpcg_solve<float>(Operator<float>&, SlabMultigrid&, const float*, float*, double, long long, cudaStream_t, int);
template PcgResult slab_mgpcg_solve<double>(Operator<double>&, SlabMultigrid&, const double*, double*, double, long long, cudaStream_t, int);

}  // namespace fi
