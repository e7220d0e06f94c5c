// Specialised 3D smoothness kernel: q = S p (+ p.q) for star-shaped S (model_0..model_4, no gradient-smoothness
// cross terms) on lattices whose x size is a multiple of the 16-byte pack.
//
// 2.5-D blocking.  A block owns an xy tile of 32 packs x TYT rows (pack = 16 bytes = 4 floats / 2 doubles, one
// per thread, so every global access is a 128-bit, fully coalesced LDG/STG) and marches a chunk of z planes:
//   * the z neighbours of a thread's pack live in a register pipeline of 2R+1 packs (each plane of p is read
//     from global memory once per block, R planes ahead of use);
//   * the x / y neighbours come from a double-buffered shared-memory copy of the current plane (tile plus R
//     halo rows above/below and ceil(R/V) halo packs left/right), one __syncthreads per plane;
//   * boundary truncation of the difference rows (reference field_interpolation.cpp:257-301: a row exists only
//     while coord+k < size) is folded into per-thread coefficient registers chosen once per kernel from the
//     9-class tables (x, y) and a per-plane uniform row (z), so the inner loop is branch-free and identical for
//     interior and boundary nodes; out-of-lattice halo cells are stored as zeros.
// Optional fusion (Fused = true): the CG direction update p = M r + beta p_old is evaluated while loading
// (including halos) and written back by the owner, which removes one full pass over the vectors per iteration.
#include "internal.hpp"
#include "solver.hpp"

namespace fi {

namespace {

__host__ __device__ __forceinline__ int row_class(int i, int n)
{
	return n <= 9 ? i : (i < 4 ? i : (i >= n - 4 ? i - n + 9 : 4));
}

template <typename T>
struct PackOf;
template <>
struct PackOf<float>
{
	using type = float4;
};
template <>
struct PackOf<double>
{
	using type = double2;
};

template <typename T>
struct FastTables
{
	T band[kMaxDim][9][9];
};

template <typename T>
struct FuseArgs  // direction update folded into the load stage
{
	const T*        r;
	const T*        minv;
	const T*        p_old;
	T*              p_new;
	const PcgState* st;
	int             par;
};

template <typename T, int V>
union PackU
{
	typename PackOf<T>::type v;
	T                        a[V];
};

template <typename T, int R, int TYT, bool Fused>
__global__ void __launch_bounds__(32 * TYT) stencil3d_kernel(int nx, int ny, int nz, int zchunk, FastTables<T> tab,
                                                             const T* __restrict__ p, T* __restrict__ q, FuseArgs<T> fz,
                                                             double* dot_out, double* partial, unsigned* ticket, const int* done)
{
	constexpr int V   = 16 / sizeof(T);
	constexpr int NP  = (R + V - 1) / V;  // halo packs per side in x
	constexpr int TXT = 32;
	constexpr int SWP = TXT + 2 * NP;     // smem row width in packs
	constexpr int SH  = TYT + 2 * R;
	using Pack        = typename PackOf<T>::type;
	using PU          = PackU<T, V>;

	__shared__ __align__(16) Pack tile[2][SH][SWP];
	__shared__ T                  zband[9][2 * R + 1];
	__shared__ double             red[32];

	if (done && *done) { return; }

	const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
	const int px  = blockIdx.x * TXT + tx;  // pack column
	const int x0  = px * V;
	const int y   = blockIdx.y * TYT + ty;
	const int zb  = blockIdx.z * zchunk;
	const int ze  = min(nz, zb + zchunk);
	const bool in_xy = (x0 < nx) && (y < ny);
	const size_t plane = static_cast<size_t>(nx) * ny;

	// beta of this iteration: rho[par] is r.z of the current residual, rho[par^1] the previous one; the first
	// iteration of a solve starts from p = M r
	T beta = 0;
	if (Fused) { beta = fz.st->iters == 0 ? T(0) : static_cast<T>(fz.st->rho[fz.par] / fz.st->rho[fz.par ^ 1]); }

	// per-thread x / y coefficient rows, per-plane z rows in shared memory
	T cx[V][2 * R + 1], cy[2 * R + 1];
#pragma unroll
	for (int j = 0; j < V; ++j) {
		const int cls = row_class(min(x0 + j, nx - 1), nx);
#pragma unroll
		for (int t = 0; t <= 2 * R; ++t) { cx[j][t] = tab.band[0][cls][t + 4 - R]; }
	}
	{
		const int cls = row_class(min(y, ny - 1), ny);
#pragma unroll
		for (int t = 0; t <= 2 * R; ++t) { cy[t] = tab.band[1][cls][t + 4 - R]; }
	}
	for (int k = tid; k < 9 * (2 * R + 1); k += 32 * TYT) { zband[k / (2 * R + 1)][k % (2 * R + 1)] = tab.band[2][k / (2 * R + 1)][k % (2 * R + 1) + 4 - R]; }

	// pack loader with the optional fused direction update; returns zeros outside the lattice
	auto load_pack = [&](int gx, int gy, int gz, bool write_back) -> Pack {
		PU out;
#pragma unroll
		for (int j = 0; j < V; ++j) { out.a[j] = T(0); }
		if (gx < 0 || gx >= nx || gy < 0 || gy >= ny || gz < 0 || gz >= nz) { return out.v; }
		const size_t at = static_cast<size_t>(gz) * plane + static_cast<size_t>(gy) * nx + gx;
		if (!Fused) {
			out.v = *reinterpret_cast<const Pack*>(p + at);
		} else {
			PU rr, mm, pp;
			rr.v = *reinterpret_cast<const Pack*>(fz.r + at);
			mm.v = *reinterpret_cast<const Pack*>(fz.minv + at);
			pp.v = *reinterpret_cast<const Pack*>(fz.p_old + at);
#pragma unroll
			for (int j = 0; j < V; ++j) { out.a[j] = mm.a[j] * rr.a[j] + beta * pp.a[j]; }
			if (write_back) { *reinterpret_cast<Pack*>(fz.p_new + at) = out.v; }
		}
		return out.v;
	};

	// halo duties of this thread: one y-halo pack (threads with ty < 2R) and one x-halo pack (tid < 2*NP*TYT)
	const bool has_yh = ty < 2 * R;
	const int  yh_row = ty < R ? ty : TYT + ty;              // smem row of the y-halo pack (0..R-1, TYT+R..TYT+2R-1)
	const int  yh_gy  = blockIdx.y * TYT + (yh_row - R);
	const bool has_xh = tid < 2 * NP * TYT;
	const int  xh_r   = tid / (2 * NP);                       // tile row 0..TYT-1
	const int  xh_k   = tid % (2 * NP);
	const int  xh_col = xh_k < NP ? xh_k : TXT + xh_k;        // smem pack column (0..NP-1, TXT+NP..TXT+2NP-1)
	const int  xh_gx  = (blockIdx.x * TXT + (xh_col - NP)) * V;
	const int  xh_gy  = blockIdx.y * TYT + xh_r;

	// register pipeline: pipe[t] = own pack of plane z + t - R
	PU pipe[2 * R + 1];
#pragma unroll
	for (int t = 0; t <= 2 * R; ++t) {
		const int gz = zb + t - R;
		// a plane is written back (fused) by the chunk that owns it
		pipe[t].v = in_xy ? load_pack(x0, y, gz, gz >= zb && gz < ze) : load_pack(-1, 0, 0, false);
	}
	Pack yh = load_pack(has_yh ? x0 : -1, yh_gy, zb, false);
	Pack xh = load_pack(has_xh ? xh_gx : -1, xh_gy, zb, false);

	double acc = 0.0;
	int    buf = 0;
	for (int z = zb; z < ze; ++z, buf ^= 1) {
		tile[buf][ty + R][tx + NP] = pipe[R].v;
		if (has_yh) { tile[buf][yh_row][tx + NP] = yh; }
		if (has_xh) { tile[buf][xh_r + R][xh_col] = xh; }
		// loads for the next plane fly during this plane's arithmetic
		PU nxt;
		{
			const int gz = z + R + 1;
			nxt.v = in_xy ? load_pack(x0, y, gz, gz < ze) : load_pack(-1, 0, 0, false);
		}
		if (z + 1 < ze) {
			yh = load_pack(has_yh ? x0 : -1, yh_gy, z + 1, false);
			xh = load_pack(has_xh ? xh_gx : -1, xh_gy, z + 1, false);
		}
		__syncthreads();

		if (in_xy) {
			const T* cz = zband[row_class(z, nz)];
			PU       out;
			// z taps from the register pipeline
#pragma unroll
			for (int j = 0; j < V; ++j) {
				T s = T(0);
#pragma unroll
				for (int t = 0; t <= 2 * R; ++t) { s += cz[t] * pipe[t].a[j]; }
				out.a[j] = s;
			}
			// y taps from shared memory
#pragma unroll
			for (int t = 0; t <= 2 * R; ++t) {
				if (t == R) {
#pragma unroll
					for (int j = 0; j < V; ++j) { out.a[j] += cy[t] * pipe[R].a[j]; }
				} else {
					PU nb;
					nb.v = tile[buf][ty + t][tx + NP];
#pragma unroll
					for (int j = 0; j < V; ++j) { out.a[j] += cy[t] * nb.a[j]; }
				}
			}
			// x taps: the row segment [x0 - NP*V, x0 + V + NP*V)
			T xs[(2 * NP + 1) * V];
#pragma unroll
			for (int k = 0; k < 2 * NP + 1; ++k) {
				PU nb;
				if (k == NP) { nb = pipe[R]; } else { nb.v = tile[buf][ty + R][tx + k]; }
#pragma unroll
				for (int j = 0; j < V; ++j) { xs[k * V + j] = nb.a[j]; }
			}
#pragma unroll
			for (int j = 0; j < V; ++j) {
#pragma unroll
				for (int t = 0; t <= 2 * R; ++t) { out.a[j] += cx[j][t] * xs[NP * V + j + t - R]; }
			}
			*reinterpret_cast<Pack*>(q + static_cast<size_t>(z) * plane + static_cast<size_t>(y) * nx + x0) = out.v;
			T d = T(0);
#pragma unroll
			for (int j = 0; j < V; ++j) { d += out.a[j] * pipe[R].a[j]; }
			acc += static_cast<double>(d);
		}
#pragma unroll
		for (int t = 0; t < 2 * R; ++t) { pipe[t] = pipe[t + 1]; }
		pipe[2 * R] = nxt;
	}

	if (dot_out) {
		double mine[1] = {block_sum(acc, red)};
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { *dot_out = tot[0]; });
	}
}

template <typename T, int R, bool Fused>
void launch(const Geom& g, const StencilTables& t, const T* p, T* q, const FuseArgs<T>& fz, double* d_dot_out, double* d_partial,
            unsigned* d_ticket, const int* d_done, cudaStream_t s)
{
	constexpr int TYT = 8;
	constexpr int V   = 16 / sizeof(T);
	FastTables<T> tab;
	for (int a = 0; a < kMaxDim; ++a) {
		for (int c = 0; c < 9; ++c) {
			for (int k = 0; k < 9; ++k) { tab.band[a][c][k] = static_cast<T>(t.band[a][c][k]); }
		}
	}
	const int tiles_x = div_up(g.size[0], 32 * V), tiles_y = div_up(g.size[1], TYT);
	// z chunking: aim for >= 8 waves of 3 resident blocks per SM, chunks of at least 8 planes
	const int64_t want_blocks = static_cast<int64_t>(sm_count()) * 3 * 8;
	int           chunks      = static_cast<int>(std::max<int64_t>(1, want_blocks / (static_cast<int64_t>(tiles_x) * tiles_y)));
	chunks                    = std::min(chunks, std::max(1, g.size[2] / 8));
	const int zchunk          = div_up(g.size[2], chunks);
	chunks                    = div_up(g.size[2], zchunk);
	dim3 grid(tiles_x, tiles_y, chunks);
	auto kern = stencil3d_kernel<T, R, TYT, Fused>;
	FI_LAUNCH(kern, grid, 32 * TYT, 0, s, g.size[0], g.size[1], g.size[2], zchunk, tab, p, q, fz, d_dot_out, d_partial, d_ticket,
	          d_done);
	note_stencil(FI_PCG_KERNEL_TILED_3D, R, false, TYT, chunks);
}

template <typename T>
bool eligible(const Geom& g, const StencilTables& t)
{
	constexpr int V = 16 / sizeof(T);
	return g.ndim == 3 && t.gs2 == 0.0 && t.radius >= 1 && g.size[0] % V == 0 && g.size[0] >= 32 && g.size[1] >= 8 && g.size[2] >= 8 && !g.sharded();
}

}  // namespace

template <typename T>
bool stencil_fast_3d(const Geom& g, const StencilTables& t, const T* p, T* q, double* d_dot_out, double* d_partial,
                     unsigned* d_ticket, const int* d_done, cudaStream_t s)
{
	if (!eligible<T>(g, t)) { return false; }
	FuseArgs<T> none{nullptr, nullptr, nullptr, nullptr, nullptr, 0};
	if (t.radius <= 1) {
		launch<T, 1, false>(g, t, p, q, none, d_dot_out, d_partial, d_ticket, d_done, s);
	} else if (t.radius == 2) {
		launch<T, 2, false>(g, t, p, q, none, d_dot_out, d_partial, d_ticket, d_done, s);
	} else {
		launch<T, 4, false>(g, t, p, q, none, d_dot_out, d_partial, d_ticket, d_done, s);
	}
	return true;
}

// Fused CG step: p_new = M r + beta p_old, q = S p_new, p_new.q — see solver.cu.
template <typename T>
bool stencil_fast_3d_fused(const Geom& g, const StencilTables& t, const T* r, const T* minv, const T* p_old, T* p_new, T* q,
                           const PcgState* st, int par, double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done,
                           cudaStream_t s)
{
	if (!eligible<T>(g, t)) { return false; }
	FuseArgs<T> fz{r, minv, p_old, p_new, st, par};
	if (t.radius <= 1) {
		launch<T, 1, true>(g, t, nullptr, q, fz, d_dot_out, d_partial, d_ticket, d_done, s);
	} else if (t.radius == 2) {
		launch<T, 2, true>(g, t, nullptr, q, fz, d_dot_out, d_partial, d_ticket, d_done, s);
	} else {
		launch<T, 4, true>(g, t, nullptr, q, fz, d_dot_out, d_partial, d_ticket, d_done, s);
	}
	return true;
}

template bool stencil_fast_3d<float>(const Geom&, const StencilTables&, const float*, float*, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_fast_3d<double>(const Geom&, const StencilTables&, const double*, double*, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_fast_3d_fused<float>(const Geom&, const StencilTables&, const float*, const float*, const float*, float*, float*, const PcgState*, int, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_fast_3d_fused<double>(const Geom&, const StencilTables&, const double*, const double*, const double*, double*, double*, const PcgState*, int, double*, double*, unsigned*, const int*, cudaStream_t);

}  // namespace fi
