// TMA-staged smoothness kernel for 2D lattices on sm_100a: q = S p (+ p.q), optionally with the CG direction update
// p = M r + beta p_old folded into the load stage, or — epilogue mode, the multigrid smoother — consumed in place.
//
// Same mathematics as the 3D kernel (stencil_tma.cu; operator built from the reference's model rows,
// field_interpolation/field_interpolation.cpp:243-316), including the gradient-smoothness cross terms
// 2 w_gs^2 (D_1^T D_1)_x (x) (D_1^T D_1)_y (:303-315), which in 2D are a compact 3x3 stencil.  Different blocking: a 2D
// lattice has no third axis to march along, so a block owns one TX x TY tile, one elected thread fetches the tile and
// its halo — (TX + 2 halo) x (TY + 2R), one box per input array — with cp.async.bulk.tensor into shared memory, all
// threads wait on the mbarrier, turn the staged arrays into the direction p in place, and evaluate the star (and the
// 3x3 cross term) from shared memory.  Lattice boundaries need no branches: out-of-bounds box elements arrive as zeros,
// which is what the dropped difference rows imply, and the per-axis coefficient rows already contain the truncation.
// Several blocks per SM overlap each other's load and compute phases.  BASELINE configs[1] and [2] (512^2, 2048^2) are
// L2-resident: the kernel is bound by L2 bandwidth and launch latency there, by HBM from ~8192^2 up.
//
// The lattice is described to TMA as a 3D tensor (nx, ny, 1) so that the kernel uses the same load instruction (and the
// same emulation hook in tests/emu) as the 3D kernel.
#include "solver.hpp"
#include "tma.cuh"

namespace fi {

namespace {

using namespace tma;

template <typename T, int R, int TY_>
struct Tile2
{
	static constexpr int V    = 16 / sizeof(T);   // elements per 16-byte pack
	static constexpr int NP   = (R + V - 1) / V;  // halo packs per side in x
	static constexpr int TXP  = 32;               // packs per tile row (one per lane)
	static constexpr int TY   = TY_;              // tile rows (8 warps, TY / 8 rows each)
	static constexpr int BXP  = TXP + 2 * NP;     // box row in packs
	static constexpr int BY   = TY + 2 * R;       // box rows
	static constexpr int TILE_BYTES = ((BXP * BY * 16 + 127) / 128) * 128;
	static constexpr int BOX_BYTES  = BXP * BY * 16;
};

template <typename T, int R, int TY, bool Fused>
constexpr size_t smem_bytes_2d()
{
	using G = Tile2<T, R, TY>;
	return 128 /* alignment slack */ + static_cast<size_t>(Fused ? 3 : 1) * G::TILE_BYTES + sizeof(uint64_t) + 32 * sizeof(double) + 64;
}

// (D_1^T D_1)[i][i] on an axis of n nodes: how many first-difference rows touch node i
__device__ __forceinline__ int lap_center(int i, int n) { return (i > 0 ? 1 : 0) + (i < n - 1 ? 1 : 0); }

template <typename T, int R, int TY, bool Fused, bool Epi, bool GS>
__global__ void __launch_bounds__(256)
    stencil2d_tma_kernel(const __grid_constant__ CUtensorMap map_a,  // p (plain) or r (fused)
                         const __grid_constant__ CUtensorMap map_b,  // M^-1 (fused)
                         const __grid_constant__ CUtensorMap map_c,  // p_old (fused)
                         int nx, int ny, TmaTables<T> tab, T gs2, T* __restrict__ q, T* __restrict__ p_new, const PcgState* st, int par,
                         double* dot_out, double* partial, unsigned* ticket, const int* done, EpiArgs<T> epi)
{
	static_assert(!(Fused && Epi), "the epilogue mode takes a plain input");
	using G          = Tile2<T, R, TY>;
	constexpr int V  = G::V;
	constexpr int NP = G::NP;
	constexpr int NA = Fused ? 3 : 1;
	constexpr int W  = 2 * R + 1;
	constexpr int RPT = TY / 8;  // rows per thread
	using Pack       = typename PackOf<T>::type;
	using PU         = PackU<T, V>;

	if (done && *done) { return; }

#ifdef FI_B200_EMU
	unsigned char* smem_raw = ::cuda_emu::dynamic_smem();
#else
	extern __shared__ unsigned char smem_raw[];
#endif
	unsigned char* base = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
	auto     tile_ptr = [&](int a) { return reinterpret_cast<Pack*>(base + static_cast<size_t>(a) * G::TILE_BYTES); };
	uint64_t* full = reinterpret_cast<uint64_t*>(base + static_cast<size_t>(NA) * G::TILE_BYTES);
	double*   red  = reinterpret_cast<double*>(full + 1);

	const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
	const int x0t = blockIdx.x * (G::TXP * V);  // first element column of the tile
	const int y0t = blockIdx.y * TY;
	const int x0  = x0t + tx * V;

	if (tid == 0) {
		mbar_init(full, 1);
		fence_barrier_init();
	}
	__syncthreads();
	if (tid == 0) {
		mbar_expect_tx(full, NA * G::BOX_BYTES);
		tma_load_3d(tile_ptr(0), &map_a, full, x0t - NP * V, y0t - R, 0);
		if (Fused) {
			tma_load_3d(tile_ptr(1), &map_b, full, x0t - NP * V, y0t - R, 0);
			tma_load_3d(tile_ptr(2), &map_c, full, x0t - NP * V, y0t - R, 0);
		}
	}

	// while the boxes are in flight: coefficients, and the epilogue's pointwise operands of this thread's packs
	T beta = 0;
	if (Fused) { beta = st->iters == 0 ? T(0) : static_cast<T>(st->rho[par] / st->rho[par ^ 1]); }
	T cx[V][W];
	T lx0[V];  // gradient smoothness: (D_1^T D_1)_x diagonal at this thread's columns
#pragma unroll
	for (int j = 0; j < V; ++j) {
		const int xi  = min(x0 + j, nx - 1);
		const int cls = row_class(xi, nx);
#pragma unroll
		for (int t = 0; t < W; ++t) { cx[j][t] = tab.band[0][cls][t + 4 - R]; }
		lx0[j] = static_cast<T>(lap_center(xi, nx));
	}
	const bool in_x    = x0 < nx;
	const bool epi_upd = Epi && epi.d_new != nullptr;
	PU         pre_r[RPT], pre_m[RPT], pre_e[RPT];
	if (Epi) {
#pragma unroll
		for (int k = 0; k < RPT; ++k) {
			const int y = y0t + ty + 8 * k;
			if (in_x && y < ny) {
				const size_t at = static_cast<size_t>(y) * nx + x0;
				pre_r[k].v      = *reinterpret_cast<const Pack*>(epi.res_in + at);
				if (epi_upd) {
					pre_m[k].v = *reinterpret_cast<const Pack*>(epi.minv + at);
					pre_e[k].v = *reinterpret_cast<const Pack*>(epi.e + at);
				}
			}
		}
	}

	mbar_wait(full, 0);
	Pack* pt = tile_ptr(0);
	if (Fused) {  // the new direction over the whole box, in place over r
		const Pack* sb = tile_ptr(1);
		const Pack* sc = tile_ptr(2);
		for (int i = tid; i < G::BXP * G::BY; i += 256) {
			PU rr, mm, pp;
			rr.v = pt[i];
			mm.v = sb[i];
			pp.v = sc[i];
#pragma unroll
			for (int j = 0; j < V; ++j) { rr.a[j] = mm.a[j] * rr.a[j] + beta * pp.a[j]; }
			pt[i] = rr.v;
		}
		__syncthreads();
	}

	double acc = 0.0;
#pragma unroll
	for (int k = 0; k < RPT; ++k) {
		const int row = ty + 8 * k;  // tile row
		const int y   = y0t + row;
		if (!in_x || y >= ny) { continue; }
		const int cls_y = row_class(y, ny);
		PU        ctr;
		ctr.v = pt[(row + R) * G::BXP + tx + NP];
		PU out;
#pragma unroll
		for (int j = 0; j < V; ++j) { out.a[j] = T(0); }
		// y taps: this thread's pack column
#pragma unroll
		for (int t = 0; t < W; ++t) {
			const T c = tab.band[1][cls_y][t + 4 - R];
			PU      nb;
			if (t == R) { nb = ctr; } else { nb.v = pt[(row + t) * G::BXP + tx + NP]; }
#pragma unroll
			for (int j = 0; j < V; ++j) { out.a[j] += c * nb.a[j]; }
		}
		// x taps: the centre row
		T xs[(2 * NP + 1) * V];
#pragma unroll
		for (int kk = 0; kk < 2 * NP + 1; ++kk) {
			PU nb;
			if (kk == NP) { nb = ctr; } else { nb.v = pt[(row + R) * G::BXP + tx + kk]; }
#pragma unroll
			for (int j = 0; j < V; ++j) { xs[kk * V + j] = nb.a[j]; }
		}
#pragma unroll
		for (int j = 0; j < V; ++j) {
#pragma unroll
			for (int t = 0; t < W; ++t) { out.a[j] += cx[j][t] * xs[NP * V + j + t - R]; }
		}
		if (GS) {
			// gs2 * sum_{a,b in {-1,0,1}} lx(a) ly(b) p(x+a, y+b): lx(0) = lx0, lx(+-1) = -1 where the neighbour exists (zeros arrive otherwise)
			const T ly0 = static_cast<T>(lap_center(y, ny));
			T up[(2 * NP + 1) * V], dn[(2 * NP + 1) * V];
#pragma unroll
			for (int kk = 0; kk < 2 * NP + 1; ++kk) {
				PU a, b;
				a.v = pt[(row + R - 1) * G::BXP + tx + kk];
				b.v = pt[(row + R + 1) * G::BXP + tx + kk];
#pragma unroll
				for (int j = 0; j < V; ++j) {
					up[kk * V + j] = a.a[j];
					dn[kk * V + j] = b.a[j];
				}
			}
#pragma unroll
			for (int j = 0; j < V; ++j) {
				const int c = NP * V + j;
				const T   s = lx0[j] * ly0 * xs[c] - ly0 * (xs[c - 1] + xs[c + 1]) - lx0[j] * (up[c] + dn[c]) + (up[c - 1] + up[c + 1] + dn[c - 1] + dn[c + 1]);
				out.a[j] += gs2 * s;
			}
		}
		const size_t at = static_cast<size_t>(y) * nx + x0;
		if (Epi) {
			PU rn;
#pragma unroll
			for (int j = 0; j < V; ++j) { rn.a[j] = pre_r[k].a[j] - out.a[j]; }
			if (epi.res_out) { *reinterpret_cast<Pack*>(epi.res_out + at) = rn.v; }
			if (epi_upd) {
				PU dnew, en;
#pragma unroll
				for (int j = 0; j < V; ++j) {
					dnew.a[j] = epi.a * ctr.a[j] + epi.b * pre_m[k].a[j] * rn.a[j];
					en.a[j]   = pre_e[k].a[j] + dnew.a[j];
				}
				*reinterpret_cast<Pack*>(epi.d_new + at) = dnew.v;
				*reinterpret_cast<Pack*>(epi.e + at)     = en.v;
			}
		} else {
			*reinterpret_cast<Pack*>(q + at) = out.v;
			if (Fused) { *reinterpret_cast<Pack*>(p_new + at) = ctr.v; }
			T d = T(0);
#pragma unroll
			for (int j = 0; j < V; ++j) { d += out.a[j] * ctr.a[j]; }
			acc += static_cast<double>(d);
		}
	}

	if (dot_out) {
		double mine[1] = {block_sum(acc, red)};
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { *dot_out = tot[0]; });
	}
}

// ---- host side ------------------------------------------------------------------------------------------------
template <typename T, int R, int TY>
CUtensorMap make_map_2d(const Geom& g, const T* ptr)
{
	using G = Tile2<T, R, TY>;
	CUtensorMap m;
	std::memset(&m, 0, sizeof(m));
	EncodeFn fn = encode_fn();
	FI_REQUIRE(fn != nullptr, FI_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
	const cuuint64_t dims[3]    = {static_cast<cuuint64_t>(g.size[0]), static_cast<cuuint64_t>(g.size[1]), 1u};
	const cuuint64_t strides[2] = {static_cast<cuuint64_t>(g.size[0]) * sizeof(T), static_cast<cuuint64_t>(g.size[0]) * g.size[1] * sizeof(T)};
	const cuuint32_t box[3]     = {static_cast<cuuint32_t>(G::BXP * G::V), static_cast<cuuint32_t>(G::BY), 1u};
	const cuuint32_t estr[3]    = {1u, 1u, 1u};
	const CUresult   r = fn(&m, sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<T*>(ptr), dims, strides, box,
	                        estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	FI_REQUIRE(r == CUDA_SUCCESS, FI_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
	return m;
}

template <typename T, int R, bool Fused, bool Epi, bool GS>
void launch_2d(const Geom& g, const StencilTables& t, const T* a, const T* b, const T* c, T* q, T* p_new, const PcgState* st, int par, double* d_dot_out,
               double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s, const EpiArgs<T>& epi)
{
	constexpr int TY = 16;
	using G          = Tile2<T, R, TY>;
	TmaTables<T> tab;
	for (int ax = 0; ax < kMaxDim; ++ax) {
		for (int cl = 0; cl < 9; ++cl) {
			for (int k = 0; k < 9; ++k) { tab.band[ax][cl][k] = static_cast<T>(t.band[ax][cl][k]); }
		}
	}
	const CUtensorMap ma = make_map_2d<T, R, TY>(g, a);
	const CUtensorMap mb = Fused ? make_map_2d<T, R, TY>(g, b) : ma;
	const CUtensorMap mc = Fused ? make_map_2d<T, R, TY>(g, c) : ma;
	dim3 grid(div_up(g.size[0], G::TXP * G::V), div_up(g.size[1], TY), 1);
	auto kern = stencil2d_tma_kernel<T, R, TY, Fused, Epi, GS>;
	constexpr size_t smem = smem_bytes_2d<T, R, TY, Fused>();
	static bool configured = false;  // per instantiation
	if (!configured) {
		FI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
		configured = true;
	}
	FI_LAUNCH(kern, grid, 256, smem, s, ma, mb, mc, g.size[0], g.size[1], tab, static_cast<T>(t.gs2), q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done,
	          epi);
	note_stencil(FI_PCG_KERNEL_TMA_2D, R, GS, TY, 1);
}

template <typename T, bool Fused, bool Epi>
void dispatch_2d(const Geom& g, const StencilTables& t, const T* a, const T* b, const T* c, T* q, T* p_new, const PcgState* st, int par, double* d_dot_out,
                 double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s, const EpiArgs<T>& epi = EpiArgs<T>())
{
	const bool gs = t.gs2 != 0.0;
#define FI_2D(RR)                                                                                                                          \
	do {                                                                                                                                   \
		if (gs) {                                                                                                                          \
			launch_2d<T, RR, Fused, Epi, true>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s, epi);            \
		} else {                                                                                                                           \
			launch_2d<T, RR, Fused, Epi, false>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s, epi);           \
		}                                                                                                                                  \
	} while (0)
	if (t.radius <= 1) {
		FI_2D(1);
	} else if (t.radius == 2) {
		FI_2D(2);
	} else {
		FI_2D(4);
	}
#undef FI_2D
}

}  // namespace

template <typename T>
bool stencil_2d_eligible(const Geom& g, const StencilTables& t)
{
	constexpr int V = 16 / sizeof(T);
	return g.ndim == 2 && !g.tile && t.radius >= 1 && g.size[0] % V == 0 && g.size[0] >= 32 && g.size[1] >= 8 && encode_fn() != nullptr;
}

template <typename T>
bool stencil_tma_2d(const Geom& g, const StencilTables& t, const T* p, T* q, double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done,
                    cudaStream_t s)
{
	if (!stencil_2d_eligible<T>(g, t)) { return false; }
	dispatch_2d<T, false, false>(g, t, p, nullptr, nullptr, q, nullptr, nullptr, 0, d_dot_out, d_partial, d_ticket, d_done, s);
	return true;
}

template <typename T>
bool stencil_tma_2d_fused(const Geom& g, const StencilTables& t, const T* r, const T* minv, const T* p_old, T* p_new, T* q, const PcgState* st, int par,
                          double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s)
{
	if (!stencil_2d_eligible<T>(g, t)) { return false; }
	dispatch_2d<T, true, false>(g, t, r, minv, p_old, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s);
	return true;
}

template <typename T>
bool stencil_tma_2d_epilogue(const Geom& g, const StencilTables& t, const T* in, const T* res_in, T* res_out, const T* minv, T* e, T* d_new, T a, T b,
                             cudaStream_t s)
{
	if (!stencil_2d_eligible<T>(g, t)) { return false; }
	EpiArgs<T> epi;
	epi.res_in  = res_in;
	epi.res_out = res_out;
	epi.minv    = minv;
	epi.e       = e;
	epi.d_new   = d_new;
	epi.a       = a;
	epi.b       = b;
	dispatch_2d<T, false, true>(g, t, in, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, s, epi);
	return true;
}

template bool stencil_tma_2d<float>(const Geom&, const StencilTables&, const float*, float*, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_tma_2d<double>(const Geom&, const StencilTables&, const double*, double*, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_tma_2d_fused<float>(const Geom&, const StencilTables&, const float*, const float*, const float*, float*, float*, const PcgState*, int, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_tma_2d_fused<double>(const Geom&, const StencilTables&, const double*, const double*, const double*, double*, double*, const PcgState*, int, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_tma_2d_epilogue<float>(const Geom&, const StencilTables&, const float*, const float*, float*, const float*, float*, float*, float, float, cudaStream_t);

}  // namespace fi
