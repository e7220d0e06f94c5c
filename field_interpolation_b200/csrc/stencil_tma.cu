// TMA-staged 3D smoothness kernel for sm_100a: q = S p (+ p.q), optionally with the CG direction update
// p = M r + beta p_old folded into the load stage — north-star item (b), the roofline kernel of the solve.
//
// Same mathematics as stencil_fast.cu (2.5-D blocking of the star-shaped operator built from the reference's
// model rows, field_interpolation/field_interpolation.cpp:243-316), different data movement:
//   * one elected thread issues cp.async.bulk.tensor (TMA) loads of whole xy boxes — tile plus halo, one z
//     plane per stage, for each of the 1 (plain) or 3 (fused: r, M^-1, p_old) input arrays — into a ring of
//     S shared-memory stages guarded by mbarriers, S planes ahead of use.  Loads cost no registers and no
//     address arithmetic in the compute warps, and lattice boundaries need no branches: the tensor map's
//     out-of-bounds fill supplies the zeros that the dropped difference rows imply;
//   * the 256 compute threads turn a landed stage into the new direction p (tile and halo) in a second
//     shared-memory ring of R+2 planes, keep their own z column in a register pipeline of 2R+1 packs (the
//     plane loop is unrolled 2R+1 times so the pipeline rotates by renaming, not by moves), and evaluate the
//     2R+1 taps per axis with per-thread coefficient rows that already contain the boundary truncation;
//   * q and p are written with 128-bit coalesced stores straight from registers.
// One __syncthreads and one mbarrier wait per plane.
#include <cstdlib>
#include <type_traits>

#include "solver.hpp"
#include "tma.cuh"

namespace fi {

namespace {

using namespace tma;

// ---- geometry of one block -----------------------------------------------------------------------------------
template <typename T, int R, int TY_ = 8>
struct Tile
{
	static constexpr int V    = 16 / sizeof(T);       // elements per 16-byte pack
	static constexpr int NP   = (R + V - 1) / V;      // halo packs per side in x
	static constexpr int TXP  = 32;                   // packs per tile row (one per lane)
	static constexpr int TY   = TY_;                  // tile rows: 8 (one per warp) or 7 (the eighth warp only fills halos; see launch)
	static constexpr int BXP  = TXP + 2 * NP;         // box row in packs
	static constexpr int BY   = TY + 2 * R;           // box rows
	// planes of the new direction kept in shared memory: the star reads plane z while the fastest warp may already be writing
	// plane z + R + 1 (one barrier per plane), so R + 2; the gradient-smoothness cross terms also read plane z - 1: R + 3
	__host__ __device__ static constexpr int ring(bool gs) { return R + 2 + (gs ? 1 : 0); }
	static constexpr int TILE_BYTES = ((BXP * BY * 16 + 127) / 128) * 128;
	static constexpr int BOX_BYTES  = BXP * BY * 16;  // what one TMA load delivers
};

template <typename T, int R, int S, bool Fused, bool GS, int TY = 8>
constexpr size_t smem_bytes()
{
	using G = Tile<T, R, TY>;
	return 128 /* alignment slack */ + static_cast<size_t>(S) * (Fused ? 3 : 1) * G::TILE_BYTES + static_cast<size_t>(G::ring(GS)) * G::TILE_BYTES +
	       S * sizeof(uint64_t) + 9 * (2 * R + 1) * sizeof(T) + 32 * sizeof(double) + 64;
}

template <typename T, int R, int S, bool Fused, int MINB, bool Epi, bool GS, int TY>
__global__ void __launch_bounds__(256, MINB)
    stencil3d_tma_kernel(const __grid_constant__ CUtensorMap map_a,  // p (plain) or r (fused)
                         const __grid_constant__ CUtensorMap map_b,  // M^-1 (fused)
                         const __grid_constant__ CUtensorMap map_c,  // p_old (fused)
                         int nx, int ny, int nzl, int zo0, int zo1, int zoff, int nzg, int zchunk, TmaTables<T> tab, T gs2,
                         T* __restrict__ q, T* __restrict__ p_new,
                         const PcgState* st, int par, double* dot_out, double* partial, unsigned* ticket, const int* done, EpiArgs<T> epi)
{
	static_assert(!(Fused && Epi), "the epilogue mode takes a plain input");
	using G           = Tile<T, R, TY>;
	constexpr int V   = G::V;
	constexpr int NP  = G::NP;
	constexpr int NA  = Fused ? 3 : 1;
	constexpr int W   = 2 * R + 1;
	constexpr int RING = G::ring(GS);
	using Pack        = typename PackOf<T>::type;
	using PU          = PackU<T, V>;

	if (done && *done) { return; }

#ifdef FI_B200_EMU
	unsigned char* smem_raw = ::cuda_emu::dynamic_smem();
#else
	extern __shared__ unsigned char smem_raw[];
#endif
	unsigned char* base = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
	auto stage_ptr = [&](int s, int a) { return reinterpret_cast<Pack*>(base + (static_cast<size_t>(s) * NA + a) * G::TILE_BYTES); };
	unsigned char* ring_base = base + static_cast<size_t>(S) * NA * G::TILE_BYTES;
	auto ring_ptr = [&](int slot) { return reinterpret_cast<Pack*>(ring_base + static_cast<size_t>(slot) * G::TILE_BYTES); };
	uint64_t* full  = reinterpret_cast<uint64_t*>(ring_base + static_cast<size_t>(RING) * G::TILE_BYTES);
	T*        zband = reinterpret_cast<T*>(full + S);                                      // [9][W]
	double*   red   = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(zband + 9 * W) + 7) & ~uintptr_t(7));

	const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
	const int x0t = blockIdx.x * (G::TXP * V);  // first element column of the tile
	const int y0t = blockIdx.y * G::TY;
	const int x0  = x0t + tx * V;
	const int y   = y0t + ty;
	// local planes [zo0, zo1) are owned (q is computed there) and split into chunks; lattice z = local z + zoff
	const int zb  = zo0 + blockIdx.z * zchunk;
	const int ze  = min(zo1, zb + zchunk);
	// the new direction is also written on up to R stored planes either side of the owned range (slab halos:
	// every slab recomputes its neighbours' boundary planes instead of exchanging p)
	const int wlo = blockIdx.z == 0 ? max(0, zo0 - R) : zb;
	const int whi = ze == zo1 ? min(nzl, zo1 + R) : ze;
	const bool   has_own = ty < G::TY;  // with 7-row tiles the eighth warp owns no row: it only fills halos
	const bool   in_xy = has_own && (x0 < nx) && (y < ny);
	const size_t plane = static_cast<size_t>(nx) * ny;

	if (tid == 0) {
#pragma unroll
		for (int s = 0; s < S; ++s) { mbar_init(&full[s], 1); }
		fence_barrier_init();
	}
	for (int k = tid; k < 9 * W; k += 256) { zband[k] = tab.band[2][k / W][k % W + 4 - R]; }

	T beta = 0;
	if (Fused) { beta = st->iters == 0 ? T(0) : static_cast<T>(st->rho[par] / st->rho[par ^ 1]); }

	// per-thread x / y coefficient rows (boundary truncation included)
	T cx[V][W], cy[W];
#pragma unroll
	for (int j = 0; j < V; ++j) {
		const int cls = row_class(min(x0 + j, nx - 1), nx);
#pragma unroll
		for (int t = 0; t < W; ++t) { cx[j][t] = tab.band[0][cls][t + 4 - R]; }
	}
	{
		const int cls = row_class(min(y, ny - 1), ny);
#pragma unroll
		for (int t = 0; t < W; ++t) { cy[t] = tab.band[1][cls][t + 4 - R]; }
	}
	// gradient smoothness (GS): diagonals of (D_1^T D_1) along x (per column of the pack) and y
	T lx0[V], ly0 = T(0);
	if (GS) {
#pragma unroll
		for (int j = 0; j < V; ++j) {
			const int xi = min(x0 + j, nx - 1);
			lx0[j]       = static_cast<T>((xi > 0 ? 1 : 0) + (xi < nx - 1 ? 1 : 0));
		}
		const int yi = min(y, ny - 1);
		ly0          = static_cast<T>((yi > 0 ? 1 : 0) + (yi < ny - 1 ? 1 : 0));
	}

	const int lp0    = zb - R;             // first plane loaded
	const int n_iter = ze + R - lp0;       // planes loaded by this block
	auto issue = [&](int i) {              // thread 0 only: plane lp0 + i into stage i % S
		const int s = i % S;
		mbar_expect_tx(&full[s], NA * G::BOX_BYTES);
		tma_load_3d(stage_ptr(s, 0), &map_a, &full[s], x0t - NP * V, y0t - R, lp0 + i);
		if (Fused) {
			tma_load_3d(stage_ptr(s, 1), &map_b, &full[s], x0t - NP * V, y0t - R, lp0 + i);
			tma_load_3d(stage_ptr(s, 2), &map_c, &full[s], x0t - NP * V, y0t - R, lp0 + i);
		}
	};
	__syncthreads();  // barriers initialised, zband visible
	if (tid == 0) {
		for (int i = 0; i < S && i < n_iter; ++i) { issue(i); }
	}

	// halo duties: one y-halo pack (warps 0..2R-1) and one x-halo pack (first 2*NP*TY threads) per plane
	const bool has_yh = ty < 2 * R;
	const int  yh_row = ty < R ? ty : G::TY + ty;
	const bool has_xh = tid < 2 * NP * G::TY;
	const int  xh_r   = (tid / (2 * NP)) + R;
	const int  xh_k   = tid % (2 * NP);
	const int  xh_col = xh_k < NP ? xh_k : G::TXP + xh_k;
	const int  own_at = (ty + R) * G::BXP + tx + NP;
	const int  yh_at  = yh_row * G::BXP + tx + NP;
	const int  xh_at  = xh_r * G::BXP + xh_col;
	// the box corners (x-halo columns of the y-halo rows) matter to the gradient-smoothness cross terms only: the first
	// 2 NP lanes of every y-halo warp fill them
	const bool has_ch = GS && has_yh && tx < 2 * NP;
	const int  ch_at  = yh_row * G::BXP + (tx < NP ? tx : G::TXP + tx);

	auto direction = [&](const Pack* sa, const Pack* sb, const Pack* sc, int at) -> Pack {
		if (!Fused) { return sa[at]; }
		PU rr, mm, pp, out;
		rr.v = sa[at];
		mm.v = sb[at];
		pp.v = sc[at];
#pragma unroll
		for (int j = 0; j < V; ++j) { out.a[j] = mm.a[j] * rr.a[j] + beta * pp.a[j]; }
		return out.v;
	};

	PU     pipe[W];
	double acc = 0.0;
	T*       qout = q + static_cast<size_t>(y) * nx + x0;
	T*       pout = Fused ? p_new + static_cast<size_t>(y) * nx + x0 : nullptr;

	// epilogue operands of this thread's pack, one plane ahead
	PU         pre_r, pre_m, pre_e;
	const bool epi_upd = Epi && epi.d_new != nullptr;
	const size_t xy_off = static_cast<size_t>(y) * nx + x0;
	auto epi_load = [&](int z) {
		const size_t at = static_cast<size_t>(z) * plane + xy_off;
		pre_r.v = *reinterpret_cast<const Pack*>(epi.res_in + at);
		if (epi_upd) {
			pre_m.v = *reinterpret_cast<const Pack*>(epi.minv + at);
			pre_e.v = *reinterpret_cast<const Pack*>(epi.e + at);
		}
	};
	if (Epi && in_xy && zb < ze) { epi_load(zb); }

	int stage = 0, slot = 0;
	uint32_t phase = 0;
	for (int i0 = 0; i0 < n_iter; i0 += W) {
#pragma unroll
		for (int k = 0; k < W; ++k) {
			const int i = i0 + k;
			if (i >= n_iter) { break; }
			const int lp = lp0 + i;
			mbar_wait(&full[stage], phase);
			const Pack* sa = stage_ptr(stage, 0);
			const Pack* sb = Fused ? stage_ptr(stage, 1) : nullptr;
			const Pack* sc = Fused ? stage_ptr(stage, 2) : nullptr;
			Pack*       rg = ring_ptr(slot);
			// newest plane of the own column -> pipe[k]; plane lp - 2R + t sits in pipe[(k + 1 + t) % W]
			if (has_own) {
				pipe[k].v  = direction(sa, sb, sc, own_at);
				rg[own_at] = pipe[k].v;
			}
			if (has_yh) { rg[yh_at] = direction(sa, sb, sc, yh_at); }
			if (has_xh) { rg[xh_at] = direction(sa, sb, sc, xh_at); }
			if (has_ch) { rg[ch_at] = direction(sa, sb, sc, ch_at); }
			if (Fused && in_xy && lp >= wlo && lp < whi) { *reinterpret_cast<Pack*>(pout + static_cast<size_t>(lp) * plane) = pipe[k].v; }
			__syncthreads();
			if (tid == 0 && i + S < n_iter) { issue(i + S); }

			const int z = lp - R;
			if (z >= zb && in_xy) {
				int zslot = slot - R;
				if (zslot < 0) { zslot += RING; }
				const Pack* pz = ring_ptr(zslot);
				const T*    cz = zband + row_class(z + zoff, nzg) * W;
				const PU&   ctr = pipe[(k + 1 + R) % W];
				PU          out;
				PU          cur_r, cur_m, cur_e;
				if (Epi) {
					cur_r = pre_r;
					cur_m = pre_m;
					cur_e = pre_e;
					if (z + 1 < ze) { epi_load(z + 1); }
				}
#pragma unroll
				for (int j = 0; j < V; ++j) {
					T s = T(0);
#pragma unroll
					for (int t = 0; t < W; ++t) { s += cz[t] * pipe[(k + 1 + t) % W].a[j]; }
					out.a[j] = s;
				}
				PU y_lo, y_hi;  // p(x, y -+ 1, z), kept for the cross terms
#pragma unroll
				for (int t = 0; t < W; ++t) {
					if (t == R) {
#pragma unroll
						for (int j = 0; j < V; ++j) { out.a[j] += cy[t] * ctr.a[j]; }
					} else {
						PU nb;
						nb.v = pz[(ty + t) * G::BXP + tx + NP];
#pragma unroll
						for (int j = 0; j < V; ++j) { out.a[j] += cy[t] * nb.a[j]; }
						if (GS && t == R - 1) { y_lo = nb; }
						if (GS && t == R + 1) { y_hi = nb; }
					}
				}
				T xs[(2 * NP + 1) * V];
#pragma unroll
				for (int kk = 0; kk < 2 * NP + 1; ++kk) {
					PU nb;
					if (kk == NP) { nb = ctr; } else { nb.v = pz[(ty + R) * G::BXP + tx + kk]; }
#pragma unroll
					for (int j = 0; j < V; ++j) { xs[kk * V + j] = nb.a[j]; }
				}
#pragma unroll
				for (int j = 0; j < V; ++j) {
#pragma unroll
					for (int t = 0; t < W; ++t) { out.a[j] += cx[j][t] * xs[NP * V + j + t - R]; }
				}
				if (GS) {
					// 2 w_gs^2 sum over axis pairs of (D_1^T D_1)_d (x) (D_1^T D_1)_o (field_interpolation.cpp:303-315): per pair
					// l_d l_o p - l_o (p at d -+ 1) - l_d (p at o -+ 1) + the four diagonal neighbours; neighbours outside the lattice
					// arrive as zeros.  Planes z - 1 and z + 1 of the new direction are in the ring (xy) and in the pipe (own column).
					const int zg  = z + zoff;
					const T   lz0 = static_cast<T>((zg > 0 ? 1 : 0) + (zg < nzg - 1 ? 1 : 0));
					int       sm  = zslot - 1, sp = zslot + 1;
					if (sm < 0) { sm += RING; }
					if (sp >= RING) { sp -= RING; }
					const Pack* pm = ring_ptr(sm);
					const Pack* pp = ring_ptr(sp);
					const PU&   z_lo = pipe[(k + R) % W];      // p(x, y, z - 1)
					const PU&   z_hi = pipe[(k + 2 + R) % W];  // p(x, y, z + 1)
					// three packs around the own column: [left, centre, right] -> element j sits at V + j
					T a_lo[3 * V], a_hi[3 * V], b_lo[3 * V], b_hi[3 * V];  // rows y -+ 1 of plane z; row y of planes z -+ 1
#pragma unroll
					for (int kk = 0; kk < 3; ++kk) {
						PU u0, u1, u2, u3;
						if (kk == 1) {
							u0 = y_lo;
							u1 = y_hi;
							u2 = z_lo;
							u3 = z_hi;
						} else {
							u0.v = pz[(ty + R - 1) * G::BXP + tx + NP - 1 + kk];
							u1.v = pz[(ty + R + 1) * G::BXP + tx + NP - 1 + kk];
							u2.v = pm[(ty + R) * G::BXP + tx + NP - 1 + kk];
							u3.v = pp[(ty + R) * G::BXP + tx + NP - 1 + kk];
						}
#pragma unroll
						for (int j = 0; j < V; ++j) {
							a_lo[kk * V + j] = u0.a[j];
							a_hi[kk * V + j] = u1.a[j];
							b_lo[kk * V + j] = u2.a[j];
							b_hi[kk * V + j] = u3.a[j];
						}
					}
					PU c0, c1, c2, c3;  // p(x, y -+ 1, z -+ 1): own column
					c0.v = pm[(ty + R - 1) * G::BXP + tx + NP];
					c1.v = pm[(ty + R + 1) * G::BXP + tx + NP];
					c2.v = pp[(ty + R - 1) * G::BXP + tx + NP];
					c3.v = pp[(ty + R + 1) * G::BXP + tx + NP];
#pragma unroll
					for (int j = 0; j < V; ++j) {
						const int cc = V + j, cx0 = NP * V + j;
						const T   lx = lx0[j];
						T g = (lx * ly0 + lx * lz0 + ly0 * lz0) * ctr.a[j];
						g -= (ly0 + lz0) * (xs[cx0 - 1] + xs[cx0 + 1]);
						g -= (lx + lz0) * (y_lo.a[j] + y_hi.a[j]);
						g -= (lx + ly0) * (z_lo.a[j] + z_hi.a[j]);
						g += a_lo[cc - 1] + a_lo[cc + 1] + a_hi[cc - 1] + a_hi[cc + 1];  // (x -+ 1, y -+ 1)
						g += b_lo[cc - 1] + b_lo[cc + 1] + b_hi[cc - 1] + b_hi[cc + 1];  // (x -+ 1, z -+ 1)
						g += c0.a[j] + c1.a[j] + c2.a[j] + c3.a[j];                      // (y -+ 1, z -+ 1)
						out.a[j] += gs2 * g;
					}
				}
				if (Epi) {
					const size_t at = static_cast<size_t>(z) * plane + xy_off;
					PU           rn;
#pragma unroll
					for (int j = 0; j < V; ++j) { rn.a[j] = cur_r.a[j] - out.a[j]; }
					if (epi.res_out) { *reinterpret_cast<Pack*>(epi.res_out + at) = rn.v; }
					if (epi_upd) {
						PU dn, en;
#pragma unroll
						for (int j = 0; j < V; ++j) {
							dn.a[j] = epi.a * ctr.a[j] + epi.b * cur_m.a[j] * rn.a[j];
							en.a[j] = cur_e.a[j] + dn.a[j];
						}
						*reinterpret_cast<Pack*>(epi.d_new + at) = dn.v;
						*reinterpret_cast<Pack*>(epi.e + at)     = en.v;
					}
				} else {
					*reinterpret_cast<Pack*>(qout + static_cast<size_t>(z) * plane) = out.v;
					T d = T(0);
#pragma unroll
					for (int j = 0; j < V; ++j) { d += out.a[j] * ctr.a[j]; }
					acc += static_cast<double>(d);
				}
			}
			if (++stage == S) { stage = 0; phase ^= 1u; }
			if (++slot == RING) { slot = 0; }
		}
	}

	if (dot_out) {
		double mine[1] = {block_sum(acc, red)};
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { *dot_out = tot[0]; });
	}
}

// ---- host side ------------------------------------------------------------------------------------------------
template <typename T, int R, int TY>
CUtensorMap make_map(const Geom& g, const T* ptr)
{
	using G = Tile<T, R, TY>;
	CUtensorMap m;
	std::memset(&m, 0, sizeof(m));
	EncodeFn fn = encode_fn();
	FI_REQUIRE(fn != nullptr, FI_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
	const cuuint64_t dims[3]    = {static_cast<cuuint64_t>(g.size[0]), static_cast<cuuint64_t>(g.size[1]), static_cast<cuuint64_t>(g.nzl)};
	const cuuint64_t strides[2] = {static_cast<cuuint64_t>(g.size[0]) * sizeof(T), static_cast<cuuint64_t>(g.size[0]) * g.size[1] * sizeof(T)};
	const cuuint32_t box[3]     = {static_cast<cuuint32_t>(G::BXP * G::V), static_cast<cuuint32_t>(G::BY), 1u};
	const cuuint32_t estr[3]    = {1u, 1u, 1u};
	const CUresult   r = fn(&m, sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3,
	                        const_cast<T*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
	                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	FI_REQUIRE(r == CUDA_SUCCESS, FI_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
	return m;
}

// z chunking.  A block marches its chunk plane by plane and pays 2R halo planes plus the pipeline fill per chunk, so
// chunks should be long; blocks run in waves of `resident`, so their number should fill whole waves.  Returns the chunk
// count that minimises waves * (planes per chunk + 2R + fill) for tiles of `ty` rows, and that cost.
inline double plan_chunks(const Geom& g, int R, int S, int minb, int tx_cells, int ty, int* out_chunks)
{
	const int     tiles_x = div_up(g.size[0], tx_cells), tiles_y = div_up(g.size[1], ty);
	const int64_t resident = static_cast<int64_t>(sm_count()) * minb;
	const int64_t tiles    = static_cast<int64_t>(tiles_x) * tiles_y;
	const int     nown     = g.zown1 - g.zown0;
	int           chunks   = 1;
	double        best     = 1e300;
	for (int c = 1; c <= std::max(1, nown / (2 * R + 1)) && c <= 256; ++c) {
		const int     zc    = div_up(nown, c);
		const int     cc    = div_up(nown, zc);
		const int64_t waves = (tiles * cc + resident - 1) / resident;
		// a last wave that is mostly empty still costs a whole chunk: charge partial waves at least half
		const double  frac  = static_cast<double>(tiles * cc) / static_cast<double>(resident);
		const double  cost  = std::max(static_cast<double>(waves) - 0.5, frac) * (zc + 2 * R + S + 1);
		if (cost < best - 1e-9) {
			best   = cost;
			chunks = cc;
		}
	}
	*out_chunks = chunks;
	return best;
}

template <typename T, int R, int S, bool Fused, int MINB, bool Epi, bool GS, int TY>
void launch_ty(const Geom& g, const StencilTables& t, int chunks, const T* a, const T* b, const T* c, T* q, T* p_new, const PcgState* st, int par,
               double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s, const EpiArgs<T>& epi)
{
	using G = Tile<T, R, TY>;
	TmaTables<T> tab;
	for (int ax = 0; ax < kMaxDim; ++ax) {
		for (int cl = 0; cl < 9; ++cl) {
			for (int k = 0; k < 9; ++k) { tab.band[ax][cl][k] = static_cast<T>(t.band[ax][cl][k]); }
		}
	}
	const CUtensorMap ma = make_map<T, R, TY>(g, a);
	const CUtensorMap mb = Fused ? make_map<T, R, TY>(g, b) : ma;
	const CUtensorMap mc = Fused ? make_map<T, R, TY>(g, c) : ma;
	const int tiles_x = div_up(g.size[0], G::TXP * G::V), tiles_y = div_up(g.size[1], G::TY);
	const int nown    = g.zown1 - g.zown0;
	const int zchunk  = div_up(nown, chunks);
	chunks            = div_up(nown, zchunk);
	dim3 grid(tiles_x, tiles_y, chunks);
	auto kern = stencil3d_tma_kernel<T, R, S, Fused, MINB, Epi, GS, TY>;
	constexpr size_t smem = smem_bytes<T, R, S, Fused, GS, TY>();
	static bool configured = false;  // per instantiation
	if (!configured) {
		FI_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
		configured = true;
	}
	FI_LAUNCH(kern, grid, 256, smem, s, ma, mb, mc, g.size[0], g.size[1], g.nzl, g.zown0, g.zown1, g.zoff, g.size[2], zchunk, tab,
	          static_cast<T>(t.gs2), q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, epi);
	note_stencil(FI_PCG_KERNEL_TMA_3D, R, GS, TY, chunks);
}

// Tile height.  Inside a long timed loop the GPU runs power-capped (SM clock ~1.78 of 1.97 GHz) and the kernel is bound by
// the SMs, not by HBM: what counts is the work of the busiest SM.  512^2 planes give 4 x 64 = 256 tiles of 8 rows on 296
// resident slots — 108 SMs carry two blocks, 40 carry one; with 7-row tiles they are 4 x 74 = 296 blocks, two per SM, each
// 7/8 of the work (the eighth warp only fills halo rows).  Measured (r2g): see profiles.  The choice minimises
// waves x planes x rows per block over {8, 7}; FI_B200_STENCIL_TY=7|8 forces one.
template <typename T, int R, int S, bool Fused, int MINB, bool Epi, bool GS>
void launch_gs(const Geom& g, const StencilTables& t, const T* a, const T* b, const T* c, T* q, T* p_new, const PcgState* st, int par,
               double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s, const EpiArgs<T>& epi = EpiArgs<T>())
{
	using G8 = Tile<T, R, 8>;
	int c8 = 1, c7 = 1;
	plan_chunks(g, R, S, MINB, G8::TXP * G8::V, 8, &c8);
	bool seven = false;
	if (R <= 2) {
		static const int forced = [] {
			const char* e = getenv("FI_B200_STENCIL_TY");
			return e ? atoi(e) : 0;
		}();
		plan_chunks(g, R, S, MINB, G8::TXP * G8::V, 7, &c7);
		// work of the busiest SM: whole waves x planes marched per block x rows per block
		auto busiest = [&](int ty, int chunks) {
			const int64_t blocks = static_cast<int64_t>(div_up(g.size[0], G8::TXP * G8::V)) * div_up(g.size[1], ty) * chunks;
			const int64_t waves  = (blocks + static_cast<int64_t>(sm_count()) * MINB - 1) / (static_cast<int64_t>(sm_count()) * MINB);
			return static_cast<double>(waves) * (div_up(g.zown1 - g.zown0, chunks) + 2 * R + S + 1) * ty;
		};
		seven = forced == 7 || (forced != 8 && busiest(7, c7) < 0.97 * busiest(8, c8));
	}
	if constexpr (R <= 2) {
		if (seven) {
			launch_ty<T, R, S, Fused, MINB, Epi, GS, 7>(g, t, c7, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s, epi);
			return;
		}
	}
	launch_ty<T, R, S, Fused, MINB, Epi, GS, 8>(g, t, c8, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s, epi);
}

template <typename T, int R, int S, bool Fused, int MINB, bool Epi = false>
void launch(const Geom& g, const StencilTables& t, const T* a, const T* b, const T* c, T* q, T* p_new, const PcgState* st, int par,
            double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s, const EpiArgs<T>& epi = EpiArgs<T>())
{
	if (t.gs2 != 0.0) {
		launch_gs<T, R, S, Fused, MINB, Epi, true>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s, epi);
	} else {
		launch_gs<T, R, S, Fused, MINB, Epi, false>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s, epi);
	}
}

template <typename T>
bool eligible(const Geom& g, const StencilTables& t)
{
	constexpr int V = 16 / sizeof(T);
	return g.ndim == 3 && t.radius >= 1 && g.size[0] % V == 0 && g.size[0] >= 32 && g.size[1] >= 8 && g.zown1 - g.zown0 >= 1 &&
	       (g.sharded() || g.size[2] >= 8) && encode_fn() != nullptr;
}

template <typename T, bool Fused>
void dispatch(const Geom& g, const StencilTables& t, const T* a, const T* b, const T* c, T* q, T* p_new, const PcgState* st, int par,
              double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done, cudaStream_t s)
{
	if (t.radius <= 1) {
		launch<T, 1, 3, Fused, 2>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s);
	} else if (t.radius == 2) {
		// FI_B200_STENCIL_VARIANT (tuning experiments on the default model_2 operator): 3 = two stages, three blocks per SM;
		// 4 = four stages, two blocks per SM; anything else = three stages, two blocks per SM (the measured default)
		static const int variant = [] {
			const char* e = getenv("FI_B200_STENCIL_VARIANT");
			return e ? atoi(e) : 0;
		}();
		if (variant == 3 && std::is_same<T, float>::value) {
			launch<T, 2, 2, Fused, 3>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s);
		} else if (variant == 4 && std::is_same<T, float>::value) {
			launch<T, 2, 4, Fused, 2>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s);
		} else {
			launch<T, 2, 3, Fused, 2>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s);
		}
	} else {
		launch<T, 4, 2, Fused, 1>(g, t, a, b, c, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s);
	}
}

}  // namespace

template <typename T>
bool stencil_tma_3d(const Geom& g, const StencilTables& t, const T* p, T* q, double* d_dot_out, double* d_partial, unsigned* d_ticket,
                    const int* d_done, cudaStream_t s)
{
	if (!eligible<T>(g, t)) { return false; }
	dispatch<T, false>(g, t, p, nullptr, nullptr, q, nullptr, nullptr, 0, d_dot_out, d_partial, d_ticket, d_done, s);
	return true;
}

template <typename T>
bool stencil_tma_3d_fused(const Geom& g, const StencilTables& t, const T* r, const T* minv, const T* p_old, T* p_new, T* q,
                          const PcgState* st, int par, double* d_dot_out, double* d_partial, unsigned* d_ticket, const int* d_done,
                          cudaStream_t s)
{
	if (!eligible<T>(g, t)) { return false; }
	dispatch<T, true>(g, t, r, minv, p_old, q, p_new, st, par, d_dot_out, d_partial, d_ticket, d_done, s);
	return true;
}

// q is not formed: res_out = res_in - S in, and with d_new: d_new = a in + b minv res_out, e += d_new.  false: not applicable.
template <typename T>
bool stencil_tma_3d_epilogue(const Geom& g, const StencilTables& t, const T* in, const T* res_in, T* res_out, const T* minv, T* e, T* d_new,
                             T a, T b, cudaStream_t s)
{
	// On a slab (g.sharded()) the owned planes are updated; the halo planes of `in` must be current, those of the outputs
	// are the caller's business.
	if (!eligible<T>(g, t)) { return false; }
	EpiArgs<T> epi;
	epi.res_in  = res_in;
	epi.res_out = res_out;
	epi.minv    = minv;
	epi.e       = e;
	epi.d_new   = d_new;
	epi.a       = a;
	epi.b       = b;
	if (t.radius <= 1) {
		launch<T, 1, 3, false, 2, true>(g, t, in, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, s, epi);
	} else if (t.radius == 2) {
		launch<T, 2, 3, false, 2, true>(g, t, in, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, s, epi);
	} else {
		launch<T, 4, 2, false, 1, true>(g, t, in, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr, s, epi);
	}
	return true;
}

template bool stencil_tma_3d_epilogue<float>(const Geom&, const StencilTables&, const float*, const float*, float*, const float*, float*, float*, float, float, cudaStream_t);
template bool stencil_tma_3d<float>(const Geom&, const StencilTables&, const float*, float*, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_tma_3d<double>(const Geom&, const StencilTables&, const double*, double*, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_tma_3d_fused<float>(const Geom&, const StencilTables&, const float*, const float*, const float*, float*, float*, const PcgState*, int, double*, double*, unsigned*, const int*, cudaStream_t);
template bool stencil_tma_3d_fused<double>(const Geom&, const StencilTables&, const double*, const double*, const double*, double*, double*, const PcgState*, int, double*, double*, unsigned*, const int*, cudaStream_t);

}  // namespace fi
