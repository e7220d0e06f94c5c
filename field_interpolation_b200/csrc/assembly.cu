// Assembly kernels: data constraints -> rows / normal-equation contributions, model rows for the triplet
// view, and multilinear upscaling.  This translation unit is compiled with -fmad=false so every fp32
// product and sum rounds exactly like the reference's scalar code (built without FMA, reference
// build.sh:68), which is what makes the exported triplets bit-identical.
//
// Reference behaviour restated here (paths relative to the reference tree):
//   multilerp                              field_interpolation/field_interpolation.cpp:15-55
//   add_value_constraint                   :57-80      add_value_constraint_nearest_neighbor  :82-107
//   cell_index                             :110-121    add_gradient_constraint                :123-240
//   add_model_constraint                   :243-316    add_field_constraints                  :326-341
//   add_points                             :343-371    upscale_field                          :431-485
//   add_equation                           field_interpolation/sparse_linear.cpp:34-50
#include <type_traits>

#include "internal.hpp"
#include "peer.cuh"

namespace fi {

namespace {

constexpr int kThreads = 256;

template <typename F>
void by_dim(int ndim, F&& f)
{
	switch (ndim) {
		case 1: f(std::integral_constant<int, 1>{}); break;
		case 2: f(std::integral_constant<int, 2>{}); break;
		default: f(std::integral_constant<int, 3>{}); break;
	}
}

__device__ __forceinline__ int floor_to_int(float x) { return static_cast<int>(floorf(x)); }

// Corners of the cell containing `pos` that lie inside the lattice (with `margin` extra room above),
// compacted in ascending corner order.  Returns how many were kept.
__device__ __forceinline__ int corner_weights(const Geom& g, const float* pos, int margin, int64_t* idx, float* w, int* cid)
{
	int   base[kMaxDim];
	float frac[kMaxDim];
	for (int d = 0; d < g.ndim; ++d) {
		base[d] = floor_to_int(pos[d]);
		frac[d] = pos[d] - static_cast<float>(base[d]);
	}
	int kept = 0;
	for (int corner = 0; corner < (1 << g.ndim); ++corner) {
		int64_t index = g.shift;
		float   wt    = 1.0f;
		bool    ok    = true;
		for (int d = 0; d < g.ndim; ++d) {
			const int bit = (corner >> d) & 1;
			const int c   = base[d] + bit;
			index += g.stride[d] * c;
			wt = wt * (bit ? frac[d] : 1.0f - frac[d]);
			ok = ok && (0 <= c) && (c + margin < g.size[d]);
		}
		if (ok) {
			idx[kept] = index;
			w[kept]   = wt;
			cid[kept] = corner;
			++kept;
		}
	}
	return kept;
}

// Everything one data point contributes, in the reference's emission order.
struct PointPlan
{
	// value row
	int     nv;          // triplets of the value row (0: no row)
	int64_t vidx[8];
	float   vcoef[8];
	int     vcorner[8];  // corner id inside cell floor(pos)
	float   vrhs;
	// gradient rows: gkind -1 none, else the GradientKernel
	int     gkind;
	int64_t cell;        // containing cell (kernels 0, 1)
	int     ng;          // interpolation samples (kernel 2)
	int64_t gidx[8];
	float   gcoef[8];    // k_i * cw
	float   gsum;        // sum of gcoef in sample order
	float   gw;
	float   grad[kMaxDim];
	int     base[kMaxDim];  // floor(pos)
};

__device__ __forceinline__ void analyse_point(const Geom& g, const PointView& pv, int64_t i, PointPlan& r)
{
	const int    D    = g.ndim;
	const float* pos  = pv.pos + i * D;
	const int    kind = pv.kind[i];
	const float  vw = pv.vw[i], gw = pv.gw[i], value = pv.value[i];
	for (int d = 0; d < D; ++d) {
		r.base[d] = floor_to_int(pos[d]);
		r.grad[d] = pv.grad[i * D + d];
	}
	r.nv    = 0;
	r.vrhs  = 0.0f;
	r.gkind = -1;
	r.ng    = 0;
	r.gw    = gw;
	r.cell  = -1;
	r.gsum  = 0.0f;

	if (kind & 1) {  // linear interpolation, :57-80
		if (vw != 0) {
			float     k[8];
			const int n = corner_weights(g, pos, 0, r.vidx, k, r.vcorner);
			float     sum = 0.0f;
			for (int c = 0; c < n; ++c) {
				r.vcoef[c] = k[c] * vw;
				sum        = sum + r.vcoef[c];
			}
			r.nv   = n;
			r.vrhs = sum * value;
		}
	} else {  // nearest neighbour, :82-107 (the row goes through add_equation: dropped when the weight is 0)
		int64_t node = g.shift;
		float   along = 0.0f;
		int     corner = 0;
		bool    inside = true;
		for (int d = 0; d < D; ++d) {
			const int nd = static_cast<int>(roundf(pos[d]));
			if (nd < 0 || g.size[d] <= nd) { inside = false; break; }
			along = along + (pos[d] - static_cast<float>(nd)) * r.grad[d];
			node += nd * g.stride[d];
			corner |= (nd - r.base[d]) << d;
		}
		if (inside && vw != 0) {
			r.nv         = 1;
			r.vidx[0]    = node;
			r.vcoef[0]   = 1.0f * vw;
			r.vcorner[0] = corner;
			r.vrhs       = (value - along) * vw;
		}
	}

	if ((kind & 8) && gw != 0) {  // :123-240
		const int gk = (kind >> 1) & 3;
		if (gk == 0 || gk == 1) {
			int64_t cell = g.shift;
			bool    ok   = true;
			for (int d = 0; d < D; ++d) {
				ok = ok && (0 <= r.base[d]) && (r.base[d] + 1 < g.size[d]);
				cell += r.base[d] * g.stride[d];
			}
			if (ok) {
				r.gkind = gk;
				r.cell  = cell;
			}
		} else {
			float shifted[kMaxDim];
			for (int d = 0; d < D; ++d) { shifted[d] = pos[d] - 0.5f; }
			float     k[8];
			int       cid[8];
			const int n = corner_weights(g, shifted, 1, r.gidx, k, cid);
			if (n > 0) {
				float sum = 0.0f;
				for (int c = 0; c < n; ++c) {
					r.gcoef[c] = k[c] * gw;
					sum        = sum + r.gcoef[c];
				}
				r.gkind = 2;
				r.ng    = n;
				r.gsum  = sum;
			}
		}
	}
}

__device__ __forceinline__ void plan_counts(const Geom& g, const PointPlan& r, unsigned& rows, unsigned& trips)
{
	rows  = r.nv > 0 ? 1u : 0u;
	trips = static_cast<unsigned>(r.nv);
	if (r.gkind == 0) { rows += g.ndim; trips += 2u * g.ndim; }
	if (r.gkind == 1) { rows += g.ndim; trips += static_cast<unsigned>(g.ndim << g.ndim); }
	if (r.gkind == 2) { rows += g.ndim; trips += 2u * r.ng * g.ndim; }
}

// ---- canonical point records ----------------------------------------------------------------------------
__global__ void canonicalise_kernel(int D, int64_t n, int64_t at, const float* __restrict__ pos, const float* __restrict__ nrm,
                                    const float* __restrict__ pw, const float* __restrict__ val, float value_weight,
                                    float gradient_weight, int kind, float* o_pos, float* o_grad, float* o_value,
                                    float* o_vw, float* o_gw, uint8_t* o_kind)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	const float w = pw ? pw[i] : 1.0f;  // add_points :357
	for (int d = 0; d < D; ++d) {
		o_pos[(at + i) * D + d]  = pos[i * D + d];
		o_grad[(at + i) * D + d] = nrm ? nrm[i * D + d] : 0.0f;
	}
	o_value[at + i] = val ? val[i] : 0.0f;
	o_vw[at + i]    = w * value_weight;     // :362,364
	o_gw[at + i]    = w * gradient_weight;  // :368
	o_kind[at + i]  = static_cast<uint8_t>(kind);
}

__global__ void point_counts_kernel(Geom g, PointView pv, int64_t p0, int64_t n, uint64_t* rows, uint64_t* trips)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	PointPlan r;
	analyse_point(g, pv, p0 + i, r);
	unsigned nr, nt;
	plan_counts(g, r, nr, nt);
	rows[i]  = nr;
	trips[i] = nt;
}

__global__ void point_emit_kernel(Geom g, PointView pv, int64_t p0, int64_t n, const uint64_t* __restrict__ rowoff,
                                  const uint64_t* __restrict__ tripoff, int64_t row_base, int64_t trip_base,
                                  fi_triplet* __restrict__ trips, float* __restrict__ rhs)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	PointPlan r;
	analyse_point(g, pv, p0 + i, r);
	int64_t row = row_base + static_cast<int64_t>(rowoff[i]);
	int64_t t   = trip_base + static_cast<int64_t>(tripoff[i]);
	const int D = g.ndim;
	if (r.nv > 0) {
		for (int c = 0; c < r.nv; ++c) { trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(r.vidx[c]), r.vcoef[c]}; }
		rhs[row++] = r.vrhs;
	}
	if (r.gkind == 0) {  // :134-149 via add_equation: coefficient = pair.value * weight
		for (int d = 0; d < D; ++d) {
			trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(r.cell), -1.0f * r.gw};
			trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(r.cell + g.stride[d]), +1.0f * r.gw};
			rhs[row++] = r.grad[d] * r.gw;
		}
	} else if (r.gkind == 1) {  // :150-187
		const int   corners = 1 << D;
		const float term    = r.gw * 2.0f / static_cast<float>(corners);
		for (int d = 0; d < D; ++d) {
			for (int c = 0; c < corners; ++c) {
				int64_t node = r.cell;
				for (int a = 0; a < D; ++a) { node += g.stride[a] * ((c >> a) & 1); }
				const float sign = ((c >> d) & 1) ? +1.0f : -1.0f;
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(node), sign * term};
			}
			rhs[row++] = r.gw * r.grad[d];
		}
	} else if (r.gkind == 2) {  // :188-236
		for (int d = 0; d < D; ++d) {
			for (int c = 0; c < r.ng; ++c) {
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(r.gidx[c]), -r.gcoef[c]};
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(r.gidx[c] + g.stride[d]), +r.gcoef[c]};
			}
			rhs[row++] = r.gsum * r.grad[d];
		}
	}
}

// ---- model rows (triplet view only; the solver applies them matrix-free, see stencil.cu) -------------------
__device__ __forceinline__ void coords_of(const Geom& g, int64_t index, int* c)
{
	for (int d = 0; d < g.ndim; ++d) {
		c[d] = static_cast<int>(index % g.size[d]);
		index /= g.size[d];
	}
}

__global__ void model_counts_kernel(Geom g, fi_weights w, uint64_t* rows, uint64_t* trips)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= g.N) { return; }
	int c[kMaxDim];
	coords_of(g, i, c);
	const float wk[5] = {w.model_0, w.model_1, w.model_2, w.model_3, w.model_4};
	unsigned    nr = 0, nt = 0;
	for (int d = 0; d < g.ndim; ++d) {
		for (int k = 0; k <= 4; ++k) {
			if (wk[k] > 0 && c[d] + k < g.size[d]) { nr += 1; nt += k + 1; }
		}
		if (w.gradient_smoothness > 0 && c[d] + 1 < g.size[d]) {
			for (int o = 0; o < g.ndim; ++o) {
				if (o != d && c[o] + 1 < g.size[o]) { nr += 1; nt += 4; }
			}
		}
	}
	rows[i]  = nr;
	trips[i] = nt;
}

__global__ void model_emit_kernel(Geom g, fi_weights w, const uint64_t* __restrict__ rowoff, const uint64_t* __restrict__ tripoff,
                                  int64_t row_base, int64_t trip_base, fi_triplet* __restrict__ trips, float* __restrict__ rhs)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= g.N) { return; }
	int c[kMaxDim];
	coords_of(g, i, c);
	const float wk[5]       = {w.model_0, w.model_1, w.model_2, w.model_3, w.model_4};
	const float binom[5][5] = {{1, 0, 0, 0, 0}, {-1, 1, 0, 0, 0}, {1, -2, 1, 0, 0}, {1, -3, 3, -1, 0}, {1, -4, 6, -4, 1}};
	int64_t row = row_base + static_cast<int64_t>(rowoff[i]);
	int64_t t   = trip_base + static_cast<int64_t>(tripoff[i]);
	for (int d = 0; d < g.ndim; ++d) {
		for (int k = 0; k <= 4; ++k) {
			if (!(wk[k] > 0 && c[d] + k < g.size[d])) { continue; }
			for (int m = 0; m <= k; ++m) {
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(i + m * g.stride[d]), binom[k][m] * wk[k]};
			}
			rhs[row++] = 0.0f * wk[k];
		}
		if (w.gradient_smoothness > 0 && c[d] + 1 < g.size[d]) {
			for (int o = 0; o < g.ndim; ++o) {
				if (o == d || c[o] + 1 >= g.size[o]) { continue; }
				const float   gs = w.gradient_smoothness;
				const int64_t sd = g.stride[d], so = g.stride[o];
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(i), -1.0f * gs};
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(i + sd), +1.0f * gs};
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(i + so), +1.0f * gs};
				trips[t++] = fi_triplet{static_cast<int32_t>(row), static_cast<int32_t>(i + so + sd), -1.0f * gs};
				rhs[row++] = 0.0f * gs;
			}
		}
	}
}

// ---- upscale_field ---------------------------------------------------------------------------------------
__global__ void upscale_kernel(Geom small, Geom large, const float* __restrict__ src, float* __restrict__ dst, float post_scale)
{
	const int64_t li = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (li >= large.N) { return; }
	int c[kMaxDim];
	coords_of(large, li, c);
	float pos[kMaxDim];
	for (int d = 0; d < small.ndim; ++d) {
		// :462  (float)coord * (small - 1.0f) / (large - 1.0f), evaluated left to right in fp32
		pos[d] = static_cast<float>(c[d]) * (static_cast<float>(small.size[d]) - 1.0f) / (static_cast<float>(large.size[d]) - 1.0f);
	}
	int64_t   idx[8];
	float     k[8];
	int       cid[8];
	const int n = corner_weights(small, pos, 0, idx, k, cid);
	float wsum = 0.0f, fsum = 0.0f;
	for (int s = 0; s < n; ++s) {
		wsum = wsum + k[s];
		fsum = fsum + k[s] * src[idx[s]];
	}
	float out = (wsum == 0.0f) ? 0.0f : fsum / wsum;
	if (post_scale != 1.0f) { out = out * post_scale; }  // src/sdf_field.cpp:286-288
	dst[li] = out;
}

// ---- data term: keys, scatter ------------------------------------------------------------------------------
// Key of cell floor(pos) over the extended range base_d in [-1, size_d - 1]; `no_cell` (one past the largest key) for points that add
// nothing to a cell block (no value row and no nearest-neighbour / cell-edge gradient rows).
__global__ void cell_keys_kernel(Geom g, PointView pv, int64_t n, uint64_t no_cell, uint64_t* keys, uint32_t* order,
                                 unsigned long long* valid)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	PointPlan r;
	analyse_point(g, pv, i, r);
	uint64_t key = no_cell;
	// a slab keeps the cells that touch a plane it owns: floor(pos_z) in [first owned - 1, last owned]
	const bool in_window = !g.sharded() || (r.base[2] - g.zoff >= g.zown0 - 1 && r.base[2] - g.zoff <= g.zown1 - 1);
	if (in_window && (r.nv > 0 || r.gkind == 0 || r.gkind == 1)) {
		key            = 0;
		uint64_t kstr  = 1;
		for (int d = 0; d < g.ndim; ++d) {
			key += static_cast<uint64_t>(r.base[d] + 1) * kstr;
			kstr *= static_cast<uint64_t>(g.size[d] + 1);
		}
		atomicAdd(valid, 1ull);
	}
	keys[i]  = key;
	order[i] = static_cast<uint32_t>(i);
}

__global__ void mark_heads_kernel(const uint64_t* __restrict__ keys, int64_t n, uint64_t* flags)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	flags[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1ull : 0ull;
}

__global__ void slots_kernel(const uint64_t* __restrict__ keys, const uint64_t* __restrict__ flags,
                             const uint64_t* __restrict__ scan, int64_t n, uint32_t* slot, uint64_t* cell_key)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	const uint64_t s = scan[i] + flags[i] - 1;
	slot[i]          = static_cast<uint32_t>(s);
	if (flags[i]) { cell_key[s] = keys[i]; }
}

template <typename T>
__device__ __forceinline__ void atomic_add(T* p, T v) { atomicAdd(p, v); }

// (Pairing the reductions of x-neighbouring corners into REDG.ADD.F32x2 was tried in round 2 and measured slower on the
// B200: 0.085 vs 0.078 ms for the 512^3 bench cloud, profiles/r2f_time_iters_variant0.jsonl — scalar reductions stay.)

// One lane per (cell-sorted) point.  Each lane forms its point's contribution to the cell's symmetric block,
// right-hand side and diagonal; lanes of the same cell are contiguous, so a segmented shuffle reduction folds
// them and only the head lane of every run issues atomics.
template <typename T, int D>
__global__ void __launch_bounds__(kThreads) scatter_points_kernel(Geom g, PointView pv, const uint32_t* __restrict__ order,
                                                                  const uint32_t* __restrict__ slot, int64_t n, int64_t nocc,
                                                                  T* __restrict__ blocks, T* __restrict__ atb, T* __restrict__ diag)
{
	constexpr int C    = 1 << D;
	const int64_t i    = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	const int     lane = threadIdx.x & 31;
	const bool    live = i < n;

	T        a[C];        // value-row coefficients by corner
	T        s[D][C];     // gradient-row coefficients by corner
	T        vr = 0, gr[D];
	int      base[D];
	unsigned my_slot = 0xffffffffu;
#pragma unroll
	for (int c = 0; c < C; ++c) {
		a[c] = 0;
#pragma unroll
		for (int d = 0; d < D; ++d) { s[d][c] = 0; }
	}
#pragma unroll
	for (int d = 0; d < D; ++d) { gr[d] = 0; base[d] = 0; }

	if (live) {
		PointPlan r;
		analyse_point(g, pv, order[i], r);
		my_slot = slot[i];
#pragma unroll
		for (int d = 0; d < D; ++d) { base[d] = r.base[d]; }
		for (int k = 0; k < r.nv; ++k) {
#pragma unroll
			for (int c = 0; c < C; ++c) {
				if (c == r.vcorner[k]) { a[c] = static_cast<T>(r.vcoef[k]); }
			}
		}
		vr = static_cast<T>(r.vrhs);
		if (r.gkind == 0) {
#pragma unroll
			for (int d = 0; d < D; ++d) {
				s[d][0]      = static_cast<T>(-1.0f * r.gw);
				s[d][1 << d] = static_cast<T>(+1.0f * r.gw);
				gr[d]        = static_cast<T>(r.grad[d] * r.gw);
			}
		} else if (r.gkind == 1) {
			const float term = r.gw * 2.0f / static_cast<float>(C);
#pragma unroll
			for (int d = 0; d < D; ++d) {
#pragma unroll
				for (int c = 0; c < C; ++c) { s[d][c] = static_cast<T>(((c >> d) & 1) ? +1.0f * term : -1.0f * term); }
				gr[d] = static_cast<T>(r.gw * r.grad[d]);
			}
		}
	}

	// run structure inside the warp
	bool same[5];
#pragma unroll
	for (int k = 0; k < 5; ++k) {
		const unsigned other = __shfl_down_sync(0xffffffffu, my_slot, 1 << k);
		same[k]              = (lane + (1 << k) < 32) && (other == my_slot);
	}
	const unsigned prev = __shfl_up_sync(0xffffffffu, my_slot, 1);
	const bool     head = live && (lane == 0 || prev != my_slot);

	auto fold = [&](T v) {
#pragma unroll
		for (int k = 0; k < 5; ++k) {
			const T y = __shfl_down_sync(0xffffffffu, v, 1 << k);
			if (same[k]) { v += y; }
		}
		return v;
	};

	int tri = 0;
#pragma unroll
	for (int ci = 0; ci < C; ++ci) {
#pragma unroll
		for (int cj = ci; cj < C; ++cj) {
			T v = a[ci] * a[cj];
#pragma unroll
			for (int d = 0; d < D; ++d) { v += s[d][ci] * s[d][cj]; }
			v = fold(v);
			if (head && v != T(0)) { atomic_add(&blocks[static_cast<size_t>(tri) * nocc + my_slot], v); }
			if (ci == cj) {
				bool    inside = true;
				int64_t node   = g.shift;
#pragma unroll
				for (int d = 0; d < D; ++d) {
					const int c = base[d] + ((ci >> d) & 1);
					inside      = inside && (0 <= c) && (c < g.size[d]);
					node += g.stride[d] * c;
				}
				T b = a[ci] * vr;
#pragma unroll
				for (int d = 0; d < D; ++d) { b += s[d][ci] * gr[d]; }
				b = fold(b);
				if (head && inside) {
					if (v != T(0)) { atomic_add(&diag[node], v); }
					if (b != T(0)) { atomic_add(&atb[node], b); }
				}
			}
			++tri;
		}
	}
}

// ---- rows that do not fit one cell: linear-interpolation gradient rows -> CSR -------------------------------
__global__ void derived_counts_kernel(Geom g, PointView pv, int64_t n, uint64_t* rows, uint64_t* ents)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	PointPlan r;
	analyse_point(g, pv, i, r);
	rows[i] = r.gkind == 2 ? g.ndim : 0;
	ents[i] = r.gkind == 2 ? 2ull * r.ng * g.ndim : 0;
}

template <typename T>
__global__ void derived_emit_kernel(Geom g, PointView pv, int64_t n, const uint64_t* __restrict__ rowoff,
                                    const uint64_t* __restrict__ entoff, uint64_t* __restrict__ row_ptr,
                                    int32_t* __restrict__ col, float* __restrict__ val, T* __restrict__ atb, T* __restrict__ diag)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	PointPlan r;
	analyse_point(g, pv, i, r);
	if (r.gkind != 2) { return; }
	uint64_t row = rowoff[i], e = entoff[i];
	for (int d = 0; d < g.ndim; ++d) {
		row_ptr[row++] = e;
		const T rhs    = static_cast<T>(r.gsum * r.grad[d]);
		for (int c = 0; c < r.ng; ++c) {
			const T       v  = static_cast<T>(r.gcoef[c]);
			const int64_t lo = r.gidx[c], hi = r.gidx[c] + g.stride[d];
			col[e] = static_cast<int32_t>(lo); val[e++] = -r.gcoef[c];
			col[e] = static_cast<int32_t>(hi); val[e++] = +r.gcoef[c];
			atomic_add(&atb[lo], -v * rhs);
			atomic_add(&atb[hi], +v * rhs);
			// duplicate columns inside a row are separate triplets that AtA sums: diag gets (sum of dups)^2,
			// handled below by accumulating the row's per-column totals first
		}
		// diagonal: per distinct column, (sum of its coefficients in this row)^2
		for (int c = 0; c < 2 * r.ng; ++c) {
			const int64_t node = (c & 1) ? r.gidx[c >> 1] + g.stride[d] : r.gidx[c >> 1];
			bool first = true;
			T    tot   = 0;
			for (int c2 = 0; c2 < 2 * r.ng; ++c2) {
				const int64_t node2 = (c2 & 1) ? r.gidx[c2 >> 1] + g.stride[d] : r.gidx[c2 >> 1];
				if (node2 != node) { continue; }
				if (c2 < c) { first = false; }
				tot += static_cast<T>((c2 & 1) ? r.gcoef[c2 >> 1] : -r.gcoef[c2 >> 1]);
			}
			if (first) { atomic_add(&diag[node], tot * tot); }
		}
	}
}

// Caller rows: accumulate Atb and the diagonal (duplicates inside a row summed first, as setFromTriplets does).
template <typename T>
__global__ void user_rows_accumulate_kernel(int64_t nrows, const uint64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                                            const float* __restrict__ val, const float* __restrict__ rhs, T* __restrict__ atb,
                                            T* __restrict__ diag)
{
	const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (r >= nrows) { return; }
	const uint64_t b = row_ptr[r], e = row_ptr[r + 1];
	const T        rh = static_cast<T>(rhs[r]);
	for (uint64_t k = b; k < e; ++k) {
		atomic_add(&atb[col[k]], static_cast<T>(val[k]) * rh);
		bool first = true;
		T    tot   = 0;
		for (uint64_t k2 = b; k2 < e; ++k2) {
			if (col[k2] != col[k]) { continue; }
			if (k2 < k) { first = false; }
			tot += static_cast<T>(val[k2]);
		}
		if (first) { atomic_add(&diag[col[k]], tot * tot); }
	}
}

__global__ void shift_ptr_kernel(uint64_t* ptr, int64_t n, uint64_t add)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i < n) { ptr[i] += add; }
}

// ---- apply: q += P p ------------------------------------------------------------------------------------------
// Decodes the sorted cell keys once per operator build: corner-0 index and which corners exist / are owned.
template <int D>
__global__ void cell_nodes_kernel(Geom g, int64_t nocc, const uint64_t* __restrict__ cell_key, int64_t* __restrict__ cell_base,
                                  uint32_t* __restrict__ cell_mask)
{
	constexpr int C = 1 << D;
	const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (cell >= nocc) { return; }
	uint64_t key = cell_key[cell];
	int      base[D];
	int64_t  node = g.shift;
#pragma unroll
	for (int d = 0; d < D; ++d) {
		const uint64_t ext = static_cast<uint64_t>(g.size[d] + 1);
		base[d] = static_cast<int>(key % ext) - 1;
		key /= ext;
		node += g.stride[d] * base[d];
	}
	uint32_t mask = 0;
#pragma unroll
	for (int c = 0; c < C; ++c) {
		bool ok = true;
#pragma unroll
		for (int d = 0; d < D; ++d) {
			const int x = base[d] + ((c >> d) & 1);
			ok          = ok && (0 <= x) && (x < g.size[d]);
		}
		bool own = ok;
		if (D == 3 && g.sharded()) {  // rows of nodes another slab owns are that slab's business
			const int zl = base[D - 1] + ((c >> (D - 1)) & 1) - g.zoff;
			own          = ok && zl >= g.zown0 && zl < g.zown1;
		}
		mask |= (ok ? 1u : 0u) << c;
		mask |= (own ? 1u : 0u) << (8 + c);
	}
	cell_base[cell] = node;
	cell_mask[cell] = mask;
}

// q += P p over the occupied cells: one thread per cell reads its 2^D corner values of p, multiplies by the
// symmetric block (upper triangle, [tri][cell] so that a warp reads consecutive cells of one entry) and adds the
// 2^D results to q with atomics (neighbouring cells share corners).
// TILED (tile mode, Geom::tile): entries between corners that lie in different tiles are dropped; the cell's base
// coordinates come from its key.
template <typename T, int D, bool TILED>
__global__ void __launch_bounds__(kThreads, 3) apply_blocks_kernel(Geom g, int64_t nocc, const int64_t* __restrict__ cell_base,
                                                                const uint32_t* __restrict__ cell_mask, const T* __restrict__ blocks,
                                                                const T* __restrict__ p, T* __restrict__ q, double* partial,
                                                                unsigned* ticket, double* dot_accum, const int* done,
                                                                const uint64_t* __restrict__ cell_key, PeerPublish pub, int do_pub)
{
	constexpr int C = 1 << D;
	__shared__ double red[32];
	__shared__ double s_tot;
	__shared__ int    s_pub;
	if (done && *done) {
		// a finished solve still publishes (zeros): the peers' kernels of this round are already waiting
		if (do_pub && blockIdx.x == 0 && threadIdx.x < 32) {
			const double zero[1] = {0.0};
			peer_publish_warp(pub.link, pub.which, pub.par, seq_of(pub.base, pub.st, pub.which), zero, 1);
		}
		return;
	}
	if (threadIdx.x == 0) { s_pub = 0; }
	const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	double        mine[1] = {0.0};
	if (cell < nocc) {
		// every load of this thread is issued before the first use: the kernel is latency-bound otherwise
		constexpr int NT = C * (C + 1) / 2;
		T             blk[NT];
#pragma unroll
		for (int t = 0; t < NT; ++t) { blk[t] = __ldcs(&blocks[static_cast<size_t>(t) * nocc + cell]); }
		const int64_t  base = cell_base[cell];
		const uint32_t mask = cell_mask[cell];
		T pc[C], out[C];
#pragma unroll
		for (int c = 0; c < C; ++c) {
			int64_t off = 0;
#pragma unroll
			for (int d = 0; d < D; ++d) { off += ((c >> d) & 1) ? g.stride[d] : 0; }
			pc[c]  = ((mask >> c) & 1u) ? p[base + off] : T(0);
			out[c] = 0;
		}
		int cross = 0;  // bit d: the cell straddles a tile boundary along axis d
		if (TILED) {
			uint64_t key = cell_key[cell];
#pragma unroll
			for (int d = 0; d < D; ++d) {
				const uint64_t ext = static_cast<uint64_t>(g.size[d] + 1);
				const int      b1  = static_cast<int>(key % ext);  // base coordinate + 1
				key /= ext;
				cross |= (b1 % g.tile == 0 ? 1 : 0) << d;
			}
		}
		int tri = 0;
#pragma unroll
		for (int ci = 0; ci < C; ++ci) {
#pragma unroll
			for (int cj = ci; cj < C; ++cj) {
				T b = blk[tri];
				if (TILED && ((ci ^ cj) & cross)) { b = T(0); }
				out[ci] += b * pc[cj];
				if (cj != ci) { out[cj] += b * pc[ci]; }
				++tri;
			}
		}
		T dot = 0;
#pragma unroll
		for (int c = 0; c < C; ++c) {
			if ((mask >> (8 + c)) & 1u) {
				int64_t off = 0;
#pragma unroll
				for (int d = 0; d < D; ++d) { off += ((c >> d) & 1) ? g.stride[d] : 0; }
				atomic_add(&q[base + off], out[c]);
				dot += pc[c] * out[c];
			}
		}
		mine[0] = static_cast<double>(dot);
	}
	if (dot_accum) {
		mine[0] = block_sum(mine[0], red);
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) {
			const double all = *dot_accum + tot[0];
			*dot_accum       = all;
			s_tot            = all;
			s_pub            = 1;
		});
	}
	if (do_pub) {  // the block that completed p.Ap of this rank sends it to every rank (solver.cu: peer-memory path)
		__syncthreads();
		if (s_pub && threadIdx.x < 32) {
			const double v[1] = {s_tot};
			if (threadIdx.x == 0) { pub.link.local->stamp[0][pub.st->iters & 511] = global_ns(); }
			peer_publish_warp(pub.link, pub.which, pub.par, seq_of(pub.base, pub.st, pub.which), v, 1);
		}
	}
}

// The same product with one thread per (cell, corner row): a block covers 256 consecutive cells, thread group ci (one
// warp in 3D) owns output row ci of every cell and walks the block's cells in 2^D strides of 256 / 2^D.  Each thread
// issues 2^D coalesced block loads + 2^D gathers of p and one atomic — 2^D times the threads of the per-cell kernel
// with 1 / 2^D of its dependent work each, which is what this latency-bound kernel needs (the per-cell form holds
// 36 + 16 values in registers and runs at a third of the SM's warp slots).  A block element is read by the two rows
// that share it; the second read hits L1.
template <typename T, int D>
__global__ void __launch_bounds__(kThreads) apply_blocks_split_kernel(Geom g, int64_t nocc, const int64_t* __restrict__ cell_base,
                                                                      const uint32_t* __restrict__ cell_mask, const T* __restrict__ blocks,
                                                                      const T* __restrict__ p, T* __restrict__ q, double* partial,
                                                                      unsigned* ticket, double* dot_accum, const int* done)
{
	constexpr int C = 1 << D, CPB = kThreads / C;
	__shared__ double red[32];
	if (done && *done) { return; }
	const int ci = threadIdx.x / CPB, lane = threadIdx.x % CPB;
	int64_t   off[C];
#pragma unroll
	for (int c = 0; c < C; ++c) {
		off[c] = 0;
#pragma unroll
		for (int d = 0; d < D; ++d) { off[c] += ((c >> d) & 1) ? g.stride[d] : 0; }
	}
	int64_t off_ci = 0;
#pragma unroll
	for (int d = 0; d < D; ++d) { off_ci += ((ci >> d) & 1) ? g.stride[d] : 0; }
	T dot = 0;
#pragma unroll 2
	for (int it = 0; it < C; ++it) {
		const int64_t cell = static_cast<int64_t>(blockIdx.x) * kThreads + it * CPB + lane;
		if (cell >= nocc) { continue; }
		T b[C];
#pragma unroll
		for (int cj = 0; cj < C; ++cj) {
			const int lo = min(ci, cj), hi = max(ci, cj);
			const int tri = lo * C - (lo * (lo - 1)) / 2 + (hi - lo);  // row-major upper triangle, as build_data_term stores it
			b[cj] = __ldg(&blocks[static_cast<size_t>(tri) * nocc + cell]);
		}
		const int64_t  base = cell_base[cell];
		const uint32_t mask = cell_mask[cell];
		T out = 0, pci = 0;
#pragma unroll
		for (int cj = 0; cj < C; ++cj) {
			const T pv = ((mask >> cj) & 1u) ? p[base + off[cj]] : T(0);
			out += b[cj] * pv;
			if (cj == ci) { pci = pv; }
		}
		if ((mask >> (8 + ci)) & 1u) {
			atomic_add(&q[base + off_ci], out);
			dot += pci * out;
		}
	}
	if (dot_accum) {
		double mine[1] = {static_cast<double>(dot)};
		mine[0] = block_sum(mine[0], red);
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { *dot_accum += tot[0]; });
	}
}

// Epilogue form for the multigrid smoother: u = P in over the occupied cells, then res -= u and (d_new given)
// d_new -= b minv u, e -= b minv u.
template <typename T, int D>
__global__ void __launch_bounds__(kThreads, 3) apply_blocks_epilogue_kernel(Geom g, int64_t nocc, const int64_t* __restrict__ cell_base,
                                                                         const uint32_t* __restrict__ cell_mask, const T* __restrict__ blocks,
                                                                         const T* __restrict__ in, T* res, const T* __restrict__ minv, T* e,
                                                                         T* d_new, T b)
{
	constexpr int C  = 1 << D;
	constexpr int NT = C * (C + 1) / 2;
	const int64_t cell = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (cell >= nocc) { return; }
	T blk[NT];
#pragma unroll
	for (int t = 0; t < NT; ++t) { blk[t] = __ldcs(&blocks[static_cast<size_t>(t) * nocc + cell]); }
	const int64_t  base = cell_base[cell];
	const uint32_t mask = cell_mask[cell];
	T pc[C], out[C];
	int64_t off[C];
#pragma unroll
	for (int c = 0; c < C; ++c) {
		off[c] = 0;
#pragma unroll
		for (int d = 0; d < D; ++d) { off[c] += ((c >> d) & 1) ? g.stride[d] : 0; }
		pc[c]  = ((mask >> c) & 1u) ? in[base + off[c]] : T(0);
		out[c] = 0;
	}
	int tri = 0;
#pragma unroll
	for (int ci = 0; ci < C; ++ci) {
#pragma unroll
		for (int cj = ci; cj < C; ++cj) {
			const T v = blk[tri];
			out[ci] += v * pc[cj];
			if (cj != ci) { out[cj] += v * pc[ci]; }
			++tri;
		}
	}
#pragma unroll
	for (int c = 0; c < C; ++c) {
		if ((mask >> (8 + c)) & 1u) {
			const int64_t node = base + off[c];
			atomic_add(&res[node], -out[c]);
			if (d_new) {
				const T dd = -b * minv[node] * out[c];
				atomic_add(&d_new[node], dd);
				atomic_add(&e[node], dd);
			}
		}
	}
}

// ---- node-major form of P (DataTerm::node_*) ----------------------------------------------------------------------
__host__ __device__ constexpr int pow3(int d) { return d == 1 ? 3 : (d == 2 ? 9 : 27); }

// One key per (occupied cell, corner): the local index of the corner's node when this process owns its row, else
// `sentinel` (sorts behind every node).
template <int D>
__global__ void node_keys_kernel(Geom g, int64_t nocc, const int64_t* __restrict__ cell_base, const uint32_t* __restrict__ cell_mask,
                                 uint64_t sentinel, uint64_t* __restrict__ keys, uint32_t* __restrict__ vals, unsigned long long* valid)
{
	constexpr int C = 1 << D;
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	bool          own = false;
	if (i < nocc * C) {
		const int64_t cell = i / C;
		const int     c    = static_cast<int>(i % C);
		own                = (cell_mask[cell] >> (8 + c)) & 1u;
		int64_t off = 0;
#pragma unroll
		for (int d = 0; d < D; ++d) { off += ((c >> d) & 1) ? g.stride[d] : 0; }
		keys[i] = own ? static_cast<uint64_t>(cell_base[cell] + off) : sentinel;
		vals[i] = 0;
	}
	const unsigned b = __ballot_sync(0xffffffffu, own);
	if ((threadIdx.x & 31) == 0 && b) { atomicAdd(valid, static_cast<unsigned long long>(__popc(b))); }
}

// Row of P of every touched node, gathered from the blocks of the 2^D cells around it (found by binary search in the
// sorted cell keys).  Fixed summation order: cells in ascending corner order.
template <typename T, int D>
__global__ void __launch_bounds__(kThreads) node_rows_kernel(Geom g, int64_t nnode, const uint64_t* __restrict__ node_key, int64_t nocc,
                                                             const uint64_t* __restrict__ cell_key, const T* __restrict__ blocks,
                                                             int64_t* __restrict__ node_index, T* __restrict__ coef)
{
	constexpr int C = 1 << D, K = pow3(D);
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= nnode) { return; }
	const int64_t idx = static_cast<int64_t>(node_key[i]);
	node_index[i]     = idx;
	int     coord[D];
	int64_t v = idx - g.shift;  // = sum coord_d * stride_d over the whole lattice
#pragma unroll
	for (int d = 0; d < D; ++d) {
		if (d + 1 < D) {
			coord[d] = static_cast<int>(v % g.size[d]);
			v /= g.size[d];
		} else {
			coord[d] = static_cast<int>(v);
		}
	}
	T acc[K];
#pragma unroll
	for (int k = 0; k < K; ++k) { acc[k] = T(0); }
#pragma unroll
	for (int ci = 0; ci < C; ++ci) {
		uint64_t key = 0, kstr = 1;
#pragma unroll
		for (int d = 0; d < D; ++d) {
			key += static_cast<uint64_t>(coord[d] - ((ci >> d) & 1) + 1) * kstr;  // cell base in [-1, size - 1]
			kstr *= static_cast<uint64_t>(g.size[d] + 1);
		}
		int64_t lo = 0, hi = nocc;
		while (lo < hi) {
			const int64_t mid = (lo + hi) >> 1;
			if (cell_key[mid] < key) { lo = mid + 1; } else { hi = mid; }
		}
		if (lo >= nocc || cell_key[lo] != key) { continue; }
#pragma unroll
		for (int cj = 0; cj < C; ++cj) {
			bool inside = true;
			int  slot = 0, p3 = 1;
#pragma unroll
			for (int d = 0; d < D; ++d) {
				const int delta = ((cj >> d) & 1) - ((ci >> d) & 1);
				const int n     = coord[d] + delta;
				inside          = inside && (0 <= n) && (n < g.size[d]);
				slot += (delta + 1) * p3;
				p3 *= 3;
			}
			const int a = ci < cj ? ci : cj, b = ci < cj ? cj : ci;
			const int tri = a * C - (a * (a - 1)) / 2 + (b - a);  // row-major upper triangle, as the scatter kernel stores it
			if (inside) { acc[slot] += blocks[static_cast<size_t>(tri) * nocc + lo]; }
		}
	}
#pragma unroll
	for (int k = 0; k < K; ++k) { coef[static_cast<size_t>(k) * nnode + i] = acc[k]; }
}

// u = (P in)[node] for the touched node i of this thread (zero coefficients are never followed: their neighbour may
// lie outside the lattice).
template <typename T, int D>
__device__ __forceinline__ T node_row_dot(const Geom& g, int64_t nnode, int64_t i, int64_t idx, const T* __restrict__ coef, const T* __restrict__ in)
{
	constexpr int K = pow3(D);
	T c[K];
#pragma unroll
	for (int k = 0; k < K; ++k) { c[k] = __ldg(&coef[static_cast<size_t>(k) * nnode + i]); }
	T acc = T(0);
#pragma unroll
	for (int k = 0; k < K; ++k) {
		int64_t off = 0;
		int     r = k;
#pragma unroll
		for (int d = 0; d < D; ++d) {
			off += static_cast<int64_t>(r % 3 - 1) * g.stride[d];
			r /= 3;
		}
		if (c[k] != T(0)) { acc += c[k] * in[idx + off]; }
	}
	return acc;
}

// q += P p over the touched nodes, p.(P p) added to *dot_accum: one thread per node, one writer per element of q.
template <typename T, int D>
__global__ void __launch_bounds__(kThreads) apply_nodes_kernel(Geom g, int64_t nnode, const int64_t* __restrict__ node_index,
                                                               const T* __restrict__ coef, const T* __restrict__ p, T* __restrict__ q,
                                                               double* partial, unsigned* ticket, double* dot_accum, const int* done)
{
	__shared__ double red[32];
	if (done && *done) { return; }
	const int64_t i       = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	double        mine[1] = {0.0};
	if (i < nnode) {
		const int64_t idx = node_index[i];
		const T       u   = node_row_dot<T, D>(g, nnode, i, idx, coef, p);
		q[idx] += u;
		mine[0] = static_cast<double>(p[idx]) * static_cast<double>(u);
	}
	if (dot_accum) {
		mine[0] = block_sum(mine[0], red);
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { *dot_accum += tot[0]; });
	}
}

// Epilogue form for the multigrid smoother: u = P in, res -= u and (d_new given) d_new -= b minv u, e -= b minv u.
template <typename T, int D>
__global__ void __launch_bounds__(kThreads) apply_nodes_epilogue_kernel(Geom g, int64_t nnode, const int64_t* __restrict__ node_index,
                                                                        const T* __restrict__ coef, const T* __restrict__ in, T* __restrict__ res,
                                                                        const T* __restrict__ minv, T* __restrict__ e, T* __restrict__ d_new, T b)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= nnode) { return; }
	const int64_t idx = node_index[i];
	const T       u   = node_row_dot<T, D>(g, nnode, i, idx, coef, in);
	res[idx] -= u;
	if (d_new) {
		const T dd = -b * minv[idx] * u;
		d_new[idx] += dd;
		e[idx] += dd;
	}
}

template <typename T>
__global__ void __launch_bounds__(kThreads) apply_rows_kernel(int64_t nrows, const uint64_t* __restrict__ row_ptr,
                                                              const int32_t* __restrict__ col, const float* __restrict__ val,
                                                              const T* __restrict__ p, T* __restrict__ q, double* partial,
                                                              unsigned* ticket, double* dot_accum, const int* done)
{
	__shared__ double red[32];
	if (done && *done) { return; }
	const int64_t r       = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	double        mine[1] = {0.0};
	if (r < nrows) {
		const uint64_t b = row_ptr[r], e = row_ptr[r + 1];
		T              dot = 0;
		for (uint64_t k = b; k < e; ++k) { dot += static_cast<T>(val[k]) * p[col[k]]; }
		for (uint64_t k = b; k < e; ++k) { atomic_add(&q[col[k]], static_cast<T>(val[k]) * dot); }
		mine[0] = static_cast<double>(dot) * static_cast<double>(dot);
	}
	if (dot_accum) {
		mine[0] = block_sum(mine[0], red);
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { *dot_accum += tot[0]; });
	}
}

// Tile mode of the same: a row a contributes a_i a_j only for columns i, j of one tile, so every entry sums the
// row's terms of its own tile (quadratic in the row length; generic rows are short).
template <typename T>
__global__ void __launch_bounds__(kThreads) apply_rows_tiled_kernel(Geom g, int64_t nrows, const uint64_t* __restrict__ row_ptr,
                                                                    const int32_t* __restrict__ col, const float* __restrict__ val,
                                                                    const T* __restrict__ p, T* __restrict__ q, double* partial,
                                                                    unsigned* ticket, double* dot_accum, const int* done)
{
	__shared__ double red[32];
	if (done && *done) { return; }
	const int64_t r       = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	double        mine[1] = {0.0};
	if (r < nrows) {
		const uint64_t b = row_ptr[r], e = row_ptr[r + 1];
		for (uint64_t k = b; k < e; ++k) {
			const int64_t tk  = tile_of_node(g, col[k]);
			T             dot = 0;
			for (uint64_t j = b; j < e; ++j) {
				if (tile_of_node(g, col[j]) == tk) { dot += static_cast<T>(val[j]) * p[col[j]]; }
			}
			const T add = static_cast<T>(val[k]) * dot;
			atomic_add(&q[col[k]], add);
			mine[0] += static_cast<double>(p[col[k]]) * static_cast<double>(add);
		}
	}
	if (dot_accum) {
		mine[0] = block_sum(mine[0], red);
		grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { *dot_accum += tot[0]; });
	}
}

}  // namespace

// ---- host entry points ------------------------------------------------------------------------------------
void canonicalise_points(const Geom& g, PointStore& st, float value_weight, int value_kernel, float gradient_weight,
                         int gradient_kernel, int64_t n, const float* d_pos, const float* d_nrm, const float* d_pw,
                         const float* d_val, cudaStream_t s)
{
	if (n <= 0) { return; }
	const int64_t at = st.count, tot = st.count + n;
	st.pos.grow_keep(static_cast<size_t>(tot) * g.ndim, s);
	st.grad.grow_keep(static_cast<size_t>(tot) * g.ndim, s);
	st.value.grow_keep(tot, s);
	st.vw.grow_keep(tot, s);
	st.gw.grow_keep(tot, s);
	st.kind.grow_keep(tot, s);
	const int kind = (value_kernel & 1) | ((gradient_kernel & 3) << 1) | (d_nrm ? 8 : 0);
	FI_LAUNCH(canonicalise_kernel, div_up(n, kThreads), kThreads, 0, s, g.ndim, n, at, d_pos, d_nrm, d_pw, d_val,
	          value_weight, gradient_weight, kind, st.pos.data(), st.grad.data(), st.value.data(), st.vw.data(),
	          st.gw.data(), st.kind.data());
	st.count = tot;
}

static void scan_pair(uint64_t* d_rows, uint64_t* d_trips, int64_t n, uint64_t* h_rows, uint64_t* h_trips, cudaStream_t s)
{
	DevBuf<uint64_t> totals(2);
	exclusive_scan_u64(d_rows, d_rows, n, totals.data(), s);
	exclusive_scan_u64(d_trips, d_trips, n, totals.data() + 1, s);
	uint64_t h[2];
	FI_CUDA(cudaMemcpyAsync(h, totals.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	*h_rows  = h[0];
	*h_trips = h[1];
}

void count_point_rows(const Geom& g, PointView pv, int64_t p0, int64_t p1, uint64_t* d_rowoff, uint64_t* d_tripoff,
                      uint64_t* h_rows, uint64_t* h_trips, cudaStream_t s)
{
	const int64_t n = p1 - p0;
	*h_rows = *h_trips = 0;
	if (n <= 0) { return; }
	FI_LAUNCH(point_counts_kernel, div_up(n, kThreads), kThreads, 0, s, g, pv, p0, n, d_rowoff, d_tripoff);
	scan_pair(d_rowoff, d_tripoff, n, h_rows, h_trips, s);
}

void emit_point_rows(const Geom& g, PointView pv, int64_t p0, int64_t p1, const uint64_t* d_rowoff,
                     const uint64_t* d_tripoff, int64_t row_base, int64_t trip_base, fi_triplet* d_trips, float* d_rhs,
                     cudaStream_t s)
{
	const int64_t n = p1 - p0;
	if (n <= 0) { return; }
	FI_LAUNCH(point_emit_kernel, div_up(n, kThreads), kThreads, 0, s, g, pv, p0, n, d_rowoff, d_tripoff, row_base,
	          trip_base, d_trips, d_rhs);
}

void count_model_rows(const Geom& g, const fi_weights& w, uint64_t* d_rowoff, uint64_t* d_tripoff, uint64_t* h_rows,
                      uint64_t* h_trips, cudaStream_t s)
{
	FI_LAUNCH(model_counts_kernel, div_up(g.N, kThreads), kThreads, 0, s, g, w, d_rowoff, d_tripoff);
	scan_pair(d_rowoff, d_tripoff, g.N, h_rows, h_trips, s);
}

void emit_model_rows(const Geom& g, const fi_weights& w, const uint64_t* d_rowoff, const uint64_t* d_tripoff,
                     int64_t row_base, int64_t trip_base, fi_triplet* d_trips, float* d_rhs, cudaStream_t s)
{
	FI_LAUNCH(model_emit_kernel, div_up(g.N, kThreads), kThreads, 0, s, g, w, d_rowoff, d_tripoff, row_base, trip_base,
	          d_trips, d_rhs);
}

void upscale_device(const Geom& small, const Geom& large, const float* d_small, float* d_large, float post_scale,
                    cudaStream_t s)
{
	FI_LAUNCH(upscale_kernel, div_up(large.N, kThreads), kThreads, 0, s, small, large, d_small, d_large, post_scale);
}

static bool node_major_data_term()
{
	static const bool v = [] {
		const char* e = getenv("FI_B200_DATA_TERM");
		return e && e[0] == 'n';
	}();
	return v;
}

// Node-major form of the cell blocks (DataTerm::node_index / node_coef), built once per operator.
template <typename T>
static void build_node_rows(const Geom& g, DataTerm<T>& out, cudaStream_t s)
{
	out.nnode = 0;
	if (out.nocc == 0) { return; }
	const int     C = 1 << g.ndim;
	const int64_t n = out.nocc * C;
	FI_REQUIRE(n < (1ll << 32), FI_ERR_RANGE, "too many occupied cells for the node-major data term");
	DevBuf<uint64_t>           keys(n), flags(n), scan(n), total(1), uniq;
	DevBuf<uint32_t>           vals(n), slot(n);
	DevBuf<unsigned long long> valid(1);
	valid.zero(s);
	const uint64_t sentinel = static_cast<uint64_t>(g.N);
	by_dim(g.ndim, [&](auto dim) {
		auto kern = node_keys_kernel<decltype(dim)::value>;
		FI_LAUNCH(kern, div_up(n, kThreads), kThreads, 0, s, g, out.nocc, out.cell_base.data(), out.cell_mask.data(), sentinel, keys.data(), vals.data(),
		          valid.data());
	});
	int bits = 1;
	while (bits < 63 && (1ull << bits) <= sentinel) { ++bits; }
	radix_sort_pairs(keys, vals, n, bits, s);
	unsigned long long h_valid = 0;
	FI_CUDA(cudaMemcpyAsync(&h_valid, valid.data(), sizeof(h_valid), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	const int64_t V = static_cast<int64_t>(h_valid);
	if (V == 0) { return; }
	FI_LAUNCH(mark_heads_kernel, div_up(V, kThreads), kThreads, 0, s, keys.data(), V, flags.data());
	exclusive_scan_u64(flags.data(), scan.data(), V, total.data(), s);
	uint64_t h_nnode = 0;
	FI_CUDA(cudaMemcpyAsync(&h_nnode, total.data(), sizeof(h_nnode), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	out.nnode = static_cast<int64_t>(h_nnode);
	uniq.resize(out.nnode);
	FI_LAUNCH(slots_kernel, div_up(V, kThreads), kThreads, 0, s, keys.data(), flags.data(), scan.data(), V, slot.data(), uniq.data());
	int K = 1;
	for (int d = 0; d < g.ndim; ++d) { K *= 3; }
	out.node_index.resize(out.nnode);
	out.node_coef.resize(static_cast<size_t>(K) * out.nnode);
	by_dim(g.ndim, [&](auto dim) {
		auto kern = node_rows_kernel<T, decltype(dim)::value>;
		FI_LAUNCH(kern, div_up(out.nnode, kThreads), kThreads, 0, s, g, out.nnode, uniq.data(), out.nocc, out.cell_key.data(), out.blocks.data(),
		          out.node_index.data(), out.node_coef.data());
	});
	FI_CUDA(cudaStreamSynchronize(s));  // the scratch buffers go out of scope
}

template <typename T>
void build_data_term(const Geom& g, const PointStore& pts, const HostRows& user, DataTerm<T>& out, T* d_atb, T* d_diag,
                     cudaStream_t s)
{
	const int64_t   M  = pts.count;
	const PointView pv = view(pts);
	const int       C  = 1 << g.ndim;
	const int       ntri = C * (C + 1) / 2;
	out.nocc  = 0;
	out.nrows = 0;

	if (M > 0) {
		// 1. cell keys, stable sort by cell
		DevBuf<uint64_t>           keys(M);
		DevBuf<uint32_t>           order(M);
		DevBuf<unsigned long long> valid(1);
		valid.zero(s);
		uint64_t key_span = 1;
		for (int d = 0; d < g.ndim; ++d) { key_span *= static_cast<uint64_t>(g.size[d] + 1); }
		FI_LAUNCH(cell_keys_kernel, div_up(M, kThreads), kThreads, 0, s, g, pv, M, key_span, keys.data(), order.data(), valid.data());
		unsigned long long h_valid = 0;
		FI_CUDA(cudaMemcpyAsync(&h_valid, valid.data(), sizeof(h_valid), cudaMemcpyDeviceToHost, s));
		FI_CUDA(cudaStreamSynchronize(s));
		int bits = 1;
		while (bits < 63 && (1ull << bits) <= key_span) { ++bits; }  // keys lie in [0, key_span]
		radix_sort_pairs(keys, order, M, bits, s);

		const int64_t V = static_cast<int64_t>(h_valid);
		if (V > 0) {
			// 2. runs of equal keys -> occupied-cell slots
			DevBuf<uint64_t> flags(V), scan(V), total(1);
			DevBuf<uint32_t> slot(V);
			FI_LAUNCH(mark_heads_kernel, div_up(V, kThreads), kThreads, 0, s, keys.data(), V, flags.data());
			exclusive_scan_u64(flags.data(), scan.data(), V, total.data(), s);
			uint64_t h_nocc = 0;
			FI_CUDA(cudaMemcpyAsync(&h_nocc, total.data(), sizeof(h_nocc), cudaMemcpyDeviceToHost, s));
			FI_CUDA(cudaStreamSynchronize(s));
			out.nocc = static_cast<int64_t>(h_nocc);
			out.cell_key.resize(out.nocc);
			out.blocks.resize(static_cast<size_t>(ntri) * out.nocc);
			out.blocks.zero(s);
			FI_LAUNCH(slots_kernel, div_up(V, kThreads), kThreads, 0, s, keys.data(), flags.data(), scan.data(), V, slot.data(),
			          out.cell_key.data());
			out.cell_base.resize(out.nocc);
			out.cell_mask.resize(out.nocc);
			by_dim(g.ndim, [&](auto dim) {
				auto kern = cell_nodes_kernel<decltype(dim)::value>;
				FI_LAUNCH(kern, div_up(out.nocc, kThreads), kThreads, 0, s, g, out.nocc, out.cell_key.data(), out.cell_base.data(),
				          out.cell_mask.data());
			});
			// 3. warp-segmented scatter
			const int grid = div_up(V, kThreads);
			by_dim(g.ndim, [&](auto dim) {
				auto kern = scatter_points_kernel<T, decltype(dim)::value>;
				FI_LAUNCH(kern, grid, kThreads, 0, s, g, pv, order.data(), slot.data(), V, out.nocc, out.blocks.data(), d_atb, d_diag);
			});
			// 4'. the node-major form, when it was asked for (tile mode keeps using the blocks)
			if (node_major_data_term()) { build_node_rows<T>(g, out, s); }
			FI_CUDA(cudaStreamSynchronize(s));
		}
	}

	// 4. rows outside the cell-block form: linear-interpolation gradient rows, then caller-appended rows
	uint64_t drows = 0, dents = 0;
	DevBuf<uint64_t> rowoff, entoff;
	if (M > 0) {
		rowoff.resize(M);
		entoff.resize(M);
		FI_LAUNCH(derived_counts_kernel, div_up(M, kThreads), kThreads, 0, s, g, pv, M, rowoff.data(), entoff.data());
		scan_pair(rowoff.data(), entoff.data(), M, &drows, &dents, s);
	}
	const uint64_t urows = static_cast<uint64_t>(user.rows()), uents = user.col.size();
	out.nrows = static_cast<int64_t>(drows + urows);
	if (out.nrows > 0) {
		out.row_ptr.resize(out.nrows + 1);
		out.col.resize(dents + uents);
		out.val.resize(dents + uents);
		if (drows > 0) {
			auto kern = derived_emit_kernel<T>;
			FI_LAUNCH(kern, div_up(M, kThreads), kThreads, 0, s, g, pv, M, rowoff.data(), entoff.data(),
			          out.row_ptr.data(), out.col.data(), out.val.data(), d_atb, d_diag);
		}
		if (urows > 0) {
			DevBuf<float> d_rhs(urows);
			FI_CUDA(cudaMemcpyAsync(out.row_ptr.data() + drows, user.ptr.data(), (urows + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
			FI_CUDA(cudaMemcpyAsync(out.col.data() + dents, user.col.data(), uents * sizeof(int32_t), cudaMemcpyHostToDevice, s));
			FI_CUDA(cudaMemcpyAsync(out.val.data() + dents, user.val.data(), uents * sizeof(float), cudaMemcpyHostToDevice, s));
			FI_CUDA(cudaMemcpyAsync(d_rhs.data(), user.rhs.data(), urows * sizeof(float), cudaMemcpyHostToDevice, s));
			if (dents > 0) { FI_LAUNCH(shift_ptr_kernel, div_up(urows + 1, kThreads), kThreads, 0, s, out.row_ptr.data() + drows, static_cast<int64_t>(urows + 1), dents); }
			auto ukern = user_rows_accumulate_kernel<T>;
			FI_LAUNCH(ukern, div_up(urows, kThreads), kThreads, 0, s, static_cast<int64_t>(urows),
			          out.row_ptr.data() + drows, out.col.data(), out.val.data(), d_rhs.data(), d_atb, d_diag);
			FI_CUDA(cudaStreamSynchronize(s));
		} else {
			FI_CUDA(cudaMemcpyAsync(out.row_ptr.data() + drows, &dents, sizeof(uint64_t), cudaMemcpyHostToDevice, s));
			FI_CUDA(cudaStreamSynchronize(s));
		}
	}
	out.partial.resize(static_cast<size_t>(div_up(std::max<int64_t>(std::max(out.nocc, out.nnode), 1), kThreads)) + div_up(std::max<int64_t>(out.nrows, 1), kThreads) + 4);
	out.ticket.resize(2);
	out.ticket.zero(s);
	FI_CUDA(cudaStreamSynchronize(s));
}

// Which kernel applies the cell blocks.  Default: one thread per occupied cell, atomics into q.  Measured on the B200
// (512^3, 1M points = 898k occupied cells, fp32; profiles/r2b_data_term_kernels.md): per cell 0.078 ms, per (cell, row)
// 0.172 ms, node-major gather 0.192 ms.  The node-major form (FI_B200_DATA_TERM=node: no atomics, bit-reproducible) loses
// on scattered clouds because nearly every cell holds one point and touches 8 nodes of its own: 27 coefficients for each
// of ~6 nodes per cell against 36 per cell; it is kept for clouds dense enough to share nodes.
enum DataTermKernel { kDataCell, kDataNode, kDataSplit };
static DataTermKernel data_term_kernel()
{
	static const DataTermKernel v = [] {
		const char* e = getenv("FI_B200_DATA_TERM");
		return !e ? kDataCell : (e[0] == 'n' ? kDataNode : (e[0] == 's' ? kDataSplit : kDataCell));
	}();
	return v;
}

template <typename T>
bool apply_data_term(const Geom& g, const DataTerm<T>& dt, const T* p, T* q, double* d_dot_accum, const int* d_done,
                     cudaStream_t s, const PeerPublish* pub)
{
	bool published = false;
	const int gb = dt.nocc > 0 ? div_up(dt.nocc, kThreads) : 0;
	const int gr = dt.nrows > 0 ? div_up(dt.nrows, kThreads) : 0;
	const int gp = dt.nocc > 0 ? div_up(std::max(dt.nocc, dt.nnode), kThreads) : 0;  // partial sums of the rows kernel start behind the widest block / node grid
	double*   partial = const_cast<double*>(dt.partial.data());
	unsigned* ticket  = const_cast<unsigned*>(dt.ticket.data());
	if (gb > 0) {
		by_dim(g.ndim, [&](auto dim) {
			if (g.tile) {
				auto kern = apply_blocks_kernel<T, decltype(dim)::value, true>;
				FI_LAUNCH(kern, gb, kThreads, 0, s, g, dt.nocc, dt.cell_base.data(), dt.cell_mask.data(), dt.blocks.data(), p, q, partial, ticket,
				          d_dot_accum, d_done, dt.cell_key.data(), PeerPublish(), 0);
			} else if (data_term_kernel() == kDataNode) {
				if (dt.nnode > 0) {
					auto kern = apply_nodes_kernel<T, decltype(dim)::value>;
					FI_LAUNCH(kern, div_up(dt.nnode, kThreads), kThreads, 0, s, g, dt.nnode, dt.node_index.data(), dt.node_coef.data(), p, q, partial, ticket,
					          d_dot_accum, d_done);
				}
			} else if (data_term_kernel() == kDataSplit) {
				auto kern = apply_blocks_split_kernel<T, decltype(dim)::value>;
				FI_LAUNCH(kern, gb, kThreads, 0, s, g, dt.nocc, dt.cell_base.data(), dt.cell_mask.data(), dt.blocks.data(), p, q, partial, ticket,
				          d_dot_accum, d_done);
			} else {
				// the last block to finish may publish the rank's p.Ap itself (only when nothing else adds to it afterwards)
				const bool do_pub = pub != nullptr && d_dot_accum != nullptr && gr == 0;
				auto kern = apply_blocks_kernel<T, decltype(dim)::value, false>;
				FI_LAUNCH(kern, gb, kThreads, 0, s, g, dt.nocc, dt.cell_base.data(), dt.cell_mask.data(), dt.blocks.data(), p, q, partial, ticket,
				          d_dot_accum, d_done, static_cast<const uint64_t*>(nullptr), do_pub ? *pub : PeerPublish(), do_pub ? 1 : 0);
				published = do_pub;
			}
		});
	}
	if (gr > 0 && g.tile) {
		auto kern = apply_rows_tiled_kernel<T>;
		FI_LAUNCH(kern, gr, kThreads, 0, s, g, dt.nrows, dt.row_ptr.data(), dt.col.data(), dt.val.data(), p, q,
		          partial + gp + 1, ticket + 1, d_dot_accum, d_done);
	} else if (gr > 0) {
		auto kern = apply_rows_kernel<T>;
		FI_LAUNCH(kern, gr, kThreads, 0, s, dt.nrows, dt.row_ptr.data(), dt.col.data(), dt.val.data(), p, q,
		          partial + gp + 1, ticket + 1, d_dot_accum, d_done);
	}
	return published;
}

template <typename T>
bool apply_data_term_epilogue(const Geom& g, const DataTerm<T>& dt, const T* in, T* res_out, const T* minv, T* e, T* d_new, T b,
                              cudaStream_t s)
{
	// (a slab applies the rows of the nodes it owns: cell_mask bits 8..15, as in apply_blocks_kernel)
	if (dt.nrows > 0 || g.tile) { return false; }
	if (dt.nocc > 0) {
		by_dim(g.ndim, [&](auto dim) {
			if (data_term_kernel() == kDataNode) {
				if (dt.nnode > 0) {
					auto kern = apply_nodes_epilogue_kernel<T, decltype(dim)::value>;
					FI_LAUNCH(kern, div_up(dt.nnode, kThreads), kThreads, 0, s, g, dt.nnode, dt.node_index.data(), dt.node_coef.data(), in, res_out, minv, e,
					          d_new, b);
				}
			} else {
				auto kern = apply_blocks_epilogue_kernel<T, decltype(dim)::value>;
				FI_LAUNCH(kern, div_up(dt.nocc, kThreads), kThreads, 0, s, g, dt.nocc, dt.cell_base.data(), dt.cell_mask.data(), dt.blocks.data(), in,
				          res_out, minv, e, d_new, b);
			}
		});
	}
	return true;
}

template bool apply_data_term_epilogue<float>(const Geom&, const DataTerm<float>&, const float*, float*, const float*, float*, float*, float,
                                              cudaStream_t);
template void build_data_term<float>(const Geom&, const PointStore&, const HostRows&, DataTerm<float>&, float*, float*, cudaStream_t);
template void build_data_term<double>(const Geom&, const PointStore&, const HostRows&, DataTerm<double>&, double*, double*, cudaStream_t);
template bool apply_data_term<float>(const Geom&, const DataTerm<float>&, const float*, float*, double*, const int*, cudaStream_t, const PeerPublish*);
template bool apply_data_term<double>(const Geom&, const DataTerm<double>&, const double*, double*, double*, const int*, cudaStream_t, const PeerPublish*);

}  // namespace fi

// Point sampling (value and gradient at arbitrary positions) shares this translation unit and its -fmad=false build.
#include "sample_field.cuh"
// So does the error map of a field's own system (bit-identical to generate_error_map on its exported triplets).
#include "field_error_map.cuh"
// So does the exact nearest-point search (bit-identical to the brute-force loop of the reference's SDF caller).
#include "nearest_points.cuh"
