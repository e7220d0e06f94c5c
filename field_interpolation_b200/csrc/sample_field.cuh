// Point sampling of a lattice field: the value and, optionally, the gradient at arbitrary positions, as the
// reference's constraint rows measure them.  Included at the end of assembly.cu, so it shares that translation unit's
// -fmad=false build (every product and sum rounds on its own, as in the reference's scalar code).  The contract is in
// include/fi_b200.h (fi_sample_field).
//
//   value        upscale_kernel's expression at a given p: in-lattice corners of cell floor(p) in ascending corner
//                order (corner_weights, margin 0), wsum = sum k, fsum = sum k * x, fsum / wsum; NaN where wsum == 0
//   kernel 0     x[cell + s_d] - x[cell], cell = floor(p) entirely inside              field_interpolation.cpp:134-149
//   kernel 1     acc = acc + (+-2 / 2^D) * x[corner] over the cell's corners in order   :150-187
//   kernel 2     corner_weights(p - 0.5, margin 1); acc = acc + (-k) * x[i], acc = acc + k * x[i + s_d] per kept
//                corner (point_emit_kernel's triplet order), then acc / sum k            :188-236
//
// for_corners restates corner_weights for a compile-time D and visits the kept corners instead of compacting them
// into arrays: the same products and sums in the same order, without the per-thread arrays that give upscale_kernel
// a local-memory stack frame.

namespace fi {

namespace {

// Calls f(index, weight) for each corner of cell floor(pos) with 0 <= c and c + margin < size on every axis, in
// ascending corner order, with the weight corner_weights computes for it.
template <int D, typename F>
__device__ __forceinline__ void for_corners(const Geom& g, const float* pos, int margin, F&& f)
{
	int   base[D];
	float frac[D];
#pragma unroll
	for (int d = 0; d < D; ++d) {
		base[d] = floor_to_int(pos[d]);
		frac[d] = pos[d] - static_cast<float>(base[d]);
	}
#pragma unroll
	for (int corner = 0; corner < (1 << D); ++corner) {
		int64_t index = 0;
		float   wt    = 1.0f;
		bool    ok    = true;
#pragma unroll
		for (int d = 0; d < D; ++d) {
			const int bit = (corner >> d) & 1;
			const int c   = base[d] + bit;
			index += g.stride[d] * c;
			wt = wt * (bit ? frac[d] : 1.0f - frac[d]);
			ok = ok && (0 <= c) && (c + margin < g.size[d]);
		}
		if (ok) { f(index, wt); }
	}
}

// GK: -1 (values only), or the fi_gradient_kernel.  One thread per point, grid-stride, caller order.
template <int D, int GK>
__global__ void __launch_bounds__(kThreads) sample_field_kernel(Geom g, int64_t n, const float* __restrict__ pos,
                                                                const float* __restrict__ x, float* __restrict__ values,
                                                                float* __restrict__ gradients)
{
	const float nan    = __int_as_float(0x7fc00000);  // the canonical quiet NaN
	const int64_t step = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += step) {
		float p[D];
		bool  finite = true;  // |p| < 2^31 (NaN fails): floor(p) + 2 fits int32; every point outside is NaN anyway
#pragma unroll
		for (int d = 0; d < D; ++d) {
			p[d]   = pos[i * D + d];
			finite = finite && (fabsf(p[d]) < 2147483648.0f);
		}
		float value = nan;
		float grad[D];
#pragma unroll
		for (int d = 0; d < D; ++d) { grad[d] = nan; }
		if (finite) {
			if (values) {
				float wsum = 0.0f, fsum = 0.0f;
				for_corners<D>(g, p, 0, [&](int64_t idx, float k) {
					wsum = wsum + k;
					fsum = fsum + k * x[idx];
				});
				if (wsum != 0.0f) { value = fsum / wsum; }
			}
			if (GK == 0 || GK == 1) {
				int64_t cell = 0;
				bool    in   = true;
#pragma unroll
				for (int d = 0; d < D; ++d) {
					const int b = floor_to_int(p[d]);
					in          = in && (0 <= b) && (b + 1 < g.size[d]);
					cell += b * g.stride[d];
				}
				if (in && GK == 0) {
#pragma unroll
					for (int d = 0; d < D; ++d) { grad[d] = x[cell + g.stride[d]] - x[cell]; }
				} else if (in) {
					const float term = 2.0f / static_cast<float>(1 << D);
					float       acc[D];
#pragma unroll
					for (int d = 0; d < D; ++d) { acc[d] = 0.0f; }
#pragma unroll
					for (int c = 0; c < (1 << D); ++c) {
						int64_t node = cell;
#pragma unroll
						for (int a = 0; a < D; ++a) { node += ((c >> a) & 1) ? g.stride[a] : 0; }
						const float v = x[node];
#pragma unroll
						for (int d = 0; d < D; ++d) { acc[d] = acc[d] + (((c >> d) & 1) ? term : -term) * v; }
					}
#pragma unroll
					for (int d = 0; d < D; ++d) { grad[d] = acc[d]; }
				}
			} else if (GK == 2) {
				float shifted[D], acc[D];
#pragma unroll
				for (int d = 0; d < D; ++d) {
					shifted[d] = p[d] - 0.5f;
					acc[d]     = 0.0f;
				}
				float ksum = 0.0f;
				for_corners<D>(g, shifted, 1, [&](int64_t idx, float k) {
					ksum          = ksum + k;
					const float v = x[idx];
#pragma unroll
					for (int d = 0; d < D; ++d) {
						acc[d] = acc[d] + (-k) * v;
						acc[d] = acc[d] + k * x[idx + g.stride[d]];
					}
				});
				if (ksum != 0.0f) {  // no kept corner leaves ksum == 0 as well
#pragma unroll
					for (int d = 0; d < D; ++d) { grad[d] = acc[d] / ksum; }
				}
			}
		}
		if (values) { values[i] = value; }
		if (GK >= 0) {
#pragma unroll
			for (int d = 0; d < D; ++d) { gradients[i * D + d] = grad[d]; }
		}
	}
}

template <int D, int GK>
void launch_sample(const Geom& g, int64_t n, const float* pos, const float* x, float* values, float* gradients, cudaStream_t s)
{
	// one thread per point; the grid-stride loop only takes over past the largest grid
	const int grid = static_cast<int>(std::min<int64_t>((n + kThreads - 1) / kThreads, 0x7fffffff));
	FI_LAUNCH((sample_field_kernel<D, GK>), grid, kThreads, 0, s, g, n, pos, x, values, gradients);
}

template <int D>
void sample_dim(const Geom& g, int64_t n, const float* pos, const float* x, int gk, float* values, float* gradients, cudaStream_t s)
{
	switch (gradients ? gk : -1) {
		case 0: launch_sample<D, 0>(g, n, pos, x, values, gradients, s); break;
		case 1: launch_sample<D, 1>(g, n, pos, x, values, gradients, s); break;
		case 2: launch_sample<D, 2>(g, n, pos, x, values, gradients, s); break;
		default: launch_sample<D, -1>(g, n, pos, x, values, nullptr, s); break;
	}
}

}  // namespace

void sample_field_device(const Geom& g, int64_t n, const float* d_positions, const float* d_field, int gradient_kernel,
                         float* d_values, float* d_gradients, cudaStream_t s)
{
	if (n == 0 || (!d_values && !d_gradients)) { return; }
	by_dim(g.ndim, [&](auto dim) { sample_dim<decltype(dim)::value>(g, n, d_positions, d_field, gradient_kernel, d_values, d_gradients, s); });
}

}  // namespace fi
