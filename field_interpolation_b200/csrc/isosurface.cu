// The step right after the solve in the reference's callers (SURVEY.md §8f rank 4): the zero contour of the solved 2D
// field and its enclosed area, optionally on a bicubically upsampled copy of the field —
//   emilib::marching_squares / emilib::calc_area   third_party/emilib/emilib/marching_squares.cpp:11-150
//   bicubic_upsample / iso_surface                 src/sdf_field.cpp:555-614 (called at :665-670, :701)
// done on the device so that a solved field never has to travel to the host just to be contoured.
//
// Compiled with -fmad=false: every kernel restates the reference's scalar fp32 expressions in the reference's
// order, so the segment list (order included) and the upsampled field are bit-identical to the reference's.
//
// marching squares = count -> scan -> emit over the (width-1) x (height-1) cells in the reference's visiting order
// (y-major, marching_squares.cpp:15-16): a block owns 1024 consecutive cells (4 per thread, consecutive, so a thread's
// own segments stay in order), the per-block counts are scanned on the device, and the emit pass repeats the cheap
// classification, scans inside the block and stores each segment as one float4.  Nothing lattice-sized is written
// besides the segments themselves.  All HBM/L2-bound byte work: 4 B read per cell per pass, 16 B written per segment.
#include "internal.hpp"

namespace fi {

namespace {

constexpr int kMsThreads = 256;
constexpr int kMsItems   = 4;
constexpr int kMsTile    = kMsThreads * kMsItems;

// Segments per cell configuration; config = br<<3 | bl<<2 | tr<<1 | tl with bit = (value >= 0), marching_squares.cpp:21-28.
__device__ __forceinline__ int segments_of(int config)
{
	// 0b0110 and 0b1001 (saddles) emit two segments (:96-115), 0 and 15 none (:28), the rest one
	return (config == 0 || config == 15) ? 0 : ((config == 6 || config == 9) ? 2 : 1);
}

struct Corners
{
	float tl, tr, bl, br;
	int   config;
};

// Cell c of the (width-1)-wide cell grid; values are shifted by -iso first (iso_surface, src/sdf_field.cpp:609-611).
__device__ __forceinline__ Corners load_cell(const float* __restrict__ v, unsigned width, unsigned cw, unsigned c, float iso, unsigned* x, unsigned* y)
{
	const unsigned cy = c / cw, cx = c - cy * cw;
	const size_t   i  = static_cast<size_t>(cy) * width + cx;
	Corners k;
	k.tl     = v[i] - iso;
	k.tr     = v[i + 1] - iso;
	k.bl     = v[i + width] - iso;
	k.br     = v[i + width + 1] - iso;
	k.config = (k.br >= 0.0f ? 8 : 0) | (k.bl >= 0.0f ? 4 : 0) | (k.tr >= 0.0f ? 2 : 0) | (k.tl >= 0.0f ? 1 : 0);
	*x       = cx;
	*y       = cy;
	return k;
}

__global__ void __launch_bounds__(kMsThreads) ms_count_kernel(const float* __restrict__ v, unsigned width, unsigned cw, unsigned ncells, float iso,
                                                              uint64_t* __restrict__ block_count)
{
	__shared__ int warp_tot[kMsThreads / 32];
	const unsigned first = blockIdx.x * kMsTile + threadIdx.x * kMsItems;
	int            mine  = 0;
#pragma unroll
	for (int k = 0; k < kMsItems; ++k) {
		const unsigned c = first + k;
		if (c < ncells) {
			unsigned x, y;
			mine += segments_of(load_cell(v, width, cw, c, iso, &x, &y).config);
		}
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) { mine += __shfl_xor_sync(0xffffffffu, mine, o); }
	if ((threadIdx.x & 31) == 0) { warp_tot[threadIdx.x >> 5] = mine; }
	__syncthreads();
	if (threadIdx.x == 0) {
		int tot = 0;
#pragma unroll
		for (int w = 0; w < kMsThreads / 32; ++w) { tot += warp_tot[w]; }
		block_count[blockIdx.x] = static_cast<uint64_t>(tot);
	}
}

// The crossing points of a cell, marching_squares.cpp:31-34, and the directed segments of each case, :36-129.
// Edge codes: 0 = left (x, y + y_left), 1 = top (x + x_top, y), 2 = right (x + 1, y + y_right), 3 = bottom (x + x_bottom, y + 1).
__device__ __forceinline__ float2 edge_point(const Corners& k, float fx, float fy, int e)
{
	switch (e) {
		case 0: return make_float2(fx + 0.0f, fy + k.tl / (k.tl - k.bl));
		case 1: return make_float2(fx + k.tl / (k.tl - k.tr), fy + 0.0f);
		case 2: return make_float2(fx + 1.0f, fy + k.tr / (k.tr - k.br));
		default: return make_float2(fx + k.bl / (k.bl - k.br), fy + 1.0f);
	}
}

__global__ void __launch_bounds__(kMsThreads) ms_emit_kernel(const float* __restrict__ v, unsigned width, unsigned cw, unsigned ncells, float iso,
                                                             const uint64_t* __restrict__ block_off, float4* __restrict__ lines)
{
	// (from, to) edge codes packed 2 bits each: first segment in bits 0-3, second (saddles only) in bits 4-7
	//           cfg:   0     1     2     3     4     5     6     7     8     9    10    11    12    13    14   15
	// first:          --   L>T   T>R   L>R   B>L   B>T   T>L   B>R   R>B   L>T   T>B   L>B   R>L   R>T   T>L   --
	// second:                                            B>R               R>B
	constexpr unsigned kFrom1 = 0u | (0u << 2) | (1u << 4) | (0u << 6) | (3u << 8) | (3u << 10) | (1u << 12) | (3u << 14) | (2u << 16) | (0u << 18) |
	                            (1u << 20) | (0u << 22) | (2u << 24) | (2u << 26) | (1u << 28);
	constexpr unsigned kTo1 = 0u | (1u << 2) | (2u << 4) | (2u << 6) | (0u << 8) | (1u << 10) | (0u << 12) | (2u << 14) | (3u << 16) | (1u << 18) |
	                          (3u << 20) | (3u << 22) | (0u << 24) | (1u << 26) | (0u << 28);
	__shared__ int warp_tot[kMsThreads / 32];
	const unsigned first = blockIdx.x * kMsTile + threadIdx.x * kMsItems;
	Corners        cell[kMsItems];
	unsigned       cx[kMsItems], cy[kMsItems];
	int            mine = 0;
#pragma unroll
	for (int k = 0; k < kMsItems; ++k) {
		const unsigned c = first + k;
		cell[k].config   = 0;
		if (c < ncells) {
			cell[k] = load_cell(v, width, cw, c, iso, &cx[k], &cy[k]);
			mine += segments_of(cell[k].config);
		}
	}
	// exclusive scan of `mine` over the block (warp shuffles, then the warp totals)
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	int       incl = mine;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		const int up = __shfl_up_sync(0xffffffffu, incl, o);
		if (lane >= o) { incl += up; }
	}
	if (lane == 31) { warp_tot[wid] = incl; }
	__syncthreads();
	int before = 0;
#pragma unroll
	for (int w = 0; w < kMsThreads / 32; ++w) {
		if (w < wid) { before += warp_tot[w]; }
	}
	uint64_t at = block_off[blockIdx.x] + static_cast<uint64_t>(before + incl - mine);
#pragma unroll
	for (int k = 0; k < kMsItems; ++k) {
		const int cfg = cell[k].config;
		const int ns  = segments_of(cfg);
		if (ns == 0) { continue; }
		const float  fx = static_cast<float>(cx[k]), fy = static_cast<float>(cy[k]);
		const float2 a = edge_point(cell[k], fx, fy, (kFrom1 >> (2 * cfg)) & 3), b = edge_point(cell[k], fx, fy, (kTo1 >> (2 * cfg)) & 3);
		lines[at++] = make_float4(a.x, a.y, b.x, b.y);
		if (ns == 2) {  // 0b0110: bottom -> right; 0b1001: right -> bottom (:96-115)
			const float2 c2 = edge_point(cell[k], fx, fy, cfg == 6 ? 3 : 2), d2 = edge_point(cell[k], fx, fy, cfg == 6 ? 2 : 3);
			lines[at++]     = make_float4(c2.x, c2.y, d2.x, d2.y);
		}
	}
}

// calc_area, marching_squares.cpp:136-150: sum over segments of p0x*p1y - p1x*p0y in double (each product of two floats
// is exact in double, so every term equals the reference's); the terms are added in a fixed tree order instead of
// sequentially, which can differ from the reference's double sum in its last bits — invisible after the cast to float
// except at a rounding boundary.
__global__ void __launch_bounds__(256) area_kernel(int64_t nseg, const float4* __restrict__ lines, double* partial, unsigned* ticket, double* out)
{
	__shared__ double red[32];
	double            acc    = 0.0;
	const int64_t     stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < nseg; i += stride) {
		const float4 s = lines[i];
		acc += static_cast<double>(s.x) * static_cast<double>(s.w) - static_cast<double>(s.z) * static_cast<double>(s.y);
	}
	const double mine[1] = {block_sum(acc, red)};
	grid_sum<1>(mine, partial, ticket, red, [&](const double(&tot)[1]) { out[0] = tot[0]; });
}

// emath::catmull_rom, third_party/emath/emath/math.hpp:308-316, in the reference's evaluation order (the integer literals
// there are converted to float; products associate left to right).
__device__ __forceinline__ float catmull_rom(float t, float p0, float p1, float p2, float p3)
{
	const float a = p0 * t * ((2.0f - t) * t - 1.0f);
	const float b = p1 * (t * t * (3.0f * t - 5.0f) + 2.0f);
	const float c = p2 * t * ((4.0f - 3.0f * t) * t + 1.0f);
	const float d = p3 * (t - 1.0f) * t * t;
	return 0.5f * (a + b + c + d);
}

// bicubic_upsample, src/sdf_field.cpp:555-603: one thread per large-lattice sample, clamped 4 x 4 neighbourhood (:565-570),
// Catmull-Rom along x for the four rows, then along y (:587-594).  Reads hit L1/L2 (the small field is read ~upsample^2
// times); the 4 B/sample store is the HBM traffic.
__global__ void __launch_bounds__(256) bicubic_kernel(int width, int height, const float* __restrict__ v, int upsample, int lw, int lh,
                                                      float* __restrict__ out)
{
	const int lx = blockIdx.x * blockDim.x + threadIdx.x, ly = blockIdx.y * blockDim.y + threadIdx.y;
	if (lx >= lw || ly >= lh) { return; }
	const float tx = static_cast<float>(lx % upsample) / static_cast<float>(upsample);
	const float ty = static_cast<float>(ly % upsample) / static_cast<float>(upsample);
	const int   sx = lx / upsample, sy = ly / upsample;
	int         xs[4];
#pragma unroll
	for (int i = 0; i < 4; ++i) { xs[i] = min(max(sx - 1 + i, 0), width - 1); }
	float row[4];
#pragma unroll
	for (int j = 0; j < 4; ++j) {
		const float* r = v + static_cast<size_t>(min(max(sy - 1 + j, 0), height - 1)) * width;
		row[j]         = catmull_rom(tx, r[xs[0]], r[xs[1]], r[xs[2]], r[xs[3]]);
	}
	out[static_cast<size_t>(ly) * lw + lx] = catmull_rom(ty, row[0], row[1], row[2], row[3]);
}

}  // namespace

// Segments of the contour `values == iso` in the reference's order.  d_values: width * height floats on the device.
// d_lines == nullptr: count only.  Returns the number of segments; when d_lines is given it must hold `capacity`
// segments (4 floats each, 16-byte aligned) and nothing is written if the count exceeds it.
int64_t marching_squares_device(int width, int height, const float* d_values, float iso, float* d_lines, int64_t capacity, cudaStream_t s)
{
	if (width < 2 || height < 2) { return 0; }
	const int64_t ncells64 = static_cast<int64_t>(width - 1) * (height - 1);
	FI_REQUIRE(ncells64 < (int64_t{1} << 31), FI_ERR_RANGE, "marching squares: more than 2^31 cells");
	FI_REQUIRE((reinterpret_cast<uintptr_t>(d_lines) & 15u) == 0, FI_ERR_INVALID, "marching squares: the segment buffer must be 16-byte aligned");
	const unsigned   ncells = static_cast<unsigned>(ncells64), cw = static_cast<unsigned>(width - 1);
	const int        nblocks = div_up(ncells64, kMsTile);
	DevBuf<uint64_t> counts(nblocks), total(1);
	FI_LAUNCH(ms_count_kernel, nblocks, kMsThreads, 0, s, d_values, static_cast<unsigned>(width), cw, ncells, iso, counts.data());
	exclusive_scan_u64(counts.data(), counts.data(), nblocks, total.data(), s);
	uint64_t h_total = 0;
	FI_CUDA(cudaMemcpyAsync(&h_total, total.data(), sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	const int64_t nseg = static_cast<int64_t>(h_total);
	if (d_lines && nseg > 0 && nseg <= capacity) {
		FI_LAUNCH(ms_emit_kernel, nblocks, kMsThreads, 0, s, d_values, static_cast<unsigned>(width), cw, ncells, iso, counts.data(),
		          reinterpret_cast<float4*>(d_lines));
		FI_CUDA(cudaStreamSynchronize(s));  // `counts` dies here
	}
	return nseg;
}

// Twice the signed area enclosed by the segments (device, 4 floats each), as the double the reference halves and casts.
double area_twice_device(int64_t nseg, const float* d_lines, cudaStream_t s)
{
	if (nseg <= 0) { return 0.0; }
	FI_REQUIRE((reinterpret_cast<uintptr_t>(d_lines) & 15u) == 0, FI_ERR_INVALID, "calc_area: the segment buffer must be 16-byte aligned");
	const int        grid = static_cast<int>(std::min<int64_t>(div_up(nseg, 256), 4 * sm_count()));
	DevBuf<double>   partial(grid), out(1);
	DevBuf<unsigned> ticket(1);
	ticket.zero(s);
	FI_LAUNCH(area_kernel, grid, 256, 0, s, nseg, reinterpret_cast<const float4*>(d_lines), partial.data(), ticket.data(), out.data());
	double h = 0.0;
	FI_CUDA(cudaMemcpyAsync(&h, out.data(), sizeof(double), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	return h;
}

void bicubic_upsample_device(int width, int height, const float* d_values, int upsample, float* d_large, cudaStream_t s)
{
	const int64_t lw = static_cast<int64_t>(upsample) * width - upsample + 1, lh = static_cast<int64_t>(upsample) * height - upsample + 1;
	FI_REQUIRE(lw < (int64_t{1} << 31) && lh < (int64_t{1} << 31) && div_up(lh, 8) <= 65535, FI_ERR_RANGE, "bicubic_upsample: upsampled lattice too large");
	const dim3 block(32, 8), grid(div_up(lw, 32), div_up(lh, 8));
	FI_LAUNCH(bicubic_kernel, grid, block, 0, s, width, height, d_values, upsample, static_cast<int>(lw), static_cast<int>(lh), d_large);
}

}  // namespace fi

// The 3D counterpart, marching cubes, shares this translation unit and its -fmad=false build.
#include "marching_cubes.cuh"
