// Exact nearest-point search: for each query, the fp32 distance to the nearest point of a cloud and that point's
// index, bit-identical to the brute-force loop of the reference's SDF caller (src/sdf_field.cpp:212-249).  Included
// at the end of assembly.cu, so it shares that translation unit's -fmad=false build: every product and sum of the
// distance rounds on its own, as in the loop.  The contract is in include/fi_b200.h (fi_nearest_point_distance);
// DESIGN.md §3g has the exactness argument.
//
// Each call builds its structure from the cloud and frees it:
//   bounds    the fp32 bounding box of the finite points and their count (points with a non-finite coordinate never
//             win the loop, so dropping them changes nothing)
//   keys      a 30-bit Morton key of each finite point quantised over that box (non-finite points get key 2^30 and
//             sort last), stable radix sort of (key, index)
//   leaves    32 consecutive sorted points per leaf (struct of arrays) with their exact fp32 box
//   levels    8 consecutive boxes of a level per box of the next, up to one root: an implicit tree over the Morton
//             order, 6 levels at 1M points
// One thread per query walks the tree nearest child first with a stack of (lower bound, level, node).  A box is
// skipped only when a lower bound on the fp32 d2 of every point inside it is strictly greater than the best d2 so far;
// a tested point replaces the best on d2 < best, or on d2 == best at a lower index.  So the result is the loop's
// first minimum whatever order the leaves are visited in.
//
// The queries come from a caller array or from an enumeration of the border nodes of a lattice (ascending linear
// index), which is never materialised.

#include <algorithm>
#include <cmath>

namespace fi {

namespace {

constexpr int kNpLeaf      = 32;  // points per leaf
constexpr int kNpFan       = 8;   // boxes of a level per box of the next
constexpr int kNpMaxLevels = 10;  // < 2^32 points: < 2^27 leaves and at most 9 levels above them
// Popping a box of level l leaves at most kNpFan - 1 entries of each level in [l, top); its children add kNpFan.
constexpr int kNpStack   = kNpFan + (kNpFan - 1) * (kNpMaxLevels - 2);
constexpr int kNpKeyBits = 30;  // Morton key bits; 2^30 marks a non-finite point
constexpr float kNpMaxFloat = 3.40282347e38f;

struct NpBox
{
	float lo[kMaxDim], hi[kMaxDim];  // axes >= D hold 0
};

struct NpCloud  // the search structure, passed to the query kernel as a __grid_constant__ parameter
{
	const float*    p[kMaxDim];  // finite points in Morton order, one array per axis
	const uint32_t* idx;         // their input indices
	int64_t         m;           // number of finite points
	const NpBox*    box;         // every level's boxes, leaves first
	int64_t         off[kNpMaxLevels];
	int64_t         cnt[kNpMaxLevels];
	int             top;  // level of the root
};

// Border nodes of a lattice in ascending linear index.  full[d] = nodes of the sub-lattice of axes < d; bc[d] = its
// border nodes (a node is on the border when some coordinate is 0 or size - 1).
struct NpBorder
{
	int     ndim;
	int     size[kMaxDim];
	int64_t stride[kMaxDim];
	int64_t full[kMaxDim + 1], bc[kMaxDim + 1];

	__host__ __device__ int64_t count() const { return bc[ndim]; }
	// Linear index of border node number b (0 <= b < count()).  Walking down from the slowest axis: slices 0 and
	// n - 1 along an axis are all border nodes (in linear order), an interior slice holds the border nodes of the
	// sub-lattice below it.  Axes of 1 or 2 nodes have no interior slice.
	__host__ __device__ int64_t node(int64_t b) const
	{
		int64_t index = 0;
		for (int d = ndim - 1; d >= 0; --d) {
			const int n = size[d];
			if (n <= 2 || b < full[d]) { return index + b; }
			b -= full[d];
			const int64_t inner = static_cast<int64_t>(n - 2) * bc[d];
			if (b < inner) {
				index += (1 + b / bc[d]) * stride[d];
				b %= bc[d];
				continue;
			}
			return index + static_cast<int64_t>(n - 1) * stride[d] + (b - inner);
		}
		return index;
	}
};

NpBorder np_border(const Geom& g)
{
	NpBorder e{};
	e.ndim    = g.ndim;
	e.full[0] = 1;
	e.bc[0]   = 0;
	for (int d = 0; d < g.ndim; ++d) {
		e.size[d]     = g.size[d];
		e.stride[d]   = g.stride[d];
		e.full[d + 1] = e.full[d] * g.size[d];
		e.bc[d + 1]   = g.size[d] <= 2 ? e.full[d + 1] : 2 * e.full[d] + static_cast<int64_t>(g.size[d] - 2) * e.bc[d];
	}
	return e;
}

template <int D>
struct NpArrayQueries
{
	const float* q;
	__device__ void get(int64_t i, float (&out)[D]) const
	{
#pragma unroll
		for (int d = 0; d < D; ++d) { out[d] = q[i * D + d]; }
	}
};

template <int D>
struct NpBorderQueries
{
	NpBorder e;
	__device__ void get(int64_t i, float (&out)[D]) const
	{
		const int64_t node = e.node(i);
#pragma unroll
		for (int d = 0; d < D; ++d) { out[d] = static_cast<float>(static_cast<int>((node / e.stride[d]) % e.size[d])); }
	}
};

// float <-> unsigned with the order of the floats (for atomicMin / atomicMax)
__device__ __forceinline__ unsigned long long np_ordered(float v)
{
	const uint32_t u = static_cast<uint32_t>(__float_as_int(v));
	return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
float np_unordered(unsigned long long o)
{
	uint32_t u = static_cast<uint32_t>(o);
	u          = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
	float f;
	std::memcpy(&f, &u, 4);
	return f;
}

__device__ __forceinline__ bool np_finite(float v) { return fabsf(v) <= kNpMaxFloat; }

__host__ __device__ __forceinline__ int64_t np_min(int64_t a, int64_t b) { return a < b ? a : b; }

// acc[0..D) = min, acc[3..3+D) = max (ordered) of the finite points, acc[6] += their count.
template <int D>
__global__ void __launch_bounds__(kThreads) np_bounds_kernel(int64_t n, const float* __restrict__ pts, unsigned long long* __restrict__ acc)
{
	unsigned long long lo[D], hi[D], cnt = 0;
#pragma unroll
	for (int d = 0; d < D; ++d) {
		lo[d] = 0xffffffffull;
		hi[d] = 0;
	}
	const int64_t step = static_cast<int64_t>(gridDim.x) * blockDim.x;
	for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += step) {
		float p[D];
		bool  fin = true;
#pragma unroll
		for (int d = 0; d < D; ++d) {
			p[d] = pts[i * D + d];
			fin  = fin && np_finite(p[d]);
		}
		if (!fin) { continue; }
		++cnt;
#pragma unroll
		for (int d = 0; d < D; ++d) {
			const unsigned long long o = np_ordered(p[d]);
			lo[d]                      = o < lo[d] ? o : lo[d];
			hi[d]                      = o > hi[d] ? o : hi[d];
		}
	}
#pragma unroll
	for (int s = 16; s > 0; s >>= 1) {
		cnt += __shfl_xor_sync(0xffffffffu, cnt, s);
#pragma unroll
		for (int d = 0; d < D; ++d) {
			const unsigned long long a = __shfl_xor_sync(0xffffffffu, lo[d], s), b = __shfl_xor_sync(0xffffffffu, hi[d], s);
			lo[d]                      = a < lo[d] ? a : lo[d];
			hi[d]                      = b > hi[d] ? b : hi[d];
		}
	}
	if ((threadIdx.x & 31) == 0 && cnt > 0) {
#pragma unroll
		for (int d = 0; d < D; ++d) {
			atomicMin(&acc[d], lo[d]);
			atomicMax(&acc[3 + d], hi[d]);
		}
		atomicAdd(&acc[6], cnt);
	}
}

__device__ __forceinline__ uint32_t np_spread2(uint32_t x)  // 15 bits -> even bits
{
	x &= 0x7fffu;
	x = (x | (x << 8)) & 0x00ff00ffu;
	x = (x | (x << 4)) & 0x0f0f0f0fu;
	x = (x | (x << 2)) & 0x33333333u;
	x = (x | (x << 1)) & 0x55555555u;
	return x;
}

__device__ __forceinline__ uint32_t np_spread3(uint32_t x)  // 10 bits -> every third bit
{
	x &= 0x3ffu;
	x = (x | (x << 16)) & 0x030000ffu;
	x = (x | (x << 8)) & 0x0300f00fu;
	x = (x | (x << 4)) & 0x030c30c3u;
	x = (x | (x << 2)) & 0x09249249u;
	return x;
}

// Morton key of every point over the box [lo, lo + (2^bits - 1) / scale]; 2^30 for a point with a non-finite coordinate.
template <int D>
__global__ void __launch_bounds__(kThreads) np_keys_kernel(int64_t n, const float* __restrict__ pts, NpBox bb, double sx, double sy, double sz,
                                                           uint64_t* __restrict__ keys, uint32_t* __restrict__ vals)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= n) { return; }
	constexpr int    bits  = kNpKeyBits / D;
	constexpr double maxq  = static_cast<double>((1u << bits) - 1u);
	const double     sc[3] = {sx, sy, sz};
	uint32_t         q[D];
	bool             fin = true;
#pragma unroll
	for (int d = 0; d < D; ++d) {
		const float  v = pts[i * D + d];
		const double t = (static_cast<double>(v) - static_cast<double>(bb.lo[d])) * sc[d];
		fin            = fin && np_finite(v);
		q[d]           = fin ? static_cast<uint32_t>(t < 0.0 ? 0.0 : (t > maxq ? maxq : t)) : 0u;
	}
	uint64_t key;
	if (D == 1) {
		key = q[0];
	} else if (D == 2) {
		key = np_spread2(q[0]) | (np_spread2(q[D > 1 ? 1 : 0]) << 1);
	} else {
		key = np_spread3(q[0]) | (np_spread3(q[D > 1 ? 1 : 0]) << 1) | (np_spread3(q[D > 2 ? 2 : 0]) << 2);
	}
	keys[i] = fin ? key : (uint64_t{1} << kNpKeyBits);
	vals[i] = static_cast<uint32_t>(i);
}

template <int D>
__global__ void __launch_bounds__(kThreads) np_gather_kernel(int64_t m, const float* __restrict__ pts, const uint32_t* __restrict__ order, float* __restrict__ px,
                                                             float* __restrict__ py, float* __restrict__ pz, uint32_t* __restrict__ idx)
{
	const int64_t j = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (j >= m) { return; }
	const int64_t i = order[j];
	px[j]           = pts[i * D];
	if (D > 1) { py[j] = pts[i * D + 1]; }
	if (D > 2) { pz[j] = pts[i * D + 2]; }
	idx[j] = static_cast<uint32_t>(i);
}

template <int D>
__global__ void __launch_bounds__(kThreads) np_leaf_boxes_kernel(int64_t m, int64_t nleaves, const float* __restrict__ px, const float* __restrict__ py,
                                                                 const float* __restrict__ pz, NpBox* __restrict__ box)
{
	const int64_t l = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (l >= nleaves) { return; }
	const float* p[3] = {px, py, pz};
	NpBox        b{};
	const int64_t k0 = l * kNpLeaf, k1 = np_min(k0 + kNpLeaf, m);
#pragma unroll
	for (int d = 0; d < D; ++d) {
		float lo = p[d][k0], hi = lo;
		for (int64_t k = k0 + 1; k < k1; ++k) {
			lo = fminf(lo, p[d][k]);
			hi = fmaxf(hi, p[d][k]);
		}
		b.lo[d] = lo;
		b.hi[d] = hi;
	}
	box[l] = b;
}

// Box j of a level = the union of boxes [kNpFan j, kNpFan j + kNpFan) of the level below (src, nsrc of them).
__global__ void __launch_bounds__(kThreads) np_parent_boxes_kernel(const NpBox* __restrict__ src, int64_t nsrc, NpBox* __restrict__ dst, int64_t ndst)
{
	const int64_t j = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (j >= ndst) { return; }
	const int64_t c0 = j * kNpFan, c1 = np_min(c0 + kNpFan, nsrc);
	NpBox         b  = src[c0];
	for (int64_t c = c0 + 1; c < c1; ++c) {
		const NpBox& o = src[c];
#pragma unroll
		for (int d = 0; d < kMaxDim; ++d) {
			b.lo[d] = fminf(b.lo[d], o.lo[d]);
			b.hi[d] = fmaxf(b.hi[d], o.hi[d]);
		}
	}
	dst[j] = b;
}

// A lower bound on the fp32 d2 of every point in the box, in fp64: the real squared distance from q to the box,
// shrunk by the relative slack of the fp32 expression's roundings and by an absolute slack for its underflow
// (DESIGN.md §3g).
template <int D>
__device__ __forceinline__ double np_box_bound(const NpBox& b, const float (&q)[D])
{
	double s = 0.0;
#pragma unroll
	for (int d = 0; d < D; ++d) {
		const double x = q[d], lo = b.lo[d], hi = b.hi[d];
		const double gap = lo > x ? lo - x : (x > hi ? x - hi : 0.0);
		s                = s + gap * gap;
	}
	return s * (1.0 - 0x1p-20) - 0x1p-140;
}

// The largest float <= v (0 for v <= 0): stack entries carry their bound as a float that never exceeds it.
__device__ __forceinline__ float np_float_down(double v)
{
	if (!(v > 0.0)) { return 0.0f; }
	float f = static_cast<float>(v);
	if (static_cast<double>(f) > v) { f = nextafterf(f, 0.0f); }
	return f;
}

template <int D>
__device__ __forceinline__ float np_d2(const NpCloud& c, int64_t k, const float (&q)[D])
{
	const float dx = c.p[0][k] - q[0];
	float       d2 = dx * dx;
	if (D > 1) {
		const float dy = c.p[1][k] - q[D > 1 ? 1 : 0];
		d2             = d2 + dy * dy;
	}
	if (D > 2) {
		const float dz = c.p[2][k] - q[D > 2 ? 2 : 0];
		d2             = d2 + dz * dz;
	}
	return d2;
}

// One thread per query: distance (nullable) and nearest index (nullable; -1 where the distance is +inf).
template <int D, typename Src>
__global__ void __launch_bounds__(kThreads) np_query_kernel(const __grid_constant__ NpCloud c, const __grid_constant__ Src src, int64_t nq,
                                                            float* __restrict__ dist, int64_t* __restrict__ nearest)
{
	const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (i >= nq) { return; }
	float q[D];
	src.get(i, q);
	bool fin = true;
#pragma unroll
	for (int d = 0; d < D; ++d) { fin = fin && np_finite(q[d]); }
	const float inf  = __int_as_float(0x7f800000);
	float       best = inf;
	uint32_t    bi   = 0xffffffffu;
	if (fin && c.m > 0) {  // a non-finite query makes every d2 NaN or +inf: nothing wins
		uint64_t stack[kNpStack];
		int      sp  = 0;
		stack[sp++] = static_cast<uint64_t>(c.top) << 28;  // the root, bound 0
		while (sp > 0) {
			const uint64_t e = stack[--sp];
			if (__int_as_float(static_cast<int>(e >> 32)) > best) { continue; }
			const int     level = static_cast<int>((e >> 28) & 15u);
			const int64_t node  = static_cast<int64_t>(e & 0x0fffffffu);
			if (level == 0) {
				const int64_t k1 = np_min((node + 1) * kNpLeaf, c.m);
				for (int64_t k = node * kNpLeaf; k < k1; ++k) {
					const float    d2 = np_d2<D>(c, k, q);
					const uint32_t id = c.idx[k];
					if (d2 < best || (d2 == best && id < bi)) {
						best = d2;
						bi   = id;
					}
				}
				continue;
			}
			const int64_t c0 = node * kNpFan, nc = c.cnt[level - 1];
			const NpBox*  bx = c.box + c.off[level - 1];
			uint64_t      key[kNpFan];
#pragma unroll
			for (int j = 0; j < kNpFan; ++j) {
				key[j] = ~uint64_t{0};
				if (c0 + j < nc) {
					const double lb = np_box_bound<D>(bx[c0 + j], q);
					if (!(lb > static_cast<double>(best))) {
						key[j] = (static_cast<uint64_t>(static_cast<uint32_t>(__float_as_int(np_float_down(lb)))) << 32) |
						         (static_cast<uint64_t>(level - 1) << 28) | static_cast<uint64_t>(c0 + j);
					}
				}
			}
#pragma unroll
			for (int a = 1; a < kNpFan; ++a) {
#pragma unroll
				for (int b = a; b > 0; --b) {
					const uint64_t x = key[b - 1], y = key[b];
					key[b - 1]       = x < y ? x : y;
					key[b]           = x < y ? y : x;
				}
			}
#pragma unroll
			for (int j = kNpFan - 1; j >= 0; --j) {  // nearest on top
				if (key[j] != ~uint64_t{0}) { stack[sp++] = key[j]; }
			}
		}
	}
#ifdef FI_B200_EMU
	if (dist) { dist[i] = std::sqrt(best); }
#else
	if (dist) { dist[i] = __fsqrt_rn(best); }
#endif
	if (nearest) { nearest[i] = best == inf ? -1 : static_cast<int64_t>(bi); }
}

// The search structure of a cloud; its buffers live as long as the object.
struct NpTree
{
	DevBuf<float>    px, py, pz;
	DevBuf<uint32_t> idx;
	DevBuf<NpBox>    box;
	NpCloud          c{};

	template <int D>
	void build(int64_t n, const float* d_pts, cudaStream_t s)
	{
		c.m = 0;
		if (n == 0) { return; }
		unsigned long long h[7] = {0xffffffffull, 0xffffffffull, 0xffffffffull, 0, 0, 0, 0};
		DevBuf<unsigned long long> acc(7);
		FI_CUDA(cudaMemcpyAsync(acc.data(), h, sizeof(h), cudaMemcpyHostToDevice, s));
		const int grid = static_cast<int>(std::min<int64_t>(div_up(n, kThreads), 1024));
		FI_LAUNCH(np_bounds_kernel<D>, grid, kThreads, 0, s, n, d_pts, acc.data());
		FI_CUDA(cudaMemcpyAsync(h, acc.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
		FI_CUDA(cudaStreamSynchronize(s));
		const int64_t m = static_cast<int64_t>(h[6]);
		if (m == 0) { return; }
		NpBox  bb{};
		double sc[3] = {0, 0, 0};
		for (int d = 0; d < D; ++d) {
			bb.lo[d]         = np_unordered(h[d]);
			bb.hi[d]         = np_unordered(h[3 + d]);
			const double ext = static_cast<double>(bb.hi[d]) - static_cast<double>(bb.lo[d]);
			sc[d]            = ext > 0 ? static_cast<double>((1u << (kNpKeyBits / D)) - 1u) / ext : 0.0;
		}
		DevBuf<uint64_t> keys(n);
		DevBuf<uint32_t> order(n);
		FI_LAUNCH(np_keys_kernel<D>, div_up(n, kThreads), kThreads, 0, s, n, d_pts, bb, sc[0], sc[1], sc[2], keys.data(), order.data());
		radix_sort_pairs(keys, order, n, kNpKeyBits + 1, s);  // finite points first, stable
		px.resize(m);
		py.resize(D > 1 ? m : 0);
		pz.resize(D > 2 ? m : 0);
		idx.resize(m);
		FI_LAUNCH(np_gather_kernel<D>, div_up(m, kThreads), kThreads, 0, s, m, d_pts, order.data(), px.data(), py.data(), pz.data(), idx.data());
		int64_t total = 0;
		c.cnt[0]      = (m + kNpLeaf - 1) / kNpLeaf;
		c.top         = 0;
		while (c.cnt[c.top] > 1) {
			c.cnt[c.top + 1] = (c.cnt[c.top] + kNpFan - 1) / kNpFan;
			++c.top;
		}
		FI_REQUIRE(c.top < kNpMaxLevels, FI_ERR_RANGE, "nearest points: cloud too large");
		for (int l = 0; l <= c.top; ++l) {
			c.off[l] = total;
			total += c.cnt[l];
		}
		box.resize(total);
		FI_LAUNCH(np_leaf_boxes_kernel<D>, div_up(c.cnt[0], kThreads), kThreads, 0, s, m, c.cnt[0], px.data(), py.data(), pz.data(), box.data());
		for (int l = 1; l <= c.top; ++l) {
			FI_LAUNCH(np_parent_boxes_kernel, div_up(c.cnt[l], kThreads), kThreads, 0, s, box.data() + c.off[l - 1], c.cnt[l - 1],
			          box.data() + c.off[l], c.cnt[l]);
		}
		c.p[0] = px.data();
		c.p[1] = D > 1 ? py.data() : px.data();
		c.p[2] = D > 2 ? pz.data() : px.data();
		c.idx  = idx.data();
		c.box  = box.data();
		c.m    = m;
		FI_CUDA(cudaStreamSynchronize(s));  // the sort's scratch (keys, order) is released on return
	}
};

}  // namespace

void nearest_points_device(int ndim, int64_t n_points, const float* d_points, int64_t n_queries, const float* d_queries, float* d_dist,
                           int64_t* d_nearest, cudaStream_t s)
{
	if (n_queries == 0 || (!d_dist && !d_nearest)) { return; }
	by_dim(ndim, [&](auto dim) {
		constexpr int D = decltype(dim)::value;
		NpTree        t;
		t.build<D>(n_points, d_points, s);
		FI_LAUNCH((np_query_kernel<D, NpArrayQueries<D>>), div_up(n_queries, kThreads), kThreads, 0, s, t.c, NpArrayQueries<D>{d_queries}, n_queries,
		          d_dist, d_nearest);
		FI_CUDA(cudaStreamSynchronize(s));
	});
}

void append_border_rows(const Geom& g, float weight, int64_t n_points, const float* d_points, HostRows& rows, cudaStream_t s)
{
	const NpBorder e  = np_border(g);
	const int64_t  nb = e.count();
	DevBuf<float>  d(nb);
	by_dim(g.ndim, [&](auto dim) {
		constexpr int D = decltype(dim)::value;
		NpTree        t;
		t.build<D>(n_points, d_points, s);
		FI_LAUNCH((np_query_kernel<D, NpBorderQueries<D>>), div_up(nb, kThreads), kThreads, 0, s, t.c, NpBorderQueries<D>{e}, nb, d.data(),
		          static_cast<int64_t*>(nullptr));
	});
	std::vector<float> dist(static_cast<size_t>(nb));
	FI_CUDA(cudaMemcpyAsync(dist.data(), d.data(), nb * sizeof(float), cudaMemcpyDeviceToHost, s));
	FI_CUDA(cudaStreamSynchronize(s));
	// add_equation(weight, {distance}, {{node, 1.0f}}) per node (reference sparse_linear.cpp:34-50, host/sparse_linear.cpp:40-51)
	const float v = 1.0f * weight;
	rows.col.reserve(rows.col.size() + static_cast<size_t>(nb));
	rows.val.reserve(rows.val.size() + static_cast<size_t>(nb));
	rows.ptr.reserve(rows.ptr.size() + static_cast<size_t>(nb));
	rows.rhs.reserve(rows.rhs.size() + static_cast<size_t>(nb));
	for (int64_t b = 0; b < nb; ++b) {
		rows.col.push_back(static_cast<int32_t>(e.node(b)));
		rows.val.push_back(v);
		rows.ptr.push_back(rows.col.size());
		rows.rhs.push_back(dist[static_cast<size_t>(b)] * weight);
	}
}

}  // namespace fi
