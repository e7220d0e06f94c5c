// generate_error_map (reference field_interpolation.cpp:402-429) of a field's own system, computed from what the field
// holds instead of from its triplet list.  Included at the end of assembly.cu, so it shares that translation unit's
// -fmad=false build and its row emitters.  The contract is in include/fi_b200.h (fi_field_error_map).
//
// The reference adds out[col] += (v * v) / sq[row] * err[row]^2 over the triplets in global order.  The rows of every
// builder call are contiguous and the calls come in order, so taking the segments one after the other, each adding its
// terms to heat[col] in its own triplet order, adds every column's terms in the reference's order:
//
//   model rows   no triplets: one thread per node walks a host-built table of the rows that can reach it, sorted by
//                (tap offset descending = anchor ascending, axis, row type).  model_emit_kernel emits rows anchored
//                at node j in that (axis, type) order, so this is the node's triplet order.  Each row's err and sq are
//                recomputed from the taps in order (coefficients binom[k][m] * w_k or +-1 * w_gs, rhs 0 * w).
//   point rows   emitted in chunks of at most error_map_chunk_triplets() triplets by emit_point_rows itself; one thread per row
//                forms err, sq and one term per triplet; a stable radix sort of (column, triplet index) groups the
//                terms by column in triplet order; one thread per run of equal columns adds them to heat in order.
//   caller rows  the CSR of HostRows, staged in chunks, then the same row / sort / run steps.
//
// Row error sums (fp64 err^2 per row, split model / point / caller rows) are reduced per block and the block partials
// added in block order, so they repeat bit for bit from run to run.

#include <algorithm>
#include <cstdlib>

namespace fi {

namespace {

// Up to 69 entries in 3D: per axis d, taps m = 0..k of every order k (15), and 4 taps of each of the D - 1
// gradient-smoothness rows across o.
constexpr int kMaxModelTaps = 69;

struct ModelTable
{
	int   n;
	int   entry[kMaxModelTaps];  // d | type << 2 | tap << 6; type 0..4: order k, 5 + o: gradient smoothness across o
	float coef[kMaxDim + 5][5];  // row coefficients by type: [k][m] = binom[k][m] * w_k; [5 + o] = -gs, +gs, +gs, -gs
	float rhs[kMaxDim + 5];      // 0.0f * w, as model_emit_kernel writes it
};

// Displacement along axis a of the node that holds tap `tap` of row (d, type) from the row's anchor.
__host__ __device__ __forceinline__ int tap_disp(int a, int d, int type, int tap)
{
	if (type < 5) { return a == d ? tap : 0; }
	return (a == d ? (tap & 1) : 0) + (a == type - 5 ? (tap >> 1) : 0);
}

// One thread per node: heat[i] += the node's model terms, in the segment's triplet order.  Adds the fp64 err^2 of the
// rows anchored at the node (tap 0) to the block partial.  Both parameters are __grid_constant__: the table is indexed
// at run time, and a by-value copy would put it (and the Geom) in a local-memory stack frame.
template <int D>
__global__ void __launch_bounds__(kThreads) model_error_kernel(const __grid_constant__ Geom g, const __grid_constant__ ModelTable tab,
                                                               const float* __restrict__ x, float* __restrict__ heat, double* __restrict__ partial)
{
	__shared__ double red[32];
	const int64_t i    = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	double        mine = 0.0;
	if (i < g.N) {
		int     c[D];
		int64_t rest = i;
#pragma unroll
		for (int a = 0; a < D; ++a) {
			c[a] = static_cast<int>(rest % g.size[a]);
			rest /= g.size[a];
		}
		float h = heat[i];
		for (int e = 0; e < tab.n; ++e) {
			const int ent = tab.entry[e];
			const int d = ent & 3, type = (ent >> 2) & 15, tap = ent >> 6;
			// anchor of the row: inside the lattice, and the row exists there (model_counts_kernel's tests)
			bool    ok = true;
			int64_t j = i, sd = 0, so = 0;
#pragma unroll
			for (int a = 0; a < D; ++a) {
				const int disp = tap_disp(a, d, type, tap);
				const int ext  = (a == d ? (type < 5 ? type : 1) : 0) + (a == type - 5 ? 1 : 0);
				const int anc  = c[a] - disp;
				ok             = ok && anc >= 0 && anc + ext < g.size[a];
				j -= disp * g.stride[a];
				if (a == d) { sd = g.stride[a]; }
				if (a == type - 5) { so = g.stride[a]; }
			}
			if (!ok) { continue; }
			float err = tab.rhs[type], sq = 0.0f;
			if (type < 5) {
				for (int m = 0; m <= type; ++m) {
					const float v = tab.coef[type][m];
					err           = err - x[j + m * sd] * v;
					sq            = sq + v * v;
				}
			} else {
				const float gs0 = tab.coef[type][0], gs1 = tab.coef[type][1], gs2 = tab.coef[type][2], gs3 = tab.coef[type][3];
				err = err - x[j] * gs0;
				sq  = sq + gs0 * gs0;
				err = err - x[j + sd] * gs1;
				sq  = sq + gs1 * gs1;
				err = err - x[j + so] * gs2;
				sq  = sq + gs2 * gs2;
				err = err - x[j + so + sd] * gs3;
				sq  = sq + gs3 * gs3;
			}
			if (tap == 0) { mine += static_cast<double>(err) * static_cast<double>(err); }
			err = err * err;
			if (sq != 0.0f) {
				const float v = tab.coef[type][tap];
				h             = h + (v * v) / sq * err;
			}
		}
		heat[i] = h;
	}
	mine = block_sum(mine, red);
	if (threadIdx.x == 0) { partial[blockIdx.x] = mine; }
}

// Row boundaries of a chunk of emitted point rows (every emitted row has at least one triplet).
__global__ void row_starts_kernel(int64_t nt, const fi_triplet* __restrict__ t, int64_t nrows, uint64_t* __restrict__ row_ptr)
{
	const int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (k >= nt) { return; }
	if (k == 0 || t[k].row != t[k - 1].row) { row_ptr[t[k].row] = static_cast<uint64_t>(k); }
	if (k == 0) { row_ptr[nrows] = static_cast<uint64_t>(nt); }
}

struct TripletRows  // emitted point rows
{
	const fi_triplet* t;
	__device__ int32_t col(uint64_t k) const { return t[k].col; }
	__device__ float   val(uint64_t k) const { return t[k].value; }
};

struct CsrRows  // staged caller rows
{
	const int32_t* c;
	const float*   v;
	__device__ int32_t col(uint64_t k) const { return c[k]; }
	__device__ float   val(uint64_t k) const { return v[k]; }
};

// One thread per row: err = rhs - sum x[col] * v and sq = sum v * v in triplet order, then one term per triplet
// ((v * v) / sq * err^2, or -0.0f where sq == 0: adding -0.0f leaves every value as it is) and its sort key (the
// column) and value (the triplet index).  row_ptr is relative to the chunk's first triplet.
template <typename Rows>
__global__ void __launch_bounds__(kThreads) row_terms_kernel(int64_t nrows, const uint64_t* __restrict__ row_ptr, uint64_t ptr0, Rows rows,
                                                             const float* __restrict__ rhs, const float* __restrict__ x,
                                                             float* __restrict__ term, uint64_t* __restrict__ key,
                                                             uint32_t* __restrict__ idx, double* __restrict__ partial)
{
	__shared__ double red[32];
	const int64_t r    = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	double        mine = 0.0;
	if (r < nrows) {
		const uint64_t b = row_ptr[r] - ptr0, e = row_ptr[r + 1] - ptr0;
		float          err = rhs[r], sq = 0.0f;
		for (uint64_t k = b; k < e; ++k) {
			const float v = rows.val(k);
			err           = err - x[rows.col(k)] * v;
			sq            = sq + v * v;
		}
		mine = static_cast<double>(err) * static_cast<double>(err);
		err  = err * err;
		for (uint64_t k = b; k < e; ++k) {
			const float v = rows.val(k);
			term[k]       = sq != 0.0f ? (v * v) / sq * err : -0.0f;
			key[k]        = static_cast<uint64_t>(rows.col(k));
			idx[k]        = static_cast<uint32_t>(k);
		}
	}
	mine = block_sum(mine, red);
	if (threadIdx.x == 0) { partial[blockIdx.x] = mine; }
}

// After the stable sort by column: the first thread of every run of equal columns adds the run's terms to heat in
// triplet order.
__global__ void run_sum_kernel(int64_t nt, const uint64_t* __restrict__ key, const uint32_t* __restrict__ idx, const float* __restrict__ term,
                               float* __restrict__ heat)
{
	const int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
	if (k >= nt || (k > 0 && key[k] == key[k - 1])) { return; }
	const uint64_t col = key[k];
	float          h   = heat[col];
	for (int64_t j = k; j < nt && key[j] == col; ++j) { h = h + term[idx[j]]; }
	heat[col] = h;
}

// *sum += the block partials, added in a fixed order.
__global__ void add_partials_kernel(const double* __restrict__ partial, int64_t nb, double* sum)
{
	__shared__ double red[32];
	double            acc = 0.0;
	for (int64_t b = threadIdx.x; b < nb; b += blockDim.x) { acc += partial[b]; }
	acc = block_sum(acc, red);
	if (threadIdx.x == 0) { *sum += acc; }
}

ModelTable model_table(const Geom& g, const fi_weights& w)
{
	static const float binom[5][5] = {{1, 0, 0, 0, 0}, {-1, 1, 0, 0, 0}, {1, -2, 1, 0, 0}, {1, -3, 3, -1, 0}, {1, -4, 6, -4, 1}};
	const float        wk[5]       = {w.model_0, w.model_1, w.model_2, w.model_3, w.model_4};
	ModelTable         t{};
	for (int k = 0; k <= 4; ++k) {
		for (int m = 0; m <= k; ++m) { t.coef[k][m] = binom[k][m] * wk[k]; }
		t.rhs[k] = 0.0f * wk[k];
	}
	const float gs = w.gradient_smoothness;
	for (int o = 0; o < kMaxDim; ++o) {
		t.coef[5 + o][0] = -1.0f * gs;
		t.coef[5 + o][1] = +1.0f * gs;
		t.coef[5 + o][2] = +1.0f * gs;
		t.coef[5 + o][3] = -1.0f * gs;
		t.rhs[5 + o]     = 0.0f * gs;
	}
	struct Tap
	{
		int64_t off;
		int     d, type, tap;
	};
	std::vector<Tap> taps;
	auto add = [&](int d, int type, int tap) {
		int64_t off = 0;
		for (int a = 0; a < g.ndim; ++a) { off += tap_disp(a, d, type, tap) * g.stride[a]; }
		taps.push_back(Tap{off, d, type, tap});
	};
	for (int d = 0; d < g.ndim; ++d) {
		for (int k = 0; k <= 4; ++k) {
			if (!(wk[k] > 0)) { continue; }
			for (int m = 0; m <= k; ++m) { add(d, k, m); }
		}
		if (gs > 0) {
			for (int o = 0; o < g.ndim; ++o) {
				if (o == d) { continue; }
				for (int tap = 0; tap < 4; ++tap) { add(d, 5 + o, tap); }
			}
		}
	}
	// a node meets its rows in ascending anchor order (= descending offset), then in emission order at the anchor
	std::sort(taps.begin(), taps.end(), [](const Tap& a, const Tap& b) {
		if (a.off != b.off) { return a.off > b.off; }
		if (a.d != b.d) { return a.d < b.d; }
		return a.type < b.type;
	});
	t.n = static_cast<int>(taps.size());
	for (int e = 0; e < t.n; ++e) { t.entry[e] = taps[e].d | (taps[e].type << 2) | (taps[e].tap << 6); }
	return t;
}

void add_partials(const DevBuf<double>& partial, int64_t nb, double* d_sum, cudaStream_t s)
{
	FI_LAUNCH(add_partials_kernel, 1, kThreads, 0, s, partial.data(), nb, d_sum);
}

// The row / sort / run steps of one chunk of rows whose triplets sit in [0, nt) of `rows`.
template <typename Rows>
void rows_to_heat(ErrorMapScratch& sc, int64_t nrows, const uint64_t* d_row_ptr, uint64_t ptr0, Rows rows, int64_t nt, const float* d_rhs,
                  const Geom& g, const float* d_x, float* d_heat, double* d_sum, cudaStream_t s)
{
	if (nrows <= 0) { return; }
	const int64_t nb = div_up(nrows, kThreads);
	sc.partial.resize(nb);
	sc.term.resize(std::max<int64_t>(nt, 1));
	sc.key.resize(std::max<int64_t>(nt, 1));
	sc.idx.resize(std::max<int64_t>(nt, 1));
	auto kern = row_terms_kernel<Rows>;
	FI_LAUNCH(kern, nb, kThreads, 0, s, nrows, d_row_ptr, ptr0, rows, d_rhs, d_x, sc.term.data(), sc.key.data(), sc.idx.data(), sc.partial.data());
	add_partials(sc.partial, nb, d_sum, s);
	if (nt == 0) { return; }
	int bits = 1;
	while (bits < 63 && (1ull << bits) < static_cast<uint64_t>(g.N)) { ++bits; }
	radix_sort_pairs(sc.key, sc.idx, nt, bits, s);
	FI_LAUNCH(run_sum_kernel, div_up(nt, kThreads), kThreads, 0, s, nt, sc.key.data(), sc.idx.data(), sc.term.data(), d_heat);
}

}  // namespace

int64_t error_map_chunk_triplets()
{
	const char*     e = getenv("FI_B200_ERROR_MAP_CHUNK");
	const long long n = e ? atoll(e) : 0;
	return n > 0 ? static_cast<int64_t>(n) : (int64_t{1} << 26);
}

void model_error_map(const Geom& g, const fi_weights& w, const float* d_x, float* d_heat, double* d_sum, ErrorMapScratch& sc, cudaStream_t s)
{
	const ModelTable tab = model_table(g, w);
	if (tab.n == 0) { return; }
	const int64_t nb = div_up(g.N, kThreads);
	sc.partial.resize(nb);
	by_dim(g.ndim, [&](auto dim) {
		auto kern = model_error_kernel<decltype(dim)::value>;
		FI_LAUNCH(kern, nb, kThreads, 0, s, g, tab, d_x, d_heat, sc.partial.data());
	});
	add_partials(sc.partial, nb, d_sum, s);
}

void point_error_map(const Geom& g, PointView pv, int64_t p0, int64_t p1, const float* d_x, float* d_heat, double* d_sum, ErrorMapScratch& sc,
                     cudaStream_t s)
{
	// the most triplets one point emits: a linear value row and D linear-interpolation gradient rows
	const int64_t per_point = (int64_t{1} << g.ndim) + 2 * g.ndim * (int64_t{1} << g.ndim);
	const int64_t step      = std::max<int64_t>(1, error_map_chunk_triplets() / per_point);
	for (int64_t a = p0; a < p1; a += step) {
		const int64_t b = std::min(p1, a + step), n = b - a;
		sc.rowoff.resize(n);
		sc.tripoff.resize(n);
		uint64_t hr = 0, ht = 0;
		count_point_rows(g, pv, a, b, sc.rowoff.data(), sc.tripoff.data(), &hr, &ht, s);
		if (hr == 0) { continue; }
		sc.trips.resize(ht);
		sc.rhs.resize(hr);
		sc.row_ptr.resize(hr + 1);
		emit_point_rows(g, pv, a, b, sc.rowoff.data(), sc.tripoff.data(), 0, 0, sc.trips.data(), sc.rhs.data(), s);
		FI_LAUNCH(row_starts_kernel, div_up(ht, kThreads), kThreads, 0, s, static_cast<int64_t>(ht), sc.trips.data(), static_cast<int64_t>(hr),
		          sc.row_ptr.data());
		rows_to_heat(sc, static_cast<int64_t>(hr), sc.row_ptr.data(), 0, TripletRows{sc.trips.data()}, static_cast<int64_t>(ht), sc.rhs.data(), g,
		             d_x, d_heat, d_sum, s);
	}
	FI_CUDA(cudaStreamSynchronize(s));
}

void caller_rows_error_map(const Geom& g, const HostRows& R, int64_t r0, int64_t r1, const float* d_x, float* d_heat, double* d_sum,
                           ErrorMapScratch& sc, cudaStream_t s)
{
	const uint64_t cap = static_cast<uint64_t>(error_map_chunk_triplets());
	for (int64_t a = r0; a < r1;) {
		// as many rows as fit the chunk (at least one)
		int64_t b = a + 1;
		while (b < r1 && R.ptr[b + 1] - R.ptr[a] <= cap) { ++b; }
		const uint64_t t0 = R.ptr[a], nt = R.ptr[b] - t0;
		const int64_t  nr = b - a;
		sc.row_ptr.resize(nr + 1);
		sc.col.resize(std::max<uint64_t>(nt, 1));
		sc.val.resize(std::max<uint64_t>(nt, 1));
		sc.rhs.resize(nr);
		FI_CUDA(cudaMemcpyAsync(sc.row_ptr.data(), R.ptr.data() + a, (nr + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
		if (nt > 0) {
			FI_CUDA(cudaMemcpyAsync(sc.col.data(), R.col.data() + t0, nt * sizeof(int32_t), cudaMemcpyHostToDevice, s));
			FI_CUDA(cudaMemcpyAsync(sc.val.data(), R.val.data() + t0, nt * sizeof(float), cudaMemcpyHostToDevice, s));
		}
		FI_CUDA(cudaMemcpyAsync(sc.rhs.data(), R.rhs.data() + a, nr * sizeof(float), cudaMemcpyHostToDevice, s));
		rows_to_heat(sc, nr, sc.row_ptr.data(), t0, CsrRows{sc.col.data(), sc.val.data()}, static_cast<int64_t>(nt), sc.rhs.data(), g, d_x, d_heat,
		             d_sum, s);
		FI_CUDA(cudaStreamSynchronize(s));  // the staged chunk is overwritten next
		a = b;
	}
}

}  // namespace fi
