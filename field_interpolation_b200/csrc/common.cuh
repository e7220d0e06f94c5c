// Shared plumbing of libfi_b200: error propagation, device buffers, launch accounting, reductions.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/fi_b200.h"

namespace fi {

constexpr int kMaxDim = 3;  // MAX_DIM, reference field_interpolation.hpp:44

// ---- errors ---------------------------------------------------------------------------------------
struct Error
{
	int         code;
	std::string what;
};

void set_last_error(const std::string& s);

#define FI_CUDA(expr)                                                                                              \
	do {                                                                                                           \
		cudaError_t fi_e_ = (expr);                                                                                \
		if (fi_e_ != cudaSuccess) {                                                                                \
			throw ::fi::Error{FI_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(fi_e_) + " (" + __FILE__ + \
			                                    ":" + std::to_string(__LINE__) + ")"};                           \
		}                                                                                                          \
	} while (0)

#define FI_REQUIRE(cond, code, msg)                        \
	do {                                                   \
		if (!(cond)) { throw ::fi::Error{(code), (msg)}; } \
	} while (0)

// ---- launch accounting (bench.py's gpu_launches) ------------------------------------------------------
extern int64_t g_launches;
inline void count_launch(int n = 1) { g_launches += n; }

// What the last stencil and data-term launches on the host were (FI_PCG_KERNEL_* / FI_PCG_DATA_*, fi_field_pcg_stage
// reports it): the tests that compare one kernel with a reference assert the instantiation they mean to cover.
struct LaunchNote
{
	int stencil = 0, radius = 0, gs = 0, tile_rows = 0, z_chunks = 0, data_term = 0;
};
extern LaunchNote g_note;
inline void note_stencil(int kind, int radius, bool gs, int tile_rows, int z_chunks)
{
	g_note.stencil   = kind;
	g_note.radius    = radius;
	g_note.gs        = gs ? 1 : 0;
	g_note.tile_rows = tile_rows;
	g_note.z_chunks  = z_chunks;
}

#ifndef FI_LAUNCH  // tests/emu/cuda_emu.hpp (the CPU functional emulator of the build container) supplies its own
#define FI_LAUNCH(kernel, grid, block, smem, stream, ...)                 \
	do {                                                                  \
		kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);       \
		::fi::count_launch();                                             \
		FI_CUDA(cudaGetLastError());                                      \
	} while (0)
#endif

// ---- tracing (the reference logs the wall time of each phase with loguru scopes, sparse_linear.cpp:62-198) ----
// FI_B200_TRACE=1 prints one line per phase to stderr.
bool trace_enabled();
struct TraceScope
{
	const char* name;
	double      t0;
	explicit TraceScope(const char* n);
	~TraceScope();
};

// ---- device memory ----------------------------------------------------------------------------------
// Lattice-sized buffers come and go with every field and every solve; cudaMalloc / cudaFree of half-gigabyte
// blocks costs milliseconds each, so freed blocks are kept in a per-process cache (exact-size reuse) and handed
// out again.  A block is reused only after the device has been synchronised since it was released.
void*  pool_alloc(size_t bytes);
void   pool_free(void* p, size_t bytes);
void   pool_trim();             // return every cached block to the driver
size_t pool_cached_bytes();

template <typename T>
class DevBuf
{
public:
	DevBuf() = default;
	explicit DevBuf(size_t n) { resize(n); }
	DevBuf(const DevBuf&)            = delete;
	DevBuf& operator=(const DevBuf&) = delete;
	DevBuf(DevBuf&& o) noexcept { swap(o); }
	DevBuf& operator=(DevBuf&& o) noexcept
	{
		if (this != &o) { release(); swap(o); }
		return *this;
	}
	~DevBuf() { release(); }

	void swap(DevBuf& o) noexcept
	{
		std::swap(p_, o.p_);
		std::swap(n_, o.n_);
		std::swap(cap_, o.cap_);
	}
	void release()
	{
		if (p_) { pool_free(p_, cap_ * sizeof(T)); }
		p_ = nullptr;
		n_ = cap_ = 0;
	}
	// Discards contents when growing.
	void resize(size_t n)
	{
		if (n > cap_) {
			release();
			p_   = static_cast<T*>(pool_alloc(std::max<size_t>(n, 1) * sizeof(T)));
			cap_ = std::max<size_t>(n, 1);
		}
		n_ = n;
	}
	// Keeps contents when growing (amortised doubling).
	void grow_keep(size_t n, cudaStream_t s)
	{
		if (n > cap_) {
			size_t ncap = std::max<size_t>(n, cap_ * 2);
			T*     q    = static_cast<T*>(pool_alloc(ncap * sizeof(T)));
			if (n_) { FI_CUDA(cudaMemcpyAsync(q, p_, n_ * sizeof(T), cudaMemcpyDeviceToDevice, s)); }
			FI_CUDA(cudaStreamSynchronize(s));
			if (p_) { pool_free(p_, cap_ * sizeof(T)); }
			p_   = q;
			cap_ = ncap;
		}
		n_ = n;
	}
	void zero(cudaStream_t s)
	{
		if (n_) { FI_CUDA(cudaMemsetAsync(p_, 0, n_ * sizeof(T), s)); }
	}
	T*       data() { return p_; }
	const T* data() const { return p_; }
	size_t   size() const { return n_; }
	bool     empty() const { return n_ == 0; }

private:
	T*     p_   = nullptr;
	size_t n_   = 0;
	size_t cap_ = 0;
};

// cudaEvent_t that is destroyed when it goes out of scope (also when an exception unwinds past it)
class CudaEvent
{
public:
	CudaEvent() { FI_CUDA(cudaEventCreate(&e_)); }
	CudaEvent(const CudaEvent&)            = delete;
	CudaEvent& operator=(const CudaEvent&) = delete;
	~CudaEvent()
	{
		if (e_) { cudaEventDestroy(e_); }
	}
	operator cudaEvent_t() const { return e_; }
	void record(cudaStream_t s) { FI_CUDA(cudaEventRecord(e_, s)); }
	void sync() { FI_CUDA(cudaEventSynchronize(e_)); }
	// milliseconds from `from` to this event (both recorded and this one complete)
	double ms_since(const CudaEvent& from)
	{
		float ms = 0;
		FI_CUDA(cudaEventElapsedTime(&ms, from.e_, e_));
		return ms;
	}

private:
	cudaEvent_t e_ = nullptr;
};

template <typename T>
class PinnedBuf
{
public:
	PinnedBuf() = default;
	explicit PinnedBuf(size_t n) { resize(n); }
	PinnedBuf(const PinnedBuf&)            = delete;
	PinnedBuf& operator=(const PinnedBuf&) = delete;
	~PinnedBuf()
	{
		if (p_) { cudaFreeHost(p_); }
	}
	void resize(size_t n)
	{
		if (n > cap_) {
			if (p_) { cudaFreeHost(p_); }
			p_ = nullptr;
			FI_CUDA(cudaMallocHost(&p_, std::max<size_t>(n, 1) * sizeof(T)));
			cap_ = n;
		}
		n_ = n;
	}
	T*     data() { return p_; }
	size_t size() const { return n_; }

private:
	T*     p_   = nullptr;
	size_t n_   = 0;
	size_t cap_ = 0;
};

inline int div_up(int64_t a, int64_t b) { return static_cast<int>((a + b - 1) / b); }

int sm_count();  // cached multiprocessor count of the current device (148 on B200)

// ---- device-side reductions --------------------------------------------------------------------------
#if defined(__CUDACC__) || defined(FI_B200_EMU)

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) { v += __shfl_xor_sync(0xffffffffu, v, o); }
	return v;
}

// Sum over the block (any blockDim.x that is a multiple of 32, <= 1024).  Result valid in thread 0.
__device__ __forceinline__ double block_sum(double v, double* smem /* >= 32 doubles */)
{
	v = warp_sum(v);
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	if (lane == 0) { smem[wid] = v; }
	__syncthreads();
	const int nw = (blockDim.x + 31) >> 5;
	double    r  = 0.0;
	if (wid == 0) {
		r = lane < nw ? smem[lane] : 0.0;
		r = warp_sum(r);
	}
	__syncthreads();
	return r;
}

// Deterministic grid-wide sum of up to K values per block: every block stores its partials, the last block
// to arrive (ticket counter) adds them in block order and calls `finish(sums)` from its thread 0.
// partial: [K][gridDim.x] doubles; ticket: one unsigned, zero on entry, reset to zero on exit.
template <int K, typename Finish>
__device__ __forceinline__ void grid_sum(const double (&mine)[K], double* partial, unsigned* ticket, double* smem,
                                         Finish finish)
{
	__shared__ bool last;
	const unsigned  nb = gridDim.x * gridDim.y * gridDim.z;
	const unsigned  b  = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
	if (threadIdx.x == 0) {
#pragma unroll
		for (int k = 0; k < K; ++k) { partial[static_cast<size_t>(k) * nb + b] = mine[k]; }
		__threadfence();
		last = (atomicAdd(ticket, 1u) == nb - 1);
	}
	__syncthreads();
	if (!last) { return; }
	__threadfence();
	double tot[K];
#pragma unroll
	for (int k = 0; k < K; ++k) {
		double acc = 0.0;
		for (unsigned i = threadIdx.x; i < nb; i += blockDim.x) { acc += __ldcg(&partial[static_cast<size_t>(k) * nb + i]); }
		tot[k] = block_sum(acc, smem);
	}
	if (threadIdx.x == 0) {
		*ticket = 0;
		finish(tot);
	}
}

#endif  // __CUDACC__ || FI_B200_EMU

}  // namespace fi
