// common.cuh -- shared host/device helpers of libdbindex_gpu.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdio>
#include <string>

#include "../../include/dbindex_gpu.h"

namespace dbi {

// ---- error plumbing --------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_kernel_launches;

struct CudaError {
  cudaError_t e;
  const char* what;
  const char* file;
  int line;
};

#define DBI_CUDA(call)                                                      \
  do {                                                                      \
    cudaError_t _e = (call);                                                \
    if (_e != cudaSuccess) throw ::dbi::CudaError{_e, #call, __FILE__, __LINE__}; \
  } while (0)

// Every kernel launch goes through this so that dbi_kernel_launches() is exact.
#define DBI_LAUNCH(kernel, grid, block, smem, stream, ...)                  \
  do {                                                                      \
    kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);             \
    ::dbi::g_kernel_launches.fetch_add(1, std::memory_order_relaxed);       \
    DBI_CUDA(cudaGetLastError());                                           \
  } while (0)

// ---- device constants ------------------------------------------------------
constexpr int kWarp = 32;
constexpr int kNumSMsB200 = 148;

// residue class flags (one byte per residue code)
constexpr uint8_t kFlagEnzyme = 1;
constexpr uint8_t kFlagNocut = 2;
constexpr uint8_t kFlagDiffMod = 4;
constexpr uint8_t kFlagMandatory = 8;  // sparam.getMandatoryInternalAAs()
constexpr uint8_t kFlagFilterAA = 16;  // PeptideFilterByMaxOccurrencies.aa

// error bits raised by kernels (OR-ed into a device word)
constexpr uint32_t kErrZeroResidue = 1;   // residue byte 0 in the input
constexpr uint32_t kErrPepTooLong = 2;    // window longer than DBI_MAX_PEP_LEN
constexpr uint32_t kErrModPos = 4;        // modified residue beyond DBI_MAX_MOD_POS
constexpr uint32_t kErrHashCollision = 8; // equal (mass, hash) but different sequence
constexpr uint32_t kErrMergeCap = 16;     // a tile of the group merge over its shared-memory capacity

#ifdef __CUDACC__

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// Warp inclusive scan (shuffle up), any arithmetic type.
template <typename T>
__device__ __forceinline__ T warp_inclusive_sum(T v) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    T n = __shfl_up_sync(0xffffffffu, v, o);
    if ((int)lane_id() >= o) v += n;
  }
  return v;
}

// Block-wide exclusive sum for blockDim.x = THREADS (multiple of 32, <= 1024).
// `warp_sums` is THREADS/32 + 1 elements of shared memory.  Returns the exclusive
// prefix of v; *total receives the block total.  Ends with a __syncthreads() so
// the scratch can be reused immediately.
template <typename T, int THREADS>
__device__ __forceinline__ T block_exclusive_sum(T v, T* warp_sums, T* total) {
  constexpr int W = THREADS / 32;
  const int w = threadIdx.x >> 5;
  T inc = warp_inclusive_sum(v);
  if (lane_id() == 31) warp_sums[w] = inc;
  __syncthreads();
  if (w == 0) {
    T s = (lane_id() < W) ? warp_sums[lane_id()] : T(0);
    T si = warp_inclusive_sum(s);
    if (lane_id() < W) warp_sums[lane_id()] = si - s;  // exclusive warp offsets
    if (lane_id() == W - 1) warp_sums[W] = si;         // block total
  }
  __syncthreads();
  T res = warp_sums[w] + inc - v;
  *total = warp_sums[W];
  __syncthreads();
  return res;
}

// Unaligned-safe byte fetch from the residue buffer through the read-only path.
__device__ __forceinline__ uint8_t ld_res(const uint8_t* __restrict__ res, uint32_t pos) {
  return __ldg(res + pos);
}

#endif  // __CUDACC__

}  // namespace dbi
