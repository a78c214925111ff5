// Shared helpers for libjvae_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>

#include "../../include/jvae_b200.h"

namespace jvae {

// ---------------------------------------------------------------- error plumbing
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define JVAE_CHECK_ARG(cond, msg)                                                   \
  do {                                                                              \
    if (!(cond)) {                                                                  \
      jvae::set_error("%s: invalid argument: %s (%s)", __func__, msg, #cond);       \
      return JVAE_ERR_INVALID;                                                      \
    }                                                                               \
  } while (0)

#define JVAE_CUDA(call)                                                             \
  do {                                                                              \
    cudaError_t _e = (call);                                                        \
    if (_e != cudaSuccess) {                                                        \
      jvae::set_error("%s: %s failed: %s", __func__, #call, cudaGetErrorString(_e));\
      return JVAE_ERR_CUDA;                                                         \
    }                                                                               \
  } while (0)

#define JVAE_LAUNCH_CHECK()                                                         \
  do {                                                                              \
    cudaError_t _e = cudaGetLastError();                                            \
    if (_e != cudaSuccess) {                                                        \
      jvae::set_error("%s: kernel launch failed: %s", __func__, cudaGetErrorString(_e)); \
      return JVAE_ERR_CUDA;                                                         \
    }                                                                               \
    jvae::count_launch();                                                           \
  } while (0)

int sm_count();   // SMs of the current device (cached)

// per-launch profile (runtime.cu): events recorded inside the library right around a kernel launch when enabled
void* prof_begin(int tag, cudaStream_t st);
void prof_end(void* h, cudaStream_t st);

// ---------------------------------------------------------------- small device utilities
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide sum; `red` is >= 32 floats of shared memory; result valid in all threads
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}

__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

// streaming 16-byte load that does not pollute L1
__device__ __forceinline__ uint4 ld_stream16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream16(void* p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ---------------------------------------------------------------- counter-based random numbers
__device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) { return __umulhi(a, b); }

// Philox4x32-10 (Salmon et al., SC'11), counter c[4], key k[2]
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(M0, c.x), lo0 = M0 * c.x;
    const uint32_t hi1 = mulhi32(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}

// Dropout keep-mask of the dense layers (jvae_gemm_bf16_dropout forward, jvae_act_dropout_bwd backward): element (row, col)
// of the call at stream position `offset` is kept iff word (col & 3) of
//     philox4x32_10(counter = (col >> 2, row, offset_lo, offset_hi), key = (seed_lo, seed_hi))
// is >= drop_thresh = floor(p * 2^32) (a 64-bit threshold: p == 1 gives 2^32, which drops everything).  The mask depends
// on nothing but (seed, offset, row, col): not on tile shapes, leading dimensions or which kernel regenerates it.
// dropout_keep4 returns the keep bits of the four columns col4 .. col4 + 3 (col4 a multiple of 4) in bits 0..3.
__device__ __forceinline__ uint32_t dropout_keep4(uint64_t seed, uint64_t offset, uint32_t row, uint32_t col4,
                                                  uint64_t drop_thresh) {
  const uint4 r = philox4x32_10(make_uint4(col4 >> 2, row, (uint32_t)offset, (uint32_t)(offset >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  return (uint32_t)(r.x >= drop_thresh) | ((uint32_t)(r.y >= drop_thresh) << 1) | ((uint32_t)(r.z >= drop_thresh) << 2) |
         ((uint32_t)(r.w >= drop_thresh) << 3);
}
// drop_thresh of a dropout probability p in [0, 1]
inline uint64_t dropout_threshold(float p) { return (uint64_t)floor((double)p * 4294967296.0); }
__device__ __forceinline__ bool dropout_keep(uint64_t seed, uint64_t offset, uint32_t row, uint32_t col, uint64_t drop_thresh) {
  return (dropout_keep4(seed, offset, row, col & ~3u, drop_thresh) >> (col & 3)) & 1u;
}

}  // namespace jvae
