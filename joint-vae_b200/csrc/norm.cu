// BatchNorm2d (train / eval), activation backward, bias gradient, max / average pooling and nearest up-sampling on NHWC
// bf16 activations: the layers that sit between the tcgen05 convolutions of the reference's features / imager stacks
// (module/vae_layers/conv.py:189-227: Conv -> [BatchNorm2d] -> activation, MaxPool2d / AvgPool2d, UpsamplingNearest2d).
//
// All kernels are HBM-bound streaming passes over a (P pixels, C channels) matrix with leading dimension ld.  Thread
// mapping: a thread owns ONE channel chunk (8 channels = one 16-byte vector when C and every ld are multiples of 8,
// one channel otherwise) for the whole kernel and walks over pixels, so per-channel parameters live in registers and
// per-channel reductions need one shared-memory + one global atomic per block.
#include "common.cuh"
#include <mutex>
#include <unordered_map>
#include <initializer_list>

namespace jvae {

constexpr int NORM_MAX_THREADS = 256;

template <int V> struct Vec;
template <> struct Vec<8> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    v[0] = bf16_lo(u.x); v[1] = bf16_hi(u.x); v[2] = bf16_lo(u.y); v[3] = bf16_hi(u.y);
    v[4] = bf16_lo(u.z); v[5] = bf16_hi(u.z); v[6] = bf16_lo(u.w); v[7] = bf16_hi(u.w);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 u;
    u.x = pack_bf16(v[0], v[1]); u.y = pack_bf16(v[2], v[3]); u.z = pack_bf16(v[4], v[5]); u.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(p) = u;
  }
};
// packed loads kept raw until use (the reductions hold several of them in flight per thread)
template <int V> struct Raw;
template <> struct Raw<8> {
  typedef uint4 T;
  static __device__ __forceinline__ T load(const __nv_bfloat16* p) { return ld_stream16(p); }
  static __device__ __forceinline__ T zero() { return make_uint4(0u, 0u, 0u, 0u); }
  static __device__ __forceinline__ void unpack(const T& u, float (&v)[8]) {
    v[0] = bf16_lo(u.x); v[1] = bf16_hi(u.x); v[2] = bf16_lo(u.y); v[3] = bf16_hi(u.y);
    v[4] = bf16_lo(u.z); v[5] = bf16_hi(u.z); v[6] = bf16_lo(u.w); v[7] = bf16_hi(u.w);
  }
};
template <> struct Raw<1> {
  typedef float T;
  static __device__ __forceinline__ T load(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ T zero() { return 0.f; }
  static __device__ __forceinline__ void unpack(const T& u, float (&v)[1]) { v[0] = u; }
};
template <> struct Vec<1> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[1]) { v[0] = __bfloat162float(*p); }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[1]) { *p = __float2bfloat16(v[0]); }
};

// thread geometry shared by all kernels: nchunk chunks per pixel, blockDim.x = nchunk * pixels_per_block
struct Geo {
  int nchunk, ppb, threads, grid;
};
static Geo make_geo(size_t P, int C, int V, int blocks_per_sm = 8) {
  Geo g;
  g.nchunk = C / V;
  g.ppb = NORM_MAX_THREADS / g.nchunk;
  if (g.ppb < 1) g.ppb = 1;
  g.threads = g.nchunk * g.ppb;
  size_t want = (P + g.ppb - 1) / g.ppb;
  const size_t cap = (size_t)sm_count() * blocks_per_sm;
  g.grid = (int)(want < cap ? (want ? want : 1) : cap);
  return g;
}

__device__ __forceinline__ float act_fwd(float z, int act) {
  if (act == JVAE_ACT_RELU) return fmaxf(z, 0.f);
  if (act == JVAE_ACT_SIGMOID) return 1.f / (1.f + __expf(-z));
  if (act == JVAE_ACT_LEAKY) return z > 0.f ? z : JVAE_LEAKY_SLOPE * z;
  return z;
}
// derivative of the activation expressed with the pre-activation z
__device__ __forceinline__ float act_grad_z(float z, int act) {
  if (act == JVAE_ACT_RELU) return z > 0.f ? 1.f : 0.f;
  if (act == JVAE_ACT_SIGMOID) { const float s = 1.f / (1.f + __expf(-z)); return s * (1.f - s); }
  if (act == JVAE_ACT_LEAKY) return z > 0.f ? 1.f : JVAE_LEAKY_SLOPE;
  return 1.f;
}

// per-block reduction of per-thread channel partials: s_acc[(k * C) + channel] += v, then one global atomic per value.
// Shared and global accumulators are fp64: the order in which warps / blocks arrive does not change the fp32 result,
// so the statistics (and everything downstream) are reproducible run to run.
// When the chunk count divides the warp (power of two <= 16) the lanes that own the same chunk are folded with
// shuffles first, so shared memory sees one atomic per chunk and warp instead of 32 / nchunk conflicting ones.
// gld: row stride of gout (0 = C, dense (NK, C)); a wider array takes the statistics of a channel slice of a dense block
template <int V, int NK>
__device__ __forceinline__ void block_channel_reduce(float (&acc)[NK][V], int chunk, int C, double* s_acc, double* gout,
                                                     int gld = 0) {
  for (int i = threadIdx.x; i < NK * C; i += blockDim.x) s_acc[i] = 0.0;
  __syncthreads();
  const int nchunk = C / V;
  const bool fold = nchunk < 32 && (nchunk & (nchunk - 1)) == 0 && (blockDim.x & 31) == 0;
  if (fold) {
#pragma unroll
    for (int k = 0; k < NK; ++k)
#pragma unroll
      for (int j = 0; j < V; ++j) {
        float v = acc[k][j];
        for (int off = nchunk; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        acc[k][j] = v;
      }
  }
  if (!fold || (threadIdx.x & 31) < nchunk) {
#pragma unroll
    for (int k = 0; k < NK; ++k)
#pragma unroll
      for (int j = 0; j < V; ++j) atomicAdd(&s_acc[k * C + chunk * V + j], (double)acc[k][j]);
  }
  __syncthreads();
  if (gld == 0 || gld == C) {
    for (int i = threadIdx.x; i < NK * C; i += blockDim.x) atomicAdd(&gout[i], s_acc[i]);
  } else {
    for (int i = threadIdx.x; i < NK * C; i += blockDim.x) atomicAdd(&gout[(i / C) * gld + i % C], s_acc[i]);
  }
}

// same, for a float destination (bias gradients accumulate straight into the fp32 .grad buffer)
template <int V, int NK>
__device__ __forceinline__ void block_channel_reduce_f32(float (&acc)[NK][V], int chunk, int C, double* s_acc, float* gout) {
  for (int i = threadIdx.x; i < NK * C; i += blockDim.x) s_acc[i] = 0.0;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < NK; ++k)
#pragma unroll
    for (int j = 0; j < V; ++j) atomicAdd(&s_acc[k * C + chunk * V + j], (double)acc[k][j]);
  __syncthreads();
  for (int i = threadIdx.x; i < NK * C; i += blockDim.x) atomicAdd(&gout[i], (float)s_acc[i]);
}

// ------------------------------------------------------------------------------------------------ statistics
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) bn_stats_kernel(const __nv_bfloat16* __restrict__ y, size_t P, int C, int ld,
                                                                    int nchunk, int ppb, double* stats, int sld) {
  extern __shared__ double s_acc[];
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  float acc[2][V];
#pragma unroll
  for (int j = 0; j < V; ++j) acc[0][j] = acc[1][j] = 0.f;
  constexpr int U = 4;
  const size_t step = (size_t)gridDim.x * ppb;
  for (size_t p0 = (size_t)blockIdx.x * ppb + pl; p0 < P; p0 += U * step) {
    float v[U][V];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p < P) {
        Vec<V>::load(y + p * ld + chunk * V, v[u]);
      } else {
#pragma unroll
        for (int j = 0; j < V; ++j) v[u][j] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int j = 0; j < V; ++j) { acc[0][j] += v[u][j]; acc[1][j] += v[u][j] * v[u][j]; }
  }
  block_channel_reduce<V, 2>(acc, chunk, C, s_acc, stats, sld);
}

// ------------------------------------------------------------------------------------------------ BN forward
struct BnFwd {
  const __nv_bfloat16* y; __nv_bfloat16* out;
  size_t P; int C, ld_y, ld_out, nchunk, ppb, act, training;
  int sld;                // row stride of stats: sums at stats[c], sums of squares at stats[sld + c]
  const double* stats; const float* gamma; const float* beta;
  float* running_mean; float* running_var; long long* num_batches; float* save;
  float eps, momentum;
};

template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) bn_apply_fwd_kernel(const BnFwd a) {
  const int chunk = threadIdx.x % a.nchunk, pl = threadIdx.x / a.nchunk;
  float scale[V], shift[V];
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const int c = chunk * V + j;
    float mean, rstd;
    if (a.training) {
      const double inv = 1.0 / (double)a.P;
      const double mean_d = a.stats[c] * inv;
      mean = (float)mean_d;
      const float var = fmaxf((float)(a.stats[a.sld + c] * inv - mean_d * mean_d), 0.f);
      rstd = rsqrtf(var + a.eps);
      if (blockIdx.x == 0 && pl == 0) {
        a.save[c] = mean; a.save[a.C + c] = rstd;
        if (a.running_mean) {   // torch: running = (1-m) running + m batch, unbiased variance
          const float unb = a.P > 1 ? var * (float)a.P / (float)(a.P - 1) : var;
          a.running_mean[c] = (1.f - a.momentum) * a.running_mean[c] + a.momentum * mean;
          a.running_var[c] = (1.f - a.momentum) * a.running_var[c] + a.momentum * unb;
        }
      }
    } else {
      mean = a.running_mean[c];
      rstd = rsqrtf(a.running_var[c] + a.eps);
    }
    const float g = a.gamma ? a.gamma[c] : 1.f, b = a.beta ? a.beta[c] : 0.f;
    scale[j] = g * rstd;
    shift[j] = b - mean * scale[j];
  }
  if (a.training && a.num_batches && blockIdx.x == 0 && threadIdx.x == 0) *a.num_batches += 1;
  constexpr int U = 4;        // rows per thread and round, loads requested together
  const size_t step = (size_t)gridDim.x * a.ppb;
  for (size_t p0 = (size_t)blockIdx.x * a.ppb + pl; p0 < a.P; p0 += U * step) {
    typename Raw<V>::T yr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      yr[u] = p < a.P ? Raw<V>::load(a.y + p * a.ld_y + chunk * V) : Raw<V>::zero();
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p >= a.P) break;
      float v[V];
      Raw<V>::unpack(yr[u], v);
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] = act_fwd(fmaf(v[j], scale[j], shift[j]), a.act);
      Vec<V>::store(a.out + p * a.ld_out + chunk * V, v);
    }
  }
}

// ------------------------------------------------------------------------------------------------ BN backward
constexpr int BN_REDUCE_BLOCKS = 3;      // resident blocks per SM of the backward reduction (one wave)
struct BnBwd {
  const __nv_bfloat16* da; const __nv_bfloat16* y; __nv_bfloat16* dy;
  size_t P; int C, ld_da, ld_y, ld_dy, nchunk, ppb, act;
  const float* save; const float* gamma; const float* beta;
  double* sums;           // (2, C): sum g, sum g * xhat   (zeroed by the caller before the reduce kernel)
  float* dgamma; float* dbeta;
  // pre-activation BatchNorm of a dense block (jvae_bn_preact_bwd): dxf (fp32, row stride ld_dxf) += the data gradient
  // instead of storing bf16 dy; eval != 0: running statistics, the gradient is the per-channel scale only (no reduction)
  float* dxf; int ld_dxf, eval;
  const float* rmean; const float* rvar; float eps;
};

// dst[0..V) += v (fp32 accumulator of a dense block's channel gradients)
template <int V>
__device__ __forceinline__ void acc_f32(float* dst, const float (&v)[V]) {
  if constexpr (V == 8) {
    float4* d = reinterpret_cast<float4*>(dst);
    float4 x0 = d[0], x1 = d[1];
    x0.x += v[0]; x0.y += v[1]; x0.z += v[2]; x0.w += v[3];
    x1.x += v[4]; x1.y += v[5]; x1.z += v[6]; x1.w += v[7];
    d[0] = x0; d[1] = x1;
  } else {
#pragma unroll
    for (int j = 0; j < V; ++j) dst[j] += v[j];
  }
}

template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS, BN_REDUCE_BLOCKS) bn_bwd_reduce_kernel(const BnBwd a) {
  extern __shared__ double s_acc[];
  const int chunk = threadIdx.x % a.nchunk, pl = threadIdx.x / a.nchunk;
  // registers: only scale / shift live through the loop (the activation mask needs z); sum g xhat is recovered at the end
  // from sum g y, so four blocks of 256 threads fit per SM and their load / compute phases interleave
  float scale[V], shift[V], acc[2][V];
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const int c = chunk * V + j;
    const float mean = a.save[c], rstd = a.save[a.C + c];
    const float g = a.gamma ? a.gamma[c] : 1.f, b = a.beta ? a.beta[c] : 0.f;
    scale[j] = g * rstd; shift[j] = b - mean * scale[j];
    acc[0][j] = acc[1][j] = 0.f;
  }
  // U pixel rows per thread and round, all 2 U loads requested (and kept packed) before the first use: ~100 KB in flight per SM
  constexpr int U = 4;
  const size_t step = (size_t)gridDim.x * a.ppb;
  for (size_t p0 = (size_t)blockIdx.x * a.ppb + pl; p0 < a.P; p0 += U * step) {
    typename Raw<V>::T gr[U], yr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p < a.P) {
        gr[u] = Raw<V>::load(a.da + p * a.ld_da + chunk * V);
        yr[u] = Raw<V>::load(a.y + p * a.ld_y + chunk * V);
      } else {
        gr[u] = Raw<V>::zero(); yr[u] = Raw<V>::zero();
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float g[V], y[V];
      Raw<V>::unpack(gr[u], g);
      Raw<V>::unpack(yr[u], y);
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float gz = g[j] * act_grad_z(fmaf(y[j], scale[j], shift[j]), a.act);
        acc[0][j] += gz;
        acc[1][j] = fmaf(gz, y[j], acc[1][j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < V; ++j) {      // sum g xhat = (sum g y - mean sum g) rstd, per thread before the cross-thread reduction
    const int c = chunk * V + j;
    acc[1][j] = (acc[1][j] - a.save[c] * acc[0][j]) * a.save[a.C + c];
  }
  block_channel_reduce<V, 2>(acc, chunk, a.C, s_acc, a.sums);
}

template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) bn_bwd_apply_kernel(const BnBwd a) {
  const int chunk = threadIdx.x % a.nchunk, pl = threadIdx.x / a.nchunk;
  float mean[V], rstd[V], scale[V], shift[V], k1[V], k2[V];
  const float inv = 1.f / (float)a.P;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const int c = chunk * V + j;
    if (a.eval) {
      mean[j] = a.rmean[c]; rstd[j] = rsqrtf(a.rvar[c] + a.eps);
    } else {
      mean[j] = a.save[c]; rstd[j] = a.save[a.C + c];
    }
    const float g = a.gamma ? a.gamma[c] : 1.f, b = a.beta ? a.beta[c] : 0.f;
    scale[j] = g * rstd[j]; shift[j] = b - mean[j] * scale[j];
    if (a.eval) {
      k1[j] = k2[j] = 0.f;
    } else {
      k1[j] = (float)(a.sums[c] * (double)inv); k2[j] = (float)(a.sums[a.C + c] * (double)inv);
      if (blockIdx.x == 0 && pl == 0) {
        if (a.dbeta) a.dbeta[c] += (float)a.sums[c];   // accumulated: the caller passes a zeroed buffer or the live .grad
        if (a.dgamma) a.dgamma[c] += (float)a.sums[a.C + c];
      }
    }
  }
  constexpr int U = 2;        // rows per thread and round, the 2 U loads requested together
  const size_t step = (size_t)gridDim.x * a.ppb;
  for (size_t p0 = (size_t)blockIdx.x * a.ppb + pl; p0 < a.P; p0 += U * step) {
    typename Raw<V>::T gr[U], yr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p < a.P) {
        gr[u] = Raw<V>::load(a.da + p * a.ld_da + chunk * V);
        yr[u] = Raw<V>::load(a.y + p * a.ld_y + chunk * V);
      } else {
        gr[u] = Raw<V>::zero(); yr[u] = Raw<V>::zero();
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p >= a.P) break;
      float g[V], y[V];
      Raw<V>::unpack(gr[u], g);
      Raw<V>::unpack(yr[u], y);
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float gz = g[j] * act_grad_z(fmaf(y[j], scale[j], shift[j]), a.act);
        const float xh = (y[j] - mean[j]) * rstd[j];
        g[j] = scale[j] * (gz - k1[j] - xh * k2[j]);
      }
      if (a.dxf) acc_f32<V>(a.dxf + p * a.ld_dxf + chunk * V, g);
      else Vec<V>::store(a.dy + p * a.ld_dy + chunk * V, g);
    }
  }
}


// ------------------------------------------------------------------------------------------------ narrow tensors (C <= 8)
// The image head's BatchNorm (3 channels in an 8-channel padded row): with one channel per thread the generic <1> kernels moved
// 2 bytes per load (reduce 140 us, apply 90 us, forward 41 us on 8704 x 32 x 32 pixels: ~2 TB/s).  Here a thread owns a whole
// pixel: the padded 16-byte rows of y / dy are one vector, a dense row (ld < 8: the loss gradient, the image) is C scalars.
// Padded channels carry zero parameters, so they produce zeros.
__device__ __forceinline__ void narrow_load_row(const __nv_bfloat16* base, size_t p, int ld, int C, float (&v)[8]) {
  if (ld == 8) {
    Raw<8>::unpack(ld_stream16(base + p * 8), v);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = j < C ? __bfloat162float(base[p * ld + j]) : 0.f;
  }
}
__device__ __forceinline__ void narrow_store_row(__nv_bfloat16* base, size_t p, int ld, int C, const float (&v)[8]) {
  if (ld == 8) {
    Vec<8>::store(base + p * 8, v);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j < ld) base[p * ld + j] = __float2bfloat16(j < C ? v[j] : 0.f);
  }
}
// warp + block reduction of NK x 8 per-thread partials into gout[k * C + c] (fp64 atomics: order independent)
template <int NK>
__device__ __forceinline__ void narrow_reduce(float (&acc)[NK][8], int C, double* s_acc, double* gout) {
  for (int i = threadIdx.x; i < NK * 8; i += blockDim.x) s_acc[i] = 0.0;
  __syncthreads();
#pragma unroll
  for (int k = 0; k < NK; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = acc[k][j];
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if ((threadIdx.x & 31) == 0 && j < C) atomicAdd(&s_acc[k * 8 + j], (double)v);
    }
  __syncthreads();
  for (int i = threadIdx.x; i < NK * 8; i += blockDim.x)
    if ((i & 7) < C) atomicAdd(&gout[(i >> 3) * C + (i & 7)], s_acc[i]);
}

__global__ void __launch_bounds__(NORM_MAX_THREADS) bn_apply_fwd_narrow_kernel(const BnFwd a) {
  float scale[8], shift[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    scale[c] = shift[c] = 0.f;
    if (c >= a.C) continue;
    float mean, rstd;
    if (a.training) {
      const double inv = 1.0 / (double)a.P;
      const double mean_d = a.stats[c] * inv;
      mean = (float)mean_d;
      const float var = fmaxf((float)(a.stats[a.sld + c] * inv - mean_d * mean_d), 0.f);
      rstd = rsqrtf(var + a.eps);
      if (blockIdx.x == 0 && threadIdx.x == 0) {
        a.save[c] = mean; a.save[a.C + c] = rstd;
        if (a.running_mean) {
          const float unb = a.P > 1 ? var * (float)a.P / (float)(a.P - 1) : var;
          a.running_mean[c] = (1.f - a.momentum) * a.running_mean[c] + a.momentum * mean;
          a.running_var[c] = (1.f - a.momentum) * a.running_var[c] + a.momentum * unb;
        }
      }
    } else {
      mean = a.running_mean[c];
      rstd = rsqrtf(a.running_var[c] + a.eps);
    }
    const float g = a.gamma ? a.gamma[c] : 1.f, b = a.beta ? a.beta[c] : 0.f;
    scale[c] = g * rstd;
    shift[c] = b - mean * scale[c];
  }
  if (a.training && a.num_batches && blockIdx.x == 0 && threadIdx.x == 0) *a.num_batches += 1;
  constexpr int U = 4;
  const size_t step = (size_t)gridDim.x * blockDim.x;
  for (size_t p0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p0 < a.P; p0 += U * step) {
    uint4 yr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) yr[u] = p0 + u * step < a.P ? ld_stream16(a.y + (p0 + u * step) * 8) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p >= a.P) break;
      float v[8];
      Raw<8>::unpack(yr[u], v);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = j < a.C ? act_fwd(fmaf(v[j], scale[j], shift[j]), a.act) : 0.f;
      narrow_store_row(a.out, p, a.ld_out, a.C, v);
    }
  }
}

__global__ void __launch_bounds__(NORM_MAX_THREADS, BN_REDUCE_BLOCKS) bn_bwd_reduce_narrow_kernel(const BnBwd a) {
  __shared__ double s_acc[16];
  float scale[8], shift[8], acc[2][8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    scale[c] = shift[c] = 0.f; acc[0][c] = acc[1][c] = 0.f;
    if (c < a.C) {
      const float mean = a.save[c], rstd = a.save[a.C + c];
      const float g = a.gamma ? a.gamma[c] : 1.f, b = a.beta ? a.beta[c] : 0.f;
      scale[c] = g * rstd; shift[c] = b - mean * scale[c];
    }
  }
  constexpr int U = 4;
  const size_t step = (size_t)gridDim.x * blockDim.x;
  for (size_t p0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p0 < a.P; p0 += U * step) {
    uint4 yr[U];
    float g[U][8];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p < a.P) {
        yr[u] = ld_stream16(a.y + p * 8);
        narrow_load_row(a.da, p, a.ld_da, a.C, g[u]);
      } else {
        yr[u] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int j = 0; j < 8; ++j) g[u][j] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float y[8];
      Raw<8>::unpack(yr[u], y);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gz = g[u][j] * act_grad_z(fmaf(y[j], scale[j], shift[j]), a.act);
        acc[0][j] += gz;
        acc[1][j] = fmaf(gz, y[j], acc[1][j]);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c)
    if (c < a.C) acc[1][c] = (acc[1][c] - a.save[c] * acc[0][c]) * a.save[a.C + c];
    else acc[0][c] = acc[1][c] = 0.f;
  narrow_reduce<2>(acc, a.C, s_acc, a.sums);
}

__global__ void __launch_bounds__(NORM_MAX_THREADS) bn_bwd_apply_narrow_kernel(const BnBwd a) {
  float mean[8], rstd[8], scale[8], shift[8], k1[8], k2[8];
  const float inv = 1.f / (float)a.P;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    mean[c] = rstd[c] = scale[c] = shift[c] = k1[c] = k2[c] = 0.f;
    if (c >= a.C) continue;
    mean[c] = a.save[c]; rstd[c] = a.save[a.C + c];
    const float g = a.gamma ? a.gamma[c] : 1.f, b = a.beta ? a.beta[c] : 0.f;
    scale[c] = g * rstd[c]; shift[c] = b - mean[c] * scale[c];
    k1[c] = (float)(a.sums[c] * (double)inv); k2[c] = (float)(a.sums[a.C + c] * (double)inv);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      if (a.dbeta) a.dbeta[c] += (float)a.sums[c];
      if (a.dgamma) a.dgamma[c] += (float)a.sums[a.C + c];
    }
  }
  constexpr int U = 2;
  const size_t step = (size_t)gridDim.x * blockDim.x;
  for (size_t p0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p0 < a.P; p0 += U * step) {
    uint4 yr[U];
    float g[U][8];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p < a.P) {
        yr[u] = ld_stream16(a.y + p * 8);
        narrow_load_row(a.da, p, a.ld_da, a.C, g[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t p = p0 + u * step;
      if (p >= a.P) break;
      float y[8], o[8];
      Raw<8>::unpack(yr[u], y);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gz = g[u][j] * act_grad_z(fmaf(y[j], scale[j], shift[j]), a.act);
        const float xh = (y[j] - mean[j]) * rstd[j];
        o[j] = scale[j] * (gz - k1[j] - xh * k2[j]);
      }
      Vec<8>::store(a.dy + p * 8, o);
    }
  }
}

// ------------------------------------------------------------------------------------------------ activation backward + bias gradient
// dy = da * f'(a) with the derivative expressed through the OUTPUT a of the activation (relu: a > 0, sigmoid: a (1 - a));
// dbias[c] += sum_p dy[p, c].  act == none: pure channel sum of da (dy may be null).
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) act_bwd_kernel(const __nv_bfloat16* __restrict__ da, int ld_da,
                                                                   const __nv_bfloat16* __restrict__ aout, int ld_a, size_t P, int C,
                                                                   int nchunk, int ppb, int act, __nv_bfloat16* dy, int ld_dy,
                                                                   float* dbias) {
  extern __shared__ double s_acc[];
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  float acc[1][V];
#pragma unroll
  for (int j = 0; j < V; ++j) acc[0][j] = 0.f;
  for (size_t p = (size_t)blockIdx.x * ppb + pl; p < P; p += (size_t)gridDim.x * ppb) {
    float g[V];
    Vec<V>::load(da + p * ld_da + chunk * V, g);
    if (act != JVAE_ACT_NONE) {
      float o[V];
      Vec<V>::load(aout + p * ld_a + chunk * V, o);
#pragma unroll
      for (int j = 0; j < V; ++j)
        g[j] *= (act == JVAE_ACT_RELU) ? (o[j] > 0.f ? 1.f : 0.f)
                : (act == JVAE_ACT_LEAKY) ? (o[j] > 0.f ? 1.f : JVAE_LEAKY_SLOPE) : o[j] * (1.f - o[j]);
    }
    if (dy) Vec<V>::store(dy + p * ld_dy + chunk * V, g);
#pragma unroll
    for (int j = 0; j < V; ++j) acc[0][j] += g[j];
  }
  if (dbias) block_channel_reduce_f32<V, 1>(acc, chunk, C, s_acc, dbias);
}

// ------------------------------------------------------------------------------------------------ pooling / up-sampling
// k x k max pooling with stride s >= k, no padding, floor mode: out (N, (H-k)/s+1, (W-k)/s+1, C)
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ in, int H, int W, int ld_in,
                                                                       __nv_bfloat16* __restrict__ out, int ld_out, int Ho, int Wo,
                                                                       int k, int s, size_t Pout, int nchunk, int ppb) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  for (size_t p = (size_t)blockIdx.x * ppb + pl; p < Pout; p += (size_t)gridDim.x * ppb) {
    const int ox = (int)(p % Wo), oy = (int)((p / Wo) % Ho);
    const size_t n = p / ((size_t)Wo * Ho);
    const __nv_bfloat16* base = in + ((n * H + (size_t)s * oy) * W + (size_t)s * ox) * ld_in + chunk * V;
    float m[V], t[V];
    Vec<V>::load(base, m);
    for (int i = 0; i < k; ++i)
      for (int j = (i == 0 ? 1 : 0); j < k; ++j) {
        Vec<V>::load(base + ((size_t)i * W + j) * ld_in, t);
#pragma unroll
        for (int e = 0; e < V; ++e) m[e] = fmaxf(m[e], t[e]);
      }
    Vec<V>::store(out + p * ld_out + chunk * V, m);
  }
}

// gradient goes to the FIRST maximum of the window in row-major order (torch's max_pool2d tie rule); windows do not
// overlap (s >= k), so every input pixel inside a window is written exactly once (pixels outside: caller zero-fills)
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ in, int H, int W, int ld_in,
                                                                       const __nv_bfloat16* __restrict__ dout, int ld_dout,
                                                                       __nv_bfloat16* __restrict__ din, int ld_din, int Ho, int Wo,
                                                                       int k, int s, size_t Pout, int nchunk, int ppb) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  for (size_t p = (size_t)blockIdx.x * ppb + pl; p < Pout; p += (size_t)gridDim.x * ppb) {
    const int ox = (int)(p % Wo), oy = (int)((p / Wo) % Ho);
    const size_t n = p / ((size_t)Wo * Ho);
    const size_t pix = (n * H + (size_t)s * oy) * W + (size_t)s * ox;
    const __nv_bfloat16* base = in + pix * ld_in + chunk * V;
    float m[V], t[V], g[V];
    int win[V];
    Vec<V>::load(base, m);
#pragma unroll
    for (int e = 0; e < V; ++e) win[e] = 0;
    for (int i = 0; i < k; ++i)
      for (int j = (i == 0 ? 1 : 0); j < k; ++j) {
        Vec<V>::load(base + ((size_t)i * W + j) * ld_in, t);
#pragma unroll
        for (int e = 0; e < V; ++e)
          if (t[e] > m[e]) { m[e] = t[e]; win[e] = i * k + j; }
      }
    Vec<V>::load(dout + p * ld_dout + chunk * V, g);
    __nv_bfloat16* d = din + pix * ld_din + chunk * V;
    for (int i = 0; i < k; ++i)
      for (int j = 0; j < k; ++j) {
#pragma unroll
        for (int e = 0; e < V; ++e) t[e] = (win[e] == i * k + j) ? g[e] : 0.f;
        Vec<V>::store(d + ((size_t)i * W + j) * ld_din, t);
      }
  }
}

// nearest-neighbour 2x up-sampling: out (N, 2H, 2W, C); backward sums the 2x2 block
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) upsample2_kernel(const __nv_bfloat16* __restrict__ src, int ld_src,
                                                                     __nv_bfloat16* __restrict__ dst, int ld_dst, int H, int W,
                                                                     size_t Pin, int nchunk, int ppb, int backward) {
  // forward: src = small (N,H,W), dst = large (N,2H,2W).  backward: src = large gradient, dst = small gradient.
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  for (size_t p = (size_t)blockIdx.x * ppb + pl; p < Pin; p += (size_t)gridDim.x * ppb) {
    const int x = (int)(p % W), y = (int)((p / W) % H);
    const size_t n = p / ((size_t)W * H);
    const size_t big = (n * 2 * H + 2 * y) * (size_t)(2 * W) + 2 * x;
    if (!backward) {
      float v[V];
      Vec<V>::load(src + p * ld_src + chunk * V, v);
      __nv_bfloat16* d = dst + big * ld_dst + chunk * V;
      Vec<V>::store(d, v);
      Vec<V>::store(d + ld_dst, v);
      Vec<V>::store(d + (size_t)2 * W * ld_dst, v);
      Vec<V>::store(d + (size_t)(2 * W + 1) * ld_dst, v);
    } else {
      float v[V], t[V];
      const __nv_bfloat16* s = src + big * ld_src + chunk * V;
      Vec<V>::load(s, v);
      Vec<V>::load(s + ld_src, t);
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] += t[j];
      Vec<V>::load(s + (size_t)2 * W * ld_src, t);
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] += t[j];
      Vec<V>::load(s + (size_t)(2 * W + 1) * ld_src, t);
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] += t[j];
      Vec<V>::store(dst + p * ld_dst + chunk * V, v);
    }
  }
}

// ------------------------------------------------------------------------------------------------ padded / overlapping max pooling
// kernel k, stride s, padding p (padded positions never win), floor mode: torchvision's ResNet stem MaxPool2d(3, 2, 1)
struct PoolGeo { int H, W, Ho, Wo, k, s, p; };

template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) maxpool_pad_fwd_kernel(const __nv_bfloat16* __restrict__ in, int ld_in,
                                                                           __nv_bfloat16* __restrict__ out, int ld_out, PoolGeo q,
                                                                           size_t Pout, int nchunk, int ppb) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  for (size_t pp = (size_t)blockIdx.x * ppb + pl; pp < Pout; pp += (size_t)gridDim.x * ppb) {
    const int ox = (int)(pp % q.Wo), oy = (int)((pp / q.Wo) % q.Ho);
    const size_t n = pp / ((size_t)q.Wo * q.Ho);
    float m[V], t[V];
#pragma unroll
    for (int e = 0; e < V; ++e) m[e] = -__int_as_float(0x7f800000);
    for (int i = 0; i < q.k; ++i) {
      const int iy = oy * q.s - q.p + i;
      if (iy < 0 || iy >= q.H) continue;
      for (int j = 0; j < q.k; ++j) {
        const int ix = ox * q.s - q.p + j;
        if (ix < 0 || ix >= q.W) continue;
        Vec<V>::load(in + ((n * q.H + iy) * q.W + ix) * ld_in + chunk * V, t);
#pragma unroll
        for (int e = 0; e < V; ++e) m[e] = fmaxf(m[e], t[e]);
      }
    }
    Vec<V>::store(out + pp * ld_out + chunk * V, m);
  }
}

// one thread per INPUT pixel: it collects the gradient of every window that contains it and whose first maximum (row-major
// scan, torch's tie rule) it is; no atomics, every input pixel is written once
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) maxpool_pad_bwd_kernel(const __nv_bfloat16* __restrict__ in, int ld_in,
                                                                           const __nv_bfloat16* __restrict__ dout, int ld_dout,
                                                                           __nv_bfloat16* __restrict__ din, int ld_din, PoolGeo q,
                                                                           size_t Pin, int nchunk, int ppb) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  for (size_t pp = (size_t)blockIdx.x * ppb + pl; pp < Pin; pp += (size_t)gridDim.x * ppb) {
    const int ix = (int)(pp % q.W), iy = (int)((pp / q.W) % q.H);
    const size_t n = pp / ((size_t)q.W * q.H);
    float acc[V], me[V], t[V], g[V];
#pragma unroll
    for (int e = 0; e < V; ++e) acc[e] = 0.f;
    Vec<V>::load(in + pp * ld_in + chunk * V, me);
    // windows oy with oy*s - p <= iy <= oy*s - p + k - 1
    int oy0 = iy + q.p - q.k + 1;
    oy0 = oy0 <= 0 ? 0 : (oy0 + q.s - 1) / q.s;
    int ox0 = ix + q.p - q.k + 1;
    ox0 = ox0 <= 0 ? 0 : (ox0 + q.s - 1) / q.s;
    const int oy1 = min((iy + q.p) / q.s, q.Ho - 1), ox1 = min((ix + q.p) / q.s, q.Wo - 1);
    for (int oy = oy0; oy <= oy1; ++oy)
      for (int ox = ox0; ox <= ox1; ++ox) {
        // this pixel wins the window iff no EARLIER position is >= it and no LATER position is > it
        bool win[V];
#pragma unroll
        for (int e = 0; e < V; ++e) win[e] = true;
        for (int i = 0; i < q.k; ++i) {
          const int yy = oy * q.s - q.p + i;
          if (yy < 0 || yy >= q.H) continue;
          for (int j = 0; j < q.k; ++j) {
            const int xx = ox * q.s - q.p + j;
            if (xx < 0 || xx >= q.W || (yy == iy && xx == ix)) continue;
            Vec<V>::load(in + ((n * q.H + yy) * q.W + xx) * ld_in + chunk * V, t);
            const bool earlier = yy < iy || (yy == iy && xx < ix);
#pragma unroll
            for (int e = 0; e < V; ++e) win[e] = win[e] && (earlier ? t[e] < me[e] : t[e] <= me[e]);
          }
        }
        Vec<V>::load(dout + ((n * q.Ho + oy) * q.Wo + ox) * ld_dout + chunk * V, g);
#pragma unroll
        for (int e = 0; e < V; ++e) acc[e] += win[e] ? g[e] : 0.f;
      }
    Vec<V>::store(din + pp * ld_din + chunk * V, acc);
  }
}

// k x k average pooling with stride k (k = H = W: AdaptiveAvgPool2d(1)); backward spreads dout / k^2 over the window
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) avgpool_kernel(const __nv_bfloat16* __restrict__ src, int ld_src,
                                                                   __nv_bfloat16* __restrict__ dst, int ld_dst, int H, int W, int k,
                                                                   size_t Psmall, int nchunk, int ppb, int backward) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  const int Ho = H / k, Wo = W / k;
  const float inv = 1.f / (float)(k * k);
  for (size_t pp = (size_t)blockIdx.x * ppb + pl; pp < Psmall; pp += (size_t)gridDim.x * ppb) {
    const int ox = (int)(pp % Wo), oy = (int)((pp / Wo) % Ho);
    const size_t n = pp / ((size_t)Wo * Ho);
    const size_t big = (n * H + (size_t)oy * k) * W + (size_t)ox * k;
    float v[V], t[V];
    if (!backward) {      // src = large, dst = small
#pragma unroll
      for (int e = 0; e < V; ++e) v[e] = 0.f;
      for (int i = 0; i < k; ++i)
        for (int j = 0; j < k; ++j) {
          Vec<V>::load(src + (big + (size_t)i * W + j) * ld_src + chunk * V, t);
#pragma unroll
          for (int e = 0; e < V; ++e) v[e] += t[e];
        }
#pragma unroll
      for (int e = 0; e < V; ++e) v[e] *= inv;
      Vec<V>::store(dst + pp * ld_dst + chunk * V, v);
    } else {              // src = small gradient, dst = large gradient
      Vec<V>::load(src + pp * ld_src + chunk * V, v);
#pragma unroll
      for (int e = 0; e < V; ++e) v[e] *= inv;
      for (int i = 0; i < k; ++i)
        for (int j = 0; j < k; ++j) Vec<V>::store(dst + (big + (size_t)i * W + j) * ld_dst + chunk * V, v);
    }
  }
}

// nearest up-sampling by an integer factor s (UpsamplingNearest2d(scale_factor=s)).  Forward: one thread per OUTPUT pixel
// copies its source pixel (coalesced stores; the s consecutive readers of a source pixel hit L1).  Backward: one thread per
// INPUT pixel sums its s x s block of the output gradient in fp32 in a fixed order: no atomics, bit-reproducible.
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) upsample_nearest_kernel(const __nv_bfloat16* __restrict__ src, int ld_src,
                                                                            __nv_bfloat16* __restrict__ dst, int ld_dst, int H,
                                                                            int W, int s, size_t P, int nchunk, int ppb,
                                                                            int backward) {
  // forward: P = N * sH * sW output pixels, src = small.  backward: P = N * H * W input pixels, src = large gradient.
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  const int Wb = W * s, Hb = H * s;
  for (size_t p = (size_t)blockIdx.x * ppb + pl; p < P; p += (size_t)gridDim.x * ppb) {
    float v[V];
    if (!backward) {
      const int ox = (int)(p % Wb), oy = (int)((p / Wb) % Hb);
      const size_t n = p / ((size_t)Wb * Hb);
      Vec<V>::load(src + ((n * H + oy / s) * W + ox / s) * ld_src + chunk * V, v);
      Vec<V>::store(dst + p * ld_dst + chunk * V, v);
    } else {
      const int x = (int)(p % W), y = (int)((p / W) % H);
      const size_t n = p / ((size_t)W * H);
      float t[V];
#pragma unroll
      for (int e = 0; e < V; ++e) v[e] = 0.f;
      for (int i = 0; i < s; ++i) {
        const __nv_bfloat16* row = src + ((n * Hb + (size_t)y * s + i) * Wb + (size_t)x * s) * ld_src + chunk * V;
        for (int j = 0; j < s; ++j) {
          Vec<V>::load(row + (size_t)j * ld_src, t);
#pragma unroll
          for (int e = 0; e < V; ++e) v[e] += t[e];
        }
      }
      Vec<V>::store(dst + p * ld_dst + chunk * V, v);
    }
  }
}

// average pooling with torch's AvgPool2d semantics for kernel (kh, kw), stride (sh, sw), padding (ph, pw): floor output
// size, count_include_pad=True (the divisor is always kh * kw).  Forward: one thread per output pixel.  Backward in gather
// form, one thread per INPUT pixel summing dout / (kh * kw) over the windows that cover it: no atomics, every input pixel
// written once (pixels no window covers get zero).
struct AvgGeo { int H, W, Ho, Wo, kh, kw, sh, sw, ph, pw; };

template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) avgpool_pad_kernel(const __nv_bfloat16* __restrict__ src, int ld_src,
                                                                       __nv_bfloat16* __restrict__ dst, int ld_dst, AvgGeo q,
                                                                       size_t P, int nchunk, int ppb, int backward) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  const float div = (float)(q.kh * q.kw);
  for (size_t pp = (size_t)blockIdx.x * ppb + pl; pp < P; pp += (size_t)gridDim.x * ppb) {
    float acc[V], t[V];
#pragma unroll
    for (int e = 0; e < V; ++e) acc[e] = 0.f;
    if (!backward) {      // src = input (N, H, W), dst = output (N, Ho, Wo)
      const int ox = (int)(pp % q.Wo), oy = (int)((pp / q.Wo) % q.Ho);
      const size_t n = pp / ((size_t)q.Wo * q.Ho);
      const int y0 = max(oy * q.sh - q.ph, 0), y1 = min(oy * q.sh - q.ph + q.kh, q.H);
      const int x0 = max(ox * q.sw - q.pw, 0), x1 = min(ox * q.sw - q.pw + q.kw, q.W);
      for (int iy = y0; iy < y1; ++iy)
        for (int ix = x0; ix < x1; ++ix) {
          Vec<V>::load(src + ((n * q.H + iy) * q.W + ix) * ld_src + chunk * V, t);
#pragma unroll
          for (int e = 0; e < V; ++e) acc[e] += t[e];
        }
#pragma unroll
      for (int e = 0; e < V; ++e) acc[e] /= div;
    } else {              // src = output gradient (N, Ho, Wo), dst = input gradient (N, H, W)
      const int ix = (int)(pp % q.W), iy = (int)((pp / q.W) % q.H);
      const size_t n = pp / ((size_t)q.W * q.H);
      // windows o with o*s - p <= i <= o*s - p + k - 1
      int oy0 = iy + q.ph - q.kh + 1, ox0 = ix + q.pw - q.kw + 1;
      oy0 = oy0 <= 0 ? 0 : (oy0 + q.sh - 1) / q.sh;
      ox0 = ox0 <= 0 ? 0 : (ox0 + q.sw - 1) / q.sw;
      const int oy1 = min((iy + q.ph) / q.sh, q.Ho - 1), ox1 = min((ix + q.pw) / q.sw, q.Wo - 1);
      for (int oy = oy0; oy <= oy1; ++oy)
        for (int ox = ox0; ox <= ox1; ++ox) {
          Vec<V>::load(src + ((n * q.Ho + oy) * q.Wo + ox) * ld_src + chunk * V, t);
#pragma unroll
          for (int e = 0; e < V; ++e) acc[e] += t[e] / div;
        }
    }
    Vec<V>::store(dst + pp * ld_dst + chunk * V, acc);
  }
}

// out = act(a + b): the join of a residual block (torchvision BasicBlock / Bottleneck: out += identity; relu)
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) add_act_kernel(const __nv_bfloat16* __restrict__ a, int ld_a,
                                                                   const __nv_bfloat16* __restrict__ b, int ld_b,
                                                                   __nv_bfloat16* __restrict__ out, int ld_out, size_t P, int act,
                                                                   int nchunk, int ppb) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  for (size_t pp = (size_t)blockIdx.x * ppb + pl; pp < P; pp += (size_t)gridDim.x * ppb) {
    float u[V], v[V];
    Vec<V>::load(a + pp * ld_a + chunk * V, u);
    Vec<V>::load(b + pp * ld_b + chunk * V, v);
#pragma unroll
    for (int e = 0; e < V; ++e) u[e] = act_fwd(u[e] + v[e], act);
    Vec<V>::store(out + pp * ld_out + chunk * V, u);
  }
}

// ------------------------------------------------------------------------------------------------ separable narrow-output convolution
// The backward of a k x k convolution with few output channels (the image head 32 -> 3, k5: k * Co = 15 <= 16) runs as the
// backward of a 1 x k convolution to k * Co channels, T[r][(ty, co)] = sum_tx sum_ci x[r + (0, tx - p)][ci] W[co][ci][ty][tx]
// (tensor cores, k taps instead of k^2), whose vertical shift-and-add out[q][co] = sum_ty T[q + (ty - p, 0)][ty * Co + co] is
// the layer's output.  The kernels below are the adjoint of that sum: the gradient of T from the gradient of the output.

// compile-time (k, Co) with the vector layouts (U rows of 16 channels, dy rows of 8): every channel pick is a fixed register,
// the kernel streams at memory speed.  KK * CO <= 16.
template <int KK, int CO>
__global__ void __launch_bounds__(256) vstack_rows_fixed_kernel(const __nv_bfloat16* __restrict__ dy, int N, int H, int W,
                                                                __nv_bfloat16* __restrict__ U) {
  constexpr int PAD = (KK - 1) / 2;
  const size_t P = (size_t)N * H * W;
  for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < P; r += (size_t)gridDim.x * blockDim.x) {
    const int y = (int)((r / W) % H);
    float vals[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) vals[i] = 0.f;
#pragma unroll
    for (int ty = 0; ty < KK; ++ty) {
      const int yy = y - (ty - PAD);
      if (yy < 0 || yy >= H) continue;
      const uint4 d4 = *reinterpret_cast<const uint4*>(dy + (r - (size_t)(ty - PAD) * W) * 8);
      const float d[4] = {bf16_lo(d4.x), bf16_hi(d4.x), bf16_lo(d4.y), bf16_hi(d4.y)};
#pragma unroll
      for (int c = 0; c < CO; ++c) vals[ty * CO + c] = d[c];
    }
    uint4 a, b;
    a.x = pack_bf16(vals[0], vals[1]); a.y = pack_bf16(vals[2], vals[3]); a.z = pack_bf16(vals[4], vals[5]); a.w = pack_bf16(vals[6], vals[7]);
    b.x = pack_bf16(vals[8], vals[9]); b.y = pack_bf16(vals[10], vals[11]); b.z = pack_bf16(vals[12], vals[13]); b.w = pack_bf16(vals[14], vals[15]);
    uint4* u4 = reinterpret_cast<uint4*>(U + r * 16);
    u4[0] = a; u4[1] = b;
  }
}

// adjoint of the shift-and-add: U[r][ty * Co + co] = dy[r - (ty - p, 0)][co] (zero outside the image, zero in the padding channels)
__global__ void __launch_bounds__(256) vstack_rows_kernel(const __nv_bfloat16* __restrict__ dy, int ld_dy, int N, int H, int W, int k,
                                                          int p, int Co, __nv_bfloat16* __restrict__ U, int ld_u) {
  const size_t P = (size_t)N * H * W;
  const bool vec = ld_dy == 8 && ld_u == 16 && Co <= 4 && k * Co <= 16 && ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(U)) & 15) == 0;
  for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < P; r += (size_t)gridDim.x * blockDim.x) {
    const int y = (int)((r / W) % H);
    if (vec) {      // dy rows: 8 channels = one 16-byte load; U rows: 16 channels = two 16-byte stores, assembled in registers
      float vals[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) vals[i] = 0.f;
      for (int ty = 0; ty < k; ++ty) {
        const int yy = y - (ty - p);
        if (yy < 0 || yy >= H) continue;
        const uint4 d4 = *reinterpret_cast<const uint4*>(dy + (r - (size_t)(ty - p) * W) * 8);
        const float d[4] = {bf16_lo(d4.x), bf16_hi(d4.x), bf16_lo(d4.y), bf16_hi(d4.y)};
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < Co) {
            const int ch = ty * Co + c;
#pragma unroll
            for (int i = 0; i < 16; ++i) vals[i] = (i == ch) ? d[c] : vals[i];
          }
      }
      uint4 a, b;
      a.x = pack_bf16(vals[0], vals[1]); a.y = pack_bf16(vals[2], vals[3]); a.z = pack_bf16(vals[4], vals[5]); a.w = pack_bf16(vals[6], vals[7]);
      b.x = pack_bf16(vals[8], vals[9]); b.y = pack_bf16(vals[10], vals[11]); b.z = pack_bf16(vals[12], vals[13]); b.w = pack_bf16(vals[14], vals[15]);
      uint4* u4 = reinterpret_cast<uint4*>(U + r * 16);
      u4[0] = a; u4[1] = b;
      continue;
    }
    __nv_bfloat16* u = U + r * ld_u;
    int ch = 0;
    for (int ty = 0; ty < k; ++ty) {
      const int yy = y - (ty - p);
      const bool in = yy >= 0 && yy < H;
      const __nv_bfloat16* src = dy + (r - (size_t)(ty - p) * W) * ld_dy;
      for (int c = 0; c < Co; ++c, ++ch) u[ch] = in ? src[c] : __float2bfloat16(0.f);
    }
    for (; ch < ld_u; ++ch) u[ch] = __float2bfloat16(0.f);
  }
}

// ------------------------------------------------------------------------------------------------ fp32 -> bf16 channel slice
// dst (P, C) bf16 = src (P, C) fp32, both with their own leading dimension: a completed slice of a dense block's gradient
// accumulator becomes the bf16 operand of the convolutions' backward
template <int V>
__global__ void __launch_bounds__(NORM_MAX_THREADS) cast_slice_kernel(const float* __restrict__ src, int ld_src,
                                                                      __nv_bfloat16* __restrict__ dst, int ld_dst, size_t P,
                                                                      int nchunk, int ppb) {
  const int chunk = threadIdx.x % nchunk, pl = threadIdx.x / nchunk;
  const size_t step = (size_t)gridDim.x * ppb;
  for (size_t p = (size_t)blockIdx.x * ppb + pl; p < P; p += step) {
    float v[V];
    const float* s = src + p * ld_src + chunk * V;
    if constexpr (V == 8) {
      const float4 x0 = reinterpret_cast<const float4*>(s)[0], x1 = reinterpret_cast<const float4*>(s)[1];
      v[0] = x0.x; v[1] = x0.y; v[2] = x0.z; v[3] = x0.w; v[4] = x1.x; v[5] = x1.y; v[6] = x1.z; v[7] = x1.w;
    } else {
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] = s[j];
    }
    Vec<V>::store(dst + p * ld_dst + chunk * V, v);
  }
}

static bool vec_ok(int C, std::initializer_list<int> lds, std::initializer_list<const void*> ptrs) {
  if (C % 8) return false;
  for (int l : lds) if (l % 8) return false;
  for (const void* p : ptrs) if (p && (reinterpret_cast<uintptr_t>(p) & 15)) return false;
  return true;
}

}  // namespace jvae

using namespace jvae;

// all kernels here are grid-stride: the grid never exceeds what is resident at once (occupancy x SMs), so there is no partial
// second wave of blocks (bn_apply_fwd: 1184 blocks on 740 slots before)
template <typename Kern>
static int resident_grid(Kern kern, int threads, size_t smem, int want) {
  static std::mutex mu;
  static std::unordered_map<uint64_t, int> cache;
  const uint64_t key = (uint64_t)reinterpret_cast<uintptr_t>(reinterpret_cast<const void*>(kern)) ^ ((uint64_t)threads << 48) ^
                       ((uint64_t)smem << 32);
  int occ = 0;
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) occ = it->second;
  }
  if (occ == 0) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem) != cudaSuccess || occ < 1) occ = 1;
    std::lock_guard<std::mutex> lk(mu);
    cache[key] = occ;
  }
  const long long cap = (long long)occ * sm_count();
  return (int)(want < cap ? want : cap);
}

#define NORM_DISPATCH(vec, kernel, geo, smem, st, ...)                                             \
  do {                                                                                             \
    if (vec) kernel<8><<<resident_grid(kernel<8>, geo.threads, smem, geo.grid), geo.threads, smem, st>>>(__VA_ARGS__);   \
    else kernel<1><<<resident_grid(kernel<1>, geo.threads, smem, geo.grid), geo.threads, smem, st>>>(__VA_ARGS__);       \
    JVAE_LAUNCH_CHECK();                                                                           \
  } while (0)

extern "C" {

int jvae_bn_stats(const void* y, size_t P, int C, int ld, double* stats, void* stream) {
  JVAE_CHECK_ARG(y && stats && P > 0 && C > 0 && ld >= C, "bad arguments");
  const bool vec = vec_ok(C, {ld}, {y});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, bn_stats_kernel, g, 2 * C * sizeof(double), (cudaStream_t)stream,
                reinterpret_cast<const __nv_bfloat16*>(y), P, C, ld, g.nchunk, g.ppb, stats, C);
  return JVAE_OK;
}

int jvae_bn_stats_ld(const void* y, size_t P, int C, int ld, double* stats, int stats_ld, void* stream) {
  JVAE_CHECK_ARG(y && stats && P > 0 && C > 0 && ld >= C && stats_ld >= C, "bad arguments");
  const bool vec = vec_ok(C, {ld}, {y});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, bn_stats_kernel, g, 2 * C * sizeof(double), (cudaStream_t)stream,
                reinterpret_cast<const __nv_bfloat16*>(y), P, C, ld, g.nchunk, g.ppb, stats, stats_ld);
  return JVAE_OK;
}

int jvae_bn_apply_fwd(const void* y, size_t P, int C, int ld_y, const double* stats, const float* gamma, const float* beta,
                      float eps, float momentum, float* running_mean, float* running_var, int64_t* num_batches, int training,
                      int act, void* out, int ld_out, float* save_mean_rstd, void* stream) {
  JVAE_CHECK_ARG(y && out && P > 0 && C > 0 && ld_y >= C && ld_out >= C, "bad arguments");
  JVAE_CHECK_ARG(training ? (stats && save_mean_rstd) : (running_mean && running_var), "statistics missing");
  const bool vec = vec_ok(C, {ld_y, ld_out}, {y, out});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  // (a dense 3-channel output row is three 2-byte stores per thread: measured 52 us against 41 us for the generic kernel on the
  // c2 image, so only padded outputs come here)
  const bool narrow = !vec && C < 8 && ld_y == 8 && ld_out == 8 &&
                      ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  BnFwd a;
  a.y = reinterpret_cast<const __nv_bfloat16*>(y); a.out = reinterpret_cast<__nv_bfloat16*>(out);
  a.P = P; a.C = C; a.ld_y = ld_y; a.ld_out = ld_out; a.nchunk = g.nchunk; a.ppb = g.ppb; a.act = act; a.training = training;
  a.sld = C; a.stats = stats; a.gamma = gamma; a.beta = beta; a.running_mean = running_mean; a.running_var = running_var;
  a.num_batches = reinterpret_cast<long long*>(num_batches); a.save = save_mean_rstd; a.eps = eps; a.momentum = momentum;
  if (narrow) {      // a thread per pixel (the image head's BatchNorm)
    const int want = (int)((P + NORM_MAX_THREADS * 4 - 1) / (NORM_MAX_THREADS * 4));
    const int cap = sm_count() * 8;
    bn_apply_fwd_narrow_kernel<<<want < cap ? (want ? want : 1) : cap, NORM_MAX_THREADS, 0, (cudaStream_t)stream>>>(a);
    JVAE_LAUNCH_CHECK();
    return JVAE_OK;
  }
  NORM_DISPATCH(vec, bn_apply_fwd_kernel, g, 0, (cudaStream_t)stream, a);
  return JVAE_OK;
}

int jvae_bn_bwd(const void* da, int ld_da, const void* y, int ld_y, size_t P, int C, const float* save_mean_rstd,
                const float* gamma, const float* beta, int act, double* sums, void* dy, int ld_dy, float* dgamma, float* dbeta,
                void* stream) {
  JVAE_CHECK_ARG(da && y && dy && sums && save_mean_rstd && P > 0 && C > 0, "bad arguments");
  JVAE_CHECK_ARG(ld_da >= C && ld_y >= C && ld_dy >= C, "leading dimension < C");
  const bool vec = vec_ok(C, {ld_da, ld_y, ld_dy}, {da, y, dy});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  BnBwd a = {};
  a.da = reinterpret_cast<const __nv_bfloat16*>(da); a.y = reinterpret_cast<const __nv_bfloat16*>(y);
  a.dy = reinterpret_cast<__nv_bfloat16*>(dy);
  a.P = P; a.C = C; a.ld_da = ld_da; a.ld_y = ld_y; a.ld_dy = ld_dy; a.nchunk = g.nchunk; a.ppb = g.ppb; a.act = act;
  a.save = save_mean_rstd; a.gamma = gamma; a.beta = beta; a.sums = sums; a.dgamma = dgamma; a.dbeta = dbeta;
  const bool narrow = !vec && C < 8 && ld_y == 8 && ld_dy == 8 && (ld_da == 8 || ld_da < 8) &&
                      ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(dy)) & 15) == 0 &&
                      (ld_da != 8 || (reinterpret_cast<uintptr_t>(da) & 15) == 0);
  if (narrow) {      // a thread per pixel (the image head's BatchNorm)
    const int want_r = (int)((P + NORM_MAX_THREADS * 4 - 1) / (NORM_MAX_THREADS * 4));
    const int want_a = (int)((P + NORM_MAX_THREADS * 2 - 1) / (NORM_MAX_THREADS * 2));
    JVAE_CUDA(cudaMemsetAsync(sums, 0, 2 * (size_t)C * sizeof(double), (cudaStream_t)stream));
    const int cap_r = sm_count() * BN_REDUCE_BLOCKS;
    bn_bwd_reduce_narrow_kernel<<<want_r < cap_r ? (want_r ? want_r : 1) : cap_r, NORM_MAX_THREADS, 0, (cudaStream_t)stream>>>(a);
    JVAE_LAUNCH_CHECK();
    const int cap = sm_count() * 8;
    bn_bwd_apply_narrow_kernel<<<want_a < cap ? (want_a ? want_a : 1) : cap, NORM_MAX_THREADS, 0, (cudaStream_t)stream>>>(a);
    JVAE_LAUNCH_CHECK();
    return JVAE_OK;
  }
  JVAE_CUDA(cudaMemsetAsync(sums, 0, 2 * (size_t)C * sizeof(double), (cudaStream_t)stream));
  const Geo gr = make_geo(P, C, vec ? 8 : 1, BN_REDUCE_BLOCKS);     // one resident wave: the per-block reduction tail runs once
  NORM_DISPATCH(vec, bn_bwd_reduce_kernel, gr, 2 * C * sizeof(double), (cudaStream_t)stream, a);
  NORM_DISPATCH(vec, bn_bwd_apply_kernel, g, 0, (cudaStream_t)stream, a);
  return JVAE_OK;
}

int jvae_bn_preact_fwd(const void* y, size_t P, int C, int ld_y, const double* stats, int stats_ld, const float* gamma,
                       const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                       int64_t* num_batches, int training, int act, void* out, int ld_out, float* save_mean_rstd, void* stream) {
  JVAE_CHECK_ARG(y && out && P > 0 && C > 0 && ld_y >= C && ld_out >= C, "bad arguments");
  JVAE_CHECK_ARG(training ? (stats && save_mean_rstd && stats_ld >= C) : (running_mean && running_var), "statistics missing");
  JVAE_CHECK_ARG(vec_ok(C, {ld_y, ld_out}, {y, out}) && C <= 8 * NORM_MAX_THREADS,
                 "pre-activation BatchNorm needs C, ld_y, ld_out multiples of 8 and 16-byte aligned rows");
  const Geo g = make_geo(P, C, 8);
  BnFwd a;
  a.y = reinterpret_cast<const __nv_bfloat16*>(y); a.out = reinterpret_cast<__nv_bfloat16*>(out);
  a.P = P; a.C = C; a.ld_y = ld_y; a.ld_out = ld_out; a.nchunk = g.nchunk; a.ppb = g.ppb; a.act = act; a.training = training;
  a.sld = stats_ld; a.stats = stats; a.gamma = gamma; a.beta = beta; a.running_mean = running_mean; a.running_var = running_var;
  a.num_batches = reinterpret_cast<long long*>(num_batches); a.save = save_mean_rstd; a.eps = eps; a.momentum = momentum;
  NORM_DISPATCH(true, bn_apply_fwd_kernel, g, 0, (cudaStream_t)stream, a);
  return JVAE_OK;
}

int jvae_bn_preact_bwd(const void* da, int ld_da, const void* y, int ld_y, size_t P, int C, const float* save_mean_rstd,
                       const float* gamma, const float* beta, const float* running_mean, const float* running_var, float eps,
                       int training, int act, double* sums, float* dx, int ld_dx, float* dgamma, float* dbeta, void* stream) {
  JVAE_CHECK_ARG(da && y && dx && P > 0 && C > 0 && ld_da >= C && ld_y >= C && ld_dx >= C, "bad arguments");
  JVAE_CHECK_ARG(training ? (sums && save_mean_rstd) : (running_mean && running_var), "statistics missing");
  JVAE_CHECK_ARG(vec_ok(C, {ld_da, ld_y, ld_dx}, {da, y, dx}) && C <= 8 * NORM_MAX_THREADS,
                 "pre-activation BatchNorm needs C and every ld multiples of 8 and 16-byte aligned rows");
  const Geo g = make_geo(P, C, 8);
  BnBwd a = {};
  a.da = reinterpret_cast<const __nv_bfloat16*>(da); a.y = reinterpret_cast<const __nv_bfloat16*>(y);
  a.P = P; a.C = C; a.ld_da = ld_da; a.ld_y = ld_y; a.nchunk = g.nchunk; a.ppb = g.ppb; a.act = act;
  a.save = save_mean_rstd; a.gamma = gamma; a.beta = beta; a.sums = sums; a.dgamma = dgamma; a.dbeta = dbeta;
  a.dxf = dx; a.ld_dxf = ld_dx; a.eval = !training; a.rmean = running_mean; a.rvar = running_var; a.eps = eps;
  if (training) {
    JVAE_CUDA(cudaMemsetAsync(sums, 0, 2 * (size_t)C * sizeof(double), (cudaStream_t)stream));
    const Geo gr = make_geo(P, C, 8, BN_REDUCE_BLOCKS);
    NORM_DISPATCH(true, bn_bwd_reduce_kernel, gr, 2 * C * sizeof(double), (cudaStream_t)stream, a);
  }
  NORM_DISPATCH(true, bn_bwd_apply_kernel, g, 0, (cudaStream_t)stream, a);
  return JVAE_OK;
}

int jvae_cast_f32_bf16_ld(const float* src, int ld_src, void* dst, int ld_dst, size_t P, int C, void* stream) {
  JVAE_CHECK_ARG(src && dst && P > 0 && C > 0 && ld_src >= C && ld_dst >= C, "bad arguments");
  const bool vec = vec_ok(C, {ld_src, ld_dst}, {src, dst});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, cast_slice_kernel, g, 0, (cudaStream_t)stream, src, ld_src, reinterpret_cast<__nv_bfloat16*>(dst), ld_dst,
                P, g.nchunk, g.ppb);
  return JVAE_OK;
}

int jvae_act_bwd(const void* da, int ld_da, const void* a_out, int ld_a, size_t P, int C, int act, void* dy, int ld_dy,
                 float* dbias, void* stream) {
  JVAE_CHECK_ARG(da && P > 0 && C > 0 && ld_da >= C, "bad arguments");
  JVAE_CHECK_ARG(act == JVAE_ACT_NONE || (a_out && ld_a >= C), "activation output missing");
  JVAE_CHECK_ARG(dy || dbias, "nothing to compute");
  const bool vec = vec_ok(C, {ld_da, a_out ? ld_a : 8, dy ? ld_dy : 8}, {da, a_out, dy});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, act_bwd_kernel, g, C * sizeof(double), (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(da),
                ld_da, reinterpret_cast<const __nv_bfloat16*>(a_out), ld_a, P, C, g.nchunk, g.ppb, act,
                reinterpret_cast<__nv_bfloat16*>(dy), ld_dy, dbias);
  return JVAE_OK;
}

int jvae_maxpool_fwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, void* out, int ld_out, void* stream) {
  JVAE_CHECK_ARG(in && out && N > 0 && C > 0 && ld_in >= C && ld_out >= C, "bad arguments");
  JVAE_CHECK_ARG(k >= 1 && stride >= k && H >= k && W >= k, "window must fit and must not overlap (stride >= kernel)");
  const bool vec = vec_ok(C, {ld_in, ld_out}, {in, out});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const int Ho = (H - k) / stride + 1, Wo = (W - k) / stride + 1;
  const size_t Pout = (size_t)N * Ho * Wo;
  const Geo g = make_geo(Pout, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, maxpool_fwd_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(in), H, W, ld_in,
                reinterpret_cast<__nv_bfloat16*>(out), ld_out, Ho, Wo, k, stride, Pout, g.nchunk, g.ppb);
  return JVAE_OK;
}

int jvae_maxpool_bwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, const void* dout, int ld_dout,
                     void* din, int ld_din, void* stream) {
  JVAE_CHECK_ARG(in && dout && din && N > 0 && C > 0, "bad arguments");
  JVAE_CHECK_ARG(k >= 1 && stride >= k && H >= k && W >= k, "window must fit and must not overlap (stride >= kernel)");
  JVAE_CHECK_ARG(ld_in >= C && ld_dout >= C && ld_din >= C, "leading dimension < C");
  const bool vec = vec_ok(C, {ld_in, ld_dout, ld_din}, {in, dout, din});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const int Ho = (H - k) / stride + 1, Wo = (W - k) / stride + 1;
  if (stride > k || (Ho - 1) * stride + k != H || (Wo - 1) * stride + k != W)   // pixels outside every window: no gradient
    JVAE_CUDA(cudaMemsetAsync(din, 0, (size_t)N * H * W * ld_din * 2, (cudaStream_t)stream));
  const size_t Pout = (size_t)N * Ho * Wo;
  const Geo g = make_geo(Pout, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, maxpool_bwd_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(in), H, W, ld_in,
                reinterpret_cast<const __nv_bfloat16*>(dout), ld_dout, reinterpret_cast<__nv_bfloat16*>(din), ld_din, Ho, Wo, k,
                stride, Pout, g.nchunk, g.ppb);
  return JVAE_OK;
}

int jvae_upsample2(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int backward, void* stream) {
  JVAE_CHECK_ARG(src && dst && N > 0 && H > 0 && W > 0 && C > 0 && ld_src >= C && ld_dst >= C, "bad arguments");
  const bool vec = vec_ok(C, {ld_src, ld_dst}, {src, dst});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const size_t Pin = (size_t)N * H * W;
  const Geo g = make_geo(Pin, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, upsample2_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(src), ld_src,
                reinterpret_cast<__nv_bfloat16*>(dst), ld_dst, H, W, Pin, g.nchunk, g.ppb, backward);
  return JVAE_OK;
}

int jvae_maxpool_pad_fwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, int pad, void* out,
                         int ld_out, void* stream) {
  JVAE_CHECK_ARG(in && out && N > 0 && C > 0 && ld_in >= C && ld_out >= C, "bad arguments");
  JVAE_CHECK_ARG(k >= 1 && stride >= 1 && pad >= 0 && 2 * pad <= k && H + 2 * pad >= k && W + 2 * pad >= k, "bad window");
  const bool vec = vec_ok(C, {ld_in, ld_out}, {in, out});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  PoolGeo q{H, W, (H + 2 * pad - k) / stride + 1, (W + 2 * pad - k) / stride + 1, k, stride, pad};
  const size_t Pout = (size_t)N * q.Ho * q.Wo;
  const Geo g = make_geo(Pout, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, maxpool_pad_fwd_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(in), ld_in,
                reinterpret_cast<__nv_bfloat16*>(out), ld_out, q, Pout, g.nchunk, g.ppb);
  return JVAE_OK;
}

int jvae_maxpool_pad_bwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, int pad, const void* dout,
                         int ld_dout, void* din, int ld_din, void* stream) {
  JVAE_CHECK_ARG(in && dout && din && N > 0 && C > 0, "bad arguments");
  JVAE_CHECK_ARG(ld_in >= C && ld_dout >= C && ld_din >= C, "leading dimension < C");
  JVAE_CHECK_ARG(k >= 1 && stride >= 1 && pad >= 0 && 2 * pad <= k && H + 2 * pad >= k && W + 2 * pad >= k, "bad window");
  const bool vec = vec_ok(C, {ld_in, ld_dout, ld_din}, {in, dout, din});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  PoolGeo q{H, W, (H + 2 * pad - k) / stride + 1, (W + 2 * pad - k) / stride + 1, k, stride, pad};
  const size_t Pin = (size_t)N * H * W;
  const Geo g = make_geo(Pin, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, maxpool_pad_bwd_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(in), ld_in,
                reinterpret_cast<const __nv_bfloat16*>(dout), ld_dout, reinterpret_cast<__nv_bfloat16*>(din), ld_din, q, Pin,
                g.nchunk, g.ppb);
  return JVAE_OK;
}

int jvae_avgpool(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int k, int backward,
                 void* stream) {
  JVAE_CHECK_ARG(src && dst && N > 0 && H > 0 && W > 0 && C > 0 && ld_src >= C && ld_dst >= C, "bad arguments");
  JVAE_CHECK_ARG(k >= 1 && H % k == 0 && W % k == 0, "the window must tile the image (stride = kernel)");
  const bool vec = vec_ok(C, {ld_src, ld_dst}, {src, dst});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const size_t Ps = (size_t)N * (H / k) * (W / k);
  const Geo g = make_geo(Ps, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, avgpool_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(src), ld_src,
                reinterpret_cast<__nv_bfloat16*>(dst), ld_dst, H, W, k, Ps, g.nchunk, g.ppb, backward);
  return JVAE_OK;
}

int jvae_upsample_nearest(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int s, int backward,
                          void* stream) {
  JVAE_CHECK_ARG(src && dst && N > 0 && H > 0 && W > 0 && C > 0 && ld_src >= C && ld_dst >= C, "bad arguments");
  JVAE_CHECK_ARG(s >= 1 && (long long)H * s <= (1 << 20) && (long long)W * s <= (1 << 20), "up-sampling factor >= 1, output sides up to 2^20");
  const bool vec = vec_ok(C, {ld_src, ld_dst}, {src, dst});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const size_t P = backward ? (size_t)N * H * W : (size_t)N * H * s * W * s;
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, upsample_nearest_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(src), ld_src,
                reinterpret_cast<__nv_bfloat16*>(dst), ld_dst, H, W, s, P, g.nchunk, g.ppb, backward);
  return JVAE_OK;
}

int jvae_avgpool_pad(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int kh, int kw, int sh, int sw,
                     int ph, int pw, int backward, void* stream) {
  JVAE_CHECK_ARG(src && dst && N > 0 && H > 0 && W > 0 && C > 0 && ld_src >= C && ld_dst >= C, "bad arguments");
  JVAE_CHECK_ARG(kh >= 1 && kw >= 1 && sh >= 1 && sw >= 1 && ph >= 0 && pw >= 0, "bad window");
  JVAE_CHECK_ARG(2 * ph <= kh && 2 * pw <= kw, "padding must be at most half the kernel");
  JVAE_CHECK_ARG(H + 2 * ph >= kh && W + 2 * pw >= kw, "the window is larger than the padded map");
  const bool vec = vec_ok(C, {ld_src, ld_dst}, {src, dst});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  AvgGeo q{H, W, (H + 2 * ph - kh) / sh + 1, (W + 2 * pw - kw) / sw + 1, kh, kw, sh, sw, ph, pw};
  const size_t P = backward ? (size_t)N * H * W : (size_t)N * q.Ho * q.Wo;
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, avgpool_pad_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(src), ld_src,
                reinterpret_cast<__nv_bfloat16*>(dst), ld_dst, q, P, g.nchunk, g.ppb, backward);
  return JVAE_OK;
}

int jvae_vstack_rows(const void* dy, int ld_dy, int N, int H, int W, int k, int pad, int Co, void* U, int ld_u, void* stream) {
  JVAE_CHECK_ARG(dy && U && N > 0 && H > 0 && W > 0, "bad arguments");
  JVAE_CHECK_ARG(k >= 1 && pad >= 0 && Co >= 1 && ld_dy >= Co && ld_u >= k * Co, "bad channel layout");
  const size_t P = (size_t)N * H * W;
  size_t blocks = (P + 255) / 256;
  const size_t cap = (size_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  const bool fixed = ld_dy == 8 && ld_u == 16 && pad == (k - 1) / 2 && (k & 1) &&
                     ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(U)) & 15) == 0;
  const __nv_bfloat16* dp = reinterpret_cast<const __nv_bfloat16*>(dy);
  __nv_bfloat16* up = reinterpret_cast<__nv_bfloat16*>(U);
  cudaStream_t st = (cudaStream_t)stream;
  if (fixed && k == 5 && Co == 3) vstack_rows_fixed_kernel<5, 3><<<resident_grid(vstack_rows_fixed_kernel<5, 3>, 256, 0, (int)blocks), 256, 0, st>>>(dp, N, H, W, up);
  else if (fixed && k == 3 && Co == 3) vstack_rows_fixed_kernel<3, 3><<<resident_grid(vstack_rows_fixed_kernel<3, 3>, 256, 0, (int)blocks), 256, 0, st>>>(dp, N, H, W, up);
  else if (fixed && k == 5 && Co == 1) vstack_rows_fixed_kernel<5, 1><<<resident_grid(vstack_rows_fixed_kernel<5, 1>, 256, 0, (int)blocks), 256, 0, st>>>(dp, N, H, W, up);
  else if (fixed && k == 3 && Co == 1) vstack_rows_fixed_kernel<3, 1><<<resident_grid(vstack_rows_fixed_kernel<3, 1>, 256, 0, (int)blocks), 256, 0, st>>>(dp, N, H, W, up);
  else vstack_rows_kernel<<<(int)blocks, 256, 0, st>>>(dp, ld_dy, N, H, W, k, pad, Co, up, ld_u);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

int jvae_add_act(const void* a, int ld_a, const void* b, int ld_b, size_t P, int C, int act, void* out, int ld_out, void* stream) {
  JVAE_CHECK_ARG(a && b && out && P > 0 && C > 0 && ld_a >= C && ld_b >= C && ld_out >= C, "bad arguments");
  const bool vec = vec_ok(C, {ld_a, ld_b, ld_out}, {a, b, out});
  JVAE_CHECK_ARG(vec ? C <= 8 * NORM_MAX_THREADS : C <= NORM_MAX_THREADS, "too many channels for this layout");
  const Geo g = make_geo(P, C, vec ? 8 : 1);
  NORM_DISPATCH(vec, add_act_kernel, g, 0, (cudaStream_t)stream, reinterpret_cast<const __nv_bfloat16*>(a), ld_a,
                reinterpret_cast<const __nv_bfloat16*>(b), ld_b, reinterpret_cast<__nv_bfloat16*>(out), ld_out, P, act,
                g.nchunk, g.ppb);
  return JVAE_OK;
}

}  // extern "C"
