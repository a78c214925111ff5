// Fused class-conditional prior / ELBO kernels (train forward, train backward, eval/scoring forward).
//
// Replaces the ~30 ATen kernels + host syncs of cvae.py:626-902, module/priors.py:173-342 and
// module/losses.py:8-27,52-86 of the reference by ONE launch per direction (plus a tiny prior-statistics
// prologue).  The kernels are HBM-bound streaming reductions over x_reco (L*D elements per sample) with a
// latent-space epilogue executed by the last CTA that finishes a sample ("last block done" election), so
// neither the (C,B,K) nor the (L,C,B,K) broadcast of the reference is ever materialised.
//
// Work decomposition: one CTA per (sample b, group g of up to LG latent draws).  Each thread keeps 8
// pixels of x in registers and streams the matching 8 pixels of LG reconstructions with 16-byte
// no-allocate loads (LG independent loads in flight per thread), so x is read from HBM once and x_reco
// exactly once.
#include "tc_common.cuh"
#include <math_constants.h>

namespace jvae {

constexpr int ELBO_THREADS = 128;
constexpr float LOG2PI_F = 1.8378770664093453f;

struct ElboArgs {
  int B, L, K, C, Cp, D, G;
  int xr_bf16, lg_bf16, var_dim, prior_kind, conditional, has_xreco, has_logits, sigma_is_log, sigma_is_rmse;
  float beta, gamma_w, var_w, tau, alpha;
  const float* x;
  const void* xr;
  const float* mu;
  const float* lv;
  const float* z;
  const float* eps_norm;
  const void* logits;
  const long long* y;
  const float* means;
  const float* inv_trans;
  const float* sigma;
  const float* g;
  const float* wmse_in;
  // outputs
  float *kl, *zdist, *var_kl, *wmse, *cross_x, *cross_y, *total, *dzdist, *iws, *logits_out, *scores;
  int* preds;
  int* finite_flag;
  void* d_xr;
  float *d_mu, *d_lv, *d_means, *d_inv_trans, *d_sigma;
  void* d_logits;
  // workspace
  unsigned int* counters;   // (B)
  float* dict_norm_var;     // (ceil(K/32)) partial sums written by prior_stats_kernel
  int nkb;
  float* ws_mse;            // (L,B) sum_d (x_reco - x)^2
  float* dict_mean;         // (K)
  float* logdet;            // (Cp)
  float* ws_lat;            // (B,4): kl, cross_y, bad-label flag of the latent CTAs (train forward)
  // var_dim = full (inverse Cholesky T_c, priors.py:146): the main kernels run their diagonal code on
  // tdiag = sqrt(diag(T^T T)) (exact for the trace term) and take the squared distances |T_c (v - m_c)|^2 from full_dist
  // output_distribution = 'categorical' (losses.py:30-49, cvae.py:654-660, 776): 256 logits per pixel; the pre-pass
  // fills ws_mse with sum_d (argmax / 255 - x)^2 and ws_ce with sum_d cross-entropy per (draw, sample)
  int categorical, cat_group;
  int sigma_stride;         // 0: one sigma for the batch; 1: sigma[b] (Sigma coded by the encoder, cvae.py:631-634)
  float* ws_ce;             // (L, B)
  const float* full_T;      // (Cp, K, K) lower-triangular
  float* tdiag;             // (Cp, K)
  float* full_dist;         // train: (B); eval: (L+1, Cp, B)
  float* d_full_T;          // (Cp, K, K) gradient
  // eval with many classes: the cross terms z_r . m_c of the norm-expanded distances come from ONE tcgen05 GEMM (operands split
  // into bf16 hi / lo parts, three products, fp32 accumulation) run before the kernel; cross[(r * B + b) * cross_ld + c]
  const float* cross;
  const float* mnorm;       // (Cp) ||m_c||^2
  int cross_ld;
};

struct WsLayout {
  size_t counters, dnv, zero_bytes, mse, dict_mean, logdet, lat, ce, tdiag, full_dist, tc_a, tc_b, tc_cross, tc_mnorm, total;
  int tc_ld, tc_cpad;
};
// classes from which the eval kernel takes its distances from the tensor-core cross-term GEMM
constexpr int ELBO_TC_MIN_CLASSES = 32;
static bool tc_eligible(int K, int Cp, int var_dim, int prior_kind, int conditional) {
  return conditional && var_dim == JVAE_VAR_SCALAR && prior_kind == JVAE_PRIOR_GAUSSIAN && (K % 8) == 0 && Cp >= ELBO_TC_MIN_CLASSES;
}
static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
static WsLayout ws_layout(int B, int L, int K, int Cp, bool full = false, bool tc = false) {
  WsLayout w;
  w.counters = 0;
  w.zero_bytes = (size_t)B * 4;
  w.dnv = align256(w.zero_bytes);
  w.mse = w.dnv + align256((size_t)((K + 31) / 32) * 4);
  w.dict_mean = w.mse + align256((size_t)(L > 0 ? L : 1) * B * 4);
  w.logdet = w.dict_mean + align256((size_t)K * 4);
  w.lat = w.logdet + align256((size_t)Cp * 4);
  w.ce = w.lat + align256((size_t)B * 16);
  w.tdiag = w.ce + align256((size_t)(L > 0 ? L : 1) * B * 4);
  w.full_dist = w.tdiag + (full ? align256((size_t)Cp * K * 4) : 0);
  w.tc_a = w.full_dist + (full ? align256((size_t)(L + 1) * Cp * B * 4) : 0);
  w.tc_cpad = (Cp + 63) & ~63;                 // rows of the class operand (whole 64-row TMA boxes stay inside the buffer)
  w.tc_ld = (Cp + 3) & ~3;
  const size_t R = (size_t)(L + 1) * B;
  w.tc_b = w.tc_a + (tc ? align256(R * 3 * K * 2) : 0);
  w.tc_cross = w.tc_b + (tc ? align256((size_t)w.tc_cpad * 3 * K * 2) : 0);
  w.tc_mnorm = w.tc_cross + (tc ? align256(R * w.tc_ld * 4) : 0);
  w.total = w.tc_mnorm + (tc ? align256((size_t)Cp * 4) : 0);
  return w;
}

// ------------------------------------------------------------------------------------------------
// prior statistics prologue: dict_mean (K), dict_norm_var, log det Sigma_c (Cp)
//   cvae.py:747-754, priors.py:173-186
// blocks [0, nkb): 32 latent columns each; blocks [nkb, ...): 8 classes each (one warp per class)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) prior_stats_kernel(ElboArgs a, int nkb) {
  __shared__ float s1[8][33], s2[8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if ((int)blockIdx.x < nkb) {
    const int k = blockIdx.x * 32 + lane;
    float sum = 0.f, sq = 0.f;
    if (k < a.K)
      for (int c = w; c < a.Cp; c += 8) {
        float m = a.means[(size_t)c * a.K + k];
        sum += m;
        sq += m * m;
      }
    s1[w][lane] = sum;
    s2[w][lane] = sq;
    __syncthreads();
    if (w == 0) {
      float t1 = 0.f, t2 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { t1 += s1[i][lane]; t2 += s2[i][lane]; }
      float dm = t1 / (float)a.Cp;
      float part = 0.f;
      if (k < a.K) {
        a.dict_mean[k] = dm;
        part = t2 / (float)a.Cp - dm * dm;
      }
      part = warp_sum(part);
      if (lane == 0) a.dict_norm_var[blockIdx.x] = part;   // summed by the consumers (nkb <= 64 partials)
    }
  } else {
    const int c = ((int)blockIdx.x - nkb) * 8 + w;
    if (c >= a.Cp) return;
    float v;
    if (a.var_dim == JVAE_VAR_SCALAR) {
      v = -2.f * (float)a.K * logf(a.inv_trans[c]);
    } else if (a.var_dim == JVAE_VAR_DIAG) {
      float s = 0.f;
      for (int k = lane; k < a.K; k += 32) s += logf(fabsf(a.inv_trans[(size_t)c * a.K + k]));
      v = -2.f * warp_sum(s);
    } else {
      float s = 0.f;
      for (int k = lane; k < a.K; k += 32) s += logf(fabsf(a.inv_trans[((size_t)c * a.K + k) * a.K + k]));
      v = -2.f * warp_sum(s);
    }
    if (lane == 0) a.logdet[c] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// output_distribution = 'categorical' (losses.py:30-49): 256 logits per pixel variable d, target floor(255 x_d).
// Variable d of row r = (l, b) keeps its logits at  r * 256 D + (d / G) * 256 G + v * G + d % G  with G = cat_group:
//   G = channels: the conv imager's channels_last output (channel index v * C + c), x in channels_last order;
//   G = D: the reference's (256, *input_shape) layout, x in NCHW order.
// One thread per variable, online soft-max over v; a CTA reduces its variables and adds once per (l, b).
// ------------------------------------------------------------------------------------------------
template <bool BF16>
__device__ __forceinline__ float cat_load(const void* p, size_t i) {
  return BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]) : reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ int cat_target(float x) {      // (x * 255).long(), losses.py:43
  const int t = (int)(__fmul_rn(x, 255.f));
  return min(max(t, 0), 255);
}

template <bool BF16>
__global__ void __launch_bounds__(256) categorical_fwd_kernel(ElboArgs a) {
  __shared__ float red[32];
  const int row = blockIdx.x;                 // (l - 1) * B + b over the L draws
  const int b = row % a.B;
  const int D = a.D, G = a.cat_group;
  const size_t base = ((size_t)(row + a.B)) * 256 * (size_t)D;      // draw 0 (the mean) carries no loss
  float ce = 0.f, se = 0.f;
  for (int d = blockIdx.y * blockDim.x + threadIdx.x; d < D; d += gridDim.y * blockDim.x) {
    const size_t off = base + (size_t)(d / G) * 256 * G + (d % G);
    const float xv = a.x[(size_t)b * D + d];
    const int tgt = cat_target(xv);
    float m = -CUDART_INF_F, sum = 0.f, best = -CUDART_INF_F, tl = 0.f;
    int arg = 0;
    for (int v = 0; v < 256; ++v) {
      const float val = cat_load<BF16>(a.xr, off + (size_t)v * G);
      if (val > best) { best = val; arg = v; }          // first maximum, like torch.argmax
      if (v == tgt) tl = val;
      const float mn = fmaxf(m, val);
      sum = sum * expf(m - mn) + expf(val - mn);
      m = mn;
    }
    ce += m + logf(sum) - tl;
    const float e = (float)arg / 255.f - xv;
    se = fmaf(e, e, se);
  }
  ce = block_sum(ce, red);
  se = block_sum(se, red);
  if (threadIdx.x == 0) {
    atomicAdd(&a.ws_ce[row], ce);
    atomicAdd(&a.ws_mse[row], se);
  }
}

// d logits = g_b / L (softmax - onehot) for the L draws, zero for draw 0
template <bool BF16>
__global__ void __launch_bounds__(256) categorical_bwd_kernel(ElboArgs a) {
  const int row = blockIdx.x;                 // l * B + b over all L + 1 draws
  const int b = row % a.B, l = row / a.B;
  const int D = a.D, G = a.cat_group;
  const size_t base = (size_t)row * 256 * (size_t)D;
  const float coef = (l == 0) ? 0.f : a.g[b] / (float)a.L;
  for (int d = blockIdx.y * blockDim.x + threadIdx.x; d < D; d += gridDim.y * blockDim.x) {
    const size_t off = base + (size_t)(d / G) * 256 * G + (d % G);
    float m = -CUDART_INF_F, sum = 0.f;
    int tgt = -1;
    if (l > 0) {
      tgt = cat_target(a.x[(size_t)b * D + d]);
      for (int v = 0; v < 256; ++v) {
        const float val = cat_load<BF16>(a.xr, off + (size_t)v * G);
        const float mn = fmaxf(m, val);
        sum = sum * expf(m - mn) + expf(val - mn);
        m = mn;
      }
    }
    const float inv = (l > 0) ? 1.f / sum : 0.f;
    for (int v = 0; v < 256; ++v) {
      float gv = 0.f;
      if (l > 0) gv = coef * (expf(cat_load<BF16>(a.xr, off + (size_t)v * G) - m) * inv - (v == tgt ? 1.f : 0.f));
      if (BF16) reinterpret_cast<__nv_bfloat16*>(a.d_xr)[off + (size_t)v * G] = __float2bfloat16(gv);
      else reinterpret_cast<float*>(a.d_xr)[off + (size_t)v * G] = gv;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// var_dim = full (priors.py:146, 205-212, 237-240): T_c lower-triangular inverse Cholesky factors
// ------------------------------------------------------------------------------------------------
// tdiag[c][k] = sqrt(sum_i T_c[i][k]^2): trace_prod_by_var is then the diagonal formula with T^2 = diag(T^T T)
__global__ void __launch_bounds__(128) full_tdiag_kernel(const float* __restrict__ T, int K, float* __restrict__ tdiag) {
  const int c = blockIdx.x;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float s = 0.f;
    for (int i = k; i < K; ++i) { const float t = T[((size_t)c * K + i) * K + k]; s = fmaf(t, t, s); }
    tdiag[(size_t)c * K + k] = sqrtf(s);
  }
}

// out = |T_c (v_r - m_c)|^2 for 64 row vectors per CTA against class c = blockIdx.y.  T_c passes through shared memory in
// tiles of 32 rows (padded: lane i walks row i without bank conflicts); lane i owns output row i of the product.
// y != null (train): row r belongs to class y[r] only and out is (R); else (eval) out is (R / B, Cp, B).
constexpr int FD_WARPS = 8, FD_RPW = 8;
__global__ void __launch_bounds__(FD_WARPS * 32) full_dist_kernel(const float* __restrict__ T, const float* __restrict__ means,
                                                                  const float* __restrict__ rows, const long long* __restrict__ y,
                                                                  int R, int B, int K, int Cp, int C, float* __restrict__ out) {
  extern __shared__ float s_T[];      // [32][K + 1]
  const int c = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int r_base = blockIdx.x * (FD_WARPS * FD_RPW) + w * FD_RPW;
  float acc[FD_RPW];
  bool mine[FD_RPW];
#pragma unroll
  for (int j = 0; j < FD_RPW; ++j) {
    acc[j] = 0.f;
    const int r = r_base + j;
    mine[j] = r < R;
    if (mine[j] && y) {
      long long yr = y[r];
      if (yr < 0 || yr >= C) yr = 0;
      mine[j] = (Cp == 1) || (int)yr == c;
    }
  }
  const float* m = means + (size_t)c * K;
  for (int i0 = 0; i0 < K; i0 += 32) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < 32 * K; idx += FD_WARPS * 32) {
      const int ii = idx / K, k = idx - ii * K, gi = i0 + ii;
      s_T[ii * (K + 1) + k] = (gi < K && k <= gi) ? T[((size_t)c * K + gi) * K + k] : 0.f;
    }
    __syncthreads();
    const int kmax = min(K, i0 + 32);
    const float* trow = s_T + lane * (K + 1);
#pragma unroll
    for (int j = 0; j < FD_RPW; ++j) {
      if (!mine[j]) continue;      // warp-uniform
      const float* v = rows + (size_t)(r_base + j) * K;
      float sum = 0.f;
      for (int k = 0; k < kmax; ++k) sum = fmaf(trow[k], v[k] - m[k], sum);
      acc[j] = fmaf(sum, sum, acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < FD_RPW; ++j) {
    if (!mine[j]) continue;
    const float d = warp_sum(acc[j]);
    if (lane == 0) {
      const int r = r_base + j;
      if (y) out[r] = d;
      else out[((size_t)(r / B) * Cp + c) * B + (r % B)] = d;
    }
  }
}

// gradients of beta * kl through the distance, the trace and log det of a full T (one CTA per sample):
//   u = T d, d = mu - m:  d_mu += g beta T^T u;  d_m -= the same;  d_T[i][k] += g beta (u_i d_k + w T_ik exp(lv_k) - w [i = k] / T_kk)
__global__ void __launch_bounds__(128) full_prior_bwd_kernel(ElboArgs a) {
  extern __shared__ float s_fb[];      // d[K], u[K]
  float* s_d = s_fb;
  float* s_u = s_fb + a.K;
  const int b = blockIdx.x, K = a.K, tid = threadIdx.x;
  long long yb = a.y[b];
  if (yb < 0 || yb >= a.C) yb = 0;
  const int c = a.conditional ? (int)yb : 0;
  const float coef = a.g[b] * a.beta;
  const float* T = a.full_T + (size_t)c * K * K;
  for (int k = tid; k < K; k += blockDim.x) s_d[k] = a.mu[(size_t)b * K + k] - a.means[(size_t)c * K + k];
  __syncthreads();
  for (int i = tid; i < K; i += blockDim.x) {
    float sum = 0.f;
    for (int k = 0; k <= i; ++k) sum = fmaf(T[(size_t)i * K + k], s_d[k], sum);
    s_u[i] = sum;
  }
  __syncthreads();
  for (int k = tid; k < K; k += blockDim.x) {
    float v = 0.f;
    for (int i = k; i < K; ++i) v = fmaf(T[(size_t)i * K + k], s_u[i], v);
    const float dmu = coef * v;
    if (a.d_mu) a.d_mu[(size_t)b * K + k] += dmu;        // the main backward kernel wrote the other terms
    if (a.d_means) atomicAdd(&a.d_means[(size_t)c * K + k], -dmu);
  }
  if (a.d_full_T) {
    float* dT = a.d_full_T + (size_t)c * K * K;
    for (int idx = tid; idx < K * K; idx += blockDim.x) {
      const int i = idx / K, k = idx - i * K;
      if (k > i) continue;
      const float t = T[idx];
      float val = s_u[i] * s_d[k] + a.var_w * t * expf(a.lv[(size_t)b * K + k]);
      if (i == k) val -= a.var_w / t;
      atomicAdd(&dT[idx], coef * val);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// streaming part: sum_d (x_reco[l,b,d] - x[b,d])^2 for nl <= LG draws starting at l0
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sq_acc8(float& acc, const float4& x0, const float4& x1, const uint4& r) {
  float d;
  d = bf16_lo(r.x) - x0.x; acc = fmaf(d, d, acc);
  d = bf16_hi(r.x) - x0.y; acc = fmaf(d, d, acc);
  d = bf16_lo(r.y) - x0.z; acc = fmaf(d, d, acc);
  d = bf16_hi(r.y) - x0.w; acc = fmaf(d, d, acc);
  d = bf16_lo(r.z) - x1.x; acc = fmaf(d, d, acc);
  d = bf16_hi(r.z) - x1.y; acc = fmaf(d, d, acc);
  d = bf16_lo(r.w) - x1.z; acc = fmaf(d, d, acc);
  d = bf16_hi(r.w) - x1.w; acc = fmaf(d, d, acc);
}
__device__ __forceinline__ void sq_acc4(float& acc, const float4& x0, const uint4& r) {
  float d;
  d = __uint_as_float(r.x) - x0.x; acc = fmaf(d, d, acc);
  d = __uint_as_float(r.y) - x0.y; acc = fmaf(d, d, acc);
  d = __uint_as_float(r.z) - x0.z; acc = fmaf(d, d, acc);
  d = __uint_as_float(r.w) - x0.w; acc = fmaf(d, d, acc);
}

template <bool XR_BF16, int LG>
__device__ __forceinline__ void mse_partial(const ElboArgs& a, int b, int l0, int nl, float (&acc)[LG]) {
  const int D = a.D;
  const float* xb = a.x + (size_t)b * D;
  const size_t slab = (size_t)a.B * D;  // elements per latent draw
#pragma unroll
  for (int j = 0; j < LG; ++j) acc[j] = 0.f;
  const bool vec_ok = XR_BF16 ? ((D & 7) == 0) : ((D & 3) == 0);
  if (vec_ok) {
    if (XR_BF16) {
      const __nv_bfloat16* r0 = reinterpret_cast<const __nv_bfloat16*>(a.xr) + (size_t)l0 * slab + (size_t)b * D;
      const int nvec = D >> 3;
#pragma unroll 2
      for (int v = threadIdx.x; v < nvec; v += ELBO_THREADS) {
        uint4 r[LG];
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) r[j] = ld_stream16(r0 + (size_t)j * slab + (size_t)v * 8);
        const float4 x0 = __ldg(reinterpret_cast<const float4*>(xb) + 2 * v);
        const float4 x1 = __ldg(reinterpret_cast<const float4*>(xb) + 2 * v + 1);
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) sq_acc8(acc[j], x0, x1, r[j]);
      }
    } else {
      const float* r0 = reinterpret_cast<const float*>(a.xr) + (size_t)l0 * slab + (size_t)b * D;
      const int nvec = D >> 2;
#pragma unroll 2
      for (int v = threadIdx.x; v < nvec; v += ELBO_THREADS) {
        uint4 r[LG];
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) r[j] = ld_stream16(r0 + (size_t)j * slab + (size_t)v * 4);
        const float4 x0 = __ldg(reinterpret_cast<const float4*>(xb) + v);
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) sq_acc4(acc[j], x0, r[j]);
      }
    }
  } else {  // ragged D: scalar path
    for (int d = threadIdx.x; d < D; d += ELBO_THREADS) {
      const float xv = xb[d];
#pragma unroll
      for (int j = 0; j < LG; ++j)
        if (j < nl) {
          const size_t idx = (size_t)(l0 + j) * slab + (size_t)b * D + d;
          const float rv = XR_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(a.xr)[idx])
                                   : reinterpret_cast<const float*>(a.xr)[idx];
          const float df = rv - xv;
          acc[j] = fmaf(df, df, acc[j]);
        }
    }
  }
}

// Runs the streaming part for CTA (b, g) and elects the last CTA of sample b.  Returns true in every
// thread of the elected CTA, after which ws_mse[(l-1)*B + b] is complete for all l.
template <bool XR_BF16, int LG>
__device__ __forceinline__ bool stream_and_elect(const ElboArgs& a, int b, int g, float* red, int extra = 0) {
  __shared__ int s_last;
  __shared__ float s_part[ELBO_THREADS / 32][LG];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (a.has_xreco) {
    const int l0 = 1 + g * LG;
    const int nl = min(LG, a.L + 1 - l0);
    float acc[LG];
    mse_partial<XR_BF16, LG>(a, b, l0, nl, acc);
#pragma unroll
    for (int j = 0; j < LG; ++j) {
      const float s = warp_sum(acc[j]);
      if (lane == 0) s_part[wid][j] = s;
    }
    __syncthreads();
    if (threadIdx.x < nl) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < ELBO_THREADS / 32; ++w) s += s_part[w][threadIdx.x];
      a.ws_mse[(size_t)(l0 - 1 + threadIdx.x) * a.B + b] = s;
    }
  }
  if (a.G + extra == 1) {
    __syncthreads();
    return true;
  }
  // last-CTA election: every writer fences its own store, then one thread counts the arrival
  if (threadIdx.x < LG) __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int old = atomicAdd(&a.counters[b], 1u);
    s_last = (old == (unsigned int)(a.G + extra - 1));
    if (s_last) a.counters[b] = 0;   // self-cleaning: the workspace is ready for the next launch
  }
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  return true;
}

__device__ __forceinline__ float load_logit(const void* p, size_t i, int bf16) {
  return bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]) : reinterpret_cast<const float*>(p)[i];
}

// sigma handling of cvae.py:644-670: returns mean_l wmse_l in *wmse, log sigma in *log_sigma and the factor
// that turns a raw sum of squares into wmse_l in *scale  (all threads compute the same values)
__device__ __forceinline__ void sigma_terms(const ElboArgs& a, int b, float* wmse, float* log_sigma, float* scale) {
  float raw = 0.f;
#pragma unroll 8
  for (int l = 0; l < a.L; ++l) raw += __ldcg(&a.ws_mse[(size_t)l * a.B + b]);
  const float mse = raw / ((float)a.L * (float)a.D);
  if (a.categorical) {      // cvae.py:657-660: mse_loss(argmax / 255, x), no division by sigma
    *wmse = mse;
    *log_sigma = 0.f;
    *scale = 1.f / (float)a.D;
  } else if (a.sigma_is_rmse) {
    *wmse = mse / mse;
    *log_sigma = 0.5f * logf(mse);
    *scale = 1.f / ((float)a.D * mse);
  } else {
    const float s = a.sigma[(size_t)a.sigma_stride * b];
    const float sig = a.sigma_is_log ? expf(s) : s;
    *log_sigma = a.sigma_is_log ? s : logf(s);
    *wmse = mse / (sig * sig);
    *scale = 1.f / ((float)a.D * sig * sig);
  }
}

// per-latent-dimension terms of the KL for one (sample, class) pair; accumulates into 3 running sums
//   gaussian: dist += (T d)^2, tr += exp(lv) T^2            (priors.py:188-250)
//   tilted:   dist only                                       (priors.py:389-408)
//   uniform:  dist += d^2, tr += Elogq + neg, aux += Elogq + alpha   (priors.py:429-476)
__device__ __forceinline__ void kl_dim_terms(const ElboArgs& a, float mu, float lv, float m, float T, float& dist,
                                             float& tr, float& aux) {
  const float d = mu - m;
  if (a.prior_kind == JVAE_PRIOR_UNIFORM) {
    const float tau = a.tau, c = LOG2PI_F;
    const float span = 2.f * 1.7320508075688772f * expf(0.5f * lv);
    const float lo = d - 0.5f * span, hi = d + 0.5f * span;
    const float lo_ = tau * fminf(fmaxf(lo / tau, -1.f), 1.f);
    const float hi_ = tau * fminf(fmaxf(hi / tau, -1.f), 1.f);
    const float elogq = -0.5f * lv - 0.5f * 2.4849066497880004f;  // log 12
    float neg = (c + d * d + span * span / 12.f) * 0.5f;
    neg += (a.alpha - 0.5f * c) * (hi_ - lo_) / span;
    neg -= (hi_ * hi_ * hi_ - lo_ * lo_ * lo_) / span / 6.f;
    dist += d * d;
    tr += elogq + neg;
    aux += elogq + a.alpha;
  } else {
    const float w = T * d;
    dist = fmaf(w, w, dist);
    tr = fmaf(expf(lv), T * T, tr);
  }
}

// turns the reduced sums into (kl, zdist, var_kl)
__device__ __forceinline__ void kl_finish(const ElboArgs& a, float dist, float tr, float aux, float slv, float logdet,
                                          float* kl, float* var_kl) {
  if (a.prior_kind == JVAE_PRIOR_TILTED) {
    const float n = sqrtf(dist) - a.tau;
    *kl = 0.5f * n * n;
    *var_kl = 0.f;
  } else if (a.prior_kind == JVAE_PRIOR_UNIFORM) {
    float k = fmaxf(tr, aux);
    if (a.var_w != 1.f) k += (a.var_w - 1.f) * aux;
    *kl = k;
    *var_kl = 2.f * aux;
  } else {
    const float vk = tr - slv + logdet - (float)a.K;
    *var_kl = vk;
    *kl = 0.5f * (dist + a.var_w * vk);
  }
}

// ================================================================================================
// TRAIN FORWARD
// ================================================================================================
// The latent part of a sample (KL to the prior of its class, classifier cross-entropy) does not depend on the
// reconstruction stream, so it runs on its own CTAs (the first ceil(B/4) blocks, one warp per sample) while the other
// CTAs stream x_reco.  Every CTA that finishes a sample's work counts one arrival; the last one (G streaming CTAs + the
// latent warp) combines the two halves: a few scalar operations, so the kernel has no serial latent tail.
__device__ __forceinline__ void train_finalize(const ElboArgs& a, int b) {
  float wmse = 0.f, cross_x = 0.f;
  const bool has_x = a.has_xreco || a.categorical;
  if (has_x) {
    float log_sigma, scale;
    sigma_terms(a, b, &wmse, &log_sigma, &scale);
    cross_x = 0.5f * (float)a.D * (2.f * log_sigma + wmse + LOG2PI_F);
    if (a.categorical) {      // cvae.py:776: cross_x = mean_l sum_d CE
      float ce = 0.f;
      for (int l = 0; l < a.L; ++l) ce += __ldcg(&a.ws_ce[(size_t)l * a.B + b]);
      cross_x = ce / (float)a.L;
    }
  }
  const float kl = __ldcg(&a.ws_lat[4 * b]), cross_y = __ldcg(&a.ws_lat[4 * b + 1]);
  const bool bad_label = __ldcg(&a.ws_lat[4 * b + 2]) != 0.f;
  float total = a.beta * kl;
  if (has_x) total += cross_x;
  if (a.has_logits && a.gamma_w != 0.f) total += a.gamma_w * cross_y;
  if (a.wmse && has_x) a.wmse[b] = wmse;
  if (a.cross_x && has_x) a.cross_x[b] = cross_x;
  if (a.total) a.total[b] = total;
  if (a.finite_flag && (bad_label || !isfinite(total))) atomicExch(a.finite_flag, 0);
}

__device__ __forceinline__ void train_latent_warp(const ElboArgs& a, int b, int lane) {
  const int K = a.K, C = a.C;
  long long yb = a.y[b];
  const bool bad_label = (yb < 0 || yb >= C);
  if (bad_label) yb = 0;
  const int c = a.conditional ? (int)yb : 0;
  // ---- KL to the prior of class y_b (priors.py:252-326)
  float dist = 0.f, tr = 0.f, aux = 0.f, slv = 0.f, dzd = 0.f;
  const float Tc = (a.var_dim == JVAE_VAR_SCALAR) ? a.inv_trans[c] : 0.f;
#pragma unroll 4
  for (int k = lane; k < K; k += 32) {
    const float mu = a.mu[(size_t)b * K + k], lv = a.lv[(size_t)b * K + k];
    const float m = a.means[(size_t)c * K + k];
    const float T = (a.var_dim == JVAE_VAR_SCALAR) ? Tc : a.inv_trans[(size_t)c * K + k];
    kl_dim_terms(a, mu, lv, m, T, dist, tr, aux);
    slv += lv;
    if (a.conditional) {
      const float dd = mu - a.dict_mean[k];
      dzd = fmaf(dd, dd, dzd);
    }
  }
  dist = warp_sum(dist); tr = warp_sum(tr); aux = warp_sum(aux); slv = warp_sum(slv); dzd = warp_sum(dzd);
  if (a.full_dist) dist = a.full_dist[b];
  float kl, var_kl;
  kl_finish(a, dist, tr, aux, slv, a.logdet[c], &kl, &var_kl);
  // ---- cross entropy of the classifier over all L+1 draws (losses.py:73-86)
  float cross_y = 0.f;
  if (a.has_logits) {
    for (int r = 0; r <= a.L; ++r) {
      const size_t base = ((size_t)r * a.B + b) * C;
      float mx = -CUDART_INF_F;
      for (int j = lane; j < C; j += 32) mx = fmaxf(mx, load_logit(a.logits, base + j, a.lg_bf16));
      mx = warp_max(mx);
      float se = 0.f;
      for (int j = lane; j < C; j += 32) se += expf(load_logit(a.logits, base + j, a.lg_bf16) - mx);
      se = warp_sum(se);
      cross_y += logf(se) + mx - load_logit(a.logits, base + (size_t)yb, a.lg_bf16);
    }
    cross_y /= (float)(a.L + 1);
  }
  if (lane == 0) {
    if (a.kl) a.kl[b] = kl;
    if (a.zdist) a.zdist[b] = dist;
    if (a.var_kl) a.var_kl[b] = var_kl;
    if (a.cross_y && a.has_logits) a.cross_y[b] = cross_y;
    if (a.dzdist && a.conditional) {
      float dnv = 0.f;
      for (int i = 0; i < a.nkb; ++i) dnv += a.dict_norm_var[i];
      a.dzdist[b] = dzd + dnv;
    }
    a.ws_lat[4 * b] = kl; a.ws_lat[4 * b + 1] = cross_y; a.ws_lat[4 * b + 2] = bad_label ? 1.f : 0.f;
    bool last = true;
    if (a.has_xreco) {       // G streaming CTAs also arrive on this sample
      unsigned int old;
      asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(&a.counters[b]) : "memory");
      last = (old == (unsigned int)a.G);
      if (last) a.counters[b] = 0;
    }
    if (last) train_finalize(a, b);
  }
}

template <bool XR_BF16, int LG>
__global__ void __launch_bounds__(ELBO_THREADS, LG <= 4 ? 12 : 8) elbo_train_fwd_kernel(ElboArgs a) {
  __shared__ float red[32];
  const int nlat = (a.B + ELBO_THREADS / 32 - 1) / (ELBO_THREADS / 32);
  if ((int)blockIdx.x < nlat) {
    const int b = (int)blockIdx.x * (ELBO_THREADS / 32) + (threadIdx.x >> 5);
    if (b < a.B) train_latent_warp(a, b, threadIdx.x & 31);
    return;
  }
  // streaming CTAs: when the items (sample, group of draws) exceed one resident wave, every CTA takes the same number of
  // items in turn instead of leaving a partial second wave (the host sizes the grid: items / ceil(items / wave))
  const int nstream = (int)gridDim.x - nlat, items = a.B * a.G;
  for (int sid = (int)blockIdx.x - nlat; sid < items; sid += nstream) {
    const int b = sid % a.B, g = sid / a.B;   // b fastest: neighbouring CTAs stream neighbouring rows
    const bool last = stream_and_elect<XR_BF16, LG>(a, b, g, red, 1);
    if (last && threadIdx.x == 0) train_finalize(a, b);
    __syncthreads();                          // the election's shared state is reused by the next item
  }
}

// ------------------------------------------------------------------------------------------------
// Train forward, register-staged streaming (bf16 reconstructions, D a multiple of 8): ONE item (sample b, LG draws) per CTA and
// every load of U vector rounds issued before the first use (U * LG 16-byte x_reco loads + 2 U x loads in flight per thread:
// at c2, D = 3072 = 3 * 128 vectors, the whole item is one memory round trip).  The warp partials meet in shared memory;
// thread 0 alone adds them in a fixed order (deterministic), publishes ws_mse, counts the sample's arrival with one
// acq_rel atomic and, if it is the last of the sample's G + 1 arrivals, finalises: one barrier per CTA, no fence / barrier chain.
// ------------------------------------------------------------------------------------------------
template <int LG, int U, int MINB>
__global__ void __launch_bounds__(ELBO_THREADS, MINB) elbo_train_fwd_v2_kernel(ElboArgs a) {
  __shared__ float s_part[ELBO_THREADS / 32][LG];
  const int nlat = (a.B + ELBO_THREADS / 32 - 1) / (ELBO_THREADS / 32);
  if ((int)blockIdx.x < nlat) {
    const int b = (int)blockIdx.x * (ELBO_THREADS / 32) + (threadIdx.x >> 5);
    if (b < a.B) train_latent_warp(a, b, threadIdx.x & 31);
    return;
  }
  const int sid = (int)blockIdx.x - nlat;
  const int b = sid % a.B, g = sid / a.B;
  const int D = a.D, nvec = D >> 3;
  const int l0 = 1 + g * LG, nl = min(LG, a.L + 1 - l0);
  const size_t slab = (size_t)a.B * D;
  const __nv_bfloat16* r0 = reinterpret_cast<const __nv_bfloat16*>(a.xr) + (size_t)l0 * slab + (size_t)b * D;
  const float4* xb = reinterpret_cast<const float4*>(a.x + (size_t)b * D);
  float acc[LG];
#pragma unroll
  for (int j = 0; j < LG; ++j) acc[j] = 0.f;
  for (int v0 = threadIdx.x; v0 < nvec; v0 += U * ELBO_THREADS) {
    uint4 r[U][LG];
    float4 x0[U], x1[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int v = v0 + u * ELBO_THREADS;
#pragma unroll
      for (int j = 0; j < LG; ++j)
        if (v < nvec && j < nl) r[u][j] = ld_stream16(r0 + (size_t)j * slab + (size_t)v * 8);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int v = v0 + u * ELBO_THREADS;
      if (v < nvec) { x0[u] = __ldg(xb + 2 * v); x1[u] = __ldg(xb + 2 * v + 1); }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int v = v0 + u * ELBO_THREADS;
#pragma unroll
      for (int j = 0; j < LG; ++j)
        if (v < nvec && j < nl) sq_acc8(acc[j], x0[u], x1[u], r[u][j]);
    }
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < LG; ++j) {
    const float t = warp_sum(acc[j]);
    if (lane == 0) s_part[wid][j] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int j = 0; j < nl; ++j) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < ELBO_THREADS / 32; ++w) t += s_part[w][j];
      a.ws_mse[(size_t)(l0 - 1 + j) * a.B + b] = t;
    }
    unsigned int old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(&a.counters[b]) : "memory");
    if (old == (unsigned int)a.G) {       // G streaming CTAs + the latent warp
      a.counters[b] = 0;
      train_finalize(a, b);
    }
  }
}

// ================================================================================================
// TRAIN BACKWARD  (SURVEY.md §8a backward contract)
// ================================================================================================
template <bool XR_BF16, int LG>
__global__ void __launch_bounds__(ELBO_THREADS) elbo_train_bwd_kernel(ElboArgs a) {
  const int b = blockIdx.x % a.B, g = blockIdx.x / a.B;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const float gb = a.g[b];
  const int D = a.D, K = a.K, C = a.C;
  float sig = 1.f;
  if (a.has_xreco && a.sigma_is_rmse) {
    // sigma^2 := this sample's mean squared error (cvae.py:662-670); it is not detached in the reference, but wmse = mse / sigma^2
    // is then constant and cross_x = D/2 (log mse + 1 + log 2pi): d/dx_reco = (x_reco - x) / (L mse), the usual formula with
    // sigma^2 = mse.  The caller passes cross_x in the wmse slot: mse = exp(2 cross_x / D - 1 - log 2pi).
    sig = expf(a.wmse_in[b] / (float)D - 0.5f - 0.5f * LOG2PI_F);
  } else if (a.has_xreco) {
    const float s = a.sigma[(size_t)a.sigma_stride * b];
    sig = a.sigma_is_log ? expf(s) : s;
  }
  // ---- d x_reco[l,b,:] = g_b (x_reco - x) / (L sigma^2), l >= 1; slab 0 gets zeros
  if (a.has_xreco && a.d_xr) {
    const float coef = gb / ((float)a.L * sig * sig);
    const int l0 = 1 + g * LG;
    const int nl = min(LG, a.L + 1 - l0);
    const size_t slab = (size_t)a.B * D;
    const float* xb = a.x + (size_t)b * D;
    const bool vec_ok = XR_BF16 ? ((D & 7) == 0) : ((D & 3) == 0);
    if (vec_ok && XR_BF16) {
      const __nv_bfloat16* r0 = reinterpret_cast<const __nv_bfloat16*>(a.xr) + (size_t)l0 * slab + (size_t)b * D;
      __nv_bfloat16* o0 = reinterpret_cast<__nv_bfloat16*>(a.d_xr) + (size_t)l0 * slab + (size_t)b * D;
      const int nvec = D >> 3;
      for (int v = tid; v < nvec; v += ELBO_THREADS) {
        uint4 r[LG];
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) r[j] = ld_stream16(r0 + (size_t)j * slab + (size_t)v * 8);
        const float4 x0 = __ldg(reinterpret_cast<const float4*>(xb) + 2 * v);
        const float4 x1 = __ldg(reinterpret_cast<const float4*>(xb) + 2 * v + 1);
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) {
            uint4 o;
            o.x = pack_bf16(coef * (bf16_lo(r[j].x) - x0.x), coef * (bf16_hi(r[j].x) - x0.y));
            o.y = pack_bf16(coef * (bf16_lo(r[j].y) - x0.z), coef * (bf16_hi(r[j].y) - x0.w));
            o.z = pack_bf16(coef * (bf16_lo(r[j].z) - x1.x), coef * (bf16_hi(r[j].z) - x1.y));
            o.w = pack_bf16(coef * (bf16_lo(r[j].w) - x1.z), coef * (bf16_hi(r[j].w) - x1.w));
            st_stream16(o0 + (size_t)j * slab + (size_t)v * 8, o);
          }
        if (g == 0) st_stream16(reinterpret_cast<__nv_bfloat16*>(a.d_xr) + (size_t)b * D + (size_t)v * 8, make_uint4(0, 0, 0, 0));
      }
    } else if (vec_ok) {
      const float* r0 = reinterpret_cast<const float*>(a.xr) + (size_t)l0 * slab + (size_t)b * D;
      float* o0 = reinterpret_cast<float*>(a.d_xr) + (size_t)l0 * slab + (size_t)b * D;
      const int nvec = D >> 2;
      for (int v = tid; v < nvec; v += ELBO_THREADS) {
        uint4 r[LG];
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) r[j] = ld_stream16(r0 + (size_t)j * slab + (size_t)v * 4);
        const float4 x0 = __ldg(reinterpret_cast<const float4*>(xb) + v);
#pragma unroll
        for (int j = 0; j < LG; ++j)
          if (j < nl) {
            uint4 o;
            o.x = __float_as_uint(coef * (__uint_as_float(r[j].x) - x0.x));
            o.y = __float_as_uint(coef * (__uint_as_float(r[j].y) - x0.y));
            o.z = __float_as_uint(coef * (__uint_as_float(r[j].z) - x0.z));
            o.w = __float_as_uint(coef * (__uint_as_float(r[j].w) - x0.w));
            st_stream16(o0 + (size_t)j * slab + (size_t)v * 4, o);
          }
        if (g == 0) st_stream16(reinterpret_cast<float*>(a.d_xr) + (size_t)b * D + (size_t)v * 4, make_uint4(0, 0, 0, 0));
      }
    } else {
      for (int d = tid; d < D; d += ELBO_THREADS) {
        const float xv = xb[d];
        for (int j = 0; j < nl; ++j) {
          const size_t idx = (size_t)(l0 + j) * slab + (size_t)b * D + d;
          if (XR_BF16) {
            const float rv = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(a.xr)[idx]);
            reinterpret_cast<__nv_bfloat16*>(a.d_xr)[idx] = __float2bfloat16(coef * (rv - xv));
          } else {
            reinterpret_cast<float*>(a.d_xr)[idx] = coef * (reinterpret_cast<const float*>(a.xr)[idx] - xv);
          }
        }
        if (g == 0) {
          if (XR_BF16) reinterpret_cast<__nv_bfloat16*>(a.d_xr)[(size_t)b * D + d] = __float2bfloat16(0.f);
          else reinterpret_cast<float*>(a.d_xr)[(size_t)b * D + d] = 0.f;
        }
      }
    }
  }
  if (g != 0) return;

  // ---- latent-space gradients, once per sample
  long long yb = a.y[b];
  if (yb < 0 || yb >= C) yb = 0;
  const int c = a.conditional ? (int)yb : 0;
  if (a.has_xreco && a.d_sigma && !a.sigma_is_rmse && tid == 0) {
    // cross_x = D/2 (2 log sigma + wmse + log 2pi), wmse ~ sigma^-2
    float ds = gb * (float)D * (1.f - a.wmse_in[b]);
    if (!a.sigma_is_log) ds /= sig;
    atomicAdd(&a.d_sigma[(size_t)a.sigma_stride * b], ds);
  }
  const float Tc = (a.var_dim == JVAE_VAR_SCALAR) ? a.inv_trans[c] : 0.f;
  float tilt = 1.f;
  if (a.prior_kind == JVAE_PRIOR_TILTED) {
    __shared__ float red[32];
    float dist = 0.f;
    for (int k = tid; k < K; k += ELBO_THREADS) {
      const float w = Tc * (a.mu[(size_t)b * K + k] - a.means[(size_t)c * K + k]);
      dist = fmaf(w, w, dist);
    }
    dist = block_sum(dist, red);
    const float n = sqrtf(dist);
    tilt = (n > 0.f) ? (n - a.tau) / n : 0.f;
  }
  // uniform-with-gaussian-tail prior (priors.py:429-476): kl = max(sum_k (Elogq + neg), sum_k (Elogq + alpha)) [+ (w - 1) aux];
  // the max is taken on the sums, so the branch is per sample
  bool uni_first = true;
  if (a.prior_kind == JVAE_PRIOR_UNIFORM) {
    __shared__ float red_u[32];
    float dist = 0.f, tr = 0.f, aux = 0.f;
    for (int k = tid; k < K; k += ELBO_THREADS)
      kl_dim_terms(a, a.mu[(size_t)b * K + k], a.lv[(size_t)b * K + k], a.means[(size_t)c * K + k], 1.f, dist, tr, aux);
    tr = block_sum(tr, red_u);
    aux = block_sum(aux, red_u);
    uni_first = tr >= aux;      // torch.max(a, b) back-propagates into a where a >= b (ties: half each; measure-zero here)
  }
  for (int k = tid; k < K; k += ELBO_THREADS) {
    const float mu = a.mu[(size_t)b * K + k], lv = a.lv[(size_t)b * K + k];
    const float m = a.means[(size_t)c * K + k];
    const float T = (a.var_dim == JVAE_VAR_SCALAR) ? Tc : a.inv_trans[(size_t)c * K + k];
    const float t2 = T * T;
    float dmu, dlv;
    if (a.prior_kind == JVAE_PRIOR_UNIFORM) {
      // d/d(mu - m) and d/d(log_var) of Elogq + neg (first branch) or of Elogq + alpha (second branch, and the (w - 1) term)
      const float d = mu - m, tau = a.tau, A = a.alpha - 0.5f * LOG2PI_F;
      const float span = 2.f * 1.7320508075688772f * expf(0.5f * lv);
      const float lo = d - 0.5f * span, hi = d + 0.5f * span;
      const float lo_ = tau * fminf(fmaxf(lo / tau, -1.f), 1.f), hi_ = tau * fminf(fmaxf(hi / tau, -1.f), 1.f);
      const float dlo = (fabsf(lo) < tau) ? 1.f : 0.f, dhi = (fabsf(hi) < tau) ? 1.f : 0.f;      // hardtanh slopes
      const float neg_d = d + A * (dhi - dlo) / span - (hi_ * hi_ * dhi - lo_ * lo_ * dlo) / (2.f * span);
      const float neg_lv = span * span / 24.f + A * ((dhi + dlo) * 0.25f - (hi_ - lo_) / (2.f * span))
                           - ((hi_ * hi_ * dhi + lo_ * lo_ * dlo) * 0.125f - (hi_ * hi_ * hi_ - lo_ * lo_ * lo_) / (12.f * span));
      const float gk = gb * a.beta;
      dmu = uni_first ? gk * neg_d : 0.f;
      dlv = gk * ((uni_first ? neg_lv - 0.5f : -0.5f) + (a.var_w - 1.f) * -0.5f);
    } else if (a.prior_kind == JVAE_PRIOR_TILTED) {
      dmu = gb * a.beta * tilt * t2 * (mu - m);
      dlv = 0.f;
    } else {
      dmu = a.full_T ? 0.f : gb * a.beta * t2 * (mu - m);      // full T: full_prior_bwd_kernel adds T^T T (mu - m)
      dlv = gb * a.beta * 0.5f * a.var_w * (t2 * expf(lv) - 1.f);
    }
    if (a.d_mu) a.d_mu[(size_t)b * K + k] = dmu;
    if (a.d_lv) a.d_lv[(size_t)b * K + k] = dlv;
    if (a.d_means && !a.full_T) atomicAdd(&a.d_means[(size_t)c * K + k], -dmu);
    if (a.d_inv_trans && a.var_dim == JVAE_VAR_DIAG && a.prior_kind == JVAE_PRIOR_GAUSSIAN) {
      // d/dT of 1/2 [ T^2 d^2 + w (exp(lv) T^2 - 2 log|T|) ]
      const float d = mu - m;
      atomicAdd(&a.d_inv_trans[(size_t)c * K + k], gb * a.beta * (T * d * d + a.var_w * (expf(lv) * T - 1.f / T)));
    }
  }
  // ---- d logits = g gamma_w/(L+1) (softmax - onehot) for all L+1 draws
  if (a.has_logits && a.d_logits) {
    const float coef = (a.gamma_w != 0.f) ? gb * a.gamma_w / (float)(a.L + 1) : 0.f;
    for (int r = wid; r <= a.L; r += ELBO_THREADS / 32) {
      const size_t base = ((size_t)r * a.B + b) * C;
      float mx = -CUDART_INF_F;
      for (int j = lane; j < C; j += 32) mx = fmaxf(mx, load_logit(a.logits, base + j, a.lg_bf16));
      mx = warp_max(mx);
      float se = 0.f;
      for (int j = lane; j < C; j += 32) se += expf(load_logit(a.logits, base + j, a.lg_bf16) - mx);
      se = warp_sum(se);
      const float inv = 1.f / se;
      for (int j = lane; j < C; j += 32) {
        const float p = expf(load_logit(a.logits, base + j, a.lg_bf16) - mx) * inv;
        const float v = coef * (p - ((long long)j == yb ? 1.f : 0.f));
        if (a.lg_bf16) reinterpret_cast<__nv_bfloat16*>(a.d_logits)[base + j] = __float2bfloat16(v);
        else reinterpret_cast<float*>(a.d_logits)[base + j] = v;
      }
    }
  }
}

// ================================================================================================
// EVAL / SCORING FORWARD: losses for every class, importance-weighted score, logits, OOD scores, predictions
// ================================================================================================
__device__ __forceinline__ float block_max(float v, float* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : -CUDART_INF_F;
  return warp_max(r);
}

// first index attaining `target` (ties -> smallest index, like torch.argmax / argmin)
__device__ __forceinline__ int block_first_index(const float* v, int n, float target, int* red_i) {
  int best = 0x7fffffff;
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (v[i] == target) best = min(best, i);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) red_i[wid] = best;
  __syncthreads();
  int r = (lane < nw) ? red_i[lane] : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) r = min(r, __shfl_xor_sync(0xffffffffu, r, o));
  return r;
}

// Operands of the cross-term GEMM (eval with many classes).  A value v is split as hi = bf16(v), lo = bf16(v - hi); rows of
// the sample operand hold [hi | lo | hi], rows of the class operand [hi | hi | lo], so one bf16 GEMM over 3K columns returns
// hi.hi + lo.hi + hi.lo (the dropped lo.lo term is 2^-16 of a product).  blockIdx.x < R: row r * B + b of (mu; z[1..L]);
// then one block per class, which also leaves ||m_c||^2 in fp32.
__global__ void __launch_bounds__(128) dist_split_kernel(const float* __restrict__ mu, const float* __restrict__ z,
                                                         const float* __restrict__ means, int R, int B, int K, int Cp,
                                                         __nv_bfloat16* __restrict__ xa, __nv_bfloat16* __restrict__ xb,
                                                         float* __restrict__ mnorm) {
  __shared__ float red[32];
  const int row = blockIdx.x;
  const bool is_class = row >= R;
  const float* src = is_class ? means + (size_t)(row - R) * K : (row < B ? mu + (size_t)row * K : z + (size_t)row * K);
  __nv_bfloat16* dst = is_class ? xb + (size_t)(row - R) * 3 * K : xa + (size_t)row * 3 * K;
  float nrm = 0.f;
  for (int k = threadIdx.x; k < K; k += 128) {
    const float v = src[k];
    const __nv_bfloat16 hi = __float2bfloat16(v);
    const __nv_bfloat16 lo = __float2bfloat16(v - __bfloat162float(hi));
    dst[k] = hi;
    dst[K + k] = is_class ? hi : lo;
    dst[2 * K + k] = is_class ? lo : hi;
    nrm = fmaf(v, v, nrm);
  }
  if (is_class) {
    nrm = block_sum(nrm, red);
    if (threadIdx.x == 0) mnorm[row - R] = nrm;
  }
}

template <bool XR_BF16, int LG>
__global__ void __launch_bounds__(ELBO_THREADS) elbo_eval_fwd_kernel(ElboArgs a) {
  extern __shared__ float sm[];
  __shared__ float red[32];
  __shared__ int red_i[32];
  const int b = blockIdx.x % a.B, g = blockIdx.x / a.B;
  if (!stream_and_elect<XR_BF16, LG>(a, b, g, red)) return;

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int K = a.K, C = a.C, Cp = a.Cp, L = a.L, B = a.B;
  // dynamic shared memory carve-up
  float* zs = sm;                       // (L+1, K): row 0 = mu, rows 1..L = z[1..L]
  float* evar = zs + (size_t)(L + 1) * K;  // (K) log_var
  float* base_l = evar + K;             // (L) per-draw class-independent part of log_iws
  float* s_kl = base_l + L;             // (Cp)
  float* s_zd = s_kl + Cp;              // (Cp)
  float* s_vk = s_zd + Cp;              // (Cp)
  float* s_iws = s_vk + Cp;             // (Cp)
  float* s_tot = s_iws + Cp;            // (max(C,Cp))
  float* s_lo = s_tot + max(C, Cp);     // (C) mean logits
  float* s_cy = s_lo + C;               // (C) cross_y per class
  float* s_li = s_cy + C;               // (warps, L) log importance weights of the class a warp works on
  float* s_zn = s_li + (size_t)(ELBO_THREADS / 32) * L;   // (L+1) squared norms of mu and of the draws (fast path)

  for (int k = tid; k < K; k += ELBO_THREADS) {
    zs[k] = a.mu[(size_t)b * K + k];
    evar[k] = a.lv[(size_t)b * K + k];
  }
  if (a.z)
    for (int i = tid; i < L * K; i += ELBO_THREADS) {
      const int l = i / K, k = i - l * K;
      zs[(size_t)(l + 1) * K + k] = a.z[((size_t)(l + 1) * B + b) * K + k];
    }
  __syncthreads();

  // ---- per-sample scalars
  float slv = 0.f, dzd = 0.f;
  for (int k = tid; k < K; k += ELBO_THREADS) {
    slv += evar[k];
    if (a.conditional) {
      const float dd = zs[k] - a.dict_mean[k];
      dzd = fmaf(dd, dd, dzd);
    }
  }
  slv = block_sum(slv, red);
  dzd = block_sum(dzd, red);

  float wmse = 0.f, cross_x = 0.f, log_sigma = 0.f, scale = 0.f;
  const bool has_x = a.has_xreco || a.categorical;
  const bool do_iws = has_x && a.z && a.eps_norm;
  if (has_x) {
    sigma_terms(a, b, &wmse, &log_sigma, &scale);
    cross_x = 0.5f * (float)a.D * (2.f * log_sigma + wmse + LOG2PI_F);
    if (a.categorical) {
      float ce = 0.f;
      for (int l = 0; l < L; ++l) ce += __ldcg(&a.ws_ce[(size_t)l * B + b]);
      cross_x = ce / (float)L;
    }
    if (do_iws)
      for (int l = tid; l < L; l += ELBO_THREADS) {
        const float wl = __ldcg(&a.ws_mse[(size_t)l * B + b]) * scale;
        // cvae.py:676-683 and 837-850
        float v = -0.5f * (float)a.D * (wl + 2.f * log_sigma + LOG2PI_F);
        if (a.categorical) v = -__ldcg(&a.ws_ce[(size_t)l * B + b]);      // cvae.py:683: log_iws = -CE
        v += 0.5f * (a.eps_norm[(size_t)l * B + b] + slv) + 0.5f * (float)K * LOG2PI_F;
        base_l[l] = v;
      }
  }
  __syncthreads();

  // ---- logits: mean over draws 1..L, and per-class cross_y = -mean_l log(softmax_l + 1e-6)  (losses.py:62-71)
  if (a.has_logits) {
    for (int j = tid; j < C; j += ELBO_THREADS) { s_lo[j] = 0.f; s_cy[j] = 0.f; }
    __syncthreads();
    const int r0 = (L >= 1) ? 1 : 0, nr = (L >= 1) ? L : 1;
    for (int r = r0 + wid; r < r0 + nr; r += ELBO_THREADS / 32) {
      const size_t base = ((size_t)r * B + b) * C;
      float mx = -CUDART_INF_F;
      for (int j = lane; j < C; j += 32) mx = fmaxf(mx, load_logit(a.logits, base + j, a.lg_bf16));
      mx = warp_max(mx);
      float se = 0.f;
      for (int j = lane; j < C; j += 32) se += expf(load_logit(a.logits, base + j, a.lg_bf16) - mx);
      se = warp_sum(se);
      const float inv = 1.f / se;
      for (int j = lane; j < C; j += 32) {
        const float v = load_logit(a.logits, base + j, a.lg_bf16);
        atomicAdd(&s_lo[j], v);
        atomicAdd(&s_cy[j], logf(expf(v - mx) * inv + 1e-6f));
      }
    }
    __syncthreads();
    for (int j = tid; j < C; j += ELBO_THREADS) {
      s_lo[j] = s_lo[j] / (float)nr;
      s_cy[j] = -s_cy[j] / (float)nr;
    }
    __syncthreads();
  }

  // ---- fast class loop (Gaussian prior, scalar variance, K <= 256: the default model).  ||T(z - m)||^2 is expanded as
  // T^2 (||z||^2 - 2 z.m + ||m||^2): per class only the L+1 dot products z_l . m_c remain (class mean in registers, 8
  // latent dims per lane, four rows reduced at a time), ||z_l||^2 and sum exp(log_var) are per-sample scalars.
  const bool fast = a.var_dim == JVAE_VAR_SCALAR && a.prior_kind == JVAE_PRIOR_GAUSSIAN && (K <= 256 || a.cross);
  if (fast) {
    for (int r = wid; r <= (do_iws ? L : 0); r += ELBO_THREADS / 32) {
      float t = 0.f;
      for (int k = lane; k < K; k += 32) { const float v = zs[(size_t)r * K + k]; t = fmaf(v, v, t); }
      t = warp_sum(t);
      if (lane == 0) s_zn[r] = t;
    }
    float sexp = 0.f;
    for (int k = tid; k < K; k += ELBO_THREADS) sexp += expf(evar[k]);
    sexp = block_sum(sexp, red);       // contains the __syncthreads that publishes s_zn
    const int nrows = do_iws ? L + 1 : 1;
    // many classes: one THREAD per class, the dot products z_r . m_c read from the tensor-core GEMM's output (consecutive
    // classes = consecutive addresses); the log importance weights are evaluated twice (max, then sum) instead of staged
    for (int c = tid; c < (a.cross ? Cp : 0); c += ELBO_THREADS) {
      const float Tc = a.inv_trans[c], T2 = Tc * Tc, logdet = a.logdet[c], mn = a.mnorm[c];
      const float* cr = a.cross + (size_t)b * a.cross_ld + c;
      const size_t rs = (size_t)B * a.cross_ld;
      const float dist = fmaxf(T2 * (s_zn[0] - 2.f * __ldg(cr) + mn), 0.f);
      float kl, var_kl, iws = 0.f;
      kl_finish(a, dist, T2 * sexp, 0.f, slv, logdet, &kl, &var_kl);
      if (do_iws) {
        const float off = -0.5f * (float)K * LOG2PI_F - 0.5f * logdet;
        float mxl = -CUDART_INF_F;
        for (int l = 1; l <= L; ++l) {
          const float d = fmaxf(T2 * (s_zn[l] - 2.f * __ldg(cr + (size_t)l * rs) + mn), 0.f);
          mxl = fmaxf(mxl, base_l[l - 1] + off - 0.5f * d);
        }
        float se = 0.f;
        for (int l = 1; l <= L; ++l) {
          const float d = fmaxf(T2 * (s_zn[l] - 2.f * __ldg(cr + (size_t)l * rs) + mn), 0.f);
          se += expf(base_l[l - 1] + off - 0.5f * d - mxl);
        }
        iws = se / (float)L + mxl;  // cvae.py:870: mean_l exp(.) + max, no log
      }
      s_kl[c] = kl;
      s_zd[c] = dist;
      s_vk[c] = var_kl;
      s_iws[c] = iws;
    }
    for (int c = wid; c < (a.cross ? 0 : Cp); c += ELBO_THREADS / 32) {
      const float Tc = a.inv_trans[c], T2 = Tc * Tc, logdet = a.logdet[c];
      float mreg[8], mn = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = lane + 32 * i;
        mreg[i] = (k < K) ? a.means[(size_t)c * K + k] : 0.f;
        mn = fmaf(mreg[i], mreg[i], mn);
      }
      mn = warp_sum(mn);
      float* li_w = s_li + (size_t)wid * L;
      float kl = 0.f, var_kl = 0.f, dist = 0.f;
      for (int r0 = 0; r0 < nrows; r0 += 4) {
        float q[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int k = min(lane + 32 * i, K - 1);
#pragma unroll
          for (int j = 0; j < 4; ++j) q[j] = fmaf(zs[(size_t)min(r0 + j, nrows - 1) * K + k], mreg[i], q[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) q[j] = warp_sum(q[j]);
        if (lane < 4 && r0 + lane < nrows) {
          const int row = r0 + lane;
          const float dot = lane == 0 ? q[0] : (lane == 1 ? q[1] : (lane == 2 ? q[2] : q[3]));
          const float d = fmaxf(T2 * (s_zn[row] - 2.f * dot + mn), 0.f);
          if (row == 0) {
            dist = d;
            kl_finish(a, d, T2 * sexp, 0.f, slv, logdet, &kl, &var_kl);
          } else {
            li_w[row - 1] = base_l[row - 1] - 0.5f * (float)K * LOG2PI_F - 0.5f * d - 0.5f * logdet;
          }
        }
      }
      float iws = 0.f;
      if (do_iws) {
        __syncwarp();
        float mxl = -CUDART_INF_F;
        for (int l = lane; l < L; l += 32) mxl = fmaxf(mxl, li_w[l]);
        mxl = warp_max(mxl);
        float se = 0.f;
        for (int l = lane; l < L; l += 32) se += expf(li_w[l] - mxl);
        se = warp_sum(se);
        iws = se / (float)L + mxl;  // cvae.py:870: mean_l exp(.) + max, no log
        __syncwarp();
      }
      if (lane == 0) {
        s_kl[c] = kl;
        s_zd[c] = dist;
        s_vk[c] = var_kl;
        s_iws[c] = iws;
      }
    }
  }
  // ---- class loop: one warp per class, all L+1 rows of zs against mean_c
  for (int c = wid; c < (fast ? 0 : Cp); c += ELBO_THREADS / 32) {
    const float Tc = (a.var_dim == JVAE_VAR_SCALAR) ? a.inv_trans[c] : 0.f;
    const float logdet = a.logdet[c];
    // KL terms on mu (row 0)
    float dist = 0.f, tr = 0.f, aux = 0.f;
    for (int k = lane; k < K; k += 32) {
      const float m = a.means[(size_t)c * K + k];
      const float T = (a.var_dim == JVAE_VAR_SCALAR) ? Tc : a.inv_trans[(size_t)c * K + k];
      kl_dim_terms(a, zs[k], evar[k], m, T, dist, tr, aux);
    }
    dist = warp_sum(dist);
    tr = warp_sum(tr);
    aux = warp_sum(aux);
    if (a.full_dist) dist = a.full_dist[(size_t)c * B + b];
    float kl, var_kl;
    kl_finish(a, dist, tr, aux, slv, logdet, &kl, &var_kl);
    // log p(z_l | c) for the L draws (priors.py:328-342, 381-383, 478-491) and the importance weights
    float iws = 0.f;
    if (do_iws) {
      float* li_w = s_li + (size_t)wid * L;
      if (K <= 256 && a.prior_kind != JVAE_PRIOR_UNIFORM) {
        // register-blocked path: the class mean / scale stay in registers (8 latent dims per lane) for all L draws,
        // four draws are reduced at a time (independent shuffle chains)
        float mreg[8], treg[8], vreg[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int k = lane + 32 * i;
          const bool valid = k < K;
          mreg[i] = valid ? a.means[(size_t)c * K + k] : 0.f;
          treg[i] = valid ? ((a.var_dim == JVAE_VAR_SCALAR) ? Tc : a.inv_trans[(size_t)c * K + k]) : 0.f;
          vreg[i] = valid ? 1.f : 0.f;
        }
        for (int l0 = 0; l0 < L; l0 += 4) {
          float q[4] = {0.f, 0.f, 0.f, 0.f}, nz[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int k = min(lane + 32 * i, K - 1);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int l = min(l0 + j, L - 1);
              const float zv = zs[(size_t)(l + 1) * K + k];
              const float w = treg[i] * (zv - mreg[i]);
              q[j] = fmaf(w, w, q[j]);
              nz[j] = fmaf(zv * vreg[i], zv, nz[j]);
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) q[j] = warp_sum(q[j]);
          if (a.prior_kind == JVAE_PRIOR_TILTED) {
#pragma unroll
            for (int j = 0; j < 4; ++j) nz[j] = warp_sum(nz[j]);
          }
          if (lane < 4 && l0 + lane < L) {
            float qq = lane == 0 ? q[0] : (lane == 1 ? q[1] : (lane == 2 ? q[2] : q[3]));
            if (a.full_dist) qq = a.full_dist[((size_t)(l0 + lane + 1) * Cp + c) * B + b];
            const float nn = lane == 0 ? nz[0] : (lane == 1 ? nz[1] : (lane == 2 ? nz[2] : nz[3]));
            float logp = -0.5f * (float)K * LOG2PI_F - 0.5f * qq - 0.5f * logdet;
            if (a.prior_kind == JVAE_PRIOR_TILTED) logp -= sqrtf(nn);
            li_w[l0 + lane] = base_l[l0 + lane] + logp;
          }
        }
      } else
      for (int l = 0; l < L; ++l) {

        const float* zr = zs + (size_t)(l + 1) * K;
        float q = 0.f, nz = 0.f;
        for (int k = lane; k < K; k += 32) {
          const float zv = zr[k];
          const float m = a.means[(size_t)c * K + k];
          if (a.prior_kind == JVAE_PRIOR_UNIFORM) {
            const float d = a.conditional ? zv - m : zv;
            q += (fabsf(d) > a.tau) ? (-0.5f * LOG2PI_F - 0.5f * d * d) : -a.alpha;
          } else {
            const float T = (a.var_dim == JVAE_VAR_SCALAR) ? Tc : a.inv_trans[(size_t)c * K + k];
            const float w = T * (zv - m);
            q = fmaf(w, w, q);
            nz = fmaf(zv, zv, nz);
          }
        }
        q = warp_sum(q);
        if (a.full_dist) q = a.full_dist[((size_t)(l + 1) * Cp + c) * B + b];
        float logp;
        if (a.prior_kind == JVAE_PRIOR_UNIFORM) {
          logp = q;
        } else {
          logp = -0.5f * (float)K * LOG2PI_F - 0.5f * q - 0.5f * logdet;
          if (a.prior_kind == JVAE_PRIOR_TILTED) logp -= sqrtf(warp_sum(nz));
        }
        if (lane == 0) li_w[l] = base_l[l] + logp;
      }
      __syncwarp();
      float mxl = -CUDART_INF_F;
      for (int l = lane; l < L; l += 32) mxl = fmaxf(mxl, li_w[l]);
      mxl = warp_max(mxl);
      float se = 0.f;
      for (int l = lane; l < L; l += 32) se += expf(li_w[l] - mxl);
      se = warp_sum(se);
      iws = se / (float)L + mxl;  // cvae.py:870: mean_l exp(.) + max, no log
      __syncwarp();
    }
    if (lane == 0) {
      s_kl[c] = kl;
      s_zd[c] = dist;
      s_vk[c] = var_kl;
      s_iws[c] = iws;
    }
  }
  __syncthreads();

  // ---- totals (cvae.py:744, 791, 875-902): beta is cfg.beta (1 unless with_beta)
  const bool add_cy = a.has_logits && a.gamma_w != 0.f;
  const int nT = (Cp > 1) ? Cp : (add_cy ? C : 1);
  for (int j = tid; j < nT; j += ELBO_THREADS) {
    float t = a.beta * s_kl[(Cp > 1) ? j : 0];
    if (has_x) t += cross_x;
    if (add_cy) t += a.gamma_w * s_cy[j];
    s_tot[j] = t;
  }
  __syncthreads();

  // ---- write the per-class tensors, (C,B) layout
  for (int j = tid; j < Cp; j += ELBO_THREADS) {
    const size_t o = (size_t)j * B + b;
    if (a.kl) a.kl[o] = s_kl[j];
    if (a.zdist) a.zdist[o] = s_zd[j];
    if (a.var_kl) a.var_kl[o] = s_vk[j];
    if (a.iws && do_iws) a.iws[o] = s_iws[j];
  }
  for (int j = tid; j < nT; j += ELBO_THREADS)
    if (a.total) a.total[(size_t)j * B + b] = s_tot[j];
  if (a.has_logits)
    for (int j = tid; j < C; j += ELBO_THREADS) {
      if (a.cross_y) a.cross_y[(size_t)j * B + b] = s_cy[j];
      if (a.logits_out) a.logits_out[(size_t)b * C + j] = s_lo[j];
    }
  if (tid == 0) {
    if (a.wmse && has_x) a.wmse[b] = wmse;
    if (a.cross_x && has_x) a.cross_x[b] = cross_x;
    if (a.dzdist && a.conditional) {
      float dnv = 0.f;
      for (int i = 0; i < a.nkb; ++i) dnv += __ldcg(&a.dict_norm_var[i]);
      a.dzdist[b] = dzd + dnv;
    }
  }
  if (!a.scores && !a.preds) return;

  // ---- fused batch_dist_measures (cvae.py:972-1085) and predict_after_evaluate (cvae.py:938-970)
  // reductions over classes of -total, iws, -kl, -zdist and logits
  float v_negtot = -CUDART_INF_F, v_iws = -CUDART_INF_F, v_negkl = -CUDART_INF_F, v_negzd = -CUDART_INF_F,
        v_lo = -CUDART_INF_F;
  for (int j = tid; j < nT; j += ELBO_THREADS) v_negtot = fmaxf(v_negtot, -s_tot[j]);
  for (int j = tid; j < Cp; j += ELBO_THREADS) {
    v_iws = fmaxf(v_iws, s_iws[j]);
    v_negkl = fmaxf(v_negkl, -s_kl[j]);
    v_negzd = fmaxf(v_negzd, -s_zd[j]);
  }
  if (a.has_logits)
    for (int j = tid; j < C; j += ELBO_THREADS) v_lo = fmaxf(v_lo, s_lo[j]);
  const float mx_negtot = block_max(v_negtot, red);
  const float mx_iws = block_max(v_iws, red);
  const float mx_negkl = block_max(v_negkl, red);
  const float mx_negzd = block_max(v_negzd, red);
  const float mx_lo = block_max(v_lo, red);

  float se_tot = 0.f, s1 = 0.f, se_iws = 0.f, se_kl = 0.f, se_lo = 0.f, plogp = 0.f;
  for (int j = tid; j < nT; j += ELBO_THREADS) {
    se_tot += expf(-s_tot[j] - mx_negtot);
    s1 += -s_tot[j];
  }
  for (int j = tid; j < Cp; j += ELBO_THREADS) {
    se_iws += expf(s_iws[j] - mx_iws);
    se_kl += expf(-s_kl[j] - mx_negkl);
  }
  if (a.has_logits)
    for (int j = tid; j < C; j += ELBO_THREADS) se_lo += expf(s_lo[j] - mx_lo);
  se_tot = block_sum(se_tot, red);
  s1 = block_sum(s1, red);
  se_iws = block_sum(se_iws, red);
  se_kl = block_sum(se_kl, red);
  se_lo = block_sum(se_lo, red);
  const float mean_negtot = s1 / (float)nT;
  float ss = 0.f;
  for (int j = tid; j < nT; j += ELBO_THREADS) {
    const float d = -s_tot[j] - mean_negtot;
    ss = fmaf(d, d, ss);
  }
  ss = block_sum(ss, red);
  if (a.has_logits) {
    for (int j = tid; j < C; j += ELBO_THREADS) {
      const float p = expf(s_lo[j] - mx_lo) / se_lo;
      plogp += p * logf(p);
    }
    plogp = block_sum(plogp, red);
  }
  if (a.scores && tid == 0) {
    float* s = a.scores + (size_t)b * JVAE_NSCORES;
    s[JVAE_S_ELBO] = mx_negtot;
    s[JVAE_S_SUM] = logf(se_tot) + mx_negtot;
    s[JVAE_S_MEAN] = logf(se_tot / (float)nT) + mx_negtot;
    s[JVAE_S_IWS] = (Cp > 1) ? logf(se_iws) + mx_iws + logf((float)C) : mx_iws;
    s[JVAE_S_SOFTKL] = 1.f / se_kl;
    s[JVAE_S_ZDIST] = mx_negzd;
    s[JVAE_S_KL] = mx_negkl;
    s[JVAE_S_MSE] = -cross_x;
    s[JVAE_S_WMSE] = -wmse;
    s[JVAE_S_LOGITS] = a.has_logits ? mx_lo : 0.f;
    s[JVAE_S_BASELINE] = a.has_logits ? 1.f / se_lo : 0.f;
    s[JVAE_S_HYZ] = a.has_logits ? plogp : 0.f;
    s[JVAE_S_STD] = (nT > 1) ? sqrtf(ss / (float)(nT - 1)) : 0.f;
    s[JVAE_S_SOFTIWS] = 1.f / se_iws;
    s[14] = 0.f;
    s[15] = 0.f;
  }
  if (a.preds) {
    // argmin total == first index with -total == max(-total)
    for (int j = tid; j < nT; j += ELBO_THREADS) s_tot[j] = -s_tot[j];
    __syncthreads();
    const int p_loss = block_first_index(s_tot, nT, mx_negtot, red_i);
    const int p_esty = a.has_logits ? block_first_index(s_lo, C, mx_lo, red_i) : 0;
    for (int j = tid; j < Cp; j += ELBO_THREADS) s_zd[j] = -s_zd[j];
    __syncthreads();
    const int p_closest = block_first_index(s_zd, Cp, mx_negzd, red_i);
    const int p_iws = block_first_index(s_iws, Cp, mx_iws, red_i);
    if (tid == 0) {
      int* p = a.preds + (size_t)b * JVAE_NPRED;
      p[JVAE_P_LOSS] = p_loss;
      p[JVAE_P_ESTY] = p_esty;
      p[JVAE_P_CLOSEST] = p_closest;
      p[JVAE_P_IWS] = p_iws;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int check_cfg(const jvae_elbo_cfg* cfg, const char* fn) {
  if (!cfg) { set_error("%s: cfg is NULL", fn); return JVAE_ERR_INVALID; }
  if (cfg->B <= 0 || cfg->K <= 0 || cfg->C <= 0 || cfg->L < 0) {
    set_error("%s: bad dims B=%d L=%d K=%d C=%d", fn, cfg->B, cfg->L, cfg->K, cfg->C);
    return JVAE_ERR_INVALID;
  }
  if (cfg->has_xreco && (cfg->D <= 0 || cfg->L < 1)) {
    set_error("%s: a reconstruction term needs D > 0 and L >= 1 (D=%d L=%d)", fn, cfg->D, cfg->L);
    return JVAE_ERR_INVALID;
  }
  if (cfg->categorical && (!cfg->has_xreco || cfg->cat_group <= 0 || cfg->D % cfg->cat_group != 0 || cfg->sigma_is_rmse)) {
    set_error("%s: categorical output needs has_xreco, cat_group dividing D (D=%d cat_group=%d) and no rmse sigma", fn, cfg->D,
              cfg->cat_group);
    return JVAE_ERR_INVALID;
  }
  if (cfg->var_dim == JVAE_VAR_FULL && cfg->K > 1024) {
    set_error("%s: var_dim='full' supports K <= 1024 (K=%d)", fn, cfg->K);
    return JVAE_ERR_UNSUPPORTED;
  }
  if (cfg->var_dim != JVAE_VAR_SCALAR && cfg->var_dim != JVAE_VAR_DIAG && cfg->var_dim != JVAE_VAR_FULL) {
    set_error("%s: bad var_dim %d", fn, cfg->var_dim);
    return JVAE_ERR_INVALID;
  }
  if (cfg->prior_kind < JVAE_PRIOR_GAUSSIAN || cfg->prior_kind > JVAE_PRIOR_UNIFORM) {
    set_error("%s: bad prior_kind %d", fn, cfg->prior_kind);
    return JVAE_ERR_INVALID;
  }
  if (cfg->prior_kind != JVAE_PRIOR_GAUSSIAN && cfg->var_dim != JVAE_VAR_SCALAR) {
    set_error("%s: tilted / uniform priors are scalar-variance only (priors.py:44-51)", fn);
    return JVAE_ERR_INVALID;
  }
  return JVAE_OK;
}

// latent draws streamed per CTA by the train forward / backward and eval kernels
constexpr int ELBO_LG = 4;

static void fill_args(ElboArgs& a, const jvae_elbo_cfg* cfg, void* workspace) {
  memset(&a, 0, sizeof(a));
  a.B = cfg->B; a.L = cfg->L; a.K = cfg->K; a.C = cfg->C; a.D = cfg->D;
  a.Cp = cfg->conditional ? cfg->C : 1;
  a.nkb = (cfg->K + 31) / 32;
  a.G = cfg->has_xreco ? (cfg->L + ELBO_LG - 1) / ELBO_LG : 1;
  a.xr_bf16 = cfg->xreco_dtype == JVAE_BF16;
  a.lg_bf16 = cfg->logits_dtype == JVAE_BF16;
  a.var_dim = cfg->var_dim; a.prior_kind = cfg->prior_kind; a.conditional = cfg->conditional;
  a.has_xreco = cfg->has_xreco; a.has_logits = cfg->has_logits;
  a.categorical = cfg->categorical ? 1 : 0; a.cat_group = cfg->cat_group;
  a.sigma_stride = cfg->sigma_per_sample ? 1 : 0;
  if (a.categorical) { a.has_xreco = 0; a.G = 1; }      // the pre-pass replaces the (x_reco - x)^2 stream
  a.sigma_is_log = cfg->sigma_is_log; a.sigma_is_rmse = cfg->sigma_is_rmse;
  a.beta = cfg->beta; a.gamma_w = cfg->gamma_w; a.var_w = cfg->var_w; a.tau = cfg->tau; a.alpha = cfg->alpha;
  const bool full = cfg->var_dim == JVAE_VAR_FULL;
  const WsLayout w = ws_layout(a.B, a.L, a.K, a.Cp, full,
                               tc_eligible(cfg->K, a.Cp, cfg->var_dim, cfg->prior_kind, cfg->conditional));
  char* p = reinterpret_cast<char*>(workspace);
  if (full) {
    a.tdiag = reinterpret_cast<float*>(p + w.tdiag);
    a.full_dist = reinterpret_cast<float*>(p + w.full_dist);
  }
  a.counters = reinterpret_cast<unsigned int*>(p + w.counters);
  a.dict_norm_var = reinterpret_cast<float*>(p + w.dnv);
  a.ws_mse = reinterpret_cast<float*>(p + w.mse);
  a.dict_mean = reinterpret_cast<float*>(p + w.dict_mean);
  a.logdet = reinterpret_cast<float*>(p + w.logdet);
  a.ws_lat = reinterpret_cast<float*>(p + w.lat);
  a.ws_ce = reinterpret_cast<float*>(p + w.ce);
}

// categorical output: cross-entropy / arg-max error sums per (draw, sample) into ws_ce / ws_mse
static int categorical_prepass(const ElboArgs& a, cudaStream_t st) {
  JVAE_CUDA(cudaMemsetAsync(a.ws_mse, 0, (size_t)a.L * a.B * 4, st));
  JVAE_CUDA(cudaMemsetAsync(a.ws_ce, 0, (size_t)a.L * a.B * 4, st));
  int chunks = (a.D + 255) / 256;
  if (chunks > 8) chunks = 8;
  dim3 grid(a.L * a.B, chunks);
  if (a.xr_bf16) categorical_fwd_kernel<true><<<grid, 256, 0, st>>>(a);
  else categorical_fwd_kernel<false><<<grid, 256, 0, st>>>(a);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

static int launch_prologue(const ElboArgs& a, cudaStream_t st) {
  const int nkb = (a.K + 31) / 32;
  const int ncb = (a.Cp + 7) / 8;
  prior_stats_kernel<<<nkb + ncb, 256, 0, st>>>(a, nkb);
  JVAE_LAUNCH_CHECK();
  if (a.var_dim == JVAE_VAR_FULL) {
    full_tdiag_kernel<<<a.Cp, 128, 0, st>>>(a.inv_trans, a.K, a.tdiag);
    JVAE_LAUNCH_CHECK();
  }
  return JVAE_OK;
}

// var_dim = full: squared distances of `rows` (R, K) to the class means under T_c, then the main kernels see a diagonal
// prior (tdiag) plus the precomputed distances
static int full_distances(ElboArgs& a, const float* rows, int R, const long long* y, cudaStream_t st) {
  const size_t smem = (size_t)32 * (a.K + 1) * sizeof(float);
  if (smem > 48 * 1024)
    JVAE_CUDA(cudaFuncSetAttribute(full_dist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((R + FD_WARPS * FD_RPW - 1) / (FD_WARPS * FD_RPW), a.Cp);
  full_dist_kernel<<<grid, FD_WARPS * 32, smem, st>>>(a.inv_trans, a.means, rows, y, R, a.B, a.K, a.Cp, a.C, a.full_dist);
  JVAE_LAUNCH_CHECK();
  a.full_T = a.inv_trans;
  a.inv_trans = a.tdiag;
  a.var_dim = JVAE_VAR_DIAG;
  return JVAE_OK;
}

}  // namespace jvae

using namespace jvae;

extern "C" {

size_t jvae_elbo_workspace_bytes(const jvae_elbo_cfg* cfg) {
  if (!cfg) return 0;
  const int Cp = cfg->conditional ? cfg->C : 1;
  return ws_layout(cfg->B, cfg->L, cfg->K, Cp, cfg->var_dim == JVAE_VAR_FULL,
                   tc_eligible(cfg->K, Cp, cfg->var_dim, cfg->prior_kind, cfg->conditional)).total;
}

int jvae_elbo_train_fwd(const jvae_elbo_cfg* cfg, const float* x, const void* x_reco, const float* mu,
                        const float* log_var, const void* logits, const int64_t* y, const float* means,
                        const float* inv_trans, const float* sigma, float* kl, float* zdist, float* var_kl,
                        float* wmse, float* cross_x, float* cross_y, float* total, float* dzdist,
                        int32_t* finite_flag, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_cfg(cfg, __func__);
  if (rc) return rc;
  JVAE_CHECK_ARG(mu && log_var && y && means && inv_trans, "mu, log_var, y, means, inv_trans are required");
  JVAE_CHECK_ARG(!cfg->has_xreco || (x && x_reco && sigma), "x, x_reco and sigma are required when has_xreco");
  JVAE_CHECK_ARG(!cfg->has_logits || logits, "logits is required when has_logits");
  JVAE_CHECK_ARG(workspace && workspace_bytes >= jvae_elbo_workspace_bytes(cfg), "workspace too small");
  JVAE_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)x_reco & 15) == 0, "x and x_reco must be 16-byte aligned");
  ElboArgs a;
  fill_args(a, cfg, workspace);
  a.x = x; a.xr = x_reco; a.mu = mu; a.lv = log_var; a.logits = logits; a.y = (const long long*)y;
  a.means = means; a.inv_trans = inv_trans; a.sigma = sigma;
  a.kl = kl; a.zdist = zdist; a.var_kl = var_kl; a.wmse = wmse; a.cross_x = cross_x; a.cross_y = cross_y;
  a.total = total; a.dzdist = dzdist; a.finite_flag = finite_flag;
  cudaStream_t st = (cudaStream_t)stream;
  if (!cfg->prior_stats_ready) {
    rc = launch_prologue(a, st);
    if (rc) return rc;
  }
  if (cfg->var_dim == JVAE_VAR_FULL) {
    rc = full_distances(a, mu, a.B, a.y, st);
    if (rc) return rc;
  }
  if (a.categorical) {
    rc = categorical_prepass(a, st);
    if (rc) return rc;
  }
  // register-staged variant (bf16 reconstructions, vector-aligned rows): 2 draws per CTA, 3 vector rounds in flight, 6 resident
  // CTAs per SM, measured best at B = 512 and B = 2048 (tools/elbo_tune.py)
  if (a.has_xreco && a.xr_bf16 && (a.D & 7) == 0) {
    const int nlat = (a.B + ELBO_THREADS / 32 - 1) / (ELBO_THREADS / 32);
    constexpr int LG = 2, U = 3, MINB = 6;
    a.G = (a.L + LG - 1) / LG;
    void* prof = prof_begin(JVAE_PROF_ELBO_TRAIN_FWD, st);
    elbo_train_fwd_v2_kernel<LG, U, MINB><<<nlat + a.B * a.G, ELBO_THREADS, 0, st>>>(a);
    prof_end(prof, st);
    JVAE_LAUNCH_CHECK();
    return JVAE_OK;
  }
  // latent CTAs (one warp per sample) first, then the streaming CTAs (none without a reconstruction term)
  int grid = (a.B + ELBO_THREADS / 32 - 1) / (ELBO_THREADS / 32);
  if (a.has_xreco) {
    const int items = a.B * a.G;
    const int wave = 12 * sm_count() - grid;      // 12 resident CTAs per SM
    // between one and two waves (c2: 2048 items, 1648 slots) a partial second wave costs ~1.2 us of a 17 us launch: two items
    // per CTA instead.  With several waves the hardware scheduler's refill beats a static split (measured at B = 2048).
    const int per_cta = (wave > 0 && items > wave && items <= 2 * wave) ? 2 : 1;
    grid += (items + per_cta - 1) / per_cta;
  }
#define JVAE_ELBO_LAUNCH(kern, smem_)                                           \
  do {                                                                        \
    if (a.xr_bf16) kern<true, ELBO_LG><<<grid, ELBO_THREADS, smem_, st>>>(a);  \
    else kern<false, ELBO_LG><<<grid, ELBO_THREADS, smem_, st>>>(a);           \
  } while (0)
  void* prof = prof_begin(JVAE_PROF_ELBO_TRAIN_FWD, st);
  JVAE_ELBO_LAUNCH(elbo_train_fwd_kernel, 0);
  prof_end(prof, st);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

int jvae_elbo_prior_stats(const jvae_elbo_cfg* cfg, const float* means, const float* inv_trans, void* workspace,
                          size_t workspace_bytes, void* stream) {
  int rc = check_cfg(cfg, __func__);
  if (rc) return rc;
  JVAE_CHECK_ARG(means && inv_trans, "means and inv_trans are required");
  JVAE_CHECK_ARG(workspace && workspace_bytes >= jvae_elbo_workspace_bytes(cfg), "workspace too small");
  ElboArgs a;
  fill_args(a, cfg, workspace);
  a.means = means; a.inv_trans = inv_trans;
  return launch_prologue(a, (cudaStream_t)stream);
}

int jvae_elbo_train_bwd(const jvae_elbo_cfg* cfg, const float* g, const float* x, const void* x_reco,
                        const float* mu, const float* log_var, const void* logits, const int64_t* y,
                        const float* means, const float* inv_trans, const float* sigma, const float* wmse,
                        void* d_x_reco, float* d_mu, float* d_log_var, void* d_logits, float* d_means,
                        float* d_inv_trans, float* d_sigma, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_cfg(cfg, __func__);
  if (rc) return rc;
  JVAE_CHECK_ARG(g && mu && log_var && y && means && inv_trans, "g, mu, log_var, y, means, inv_trans are required");
  JVAE_CHECK_ARG(!cfg->has_xreco || (x && x_reco && sigma && wmse), "x, x_reco, sigma, wmse are required when has_xreco");
  JVAE_CHECK_ARG(!cfg->has_logits || logits, "logits is required when has_logits");
  JVAE_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)x_reco & 15) == 0 && ((uintptr_t)d_x_reco & 15) == 0,
                 "x, x_reco and d_x_reco must be 16-byte aligned");
  const bool full = cfg->var_dim == JVAE_VAR_FULL;
  JVAE_CHECK_ARG(!full || (workspace && workspace_bytes >= jvae_elbo_workspace_bytes(cfg)),
                 "var_dim='full' needs the workspace in the backward pass");
  ElboArgs a;
  char dummy[4096];
  fill_args(a, cfg, full ? workspace : dummy);
  a.counters = nullptr; a.dict_norm_var = nullptr; a.ws_mse = nullptr; a.dict_mean = nullptr; a.logdet = nullptr;
  a.ws_lat = nullptr; a.full_dist = nullptr;
  a.g = g; a.x = x; a.xr = x_reco; a.mu = mu; a.lv = log_var; a.logits = logits; a.y = (const long long*)y;
  a.means = means; a.inv_trans = inv_trans; a.sigma = sigma; a.wmse_in = wmse;
  a.d_xr = d_x_reco; a.d_mu = d_mu; a.d_lv = d_log_var; a.d_logits = d_logits; a.d_means = d_means;
  a.d_inv_trans = d_inv_trans; a.d_sigma = d_sigma;
  cudaStream_t st = (cudaStream_t)stream;
  if (d_means) JVAE_CUDA(cudaMemsetAsync(d_means, 0, (size_t)a.Cp * a.K * 4, st));
  if (d_sigma) JVAE_CUDA(cudaMemsetAsync(d_sigma, 0, (cfg->sigma_per_sample ? (size_t)a.B : 1) * 4, st));
  if (d_inv_trans)
    JVAE_CUDA(cudaMemsetAsync(d_inv_trans, 0,
                              (size_t)a.Cp * (full ? (size_t)a.K * a.K : (cfg->var_dim == JVAE_VAR_DIAG ? a.K : 1)) * 4, st));
  if (full) {      // the streaming kernel sees the diagonal view; the distance / T gradients come from full_prior_bwd_kernel
    full_tdiag_kernel<<<a.Cp, 128, 0, st>>>(inv_trans, a.K, a.tdiag);
    JVAE_LAUNCH_CHECK();
    a.full_T = inv_trans; a.inv_trans = a.tdiag; a.var_dim = JVAE_VAR_DIAG;
    a.d_full_T = d_inv_trans; a.d_inv_trans = nullptr;
  }
  if (a.categorical) {
    JVAE_CHECK_ARG(d_x_reco, "d_x_reco is required for the categorical output");
    int chunks = (a.D + 255) / 256;
    if (chunks > 8) chunks = 8;
    dim3 cgrid((a.L + 1) * a.B, chunks);
    if (a.xr_bf16) categorical_bwd_kernel<true><<<cgrid, 256, 0, st>>>(a);
    else categorical_bwd_kernel<false><<<cgrid, 256, 0, st>>>(a);
    JVAE_LAUNCH_CHECK();
  }
  const int grid = a.B * a.G;
  void* prof = prof_begin(JVAE_PROF_ELBO_TRAIN_BWD, st);
  JVAE_ELBO_LAUNCH(elbo_train_bwd_kernel, 0);
  prof_end(prof, st);
  JVAE_LAUNCH_CHECK();
  if (full) {
    full_prior_bwd_kernel<<<a.B, 128, 2 * (size_t)a.K * sizeof(float), st>>>(a);
    JVAE_LAUNCH_CHECK();
  }
  return JVAE_OK;
}

int jvae_elbo_eval_fwd(const jvae_elbo_cfg* cfg, const float* x, const void* x_reco, const float* mu,
                       const float* log_var, const float* z, const float* eps_norm, const void* logits,
                       const float* means, const float* inv_trans, const float* sigma, float* kl, float* zdist,
                       float* var_kl, float* total, float* iws, float* cross_y, float* wmse, float* cross_x,
                       float* dzdist, float* logits_out, float* scores, int32_t* preds, void* workspace,
                       size_t workspace_bytes, void* stream) {
  int rc = check_cfg(cfg, __func__);
  if (rc) return rc;
  JVAE_CHECK_ARG(mu && log_var && means && inv_trans, "mu, log_var, means, inv_trans are required");
  JVAE_CHECK_ARG(!cfg->has_xreco || (x && x_reco && sigma), "x, x_reco and sigma are required when has_xreco");
  JVAE_CHECK_ARG(!cfg->has_logits || logits, "logits is required when has_logits");
  JVAE_CHECK_ARG(workspace && workspace_bytes >= jvae_elbo_workspace_bytes(cfg), "workspace too small");
  JVAE_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)x_reco & 15) == 0, "x and x_reco must be 16-byte aligned");
  ElboArgs a;
  fill_args(a, cfg, workspace);
  a.x = x; a.xr = x_reco; a.mu = mu; a.lv = log_var; a.z = z; a.eps_norm = eps_norm; a.logits = logits;
  a.means = means; a.inv_trans = inv_trans; a.sigma = sigma;
  a.kl = kl; a.zdist = zdist; a.var_kl = var_kl; a.total = total; a.iws = iws; a.cross_y = cross_y;
  a.wmse = wmse; a.cross_x = cross_x; a.dzdist = dzdist; a.logits_out = logits_out; a.scores = scores; a.preds = preds;
  cudaStream_t st = (cudaStream_t)stream;
  const int Cmax = a.C > a.Cp ? a.C : a.Cp;
  const size_t smem = ((size_t)(a.L + 1) * a.K + a.K + a.L + 4 * (size_t)a.Cp + Cmax + 2 * (size_t)a.C +
                       (size_t)(ELBO_THREADS / 32) * a.L + (size_t)(a.L + 1)) * sizeof(float);
  if (smem > 200 * 1024) {
    set_error("%s: (L+1)*K + 7*C floats = %zu bytes of shared memory exceed 200 KB", __func__, smem);
    return JVAE_ERR_UNSUPPORTED;
  }
  if (!cfg->prior_stats_ready) {
    rc = launch_prologue(a, st);
    if (rc) return rc;
  }
  if (cfg->var_dim == JVAE_VAR_FULL) {
    JVAE_CHECK_ARG(z, "z (L+1, B, K) is required for var_dim='full'");
    rc = full_distances(a, z, (a.L + 1) * a.B, nullptr, st);
    if (rc) return rc;
  }
  if (a.categorical) {
    rc = categorical_prepass(a, st);
    if (rc) return rc;
  }
  void* prof = prof_begin(JVAE_PROF_ELBO_EVAL_FWD, st);      // the cross-term GEMM is part of the figure
  if (tc_eligible(a.K, a.Cp, a.var_dim, a.prior_kind, a.conditional)) {
    // cross terms of every (row, class) pair on the tensor cores: (R x 3K) . (Cp x 3K)^T -> fp32 (R x Cp)
    const bool rows_z = a.z && a.eps_norm && (a.has_xreco || a.categorical);
    const int R = rows_z ? (a.L + 1) * a.B : a.B;
    const WsLayout w = ws_layout(a.B, a.L, a.K, a.Cp, false, true);
    char* wp = reinterpret_cast<char*>(workspace);
    __nv_bfloat16* xa = reinterpret_cast<__nv_bfloat16*>(wp + w.tc_a);
    __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(wp + w.tc_b);
    float* cross = reinterpret_cast<float*>(wp + w.tc_cross);
    float* mnorm = reinterpret_cast<float*>(wp + w.tc_mnorm);
    dist_split_kernel<<<R + a.Cp, 128, 0, st>>>(mu, z, means, R, a.B, a.K, a.Cp, xa, xb, mnorm);
    JVAE_LAUNCH_CHECK();
    rc = jvae_gemm_bf16(JVAE_GEMM_NT, R, a.Cp, 3 * a.K, xa, 3 * a.K, xb, 3 * a.K, nullptr, JVAE_ACT_NONE, nullptr, cross, w.tc_ld,
                        nullptr, 0, stream);
    if (rc) return rc;
    a.cross = cross; a.mnorm = mnorm; a.cross_ld = w.tc_ld;
  }
  const int grid = a.B * a.G;
  if (smem > 48 * 1024) {
    JVAE_CUDA(cudaFuncSetAttribute(elbo_eval_fwd_kernel<true, ELBO_LG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    JVAE_CUDA(cudaFuncSetAttribute(elbo_eval_fwd_kernel<false, ELBO_LG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  JVAE_ELBO_LAUNCH(elbo_eval_fwd_kernel, smem);
  prof_end(prof, st);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

}  // extern "C"
