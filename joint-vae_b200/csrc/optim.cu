// Global-norm gradient clipping + Adam (optionally AMSGrad) or SGD (momentum, dampening, Nesterov) with L2 weight decay on
// one flat buffer (module/optimizers.py:79-81,120-121 of the reference: clip_grad_norm_ then torch.optim.Adam / SGD).
// The clip coefficient is computed on the device from the squared norm, so a step needs no host sync.
#include "common.cuh"

namespace jvae {

constexpr int OPT_THREADS = 256;

template <bool BF16>
__device__ __forceinline__ float4 load_grad4(const void* g, size_t i4) {
  if (BF16) {
    const uint2 u = reinterpret_cast<const uint2*>(g)[i4];
    return make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
  }
  return reinterpret_cast<const float4*>(g)[i4];
}
template <bool BF16>
__device__ __forceinline__ float load_grad1(const void* g, size_t i) {
  return BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(g)[i]) : reinterpret_cast<const float*>(g)[i];
}

constexpr int SEG_CHUNK = 256;      // JVAE_OPT_CHUNK: every parameter's slice of the flat buffers starts on a multiple of this

// sum of squares of the gradient; with a chunk -> parameter table also marks the parameters whose gradient has a non-zero
// element (seg_active[s] = 1): torch.optim skips parameters without a gradient (grad is None), here those are the
// parameters whose slice of the zeroed flat gradient nobody wrote.
template <bool BF16>
__global__ void __launch_bounds__(OPT_THREADS) grad_sqnorm_kernel(const void* __restrict__ g, size_t n, float* out,
                                                                   const int32_t* __restrict__ chunk_seg, int32_t* seg_active) {
  __shared__ float red[32];
  float acc = 0.f;
  const size_t n4 = n >> 2;
  for (size_t i = (size_t)blockIdx.x * OPT_THREADS + threadIdx.x; i < n4; i += (size_t)gridDim.x * OPT_THREADS) {
    const float4 v = load_grad4<BF16>(g, i);
    const float q = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
    acc += q;
    if (chunk_seg && q != 0.f) {
      const int sgm = chunk_seg[(i << 2) / SEG_CHUNK];
      if (seg_active[sgm] == 0) seg_active[sgm] = 1;          // benign race: every writer stores 1
    }
  }
  if (blockIdx.x == 0)
    for (size_t i = (n4 << 2) + threadIdx.x; i < n; i += OPT_THREADS) {
      const float v = load_grad1<BF16>(g, i);
      acc = fmaf(v, v, acc);
      if (chunk_seg && v != 0.f) seg_active[chunk_seg[i / SEG_CHUNK]] = 1;
    }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) atomicAdd(out, acc);
}

// per parameter: step count += active, and (Adam, seg_bc != nullptr) bias corrections of ITS step count (torch keeps
// `step` per parameter; SGD uses the count only to tell a parameter's first update)
__global__ void adam_prepare_kernel(int nseg, const int32_t* __restrict__ seg_active, int32_t* __restrict__ seg_step,
                                    float* __restrict__ seg_bc, float beta1, float beta2) {
  const int sgm = blockIdx.x * blockDim.x + threadIdx.x;
  if (sgm >= nseg) return;
  const int st = seg_step[sgm] + (seg_active[sgm] ? 1 : 0);
  seg_step[sgm] = st;
  if (!seg_bc) return;
  const float t = (float)(st > 0 ? st : 1);
  seg_bc[2 * sgm] = 1.f - powf(beta1, t);
  seg_bc[2 * sgm + 1] = sqrtf(1.f - powf(beta2, t));
}

// clip_grad_norm_: coef = clamp(max_norm / (total_norm + 1e-6), max=1); the norm is of the scaled gradient
__device__ __forceinline__ float clip_coef(const float* norm2, float max_norm, float grad_scale) {
  float clip = grad_scale;
  if (max_norm > 0.f && norm2) {
    const float tn = sqrtf(*norm2) * grad_scale;
    clip *= fminf(1.f, max_norm / (tn + 1e-6f));
  }
  return clip;
}

struct AdamArgs {
  float max_norm, lr, beta1, beta2, eps, weight_decay, grad_scale;
};

// AMSGRAD: torch.optim.Adam(amsgrad=True) normalises by the running maximum of the second moment
template <bool AMSGRAD>
__device__ __forceinline__ void adam1(float& p, float& m, float& v, float& vmax, float g, const AdamArgs& a, float clip,
                                      float bc1, float bc2_sqrt) {
  g = g * clip + a.weight_decay * p;
  m = a.beta1 * m + (1.f - a.beta1) * g;
  v = a.beta2 * v + (1.f - a.beta2) * g * g;
  float vd = v;
  if (AMSGRAD) {
    vmax = fmaxf(vmax, v);
    vd = vmax;
  }
  const float denom = sqrtf(vd) / bc2_sqrt + a.eps;
  p -= (a.lr / bc1) * (m / denom);
}

template <bool BF16, bool AMSGRAD>
__global__ void __launch_bounds__(OPT_THREADS) adam_kernel(float* __restrict__ p, float* __restrict__ m,
                                                           float* __restrict__ v, float* __restrict__ vmax,
                                                           const void* __restrict__ g, size_t n,
                                                           const float* __restrict__ norm2, const int32_t* __restrict__ chunk_seg,
                                                           const int32_t* __restrict__ seg_active,
                                                           const float* __restrict__ seg_bc, AdamArgs a) {
  const float clip = clip_coef(norm2, a.max_norm, a.grad_scale);
  const size_t n4 = n >> 2;      // n is a multiple of SEG_CHUNK
  for (size_t i = (size_t)blockIdx.x * OPT_THREADS + threadIdx.x; i < n4; i += (size_t)gridDim.x * OPT_THREADS) {
    const int sgm = chunk_seg[(i << 2) / SEG_CHUNK];
    if (!seg_active[sgm]) continue;                           // no gradient: torch skips the parameter entirely
    const float bc1 = seg_bc[2 * sgm], bc2s = seg_bc[2 * sgm + 1];
    float4 pp = reinterpret_cast<float4*>(p)[i], mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    float4 xx = AMSGRAD ? reinterpret_cast<float4*>(vmax)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 gg = load_grad4<BF16>(g, i);
    adam1<AMSGRAD>(pp.x, mm.x, vv.x, xx.x, gg.x, a, clip, bc1, bc2s);
    adam1<AMSGRAD>(pp.y, mm.y, vv.y, xx.y, gg.y, a, clip, bc1, bc2s);
    adam1<AMSGRAD>(pp.z, mm.z, vv.z, xx.z, gg.z, a, clip, bc1, bc2s);
    adam1<AMSGRAD>(pp.w, mm.w, vv.w, xx.w, gg.w, a, clip, bc1, bc2s);
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (AMSGRAD) reinterpret_cast<float4*>(vmax)[i] = xx;
  }
}

struct SgdArgs {
  float max_norm, lr, momentum, dampening, weight_decay, grad_scale;
  int nesterov;
};

// torch.optim.SGD (_single_tensor_sgd): d = g + wd p; buf = d on the parameter's first update, else
// momentum buf + (1 - dampening) d; d = nesterov ? d + momentum buf : buf; p -= lr d
template <bool MOMENTUM>
__device__ __forceinline__ void sgd1(float& p, float& buf, float g, const SgdArgs& a, float clip, bool first) {
  float d = g * clip + a.weight_decay * p;
  if (MOMENTUM) {
    buf = first ? d : a.momentum * buf + (1.f - a.dampening) * d;
    d = a.nesterov ? d + a.momentum * buf : buf;
  }
  p -= a.lr * d;
}

// MOMENTUM false: buf is not touched (it may be null), the kernel streams p and g only
template <bool BF16, bool MOMENTUM>
__global__ void __launch_bounds__(OPT_THREADS) sgd_kernel(float* __restrict__ p, float* __restrict__ buf,
                                                          const void* __restrict__ g, size_t n, const float* __restrict__ norm2,
                                                          const int32_t* __restrict__ chunk_seg,
                                                          const int32_t* __restrict__ seg_active,
                                                          const int32_t* __restrict__ seg_step, SgdArgs a) {
  const float clip = clip_coef(norm2, a.max_norm, a.grad_scale);
  const size_t n4 = n >> 2;      // n is a multiple of SEG_CHUNK
  for (size_t i = (size_t)blockIdx.x * OPT_THREADS + threadIdx.x; i < n4; i += (size_t)gridDim.x * OPT_THREADS) {
    const int sgm = chunk_seg[(i << 2) / SEG_CHUNK];
    if (!seg_active[sgm]) continue;                           // no gradient: torch skips the parameter entirely
    const bool first = seg_step[sgm] == 1;                    // counted by adam_prepare_kernel before this launch
    float4 pp = reinterpret_cast<float4*>(p)[i];
    float4 bb = MOMENTUM ? reinterpret_cast<float4*>(buf)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 gg = load_grad4<BF16>(g, i);
    sgd1<MOMENTUM>(pp.x, bb.x, gg.x, a, clip, first);
    sgd1<MOMENTUM>(pp.y, bb.y, gg.y, a, clip, first);
    sgd1<MOMENTUM>(pp.z, bb.z, gg.z, a, clip, first);
    sgd1<MOMENTUM>(pp.w, bb.w, gg.w, a, clip, first);
    reinterpret_cast<float4*>(p)[i] = pp;
    if (MOMENTUM) reinterpret_cast<float4*>(buf)[i] = bb;
  }
}

static int grid_for(size_t n) {
  const size_t want = (n / 4 + OPT_THREADS - 1) / OPT_THREADS;
  const size_t cap = (size_t)sm_count() * 8;
  size_t g = want < cap ? want : cap;
  return (int)(g ? g : 1);
}

}  // namespace jvae

using namespace jvae;

extern "C" {

int jvae_grad_sqnorm(const void* grad, int grad_dtype, size_t n, float* norm2_out, const int32_t* chunk_seg, int32_t* seg_active,
                     void* stream) {
  JVAE_CHECK_ARG(grad && norm2_out, "grad and norm2_out are required");
  JVAE_CHECK_ARG(((uintptr_t)grad & 15) == 0, "grad must be 16-byte aligned");
  JVAE_CHECK_ARG((chunk_seg == nullptr) == (seg_active == nullptr), "chunk_seg and seg_active go together");
  if (n == 0) return JVAE_OK;
  if (grad_dtype == JVAE_BF16)
    grad_sqnorm_kernel<true><<<grid_for(n), OPT_THREADS, 0, (cudaStream_t)stream>>>(grad, n, norm2_out, chunk_seg, seg_active);
  else
    grad_sqnorm_kernel<false><<<grid_for(n), OPT_THREADS, 0, (cudaStream_t)stream>>>(grad, n, norm2_out, chunk_seg, seg_active);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

int jvae_adam_step(float* p, float* m, float* v, const void* grad, int grad_dtype, size_t n, const float* norm2,
                   float max_norm, float lr, float beta1, float beta2, float eps, float weight_decay, int nseg,
                   const int32_t* chunk_seg, const int32_t* seg_active, int32_t* seg_step, float* seg_bc, float grad_scale,
                   void* stream) {
  JVAE_CHECK_ARG(p && m && v && grad, "p, m, v, grad are required");
  JVAE_CHECK_ARG(nseg >= 1 && chunk_seg && seg_active && seg_step && seg_bc, "the parameter table is required");
  JVAE_CHECK_ARG((n % SEG_CHUNK) == 0, "the flat buffers are a whole number of JVAE_OPT_CHUNK chunks");
  JVAE_CHECK_ARG((((uintptr_t)p | (uintptr_t)m | (uintptr_t)v | (uintptr_t)grad) & 15) == 0, "buffers must be 16-byte aligned");
  if (n == 0) return JVAE_OK;
  adam_prepare_kernel<<<(nseg + 127) / 128, 128, 0, (cudaStream_t)stream>>>(nseg, seg_active, seg_step, seg_bc, beta1, beta2);
  JVAE_LAUNCH_CHECK();
  AdamArgs a;
  a.max_norm = max_norm; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay;
  a.grad_scale = grad_scale;
  if (grad_dtype == JVAE_BF16)
    adam_kernel<true, false><<<grid_for(n), OPT_THREADS, 0, (cudaStream_t)stream>>>(p, m, v, nullptr, grad, n, norm2, chunk_seg,
                                                                                     seg_active, seg_bc, a);
  else
    adam_kernel<false, false><<<grid_for(n), OPT_THREADS, 0, (cudaStream_t)stream>>>(p, m, v, nullptr, grad, n, norm2, chunk_seg,
                                                                                      seg_active, seg_bc, a);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

int jvae_adam_amsgrad_step(float* p, float* m, float* v, float* vmax, const void* grad, int grad_dtype, size_t n,
                           const float* norm2, float max_norm, float lr, float beta1, float beta2, float eps,
                           float weight_decay, int nseg, const int32_t* chunk_seg, const int32_t* seg_active, int32_t* seg_step,
                           float* seg_bc, float grad_scale, void* stream) {
  JVAE_CHECK_ARG(p && m && v && vmax && grad, "p, m, v, vmax, grad are required");
  JVAE_CHECK_ARG(nseg >= 1 && chunk_seg && seg_active && seg_step && seg_bc, "the parameter table is required");
  JVAE_CHECK_ARG((n % SEG_CHUNK) == 0, "the flat buffers are a whole number of JVAE_OPT_CHUNK chunks");
  JVAE_CHECK_ARG((((uintptr_t)p | (uintptr_t)m | (uintptr_t)v | (uintptr_t)vmax | (uintptr_t)grad) & 15) == 0,
                 "buffers must be 16-byte aligned");
  if (n == 0) return JVAE_OK;
  adam_prepare_kernel<<<(nseg + 127) / 128, 128, 0, (cudaStream_t)stream>>>(nseg, seg_active, seg_step, seg_bc, beta1, beta2);
  JVAE_LAUNCH_CHECK();
  AdamArgs a;
  a.max_norm = max_norm; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay;
  a.grad_scale = grad_scale;
  if (grad_dtype == JVAE_BF16)
    adam_kernel<true, true><<<grid_for(n), OPT_THREADS, 0, (cudaStream_t)stream>>>(p, m, v, vmax, grad, n, norm2, chunk_seg,
                                                                                    seg_active, seg_bc, a);
  else
    adam_kernel<false, true><<<grid_for(n), OPT_THREADS, 0, (cudaStream_t)stream>>>(p, m, v, vmax, grad, n, norm2, chunk_seg,
                                                                                     seg_active, seg_bc, a);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

int jvae_sgd_step(float* p, float* buf, const void* grad, int grad_dtype, size_t n, const float* norm2, float max_norm,
                  float lr, float momentum, float dampening, int nesterov, float weight_decay, int nseg,
                  const int32_t* chunk_seg, const int32_t* seg_active, int32_t* seg_step, float grad_scale, void* stream) {
  JVAE_CHECK_ARG(p && grad, "p and grad are required");
  JVAE_CHECK_ARG((buf != nullptr) == (momentum != 0.f), "buf is required iff momentum != 0");
  JVAE_CHECK_ARG(nseg >= 1 && chunk_seg && seg_active && seg_step, "the parameter table is required");
  JVAE_CHECK_ARG((n % SEG_CHUNK) == 0, "the flat buffers are a whole number of JVAE_OPT_CHUNK chunks");
  JVAE_CHECK_ARG((((uintptr_t)p | (uintptr_t)buf | (uintptr_t)grad) & 15) == 0, "buffers must be 16-byte aligned");
  if (n == 0) return JVAE_OK;
  adam_prepare_kernel<<<(nseg + 127) / 128, 128, 0, (cudaStream_t)stream>>>(nseg, seg_active, seg_step, nullptr, 0.f, 0.f);
  JVAE_LAUNCH_CHECK();
  SgdArgs a;
  a.max_norm = max_norm; a.lr = lr; a.momentum = momentum; a.dampening = dampening; a.weight_decay = weight_decay;
  a.grad_scale = grad_scale; a.nesterov = nesterov != 0;
  const int grid = grid_for(n);
  cudaStream_t st = (cudaStream_t)stream;
  if (grad_dtype == JVAE_BF16) {
    if (buf) sgd_kernel<true, true><<<grid, OPT_THREADS, 0, st>>>(p, buf, grad, n, norm2, chunk_seg, seg_active, seg_step, a);
    else sgd_kernel<true, false><<<grid, OPT_THREADS, 0, st>>>(p, buf, grad, n, norm2, chunk_seg, seg_active, seg_step, a);
  } else {
    if (buf) sgd_kernel<false, true><<<grid, OPT_THREADS, 0, st>>>(p, buf, grad, n, norm2, chunk_seg, seg_active, seg_step, a);
    else sgd_kernel<false, false><<<grid, OPT_THREADS, 0, st>>>(p, buf, grad, n, norm2, chunk_seg, seg_active, seg_step, a);
  }
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

}  // extern "C"
