// Reparameterisation sampler (module/vae_layers/layers.py:230-244, 388-396 of the reference).
//
// Consumes the fused [mu | raw log_var] head (one GEMM instead of the reference's two), clips the log
// variance, draws eps (Philox4x32-10 + Box-Muller, or injected noise for parity), writes z for all L+1
// draws (slab 0 = mean) in f32 and optionally bf16 (decoder operand), eps and ||eps||^2.
#include "common.cuh"

namespace jvae {

constexpr int SAMPLE_THREADS = 128;

__device__ __forceinline__ float u01(uint32_t r) { return ((float)(r >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// one draw for flat element index idx of stream (seed, offset)
__device__ __forceinline__ float draw(uint64_t seed, uint64_t offset, uint64_t idx, int uniform) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  if (uniform) return (u01(r.x) - 0.5f) * 3.4641016151377544f;  // sqrt(12)
  const float u1 = u01(r.x), u2 = u01(r.y);
  return sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
}

// one CTA per sample b
__global__ void __launch_bounds__(SAMPLE_THREADS) sample_fwd_kernel(int B, int L, int K, const float* __restrict__ head,
                                                                    const float* __restrict__ eps_in, uint64_t seed,
                                                                    uint64_t offset, const uint64_t* __restrict__ offset_dev,
                                                                    int is_sampled, int uniform,
                                                                    float* mu_o, float* lv_o, float* z,
                                                                    __nv_bfloat16* z16, float* eps_o, float* eps_norm) {
  __shared__ float red[32];
  const int b = blockIdx.x;
  const float samp = is_sampled ? 1.f : 0.f;
  if (offset_dev) offset += *offset_dev;      // stream position kept on the device (CUDA-graph replays draw fresh noise)
  // slab 0 and the clipped head
  for (int k = threadIdx.x; k < K; k += SAMPLE_THREADS) {
    const float m = head[(size_t)b * 2 * K + k];
    const float lv = fminf(fmaxf(head[(size_t)b * 2 * K + K + k], -20.f), 20.f);
    if (mu_o) mu_o[(size_t)b * K + k] = m;
    if (lv_o) lv_o[(size_t)b * K + k] = lv;
    if (z) z[(size_t)b * K + k] = m;
    if (z16) z16[(size_t)b * K + k] = __float2bfloat16(m);
  }
  for (int l = 1; l <= L; ++l) {
    float en = 0.f;
    for (int k = threadIdx.x; k < K; k += SAMPLE_THREADS) {
      const float m = head[(size_t)b * 2 * K + k];
      const float lv = fminf(fmaxf(head[(size_t)b * 2 * K + K + k], -20.f), 20.f);
      const size_t idx = ((size_t)l * B + b) * K + k;
      const float e = eps_in ? eps_in[idx] : draw(seed, offset, idx, uniform);
      const float zv = m + expf(0.5f * lv) * e * samp;
      if (z) z[idx] = zv;
      if (z16) z16[idx] = __float2bfloat16(zv);
      if (eps_o) eps_o[idx - (size_t)B * K] = e;
      en = fmaf(e, e, en);
    }
    en = block_sum(en, red);
    if (eps_norm && threadIdx.x == 0) eps_norm[(size_t)(l - 1) * B + b] = en;
  }
}

template <bool DZ_BF16>
__global__ void __launch_bounds__(SAMPLE_THREADS) sample_bwd_kernel(int B, int L, int K, const float* __restrict__ head,
                                                                    const float* __restrict__ log_var,
                                                                    const float* __restrict__ eps, const void* __restrict__ dz,
                                                                    const float* __restrict__ d_mu_direct,
                                                                    const float* __restrict__ d_lv_direct, int is_sampled,
                                                                    float* __restrict__ d_head) {
  const size_t i = (size_t)blockIdx.x * SAMPLE_THREADS + threadIdx.x;
  if (i >= (size_t)B * K) return;
  const int b = (int)(i / K), k = (int)(i - (size_t)b * K);
  const float lv = log_var[i];
  const float hs = 0.5f * expf(0.5f * lv) * (is_sampled ? 1.f : 0.f);
  float gm = d_mu_direct ? d_mu_direct[i] : 0.f;
  float gv = d_lv_direct ? d_lv_direct[i] : 0.f;
  if (dz) {
    for (int l = 0; l <= L; ++l) {
      const size_t idx = (size_t)l * B * K + i;
      const float g = DZ_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(dz)[idx])
                              : reinterpret_cast<const float*>(dz)[idx];
      gm += g;
      if (l >= 1) gv = fmaf(g * hs, eps[idx - (size_t)B * K], gv);
    }
  }
  const float raw = head[(size_t)b * 2 * K + K + k];
  if (!(raw >= -20.f && raw <= 20.f)) gv = 0.f;  // torch.clip backward (layers.py:394)
  d_head[(size_t)b * 2 * K + k] = gm;
  d_head[(size_t)b * 2 * K + K + k] = gv;
}

}  // namespace jvae

using namespace jvae;

extern "C" {

int jvae_sample_fwd(int B, int L, int K, const float* head, const float* eps_in, uint64_t seed, uint64_t offset,
                    const uint64_t* offset_dev, int is_sampled, int uniform, float* mu, float* log_var, float* z, void* z_bf16,
                    float* eps_out, float* eps_norm, void* stream) {
  JVAE_CHECK_ARG(B > 0 && L >= 0 && K > 0, "B, K > 0 and L >= 0");
  JVAE_CHECK_ARG(head != nullptr, "head is required");
  sample_fwd_kernel<<<B, SAMPLE_THREADS, 0, (cudaStream_t)stream>>>(B, L, K, head, eps_in, seed, offset, offset_dev,
                                                                     is_sampled, uniform, mu, log_var, z,
                                                                     reinterpret_cast<__nv_bfloat16*>(z_bf16), eps_out,
                                                                     eps_norm);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

int jvae_sample_bwd(int B, int L, int K, const float* head, const float* log_var, const float* eps, const void* dz,
                    int dz_dtype, const float* d_mu_direct, const float* d_lv_direct, int is_sampled, float* d_head,
                    void* stream) {
  JVAE_CHECK_ARG(B > 0 && L >= 0 && K > 0, "B, K > 0 and L >= 0");
  JVAE_CHECK_ARG(head && log_var && d_head, "head, log_var, d_head are required");
  JVAE_CHECK_ARG(!dz || L == 0 || eps, "eps is required with dz");
  const size_t n = (size_t)B * K;
  const int grid = (int)((n + SAMPLE_THREADS - 1) / SAMPLE_THREADS);
  if (dz_dtype == JVAE_BF16)
    sample_bwd_kernel<true><<<grid, SAMPLE_THREADS, 0, (cudaStream_t)stream>>>(B, L, K, head, log_var, eps, dz,
                                                                               d_mu_direct, d_lv_direct, is_sampled, d_head);
  else
    sample_bwd_kernel<false><<<grid, SAMPLE_THREADS, 0, (cudaStream_t)stream>>>(B, L, K, head, log_var, eps, dz,
                                                                                d_mu_direct, d_lv_direct, is_sampled, d_head);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

}  // extern "C"
