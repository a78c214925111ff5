// Dense bf16 GEMM on the tcgen05 tensor cores: D[M,N] = act(op(A) . op(B) + bias), fp32 accumulation in TMEM.
//
// Used for every nn.Linear of the path (module/vae_layers/layers.py:284-298, 441-453, 476-480 of the reference),
// their dgrad / wgrad, and the ConvTranspose2d-on-1x1 first deconv layer (conv-models.ini:25).
//
// One CTA computes a 128 x BN output tile.  Warp roles: warp 0 = TMA producer (one elected lane), warp 1 = TMEM
// allocator + MMA issuer (one elected lane), warps 2..5 = epilogue (TMEM -> registers -> global).  Operands are
// staged by TMA into a STAGES-deep ring of 128B-swizzled shared-memory tiles guarded by full/empty mbarriers.
// Operands may be K-major (reduction dimension contiguous) or MN-major (the "transposed" operand of dgrad / wgrad),
// selected per operand through the TMA box and the UMMA descriptors, so no transposed copies are ever made.
#include "tc_common.cuh"
#include <mutex>

namespace jvae {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_THREADS = 192;

struct GemmParams {
  int M, N, K, ldd, act, accumulate;
  int ksplit;      // > 1: gridDim.z slices of the reduction, partial results added to out_f32 with fp32 atomics
  int stages;      // ring depth actually used (<= GemmSmem::STAGES): short reductions take less shared memory, so several
                   // CTAs share an SM and their prologue / load / epilogue latencies overlap
  const float* bias;
  __nv_bfloat16* out_bf16;
  float* out_f32;
  // dropout (the DROPOUT kernels only): keep-mask of csrc/common.cuh at stream position drop_offset + *drop_offset_dev
  uint64_t seed, drop_offset, drop_thresh;
  const uint64_t* drop_offset_dev;
  float keep_scale;   // 1 / (1 - p); 0 when p == 1
};

template <int BN>
struct GemmSmem {
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;  // 16 KB
  static constexpr int B_BYTES = BN * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BN == 128) ? 6 : 8;
  static constexpr int BAR_OFFSET = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFFSET + 256 + 1024;  // barriers + alignment slack
};

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == JVAE_ACT_RELU) return fmaxf(v, 0.f);
  if (act == JVAE_ACT_SIGMOID) return 1.f / (1.f + __expf(-v));
  if (act == JVAE_ACT_LEAKY) return v > 0.f ? v : JVAE_LEAKY_SLOPE * v;
  return v;
}

// DROPOUT: the epilogue multiplies act(.) by keep(row, col) / (1 - p) (dense-layer dropout, layers.py:177-181, cvae.py:207-211)
template <int BN, bool A_MN, bool B_MN, bool DROPOUT>
__global__ void __launch_bounds__(GEMM_THREADS)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, GemmParams p) {
  using S = GemmSmem<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int STG = p.stages;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)STG * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STG;
  uint64_t* accum_bar = empty_bar + STG;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * GEMM_BM, n0 = blockIdx.y * BN;
  const int num_kb_all = (p.K + GEMM_BK - 1) / GEMM_BK;
  const int kb_per = p.ksplit > 1 ? (num_kb_all + p.ksplit - 1) / p.ksplit : num_kb_all;
  const int kb_lo = (int)blockIdx.z * kb_per;
  const int num_kb = min(kb_per, num_kb_all - kb_lo);       // k-blocks of this CTA's slice
  if (num_kb <= 0) return;                                  // empty tail slice (uniform for the CTA, before any barrier)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < STG; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc<BN>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % STG;
        const uint32_t ph = (kb / STG) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        uint8_t* sa = smem + s * S::STAGE_BYTES;
        uint8_t* sb = sa + S::A_BYTES;
        mbar_arrive_expect_tx(&full_bar[s], S::STAGE_BYTES);
        const int k0 = (kb_lo + kb) * GEMM_BK;
        if (!A_MN) {
          tma_load_2d(sa, &tmap_a, &full_bar[s], k0, m0);            // box {64 k, 128 m}
        } else {
          tma_load_2d(sa, &tmap_a, &full_bar[s], m0, k0);            // box {64 m, 64 k} x 2
          tma_load_2d(sa + 8192, &tmap_a, &full_bar[s], m0 + 64, k0);
        }
        if (!B_MN) {
          tma_load_2d(sb, &tmap_b, &full_bar[s], k0, n0);            // box {64 k, BN n}
        } else {
          tma_load_2d(sb, &tmap_b, &full_bar[s], n0, k0);            // box {64 n, 64 k} x BN/64
          if (BN == 128) tma_load_2d(sb + 8192, &tmap_b, &full_bar[s], n0 + 64, k0);
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      constexpr uint32_t idesc = make_idesc_bf16(GEMM_BM, BN, A_MN, B_MN);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % STG;
        const uint32_t ph = (kb / STG) & 1;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + s * S::STAGE_BYTES);
        const uint32_t sb = sa + S::A_BYTES;
        // K-major: rows of 128 B, 8-row groups 1024 B apart, k-step of 16 elements = +32 B
        // MN-major: 64-wide blocks 8192 B apart (LBO), 8-k-row groups 1024 B apart (SBO), k-step of 16 rows = +2048 B
        const uint64_t a_desc = A_MN ? make_smem_desc(sa, 8192, 1024, SWZ_128B) : make_smem_desc(sa, 16, 1024, SWZ_128B);
        const uint64_t b_desc = B_MN ? make_smem_desc(sb, 8192, 1024, SWZ_128B) : make_smem_desc(sb, 16, 1024, SWZ_128B);
#pragma unroll
        for (int k = 0; k < GEMM_BK / 16; ++k) {
          const uint64_t ad = a_desc + (uint64_t)((A_MN ? 2048 : 32) * k >> 4);
          const uint64_t bd = b_desc + (uint64_t)((B_MN ? 2048 : 32) * k >> 4);
          umma_bf16(tmem_base, ad, bd, idesc, (kb | k) != 0);
        }
        umma_commit(&empty_bar[s]);   // frees the smem slot once these MMAs have read it
      }
      umma_commit(accum_bar);         // accumulator complete
    }
  } else {
    // ================= epilogue: warps 2..5, TMEM lane quarter = warp % 4 =================
    const int q = warp & 3;
    // DROPOUT: the keep bits of the thread's row in the tile's BN columns (8 Philox draws per 32 columns), drawn while the
    // MMAs run; kb[0] always holds the current chunk's (shifted down once per chunk: no dynamically indexed registers)
    uint32_t kb[BN / 32];
    if (DROPOUT) {
      const uint64_t off = p.drop_offset + (p.drop_offset_dev ? *p.drop_offset_dev : 0ull);
#pragma unroll
      for (int c = 0; c < BN / 32; ++c) {
        kb[c] = 0;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          kb[c] |= dropout_keep4(p.seed, off, (uint32_t)(m0 + q * 32 + lane), (uint32_t)(n0 + c * 32 + j), p.drop_thresh) << j;
      }
    }
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    const int row = m0 + q * 32 + lane;
    const bool row_ok = row < p.M;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      if (n0 + c0 >= p.N) break;   // warp-uniform
      uint32_t keep = 0;
      if (DROPOUT) {
        keep = kb[0];
#pragma unroll
        for (int c = 0; c + 1 < BN / 32; ++c) kb[c] = kb[c + 1];
      }
      uint32_t r[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
      tmem_ld_wait();
      if (!row_ok) continue;
      // bias and activation are decided ONCE per chunk (the ncu source view of the K = 128 decoder GEMM showed ~57 instructions
      // per output element -- a bounds test, a scalar bias load and the activation switch each -- and 19 us per 128 x 128 tile)
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      if (p.bias) {
        if (n0 + c0 + 32 <= p.N && ((reinterpret_cast<uintptr_t>(p.bias + n0 + c0) & 15) == 0)) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c0 + j));
            v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
          }
        } else {
          for (int j = 0; j < 32; ++j)
            if (n0 + c0 + j < p.N) v[j] += __ldg(&p.bias[n0 + c0 + j]);
        }
      }
      if (p.act == JVAE_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
      } else if (p.act == JVAE_ACT_SIGMOID) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 1.f / (1.f + __expf(-v[j]));
      } else if (p.act == JVAE_ACT_LEAKY) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = v[j] > 0.f ? v[j] : JVAE_LEAKY_SLOPE * v[j];
      }
      if (DROPOUT) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = ((keep >> j) & 1u) ? v[j] * p.keep_scale : 0.f;
      }
      const size_t off = (size_t)row * p.ldd + n0 + c0;
      const bool full = (n0 + c0 + 32 <= p.N);
      if (p.out_f32 && p.ksplit > 1) {
        float* o = p.out_f32 + off;
        for (int j = 0; j < 32; ++j)
          if (n0 + c0 + j < p.N) atomicAdd(o + j, v[j]);
      } else if (p.out_f32) {
        float* o = p.out_f32 + off;
        if (full && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 t = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            if (p.accumulate) {
              const float4 old = *reinterpret_cast<float4*>(o + j);
              t.x += old.x; t.y += old.y; t.z += old.z; t.w += old.w;
            }
            *reinterpret_cast<float4*>(o + j) = t;
          }
        } else {
          for (int j = 0; j < 32; ++j)
            if (n0 + c0 + j < p.N) o[j] = p.accumulate ? o[j] + v[j] : v[j];
        }
      }
      if (p.out_bf16) {
        __nv_bfloat16* o = p.out_bf16 + off;
        if (full && ((reinterpret_cast<uintptr_t>(o) & 31) == 0)) {
#pragma unroll
          for (int j = 0; j < 32; j += 16)
            st_global_v8(o + j, pack_bf16(v[j], v[j + 1]), pack_bf16(v[j + 2], v[j + 3]), pack_bf16(v[j + 4], v[j + 5]),
                         pack_bf16(v[j + 6], v[j + 7]), pack_bf16(v[j + 8], v[j + 9]), pack_bf16(v[j + 10], v[j + 11]),
                         pack_bf16(v[j + 12], v[j + 13]), pack_bf16(v[j + 14], v[j + 15]));
        } else if (full && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            uint4 t;
            t.x = pack_bf16(v[j], v[j + 1]); t.y = pack_bf16(v[j + 2], v[j + 3]);
            t.z = pack_bf16(v[j + 4], v[j + 5]); t.w = pack_bf16(v[j + 6], v[j + 7]);
            *reinterpret_cast<uint4*>(o + j) = t;
          }
        } else {
          for (int j = 0; j < 32; ++j)
            if (n0 + c0 + j < p.N) o[j] = __float2bfloat16(v[j]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<BN>(tmem_base);
}

// ------------------------------------------------------------------------------------------------ host
PFN_cuTensorMapEncodeTiled_v12000 get_tmap_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, const uint32_t* elem_strides, int swizzle_bytes) {
  auto enc = get_tmap_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return JVAE_ERR_CUDA;
  }
  CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_NONE;
  if (swizzle_bytes == 128) sw = CU_TENSOR_MAP_SWIZZLE_128B;
  else if (swizzle_bytes == 64) sw = CU_TENSOR_MAP_SWIZZLE_64B;
  else if (swizzle_bytes == 32) sw = CU_TENSOR_MAP_SWIZZLE_32B;
  cuuint64_t gd[5], gs[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = elem_strides ? elem_strides[i] : 1;
    if (i > 0) gs[i - 1] = strides_bytes[i - 1];
  }
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d): rank %d dims [%llu,%llu,..] stride0 %llu box [%u,%u,..]", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 1 ? strides_bytes[0] : 0), box[0], rank > 1 ? box[1] : 0);
    return JVAE_ERR_CUDA;
  }
  return JVAE_OK;
}

// operand tensor map: K-major: dims {K, R}, box {64, rows}; MN-major: dims {R, K}, box {64, 64}
static int operand_tmap(CUtensorMap* t, const void* base, bool mn_major, int R, int K, int ld, int rows_box) {
  uint64_t dims[2], strides[1];
  uint32_t box[2];
  if (!mn_major) {
    dims[0] = (uint64_t)K; dims[1] = (uint64_t)R;
    box[0] = GEMM_BK; box[1] = (uint32_t)rows_box;
  } else {
    dims[0] = (uint64_t)R; dims[1] = (uint64_t)K;
    box[0] = 64; box[1] = GEMM_BK;
  }
  strides[0] = (uint64_t)ld * 2;
  return make_tmap_bf16(t, base, 2, dims, strides, box, nullptr, 128);
}

template <int BN, bool A_MN, bool B_MN, bool DROPOUT>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const GemmParams& p, cudaStream_t st) {
  using S = GemmSmem<BN>;
  static bool attr_done = false;
  if (!attr_done) {
    JVAE_CUDA(cudaFuncSetAttribute(gemm_bf16_kernel<BN, A_MN, B_MN, DROPOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    attr_done = true;
  }
  dim3 grid((p.M + GEMM_BM - 1) / GEMM_BM, (p.N + BN - 1) / BN, p.ksplit > 1 ? p.ksplit : 1);
  GemmParams q = p;
  const int num_kb_all = (p.K + GEMM_BK - 1) / GEMM_BK;
  const int num_kb = p.ksplit > 1 ? (num_kb_all + p.ksplit - 1) / p.ksplit : num_kb_all;
  q.stages = num_kb < S::STAGES ? (num_kb < 2 ? 2 : num_kb) : S::STAGES;
  const size_t smem = (size_t)q.stages * S::STAGE_BYTES + 256 + 1024;
  gemm_bf16_kernel<BN, A_MN, B_MN, DROPOUT><<<grid, GEMM_THREADS, smem, st>>>(ta, tb, q);
  JVAE_LAUNCH_CHECK();
  return JVAE_OK;
}

// argument checks, tensor maps and parameters shared by both entry points; *bn receives the N tile
static int prepare_gemm(int mode, int M, int N, int K, const void* a, int lda, const void* b, int ldb, const float* bias, int act,
                        void* out_bf16, float* out_f32, int ldd, float* col_stats, int accumulate, CUtensorMap* ta,
                        CUtensorMap* tb, GemmParams* p, int* bn) {
  JVAE_CHECK_ARG(mode >= JVAE_GEMM_NT && mode <= JVAE_GEMM_TN, "mode must be NT, NN or TN");
  JVAE_CHECK_ARG(M > 0 && N > 0 && K > 0, "M, N, K must be positive");
  JVAE_CHECK_ARG(a && b && (out_bf16 || out_f32), "a, b and one output are required");
  JVAE_CHECK_ARG((lda % 8) == 0 && (ldb % 8) == 0, "lda and ldb must be multiples of 8 elements (TMA 16-byte strides)");
  JVAE_CHECK_ARG((((uintptr_t)a | (uintptr_t)b) & 15) == 0, "a and b must be 16-byte aligned");
  JVAE_CHECK_ARG(ldd >= N, "ldd < N");
  JVAE_CHECK_ARG(!accumulate || out_f32, "accumulate needs out_f32");
  JVAE_CHECK_ARG(accumulate < 2 || (!out_bf16 && !bias && act == JVAE_ACT_NONE), "a split reduction only adds into out_f32");
  if (col_stats) {
    set_error("jvae_gemm_bf16: col_stats is only implemented by the convolution kernels");
    return JVAE_ERR_UNSUPPORTED;
  }
  const bool a_mn = (mode == JVAE_GEMM_TN);
  const bool b_mn = (mode != JVAE_GEMM_NT);
  JVAE_CHECK_ARG(lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K), "leading dimension smaller than the row length");
  const int BN = (N > 64) ? 128 : 64;
  int rc = operand_tmap(ta, a, a_mn, M, K, lda, GEMM_BM);
  if (rc) return rc;
  rc = operand_tmap(tb, b, b_mn, N, K, ldb, BN);
  if (rc) return rc;
  *p = GemmParams{};
  p->M = M; p->N = N; p->K = K; p->ldd = ldd; p->act = act; p->accumulate = accumulate ? 1 : 0;
  p->ksplit = accumulate >= 2 ? accumulate : 1;
  p->bias = bias; p->out_bf16 = reinterpret_cast<__nv_bfloat16*>(out_bf16); p->out_f32 = out_f32;
  *bn = BN;
  return JVAE_OK;
}

}  // namespace jvae

using namespace jvae;

extern "C" int jvae_gemm_bf16(int mode, int M, int N, int K, const void* a, int lda, const void* b, int ldb,
                              const float* bias, int act, void* out_bf16, float* out_f32, int ldd, float* col_stats,
                              int accumulate, void* stream) {
  CUtensorMap ta, tb;
  GemmParams p;
  int BN;
  const int rc = prepare_gemm(mode, M, N, K, a, lda, b, ldb, bias, act, out_bf16, out_f32, ldd, col_stats, accumulate, &ta,
                              &tb, &p, &BN);
  if (rc) return rc;
  const bool a_mn = (mode == JVAE_GEMM_TN);
  const bool b_mn = (mode != JVAE_GEMM_NT);
  cudaStream_t st = (cudaStream_t)stream;
#define JVAE_GEMM_CASE(bn, am, bm) return launch_gemm<bn, am, bm, false>(ta, tb, p, st)
  if (BN == 128) {
    if (!a_mn && !b_mn) JVAE_GEMM_CASE(128, false, false);
    if (!a_mn && b_mn) JVAE_GEMM_CASE(128, false, true);
    JVAE_GEMM_CASE(128, true, true);
  } else {
    if (!a_mn && !b_mn) JVAE_GEMM_CASE(64, false, false);
    if (!a_mn && b_mn) JVAE_GEMM_CASE(64, false, true);
    JVAE_GEMM_CASE(64, true, true);
  }
#undef JVAE_GEMM_CASE
}

extern "C" int jvae_gemm_bf16_dropout(int mode, int M, int N, int K, const void* a, int lda, const void* b, int ldb,
                                      const float* bias, int act, void* out_bf16, float* out_f32, int ldd, float* col_stats,
                                      int accumulate, float p, uint64_t seed, uint64_t offset, const uint64_t* offset_dev,
                                      void* stream) {
  JVAE_CHECK_ARG(p >= 0.f && p <= 1.f, "dropout probability p must be in [0, 1]");
  JVAE_CHECK_ARG(mode == JVAE_GEMM_NT, "dropout applies to the forward GEMM (mode NT)");
  JVAE_CHECK_ARG(accumulate == 0, "dropout does not accumulate or split the reduction");
  JVAE_CHECK_ARG(col_stats == nullptr, "dropout takes no col_stats");
  CUtensorMap ta, tb;
  GemmParams q;
  int BN;
  const int rc = prepare_gemm(mode, M, N, K, a, lda, b, ldb, bias, act, out_bf16, out_f32, ldd, nullptr, 0, &ta, &tb, &q, &BN);
  if (rc) return rc;
  q.seed = seed;
  q.drop_offset = offset;
  q.drop_offset_dev = offset_dev;
  q.drop_thresh = dropout_threshold(p);
  q.keep_scale = p < 1.f ? 1.f / (1.f - p) : 0.f;
  cudaStream_t st = (cudaStream_t)stream;
  if (BN == 128) return launch_gemm<128, false, false, true>(ta, tb, q, st);
  return launch_gemm<64, false, false, true>(ta, tb, q, st);
}
