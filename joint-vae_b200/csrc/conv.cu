// Implicit-GEMM convolutions on tcgen05 for NHWC bf16 activations: Conv2d (stride 1..8), ConvTranspose2d (stride 1, and
// stride s = 2..8 through its s*s sub-pixel phases), their data gradients (the same kernel with transformed weights / geometry) and the
// weight gradient (second kernel, MN-major operands, split over the pixel dimension).
//
// Replaces nn.Conv2d / nn.ConvTranspose2d of the reference's features / imager stacks
// (module/vae_layers/conv.py:189-219, conv-models.ini:11-30).
//
// Forward / dgrad kernel ("gather GEMM"): the output tile is 128 positions q = (image, y, x) of a TW x TH x NB box by
// BN output channels.  For every tap (dy,dx) of the filter the A operand is ONE TMA box load of the NHWC input at the
// shifted coordinate (q*stride + d): out-of-image rows / columns are zero-filled by TMA, which is the padding.  No
// im2col buffer exists anywhere.  B is the [BN x Cblk] slice of the pre-arranged weight matrix for that tap.
// The kernel is persistent (static round-robin over tiles) with a double-buffered TMEM accumulator so the epilogue
// of tile i overlaps the MMAs of tile i+1.
#include "tc_common.cuh"
#include <vector>
#include <algorithm>

namespace jvae {

constexpr int CONV_THREADS = 192;
constexpr int CONV_MAX_TAPS = 64;
// which kernel the last convolution entry point of this thread launched (jvae_last_conv_kernel: bench.py attributes its
// per-launch CUDA-event times to the dominant kernel with it)
static thread_local int g_last_conv_kernel = 0;

struct ConvParams {
  // iteration space
  int N, Hq, Wq;               // positions q: image, row, column
  int TW, TH, NB;              // tile box, TW*TH*NB == 128
  int tiles_x, tiles_y, tiles_n, num_tiles, n_tiles_n;  // n_tiles_n: output-channel tiles
  // reduction
  int Cblk, nCk, ntaps;        // channel chunk (16/32/64 elements = swizzle span), chunks per tap, taps
  int in_stride;               // input coordinate = q * in_stride + d
  short dy[CONV_MAX_TAPS], dx[CONV_MAX_TAPS];
  int BN;                      // output channels per CTA tile (multiple of 16, <= 256)
  // output
  int Ho, Wo, Cout, ldc;       // output tensor (N, Ho, Wo, ldc channels); Cout real channels written
  int out_sy, out_sx, out_oy, out_ox;   // output pixel = q * out_s + out_o
  int act;
  const float* bias;
  __nv_bfloat16* out;
  double* stats;               // (2, Cout) per-channel sum / sum of squares of the pre-activation, += (or null)
  int cout_pad;                // padded channel count (size of the shared-memory statistics accumulators)
  uint32_t stage_bytes, a_bytes, tx_bytes, tmem_cols;
  int stages;
};

// Sum of v[j] over the 32 lanes of a warp for 16 values at once (16 shuffles instead of 80): after the call the
// lane pair (2c, 2c+1) holds the warp total of v[c'] with c' = bit-reversed routing below, returned with its index.
__device__ __forceinline__ float warp_sum16(const float (&v)[16], int lane, int* channel) {
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
  float w[8], u[4], t[2];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float send = b4 ? v[j] : v[j + 8], keep = b4 ? v[j + 8] : v[j];
    w[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float send = b3 ? w[j] : w[j + 4], keep = b3 ? w[j + 4] : w[j];
    u[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const float send = b2 ? u[j] : u[j + 2], keep = b2 ? u[j + 2] : u[j];
    t[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  float s = (b1 ? t[1] : t[0]) + __shfl_xor_sync(0xffffffffu, b1 ? t[0] : t[1], 2);
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  *channel = (b4 ? 8 : 0) + (b3 ? 4 : 0) + (b2 ? 2 : 0) + (b1 ? 1 : 0);
  return s;
}

__device__ __forceinline__ void tmem_alloc_dyn(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc_dyn(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols));
}

constexpr int TAPBOX_THREADS = 320;     // TMA warp, MMA warp, 8 epilogue warps (two per TMEM lane quarter, alternating chunks)
__global__ void __launch_bounds__(TAPBOX_THREADS, 1)
conv_gather_gemm_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_w,
                        const __grid_constant__ ConvParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tfull_bar = empty_bar + p.stages;   // [2] accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;         // [2] accumulator drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  double* s_stats = reinterpret_cast<double*>(tmem_slot + 4);   // [2][cout_pad] when p.stats (fp64: order-independent sums)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kb_per_tile = p.ntaps * p.nCk;
  if (p.stats)
    for (int i = threadIdx.x; i < 2 * p.cout_pad; i += TAPBOX_THREADS) s_stats[i] = 0.0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_in);
    tma_prefetch_desc(&tmap_w);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 8);
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc_dyn(tmem_slot, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t acc_stride = p.tmem_cols >> 1;

  if (warp == 0) {
    // ================= TMA producer =================
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_tiles_n;
        int m = tile / p.n_tiles_n;
        const int tx = m % p.tiles_x; m /= p.tiles_x;
        const int ty = m % p.tiles_y; m /= p.tiles_y;
        const int x0 = tx * p.TW * p.in_stride, y0 = ty * p.TH * p.in_stride, n0 = m * p.NB;
        for (int t = 0; t < p.ntaps; ++t) {
          for (int c = 0; c < p.nCk; ++c, ++it) {
            const int s = it % p.stages;
            const uint32_t ph = (it / p.stages) & 1;
            mbar_wait(&empty_bar[s], ph ^ 1);
            uint8_t* sa = smem + (size_t)s * p.stage_bytes;
            mbar_arrive_expect_tx(&full_bar[s], p.tx_bytes);
            tma_load_4d(sa, &tmap_in, &full_bar[s], c * p.Cblk, x0 + p.dx[t], y0 + p.dy[t], n0);
            tma_load_2d(sa + p.a_bytes, &tmap_w, &full_bar[s], (t * p.nCk + c) * p.Cblk, nt * p.BN);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      const uint32_t idesc = make_idesc_bf16(128, p.BN, false, false);
      const uint32_t swz = (p.Cblk == 64) ? SWZ_128B : (p.Cblk == 32 ? SWZ_64B : SWZ_32B);
      const uint32_t sbo = 8u * (uint32_t)p.Cblk * 2u;      // 8 rows of Cblk bf16
      const int ksteps = p.Cblk >> 4;
      uint32_t it = 0, local = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++local) {
        const uint32_t acc = local & 1;
        mbar_wait(&tempty_bar[acc], ((local >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * acc_stride;
        for (int kb = 0; kb < kb_per_tile; ++kb, ++it) {
          const int s = it % p.stages;
          const uint32_t ph = (it / p.stages) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)s * p.stage_bytes);
          const uint64_t a_desc = make_smem_desc(sa, 16, sbo, swz);
          const uint64_t b_desc = make_smem_desc(sa + p.a_bytes, 16, sbo, swz);
          for (int k = 0; k < ksteps; ++k)
            umma_bf16(d_tmem, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (kb | k) != 0);
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&tfull_bar[acc]);
      }
    }
  } else {
    // ================= epilogue =================
    // two warps per TMEM lane quarter take alternate 16-channel chunks of a tile (the early vgg19 layers were drain-bound:
    // 36 MMAs of 64 cycles against ~250 epilogue instructions per chunk on one warp per scheduler)
    const int q = warp & 3, set = (warp - 2) >> 2;
    const int mrow = q * 32 + lane;
    const bool bias_vec = p.bias && ((reinterpret_cast<uintptr_t>(p.bias) & 15) == 0) && (p.Cout & 3) == 0;
    const int tx_in = mrow % p.TW, ty_in = (mrow / p.TW) % p.TH, nb_in = mrow / (p.TW * p.TH);
    uint32_t local = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++local) {
      const uint32_t acc = local & 1;
      const int nt = tile % p.n_tiles_n;
      int m = tile / p.n_tiles_n;
      const int tx = m % p.tiles_x; m /= p.tiles_x;
      const int ty = m % p.tiles_y; m /= p.tiles_y;
      const int qx = tx * p.TW + tx_in, qy = ty * p.TH + ty_in, n = m * p.NB + nb_in;
      const bool ok = (n < p.N) && (qy < p.Hq) && (qx < p.Wq);
      const int oy = qy * p.out_sy + p.out_oy, ox = qx * p.out_sx + p.out_ox;
      __nv_bfloat16* orow = p.out + (((size_t)n * p.Ho + oy) * p.Wo + ox) * p.ldc + (size_t)nt * p.BN;
      mbar_wait(&tfull_bar[acc], (local >> 1) & 1);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + acc * acc_stride + ((uint32_t)(q * 32) << 16);
      const int ch0 = nt * p.BN;
#pragma unroll 1
      for (int c0 = set * 16; c0 < p.BN; c0 += 32) {
        if (ch0 + c0 >= p.Cout) continue;       // warp-uniform
        uint32_t r[16];
        tmem_ld_32x16(t_addr + (uint32_t)c0, r);
        tmem_ld_wait();
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
        if (p.bias) {
          if (bias_vec && ch0 + c0 + 16 <= p.Cout) {
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + ch0 + c0 + j));
              v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (ch0 + c0 + j < p.Cout) v[j] += __ldg(&p.bias[ch0 + c0 + j]);
          }
        }
        if (!ok || ch0 + c0 + 16 > p.Cout) {     // rows outside the image / channels past Cout contribute nothing
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = (ok && ch0 + c0 + j < p.Cout) ? v[j] : 0.f;
        }
        if (p.stats) {      // batch statistics of the pre-activation (BatchNorm2d in train mode), fp32 accumulators
          float sq[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) sq[j] = v[j] * v[j];
          int chn;
          const float s1 = warp_sum16(v, lane, &chn);
          const float s2 = warp_sum16(sq, lane, &chn);
          if ((lane & 1) == 0 && ch0 + c0 + chn < p.Cout) {
            atomicAdd(&s_stats[ch0 + c0 + chn], (double)s1);
            atomicAdd(&s_stats[p.cout_pad + ch0 + c0 + chn], (double)s2);
          }
        }
        if (ok) {
          if (p.act == JVAE_ACT_RELU) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
          } else if (p.act == JVAE_ACT_SIGMOID) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = (ch0 + c0 + j < p.Cout) ? 1.f / (1.f + __expf(-v[j])) : 0.f;
          } else if (p.act == JVAE_ACT_LEAKY) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = v[j] > 0.f ? v[j] : JVAE_LEAKY_SLOPE * v[j];
          }
          if (ch0 + c0 + 16 <= p.ldc && (p.ldc & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 31) == 0) {
            st_global_v8(orow + c0, pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]),
                         pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
          } else if (ch0 + c0 + 16 <= p.ldc && (p.ldc & 7) == 0) {
            uint4 o0, o1;
            o0.x = pack_bf16(v[0], v[1]); o0.y = pack_bf16(v[2], v[3]); o0.z = pack_bf16(v[4], v[5]); o0.w = pack_bf16(v[6], v[7]);
            o1.x = pack_bf16(v[8], v[9]); o1.y = pack_bf16(v[10], v[11]); o1.z = pack_bf16(v[12], v[13]); o1.w = pack_bf16(v[14], v[15]);
            *reinterpret_cast<uint4*>(orow + c0) = o0;
            *reinterpret_cast<uint4*>(orow + c0 + 8) = o1;
          } else {
            for (int j = 0; j < 16; ++j)
              if (ch0 + c0 + j < p.ldc) orow[c0 + j] = __float2bfloat16(v[j]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
    }
    if (p.stats) {
      asm volatile("bar.sync 1, 256;" ::: "memory");       // the eight epilogue warps
      const int t = threadIdx.x - 64;
      for (int i = t; i < 2 * p.cout_pad; i += 256) {
        const int ch = i % p.cout_pad;
        const double val = s_stats[i];
        if (ch < p.Cout && val != 0.0) atomicAdd(&p.stats[(i / p.cout_pad) * p.Cout + ch], val);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc_dyn(tmem_base, p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// Halo-tile gather GEMM (input stride 1, one channel chunk): the A operand of EVERY filter tap is read out of ONE
// TMA-loaded halo box of the NHWC input.  A box is an 8-pixel-wide strip, RT output rows (+ the taps' vertical extent)
// of NBt consecutive images, stacked in shared memory as "slots" (rows of HWp = 8 + horizontal extent pixels).  An MMA
// M-tile is 16 consecutive slots x 8 pixels; for tap (dy,dx) its K-major descriptor simply starts (dy*HWp + dx) pixel
// rows further into the same box (8-row groups one slot = HWp pixel rows apart).  Shifted start addresses and arbitrary
// group strides are legal for swizzled K-major descriptors with base_offset 0: measured by jvae_probe_descriptors
// (profiles/r01_umma_descriptor_probe.txt).  Slots between two stacked images compute junk rows that are discarded;
// in exchange the input is read from L2 ~1.7x instead of 25x (k = 5), and the layer's weights stay resident in shared
// memory (or stream per tap when they do not fit, amortised over the MT M-tiles of the box).
// ------------------------------------------------------------------------------------------------
constexpr int HALO_MAX_CK = 128;
struct HaloParams {
  int N, Hq, Wq;
  int RT, NBt, HHs, HWp, MT;            // rows / images per box, slots per image, halo width (pixels), M-tiles per box
  int strips_x, blocks_y, blocks_n, num_boxes, n_tiles_n;
  int Cblk, ntaps, BN;
  int nkc;                               // input-channel chunks of Cblk (2: a 33..64-channel input in 32-channel chunks); 1 otherwise
  int dymin, dxmin;                      // smallest tap offset in PLANE coordinates (e = (d - r) / in_stride)
  int in_stride, nplanes;                // input stride s: the input is read as up to s*s parity planes P_r[j] = in[s*j + r]
  short plane_ry[4], plane_rx[4];
  uint32_t plane_bytes;                  // bytes of one plane's box region inside a stage
  short dy[CONV_MAX_TAPS], dx[CONV_MAX_TAPS];
  uint32_t tap_off16[CONV_MAX_TAPS];     // (plane * plane_bytes + ((ey-eymin)*HWp + (ex-exmin)) * row bytes) / 16
  int Ho, Wo, Cout, ldc, out_sy, out_sx, out_oy, out_ox, act;
  const float* bias;
  __nv_bfloat16* out;
  double* stats;
  int cout_pad;
  uint32_t stage_bytes, box_bytes, w_tap_bytes, w_bytes, tmem_cols, acc_stride;
  int stages, resident, wstages;
  // Vertical tap stacking (G > 1): one M row stands for G consecutive output rows (slots) of one pixel column; the N side of an
  // MMA stacks the weights of up to G vertically adjacent taps, D[(row group, px)][(j, co)] += X[slot g*G + u][px + x][ci] *
  // W[tap (e = u - j, x)][co][ci] for every j that has such a tap.  An MMA then does count * BN columns instead of BN for the
  // same A-operand fetch, which is what bounds the N <= 64 layers (DESIGN.md section 3.2).  Chunks = (plane, x, u) triples.
  int G, nck;
  // Merged sub-pixel phases (PH > 1, G == 1; jvae_conv_subpixel_gemm): the PH phases of a stride-2 transposed convolution are
  // computed from ONE box.  An M-tile owns PH accumulator blocks (one per phase, in the order the planner chose); a chunk is one
  // input shift whose MMA stacks the weights of every phase that has a tap at that shift along N (a run of consecutive blocks),
  // so the box is read once instead of once per phase launch and the epilogue writes whole output rows.  ph_oy / ph_ox: output
  // offset of the phase that owns block position i.
  int PH;
  short ph_oy[4], ph_ox[4];
  // one 16-byte record per chunk (ONE uniform load in the issue loop; the MMA thread was issue-bound at ~12 uniform
  // instructions per MMA when these were five byte / short tables and the instruction descriptor was rebuilt per chunk):
  //   x = A start shift (plane * plane_bytes + (u * HWp + x) * row bytes) / 16,  y = B start shift (first tap block) / 16,
  //   z = instruction descriptor (M = 128, N = count * BN),  w = first accumulator column (j0 * BN) | fresh << 31
  uint4 ck[HALO_MAX_CK];
  short w_pos[CONV_MAX_TAPS];            // position of tap t's weight block in shared memory (resident weights)
};

__device__ __forceinline__ int2 lds_int2(uint32_t addr) {
  int2 v;
  asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}

__device__ __forceinline__ uint64_t desc64(uint32_t hi, uint32_t lo) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}

// All MMAs of one box: taps outer, (M-tile, k-step) fully unrolled.  Descriptors are (hi, lo) words; only the low word
// (start address >> 4) moves: + tap_off16[t] per tap, + m_step16 per M-tile, + 2 per k-step.
template <int KSTEPS, int MT>
__device__ __forceinline__ void halo_mma_box(const HaloParams& p, uint32_t d0, uint32_t a_hi, uint32_t a_lo0, uint32_t m_step16,
                                             uint32_t b_hi, uint32_t b_lo_base, uint32_t w_tap16, uint32_t idesc,
                                             uint64_t* wfull_bar, uint64_t* wempty_bar, uint32_t& ws, uint32_t& wph,
                                             uint32_t later_chunk) {
  uint32_t b_lo = b_lo_base;
  for (int t = 0; t < p.ntaps; ++t) {
    if (!p.resident) {
      mbar_wait(&wfull_bar[ws], wph);
      tc_fence_after();
      b_lo = b_lo_base + ws * w_tap16;
    }
    const uint32_t a_lo = a_lo0 + p.tap_off16[t];
    const uint32_t acc_first = (t != 0) | later_chunk;      // the first tap of the first channel chunk overwrites
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
      for (int k = 0; k < KSTEPS; ++k)
        umma_bf16(d0 + (uint32_t)(m * p.BN), desc64(a_hi, a_lo + (uint32_t)m * m_step16 + 2u * k), desc64(b_hi, b_lo + 2u * k), idesc,
                  k == 0 ? acc_first : 1u);
    if (p.resident) {
      b_lo += w_tap16;
    } else {
      umma_commit(&wempty_bar[ws]);
      if (++ws == (uint32_t)p.wstages) { ws = 0; wph ^= 1; }
    }
  }
}

// All MMAs of one box with vertical tap stacking (HaloParams::G > 1): M-tiles outer, chunks inner.  The chunks flagged fresh come
// first and cover every column block of the tile exactly once (they overwrite), the others accumulate.
template <int KSTEPS>
__device__ __forceinline__ void halo_mma_box_g(const HaloParams& p, uint32_t d0, uint32_t a_hi, uint32_t a_lo0, uint32_t m_step16,
                                               uint32_t b_hi, uint32_t b_lo_base, uint32_t idesc0, uint32_t later_chunk) {
  const uint32_t gbn = (uint32_t)(p.G * p.PH * p.BN);
  for (int m = 0; m < p.MT; ++m) {
    const uint32_t a_m = a_lo0 + (uint32_t)m * m_step16;
    const uint32_t d_m = d0 + (uint32_t)m * gbn;
    for (int c = 0; c < p.nck; ++c) {
      const uint4 ck = p.ck[c];
      const uint32_t a_lo = a_m + ck.x, b_lo = b_lo_base + ck.y;
      const uint32_t d = d_m + (ck.w & 0x7fffffffu);
      const uint32_t idesc = ck.z;
      const uint32_t acc0 = ((ck.w >> 31) ^ 1u) | later_chunk;      // fresh chunks overwrite only in the first channel chunk
#pragma unroll
      for (int k = 0; k < KSTEPS; ++k)
        umma_bf16(d, desc64(a_hi, a_lo + 2u * k), desc64(b_hi, b_lo + 2u * k), idesc, k == 0 ? acc0 : 1u);
    }
  }
}

// Epilogue of the halo kernel, run by EIGHT warps.  The ncu source view of the
// generic role above showed ~420 warp instructions per 32-channel accumulator block, of which ~90 are the work, executed by one
// epilogue warp per scheduler at an IPC of 0.15: the accumulator drain, not the MMAs, paced the narrow layers (the MMA thread
// spent its time waiting for a free accumulator).  Two changes:
//   * a per-thread table in shared memory holds, for each of the MT * G accumulator blocks of a box, the thread's output offset
//     from the box origin and its (row, image) inside the box: a block costs one 8-byte shared load and four compares instead of
//     a division and the pointer arithmetic; rows that are not written skip the arithmetic, dead blocks skip the TMEM load;
//   * two warps per TMEM lane quarter (set = 0 / 1): a set takes every other 16-channel chunk of each block (every other block
//     for 16-channel tiles), so a scheduler interleaves two independent drains and a thread keeps statistics for at most 32
//     channels.
// STATS: BatchNorm batch statistics of the output (sum y, sum y^2).
template <int NCH, bool STATS>
__device__ __forceinline__ void halo_epilogue_fast(const HaloParams& p, uint32_t tmem_base, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                                   double* s_stats, const float* s_bias, int2* s_tab, int warp, int lane, int nt,
                                                   int box0, int box_step) {
  constexpr int LC = (NCH + 1) / 2;              // chunks a thread handles at most
  const int set = (warp - 2) >> 2;               // warps 2..5: set 0, warps 6..9: set 1
  const int q = warp & 3;
  const int mrow = q * 32 + lane;
  const int ch0 = nt * p.BN;
  const int per = p.G * p.PH;                    // accumulator blocks of an M-tile: (row j of the group, phase)
  const int nblk = p.MT * per;
  const int c_first = NCH == 1 ? 0 : set;        // chunks c_first, c_first + 2
  // the table does not depend on the pixel column of a row: 16 entries (slot groups of an M-tile) per block
  for (int i = threadIdx.x - 64; i < nblk * 16; i += 256) {
    const int blk = i >> 4;
    const int m = blk / per, r = blk - m * per;
    const int j = r / p.PH, ph = r - j * p.PH;
    const int slot = (m * 16 + (i & 15)) * p.G + j;
    const int nb = slot / p.HHs, yy = slot - nb * p.HHs;
    const bool valid = nb < p.NBt && yy < p.RT;
    s_tab[i] = make_int2(valid ? (nb * p.Ho + yy * p.out_sy + p.ph_oy[ph]) * p.Wo + p.ph_ox[ph] : -1,
                         yy | (nb << 16));      // pixel offset from the box origin
  }
  asm volatile("bar.sync 1, 256;" ::: "memory");      // the table is shared by the two warps of a lane quarter
  float s1[STATS ? LC * 16 : 1], s2[STATS ? LC * 16 : 1];
  if (STATS) {
#pragma unroll
    for (int j = 0; j < LC * 16; ++j) s1[j] = s2[j] = 0.f;
  }
  const bool has_bias = p.bias != nullptr;
  const uint32_t sb = smem_u32(s_bias);
  const uint32_t stab = smem_u32(s_tab) + 8u * (uint32_t)(mrow >> 3);      // this thread's entry of block 0
  const bool vec_bf16 = (p.ldc & 7) == 0;
  // 32-byte stores (st.global.v8.b32) when the thread's 16 channels start on a 32-byte boundary: one full sector per instruction
  // instead of two half sectors (the scattered 16-byte stores of the sub-pixel / narrow layers kept L1TEX 67 % busy)
  const bool al32 = (reinterpret_cast<uintptr_t>(p.out) & 31) == 0;
  const bool v8_bf16 = al32 && (p.ldc & 15) == 0;
  uint32_t it = 0;
  // (strip, row block, image block) of the box, advanced by the decomposition of box_step with carries: the two runtime
  // divisions per box were a fifth of the epilogue's stall samples on launches with few blocks per box (ncu source view)
  int sx, by, mm, dsx, dby, dmm;
  {
    int t = box0;
    sx = t % p.strips_x; t /= p.strips_x;
    by = t % p.blocks_y; mm = t / p.blocks_y;
    t = box_step;
    dsx = t % p.strips_x; t /= p.strips_x;
    dby = t % p.blocks_y; dmm = t / p.blocks_y;
  }
  for (int box = box0; box < p.num_boxes; box += box_step, ++it) {
    const uint32_t acc = it & 1;
    if (it != 0) {
      sx += dsx;
      if (sx >= p.strips_x) { sx -= p.strips_x; ++by; }
      by += dby;
      if (by >= p.blocks_y) { by -= p.blocks_y; ++mm; }
      mm += dmm;
    }
    const int qx = sx * 8 + (mrow & 7);
    const bool pxok = qx < p.Wq;
    const int ylim = p.Hq - by * p.RT, nlim = p.N - mm * p.NBt;
    const size_t pix0 = ((size_t)(mm * p.NBt) * p.Ho + (size_t)(by * p.RT * p.out_sy + p.out_oy)) * p.Wo +
                        (size_t)(qx * p.out_sx + p.out_ox);
    mbar_wait(&tfull_bar[acc], (it >> 1) & 1);
    tc_fence_after();
    constexpr int BSTEP = NCH == 1 ? 2 : 1;
    int2 e_next = lds_int2(stab + 8u * (uint32_t)(NCH == 1 ? set : 0) * 16u);
    for (int blk = (NCH == 1 ? set : 0); blk < nblk; blk += BSTEP) {
      // the table entry of the NEXT block is requested now: its latency used to head the dependent chain of every block
      // (ncu source view of the merged sub-pixel launch: the top stall after the accumulator wait)
      const int2 e = e_next;
      if (blk + BSTEP < nblk) e_next = lds_int2(stab + 8u * (uint32_t)(blk + BSTEP) * 16u);
      const bool ok = pxok && e.x >= 0 && (e.y & 0xffff) < ylim && (e.y >> 16) < nlim;
      if (!__any_sync(0xffffffffu, ok)) continue;
      const uint32_t t_addr = tmem_base + acc * p.acc_stride + (uint32_t)(blk * p.BN) + ((uint32_t)(q * 32) << 16);
      const size_t pix = pix0 + (size_t)(ok ? e.x : 0);
      // the bias of the thread's channels is requested BEFORE the accumulator (its latency hides under the TMEM load, and the
      // sum lands in the accumulator's own registers: with the loads after the wait the compiler copied all 16 values away
      // and back, 32 of ~145 instructions per block)
      float bq[LC][16];
      if (has_bias) {
#pragma unroll
        for (int lc = 0; lc < LC; ++lc)
          if (c_first + 2 * lc < NCH) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                           : "=f"(bq[lc][j]), "=f"(bq[lc][j + 1]), "=f"(bq[lc][j + 2]), "=f"(bq[lc][j + 3])
                           : "r"(sb + 4u * ((c_first + 2 * lc) * 16 + j)));
          }
      }
      uint32_t r[LC][16];
#pragma unroll
      for (int lc = 0; lc < LC; ++lc)
        if (c_first + 2 * lc < NCH) tmem_ld_32x16(t_addr + (uint32_t)((c_first + 2 * lc) * 16), r[lc]);
      tmem_ld_wait();
      if (!ok) continue;
#pragma unroll
      for (int lc = 0; lc < LC; ++lc) {
        const int c = c_first + 2 * lc;
        if (c >= NCH || ch0 + c * 16 >= p.Cout) continue;      // warp-uniform
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[lc][j]);
        if (has_bias) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] += bq[lc][j];
        }
        if (STATS) {
#pragma unroll
          for (int j = 0; j < 16; ++j) { s1[lc * 16 + j] += v[j]; s2[lc * 16 + j] = fmaf(v[j], v[j], s2[lc * 16 + j]); }
          // keeps the sums ahead of the activation: sunk below it they needed a second copy of the 16 values (32 moves per block)
#pragma unroll
          for (int j = 0; j < 16; ++j) asm volatile("" : "+f"(v[j]));
        }
        if (p.act != JVAE_ACT_NONE) {      // one uniform test in the common case (BatchNorm layers, data gradients)
          if (p.act == JVAE_ACT_RELU) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
          } else if (p.act == JVAE_ACT_SIGMOID) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = 1.f / (1.f + __expf(-v[j]));
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = v[j] > 0.f ? v[j] : JVAE_LEAKY_SLOPE * v[j];
          }
        }
        const int c0 = c * 16;
        __nv_bfloat16* o = p.out + pix * (size_t)p.ldc + (size_t)(ch0 + c0);
        if (ch0 + c0 + 16 <= p.ldc && v8_bf16) {
          st_global_v8(o, pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]),
                       pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
        } else if (ch0 + c0 + 16 <= p.ldc && vec_bf16) {
          uint4 o0, o1;
          o0.x = pack_bf16(v[0], v[1]); o0.y = pack_bf16(v[2], v[3]); o0.z = pack_bf16(v[4], v[5]); o0.w = pack_bf16(v[6], v[7]);
          o1.x = pack_bf16(v[8], v[9]); o1.y = pack_bf16(v[10], v[11]); o1.z = pack_bf16(v[12], v[13]); o1.w = pack_bf16(v[14], v[15]);
          *reinterpret_cast<uint4*>(o) = o0;
          *reinterpret_cast<uint4*>(o + 8) = o1;
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (ch0 + c0 + j < p.ldc) o[j] = __float2bfloat16(ch0 + c0 + j < p.Cout ? v[j] : 0.f);
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&tempty_bar[acc]);
  }
  if (STATS) {
    // CTA-level reduction of the per-thread sums: warp butterfly (16 values at a time), then shared + global atomics
#pragma unroll
    for (int lc = 0; lc < LC; ++lc) {
      const int c = c_first + 2 * lc;
      float a[16], b[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) { a[j] = s1[STATS ? lc * 16 + j : 0]; b[j] = s2[STATS ? lc * 16 + j : 0]; }
      int chn;
      const float t1 = warp_sum16(a, lane, &chn);
      const float t2 = warp_sum16(b, lane, &chn);
      if (c < NCH && (lane & 1) == 0 && ch0 + c * 16 + chn < p.Cout) {
        atomicAdd(&s_stats[ch0 + c * 16 + chn], (double)t1);
        atomicAdd(&s_stats[p.cout_pad + ch0 + c * 16 + chn], (double)t2);
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const int t = threadIdx.x - 64;
    for (int i = t; i < 2 * p.cout_pad; i += 256) {
      const int ch = i % p.cout_pad;
      const double val = s_stats[i];
      if (ch < p.Cout && val != 0.0) atomicAdd(&p.stats[(i / p.cout_pad) * p.Cout + ch], val);
    }
  }
}

constexpr int HALO_THREADS = 320;      // TMA warp, MMA warp, 8 epilogue warps (two per TMEM lane quarter)
__global__ void __launch_bounds__(HALO_THREADS, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap tmap_in, const __grid_constant__ CUtensorMap tmap_w,
                 const __grid_constant__ HaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* wsm = smem + (size_t)p.stages * p.stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(wsm + p.w_bytes);
  uint64_t* empty_bar = full_bar + 4;
  uint64_t* wfull_bar = empty_bar + 4;      // [wstages] (resident: only [0])
  uint64_t* wempty_bar = wfull_bar + 8;
  uint64_t* tfull_bar = wempty_bar + 8;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  double* s_stats = reinterpret_cast<double*>(tmem_slot + 4);              // [2][cout_pad] when p.stats (fp64 sums)
  float* s_bias = reinterpret_cast<float*>(s_stats + (p.stats ? 2 * p.cout_pad : 0));   // [BN] bias of this CTA's channel tile

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nt = (int)blockIdx.x % p.n_tiles_n;
  int2* s_tab = reinterpret_cast<int2*>(s_bias + 64);                      // [MT * G][16]: block table of the fast epilogue
  for (int i = threadIdx.x; i < p.BN; i += HALO_THREADS) {
    const int ch = nt * p.BN + i;
    s_bias[i] = (p.bias && ch < p.Cout) ? p.bias[ch] : 0.f;
  }
  const int box0 = (int)blockIdx.x / p.n_tiles_n, box_step = (int)gridDim.x / p.n_tiles_n;
  const uint32_t rb = (uint32_t)p.Cblk * 2u;

  if (p.stats)
    for (int i = threadIdx.x; i < 2 * p.cout_pad; i += HALO_THREADS) s_stats[i] = 0.0;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_in);
    tma_prefetch_desc(&tmap_w);
    for (int s = 0; s < 4; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 8; ++s) { mbar_init(&wfull_bar[s], 1); mbar_init(&wempty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 8); }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc_dyn(tmem_slot, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      if (p.resident) {      // every channel chunk's weights (nkc > 1: two 32-channel chunks of a 64-channel input)
        mbar_arrive_expect_tx(&wfull_bar[0], (uint32_t)(p.ntaps * p.nkc) * p.w_tap_bytes);
        for (int kc = 0; kc < p.nkc; ++kc)
          for (int t = 0; t < p.ntaps; ++t)
            tma_load_2d(wsm + (size_t)(kc * p.ntaps + (p.nck > 0 ? p.w_pos[t] : t)) * p.w_tap_bytes, &tmap_w, &wfull_bar[0],
                        (t * p.nkc + kc) * p.Cblk, nt * p.BN);
      }
      // one shared-memory stage per unit = (box, input-channel chunk); the unit after the current one is requested before the
      // current unit's weights (streamed per tap when they are not resident)
      auto load_unit = [&](int box, int kc, uint32_t iu) {
        int m = box;
        const int sx = m % p.strips_x; m /= p.strips_x;
        const int by = m % p.blocks_y; m /= p.blocks_y;
        const int s = iu % p.stages;
        mbar_wait(&empty_bar[s], ((iu / p.stages) & 1) ^ 1);
        mbar_arrive_expect_tx(&full_bar[s], p.box_bytes);
        for (int pl = 0; pl < p.nplanes; ++pl)
          tma_load_4d(smem + (size_t)s * p.stage_bytes + (size_t)pl * p.plane_bytes, &tmap_in, &full_bar[s], kc * p.Cblk,
                      p.in_stride * (sx * 8 + p.dxmin) + p.plane_rx[pl], p.in_stride * (by * p.RT + p.dymin) + p.plane_ry[pl],
                      m * p.NBt);
      };
      uint32_t iu = 0, wit = 0;
      if (box0 < p.num_boxes) load_unit(box0, 0, 0);
      for (int box = box0; box < p.num_boxes; box += box_step) {
        for (int kc = 0; kc < p.nkc; ++kc, ++iu) {
          if (kc + 1 < p.nkc) load_unit(box, kc + 1, iu + 1);
          else if (box + box_step < p.num_boxes) load_unit(box + box_step, 0, iu + 1);
          if (!p.resident) {
            for (int t = 0; t < p.ntaps; ++t, ++wit) {
              const int ws = wit % p.wstages;
              mbar_wait(&wempty_bar[ws], ((wit / p.wstages) & 1) ^ 1);
              mbar_arrive_expect_tx(&wfull_bar[ws], p.w_tap_bytes);
              tma_load_2d(wsm + (size_t)ws * p.w_tap_bytes, &tmap_w, &wfull_bar[ws], (t * p.nkc + kc) * p.Cblk, nt * p.BN);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      const uint32_t idesc = make_idesc_bf16(128, p.BN, false, false);
      const uint32_t swz = (p.Cblk == 64) ? SWZ_128B : (p.Cblk == 32 ? SWZ_64B : SWZ_32B);
      const uint32_t sbo_a = (uint32_t)(p.G * p.HWp) * rb, sbo_b = 8u * rb;      // 8-row groups of A: one slot (row group) apart
      // descriptor words: lo = start >> 4 | LBO(16 B) << 16; hi = SBO >> 4 | version 1 << 14 | swizzle << 29
      const uint32_t a_hi = ((sbo_a >> 4) & 0x3fffu) | (1u << 14) | (swz << 29);
      const uint32_t b_hi = ((sbo_b >> 4) & 0x3fffu) | (1u << 14) | (swz << 29);
      const uint32_t m_step16 = (16u * sbo_a) >> 4, w_tap16 = p.w_tap_bytes >> 4;
      const int ksteps = p.Cblk >> 4;
      if (p.resident) { mbar_wait(&wfull_bar[0], 0); tc_fence_after(); }
      uint32_t it = 0, s = 0, sph = 0, ws = 0, wph = 0;
      for (int box = box0; box < p.num_boxes; box += box_step, ++it) {
        const uint32_t acc = it & 1;
        mbar_wait(&tempty_bar[acc], ((it >> 1) & 1) ^ 1);
        const uint32_t d0 = tmem_base + acc * p.acc_stride;
        const uint32_t b_lo = ((smem_u32(wsm) >> 4) & 0x3fffu) | (1u << 16);
        for (int kc = 0; kc < p.nkc; ++kc) {
          mbar_wait(&full_bar[s], sph);
          tc_fence_after();
          const uint32_t a_lo0 = ((smem_u32(smem + (size_t)s * p.stage_bytes) >> 4) & 0x3fffu) | (1u << 16);
          const uint32_t later = kc != 0;
#define HALO_BOX(KS, M) halo_mma_box<KS, M>(p, d0, a_hi, a_lo0, m_step16, b_hi, b_lo, w_tap16, idesc, wfull_bar, wempty_bar, ws, wph, later)
#define HALO_BOX_M(KS)                                                                 \
          switch (p.MT) {                                                              \
            case 1: HALO_BOX(KS, 1); break;                                            \
            case 2: HALO_BOX(KS, 2); break;                                            \
            case 3: HALO_BOX(KS, 3); break;                                            \
            case 4: HALO_BOX(KS, 4); break;                                            \
            default: HALO_BOX(KS, 5); break;                                           \
          }
          if (p.nck > 0) {
            const uint32_t idesc0 = make_idesc_bf16(128, 0, false, false);
            const uint32_t b_kc = b_lo + (uint32_t)(kc * p.ntaps) * w_tap16;      // this chunk's resident weights
            if (ksteps == 2) halo_mma_box_g<2>(p, d0, a_hi, a_lo0, m_step16, b_hi, b_kc, idesc0, later);
            else if (ksteps == 4) halo_mma_box_g<4>(p, d0, a_hi, a_lo0, m_step16, b_hi, b_kc, idesc0, later);
            else halo_mma_box_g<1>(p, d0, a_hi, a_lo0, m_step16, b_hi, b_kc, idesc0, later);
          } else if (ksteps == 2) { HALO_BOX_M(2) } else if (ksteps == 4) { HALO_BOX_M(4) } else { HALO_BOX_M(1) }
#undef HALO_BOX_M
#undef HALO_BOX
          umma_commit(&empty_bar[s]);
          if (++s == (uint32_t)p.stages) { s = 0; sph ^= 1; }
        }
        umma_commit(&tfull_bar[acc]);
      }
    }
  } else {
    // ================= epilogue =================
#define HALO_EPI_FAST(NCH_)                                                                                                      \
    if (p.stats) halo_epilogue_fast<NCH_, true>(p, tmem_base, tfull_bar, tempty_bar, s_stats, s_bias, s_tab, warp, lane, nt, box0, box_step); \
    else halo_epilogue_fast<NCH_, false>(p, tmem_base, tfull_bar, tempty_bar, s_stats, s_bias, s_tab, warp, lane, nt, box0, box_step)
    switch (p.BN >> 4) {
      case 1: HALO_EPI_FAST(1); break;
      case 2: HALO_EPI_FAST(2); break;
      case 3: HALO_EPI_FAST(3); break;
      default: HALO_EPI_FAST(4); break;
    }
#undef HALO_EPI_FAST
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc_dyn(tmem_base, p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// weight gradient: dW[tap][co][ci] = sum_q dY[q, co] * X[q*stride + d_tap, ci]
// Both operands are NHWC tiles whose contiguous dimension (channels) is the M / N dimension of the GEMM and whose
// rows (pixels) are the reduction: MN-major descriptors on the same TMA boxes the forward kernel uses.
// Each CTA owns a slice of the pixel tiles and a group of taps; partial sums are reduced with fp32 atomics.
// ------------------------------------------------------------------------------------------------
struct WgradParams {
  int N, Hq, Wq, TW, TH, NB, tiles_x, tiles_y, tiles_n, num_tiles;
  int Cblk_y, Cblk_x;          // channel block of dY (M side, 64 max) and X (N side)
  int Cy, Cx, ncx;             // channels of dY / X; blockIdx.z = (dY block) * ncx + (X block)
  int ntaps, tap0, taps_per_cta, in_stride;
  short dy[CONV_MAX_TAPS], dx[CONV_MAX_TAPS];
  float* dw;                   // (ntaps_total, Cout, Cin) fp32, accumulated atomically
  int dw_ld_tap, dw_ld_co, dw_ld_cx;     // strides of dw in elements (tap, dY channel, X channel)
  uint32_t stage_bytes, a_bytes, tx_bytes, tmem_cols;
  int stages;
};

__global__ void __launch_bounds__(CONV_THREADS, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap tmap_dy, const __grid_constant__ CUtensorMap tmap_x,
                  const __grid_constant__ WgradParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* done_bar = empty_bar + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tap_lo = p.tap0 + blockIdx.y * p.taps_per_cta;
  const int ntap = min(p.taps_per_cta, p.ntaps - tap_lo);
  const int cy0 = ((int)blockIdx.z / p.ncx) * p.Cblk_y, cx0 = ((int)blockIdx.z % p.ncx) * p.Cblk_x;
  const int M_real = min(p.Cblk_y, p.Cy - cy0), N_real = min(p.Cblk_x, p.Cx - cx0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_dy);
    tma_prefetch_desc(&tmap_x);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(done_bar, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc_dyn(tmem_slot, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t x_bytes = 128u * (uint32_t)p.Cblk_x * 2u;

  if (warp == 0) {
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        int m = tile;
        const int tx = m % p.tiles_x; m /= p.tiles_x;
        const int ty = m % p.tiles_y; m /= p.tiles_y;
        const int n0 = m * p.NB;
        // stage layout: [dY tile (128 x Cblk_y)] [X tile per tap ...]: one stage = dY + ONE tap's X tile
        for (int t = 0; t < ntap; ++t, ++it) {
          const int s = it % p.stages;
          const uint32_t ph = (it / p.stages) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* sa = smem + (size_t)s * p.stage_bytes;
          mbar_arrive_expect_tx(&full_bar[s], p.tx_bytes);
          tma_load_4d(sa, &tmap_dy, &full_bar[s], cy0, tx * p.TW, ty * p.TH, n0);
          tma_load_4d(sa + p.a_bytes, &tmap_x, &full_bar[s], cx0, tx * p.TW * p.in_stride + p.dx[tap_lo + t],
                      ty * p.TH * p.in_stride + p.dy[tap_lo + t], n0);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {      // one elected lane (elect.sync lets the compiler keep descriptors in uniform registers)
      // D[M = dY channels (64 rows), N = X channels] += dY^T[M x 128 px] * X[128 px x N]; both MN-major
      const uint32_t idesc = make_idesc_bf16(64, p.Cblk_x, true, true);
      const uint32_t swz_y = (p.Cblk_y == 64) ? SWZ_128B : (p.Cblk_y == 32 ? SWZ_64B : SWZ_32B);
      const uint32_t swz_x = (p.Cblk_x == 64) ? SWZ_128B : (p.Cblk_x == 32 ? SWZ_64B : SWZ_32B);
      const uint32_t row_y = (uint32_t)p.Cblk_y * 2u, row_x = (uint32_t)p.Cblk_x * 2u;
      uint32_t it = 0;
      bool first_tile = true;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        for (int t = 0; t < ntap; ++t, ++it) {
          const int s = it % p.stages;
          const uint32_t ph = (it / p.stages) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)s * p.stage_bytes);
          // MN-major: one block of Cblk channels wide; 8-pixel groups are 8 rows apart (SBO); LBO (next channel block)
          // is unused for a single block but must be valid: point it at the same block
          const uint64_t a_desc = make_smem_desc(sa, 8 * row_y, 8 * row_y, swz_y);
          const uint64_t b_desc = make_smem_desc(sa + p.a_bytes, 8 * row_x, 8 * row_x, swz_x);
          const uint32_t d_tmem = tmem_base + (uint32_t)(t * p.Cblk_x);
#pragma unroll
          for (int k = 0; k < 8; ++k)   // 128 pixels = 8 x K16
            umma_bf16(d_tmem, a_desc + (uint64_t)((16 * row_y * k) >> 4), b_desc + (uint64_t)((16 * row_x * k) >> 4), idesc,
                      (!first_tile || k != 0));
          umma_commit(&empty_bar[s]);
        }
        first_tile = false;
      }
      umma_commit(done_bar);
    }
  } else {
    // epilogue: accumulator rows = dY channels (M = 64: TMEM lanes 0..15 of each lane quarter hold rows 16q..16q+15),
    // columns = taps x X channels
    const int q = warp & 3;
    mbar_wait(done_bar, 0);
    tc_fence_after();
    const bool has_work = blockIdx.x < p.num_tiles;
    for (int t = 0; t < ntap && has_work; ++t) {
      for (int c0 = 0; c0 < p.Cblk_x; c0 += 16) {
        uint32_t r[16];
        tmem_ld_32x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(t * p.Cblk_x + c0), r);
        tmem_ld_wait();
        const int row = q * 16 + lane;     // valid for lane < 16
        if (lane < 16 && row < M_real) {
          float* o = p.dw + (size_t)(tap_lo + t) * p.dw_ld_tap + (size_t)(cy0 + row) * p.dw_ld_co + (size_t)(cx0 + c0) * p.dw_ld_cx;
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (c0 + j < N_real) atomicAdd(o + (size_t)j * p.dw_ld_cx, __uint_as_float(r[j]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc_dyn(tmem_base, p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------
// Halo-tile weight gradient (input stride 1):  dW[t][a][b] += sum_px G[px, a] * X[px + d_t, b]
// G = grid tensor (dY for a Conv2d, x for a ConvTranspose2d), X = gathered tensor.  K of the MMA = pixels; both
// operands are MN-major views of NHWC boxes.  The X box is the same stacked halo box the forward kernel uses; up to
// 128 / Cblk_x horizontally adjacent taps are ONE MMA: they are stacked along M through the descriptor's leading byte
// offset (LBO = one pixel row).  D[(tap j, X channel)][G channel] accumulates in TMEM over every box the CTA owns;
// one epilogue at the end adds it to dW with fp32 atomics.  Junk slots between stacked images contribute nothing
// because the G box is zero there (rows beyond the image are TMA OOB fill); stage slack is zeroed once.
// ------------------------------------------------------------------------------------------------
constexpr int WH_MAX_GROUPS = 64;
struct WHaloParams {
  int N, Hq, Wq;
  int NBt, HHs, HWp, MT, strips_x, num_boxes;
  int RT, blocks_y;                         // rows per box and row blocks per image (maps taller than 32 rows)
  uint32_t g_img_bytes;                     // blocks_y > 1: the gradient tile arrives image by image (RT rows each, HHs slots apart)
  int Cblk_g, Cblk_x, ncx, Cg, Cx;          // blockIdx.z = (G channel block) * ncx + (X channel block)
  int ngroups, groups_per_cta;              // blockIdx.y selects a slice of the tap groups
  int dymin, dxmin, ey;                     // smallest tap offset in plane coordinates; vertical extent of the window
  int in_stride, nplanes;                   // gathered tensor read as parity planes X_r[j] = X[s*j + r]
  short plane_ry[4], plane_rx[4];
  uint32_t plane_bytes;
  uint32_t grp_off16[WH_MAX_GROUPS];        // A (gathered tensor) descriptor start shift of the group's first tap (16-byte units)
  unsigned char grp_ntap[WH_MAX_GROUPS];    // taps stacked along M (horizontally adjacent, LBO = one pixel row)
  // Vertical stacking on the N side (full k x k windows, stride 1): the B operand's N atoms are the gradient tile read nv times,
  // each one slot (pixel row) further down -- LBO = SBO = one slot -- so atom j pairs gathered row s with gradient row
  // s - ey + v0 + j, i.e. tap row dymax - v0 - j.  One MMA then covers ntap x nv taps (20 of the 25 for k = 5, 32 channels) for
  // the same A fetch; the old form (nv = 1, the vertical shift on the A side) remains for strided / sparse windows.
  unsigned char grp_nv[WH_MAX_GROUPS];      // N atoms (vertically stacked taps) of the group
  uint32_t grp_boff16[WH_MAX_GROUPS];       // B descriptor start shift from (gradient box - ey slots), 16-byte units
  uint32_t grp_idesc[WH_MAX_GROUPS];        // instruction descriptor (M = 64 / 128, N = nv * Cblk_g)
  unsigned short grp_col[WH_MAX_GROUPS];    // first TMEM column of the group inside its CTA slice
  short grp_tap[WH_MAX_GROUPS][8][8];       // [N atom][M block] -> tap index (into dW)
  uint32_t g_gap_bytes;                     // zeroed bytes in front of the gradient box (>= ey slots)
  float* dw;
  int dw_ld_tap, dw_ld_co, dw_ld_cx;
  uint32_t x_stage_bytes, stage_bytes, x_box_bytes, g_box_bytes, tmem_cols;
  int stages;
};

__global__ void __launch_bounds__(CONV_THREADS, 1)
conv_wgrad_halo_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_x,
                       const __grid_constant__ WHaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* done_bar = empty_bar + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g_lo = (int)blockIdx.y * p.groups_per_cta;
  const int ng = min(p.groups_per_cta, p.ngroups - g_lo);
  const int cg0 = ((int)blockIdx.z / p.ncx) * p.Cblk_g, cx0 = ((int)blockIdx.z % p.ncx) * p.Cblk_x;
  const uint32_t rbx = (uint32_t)p.Cblk_x * 2u, rbg = (uint32_t)p.Cblk_g * 2u;

  // zero every stage once: slots past the TMA boxes stay zero for the whole kernel
  for (uint32_t i = threadIdx.x; i < (uint32_t)p.stages * p.stage_bytes / 16u; i += CONV_THREADS)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_g);
    tma_prefetch_desc(&tmap_x);
    for (int s = 0; s < 8; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(done_bar, 1);
    fence_barrier_init();
  }
  fence_proxy_async();
  if (warp == 1) tmem_alloc_dyn(tmem_slot, p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      uint32_t s = 0, ph = 0;
      for (int box = blockIdx.x; box < p.num_boxes; box += gridDim.x) {
        int m = box;
        const int sx = m % p.strips_x; m /= p.strips_x;
        const int by = m % p.blocks_y; const int nb = m / p.blocks_y;
        mbar_wait(&empty_bar[s], ph ^ 1);
        uint8_t* st = smem + (size_t)s * p.stage_bytes;
        mbar_arrive_expect_tx(&full_bar[s], p.x_box_bytes + p.g_box_bytes);
        for (int pl = 0; pl < p.nplanes; ++pl)
          tma_load_4d(st + (size_t)pl * p.plane_bytes, &tmap_x, &full_bar[s], cx0, p.in_stride * (sx * 8 + p.dxmin) + p.plane_rx[pl],
                      p.in_stride * (by * p.RT + p.dymin) + p.plane_ry[pl], nb * p.NBt);
        if (p.blocks_y == 1) {
          tma_load_4d(st + p.x_stage_bytes + p.g_gap_bytes, &tmap_g, &full_bar[s], cg0, sx * 8, 0, nb * p.NBt);
        } else {
          // row blocks: RT gradient rows per image, the ey halo slots behind them keep the zeros the stage was initialised with
          // (a box of HHs rows would bring the NEXT block's rows there); rows past the image are zero-filled by TMA
          for (int i = 0; i < p.NBt; ++i)
            tma_load_4d(st + p.x_stage_bytes + p.g_gap_bytes + (size_t)i * p.HHs * 8u * rbg, &tmap_g, &full_bar[s], cg0, sx * 8,
                        by * p.RT, nb * p.NBt + i);
        }
        if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t swx = (p.Cblk_x == 64) ? SWZ_128B : (p.Cblk_x == 32 ? SWZ_64B : SWZ_32B);
      const uint32_t swg = (p.Cblk_g == 64) ? SWZ_128B : (p.Cblk_g == 32 ? SWZ_64B : SWZ_32B);
      // MN-major descriptors: LBO = next M block (= next stacked tap = one pixel row), SBO = next 8-pixel K group (= next slot)
      const uint32_t a_hi = (((uint32_t)p.HWp * rbx >> 4) & 0x3fffu) | (1u << 14) | (swx << 29);
      const uint32_t b_hi = (((8u * rbg) >> 4) & 0x3fffu) | (1u << 14) | (swg << 29);
      const uint32_t a_lbo = ((rbx >> 4) & 0x3fffu) << 16, b_lbo = (((8u * rbg) >> 4) & 0x3fffu) << 16;    // B atoms: one slot apart
      const uint32_t ak16 = (2u * (uint32_t)p.HWp * rbx) >> 4, bk16 = (16u * rbg) >> 4;   // one MMA = 16 pixels = 2 slots
      const uint32_t am16 = (16u * (uint32_t)p.HWp * rbx) >> 4, bm16 = (128u * rbg) >> 4;  // one M-tile = 16 slots
      const uint32_t ey_slots16 = ((uint32_t)p.ey * 8u * rbg) >> 4;
      uint32_t s = 0, ph = 0, first = 0;
      for (int box = blockIdx.x; box < p.num_boxes; box += gridDim.x) {
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t sx_ = smem_u32(smem + (size_t)s * p.stage_bytes);
        const uint32_t a_lo0 = ((sx_ >> 4) & 0x3fffu) | a_lbo;
        const uint32_t b_lo0 = ((((sx_ + p.x_stage_bytes + p.g_gap_bytes) >> 4) - ey_slots16) & 0x3fffu) | b_lbo;
        for (int m = 0; m < p.MT; ++m) {
          const uint32_t b_lo = b_lo0 + (uint32_t)m * bm16;
          for (int g = 0; g < ng; ++g) {
            const uint32_t a_lo = a_lo0 + (uint32_t)m * am16 + p.grp_off16[g_lo + g];
            const uint32_t bg_lo = b_lo + p.grp_boff16[g_lo + g];
            const uint32_t idesc = p.grp_idesc[g_lo + g];
            const uint32_t d = tmem_base + (uint32_t)p.grp_col[g_lo + g];
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_bf16(d, desc64(a_hi, a_lo + (uint32_t)k * ak16), desc64(b_hi, bg_lo + (uint32_t)k * bk16), idesc,
                        k == 0 ? first : 1u);
          }
          first = 1;
        }
        umma_commit(&empty_bar[s]);
        if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1; }
      }
      umma_commit(done_bar);
    }
  } else {
    const int q = warp & 3;
    mbar_wait(done_bar, 0);
    tc_fence_after();
    const bool has_work = (int)blockIdx.x < p.num_boxes;
    const int Ng = min(p.Cblk_g, p.Cg - cg0), Nx = min(p.Cblk_x, p.Cx - cx0);
    for (int g = 0; g < ng && has_work; ++g) {
      const int ntap = p.grp_ntap[g_lo + g];
      const bool m128 = ntap * p.Cblk_x > 64;
      // accumulator row of this thread: M = 128 -> lane quarter q holds rows 32q..32q+31; M = 64 -> rows 16q..16q+15
      const int row = m128 ? q * 32 + lane : q * 16 + lane;
      const bool row_ok = m128 || lane < 16;
      const int j = row / p.Cblk_x, cx = row - j * p.Cblk_x;
      const bool live = row_ok && j < ntap && cx < Nx;
      const int nv = p.grp_nv[g_lo + g];
      for (int jv = 0; jv < nv; ++jv) {
        const int t = live ? p.grp_tap[g_lo + g][jv][j] : 0;
        for (int c0 = 0; c0 < p.Cblk_g; c0 += 16) {
          uint32_t r[16];
          tmem_ld_32x16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(p.grp_col[g_lo + g] + jv * p.Cblk_g + c0), r);
          tmem_ld_wait();
          if (live) {
            float* o = p.dw + (size_t)t * p.dw_ld_tap + (size_t)(cg0 + c0) * p.dw_ld_co + (size_t)(cx0 + cx) * p.dw_ld_cx;
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (c0 + i < Ng) atomicAdd(o + (size_t)i * p.dw_ld_co, __uint_as_float(r[i]));
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc_dyn(tmem_base, p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------ host helpers
static int pow2_floor(int v) { int p = 1; while (p * 2 <= v) p *= 2; return p; }
static int pow2_ceil(int v) { int p = 1; while (p < v) p *= 2; return p; }

// tile box of the tap-box kernels for input stride s: the strided input box spans TW*s x TH*s elements, and a TMA box
// dimension is at most 256, so TW and TH are capped at pow2_floor(256 / s) (no cap below 128 for s <= 2)
static void tile_shape(int Hq, int Wq, int s, int* TW, int* TH, int* NB) {
  const int cap = min(128, pow2_floor(256 / s));
  int tw = pow2_floor(Wq); if (tw > cap) tw = cap;
  if (tw < Wq && tw * 2 <= cap && (tw * 2 - Wq) * 4 <= Wq) tw *= 2;   // e.g. W=28 -> 32 rather than 16
  int th = pow2_ceil(Hq); if (th > 128 / tw) th = 128 / tw;
  if (th > cap) th = cap;
  *TW = tw; *TH = th; *NB = 128 / (tw * th);
}

static int cblk_of(int C) { return C > 32 ? 64 : (C > 16 ? 32 : 16); }

// NHWC bf16 activation map: dims {C, W, H, N}, box {Cblk, TW*s, TH*s, NB}, element strides {1, s, s, 1}
static int act_tmap(CUtensorMap* t, const void* base, int N, int H, int W, int C, int ldc, int Cblk, int TW, int TH, int NB,
                    int stride) {
  uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
  uint64_t strides[3] = {(uint64_t)ldc * 2, (uint64_t)W * ldc * 2, (uint64_t)H * W * ldc * 2};
  uint32_t box[4] = {(uint32_t)Cblk, (uint32_t)(TW * stride), (uint32_t)(TH * stride), (uint32_t)NB};
  uint32_t es[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
  return make_tmap_bf16(t, base, 4, dims, strides, box, es, Cblk * 2);
}

// merged sub-pixel phases (jvae_conv_subpixel_gemm): the tap table lists the taps of phase 0, then phase 1, ...
struct PhaseSpec { int n; const int16_t* ntaps; const int16_t* oy; const int16_t* ox; };

// plans and launches the halo kernel; returns 1 if the geometry is not covered (caller falls back to the tap-box kernel)
static int try_launch_halo(const void* in, int N, int H, int W, int Cin, int ld_in, const void* wmat, int Cout_pad, int ldw,
                           int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, int Hq, int Wq, void* out,
                           int Ho, int Wo, int Cout, int ld_out, int out_sy, int out_sx, int out_oy, int out_ox,
                           const float* bias, int act, double* stats, cudaStream_t stream, const PhaseSpec* phs = nullptr,
                           HaloParams* plan_out = nullptr, int force_cblk = 0, double* score_out = nullptr) {
  if (Wq < 6) return 1;
  // strides 3..8 read s*s parity planes: more than the plane tables hold and the stage budget fits; the tap-box kernel runs them
  if (in_stride > 2) return 1;
  // wide layers (Cin > 64 or more than 64 output channels) run on the tap-box kernel: a halo form with 64-channel output tiles
  // and weights streamed per (tap, chunk) measured slower on B200 (DESIGN.md section 6)
  if (Cin > 64 || Cout_pad > 64) return 1;
  if (phs && (in_stride != 1 || phs->n < 2 || phs->n > 4)) return 1;
  // 33..64 input channels, narrow output: either ONE 64-channel chunk (128-byte rows; the resident weights then leave no room for
  // tap stacking: N = BN MMAs bound by the A-operand fetch) or TWO 32-channel chunks per box (64-byte rows, half-size stages, the
  // weights of both chunks resident) with tap stacking.  Both are planned, the better modelled one runs.
  if (!phs && force_cblk == 0 && Cin > 32) {
    HaloParams pa, pb;
    double sa = 0.0, sb = 0.0;
    const int ra = try_launch_halo(in, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, ntaps, tap_dy, tap_dx, in_stride, Hq, Wq, out, Ho, Wo,
                                   Cout, ld_out, out_sy, out_sx, out_oy, out_ox, bias, act, stats, stream, nullptr, &pa, 64, &sa);
    const int rb2 = try_launch_halo(in, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, ntaps, tap_dy, tap_dx, in_stride, Hq, Wq, out, Ho, Wo,
                                    Cout, ld_out, out_sy, out_sx, out_oy, out_ox, bias, act, stats, stream, nullptr, &pb, 32, &sb);
    if (ra < 0) return ra;
    const int pick = (rb2 == 0 && (ra != 0 || sb > 1.15 * sa)) ? 32 : 64;
    if (score_out) *score_out = pick == 32 ? sb : sa;
    return try_launch_halo(in, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, ntaps, tap_dy, tap_dx, in_stride, Hq, Wq, out, Ho, Wo, Cout,
                           ld_out, out_sy, out_sx, out_oy, out_ox, bias, act, stats, stream, nullptr, plan_out, pick, nullptr);
  }
  HaloParams p;
  memset(&p, 0, sizeof(p));
  p.PH = 1;
  // tap offset d = s * e + r: parity plane r, offset e inside the plane (floor division for negative d)
  const int st = in_stride;
  int tey[CONV_MAX_TAPS], tex[CONV_MAX_TAPS], tpl[CONV_MAX_TAPS];
  int dymin = 1 << 20, dymax = -(1 << 20), dxmin = 1 << 20, dxmax = -(1 << 20);
  p.in_stride = st; p.nplanes = 0;
  for (int t = 0; t < ntaps; ++t) {
    p.dy[t] = tap_dy[t]; p.dx[t] = tap_dx[t];
    const int ry = ((tap_dy[t] % st) + st) % st, rx = ((tap_dx[t] % st) + st) % st;
    tey[t] = (tap_dy[t] - ry) / st; tex[t] = (tap_dx[t] - rx) / st;
    int pl = -1;
    for (int i = 0; i < p.nplanes; ++i)
      if (p.plane_ry[i] == ry && p.plane_rx[i] == rx) pl = i;
    if (pl < 0) { pl = p.nplanes++; p.plane_ry[pl] = (short)ry; p.plane_rx[pl] = (short)rx; }
    tpl[t] = pl;
    dymin = min(dymin, tey[t]); dymax = max(dymax, tey[t]);
    dxmin = min(dxmin, tex[t]); dxmax = max(dxmax, tex[t]);
  }
  const int ey = dymax - dymin, ex = dxmax - dxmin;
  if (ey > 16 || ex > 16) return 1;
  p.N = N; p.Hq = Hq; p.Wq = Wq; p.dymin = dymin; p.dxmin = dxmin;
  p.Cblk = force_cblk ? force_cblk : cblk_of(Cin); p.ntaps = ntaps;
  p.nkc = (Cin + p.Cblk - 1) / p.Cblk;
  p.BN = Cout_pad; p.n_tiles_n = 1;
  const uint32_t rb = (uint32_t)p.Cblk * 2u;
  p.HWp = 8 + ex;
  p.RT = Hq <= 32 ? Hq : 32;
  p.HHs = p.RT + ey;
  p.w_tap_bytes = (uint32_t)p.BN * rb;
  const uint32_t budget = 200u * 1024u;
  const uint32_t stats_bytes = stats ? 2u * (uint32_t)Cout_pad * 8u : 0u;
  const uint32_t w_res = (uint32_t)ntaps * p.w_tap_bytes * (uint32_t)p.nkc;      // every chunk's weights resident
  const bool ksplit = p.nkc > 1;
  const int ksteps = p.Cblk >> 4;
  // modelled cycles of one 128 x n x 16 MMA with both operands in shared memory (measured: profiles/r01_umma_rate_probe.txt):
  // the tensor pipe needs n / 2, the operand fetch (4 KB of A + 32 n bytes of B at 128 B / cycle) 32 + n / 4
  auto mma_cycles = [](int n) { const double t = n / 2.0, f = 32.0 + n / 4.0; return t > f ? t : f; };

  // ---- tap rectangles per parity plane (vertical stacking needs, for every tap column, a contiguous run of tap rows)
  struct Col { int pl, x, e_lo, e_hi; };
  std::vector<Col> cols;
  bool stackable = true;
  for (int t = 0; t < ntaps && stackable; ++t) {
    const int x = tex[t] - dxmin, e = tey[t] - dymin;
    Col* c = nullptr;
    for (auto& q : cols) if (q.pl == tpl[t] && q.x == x) c = &q;
    if (!c) { cols.push_back({tpl[t], x, e, e}); continue; }
    c->e_lo = min(c->e_lo, e); c->e_hi = max(c->e_hi, e);
  }
  if (stackable) {
    int covered = 0;
    for (auto& q : cols) covered += q.e_hi - q.e_lo + 1;
    stackable = covered == ntaps;                          // no holes, no duplicates
  }

  // ---- merged phases: one chunk per (input shift, run of consecutive phase blocks that have a tap there)
  struct Run { int shift, pos0, len, fresh; };
  std::vector<Run> runs;
  std::vector<int> shift_y, shift_x;
  int tap_shift[CONV_MAX_TAPS], tap_phase[CONV_MAX_TAPS], ph_pos[4] = {0, 1, 2, 3};
  if (phs) {
    int t = 0;
    for (int ph = 0; ph < phs->n; ++ph)
      for (int i = 0; i < phs->ntaps[ph]; ++i, ++t) {
        if (t >= ntaps) return 1;
        tap_phase[t] = ph;
        int sidx = -1;
        for (size_t q = 0; q < shift_y.size(); ++q)
          if (shift_y[q] == tey[t] && shift_x[q] == tex[t]) sidx = (int)q;
        if (sidx < 0) { sidx = (int)shift_y.size(); shift_y.push_back(tey[t]); shift_x.push_back(tex[t]); }
        for (int u = 0; u < t; ++u)
          if (tap_shift[u] == sidx && tap_phase[u] == ph) return 1;      // two taps of a phase at one shift
        tap_shift[t] = sidx;
      }
    if (t != ntaps) return 1;
    // order of the phase blocks with the fewest runs (k = 5, stride 2: (0,1) (0,0) (1,0) (1,1) makes every shift ONE run)
    auto runs_of = [&](const int* pos, std::vector<Run>* out) {
      int count = 0;
      for (size_t q = 0; q < shift_y.size(); ++q) {
        bool used[4] = {false, false, false, false};
        for (int u = 0; u < ntaps; ++u)
          if (tap_shift[u] == (int)q) used[pos[tap_phase[u]]] = true;
        for (int b = 0; b < phs->n;) {
          if (!used[b]) { ++b; continue; }
          int e = b;
          while (e + 1 < phs->n && used[e + 1]) ++e;
          if (out) out->push_back({(int)q, b, e - b + 1, 0});
          ++count;
          b = e + 1;
        }
      }
      return count;
    };
    int perm[4] = {0, 1, 2, 3}, best_runs = 1 << 20;
    do {
      if (phs->n < 4 && (perm[3] != 3 || (phs->n < 3 && perm[2] != 2))) continue;      // only the first n entries move
      const int c = runs_of(perm, nullptr);
      if (c < best_runs) { best_runs = c; for (int i = 0; i < 4; ++i) ph_pos[i] = perm[i]; }
    } while (std::next_permutation(perm, perm + 4));
    runs_of(ph_pos, &runs);
    // the fresh (overwriting) chunks: a disjoint cover of the phase blocks, longest runs first
    std::stable_sort(runs.begin(), runs.end(), [](const Run& a, const Run& b) { return a.len > b.len; });
    unsigned covered = 0;
    for (auto& r : runs) {
      const unsigned bits = ((1u << r.len) - 1u) << r.pos0;
      if ((covered & bits) == 0) { r.fresh = 1; covered |= bits; }
    }
    if (covered != (1u << phs->n) - 1u) return 1;
    std::stable_sort(runs.begin(), runs.end(), [](const Run& a, const Run& b) { return a.fresh > b.fresh; });
    if ((int)runs.size() > HALO_MAX_CK) return 1;
    p.PH = phs->n;
    for (int ph = 0; ph < phs->n; ++ph) { p.ph_oy[ph_pos[ph]] = phs->oy[ph]; p.ph_ox[ph_pos[ph]] = phs->ox[ph]; }
  }

  // ---- choose (G, resident, images per box): most useful output rows per modelled MMA cycle
  double best = 0.0;
  int bestG = 1;
  uint32_t best_extent = 0;
  if (phs) {
    // G = 1, resident weights; the channel tile is halved until all the taps' weights fit beside two stages
    for (int bn_try = p.BN; bn_try >= 16 && (bn_try % 16) == 0 && (Cout_pad % bn_try) == 0; bn_try /= 2) {
      const uint32_t wtap = (uint32_t)bn_try * rb, wb = (uint32_t)ntaps * wtap;
      for (int nbt = 1; nbt <= 16 && nbt <= N; ++nbt) {
        const int S = nbt * p.HHs;
        const int groups = S - ey, MT = (groups + 15) / 16;
        if (nbt > 1 && p.RT < Hq) break;
        if (pow2_ceil(2 * MT * p.PH * bn_try) > 512) break;
        const uint32_t plane = ((uint32_t)(16 * MT + ey) * p.HWp * rb + 1023u) & ~1023u;
        if (2u * plane + wb + stats_bytes + 1792u + (uint32_t)(MT * p.PH) * 128u > budget) break;
        double cyc = 0.0;
        for (auto& r : runs) cyc += (double)MT * ksteps * mma_cycles(r.len * bn_try);
        cyc *= (double)(Cout_pad / bn_try);
        const double score = (double)(nbt * p.RT) / cyc;
        if (score > best * 1.02) {
          best = score; p.NBt = nbt; p.MT = MT; p.stage_bytes = plane; p.plane_bytes = plane; p.resident = 1; p.w_bytes = wb;
          p.BN = bn_try; p.n_tiles_n = Cout_pad / bn_try; p.w_tap_bytes = wtap;
        }
      }
    }
  }
  for (int G = 1; G <= 8 && !phs; ++G) {
    if (G > 1 && (!stackable || G * p.BN > 256)) break;
    for (int resident = 1; resident >= 0; --resident) {
      if (G > 1 && !resident) continue;
      if (ksplit && (G == 1 || !resident)) continue;       // two resident chunks: only the stacked form is built
      const uint32_t wb = resident ? w_res : 4u * p.w_tap_bytes;
      bool found = false;
      for (int nbt = 1; nbt <= 16 && nbt <= N; ++nbt) {
        const int S = nbt * p.HHs;
        const int groups = (S - ey + G - 1) / G, MT = (groups + 15) / 16;
        if (nbt > 1 && p.RT < Hq) break;                   // several row blocks per image: one image per box
        if (pow2_ceil(2 * MT * G * p.BN) > 512) break;
        // a plane holds the box; the MMAs of the last (partly filled) M-tile read up to slot 16 MT G + ey - 1: past the box they
        // fetch whatever follows in shared memory (the next plane / stage / the weights) into rows that are discarded, so only
        // the END of the last stage's last plane has to stay inside the allocation
        const uint32_t plane = G == 1 ? (((uint32_t)(16 * MT + ey) * p.HWp * rb + 1023u) & ~1023u)
                                      : (((uint32_t)S * p.HWp * rb + 1023u) & ~1023u);
        const uint32_t extent = (uint32_t)(16 * MT * G + ey) * p.HWp * rb;      // bytes an M-tile sweep can touch in a plane
        const uint32_t stage = plane * (uint32_t)p.nplanes;
        const uint32_t ystage = 0u;
        const uint32_t over = extent > plane ? extent - plane : 0u;             // overshoot of the very last plane
        const uint32_t tail = over > wb + 3u * ystage ? over - wb - 3u * ystage : 0u;
        if (2u * stage + wb + stats_bytes + 1792u + 3u * ystage + tail + (uint32_t)(MT * G) * 128u > budget + (G > 1 ? 20u * 1024u : 0u)) break;
        double cyc = 0.0;
        if (G == 1) cyc = (double)MT * ntaps * ksteps * mma_cycles(p.BN) * (resident ? 1.0 : 1.03);
        else
          for (auto& q : cols)
            for (int u = q.e_lo; u <= q.e_hi + G - 1; ++u) {
              const int j0 = max(0, u - q.e_hi), j1 = min(G - 1, u - q.e_lo);
              cyc += (double)MT * ksteps * mma_cycles((j1 - j0 + 1) * p.BN);
            }
        cyc *= (double)p.nkc;
        const double score = (double)(nbt * p.RT) / cyc;
        if (score > best * 1.02) {
          best = score; bestG = G; p.NBt = nbt; p.MT = MT; p.stage_bytes = stage; p.plane_bytes = plane; p.resident = resident;
          p.w_bytes = wb + tail; best_extent = extent;
        }
        found = true;
      }
      if (found && resident) break;                        // resident weights fit: take them
    }
  }
  if (best <= 0.0) return 1;
  if (score_out) *score_out = best;
  p.G = bestG;
  (void)best_extent;
  p.wstages = p.resident ? 1 : 4;
  if ((size_t)p.stage_bytes + (size_t)(p.G * p.HWp) * rb * 16 >= (1u << 18)) return 1;      // descriptor start field is 14 bits of 16 B
  if (((uint32_t)(p.G * p.HWp) * rb >> 4) > 0x3fffu) return 1;                              // SBO field
  for (int t = 0; t < ntaps; ++t)
    p.tap_off16[t] = ((uint32_t)tpl[t] * p.plane_bytes + (uint32_t)((tey[t] - dymin) * p.HWp + (tex[t] - dxmin)) * rb) >> 4;
  if (phs) {
    // weight blocks in shared memory: run after run, inside a run in block order (= the N rows of the run's MMA)
    int pos = 0, nck = 0;
    for (auto& r : runs) {
      for (int b = 0; b < r.len; ++b)
        for (int t = 0; t < ntaps; ++t)
          if (tap_shift[t] == r.shift && ph_pos[tap_phase[t]] == r.pos0 + b) p.w_pos[t] = (short)(pos + b);
      p.ck[nck].x = ((uint32_t)((shift_y[r.shift] - dymin) * p.HWp + (shift_x[r.shift] - dxmin)) * rb) >> 4;
      p.ck[nck].y = ((uint32_t)pos * p.w_tap_bytes) >> 4;
      p.ck[nck].z = make_idesc_bf16(128, r.len * p.BN, false, false);
      p.ck[nck].w = (uint32_t)(r.pos0 * p.BN) | (r.fresh ? 0x80000000u : 0u);
      ++nck;
      pos += r.len;
    }
    if (pos != ntaps) return 1;
    p.nck = nck;
    if ((((uint32_t)pos * p.w_tap_bytes) >> 4) > 0xffffu) return 1;
  } else if (p.G > 1) {
    // weight blocks in shared memory: per tap column, rows of taps DESCENDING (the column block j of a chunk reads tap e = u - j)
    int pos = 0, nck = 0;
    std::vector<int> col_base(cols.size());
    for (size_t ci = 0; ci < cols.size(); ++ci) {
      col_base[ci] = pos;
      for (int t = 0; t < ntaps; ++t)
        if (tpl[t] == cols[ci].pl && tex[t] - dxmin == cols[ci].x) p.w_pos[t] = (short)(pos + cols[ci].e_hi - (tey[t] - dymin));
      pos += cols[ci].e_hi - cols[ci].e_lo + 1;
    }
    auto add_chunk = [&](size_t ci, int u, int fresh) {
      const Col& q = cols[ci];
      const int j0 = max(0, u - q.e_hi), j1 = min(p.G - 1, u - q.e_lo);
      p.ck[nck].x = ((uint32_t)q.pl * p.plane_bytes + (uint32_t)(u * p.HWp + q.x) * rb) >> 4;
      p.ck[nck].y = ((uint32_t)(col_base[ci] + q.e_hi - (u - j0)) * p.w_tap_bytes) >> 4;
      p.ck[nck].z = make_idesc_bf16(128, (j1 - j0 + 1) * p.BN, false, false);
      p.ck[nck].w = (uint32_t)(j0 * p.BN) | (fresh ? 0x80000000u : 0u);
      ++nck;
    };
    // fresh chunks: a disjoint cover of the G column blocks out of the first tap column
    std::vector<int> fresh_u;
    for (int jn = 0; jn < p.G;) {
      const int u = jn + cols[0].e_hi;
      fresh_u.push_back(u);
      jn = min(p.G - 1, u - cols[0].e_lo) + 1;
    }
    for (int u : fresh_u) add_chunk(0, u, 1);
    for (size_t ci = 0; ci < cols.size(); ++ci)
      for (int u = cols[ci].e_lo; u <= cols[ci].e_hi + p.G - 1; ++u) {
        if (ci == 0 && std::find(fresh_u.begin(), fresh_u.end(), u) != fresh_u.end()) continue;
        if (nck >= HALO_MAX_CK) return 1;
        add_chunk(ci, u, 0);
      }
    p.nck = nck;
    if ((((uint32_t)pos * p.w_tap_bytes) >> 4) > 0xffffu) return 1;
  }
  p.box_bytes = (uint32_t)p.nplanes * (uint32_t)(p.NBt * p.HHs) * p.HWp * rb;
  {
    const uint32_t bud = budget + (p.G > 1 ? 20u * 1024u : 0u);
    p.stages = (int)((bud - p.w_bytes - stats_bytes - 1792u - (uint32_t)(p.MT * p.G * p.PH) * 128u) / p.stage_bytes);
  }
  if (p.stages > 4) p.stages = 4;
  if (p.stages < 2) return 1;
  p.acc_stride = (uint32_t)(p.MT * p.G * p.PH * p.BN);
  p.tmem_cols = (uint32_t)pow2_ceil(2 * p.acc_stride < 32 ? 32 : 2 * p.acc_stride);
  p.strips_x = (Wq + 7) / 8; p.blocks_y = (Hq + p.RT - 1) / p.RT; p.blocks_n = (N + p.NBt - 1) / p.NBt;
  p.num_boxes = p.strips_x * p.blocks_y * p.blocks_n;
  p.Ho = Ho; p.Wo = Wo; p.Cout = Cout; p.ldc = ld_out;
  p.out_sy = out_sy; p.out_sx = out_sx; p.out_oy = out_oy; p.out_ox = out_ox;
  p.act = act & 0xff;
  p.bias = bias; p.out = reinterpret_cast<__nv_bfloat16*>(out); p.stats = stats; p.cout_pad = Cout_pad;
  if (plan_out) { *plan_out = p; return JVAE_OK; }      // jvae_conv_halo_emulate: the plan only, nothing touches the device
  CUtensorMap tin, tw;
  {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t strides[3] = {(uint64_t)ld_in * 2, (uint64_t)W * ld_in * 2, (uint64_t)H * W * ld_in * 2};
    uint32_t box[4] = {(uint32_t)p.Cblk, (uint32_t)(p.HWp * st), (uint32_t)(p.HHs * st), (uint32_t)p.NBt};
    uint32_t es[4] = {1u, (uint32_t)st, (uint32_t)st, 1u};
    if (box[1] > 256 || box[2] > 256) return 1;
    int rc = make_tmap_bf16(&tin, in, 4, dims, strides, box, es, p.Cblk * 2);
    if (rc) return rc;
    const int Ktot = ntaps * p.nkc * p.Cblk;
    uint64_t wd[2] = {(uint64_t)Ktot, (uint64_t)Cout_pad};
    uint64_t ws[1] = {(uint64_t)ldw * 2};
    uint32_t wbox[2] = {(uint32_t)p.Cblk, (uint32_t)p.BN};
    if (ldw < Ktot) { set_error("jvae_conv_gather_gemm: weight matrix row shorter than taps*Cblk"); return JVAE_ERR_INVALID; }
    rc = make_tmap_bf16(&tw, wmat, 2, wd, ws, wbox, nullptr, p.Cblk * 2);
    if (rc) return rc;
  }
  const size_t tab_bytes = (size_t)p.MT * p.G * p.PH * 16 * sizeof(int2);       // block table of the fast epilogue
  const size_t smem = (size_t)p.stages * p.stage_bytes + p.w_bytes + 512 + stats_bytes + 256 + 1024 + tab_bytes;
  if (smem > 227u * 1024u) return 1;
  static bool attr = false;
  if (!attr) {
    JVAE_CUDA(cudaFuncSetAttribute(conv_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr = true;
  }
  int grid = p.num_boxes * p.n_tiles_n < sm_count() ? p.num_boxes * p.n_tiles_n : (sm_count() / p.n_tiles_n) * p.n_tiles_n;
  if (grid < p.n_tiles_n) return 1;
  void* prof = prof_begin(JVAE_PROF_CONV_HALO, stream);
  conv_halo_kernel<<<grid, HALO_THREADS, smem, stream>>>(tin, tw, p);
  prof_end(prof, stream);
  JVAE_LAUNCH_CHECK();
  g_last_conv_kernel = JVAE_KERNEL_CONV_HALO;
  return JVAE_OK;
}

// plans and launches the halo weight-gradient kernel; returns 1 when the geometry is not covered
static int try_launch_wgrad_halo(const void* g, int N, int Hq, int Wq, int Cg, int ld_g, const void* x, int H, int W, int Cx,
                                 int ld_x, int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, float* dw,
                                 int dw_ld_tap, int dw_ld_co, int dw_ld_cx, cudaStream_t stream, const int* tap_ids = nullptr,
                                 bool dry_run = false, WHaloParams* plan_out = nullptr) {
  // tap_ids: position of tap t in dW when the list is a subset of the layer's taps (per-plane launches, jvae_conv_wgrad);
  // dry_run: plan only (is the geometry covered?)
  if (Wq < 6) return 1;
  if (in_stride > 2) return 1;          // s*s parity planes for s >= 3: the tap-box kernel runs them
  WHaloParams p;
  memset(&p, 0, sizeof(p));
  const int st = in_stride;
  std::vector<int> tey(ntaps), tex(ntaps), tpl(ntaps);
  int dymin = 1 << 20, dymax = -(1 << 20), dxmin = 1 << 20, dxmax = -(1 << 20);
  p.in_stride = st; p.nplanes = 0;
  for (int t = 0; t < ntaps; ++t) {
    const int ry = ((tap_dy[t] % st) + st) % st, rx = ((tap_dx[t] % st) + st) % st;
    tey[t] = (tap_dy[t] - ry) / st; tex[t] = (tap_dx[t] - rx) / st;
    int pl = -1;
    for (int i = 0; i < p.nplanes; ++i)
      if (p.plane_ry[i] == ry && p.plane_rx[i] == rx) pl = i;
    if (pl < 0) { pl = p.nplanes++; p.plane_ry[pl] = (short)ry; p.plane_rx[pl] = (short)rx; }
    tpl[t] = pl;
    dymin = min(dymin, tey[t]); dymax = max(dymax, tey[t]);
    dxmin = min(dxmin, tex[t]); dxmax = max(dxmax, tex[t]);
  }
  const int ey = dymax - dymin, ex = dxmax - dxmin;
  if (ey > 16 || ex > 16) return 1;
  p.N = N; p.Hq = Hq; p.Wq = Wq; p.dymin = dymin; p.dxmin = dxmin;
  p.Cg = Cg; p.Cx = Cx;
  p.Cblk_g = cblk_of(Cg > 64 ? 64 : Cg); p.Cblk_x = cblk_of(Cx > 64 ? 64 : Cx);
  const int ncg = (Cg + p.Cblk_g - 1) / p.Cblk_g;
  p.ncx = (Cx + p.Cblk_x - 1) / p.Cblk_x;
  const uint32_t rbx = (uint32_t)p.Cblk_x * 2u, rbg = (uint32_t)p.Cblk_g * 2u;
  p.RT = Hq <= 32 ? Hq : 32; p.blocks_y = (Hq + p.RT - 1) / p.RT;      // taller maps: row blocks of 32
  p.HWp = 8 + ex; p.HHs = p.RT + ey;
  // tap groups.  Full k x k windows at stride 1: runs of horizontally adjacent taps (at most 128 / Cblk_x) along M, sets of
  // vertically adjacent taps (at most 256 / Cblk_g) along N.  Otherwise (parity planes, sparse windows): horizontal runs only,
  // the vertical shift on the A side.
  const int tpm = 128 / p.Cblk_x;
  p.ey = ey;
  std::vector<int> tap_at((size_t)(ey + 1) * (ex + 1), -1);
  // Measured on B200 (tools/bench_layers.py, old form / stacked form): 32 -> 32 k5 at 32 x 32: 850 / 600 us; 256-channel k3 layers at
  // 8 x 8: 142 / 117 us; but 64-channel tiles on 16 x 16 and 32 x 32 maps and the 64 -> 64 k5 layer at 8 x 8 lose (a stacked B
  // fetch costs ~1.5x per MMA, so the form pays only when it removes most of the MMAs): enabled for 32-channel gradient tiles
  // with at least four tap rows, and for 3 x 3 windows on maps of at most 8 x 8 with >= 128 channels.
  const bool want = (cblk_of(Cg > 64 ? 64 : Cg) == 32 && ey + 1 >= 4) || (ey + 1 == 3 && Hq * Wq <= 64 && Cg >= 128);
  bool full = want && st == 1 && p.nplanes == 1 && ntaps == (ey + 1) * (ex + 1);
  for (int t = 0; t < ntaps && full; ++t) {
    int& slot = tap_at[(size_t)(tey[t] - dymin) * (ex + 1) + (tex[t] - dxmin)];
    if (slot >= 0) full = false;
    slot = t;
  }
  int ngr = 0;
  std::vector<int> grp_first;
  const uint32_t gslot16 = (8u * rbg) >> 4;               // one slot of the gradient tile (8 pixels), 16-byte units
  const int E = ey;
  if (full) {
    const int nvmax = min(ey + 1, 256 / p.Cblk_g);
    const int nsets = (ey + 1 + nvmax - 1) / nvmax;
    for (int x0 = 0; x0 <= ex; x0 += min(tpm, 8)) {
      const int n = min(min(tpm, 8), ex + 1 - x0);
      for (int vs = 0, v0 = 0; vs < nsets; ++vs) {
        const int nv = (ey + 1 - v0 + (nsets - vs) - 1) / (nsets - vs);      // balanced sets
        if (ngr >= WH_MAX_GROUPS) return 1;
        p.grp_ntap[ngr] = (unsigned char)n;
        p.grp_nv[ngr] = (unsigned char)nv;
        p.grp_off16[ngr] = ((uint32_t)x0 * rbx) >> 4;
        p.grp_boff16[ngr] = (uint32_t)v0 * gslot16;
        for (int jv = 0; jv < nv; ++jv)
          for (int j = 0; j < n; ++j) {
            const int t = tap_at[(size_t)(ey - v0 - jv) * (ex + 1) + (x0 + j)];
            p.grp_tap[ngr][jv][j] = (short)(tap_ids ? tap_ids[t] : t);
          }
        ++ngr;
        v0 += nv;
      }
    }
  } else {
    std::vector<int> order(ntaps);
    for (int t = 0; t < ntaps; ++t) order[t] = t;
    // groups = runs of taps adjacent in x INSIDE one parity plane and one plane row
    std::sort(order.begin(), order.end(), [&](int a, int b) {
      if (tpl[a] != tpl[b]) return tpl[a] < tpl[b];
      return tey[a] != tey[b] ? tey[a] < tey[b] : tex[a] < tex[b];
    });
    for (int i = 0; i < ntaps;) {
      if (ngr >= WH_MAX_GROUPS) return 1;
      int n = 1;
      while (i + n < ntaps && n < tpm && n < 8 && tpl[order[i + n]] == tpl[order[i]] && tey[order[i + n]] == tey[order[i]] &&
             tex[order[i + n]] == tex[order[i]] + n)
        ++n;
      p.grp_ntap[ngr] = (unsigned char)n;
      p.grp_nv[ngr] = 1;
      p.grp_boff16[ngr] = (uint32_t)E * gslot16;           // the gradient tile itself
      grp_first.push_back(order[i]);
      for (int j = 0; j < n; ++j) p.grp_tap[ngr][0][j] = (short)(tap_ids ? tap_ids[order[i + j]] : order[i + j]);
      ++ngr;
      i += n;
    }
  }
  p.ngroups = ngr;
  int wmax = 0;
  for (int gi = 0; gi < ngr; ++gi) {
    const int M = ((int)p.grp_ntap[gi] * p.Cblk_x > 64) ? 128 : 64;
    p.grp_idesc[gi] = make_idesc_bf16(M, (int)p.grp_nv[gi] * p.Cblk_g, true, true);
    wmax = max(wmax, (int)p.grp_nv[gi] * p.Cblk_g);
  }
  p.groups_per_cta = 512 / wmax;
  if (p.groups_per_cta > ngr) p.groups_per_cta = ngr;
  const int ysplit = (ngr + p.groups_per_cta - 1) / p.groups_per_cta;
  p.groups_per_cta = (ngr + ysplit - 1) / ysplit;               // balance the slices
  int cols_max = 0;
  for (int gi = 0; gi < ngr; gi += p.groups_per_cta) {
    int col = 0;
    for (int k = gi; k < min(ngr, gi + p.groups_per_cta); ++k) { p.grp_col[k] = (unsigned short)col; col += (int)p.grp_nv[k] * p.Cblk_g; }
    cols_max = max(cols_max, col);
  }
  p.tmem_cols = (uint32_t)pow2_ceil(cols_max < 32 ? 32 : cols_max);
  p.g_gap_bytes = ((uint32_t)E * 8u * rbg + 1023u) & ~1023u;
  p.ey = E;                                             // the kernel's B base sits E slots in front of the gradient box
  // images per box: best slot efficiency within the shared-memory budget
  const uint32_t budget = 200u * 1024u;
  double best = 0.0;
  for (int nbt = 1; nbt <= 16 && nbt <= N; ++nbt) {
    const int S = nbt * p.HHs, MT = full ? (S + 15) / 16 : (S - ey + 15) / 16;
    const uint32_t plane = ((uint32_t)(16 * MT + ey + 1) * p.HWp * rbx + 1023u) & ~1023u;   // +1 slot: stacked-tap overrun
    const uint32_t xs = plane * (uint32_t)p.nplanes;
    const uint32_t gs = p.g_gap_bytes + (((uint32_t)(16 * MT > S ? 16 * MT : S) * 8u * rbg + 1023u) & ~1023u);
    if (2u * (xs + gs) + 1024u > budget) break;
    if (nbt * p.HHs > 256) break;
    const double eff = (double)(nbt * p.RT) / (16.0 * MT);
    if (eff > best + 0.02) {
      best = eff; p.NBt = nbt; p.MT = MT; p.x_stage_bytes = xs; p.stage_bytes = xs + gs; p.plane_bytes = plane;
    }
  }
  if (best <= 0.0) return 1;
  if ((size_t)p.stage_bytes >= (1u << 18)) return 1;
  for (int gi = 0; gi < ngr && !full; ++gi) {
    const int t0 = grp_first[gi];
    p.grp_off16[gi] = ((uint32_t)tpl[t0] * p.plane_bytes + (uint32_t)((tey[t0] - dymin) * p.HWp + (tex[t0] - dxmin)) * rbx) >> 4;
  }
  p.x_box_bytes = (uint32_t)p.nplanes * (uint32_t)(p.NBt * p.HHs) * p.HWp * rbx;
  p.g_box_bytes = (uint32_t)(p.NBt * (p.blocks_y == 1 ? p.HHs : p.RT)) * 8u * rbg;
  p.stages = (int)((budget - 1024u) / p.stage_bytes);
  if (p.stages > 6) p.stages = 6;
  if (p.stages < 2) return 1;
  p.strips_x = (Wq + 7) / 8;
  p.num_boxes = p.strips_x * p.blocks_y * ((N + p.NBt - 1) / p.NBt);
  p.dw = dw; p.dw_ld_tap = dw_ld_tap; p.dw_ld_co = dw_ld_co; p.dw_ld_cx = dw_ld_cx;
  if (plan_out) *plan_out = p;
  if (dry_run) return JVAE_OK;
  CUtensorMap tg, tx;
  {
    uint64_t dg[4] = {(uint64_t)Cg, (uint64_t)Wq, (uint64_t)Hq, (uint64_t)N};
    uint64_t sg[3] = {(uint64_t)ld_g * 2, (uint64_t)Wq * ld_g * 2, (uint64_t)Hq * Wq * ld_g * 2};
    uint32_t bg[4] = {(uint32_t)p.Cblk_g, 8u, (uint32_t)(p.blocks_y == 1 ? p.HHs : p.RT), (uint32_t)(p.blocks_y == 1 ? p.NBt : 1)};
    int rc = make_tmap_bf16(&tg, g, 4, dg, sg, bg, nullptr, p.Cblk_g * 2);
    if (rc) return rc;
    uint64_t dx[4] = {(uint64_t)Cx, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t sx[3] = {(uint64_t)ld_x * 2, (uint64_t)W * ld_x * 2, (uint64_t)H * W * ld_x * 2};
    uint32_t bx[4] = {(uint32_t)p.Cblk_x, (uint32_t)(p.HWp * st), (uint32_t)(p.HHs * st), (uint32_t)p.NBt};
    uint32_t esx[4] = {1u, (uint32_t)st, (uint32_t)st, 1u};
    if (bx[1] > 256 || bx[2] > 256) return 1;
    rc = make_tmap_bf16(&tx, x, 4, dx, sx, bx, esx, p.Cblk_x * 2);
    if (rc) return rc;
  }
  const int nz = ncg * p.ncx;
  if (nz > 65535) return 1;
  int gx = (sm_count() + ysplit * nz - 1) / (ysplit * nz);
  if (gx < 1) gx = 1;
  if (gx > p.num_boxes) gx = p.num_boxes;
  const size_t smem = (size_t)p.stages * p.stage_bytes + 256 + 1024;
  static bool attr = false;
  if (!attr) {
    JVAE_CUDA(cudaFuncSetAttribute(conv_wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr = true;
  }
  void* prof = prof_begin(JVAE_PROF_WGRAD_HALO, stream);
  conv_wgrad_halo_kernel<<<dim3(gx, ysplit, nz), CONV_THREADS, smem, stream>>>(tg, tx, p);
  prof_end(prof, stream);
  JVAE_LAUNCH_CHECK();
  g_last_conv_kernel = JVAE_KERNEL_WGRAD_HALO;
  return JVAE_OK;
}


// Host-only execution of the halo weight-gradient PLAN (try_launch_wgrad_halo), the counterpart of jvae_conv_halo_emulate: the
// two stages (parity planes of the gathered tensor, the gradient tile behind its zeroed gap), the tap groups as MN-major
// operands -- M = (stacked horizontal tap j, X channel) through LBO = one pixel row, N = (vertically stacked atom jv, G channel)
// through LBO = one slot, K = 16 pixels = 2 slots per MMA -- and the scatter of D into dW through the group's tap table.
static void wgrad_plan_emulate(const WHaloParams& p, const float* g, int ld_g, const float* x, int H, int W, int ld_x, float* dw) {
  const int ncg = (p.Cg + p.Cblk_g - 1) / p.Cblk_g;
  const size_t plane_rows = p.plane_bytes / ((size_t)p.Cblk_x * 2u);
  const size_t x_rows = plane_rows * p.nplanes;
  const int gap_slots = (int)(p.g_gap_bytes / (8u * (uint32_t)p.Cblk_g * 2u));
  const size_t g_slots = (size_t)gap_slots + (size_t)((p.stage_bytes - p.x_stage_bytes - p.g_gap_bytes) / (8u * (uint32_t)p.Cblk_g * 2u));
  std::vector<float> sx(x_rows * p.Cblk_x), sg(g_slots * 8 * p.Cblk_g);
  const float qnan = nanf("");
  for (int zg = 0; zg < ncg; ++zg)
    for (int zx = 0; zx < p.ncx; ++zx) {
      const int cg0 = zg * p.Cblk_g, cx0 = zx * p.Cblk_x;
      std::vector<double> D((size_t)p.ngroups * 128 * 8 * p.Cblk_g, 0.0);      // [group][M row][N column]
      for (int box = 0; box < p.num_boxes; ++box) {
        int m0 = box;
        const int bx = m0 % p.strips_x; m0 /= p.strips_x;
        const int by = m0 % p.blocks_y; const int nb = m0 / p.blocks_y;
        std::fill(sx.begin(), sx.end(), 0.f);      // the stage was zeroed once; the boxes always land on the same bytes
        std::fill(sg.begin(), sg.end(), 0.f);
        for (int pl = 0; pl < p.nplanes; ++pl)
          for (int i = 0; i < p.NBt; ++i)
            for (int yy = 0; yy < p.HHs; ++yy)
              for (int xx = 0; xx < p.HWp; ++xx) {
                const size_t row = (size_t)pl * plane_rows + (size_t)(i * p.HHs + yy) * p.HWp + xx;
                const int n = nb * p.NBt + i;
                const int iy = p.in_stride * (by * p.RT + p.dymin + yy) + p.plane_ry[pl], ix = p.in_stride * (bx * 8 + p.dxmin + xx) + p.plane_rx[pl];
                for (int c = 0; c < p.Cblk_x; ++c) {
                  const bool in = n < p.N && iy >= 0 && iy < H && ix >= 0 && ix < W && cx0 + c < p.Cx;
                  if (row < x_rows) sx[row * p.Cblk_x + c] = in ? x[(((size_t)n * H + iy) * W + ix) * ld_x + cx0 + c] : 0.f;
                }
              }
        for (int i = 0; i < p.NBt; ++i)
          for (int yy = 0; yy < (p.blocks_y == 1 ? p.HHs : p.RT); ++yy)
            for (int px = 0; px < 8; ++px) {
              const size_t slot = (size_t)gap_slots + (size_t)i * p.HHs + yy;
              const int n = nb * p.NBt + i, gy = by * p.RT + yy, gx = bx * 8 + px;
              for (int c = 0; c < p.Cblk_g; ++c) {
                const bool in = n < p.N && gy < p.Hq && gx < p.Wq && cg0 + c < p.Cg;
                if (slot < g_slots) sg[(slot * 8 + px) * p.Cblk_g + c] = in ? g[(((size_t)n * p.Hq + gy) * p.Wq + gx) * ld_g + cg0 + c] : 0.f;
              }
            }
        auto xa = [&](long long row, int c) { return row >= 0 && (size_t)row < x_rows ? sx[(size_t)row * p.Cblk_x + c] : qnan; };
        auto ga = [&](long long slot, int px, int c) { return slot >= 0 && (size_t)slot < g_slots ? sg[((size_t)slot * 8 + px) * p.Cblk_g + c] : qnan; };
        for (int m = 0; m < p.MT; ++m)
          for (int gi = 0; gi < p.ngroups; ++gi) {
            const long long a_rows = (long long)p.grp_off16[gi] * 16 / (p.Cblk_x * 2);
            const long long b_slots = (long long)gap_slots - p.ey + (long long)p.grp_boff16[gi] * 16 / (8 * p.Cblk_g * 2);
            const int ntap = p.grp_ntap[gi], nv = p.grp_nv[gi];
            for (int k = 0; k < 8; ++k)
              for (int kk = 0; kk < 16; ++kk) {
                const long long s = 16 * m + 2 * k + (kk >> 3);
                for (int j = 0; j < ntap; ++j)
                  for (int cx = 0; cx < p.Cblk_x; ++cx) {
                    const float a = xa(a_rows + s * p.HWp + (kk & 7) + j, cx);
                    if (a == 0.f) continue;
                    for (int jv = 0; jv < nv; ++jv)
                      for (int cg = 0; cg < p.Cblk_g; ++cg)
                        D[(((size_t)gi * 128 + (size_t)j * p.Cblk_x + cx) * 8 + jv) * p.Cblk_g + cg] += (double)a * (double)ga(b_slots + s + jv, kk & 7, cg);
                  }
              }
          }
      }
      for (int gi = 0; gi < p.ngroups; ++gi)
        for (int j = 0; j < p.grp_ntap[gi]; ++j)
          for (int jv = 0; jv < p.grp_nv[gi]; ++jv) {
            const int t = p.grp_tap[gi][jv][j];
            for (int cx = 0; cx < p.Cblk_x && cx0 + cx < p.Cx; ++cx)
              for (int cg = 0; cg < p.Cblk_g && cg0 + cg < p.Cg; ++cg)
                dw[(size_t)t * p.dw_ld_tap + (size_t)(cg0 + cg) * p.dw_ld_co + (size_t)(cx0 + cx) * p.dw_ld_cx] +=
                    (float)D[(((size_t)gi * 128 + (size_t)j * p.Cblk_x + cx) * 8 + jv) * p.Cblk_g + cg];
          }
    }
}

}  // namespace jvae

using namespace jvae;

extern "C" {

int jvae_conv_gather_gemm(const void* in, int N, int H, int W, int Cin, int ld_in, const void* wmat, int Cout_pad, int ldw,
                          int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, int Hq, int Wq,
                          void* out, int Ho, int Wo, int Cout, int ld_out, int out_sy, int out_sx, int out_oy, int out_ox,
                          const float* bias, int act, double* stats, void* stream) {
  JVAE_CHECK_ARG(in && wmat && out && tap_dy && tap_dx, "null pointer");
  JVAE_CHECK_ARG(ntaps >= 1 && ntaps <= CONV_MAX_TAPS, "1..64 taps");
  JVAE_CHECK_ARG((ld_in % 8) == 0 && (ldw % 8) == 0, "input / weight channel strides must be multiples of 8");
  JVAE_CHECK_ARG(ld_out >= Cout, "ld_out < Cout");
  JVAE_CHECK_ARG((Cout_pad % 16) == 0 && Cout_pad >= 16 && Cout_pad >= Cout, "Cout_pad must be a multiple of 16, >= Cout");
  JVAE_CHECK_ARG(!stats || Cout_pad <= 2048, "statistics epilogue supports up to 2048 channels");
  JVAE_CHECK_ARG(in_stride >= 1 && in_stride <= 8, "input stride 1..8");
  JVAE_CHECK_ARG((((uintptr_t)in | (uintptr_t)wmat | (uintptr_t)out) & 15) == 0, "16-byte alignment");
  int rc = try_launch_halo(in, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, ntaps, tap_dy, tap_dx, in_stride, Hq, Wq, out, Ho, Wo,
                           Cout, ld_out, out_sy, out_sx, out_oy, out_ox, bias, act, stats, (cudaStream_t)stream);
  if (rc <= 0) return rc;      // launched (0) or failed (< 0); 1 = geometry not covered, use the tap-box kernel
  ConvParams p;
  memset(&p, 0, sizeof(p));
  p.N = N; p.Hq = Hq; p.Wq = Wq;
  tile_shape(Hq, Wq, in_stride, &p.TW, &p.TH, &p.NB);
  p.tiles_x = (Wq + p.TW - 1) / p.TW; p.tiles_y = (Hq + p.TH - 1) / p.TH; p.tiles_n = (N + p.NB - 1) / p.NB;
  p.BN = Cout_pad > 256 ? 256 : Cout_pad;
  if (Cout_pad > 256) JVAE_CHECK_ARG((Cout_pad % 256) == 0, "Cout_pad > 256 must be a multiple of 256");
  // small maps (vgg19's 512-channel layers at 2x2: 16 pixel tiles): narrower channel tiles until the CTAs cover the SMs
  while (p.BN > 64 && (p.BN % 32) == 0 && 2 * p.tiles_x * p.tiles_y * p.tiles_n * (Cout_pad / p.BN) <= sm_count()) p.BN /= 2;
  p.n_tiles_n = Cout_pad / p.BN;
  p.num_tiles = p.tiles_x * p.tiles_y * p.tiles_n * p.n_tiles_n;
  p.Cblk = cblk_of(Cin); p.nCk = (Cin + p.Cblk - 1) / p.Cblk; p.ntaps = ntaps; p.in_stride = in_stride;
  for (int t = 0; t < ntaps; ++t) { p.dy[t] = tap_dy[t]; p.dx[t] = tap_dx[t]; }
  p.Ho = Ho; p.Wo = Wo; p.Cout = Cout; p.ldc = ld_out;
  p.out_sy = out_sy; p.out_sx = out_sx; p.out_oy = out_oy; p.out_ox = out_ox;
  p.act = act & 0xff;
  p.bias = bias; p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.stats = stats; p.cout_pad = Cout_pad;
  const uint32_t stats_bytes = stats ? 2u * (uint32_t)Cout_pad * 8u : 0u;
  p.a_bytes = 128u * p.Cblk * 2u;
  p.tx_bytes = p.a_bytes + (uint32_t)p.BN * p.Cblk * 2u;      // bytes the two TMA boxes deliver per stage
  p.stage_bytes = (p.tx_bytes + 1023u) & ~1023u;
  p.stages = (int)((200u * 1024u - stats_bytes) / p.stage_bytes);
  if (p.stages > 12) p.stages = 12;
  JVAE_CHECK_ARG(p.stages >= 2, "tile too large for shared memory");
  p.tmem_cols = (uint32_t)pow2_ceil(2 * p.BN < 32 ? 32 : 2 * p.BN);
  CUtensorMap tin, tw;
  rc = act_tmap(&tin, in, N, H, W, Cin, ld_in, p.Cblk, p.TW, p.TH, p.NB, in_stride);
  if (rc) return rc;
  {
    const int Ktot = ntaps * p.nCk * p.Cblk;
    uint64_t dims[2] = {(uint64_t)Ktot, (uint64_t)Cout_pad};
    uint64_t strides[1] = {(uint64_t)ldw * 2};
    uint32_t box[2] = {(uint32_t)p.Cblk, (uint32_t)p.BN};
    JVAE_CHECK_ARG(ldw >= Ktot, "weight matrix row shorter than taps*chunks*Cblk");
    rc = make_tmap_bf16(&tw, wmat, 2, dims, strides, box, nullptr, p.Cblk * 2);
    if (rc) return rc;
  }
  const size_t smem = (size_t)p.stages * p.stage_bytes + 256 + stats_bytes + 1024;
  static bool attr = false;
  if (!attr) {
    JVAE_CUDA(cudaFuncSetAttribute(conv_gather_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr = true;
  }
  ConvParams pk = p;
  int grid = p.num_tiles < sm_count() ? p.num_tiles : sm_count();
  void* prof = prof_begin(JVAE_PROF_CONV_TAPBOX, (cudaStream_t)stream);
  conv_gather_gemm_kernel<<<grid, TAPBOX_THREADS, smem, (cudaStream_t)stream>>>(tin, tw, pk);
  prof_end(prof, (cudaStream_t)stream);
  JVAE_LAUNCH_CHECK();
  g_last_conv_kernel = JVAE_KERNEL_CONV_TAPBOX;
  return JVAE_OK;
}

int jvae_conv_subpixel_gemm(const void* in, int N, int H, int W, int Cin, int ld_in, const void* wmat, int Cout_pad, int ldw,
                            int nphases, const int16_t* phase_ntaps, const int16_t* phase_oy, const int16_t* phase_ox,
                            const int16_t* tap_dy, const int16_t* tap_dx, int Hq, int Wq, void* out, int Ho, int Wo, int Cout,
                            int ld_out, int out_s, const float* bias, int act, double* stats, void* stream) {
  JVAE_CHECK_ARG(in && wmat && out && tap_dy && tap_dx && phase_ntaps && phase_oy && phase_ox, "null pointer");
  JVAE_CHECK_ARG(nphases >= 1 && nphases <= 4, "1..4 phases");
  int ntaps = 0;
  for (int i = 0; i < nphases; ++i) {
    JVAE_CHECK_ARG(phase_ntaps[i] >= 1, "every phase needs a tap");
    JVAE_CHECK_ARG(phase_oy[i] >= 0 && phase_oy[i] < out_s && phase_ox[i] >= 0 && phase_ox[i] < out_s, "phase offset outside the stride");
    ntaps += phase_ntaps[i];
  }
  JVAE_CHECK_ARG(ntaps <= CONV_MAX_TAPS, "at most 64 taps over all phases");
  JVAE_CHECK_ARG((ld_in % 8) == 0 && (ldw % 8) == 0, "input / weight channel strides must be multiples of 8");
  JVAE_CHECK_ARG(ld_out >= Cout, "ld_out < Cout");
  JVAE_CHECK_ARG((Cout_pad % 16) == 0 && Cout_pad >= 16 && Cout_pad >= Cout, "Cout_pad must be a multiple of 16, >= Cout");
  JVAE_CHECK_ARG((((uintptr_t)in | (uintptr_t)wmat | (uintptr_t)out) & 15) == 0, "16-byte alignment");
  JVAE_CHECK_ARG(out_s >= 1 && (Hq - 1) * out_s + out_s <= Ho && (Wq - 1) * out_s + out_s <= Wo, "phase grid larger than the output");
  PhaseSpec ps = {nphases, phase_ntaps, phase_oy, phase_ox};
  const int rc = try_launch_halo(in, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, ntaps, tap_dy, tap_dx, 1, Hq, Wq, out, Ho, Wo, Cout,
                                 ld_out, out_s, out_s, 0, 0, bias, act, stats, (cudaStream_t)stream, &ps);
  return rc > 0 ? JVAE_NOT_COVERED : rc;
}

int jvae_conv_wgrad(const void* dy, int N, int Hq, int Wq, int Cout, int ld_dy, const void* x, int H, int W, int Cin, int ld_x,
                    int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, float* dw, int dw_ld_tap,
                    int dw_ld_co, int dw_ld_ci, void* stream) {
  JVAE_CHECK_ARG(dy && x && dw && tap_dy && tap_dx, "null pointer");
  JVAE_CHECK_ARG(ntaps >= 1 && ntaps <= CONV_MAX_TAPS, "1..64 taps");
  JVAE_CHECK_ARG((ld_dy % 8) == 0 && (ld_x % 8) == 0, "channel strides must be multiples of 8");
  JVAE_CHECK_ARG(in_stride >= 1 && in_stride <= 8, "input stride 1..8");
  int rc = try_launch_wgrad_halo(dy, N, Hq, Wq, Cout, ld_dy, x, H, W, Cin, ld_x, ntaps, tap_dy, tap_dx, in_stride, dw,
                                 dw_ld_tap, dw_ld_co, dw_ld_ci, (cudaStream_t)stream);
  if (rc <= 0) return rc;
  // Stride 2 with wide rows (the 64-channel stride-2 layers): the four parity planes of the gathered tensor do not fit one
  // stage together, but each plane alone does -- one launch per plane with that plane's taps (a tap belongs to exactly one
  // plane, so the launches add into disjoint slices of dW).  Tap-box kernel before: 375 us for the 8 -> 16 layer of c2.
  if (in_stride == 2) {
    std::vector<int16_t> sdy[4], sdx[4];
    std::vector<int> ids[4];
    for (int t = 0; t < ntaps; ++t) {
      const int pl = (((tap_dy[t] % 2) + 2) % 2) * 2 + (((tap_dx[t] % 2) + 2) % 2);
      sdy[pl].push_back(tap_dy[t]); sdx[pl].push_back(tap_dx[t]); ids[pl].push_back(t);
    }
    bool covered = true;
    for (int pass = 0; pass < 2 && covered; ++pass)      // first pass: plans only, so that either every plane launches or none
      for (int pl = 0; pl < 4; ++pl) {
        if (ids[pl].empty()) continue;
        const int r2 = try_launch_wgrad_halo(dy, N, Hq, Wq, Cout, ld_dy, x, H, W, Cin, ld_x, (int)ids[pl].size(), sdy[pl].data(),
                                             sdx[pl].data(), 2, dw, dw_ld_tap, dw_ld_co, dw_ld_ci, (cudaStream_t)stream,
                                             ids[pl].data(), pass == 0);
        if (r2 < 0) return r2;
        if (r2 > 0) { covered = false; break; }
      }
    if (covered) return JVAE_OK;
  }
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.N = N; p.Hq = Hq; p.Wq = Wq;
  tile_shape(Hq, Wq, in_stride, &p.TW, &p.TH, &p.NB);
  p.tiles_x = (Wq + p.TW - 1) / p.TW; p.tiles_y = (Hq + p.TH - 1) / p.TH; p.tiles_n = (N + p.NB - 1) / p.NB;
  p.num_tiles = p.tiles_x * p.tiles_y * p.tiles_n;
  p.Cblk_y = cblk_of(Cout); p.Cblk_x = cblk_of(Cin);
  p.ntaps = ntaps; p.in_stride = in_stride;
  for (int t = 0; t < ntaps; ++t) { p.dy[t] = tap_dy[t]; p.dx[t] = tap_dx[t]; }
  p.dw = dw; p.dw_ld_tap = dw_ld_tap; p.dw_ld_co = dw_ld_co; p.dw_ld_cx = dw_ld_ci;
  p.a_bytes = 128u * 64u * 2u;     // the M=64 MMA reads 64 channel columns: reserve a full 64-wide slot for dY
  p.stage_bytes = p.a_bytes + 128u * (uint32_t)p.Cblk_x * 2u;
  p.stage_bytes = (p.stage_bytes + 1023u) & ~1023u;
  p.tx_bytes = 128u * (uint32_t)p.Cblk_y * 2u + 128u * (uint32_t)p.Cblk_x * 2u;
  p.stages = (int)((200u * 1024u) / p.stage_bytes);
  if (p.stages > 8) p.stages = 8;
  // taps per CTA limited by TMEM: taps * Cblk_x <= 512 columns
  p.taps_per_cta = 512 / p.Cblk_x;
  if (p.taps_per_cta > ntaps) p.taps_per_cta = ntaps;
  const int tap_groups = (ntaps + p.taps_per_cta - 1) / p.taps_per_cta;
  p.tmem_cols = (uint32_t)pow2_ceil(p.taps_per_cta * p.Cblk_x < 32 ? 32 : p.taps_per_cta * p.Cblk_x);
  CUtensorMap tdy, tx;
  static bool attr = false;
  if (!attr) {
    JVAE_CUDA(cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr = true;
  }
  const size_t smem = (size_t)p.stages * p.stage_bytes + 256 + 1024;
  // grid: x = slices of the pixel tiles, y = tap groups, z = (64-wide dY channel block) x (X channel block)
  const int ncy = (Cout + p.Cblk_y - 1) / p.Cblk_y;
  p.ncx = (Cin + p.Cblk_x - 1) / p.Cblk_x;
  p.Cy = Cout; p.Cx = Cin;
  const int nz = ncy * p.ncx;
  JVAE_CHECK_ARG(nz <= 65535, "too many channel blocks");
  int gx = (2 * sm_count() + tap_groups * nz - 1) / (tap_groups * nz);
  if (gx < 1) gx = 1;
  if (gx > p.num_tiles) gx = p.num_tiles;
  rc = act_tmap(&tdy, dy, N, Hq, Wq, Cout, ld_dy, p.Cblk_y, p.TW, p.TH, p.NB, 1);
  if (rc) return rc;
  rc = act_tmap(&tx, x, N, H, W, Cin, ld_x, p.Cblk_x, p.TW, p.TH, p.NB, in_stride);
  if (rc) return rc;
  void* prof = prof_begin(JVAE_PROF_WGRAD_TAPBOX, (cudaStream_t)stream);
  conv_wgrad_kernel<<<dim3(gx, tap_groups, nz), CONV_THREADS, smem, (cudaStream_t)stream>>>(tdy, tx, p);
  prof_end(prof, (cudaStream_t)stream);
  JVAE_LAUNCH_CHECK();
  g_last_conv_kernel = JVAE_KERNEL_WGRAD_TAPBOX;
  return JVAE_OK;
}

int jvae_last_conv_kernel(void) { return g_last_conv_kernel; }

int jvae_conv_wgrad_emulate(const float* dy, int N, int Hq, int Wq, int Cout, int ld_dy, const float* x, int H, int W, int Cin, int ld_x,
                            int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, float* dw, int dw_ld_tap,
                            int dw_ld_co, int dw_ld_ci, int* launches) {
  JVAE_CHECK_ARG(dy && x && dw && tap_dy && tap_dx, "null pointer");
  JVAE_CHECK_ARG(ntaps >= 1 && ntaps <= CONV_MAX_TAPS, "1..64 taps");
  JVAE_CHECK_ARG((ld_dy % 8) == 0 && (ld_x % 8) == 0, "channel strides must be multiples of 8");
  JVAE_CHECK_ARG(in_stride >= 1 && in_stride <= 8, "input stride 1..8");
  if (launches) *launches = 0;
  WHaloParams p;
  int rc = try_launch_wgrad_halo(dy, N, Hq, Wq, Cout, ld_dy, x, H, W, Cin, ld_x, ntaps, tap_dy, tap_dx, in_stride, dw, dw_ld_tap, dw_ld_co,
                                 dw_ld_ci, nullptr, nullptr, true, &p);
  if (rc < 0) return rc;
  if (rc == 0) {
    wgrad_plan_emulate(p, dy, ld_dy, x, H, W, ld_x, dw);
    if (launches) *launches = 1;
    return JVAE_OK;
  }
  if (in_stride != 2) return JVAE_NOT_COVERED;
  // the per-plane split of jvae_conv_wgrad
  std::vector<int16_t> sdy[4], sdx[4];
  std::vector<int> ids[4];
  for (int t = 0; t < ntaps; ++t) {
    const int pl = (((tap_dy[t] % 2) + 2) % 2) * 2 + (((tap_dx[t] % 2) + 2) % 2);
    sdy[pl].push_back(tap_dy[t]); sdx[pl].push_back(tap_dx[t]); ids[pl].push_back(t);
  }
  WHaloParams pp[4];
  for (int pl = 0; pl < 4; ++pl) {
    if (ids[pl].empty()) continue;
    rc = try_launch_wgrad_halo(dy, N, Hq, Wq, Cout, ld_dy, x, H, W, Cin, ld_x, (int)ids[pl].size(), sdy[pl].data(), sdx[pl].data(), 2, dw,
                               dw_ld_tap, dw_ld_co, dw_ld_ci, nullptr, ids[pl].data(), true, &pp[pl]);
    if (rc < 0) return rc;
    if (rc > 0) return JVAE_NOT_COVERED;
  }
  for (int pl = 0; pl < 4; ++pl) {
    if (ids[pl].empty()) continue;
    wgrad_plan_emulate(pp[pl], dy, ld_dy, x, H, W, ld_x, dw);
    if (launches) ++*launches;
  }
  return JVAE_OK;
}


// ------------------------------------------------------------------------------------------------ plan emulation (host only)
// Executes the PLAN try_launch_halo makes for a geometry on the host, step by step as conv_halo_kernel does: the TMA box fill
// of a stage (zero outside the image, NaN where the kernel would see leftovers), the MMAs in the order of the chunk records /
// tap table on row addresses decoded from the descriptor words, the fresh / accumulate flags, the epilogue's block table and
// bounds.  A planning mistake (wrong shift, weight block, accumulator column, phase offset, a junk slot reaching a live row)
// shows up as a wrong or NaN output.  No GPU is needed: the `-m "not gpu"` tests run it against torch convolutions.
int jvae_conv_halo_emulate(const float* in, int N, int H, int W, int Cin, int ld_in, const float* wmat, int Cout_pad, int ldw,
                           int nphases, const int16_t* phase_ntaps, const int16_t* phase_oy, const int16_t* phase_ox, int ntaps,
                           const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, int Hq, int Wq, float* out, int Ho, int Wo,
                           int Cout, int ld_out, int out_sy, int out_sx, int out_oy, int out_ox, const float* bias, int act,
                           int* info) {
  JVAE_CHECK_ARG(in && wmat && out && tap_dy && tap_dx, "null pointer");
  JVAE_CHECK_ARG(ntaps >= 1 && ntaps <= CONV_MAX_TAPS, "1..64 taps");
  JVAE_CHECK_ARG(nphases == 0 || (nphases >= 2 && nphases <= 4 && phase_ntaps && phase_oy && phase_ox), "0 or 2..4 phases with their tables");
  JVAE_CHECK_ARG(in_stride >= 1 && in_stride <= 8, "input stride 1..8");
  JVAE_CHECK_ARG((Cout_pad % 16) == 0 && Cout_pad >= Cout && ld_out >= Cout && (ld_in % 8) == 0 && (ldw % 8) == 0, "bad channel layout");
  HaloParams p;
  PhaseSpec ps = {nphases, phase_ntaps, phase_oy, phase_ox};
  const int rc = try_launch_halo(in, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, ntaps, tap_dy, tap_dx, in_stride, Hq, Wq, out, Ho, Wo,
                                 Cout, ld_out, out_sy, out_sx, out_oy, out_ox, bias, act, nullptr, nullptr,
                                 nphases > 0 ? &ps : nullptr, &p);
  if (rc != 0) return rc > 0 ? JVAE_NOT_COVERED : rc;
  if (info) { info[0] = p.G; info[1] = p.PH; info[2] = p.MT; info[3] = p.NBt; info[4] = p.BN; info[5] = p.nck; info[6] = p.resident; info[7] = p.stages; }
  const float qnan = nanf("");
  const uint32_t rb = (uint32_t)p.Cblk * 2u;
  const size_t stage_rows = p.stage_bytes / rb;
  const int per = p.G * p.PH, nblk = p.MT * per;
  const size_t group_rows = (size_t)p.G * p.HWp;                    // SBO of the A descriptor in pixel rows
  std::vector<float> stage(stage_rows * p.Cblk), D((size_t)nblk * 128 * p.BN);
  std::vector<float> wsm;
  auto a_at = [&](size_t row, int c) { return row < stage_rows ? stage[row * p.Cblk + c] : qnan; };
  for (int nt = 0; nt < p.n_tiles_n; ++nt)
    for (int box = 0; box < p.num_boxes; ++box) {
      int mm = box;
      const int sx = mm % p.strips_x; mm /= p.strips_x;
      const int by = mm % p.blocks_y; mm /= p.blocks_y;
      for (int kc = 0; kc < p.nkc; ++kc) {
        // ---- TMA: the box of every plane (zero fill outside the tensor), leftovers elsewhere
        std::fill(stage.begin(), stage.end(), qnan);
        for (int pl = 0; pl < p.nplanes; ++pl)
          for (int nb = 0; nb < p.NBt; ++nb)
            for (int j = 0; j < p.HHs; ++j)
              for (int i = 0; i < p.HWp; ++i) {
                const size_t row = (size_t)pl * (p.plane_bytes / rb) + (size_t)(nb * p.HHs + j) * p.HWp + i;
                const int n = mm * p.NBt + nb;
                const int y = p.in_stride * (by * p.RT + p.dymin + j) + p.plane_ry[pl], x = p.in_stride * (sx * 8 + p.dxmin + i) + p.plane_rx[pl];
                for (int c = 0; c < p.Cblk; ++c) {
                  const int ci = kc * p.Cblk + c;
                  const bool inside = n < N && y >= 0 && y < H && x >= 0 && x < W && ci < Cin;
                  if (row < stage_rows) stage[row * p.Cblk + c] = inside ? in[(((size_t)n * H + y) * W + x) * ld_in + ci] : 0.f;
                }
              }
        // ---- weights of this channel tile / chunk at their shared-memory positions
        wsm.assign((size_t)p.ntaps * p.BN * p.Cblk, qnan);
        for (int t = 0; t < p.ntaps; ++t) {
          const int pos = p.nck > 0 ? p.w_pos[t] : t;
          for (int r = 0; r < p.BN; ++r)
            for (int c = 0; c < p.Cblk; ++c)
              wsm[((size_t)pos * p.BN + r) * p.Cblk + c] = wmat[(size_t)(nt * p.BN + r) * ldw + (size_t)(t * p.nkc + kc) * p.Cblk + c];
        }
        auto mma = [&](int m, size_t a_shift_rows, size_t w_block, int ncols, int dcol, bool overwrite) {
          for (int r = 0; r < 128; ++r) {
            const size_t arow = (size_t)(m * 16 + (r >> 3)) * group_rows + (size_t)(r & 7) + a_shift_rows;
            for (int nn = 0; nn < ncols; ++nn) {
              float acc = 0.f;
              for (int c = 0; c < p.Cblk; ++c) acc += a_at(arow, c) * wsm[(w_block * p.BN + nn) * p.Cblk + c];
              float& d = D[((size_t)m * 128 + r) * (size_t)(per * p.BN) + dcol + nn];
              d = overwrite ? acc : d + acc;
            }
          }
        };
        if (kc == 0) std::fill(D.begin(), D.end(), qnan);
        if (p.nck > 0) {
          for (int m = 0; m < p.MT; ++m)
            for (int c = 0; c < p.nck; ++c) {
              const uint4 ck = p.ck[c];
              mma(m, (size_t)ck.x * 16 / rb, (size_t)ck.y * 16 / p.w_tap_bytes, (int)((ck.z >> 17) & 0x3f) << 3, (int)(ck.w & 0x7fffffffu),
                  (ck.w >> 31) != 0 && kc == 0);
            }
        } else {
          for (int t = 0; t < p.ntaps; ++t)
            for (int m = 0; m < p.MT; ++m) mma(m, (size_t)p.tap_off16[t] * 16 / rb, (size_t)t, p.BN, 0, t == 0 && kc == 0);
        }
      }
      // ---- epilogue: block table, bounds, phase offsets
      for (int blk = 0; blk < nblk; ++blk) {
        const int m = blk / per, rr = blk - m * per;
        const int j = rr / p.PH, ph = rr - j * p.PH;
        for (int r = 0; r < 128; ++r) {
          const int slot = (m * 16 + (r >> 3)) * p.G + j;
          const int nb = slot / p.HHs, yy = slot - nb * p.HHs;
          const int qx = sx * 8 + (r & 7);
          if (!(nb < p.NBt && yy < p.RT) || qx >= p.Wq || yy >= p.Hq - by * p.RT || nb >= p.N - mm * p.NBt) continue;
          const size_t pix = ((size_t)(mm * p.NBt) * p.Ho + (size_t)(by * p.RT * p.out_sy + p.out_oy)) * p.Wo + (size_t)(qx * p.out_sx + p.out_ox) +
                             (size_t)((nb * p.Ho + yy * p.out_sy + p.ph_oy[ph]) * p.Wo + p.ph_ox[ph]);
          for (int c = 0; c < p.BN; ++c) {
            const int ch = nt * p.BN + c;
            if (ch >= ld_out) continue;
            float v = D[((size_t)m * 128 + r) * (size_t)(per * p.BN) + (size_t)blk % per * p.BN + c];
            if (bias && ch < Cout) v += bias[ch];
            if ((act & 0xff) == JVAE_ACT_RELU) v = v > 0.f ? v : (v != v ? v : 0.f);
            else if ((act & 0xff) == JVAE_ACT_SIGMOID) v = 1.f / (1.f + expf(-v));
            else if ((act & 0xff) == JVAE_ACT_LEAKY) v = v > 0.f ? v : JVAE_LEAKY_SLOPE * v;
            out[pix * ld_out + ch] = ch < Cout ? v : 0.f;
          }
        }
      }
    }
  return JVAE_OK;
}


}  // extern "C"

namespace jvae {

// ------------------------------------------------------------------------------------------------ self test
__global__ void conv_fill_kernel(__nv_bfloat16* p, size_t n, uint32_t seed, float scale) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t h = (uint32_t)i * 2654435761u ^ seed;
    h ^= h >> 15; h *= 2246822519u; h ^= h >> 13; h *= 3266489917u; h ^= h >> 16;
    p[i] = __float2bfloat16(scale * (((float)(h & 0xffff) / 32768.f) - 1.f));
  }
}

// naive gather conv with the same tap-table semantics; one thread per (output position q, co)
__global__ void conv_ref_kernel(const __nv_bfloat16* in, int N, int H, int W, int Cin, int ld_in, const __nv_bfloat16* wmat,
                                int ldw, int Cblk, int nCk, int ntaps, const short* dy, const short* dx, int in_stride,
                                int Hq, int Wq, float* out, int Ho, int Wo, int Cout, int out_sy, int out_sx, int out_oy,
                                int out_ox, const float* bias, int act) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)N * Hq * Wq * Cout;
  if (idx >= total) return;
  const int co = (int)(idx % Cout);
  size_t r = idx / Cout;
  const int qx = (int)(r % Wq); r /= Wq;
  const int qy = (int)(r % Hq); r /= Hq;
  const int n = (int)r;
  float acc = 0.f;
  for (int t = 0; t < ntaps; ++t) {
    const int iy = qy * in_stride + dy[t], ix = qx * in_stride + dx[t];
    if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
    for (int ci = 0; ci < Cin; ++ci) {
      const float a = __bfloat162float(in[(((size_t)n * H + iy) * W + ix) * ld_in + ci]);
      const float w = __bfloat162float(wmat[(size_t)co * ldw + (size_t)(t * nCk + ci / Cblk) * Cblk + ci % Cblk]);
      acc = fmaf(a, w, acc);
    }
  }
  if (bias) acc += bias[co];
  if (act == JVAE_ACT_RELU) acc = fmaxf(acc, 0.f);
  const int oy = qy * out_sy + out_oy, ox = qx * out_sx + out_ox;
  out[(((size_t)n * Ho + oy) * Wo + ox) * Cout + co] = acc;
}

__global__ void conv_cmp_kernel(const __nv_bfloat16* got, int ld, const float* ref, int C, size_t pixels, const float* mask,
                                float* err) {
  float e = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < pixels * C; i += (size_t)gridDim.x * blockDim.x) {
    const size_t pix = i / C;
    const int c = (int)(i % C);
    if (mask && mask[pix] == 0.f) continue;
    const float g = __bfloat162float(got[pix * ld + c]), r = ref[i];
    float d = fabsf(g - r) / (1.f + fabsf(r));
    if (!(d == d)) d = 1e30f;
    e = fmaxf(e, d);
  }
  e = warp_max(e);
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(err), __float_as_int(e));
}

__global__ void wgrad_ref_kernel(const __nv_bfloat16* dyp, int N, int Hq, int Wq, int Cout, int ld_dy, const __nv_bfloat16* x,
                                 int H, int W, int Cin, int ld_x, int ntaps, const short* dy, const short* dx, int in_stride,
                                 float* dw) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)ntaps * Cout * Cin) return;
  const int ci = (int)(idx % Cin);
  const int co = (int)((idx / Cin) % Cout);
  const int t = (int)(idx / ((size_t)Cin * Cout));
  float acc = 0.f;
  for (int n = 0; n < N; ++n)
    for (int qy = 0; qy < Hq; ++qy)
      for (int qx = 0; qx < Wq; ++qx) {
        const int iy = qy * in_stride + dy[t], ix = qx * in_stride + dx[t];
        if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
        acc = fmaf(__bfloat162float(dyp[(((size_t)n * Hq + qy) * Wq + qx) * ld_dy + co]),
                   __bfloat162float(x[(((size_t)n * H + iy) * W + ix) * ld_x + ci]), acc);
      }
  dw[idx] = acc;
}

__global__ void f32_cmp_kernel(const float* a, const float* b, size_t n, float* err) {
  float e = 0.f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float d = fabsf(a[i] - b[i]) / (1.f + fabsf(b[i]));
    if (!(d == d)) d = 1e30f;
    e = fmaxf(e, d);
  }
  e = warp_max(e);
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(err), __float_as_int(e));
}

// per-channel sum / sum of squares of a dense (pixels, C) fp32 tensor restricted to the masked pixels; one thread per channel
__global__ void stats_ref_kernel(const float* ref, int C, size_t pixels, const float* mask, const double* got, float* out, float* gotf) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s1 = 0.0, s2 = 0.0;
  for (size_t p = 0; p < pixels; ++p) {
    if (mask && mask[p] == 0.f) continue;
    const double v = ref[p * C + c];
    s1 += v; s2 += v * v;
  }
  out[c] = (float)s1; out[C + c] = (float)s2;
  gotf[c] = (float)got[c]; gotf[C + c] = (float)got[C + c];
}

struct ConvCase { int N, H, W, Cin, Cout, k, pad, in_stride, out_s, act; };

static int r8(int v) { return (v + 7) & ~7; }
static int r16(int v) { return (v + 15) & ~15; }

static int conv_case(const ConvCase& c, int verbose) {
  // regular conv geometry when out_s == 1: q is the output position; out_s == 2 emulates one sub-pixel phase
  const int Hq = (c.in_stride == 2) ? (c.H + 2 * c.pad - c.k) / 2 + 1 : c.H;
  const int Wq = (c.in_stride == 2) ? (c.W + 2 * c.pad - c.k) / 2 + 1 : c.W;
  const int Ho = Hq * c.out_s, Wo = Wq * c.out_s;
  const int ntaps = c.k * c.k;
  std::vector<int16_t> dy(ntaps), dx(ntaps);
  for (int i = 0; i < ntaps; ++i) { dy[i] = (int16_t)(i / c.k - c.pad); dx[i] = (int16_t)(i % c.k - c.pad); }
  const int ld_in = r8(c.Cin), Cblk = cblk_of(c.Cin), nCk = (c.Cin + Cblk - 1) / Cblk;
  const int Cout_pad = c.Cout > 256 ? ((c.Cout + 255) / 256) * 256 : r16(c.Cout);
  const int ldw = ntaps * nCk * Cblk, ld_out = r8(c.Cout);
  const size_t in_n = (size_t)c.N * c.H * c.W * ld_in, w_n = (size_t)Cout_pad * ldw, out_pix = (size_t)c.N * Ho * Wo;
  __nv_bfloat16 *in, *w, *out; float *ref, *bias, *err, *mask, *stats_ref = nullptr, *stats_f = nullptr; double* stats = nullptr; short *ddy, *ddx;
  if (c.act == 0) {
    cudaMalloc(&stats, 2 * c.Cout * 8); cudaMalloc(&stats_ref, 2 * c.Cout * 4); cudaMalloc(&stats_f, 2 * c.Cout * 4);
    cudaMemset(stats, 0, 2 * c.Cout * 8);
  }
  cudaMalloc(&in, in_n * 2); cudaMalloc(&w, w_n * 2); cudaMalloc(&out, out_pix * ld_out * 2);
  cudaMalloc(&ref, out_pix * c.Cout * 4); cudaMalloc(&bias, c.Cout * 4); cudaMalloc(&err, 4); cudaMalloc(&mask, out_pix * 4);
  cudaMalloc(&ddy, ntaps * 2); cudaMalloc(&ddx, ntaps * 2);
  cudaMemcpy(ddy, dy.data(), ntaps * 2, cudaMemcpyHostToDevice); cudaMemcpy(ddx, dx.data(), ntaps * 2, cudaMemcpyHostToDevice);
  conv_fill_kernel<<<128, 256>>>(in, in_n, 17u, 1.f);
  conv_fill_kernel<<<128, 256>>>(w, w_n, 99u, 0.25f);
  std::vector<float> hb(c.Cout);
  for (int i = 0; i < c.Cout; ++i) hb[i] = 0.05f * (float)(i % 13) - 0.3f;
  cudaMemcpy(bias, hb.data(), c.Cout * 4, cudaMemcpyHostToDevice);
  cudaMemset(out, 0, out_pix * ld_out * 2); cudaMemset(ref, 0, out_pix * c.Cout * 4); cudaMemset(err, 0, 4);
  // mask of output pixels this launch writes (phase (0,0) only when out_s == 2)
  std::vector<float> hm(out_pix, 0.f);
  for (int n = 0; n < c.N; ++n) for (int y = 0; y < Hq; ++y) for (int x = 0; x < Wq; ++x)
    hm[((size_t)n * Ho + y * c.out_s) * Wo + x * c.out_s] = 1.f;
  cudaMemcpy(mask, hm.data(), out_pix * 4, cudaMemcpyHostToDevice);
  int rc = jvae_conv_gather_gemm(in, c.N, c.H, c.W, c.Cin, ld_in, w, Cout_pad, ldw, ntaps, dy.data(), dx.data(), c.in_stride, Hq, Wq,
                                 out, Ho, Wo, c.Cout, ld_out, c.out_s, c.out_s, 0, 0, bias, c.act, stats, nullptr);
  float h_err = -1.f;
  if (rc == 0) {
    const size_t total = (size_t)c.N * Hq * Wq * c.Cout;
    conv_ref_kernel<<<(unsigned)((total + 255) / 256), 256>>>(in, c.N, c.H, c.W, c.Cin, ld_in, w, ldw, Cblk, nCk, ntaps, ddy, ddx,
                                                             c.in_stride, Hq, Wq, ref, Ho, Wo, c.Cout, c.out_s, c.out_s, 0, 0, bias, c.act);
    conv_cmp_kernel<<<128, 256>>>(out, ld_out, ref, c.Cout, out_pix, mask, err);
    if (stats) {
      stats_ref_kernel<<<(c.Cout + 63) / 64, 64>>>(ref, c.Cout, out_pix, mask, stats, stats_ref, stats_f);
      f32_cmp_kernel<<<1, 256>>>(stats_f, stats_ref, 2 * (size_t)c.Cout, err);      // folded into the same error word
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("[selftest] conv: CUDA error %s\n", cudaGetErrorString(e)); rc = -2; }
    else cudaMemcpy(&h_err, err, 4, cudaMemcpyDeviceToHost);
  }
  const bool ok = rc == 0 && h_err >= 0.f && h_err < 2e-2f;
  if (verbose || !ok)
    printf("[selftest] conv N=%d %dx%d Cin=%d Cout=%d k=%d pad=%d in_stride=%d out_s=%d act=%d: rc=%d rel_err=%g %s%s\n", c.N, c.H,
           c.W, c.Cin, c.Cout, c.k, c.pad, c.in_stride, c.out_s, c.act, rc, h_err, ok ? "OK" : "FAIL", rc ? jvae_last_error() : "");
  // ---- weight gradient on the same geometry: dY := out (bf16), X := in
  int fails = ok ? 0 : 1;
  if (ok && c.out_s == 1) {
    float *dw, *dwr;
    const size_t dw_n = (size_t)ntaps * c.Cout * c.Cin;
    cudaMalloc(&dw, dw_n * 4); cudaMalloc(&dwr, dw_n * 4);
    cudaMemset(dw, 0, dw_n * 4); cudaMemset(err, 0, 4);
    conv_fill_kernel<<<128, 256>>>(out, out_pix * ld_out, 5u, 0.5f);
    rc = jvae_conv_wgrad(out, c.N, Hq, Wq, c.Cout, ld_out, in, c.H, c.W, c.Cin, ld_in, ntaps, dy.data(), dx.data(), c.in_stride, dw,
                         c.Cout * c.Cin, c.Cin, 1, nullptr);
    h_err = -1.f;
    if (rc == 0) {
      wgrad_ref_kernel<<<(unsigned)((dw_n + 127) / 128), 128>>>(out, c.N, Hq, Wq, c.Cout, ld_out, in, c.H, c.W, c.Cin, ld_in, ntaps,
                                                               ddy, ddx, c.in_stride, dwr);
      f32_cmp_kernel<<<64, 256>>>(dw, dwr, dw_n, err);
      cudaError_t e = cudaDeviceSynchronize();
      if (e != cudaSuccess) { printf("[selftest] wgrad: CUDA error %s\n", cudaGetErrorString(e)); rc = -2; }
      else cudaMemcpy(&h_err, err, 4, cudaMemcpyDeviceToHost);
    }
    const bool ok2 = rc == 0 && h_err >= 0.f && h_err < 2e-2f;
    if (verbose || !ok2)
      printf("[selftest] wgrad same geometry: rc=%d rel_err=%g %s%s\n", rc, h_err, ok2 ? "OK" : "FAIL", rc ? jvae_last_error() : "");
    fails += ok2 ? 0 : 1;
    cudaFree(dw); cudaFree(dwr);
  }
  if (stats) { cudaFree(stats); cudaFree(stats_ref); cudaFree(stats_f); }
  cudaFree(in); cudaFree(w); cudaFree(out); cudaFree(ref); cudaFree(bias); cudaFree(err); cudaFree(mask); cudaFree(ddy); cudaFree(ddx);
  return fails;
}

// all four sub-pixel phases of a stride-2 ConvTranspose2d (k, pad, output 2H x 2W) in one launch against the naive kernel run
// phase by phase on the same merged weight matrix
static int subpixel_case(int N, int H, int W, int Cin, int Cout, int k, int pad, int act, int verbose) {
  const int Ho = 2 * H, Wo = 2 * W;
  std::vector<int16_t> dy, dx, pn, poy, pox;
  for (int fy = 0; fy < 2; ++fy)
    for (int fx = 0; fx < 2; ++fx) {
      int cnt = 0;
      for (int i = 0; i < k; ++i)
        for (int j = 0; j < k; ++j)
          if ((fy + pad - i) % 2 == 0 && (fx + pad - j) % 2 == 0) {
            dy.push_back((int16_t)((fy + pad - i) / 2)); dx.push_back((int16_t)((fx + pad - j) / 2));
            ++cnt;
          }
      pn.push_back((int16_t)cnt); poy.push_back((int16_t)fy); pox.push_back((int16_t)fx);
    }
  const int ntaps = (int)dy.size();
  const int ld_in = r8(Cin), Cblk = cblk_of(Cin), Cout_pad = r16(Cout), ldw = ntaps * Cblk, ld_out = r8(Cout);
  const size_t in_n = (size_t)N * H * W * ld_in, w_n = (size_t)Cout_pad * ldw, out_pix = (size_t)N * Ho * Wo;
  __nv_bfloat16 *in, *w, *out; float *ref, *bias, *err, *stats_ref = nullptr, *stats_f = nullptr; double* stats = nullptr; short *ddy, *ddx;
  if (act == 0) {
    cudaMalloc(&stats, 2 * Cout * 8); cudaMalloc(&stats_ref, 2 * Cout * 4); cudaMalloc(&stats_f, 2 * Cout * 4);
    cudaMemset(stats, 0, 2 * Cout * 8);
  }
  cudaMalloc(&in, in_n * 2); cudaMalloc(&w, w_n * 2); cudaMalloc(&out, out_pix * ld_out * 2);
  cudaMalloc(&ref, out_pix * Cout * 4); cudaMalloc(&bias, Cout * 4); cudaMalloc(&err, 4);
  cudaMalloc(&ddy, ntaps * 2); cudaMalloc(&ddx, ntaps * 2);
  cudaMemcpy(ddy, dy.data(), ntaps * 2, cudaMemcpyHostToDevice); cudaMemcpy(ddx, dx.data(), ntaps * 2, cudaMemcpyHostToDevice);
  conv_fill_kernel<<<128, 256>>>(in, in_n, 23u, 1.f);
  conv_fill_kernel<<<128, 256>>>(w, w_n, 77u, 0.25f);
  std::vector<float> hb(Cout);
  for (int i = 0; i < Cout; ++i) hb[i] = 0.05f * (float)(i % 13) - 0.3f;
  cudaMemcpy(bias, hb.data(), Cout * 4, cudaMemcpyHostToDevice);
  cudaMemset(out, 0xff, out_pix * ld_out * 2); cudaMemset(ref, 0, out_pix * Cout * 4); cudaMemset(err, 0, 4);
  int rc = jvae_conv_subpixel_gemm(in, N, H, W, Cin, ld_in, w, Cout_pad, ldw, 4, pn.data(), poy.data(), pox.data(), dy.data(), dx.data(),
                                   H, W, out, Ho, Wo, Cout, ld_out, 2, bias, act, stats, nullptr);
  float h_err = -1.f;
  if (rc == 0) {
    const size_t total = (size_t)N * H * W * Cout;
    int first = 0;
    for (int ph = 0; ph < 4; ++ph) {
      conv_ref_kernel<<<(unsigned)((total + 255) / 256), 256>>>(in, N, H, W, Cin, ld_in, w + (size_t)first * Cblk, ldw, Cblk, 1, pn[ph],
                                                               ddy + first, ddx + first, 1, H, W, ref, Ho, Wo, Cout, 2, 2, poy[ph],
                                                               pox[ph], bias, act);
      first += pn[ph];
    }
    conv_cmp_kernel<<<128, 256>>>(out, ld_out, ref, Cout, out_pix, nullptr, err);
    if (stats) {
      stats_ref_kernel<<<(Cout + 63) / 64, 64>>>(ref, Cout, out_pix, nullptr, stats, stats_ref, stats_f);
      f32_cmp_kernel<<<1, 256>>>(stats_f, stats_ref, 2 * (size_t)Cout, err);
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("[selftest] subpixel: CUDA error %s\n", cudaGetErrorString(e)); rc = -2; }
    else cudaMemcpy(&h_err, err, 4, cudaMemcpyDeviceToHost);
  }
  const bool ok = rc == 0 && h_err >= 0.f && h_err < 2e-2f;
  if (verbose || !ok)
    printf("[selftest] subpixel N=%d %dx%d Cin=%d Cout=%d k=%d pad=%d act=%d: rc=%d rel_err=%g %s%s\n", N, H, W, Cin, Cout, k, pad, act, rc,
           h_err, ok ? "OK" : (rc == JVAE_NOT_COVERED ? "NOT COVERED" : "FAIL"), rc < 0 ? jvae_last_error() : "");
  if (stats) { cudaFree(stats); cudaFree(stats_ref); cudaFree(stats_f); }
  cudaFree(in); cudaFree(w); cudaFree(out); cudaFree(ref); cudaFree(bias); cudaFree(err); cudaFree(ddy); cudaFree(ddx);
  return ok ? 0 : 1;
}

int conv_selftest(int verbose) {
  const ConvCase cases[] = {
      {4, 8, 8, 64, 64, 3, 1, 1, 1, 0},     // SW128, NB=2
      {3, 16, 16, 32, 32, 5, 2, 1, 1, 1},   // SW64, relu
      {2, 32, 32, 16, 32, 5, 2, 1, 1, 0},   // SW32
      {5, 32, 32, 3, 64, 3, 1, 1, 1, 0},    // 3 input channels (zero-filled to 16)
      {2, 32, 32, 32, 3, 5, 2, 1, 1, 0},    // 3 output channels
      {3, 8, 8, 128, 128, 3, 1, 1, 1, 0},   // two channel chunks
      {2, 4, 4, 64, 512, 3, 1, 1, 1, 0},    // two output-channel tiles
      {3, 16, 16, 32, 64, 5, 2, 2, 1, 0},   // stride-2 conv (TMA element strides)
      {3, 8, 8, 64, 64, 3, 1, 1, 2, 0},     // sub-pixel phase store (output stride 2)
      {70, 28, 28, 8, 24, 3, 1, 1, 1, 0},   // ragged W, many tiles
      {2, 1, 1, 64, 64, 1, 0, 1, 1, 0},     // 1x1 spatial
      {7, 8, 8, 64, 64, 5, 2, 1, 1, 0},     // halo kernel: streamed weights, 3 stacked images per box, ragged batch
      {5, 16, 16, 64, 32, 5, 2, 1, 1, 0},   // halo kernel: resident weights, one image per box
      {3, 32, 32, 32, 32, 5, 2, 1, 1, 0},   // halo kernel: two M-tiles per box
      {2, 40, 40, 8, 16, 3, 1, 1, 1, 0},    // halo kernel: two row blocks per image
      {9, 8, 8, 64, 64, 3, 1, 1, 2, 0},     // halo kernel: sub-pixel phase store, stacked images
      {5, 16, 16, 64, 64, 5, 2, 2, 1, 0},   // stride 2, 64 channels: weight gradient as one halo launch per parity plane
  };
  int fails = 0;
  for (const auto& c : cases) {
    fails += conv_case(c, verbose);
    if (fails > 4) { printf("[selftest] conv: too many failures, stopping\n"); break; }
  }
  fails += subpixel_case(5, 16, 16, 32, 32, 5, 2, 0, verbose);      // c2 imager 16 -> 32: one image per box, 4 x 32 columns
  fails += subpixel_case(7, 8, 8, 64, 64, 5, 2, 0, verbose);        // c2 imager 8 -> 16: channel tile halved, 3 images per box
  fails += subpixel_case(3, 16, 16, 32, 16, 4, 1, 1, verbose);      // k = 4 (two taps per axis and phase), relu
  fails += subpixel_case(2, 40, 24, 16, 24, 3, 1, 0, verbose);      // two row blocks per image, ragged channel count
  fails += subpixel_case(150, 8, 8, 16, 16, 5, 2, 0, verbose);      // more boxes than SMs
  return fails;
}
}  // namespace jvae
