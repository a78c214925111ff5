/*
 * jvae_b200.h — C ABI of libjvae_sm100.so: the B200-native (sm_100a) replacement for the
 * arithmetic of moxime/joint-vae's train/eval hot path.
 *
 * The reference has no FFI of its own (it is PyTorch eager code); every entry point below
 * replaces the interior of one reference function (file:line relative to the reference root)
 * and is called from the host-side mirror in joint-vae_b200/ through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C: raw device pointers, explicit sizes, `void* stream` is a cudaStream_t
 *     (PyTorch's current stream); no torch types, no C++ exceptions across the boundary.
 *   - every function returns 0 on success, a negative jvae_status otherwise;
 *     jvae_last_error() gives a thread-local human-readable message.
 *   - the library never allocates user-visible memory: outputs and workspaces are caller
 *     allocated (PyTorch owns all tensors, as in the reference).
 *   - dtype codes: JVAE_F32 = 0, JVAE_BF16 = 1.
 *   - all tensors are dense row-major with the shapes given in the comments.
 */
#ifndef JVAE_B200_H
#define JVAE_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JVAE_ABI_VERSION 17

enum jvae_status {
  JVAE_OK = 0,
  JVAE_ERR_INVALID = -1,    /* bad argument (shape, dtype, null pointer) */
  JVAE_ERR_CUDA = -2,       /* a CUDA runtime/driver call failed */
  JVAE_ERR_UNSUPPORTED = -3,/* valid request this build does not implement */
  JVAE_ERR_NOGPU = -4       /* no sm_100 device */
};

enum jvae_dtype { JVAE_F32 = 0, JVAE_BF16 = 1 };

/* prior variance parametrisation, module/priors.py:110-122 */
enum jvae_var_dim { JVAE_VAR_SCALAR = 0, JVAE_VAR_DIAG = 1, JVAE_VAR_FULL = 2 };
/* prior family, module/priors.py:35-52 */
enum jvae_prior_kind { JVAE_PRIOR_GAUSSIAN = 0, JVAE_PRIOR_TILTED = 1, JVAE_PRIOR_UNIFORM = 2 };

const char* jvae_last_error(void);
int jvae_abi_version(void);
/* number of SMs / compute capability of `device`; JVAE_ERR_NOGPU if it is not sm_100 */
int jvae_device_info(int device, int* sm_count, int* cc_major, int* cc_minor);
/* how many kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t jvae_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Fused class-conditional Gaussian-prior ELBO  (cvae.py:626-902, module/priors.py:173-342,
 * module/losses.py:8-27,52-86).  B samples, L latent draws (+ slab 0 = the mean), K latent
 * dims, C classes, D = prod(input_shape) pixels.
 * ------------------------------------------------------------------------------------------ */
typedef struct jvae_elbo_cfg {
  int32_t B, L, K, C, D;
  int32_t xreco_dtype;      /* jvae_dtype of x_reco (and of d_x_reco) */
  int32_t logits_dtype;     /* jvae_dtype of logits (and of d_logits) */
  int32_t var_dim;          /* jvae_var_dim */
  int32_t prior_kind;       /* jvae_prior_kind */
  int32_t conditional;      /* 1: C class means, 0: single prior (means is (1,K)) */
  int32_t has_xreco;        /* 0 for type 'vib' (no reconstruction term) */
  int32_t has_logits;       /* 1 if a classifier output exists (y_is_decoded) */
  int32_t sigma_is_log;     /* Sigma stored as log sigma (learned), layers.py:84-87 */
  int32_t sigma_is_rmse;    /* Sigma(is_rmse): sigma^2 := batch wmse, cvae.py:662-670 */
  float   beta;             /* KL weight actually applied (1 unless with_beta), cvae.py:898 */
  float   gamma_w;          /* cross_y weight actually applied (0 => not added), cvae.py:557-562 */
  float   var_w;            /* kl_var_weighting, priors.py:323 */
  float   tau;              /* tilted / uniform priors */
  float   alpha;            /* uniform prior: log rho inside [-tau,tau], priors.py:423-424 */
  int32_t prior_stats_ready;/* 1: jvae_elbo_prior_stats already ran on this workspace for the current prior parameters */
  int32_t categorical;      /* 1: output_distribution='categorical' (losses.py:30-49, cvae.py:654-660, 683, 776): x_reco holds 256
                               logits per pixel variable, cross_x = mean_l sum_d CE(logits, floor(255 x_d)),
                               wmse = mean_l mean_d (argmax / 255 - x_d)^2 (not divided by sigma), log_iws = -CE */
  int32_t cat_group;        /* logit v of variable d of row r = (l, b) sits at r*256*D + (d / cat_group)*256*cat_group +
                               v*cat_group + d % cat_group: cat_group = channels for the conv imager's channels_last output
                               (x in channels_last order), cat_group = D for the reference's (256, *input_shape) layout */
  int32_t sigma_per_sample; /* 1: sigma (and d_sigma) hold one value per sample (B): Sigma coded by the encoder's sigma head,
                               layers.py:297-298, 398-399, cvae.py:631-634 (sdim = 1) */
} jvae_elbo_cfg;

/* bytes of scratch the ELBO entry points need for `cfg`.  The first 4*B bytes (arrival counters) must be ZERO before
 * the first use; every launch leaves them zero again, so one workspace can be reused without clearing AS LONG AS the
 * layout (B, L, K, number of priors) stays the same: use one workspace per layout, or re-zero it when the layout changes. */
size_t jvae_elbo_workspace_bytes(const jvae_elbo_cfg* cfg);

/* Prior statistics (mean of the class means, its variance, log det Sigma_c: cvae.py:747-754, priors.py:173-186) into the
 * workspace.  They depend on the prior parameters only; calling this early (e.g. before the network forward) and setting
 * cfg.prior_stats_ready = 1 keeps the tiny prologue launch off the loss step.  With prior_stats_ready = 0 the forward
 * entry points run it themselves. */
int jvae_elbo_prior_stats(const jvae_elbo_cfg* cfg, const float* means, const float* inv_trans, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Train forward (y given).  Replaces cvae.py:626-902 + priors.py:252-326 + losses.py:8-27,73-86.
 *   x (B,D) f32; x_reco (L+1,B,D) [slab 0 is not read]; mu, log_var (B,K) f32;
 *   logits (L+1,B,C) or NULL; y (B) int64; means (C,K) f32; inv_trans (C)|(C,K)|(C,K,K) f32;
 *   sigma: 1 f32 on the device = the raw Sigma parameter (log sigma if sigma_is_log; sdim == 1), it is a
 *   learned parameter so it is never read back to the host.
 *   outputs, each (B) f32 (NULL = not wanted): kl zdist var_kl wmse cross_x cross_y total dzdist.
 *   finite_flag: 1 int32 the CALLER initialises to non-zero; the kernel clears it if some total is NaN/Inf or a label is
 *   out of range (replaces the per-parameter isnan scan of cvae.py:2454-2457). */
int jvae_elbo_train_fwd(const jvae_elbo_cfg* cfg, const float* x, const void* x_reco,
                        const float* mu, const float* log_var, const void* logits, const int64_t* y,
                        const float* means, const float* inv_trans, const float* sigma,
                        float* kl, float* zdist, float* var_kl, float* wmse, float* cross_x,
                        float* cross_y, float* total, float* dzdist, int32_t* finite_flag,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Train backward of sum_b g[b]*total[b] (SURVEY.md §8a backward contract; the reference uses
 * autograd over the same lines).  g (B) f32 (= 1/B for total.mean()).  wmse (B): saved forward output `wmse`; with
 * sigma_is_rmse pass the forward's `cross_x` instead (the per-sample sigma^2 = mse is recovered from it; d_sigma is not written).
 *   d_x_reco (L+1,B,D) [slab 0 written as zeros]; d_mu, d_log_var (B,K) f32: DIRECT terms only
 *   (the path through z is added by jvae_sample_bwd); d_logits (L+1,B,C); d_means (C,K) f32;
 *   d_inv_trans like inv_trans (NULL unless var_dim is diag/full); d_sigma: 1 f32 (B with sigma_per_sample). */
int jvae_elbo_train_bwd(const jvae_elbo_cfg* cfg, const float* g, const float* x, const void* x_reco,
                        const float* mu, const float* log_var, const void* logits, const int64_t* y,
                        const float* means, const float* inv_trans, const float* sigma, const float* wmse,
                        void* d_x_reco, float* d_mu, float* d_log_var, void* d_logits,
                        float* d_means, float* d_inv_trans, float* d_sigma,
                        void* workspace, size_t workspace_bytes, void* stream);

/* scores written by the eval kernel, one row of JVAE_NSCORES floats per sample
 * (cvae.py:972-1085 batch_dist_measures; -2s / -a-p-q suffixes only select the ROC mode) */
enum jvae_score {
  JVAE_S_ELBO = 0,     /* 'elbo' / 'max': max_c(-total) */
  JVAE_S_SUM = 1,      /* 'sum': logsumexp_c(-total) */
  JVAE_S_MEAN = 2,     /* 'mean': logmeanexp_c(-total) */
  JVAE_S_IWS = 3,      /* 'iws': logsumexp_c(iws) + log C */
  JVAE_S_SOFTKL = 4,   /* 'soft' / 'softkl': max softmax_c(-kl) */
  JVAE_S_ZDIST = 5,    /* 'zdist': max_c(-zdist) */
  JVAE_S_KL = 6,       /* 'kl': max_c(-kl) */
  JVAE_S_MSE = 7,      /* 'mse': -cross_x */
  JVAE_S_WMSE = 8,     /* 'wmse': -wmse */
  JVAE_S_LOGITS = 9,   /* 'logits': max_c logits */
  JVAE_S_BASELINE = 10,/* 'baseline': max softmax(logits) */
  JVAE_S_HYZ = 11,     /* 'hyz': sum p log p */
  JVAE_S_STD = 12,     /* 'std': unbiased std_c(-total) */
  JVAE_S_SOFTIWS = 13, /* 'softiws': max softmax_c(iws) */
  JVAE_NSCORES = 16
};
/* predictions written by the eval kernel, JVAE_NPRED int32 per sample (cvae.py:938-970) */
enum jvae_pred { JVAE_P_LOSS = 0, JVAE_P_ESTY = 1, JVAE_P_CLOSEST = 2, JVAE_P_IWS = 3, JVAE_NPRED = 4 };

/* Eval / scoring forward (y None: losses for every class).  Replaces cvae.py:593-600,626-917,
 * priors.py:252-342 (no (C,B,K) / (L,C,B,K) materialisation), losses.py:62-71, cvae.py:938-1085.
 *   z (L+1,B,K) f32; eps_norm (L,B) f32 = sum_k eps^2.
 *   per-class outputs (C,B) f32: kl zdist var_kl total iws cross_y; per-sample (B): wmse cross_x dzdist;
 *   logits_out (B,C) f32 = mean_{l>=1} logits; scores (B,JVAE_NSCORES) f32; preds (B,JVAE_NPRED) int32.
 *   For non-conditional priors (vae/jvae/vib) kl zdist var_kl iws are (B) and total/cross_y (C,B) only
 *   when has_logits and gamma_w != 0. Any output pointer may be NULL. */
int jvae_elbo_eval_fwd(const jvae_elbo_cfg* cfg, const float* x, const void* x_reco,
                       const float* mu, const float* log_var, const float* z, const float* eps_norm,
                       const void* logits, const float* means, const float* inv_trans, const float* sigma,
                       float* kl, float* zdist, float* var_kl, float* total, float* iws, float* cross_y,
                       float* wmse, float* cross_x, float* dzdist, float* logits_out,
                       float* scores, int32_t* preds,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Reparameterisation sampler (module/vae_layers/layers.py:230-244, 388-396).
 *   head (B,2K) f32: [mu | raw log_var] (the fused dense_mean/dense_log_var GEMM output, bias added);
 *   eps_in (L+1,B,K) f32 or NULL (NULL => Philox4x32-10 + Box-Muller from (seed, offset));
 *   writes mu, log_var = clip(raw,-20,20) (B,K) f32; z (L+1,B,K) f32 and optional bf16 copy z_bf16;
 *   eps_out (L,B,K) f32 (slabs 1..L) and eps_norm (L,B).  is_sampled: layers.py:243.
 *   uniform != 0 draws U(-sqrt3, sqrt3) instead (layers.py:237).
 *   The Philox stream position is offset + *offset_dev (offset_dev: one uint64 on the device, or NULL): a caller that
 *   advances the device word after every call gets fresh noise from a replayed CUDA graph of the step.
 * ------------------------------------------------------------------------------------------ */
int jvae_sample_fwd(int B, int L, int K, const float* head, const float* eps_in,
                    uint64_t seed, uint64_t offset, const uint64_t* offset_dev, int is_sampled, int uniform,
                    float* mu, float* log_var, float* z, void* z_bf16, float* eps_out, float* eps_norm,
                    void* stream);
/* d_head (B,2K) = [d_mu_direct + sum_l dz | (d_lv_direct + sum_l dz*0.5*exp(lv/2)*eps) * 1[|raw|<=20]] */
int jvae_sample_bwd(int B, int L, int K, const float* head, const float* log_var, const float* eps,
                    const void* dz, int dz_dtype, const float* d_mu_direct, const float* d_lv_direct,
                    int is_sampled, float* d_head, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense layers on the tcgen05 tensor cores (nn.Linear in layers.py:284-298,441-453,476-480;
 * ConvTranspose2d on a 1x1 input, conv-models.ini:25).  bf16 operands, fp32 accumulation in TMEM.
 *   D[M,N] = act( A[M,K] * W[N,K]^T + bias[N] )
 * ------------------------------------------------------------------------------------------ */
enum jvae_act { JVAE_ACT_NONE = 0, JVAE_ACT_RELU = 1, JVAE_ACT_SIGMOID = 2, JVAE_ACT_LEAKY = 3 };   /* leaky: slope 0.01 (nn.LeakyReLU default, misc.py:27) */
#define JVAE_LEAKY_SLOPE 0.01f
enum jvae_gemm_mode {
  JVAE_GEMM_NT = 0,  /* D[M,N] = A[M,K] . B[N,K]^T   forward:  y = x W^T                       */
  JVAE_GEMM_NN = 1,  /* D[M,N] = A[M,K] . B[K,N]     dgrad:    dx = dy W                        */
  JVAE_GEMM_TN = 2   /* D[M,N] = A[K,M]^T . B[K,N]   wgrad:    dW = dy^T x   (reduction over rows) */
};
/*   a, b: bf16, leading dimensions lda/ldb in elements (multiples of 8);
 *   out_bf16 / out_f32: either or both, leading dimension ldd; bias (N) f32 or NULL;
 *   col_stats (2,N) f32 or NULL: += per-column sum and sum of squares of the pre-activation
 *   (BatchNorm batch statistics, conv.py:216-217); accumulate = 1: out_f32 += result; accumulate = n >= 2: the reduction is
 *   split into n slices (one more grid dimension) whose partial products are added to out_f32 with fp32 atomics -- for
 *   weight gradients with few output tiles and a long reduction; no bias / activation / bf16 output then. */
int jvae_gemm_bf16(int mode, int M, int N, int K, const void* a, int lda, const void* b, int ldb,
                   const float* bias, int act, void* out_bf16, float* out_f32, int ldd,
                   float* col_stats, int accumulate, void* stream);
/* The forward of Linear -> activation -> Dropout(p) in training mode (layers.py:177-181, cvae.py:207-211): jvae_gemm_bf16
 * (mode NT only; accumulate 0 and col_stats NULL) whose epilogue multiplies act(.) by keep[row, col] / (1 - p).
 *   keep[row, col] = word (col & 3) of Philox4x32-10(counter (col >> 2, row, pos_lo, pos_hi), key (seed_lo, seed_hi))
 *                    >= floor(p * 2^32),   pos = offset + *offset_dev (offset_dev: one uint64 on the device, or NULL)
 * so the mask depends on (seed, pos, row, col) alone.  p in [0, 1]; p == 1 writes zeros.  Advancing the device word after
 * every call (the sampler's stream position, jvae_sample_fwd) gives a replayed CUDA graph fresh masks. */
int jvae_gemm_bf16_dropout(int mode, int M, int N, int K, const void* a, int lda, const void* b, int ldb,
                           const float* bias, int act, void* out_bf16, float* out_f32, int ldd,
                           float* col_stats, int accumulate, float p, uint64_t seed, uint64_t offset,
                           const uint64_t* offset_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Convolutions as implicit GEMM on tcgen05, NHWC bf16 activations (nn.Conv2d / nn.ConvTranspose2d of the
 * features / imager stacks, module/vae_layers/conv.py:189-219, conv-models.ini:11-30).
 *
 * jvae_conv_gather_gemm: for every position q = (n, qy, qx) of an (N, Hq, Wq) grid
 *     out[n, qy*out_sy + out_oy, qx*out_sx + out_ox, co] =
 *         act( bias[co] + sum_t sum_ci in[n, qy*in_stride + tap_dy[t], qx*in_stride + tap_dx[t], ci] * W[co][t][ci] )
 *   with out-of-image reads equal to zero.  One call is a Conv2d (stride 1..8), a ConvTranspose2d of stride 1
 *   (flipped taps), ONE sub-pixel phase of a stride-s ConvTranspose2d (out_s = s <= 8, out_o = phase), or the data
 *   gradient of any of them, depending on the tap table and weight arrangement the host passes.  in_stride is 1..8
 *   (the 'x4+0:4' / ':8' tokens of the spec grammar, conv.py:20-84): strides 1 and 2 run on the halo kernel where it
 *   takes the geometry, strides 3..8 always on the tap-box kernel.
 *   in  (N,H,W,ld_in) bf16, Cin real channels; wmat (Cout_pad, ldw) bf16 with row co = [tap][chunk][Cblk] where
 *   Cblk = 16/32/64 for Cin <= 16 / <= 32 / > 32 and chunk = ceil(Cin/Cblk) (zero padded); Cout_pad a multiple of 16
 *   (of 256 above 256); out (N,Ho,Wo,ld_out) bf16, channels >= Cout up to ld_out are written as zeros.
 *   stats (2,Cout) f64 or NULL: += per-channel sum and sum of squares of the pre-activation over the positions this
 *   call writes, taken from the fp32 accumulators (BatchNorm2d batch statistics, conv.py:216-217); fp64 so that the
 *   arrival order of warps / CTAs does not change the result (run-to-run reproducible).
 * jvae_conv_wgrad: dw[t][co][ci] += sum_q dy[n,qy,qx,co] * x[n, qy*in_stride + tap_dy[t], qx*in_stride + tap_dx[t], ci]
 *   (in_stride 1..8)
 *   (fp32, atomically accumulated into dw: the caller zeroes it, or passes the live .grad buffer to accumulate into);
 *   element (t, co, ci) lives at dw[t*dw_ld_tap + co*dw_ld_co + ci*dw_ld_ci], so the torch (Cout,Cin,kh,kw) layout is
 *   (1, Cin*kh*kw, kh*kw).
 * ------------------------------------------------------------------------------------------ */
int jvae_conv_gather_gemm(const void* in, int N, int H, int W, int Cin, int ld_in, const void* wmat, int Cout_pad, int ldw,
                          int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, int Hq, int Wq,
                          void* out, int Ho, int Wo, int Cout, int ld_out, int out_sy, int out_sx, int out_oy, int out_ox,
                          const float* bias, int act, double* stats, void* stream);
/* ALL sub-pixel phases of a stride-`out_s` ConvTranspose2d (conv.py:189-219, the imager stacks of conv-models.ini:25) or of
 * the data gradient of a strided Conv2d in ONE launch: phase i owns phase_ntaps[i] consecutive entries of the tap table (and
 * of wmat's [tap] blocks, same row layout as jvae_conv_gather_gemm) and writes
 *     out[n, qy*out_s + phase_oy[i], qx*out_s + phase_ox[i], co]
 * for every q of the (N, Hq, Wq) grid all phases share (even output sizes).  The input box is read once for all phases and
 * the taps of different phases that read the same input shift are one MMA (their weights stacked along N).
 * Returns JVAE_NOT_COVERED (nothing launched, no error text) when the geometry is outside what the merged kernel handles
 * (wide layers, weights that do not fit in shared memory): the caller then issues one
 * jvae_conv_gather_gemm per phase, which computes the same thing. */
#define JVAE_NOT_COVERED 1
int jvae_conv_subpixel_gemm(const void* in, int N, int H, int W, int Cin, int ld_in, const void* wmat, int Cout_pad, int ldw,
                            int nphases, const int16_t* phase_ntaps, const int16_t* phase_oy, const int16_t* phase_ox,
                            const int16_t* tap_dy, const int16_t* tap_dx, int Hq, int Wq, void* out, int Ho, int Wo, int Cout,
                            int ld_out, int out_s, const float* bias, int act, double* stats, void* stream);
/* Diagnostic, HOST ONLY (no GPU, every pointer is host memory, tensors as fp32): executes the plan the halo convolution kernel
 * would run for this geometry -- box fills, chunk records / tap table, accumulator columns, epilogue block table -- on the CPU,
 * so the planner is testable without a device.  nphases = 0: the plan of jvae_conv_gather_gemm (ntaps / in_stride / out_o as
 * there); nphases >= 2: the plan of jvae_conv_subpixel_gemm (out_sy = out_sx = out_s, out_o = 0).  info (8 ints, may be NULL)
 * receives {G, phases, M-tiles per box, images per box, channel tile, chunk records, resident weights, stages}.
 * Returns JVAE_NOT_COVERED when the halo kernel does not take the geometry (always for in_stride 3..8). */
int jvae_conv_halo_emulate(const float* in, int N, int H, int W, int Cin, int ld_in, const float* wmat, int Cout_pad, int ldw,
                           int nphases, const int16_t* phase_ntaps, const int16_t* phase_oy, const int16_t* phase_ox, int ntaps,
                           const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, int Hq, int Wq, float* out, int Ho, int Wo,
                           int Cout, int ld_out, int out_sy, int out_sx, int out_oy, int out_ox, const float* bias, int act,
                           int* info);
/* The same for the halo weight-gradient kernel (HOST ONLY, fp32 host tensors): the plan(s) jvae_conv_wgrad would run -- one, or one
 * per parity plane for stride-2 layers whose planes do not fit a stage together -- executed on the CPU; dw += as the kernel does.
 * *launches receives the number of kernel launches the plan stands for.  JVAE_NOT_COVERED: the tap-box kernel would run. */
int jvae_conv_wgrad_emulate(const float* dy, int N, int Hq, int Wq, int Cout, int ld_dy, const float* x, int H, int W, int Cin, int ld_x,
                            int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, float* dw, int dw_ld_tap,
                            int dw_ld_co, int dw_ld_ci, int* launches);
int jvae_conv_wgrad(const void* dy, int N, int Hq, int Wq, int Cout, int ld_dy, const void* x, int H, int W, int Cin, int ld_x,
                    int ntaps, const int16_t* tap_dy, const int16_t* tap_dx, int in_stride, float* dw, int dw_ld_tap,
                    int dw_ld_co, int dw_ld_ci, void* stream);
/* which kernel the calling thread's last jvae_conv_gather_gemm / jvae_conv_wgrad call launched (measurement aid:
 * bench.py attributes per-launch CUDA-event times to the dominant kernel of the step) */
enum jvae_conv_kernel { JVAE_KERNEL_CONV_HALO = 1, JVAE_KERNEL_CONV_TAPBOX = 2, JVAE_KERNEL_WGRAD_HALO = 3, JVAE_KERNEL_WGRAD_TAPBOX = 4 };
int jvae_last_conv_kernel(void);


/* ------------------------------------------------------------------------------------------
 * Layers between the convolutions, NHWC bf16, P = N*H*W pixels (module/vae_layers/conv.py:189-227):
 * BatchNorm2d (torch semantics: biased variance to normalise, unbiased for running_var, momentum 0.1),
 * activation backward + bias gradient, MaxPool2d, AvgPool2d, UpsamplingNearest2d.
 * ------------------------------------------------------------------------------------------ */
/* stats (2,C) f64 += per-channel sum / sum of squares of y (P,C) with leading dimension ld (zero stats first) */
int jvae_bn_stats(const void* y, size_t P, int C, int ld, double* stats, void* stream);
/* out = act(gamma * (y - mean) * rstd + beta).  training != 0: mean / biased var from stats (sums over P), writes
 * save_mean_rstd (2,C), updates running_mean / running_var / num_batches (any may be NULL); training == 0: running stats */
int jvae_bn_apply_fwd(const void* y, size_t P, int C, int ld_y, const double* stats, const float* gamma, const float* beta,
                      float eps, float momentum, float* running_mean, float* running_var, int64_t* num_batches, int training,
                      int act, void* out, int ld_out, float* save_mean_rstd, void* stream);
/* backward of act(BN_train(y)) given da = dL/d(out): dy (P,C) bf16, dgamma, dbeta (C) f32 (+=, any may be NULL);
 * sums (2,C) f64 scratch */
int jvae_bn_bwd(const void* da, int ld_da, const void* y, int ld_y, size_t P, int C, const float* save_mean_rstd,
                const float* gamma, const float* beta, int act, double* sums, void* dy, int ld_dy, float* dgamma, float* dbeta,
                void* stream);
/* DenseNet blocks (torchvision _DenseBlock): every layer appends its channels to ONE (P, C_total) bf16 buffer, whose batch
 * statistics live in ONE (2, C_total) f64 array (row stride stats_ld = C_total) written once per channel and read by every
 * later pre-activation BatchNorm; the backward accumulates the channel gradients of all consumers in ONE fp32 buffer.
 * jvae_bn_stats_ld: stats[c] / stats[stats_ld + c] += sum / sum of squares of y (P, C) for c < C (pass the statistics of
 * the channel slice's first channel; stats_ld == C is jvae_bn_stats) */
int jvae_bn_stats_ld(const void* y, size_t P, int C, int ld, double* stats, int stats_ld, void* stream);
/* jvae_bn_apply_fwd on a channel prefix of a dense block: statistics with row stride stats_ld (sums at stats[c], sums of
 * squares at stats[stats_ld + c]); gamma / beta / running statistics / num_batches of THIS consumer.  C, ld_y, ld_out
 * multiples of 8, rows 16-byte aligned. */
int jvae_bn_preact_fwd(const void* y, size_t P, int C, int ld_y, const double* stats, int stats_ld, const float* gamma,
                       const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                       int64_t* num_batches, int training, int act, void* out, int ld_out, float* save_mean_rstd, void* stream);
/* backward of act(BN(y)) given da, ACCUMULATED: dx (P, C) fp32 with row stride ld_dx += dL/dy.  training != 0: batch
 * statistics (save_mean_rstd from the forward), sums (2,C) f64 scratch, dgamma / dbeta += (either may be NULL); training == 0:
 * running statistics, dx += da * act' * gamma * rsqrt(running_var + eps) (the input gradient of an eval-mode network),
 * sums / dgamma / dbeta unused.  C and every ld multiples of 8, rows 16-byte aligned. */
int jvae_bn_preact_bwd(const void* da, int ld_da, const void* y, int ld_y, size_t P, int C, const float* save_mean_rstd,
                       const float* gamma, const float* beta, const float* running_mean, const float* running_var, float eps,
                       int training, int act, double* sums, float* dx, int ld_dx, float* dgamma, float* dbeta, void* stream);
/* dst (P, C) bf16 with row stride ld_dst = src (P, C) fp32 with row stride ld_src (a slice of the gradient accumulator) */
int jvae_cast_f32_bf16_ld(const float* src, int ld_src, void* dst, int ld_dst, size_t P, int C, void* stream);
/* dy = da * act'(.) expressed with the activation OUTPUT a_out (relu, sigmoid; act none: dy = da, dy may be NULL);
 * dbias (C) f32 += sum over pixels of dy (NULL = not wanted) */
int jvae_act_bwd(const void* da, int ld_da, const void* a_out, int ld_a, size_t P, int C, int act, void* dy, int ld_dy,
                 float* dbias, void* stream);
/* Backward of jvae_gemm_bf16_dropout's epilogue, in one launch: dz (M,N) bf16 = da * keep / (1 - p) * act', the mask
 * regenerated from the same (p, seed, offset, *offset_dev) as the forward (pass a device copy of the position the forward read);
 * act' from the saved post-dropout output a_out (relu: a_out > 0; leaky: sign of a_out; sigmoid: s (1 - s) with
 * s = a_out (1 - p); none: 1, a_out may be NULL).  dbias (N) f32 = sum over rows of dz (WRITTEN, not accumulated), summed
 * in a fixed order without atomics; either output may be NULL.  Any N; da, a_out, dz bf16 with leading dimensions >= N. */
int jvae_act_dropout_bwd(const void* da, int ld_da, const void* a_out, int ld_a, int M, int N, int act, float p, uint64_t seed,
                         uint64_t offset, const uint64_t* offset_dev, void* dz, int ld_dz, float* dbias, void* stream);
/* MaxPool2d(k, stride >= k, padding 0, floor mode): out (N,(H-k)/stride+1,(W-k)/stride+1,C) */
int jvae_maxpool_fwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, void* out, int ld_out, void* stream);
/* gradient to the first maximum of each window (torch tie rule); `in` is the pooling input */
int jvae_maxpool_bwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, const void* dout, int ld_dout,
                     void* din, int ld_din, void* stream);
/* Padded / overlapping max pooling (kernel k, stride, padding pad <= k/2, floor mode; padded positions never win): the
 * stem MaxPool2d(3, 2, 1) of torchvision's ResNets (conv.py:247-272 of the reference wraps them).  out is
 * (N, (H+2pad-k)/stride+1, (W+2pad-k)/stride+1, C); backward gives every input pixel the gradients of the windows whose FIRST
 * maximum (row-major scan, torch's tie rule) it is -- gather form, no atomics. */
int jvae_maxpool_pad_fwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, int pad, void* out,
                         int ld_out, void* stream);
int jvae_maxpool_pad_bwd(const void* in, int N, int H, int W, int C, int ld_in, int k, int stride, int pad, const void* dout,
                         int ld_dout, void* din, int ld_din, void* stream);
/* k x k average pooling with stride k (k = H = W is AdaptiveAvgPool2d(1), the last layer of the ResNet features; 'A' tokens of
 * the conv spec language): backward == 0: dst (N,H/k,W/k,C) = window means of src (N,H,W,C); backward != 0: dst (N,H,W,C) =
 * src (N,H/k,W/k,C) / k^2 spread over the windows */
int jvae_avgpool(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int k, int backward,
                 void* stream);
/* Backward of a k x k stride-1 'same' convolution with few output channels (k * Co <= 16, Co <= 4: the image head 32 -> 3 of
 * the deconv presets, conv-models.ini:25) in separable form: the gradient of the 1 x k convolution to k * Co channels,
 * T[r][ty*Co + co] = sum_tx sum_ci x[r + (0, tx - pad)][ci] W[co][ci][ty][tx], whose vertical sum is the layer's output, is
 *   jvae_vstack_rows: U[r][ty*Co + co] = dy[r - (ty - pad, 0)][co] (zero outside the image, zero padding channels up to ld_u):
 *                     the 1 x k kernel's data / weight gradients then run on U, k taps instead of k^2. */
int jvae_vstack_rows(const void* dy, int ld_dy, int N, int H, int W, int k, int pad, int Co, void* U, int ld_u, void* stream);
/* out = act(a + b) over P pixels x C channels: the join of a residual block (out += identity; relu); act = NONE adds two
 * gradient branches */
int jvae_add_act(const void* a, int ld_a, const void* b, int ld_b, size_t P, int C, int act, void* out, int ld_out,
                 void* stream);
/* backward == 0: dst (N,2H,2W,C) = nearest up-sampling of src (N,H,W,C); backward != 0: dst (N,H,W,C) = 2x2 block sums of src */
int jvae_upsample2(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int backward, void* stream);
/* UpsamplingNearest2d(scale_factor=s) for an integer s >= 1 (the 'U:s' tokens of the spec grammar, conv.py:20-84, 149-151):
 * backward == 0: dst (N,sH,sW,C) = nearest up-sampling of src (N,H,W,C); backward != 0: dst (N,H,W,C) = s x s block sums of
 * src (N,sH,sW,C), summed in fp32 in a fixed order per pixel (gather form, no atomics: bit-reproducible).  Channel strides
 * ld_src / ld_dst as for jvae_upsample2, which stays the s = 2 kernel. */
int jvae_upsample_nearest(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int s, int backward,
                          void* stream);
/* AvgPool2d(kernel (kh,kw), stride (sh,sw), padding (ph,pw)) with torch's defaults ceil_mode=False, count_include_pad=True
 * (the 'A' tokens of the spec grammar that overlap, pad or do not tile the map, conv.py:144-148; with (kh,kw) = (sh,sw) =
 * (H,W) also AdaptiveAvgPool2d(1) on a non-square map).  Output (N, (H+2ph-kh)/sh+1, (W+2pw-kw)/sw+1, C); the divisor is
 * always kh*kw.  Padding at most half the kernel.  backward == 0: dst = pooled src; backward != 0: src is the output gradient
 * and dst (N,H,W,C) the input gradient, each input pixel summing dout / (kh*kw) over the windows that cover it (gather form,
 * no atomics, deterministic; pixels no window covers get zero). */
int jvae_avgpool_pad(const void* src, int ld_src, void* dst, int ld_dst, int N, int H, int W, int C, int kh, int kw, int sh, int sw,
                     int ph, int pw, int backward, void* stream);

/* ------------------------------------------------------------------------------------------
 * Small data-movement / elementwise kernels of the step
 * ------------------------------------------------------------------------------------------ */
/* f32 -> bf16 cast of n elements (weights repack, activations) */
int jvae_cast_f32_bf16(const float* src, void* dst, size_t n, void* stream);
int jvae_cast_bf16_f32(const void* src, float* dst, size_t n, void* stream);
/* Patch matrix of a convolution (weight gradient on small maps as ONE TN GEMM, nn.Conv2d in conv.py:189-219): row (n, y, x) of
 * out (N*Hq*Wq, ld_out) holds column ci * ntaps + t = x[n, y * in_stride + dy_t, x * in_stride + dx_t, ci], zero outside the
 * map; x is NHWC bf16 with channel stride ld_x.  The column order is torch's (Cin, kh, kw), so
 * jvae_gemm_bf16(TN, Cout, Cin * ntaps, N*Hq*Wq, dY, ld_dy, out, ld_out, ..., accumulate) adds the weight gradient to .grad.
 * tap_major != 0: column t * C + ci instead (any window of up to 64 taps; the caller permutes the small result). */
int jvae_im2col_bf16(const void* x, int N, int H, int W, int C, int ld_x, int ntaps, const int16_t* tap_dy, const int16_t* tap_dx,
                     int in_stride, int Hq, int Wq, void* out, int ld_out, int tap_major, void* stream);
/* NCHW f32 -> NHWC bf16 (optionally padding channels to c_pad with zeros) and back */
int jvae_nchw_to_nhwc_bf16(const float* src, void* dst, int n, int c, int h, int w, int c_pad, void* stream);
int jvae_nhwc_bf16_to_nchw(const void* src, float* dst, int n, int c, int h, int w, int c_pad, void* stream);

/* ------------------------------------------------------------------------------------------
 * Weight re-packing.  The reference re-reads its live nn.Parameters in every step (cvae.py:2424-2461: forward, backward,
 * optimizer.step on the same tensors).  Here the optimizer updates ONE flat fp32 buffer in place and the tensor-core
 * kernels read bf16 copies in their own arrangements ([Cout_pad][tap][Cin chunk], transposed for the data gradient,
 * 1 x k rows of the separable image head, (pixel, co) rows of the 1x1 -> k x k GEMM, plain casts of Linear weights);
 * jvae_pack_weights rebuilds every arrangement of a whole layer stack in ONE launch, once per step.
 * A job describes one destination tensor dst[r][t][c] (r < rows_pad, t < T, c < cols_pad, dense, zero where r >= rows or
 * c >= cols):  dst[r][t][c] = src[(r / R0) * s_r1 + (r % R0) * s_r0 + taps[tap_off + t] * s_t + (c / C0) * s_c1 + (c % C0) * s_c0]
 * (strides in elements).  cols_pad must be a multiple of 8.  The job table and the tap table live in device memory; jobs are
 * sorted by first_block, job j owning blocks [first_block_j, first_block_j + jvae_pack_job_blocks(rows_pad, T, cols_pad)).
 * ------------------------------------------------------------------------------------------ */
typedef struct jvae_pack_job {
  const float* src;         /* fp32 parameter (device) */
  void* dst;                /* bf16 (or f32 when dst_f32) destination (device, 16-byte aligned) */
  int64_t s_r1, s_r0, s_t, s_c1, s_c0;
  int32_t rows, rows_pad, R0;
  int32_t T, tap_off;
  int32_t cols, cols_pad, C0;
  int32_t dst_f32;
  int32_t first_block;
} jvae_pack_job;
int jvae_pack_job_blocks(long long rows_pad, int T, int cols_pad);
int jvae_pack_weights(const jvae_pack_job* jobs_dev, int n_jobs, const int32_t* taps_dev, int total_blocks, void* stream);

/* ------------------------------------------------------------------------------------------
 * Input batches (SURVEY 8f row 3).  Replaces, for datasets held as uint8 (N, H, W, C) arrays (torchvision's
 * CIFAR / SVHN / MNIST `.data`), the per-sample PIL transforms of utils/torch_load.py:405-426
 * (RandomHorizontalFlip, RandomCrop(size, padding, padding_mode='edge'), Pad(2) / CenterCrop, ToTensor) and the
 * DataLoader collate + x.to(device) of cvae.py:2245-2256, 2427: one gather of B samples by index, the augmentation as
 * an index map, uint8 / 255 -> f32, written as the (B, C, out_H, out_W) NCHW batch `evaluate` takes.
 * The random decisions (flip flags, crop offsets) are inputs, so the result is bit-identical to torchvision's for the
 * same draws.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t H, W, C;                  /* source images: uint8 (n_src, H, W, C) */
  int32_t out_H, out_W;             /* size of the produced images */
  int32_t crop_pad;                 /* RandomCrop((H, W), padding=crop_pad, padding_mode='edge'); 0: no random crop */
  int32_t flip_first;               /* 1: the flip precedes the crop in data_augmentation, 0: it follows it */
  int32_t post_off_y, post_off_x;   /* output pixel (y, x) = augmented pixel (y + post_off_y, x + post_off_x), 0 outside the
                                       image: Pad(p) is (-p, -p) with out = H + 2p; CenterCrop is (+round((H-out)/2), ..) */
} jvae_batch_cfg;
/* src: device (or pinned, device-mapped) uint8 images; index (B) int64 sample numbers < n_src; flip (B) uint8 or NULL;
 * crop_ij (B, 2) int32 = RandomCrop's (i, j) in the padded image, or NULL; out (B, C, out_H, out_W) f32 */
int jvae_batch_u8_to_f32(const jvae_batch_cfg* cfg, const void* src, long long n_src, const long long* index, int B,
                         const unsigned char* flip, const int* crop_ij, float* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer (module/optimizers.py:79-81,120-121: clip_grad_norm_ then Adam / AMSGrad / SGD with L2 weight decay)
 * on one flat f32 parameter / gradient buffer.  grad may be the bf16 all-reduced bucket.
 * ------------------------------------------------------------------------------------------ */
/* The flat buffers hold the trainable parameters back to back, each starting on a multiple of JVAE_OPT_CHUNK elements;
 * chunk_seg[i / JVAE_OPT_CHUNK] = index of the parameter that owns element i (int32, n / JVAE_OPT_CHUNK entries, device).
 * torch.optim.Adam keeps a step count per parameter and skips parameters whose grad is None (here: whose slice of the zeroed
 * flat gradient stayed all zero, e.g. the classifier of a cvae with gamma = 0, cvae.py:216-218): seg_active (nseg int32,
 * ZEROED by the caller before jvae_grad_sqnorm) receives 1 for every parameter with a non-zero gradient element, seg_step
 * (nseg int32, device) holds the per-parameter step counts, seg_bc (nseg x 2 f32) is scratch for the bias corrections.
 * Nothing of the step count lives on the host, so a captured CUDA graph of the step replays correctly. */
#define JVAE_OPT_CHUNK 256
/* norm2_out[0] += sum(grad^2) (zero it first); grad_dtype is a jvae_dtype; chunk_seg / seg_active: both or neither */
int jvae_grad_sqnorm(const void* grad, int grad_dtype, size_t n, float* norm2_out, const int32_t* chunk_seg, int32_t* seg_active,
                     void* stream);
/* p,m,v (n) f32; clip_coef = min(1, max_norm/(sqrt(norm2)+1e-6)) computed on device from norm2;
 * max_norm <= 0 disables clipping.  Two launches: per-parameter step counts / bias corrections, then the update. */
int jvae_adam_step(float* p, float* m, float* v, const void* grad, int grad_dtype, size_t n,
                   const float* norm2, float max_norm, float lr, float beta1, float beta2, float eps,
                   float weight_decay, int nseg, const int32_t* chunk_seg, const int32_t* seg_active, int32_t* seg_step,
                   float* seg_bc, float grad_scale, void* stream);
/* jvae_adam_step with AMSGrad (torch.optim.Adam(amsgrad=True)): vmax (n) f32, zero-initialised, holds the running maximum
 * of v; vmax = max(vmax, v) after the v update and denom = sqrt(vmax) / sqrt(1 - beta2^t) + eps. */
int jvae_adam_amsgrad_step(float* p, float* m, float* v, float* vmax, const void* grad, int grad_dtype, size_t n,
                           const float* norm2, float max_norm, float lr, float beta1, float beta2, float eps,
                           float weight_decay, int nseg, const int32_t* chunk_seg, const int32_t* seg_active, int32_t* seg_step,
                           float* seg_bc, float grad_scale, void* stream);
/* torch.optim.SGD on the same flat buffers and parameter table: d = clip_coef * grad_scale * g + weight_decay * p; with
 * momentum != 0, buf = d on a parameter's first update (its seg_step becomes 1 in this call), else
 * buf = momentum * buf + (1 - dampening) * d, then d = nesterov ? d + momentum * buf : buf; p -= lr * d.
 * buf (n) f32 is required iff momentum != 0 (with momentum == 0 only p and g are touched).  As for Adam, a parameter whose
 * gradient slice is all zero counts as having no gradient: it is neither updated nor counted.  Two launches: per-parameter
 * step counts, then the update. */
int jvae_sgd_step(float* p, float* buf, const void* grad, int grad_dtype, size_t n, const float* norm2, float max_norm,
                  float lr, float momentum, float dampening, int nesterov, float weight_decay, int nseg,
                  const int32_t* chunk_seg, const int32_t* seg_active, int32_t* seg_step, float grad_scale, void* stream);

/* Per-launch profile: while enabled, the fused ELBO and convolution entry points bracket their main kernel launch with CUDA events recorded
 * on the launching stream inside the library (tags below); jvae_profile_drain waits for them, returns (tag, milliseconds)
 * pairs and forgets them.  Enable only around eager launches (event records are not stream-capture safe). */
enum jvae_prof_tag { JVAE_PROF_ELBO_TRAIN_FWD = 1, JVAE_PROF_ELBO_TRAIN_BWD = 2, JVAE_PROF_ELBO_EVAL_FWD = 3,
                     JVAE_PROF_CONV_HALO = 4, JVAE_PROF_CONV_TAPBOX = 5, JVAE_PROF_WGRAD_HALO = 6, JVAE_PROF_WGRAD_TAPBOX = 7 };
int jvae_profile_enable(int on);
int jvae_profile_drain(int32_t* tags, float* ms, int max_records);

/* self-test of the tensor-core kernels against naive CUDA-core references run on the device;
 * prints a report to stdout, returns the number of failed cases */
int jvae_selftest(int verbose);
/* diagnostic: which shifted / strided start addresses K-major swizzled UMMA descriptors accept on this GPU (prints a
 * table; returns the number of baseline cases that failed) */
int jvae_probe_descriptors(int verbose);
/* diagnostic: measured cycles per tcgen05.mma for small N and for 1..8 independent accumulators (prints a table) */
int jvae_probe_mma_rate(void);
/* diagnostic: fills the shared memory and TMEM of every SM with `pattern` (tests use it to show that no kernel result depends on
 * what an earlier kernel left on the SM) */
int jvae_probe_poison(unsigned pattern, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* JVAE_B200_H */
