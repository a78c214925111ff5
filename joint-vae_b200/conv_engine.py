"""Native execution of the reference's conv / deconv stacks (module/vae_layers/conv.py:128-244) on libjvae_sm100.so.

A stack (the module list build_de_conv_layers produces: Conv2d | ConvTranspose2d, optional BatchNorm2d, activation,
MaxPool2d / AvgPool2d, UpsamplingNearest2d) is compiled once into a list of steps and runs as ONE autograd node with a
hand-written backward.  Activations live in HBM as NHWC bf16 (channel stride padded to a multiple of 8 elements = the
16-byte granularity TMA needs); weights stay fp32 torch Parameters in the reference's layout (state_dict compatible) and
are re-packed to the kernels' bf16 [Cout][tap][Cin-chunk] arrangement whenever their version changes.

Every convolution flavour is one or several launches of the same tcgen05 "gather GEMM" (csrc/conv.cu):
  Conv2d stride 1/2            taps (i-p, j-p), input stride s
  ConvTranspose2d stride 1     taps (p-i, p-j)
  ConvTranspose2d stride s>1   s*s sub-pixel phases, each a small stride-1 gather written with output stride s
  data gradients               the same two forms with the roles of Conv / ConvTranspose exchanged
  ConvTranspose2d on 1x1 input a plain GEMM (csrc/gemm.cu)
Weight gradients use csrc/conv.cu's wgrad kernel (MN-major operands straight from the NHWC tensors).
BatchNorm batch statistics come out of the convolution epilogue (fp32 accumulators); normalisation + activation is one
streaming pass (csrc/norm.cu), its backward two.

`K` is the kernel backend: `NativeKernels` (ctypes -> CUDA) in the product.  tests/ substitute a torch emulation of the
same entry points to check the tap tables / weight arrangements on machines without a GPU; the product never does.
"""
import os

import torch
from torch import nn

from . import _native as nat
from . import engine


def r8(n):
    return (n + 7) & ~7


def cblk_of(c):
    return 64 if c > 32 else (32 if c > 16 else 16)


def cout_pad_of(c):
    return ((c + 255) // 256) * 256 if c > 256 else ((c + 15) // 16) * 16


_ACT_CODE = {nn.ReLU: 1, nn.Sigmoid: 2, nn.Identity: 0, nn.LeakyReLU: 3}

# Fold the BatchNorm-backward reduction of layer i-1 into the data-gradient kernel of layer i (jvae_conv_gather_gemm_bn).
# Correct and covered by the GPU tests (run them with JVAE_FUSE_BN_REDUCE=1), but measured SLOWER on B200 at c2 even with the
# saved pre-BN tile fed through its own TMA ring: +0.7 ms per fused 32-channel launch against 0.37 ms saved.  The N = 32
# MMAs of these layers already saturate the shared-memory bandwidth (measured pacing, DESIGN.md section 3.2), so every
# extra shared-memory read in the epilogue slows the MMAs themselves.  Opt-in until the per-channel constants move to
# registers / the constant bank.
import os as _os
FUSE_BN_REDUCE = _os.environ.get('JVAE_FUSE_BN_REDUCE', '0') == '1'
# opt-in, NOT yet measured on the GPU (DESIGN.md section 6, vgg19's 512-channel layers at 2x2): 'same' stride-1 convolutions on
# maps of at most 2x2 pixels as ONE dense GEMM over (pixel, channel) pairs -- every (output pixel, input pixel) pair is exactly
# one filter tap, so nothing is wasted on padding taps and the launch fills the machine (M = batch, N = K = pixels * channels)
DENSE_SMALL = _os.environ.get('JVAE_CONV_DENSE_SMALL', '0') == '1'
# the separable image head runs its FORWARD as the direct k x k convolution (tap-stacked halo kernel, one fp32 accumulation of all
# k^2 taps, no fp32 intermediate of 16 channels per pixel): 336 us against 241 + 147 us at c2 since the second epilogue pass.  The
# backward stays separable (data gradient 229 us against ~400 direct, weight gradient 184 against ~530).  0 restores the 1 x k pass.
SEP_FWD_DIRECT = _os.environ.get('JVAE_HEAD_FWD_DIRECT', '1') != '0'
# weight gradients on maps of at most this many pixels go through a patch matrix + one TN GEMM (0 disables)
IM2COL_MAXPIX = int(_os.environ.get('JVAE_CONV_IM2COL_MAXPIX', '16'))


# ------------------------------------------------------------------------------------------------ kernel backend
class NativeKernels:
    """thin adaptor from NHWC tensors to the C ABI (include/jvae_b200.h)"""
    act_dtype = torch.bfloat16

    @staticmethod
    def empty(shape, like, dtype=torch.bfloat16):
        return torch.empty(shape, dtype=dtype, device=like.device)

    @staticmethod
    def zeros(shape, like, dtype=torch.float32):
        return torch.zeros(shape, dtype=dtype, device=like.device)

    @staticmethod
    def to_nhwc(x, c_pad):
        n, c, h, w = x.shape
        x = x.float().contiguous()
        if h * w == 1 and c_pad == c:          # a (N, C) matrix: the layouts coincide, plain cast
            return nat.cast_f32_bf16(x).view(n, 1, 1, c)
        return nat.nchw_to_nhwc_bf16(x, c_pad)

    @staticmethod
    def to_nchw(t, C):
        n, h, w, ld = t.shape
        if h * w == 1 and ld == C:
            return nat.cast_bf16_f32(t).view(n, C, 1, 1)
        return nat.nhwc_bf16_to_nchw(t, C)

    @staticmethod
    def gather(x, Cin, wmat, cout_pad, taps, in_stride, Hq, Wq, out, Cout, out_s, out_o, bias, act, stats, bn=None):
        N, H, W, ld_in = x.shape
        _, Ho, Wo, _ = out.shape
        ld_out = out.stride(2)          # `out` may be a channel slice of a wider buffer (a dense block's new channels)
        return nat.conv_gather_gemm(x, N, H, W, Cin, ld_in, wmat, cout_pad, wmat.shape[1], taps, in_stride, Hq, Wq, out, Ho,
                                    Wo, Cout, ld_out, out_s, out_o, bias, act, stats, bn=bn)

    @staticmethod
    def wgrad(g, Cg, x, Cx, taps, in_stride, dw, swapped=False):
        """dw (Cg, Cx, T) fp32 (the torch weight layout with the kernel window flattened) += sum_px g x_shifted.
        swapped: dw is (Cx, Cg, T) instead (the roles of the two tensors were exchanged by the caller)"""
        N, Hq, Wq, ld_g = g.shape
        _, H, W, ld_x = x.shape
        T = len(taps[0])
        P = N * Hq * Wq
        small = Hq * Wq <= IM2COL_MAXPIX and Cx % 8 == 0 and Cg >= 128 and Cx >= 64 and T in (1, 4, 9, 25)
        if not swapped and small and dw.is_contiguous():
            # one patch matrix + ONE TN GEMM accumulating into .grad (the per-tap kernels have no operand reuse there).  With few
            # output tiles the reduction over the pixels is split over the SMs (partial products added with fp32 atomics).
            # (Tried for the ResNet stem too -- 7 x 7, stride 2, 3 channels, tap-major patch matrix: 122 us against ~90 us on the
            # halo kernel, so only the small maps come here.)
            cols = torch.empty((P, Cx * T), dtype=torch.bfloat16, device=g.device)
            nat.im2col(x, N, H, W, Cx, ld_x, taps, in_stride, Hq, Wq, cols)
            tiles = ((Cg + 127) // 128) * ((Cx * T + 127) // 128)
            ksplit = max(1, min(nat.sm_count() // tiles, (P + 511) // 512)) if tiles < 100 else 1
            nat.gemm_bf16(2, Cg, Cx * T, P, g.view(P, ld_g), ld_g, cols, Cx * T, out_f32=dw.view(Cg, Cx * T), ldd=Cx * T,
                          accumulate=ksplit if ksplit > 1 else True)
            return
        if swapped:
            nat.conv_wgrad(g, N, Hq, Wq, Cg, ld_g, x, H, W, Cx, ld_x, taps, in_stride, dw, 1, T, Cg * T)
        else:
            nat.conv_wgrad(g, N, Hq, Wq, Cg, ld_g, x, H, W, Cx, ld_x, taps, in_stride, dw, 1, Cx * T, T)

    @staticmethod
    def gemm(mode, M, N, K, a, b, bias=None, act=0, out_bf16=None, out_f32=None):
        nat.gemm_bf16(mode, M, N, K, a, a.stride(0), b, b.stride(0), bias=bias, act=act, out_bf16=out_bf16, out_f32=out_f32,
                      ldd=N)

    @staticmethod
    def phases_arg(ops):
        return nat.phases_arg(ops)

    @staticmethod
    def subpixel(x, Cin, wmat, cout_pad, phases, Hq, Wq, out, Cout, out_s, bias, act, stats):
        """all sub-pixel phases in one launch (jvae_conv_subpixel_gemm); False = not covered, nothing launched"""
        N, H, W, ld_in = x.shape
        _, Ho, Wo, ld_out = out.shape
        return nat.conv_subpixel_gemm(x, N, H, W, Cin, ld_in, wmat, cout_pad, wmat.shape[1], phases, Hq, Wq, out, Ho, Wo, Cout,
                                      ld_out, out_s, bias, act, stats)

    bn_stats = staticmethod(nat.bn_stats)
    bn_stats_ld = staticmethod(nat.bn_stats_ld)
    bn_preact_fwd = staticmethod(nat.bn_preact_fwd)
    bn_preact_bwd = staticmethod(nat.bn_preact_bwd)
    cast_f32_bf16_ld = staticmethod(nat.cast_f32_bf16_ld)
    bn_apply_fwd = staticmethod(nat.bn_apply_fwd)
    bn_bwd = staticmethod(nat.bn_bwd)
    act_bwd = staticmethod(nat.act_bwd)
    maxpool_fwd = staticmethod(nat.maxpool_fwd)
    maxpool_bwd = staticmethod(nat.maxpool_bwd)
    upsample2 = staticmethod(nat.upsample2)
    maxpool_pad_fwd = staticmethod(nat.maxpool_pad_fwd)
    maxpool_pad_bwd = staticmethod(nat.maxpool_pad_bwd)
    avgpool = staticmethod(nat.avgpool)
    add_act = staticmethod(nat.add_act)
    vsum_rows = staticmethod(nat.vsum_rows)
    vstack_rows = staticmethod(nat.vstack_rows)
    taps_arg = staticmethod(nat.taps_arg)


K = NativeKernels


# ------------------------------------------------------------------------------------------------ gather-op tables
def conv_form(k, p, s, Hq, Wq):
    """out[q] = sum_ij in[q*s + (i-p, j-p)] * G[:, ij, :]   (Conv2d forward, ConvTranspose2d data gradient)"""
    taps = [(i - p, j - p) for i in range(k) for j in range(k)]
    return [dict(taps=taps, idx=list(range(k * k)), in_stride=s, Hq=Hq, Wq=Wq, out_s=(1, 1), out_o=(0, 0))]


def deconv_form(k, p, s, Ho, Wo, allow_empty=False):
    """out[o] = sum over (i, j) with (o + p - i) divisible by s of in[(o + p - (i,j)) / s] * G[:, ij, :]
    (ConvTranspose2d forward, Conv2d data gradient): one stride-1 gather per sub-pixel phase, no zero insertion."""
    ops = []
    for fy in range(s):
        rows = [i for i in range(k) if (fy + p - i) % s == 0]
        for fx in range(s):
            cols = [j for j in range(k) if (fx + p - j) % s == 0]
            Hq, Wq = (Ho - fy + s - 1) // s, (Wo - fx + s - 1) // s
            if Hq <= 0 or Wq <= 0:
                continue
            if not rows or not cols:
                if allow_empty:      # data gradient of a kernel smaller than its stride (conv1x1 stride 2 shortcuts): this
                    continue         # sub-pixel phase receives nothing; the caller zero-fills the gradient tensor
                raise NotImplementedError('transposed convolution with kernel smaller than its stride')
            taps = [((fy + p - i) // s, (fx + p - j) // s) for i in rows for j in cols]
            ops.append(dict(taps=taps, idx=[i * k + j for i in rows for j in cols], in_stride=1, Hq=Hq, Wq=Wq,
                            out_s=(s, s), out_o=(fy, fx)))
    return ops


def pack_gather_weights(G, idx, cin):
    """G (Cout, k*k, Cin) fp32 -> bf16 (Cout_pad, T*nCk*Cblk): row co = [tap][chunk][Cblk], zero padded"""
    Co = G.shape[0]
    cb = cblk_of(cin)
    nck = (cin + cb - 1) // cb
    g = G[:, idx, :]
    T = g.shape[1]
    out = torch.zeros((cout_pad_of(Co), T, nck * cb), dtype=torch.bfloat16, device=G.device)
    out[:Co, :, :cin] = g
    return out.view(out.shape[0], T * nck * cb)


def pack_spec(name, src, rows, cols, taps, s_r0, s_c0, s_t=1, rows_pad=None, cols_pad=None, R0=None, s_r1=0, C0=None,
              s_c1=0, f32=False, index=None):
    """One destination of the native weight re-pack (include/jvae_b200.h: jvae_pack_job):
    dst[r][t][c] = src[(r // R0) * s_r1 + (r % R0) * s_r0 + taps[t] * s_t + (c // C0) * s_c1 + (c % C0) * s_c0], zero where
    r >= rows or c >= cols; dst is (rows_pad, T * cols_pad) dense.  `src` names the parameter ('w' or 'b')."""
    return dict(name=name, index=index, src=src, rows=rows, rows_pad=rows_pad or rows, R0=R0 or rows, s_r1=s_r1, s_r0=s_r0,
                taps=list(taps), s_t=s_t, cols=cols, cols_pad=cols_pad or cols, C0=C0 or cols, s_c1=s_c1, s_c0=s_c0, f32=f32)


def gather_spec(name, index, Co, cin, idx, s_row, s_col):
    """spec of pack_gather_weights(G, idx, cin) with G[co, t, ci] = w.flat[co * s_row + t + ci * s_col]"""
    cb = cblk_of(cin)
    nck = (cin + cb - 1) // cb
    return pack_spec(name, 'w', Co, cin, idx, s_row, s_col, rows_pad=cout_pad_of(Co), cols_pad=nck * cb, index=index)


def run_pack_spec(sp, src):
    """torch execution of one pack job (any device): the definition the CUDA kernel is tested against"""
    flat = src.detach().reshape(-1).float()
    r = torch.arange(sp['rows_pad'], device=flat.device)
    c = torch.arange(sp['cols_pad'], device=flat.device)
    t = torch.tensor(sp['taps'], device=flat.device, dtype=torch.long)
    ro = torch.div(r, sp['R0'], rounding_mode='floor') * sp['s_r1'] + (r % sp['R0']) * sp['s_r0']
    co = torch.div(c, sp['C0'], rounding_mode='floor') * sp['s_c1'] + (c % sp['C0']) * sp['s_c0']
    idx = ro[:, None, None] + (t * sp['s_t'])[None, :, None] + co[None, None, :]
    ok = (r < sp['rows'])[:, None, None] & (c < sp['cols'])[None, None, :]
    ok = ok.expand_as(idx)
    out = torch.zeros(idx.shape, dtype=torch.float32, device=flat.device)
    out[ok] = flat[idx[ok]]
    out = out.reshape(sp['rows_pad'], len(sp['taps']) * sp['cols_pad'])
    return out if sp['f32'] else out.to(torch.bfloat16)


class PackPlan:
    """Every bf16 weight arrangement of a stack's convolutions, rebuilt by ONE kernel launch (csrc/pack.cu) whenever
    the parameters changed: optimizer step (engine.PARAM_EPOCH), in-place torch writes (_version), re-pointed storage
    (data_ptr: Optimizer._flatten, .to(device)).  The reference reads its live nn.Parameters in every step
    (cvae.py:2424-2461); this is that read."""

    def __init__(self, steps):
        self.steps = [s for s in steps if s.pack_specs()]
        self.params = []
        for s in self.steps:
            self.params += [p for p in (s.conv.weight, s.conv.bias) if p is not None]
        self.key = None
        self.epoch = -1
        self.ptrs = None
        self.jobs_dev = self.taps_dev = None
        self.n_jobs = self.blocks = 0

    def _build(self):
        jobs, taps = [], []
        first = 0
        for s in self.steps:
            w = s.conv.weight
            assert w.dtype == torch.float32 and w.is_contiguous(), 'conv weights must be dense fp32'
            pk = {'b': s.conv.bias.detach() if s.conv.bias is not None else None}
            for sp in s.pack_specs():
                src = w if sp['src'] == 'w' else s.conv.bias
                T = len(sp['taps'])
                dst = torch.empty((sp['rows_pad'], T * sp['cols_pad']), dtype=torch.float32 if sp['f32'] else torch.bfloat16,
                                  device=w.device)
                assert sp['cols_pad'] % 8 == 0 and dst.data_ptr() % 16 == 0
                j = nat.PackJob(src=src.data_ptr(), dst=dst.data_ptr(), s_r1=sp['s_r1'], s_r0=sp['s_r0'], s_t=sp['s_t'],
                                s_c1=sp['s_c1'], s_c0=sp['s_c0'], rows=sp['rows'], rows_pad=sp['rows_pad'], R0=sp['R0'], T=T,
                                tap_off=len(taps), cols=sp['cols'], cols_pad=sp['cols_pad'], C0=sp['C0'],
                                dst_f32=int(sp['f32']), first_block=first)
                first += nat.pack_job_blocks(sp['rows_pad'], T, sp['cols_pad'])
                taps += sp['taps']
                jobs.append(j)
                if sp['index'] is None:
                    pk[sp['name']] = s.pack_view(sp, dst)
                else:
                    pk.setdefault(sp['name'], []).append(dst)
            s._pk = pk
        import ctypes
        arr = (nat.PackJob * len(jobs))(*jobs)
        dev = self.steps[0].conv.weight.device
        raw = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone()
        self.jobs_dev = raw.to(dev)
        self.taps_dev = torch.tensor(taps, dtype=torch.int32).to(dev)
        self.n_jobs, self.blocks = len(jobs), first

    def ensure(self):
        if not self.steps:
            return
        ptrs = tuple(p.data_ptr() for p in self.params)
        key = (engine.PARAM_EPOCH[0], ptrs) + tuple(p._version for p in self.params)
        self.epoch = engine.PARAM_EPOCH[0]
        if key == self.key:
            return
        if ptrs != self.ptrs:
            self._build()
            self.ptrs = ptrs
        nat.pack_weights(self.jobs_dev, self.n_jobs, self.taps_dev, self.blocks)
        self.key = key


def _live_grad(p, like):
    """the Parameter's own dense fp32 .grad (the optimizer's flat gradient buffer, zeroed by zero_grad) when the native
    kernels can accumulate into it directly; autograd then receives None for that parameter"""
    if K is not NativeKernels or p is None or p.grad is None:
        return None
    g = p.grad
    return g if (g.dtype == torch.float32 and g.is_contiguous() and g.device == like.device) else None


# ------------------------------------------------------------------------------------------------ steps
class ConvStep:
    """Conv2d | ConvTranspose2d [+ BatchNorm2d] [+ activation]"""

    def __init__(self, conv, bn, act, in_shape, final_dense):
        self.conv, self.bn, self.act = conv, bn, act
        self.transposed = isinstance(conv, nn.ConvTranspose2d)
        k, p, s = conv.kernel_size[0], conv.padding[0], conv.stride[0]
        assert conv.kernel_size[0] == conv.kernel_size[1] and conv.padding[0] == conv.padding[1] \
            and conv.stride[0] == conv.stride[1], 'square kernels / symmetric geometry only'
        if conv.dilation != (1, 1) or conv.groups != 1:
            raise NotImplementedError('dilated / grouped convolutions')
        if k * k > 64:
            raise NotImplementedError('kernels larger than 8x8')
        self.k, self.p, self.s = k, p, s
        Ci, H, W = in_shape
        self.Ci, self.H, self.W = Ci, H, W
        self.Co = conv.out_channels
        if self.transposed:
            op = conv.output_padding[0]
            self.Ho, self.Wo = (H - 1) * s - 2 * p + k + op, (W - 1) * s - 2 * p + k + op
        else:
            if s > 2:
                raise NotImplementedError('convolution stride > 2')
            self.Ho, self.Wo = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
        self.out_shape = (self.Co, self.Ho, self.Wo)
        self.gemm1x1 = (self.transposed and H == 1 and W == 1 and p == 0 and conv.output_padding[0] == 0
                        and self.Co % 8 == 0)
        self.dense_small = DENSE_SMALL and (not self.transposed) and (not self.gemm1x1) and s == 1 and k > 1 and 2 * p == k - 1 \
            and H * W <= 4 and Ci % 8 == 0 and self.Co % 8 == 0 and not final_dense
        if self.dense_small:      # (output pixel q, input pixel r) -> filter tap (ry - qy + p, rx - qx + p) when inside the window
            self.dense_pairs = [(qy * W + qx, ry * W + rx, ry - qy + p, rx - qx + p)
                                for qy in range(H) for qx in range(W) for ry in range(H) for rx in range(W)
                                if 0 <= ry - qy + p < k and 0 <= rx - qx + p < k]
        self.final_dense = final_dense
        self.ld_y = r8(self.Co) if (bn is not None or not final_dense) else self.Co
        self.ld_a = self.Co if final_dense else r8(self.Co)
        if self.gemm1x1:
            self.fwd_ops = self.dgrad_ops = None
        elif self.transposed:
            if s > 2:
                raise NotImplementedError('transposed convolution stride > 2 (weight gradient kernel)')
            self.fwd_ops = deconv_form(k, p, s, self.Ho, self.Wo)
            self.dgrad_ops = conv_form(k, p, s, H, W)
        else:
            self.fwd_ops = conv_form(k, p, s, self.Ho, self.Wo)
            self.dgrad_ops = deconv_form(k, p, s, H, W, allow_empty=True)
        # stride-2 ConvTranspose2d with an even output: the four sub-pixel phases share their grid and run as ONE launch
        # (jvae_conv_subpixel_gemm) on a weight matrix that lists the taps phase by phase; the per-phase launches stay as the
        # fallback for geometries the merged kernel does not take
        self.merged_fwd = (not self.gemm1x1) and self.transposed and s == 2 and len(self.fwd_ops) == 4 and \
            len({(op['Hq'], op['Wq']) for op in self.fwd_ops}) == 1
        if self.merged_fwd:
            self.fwd_all_idx = [i for op in self.fwd_ops for i in op['idx']]
        # phases of the data gradient that no tap reaches (kernel < stride) stay zero
        self.dgrad_sparse = (not self.gemm1x1) and (not self.transposed) and len(self.dgrad_ops) < min(s, H) * min(s, W)
        self.wgrad_taps = [(i - p, j - p) for i in range(k) for j in range(k)]
        # stride-1 Conv2d with few output channels (the image head, 32 -> 3): exchange the roles in the weight-gradient kernel
        # (grid tensor = x, gathered tensor = dy, taps negated): the kernel stacks taps of the GATHERED tensor along M, so the
        # narrow tensor packs twice as many taps per MMA (sum_p dy[p] x[p + t] = sum_q x[q] dy[q - t])
        self.wgrad_swapped = (not self.transposed) and s == 1 and (self.Ho, self.Wo) == (H, W) and \
            cblk_of(min(self.Co, 64)) < cblk_of(min(Ci, 64))
        self.wgrad_taps_neg = [(-a, -b) for a, b in self.wgrad_taps]
        # narrow image heads (32 -> 3, k5): the k x k 'same' convolution runs as a 1 x k convolution to k * Co channels on the
        # tensor cores followed by a vertical shift-and-add (include/jvae_b200.h: jvae_vsum_rows / jvae_vstack_rows): k taps
        # instead of k^2 in the forward, data-gradient and weight-gradient kernels
        # k >= 5: with a 3 x 3 head (c4's ivgg) the 9 -> 3 tap reduction does not pay for the two row passes (measured: -0.24 ms)
        self.separable = (not self.transposed) and (not self.gemm1x1) and s == 1 and k >= 5 and 2 * p == k - 1 and \
            self.Co <= 4 and k * self.Co <= 16 and W >= 8 and os.environ.get('JVAE_CONV_SEPARABLE', '1') != '0'
        if self.separable:
            self.sep_C, self.sep_ld = k * self.Co, r8(k * self.Co)
            self.sep_fwd_taps = [(0, j - p) for j in range(k)]
            self.sep_bwd_taps = [(0, p - j) for j in range(k)]
        self._packed = None
        self._packed_folded = None
        self._ctaps = {}

    def params(self):
        ps = [self.conv.weight, self.conv.bias]
        if self.bn is not None:
            ps += [self.bn.weight, self.bn.bias]
        return ps

    def _taps(self, key, taps):
        c = self._ctaps.get(key)
        if c is None:
            c = self._ctaps[key] = K.taps_arg(taps)
        return c

    def pack_specs(self):
        """jobs of the native re-pack for the training-mode (unfolded) weights: the same arrangements _pack() builds with
        torch ops (tests/test_conv_engine_cpu.py checks them against each other); [] when this layer keeps the torch path"""
        if self.dense_small:
            return []
        kk, k, Co, Ci = self.k * self.k, self.k, self.Co, self.Ci
        if self.gemm1x1:      # W (Ci, Co, k, k): Bm[(yx, co)][ci] = W[ci][co][yx]; bias repeated per output pixel
            sp = [pack_spec('bm', 'w', kk * Co, Ci, [0], kk, Co * kk, R0=Co, s_r1=1, cols_pad=r8(Ci))]
            if self.conv.bias is not None:
                sp.append(pack_spec('bias', 'b', kk, Co, [0], 0, 1, f32=True))
            return sp
        # strides of W.flat for (output channel, input channel); the tap index has stride 1 in both layouts
        s_co, s_ci = (kk, Co * kk) if self.transposed else (Ci * kk, kk)
        sp = [gather_spec('fwd', i, Co, Ci, op['idx'], s_co, s_ci) for i, op in enumerate(self.fwd_ops)]
        sp += [gather_spec('bwd', i, Ci, Co, op['idx'], s_ci, s_co) for i, op in enumerate(self.dgrad_ops)]
        if self.merged_fwd:
            sp.append(gather_spec('fwd_all', None, Co, Ci, self.fwd_all_idx, s_co, s_ci))
        if self.separable:    # rows (ky, co) of the 1 x k kernel over kx taps; and [ci][kx][(ky, co)] for the data gradient
            cb = cblk_of(Ci)
            sp.append(pack_spec('sep_fwd', 'w', k * Co, Ci, range(k), s_co, s_ci, R0=Co, s_r1=k,
                                rows_pad=cout_pad_of(k * Co), cols_pad=((Ci + cb - 1) // cb) * cb))
            cb = cblk_of(k * Co)
            sp.append(pack_spec('sep_bwd', 'w', Ci, k * Co, range(k), s_ci, s_co, C0=Co, s_c1=k,
                                rows_pad=cout_pad_of(Ci), cols_pad=((k * Co + cb - 1) // cb) * cb))
        return sp

    def pack_view(self, sp, dst):
        if sp['name'] == 'bm':
            return dst[:, :self.Ci]
        if sp['name'] == 'bias':
            return dst.view(-1)
        return dst

    def _pack(self, fold_bn=False, want_bwd=None):
        """bf16 weight arrangements, refreshed when the Parameter changes (optimizer step / load_state_dict / in-place
        writes).  Training-mode weights on the GPU come from the stack's PackPlan (one native launch per stack and step);
        this torch formulation serves the BatchNorm-folded inference weights, the opt-in dense form and the CPU emulation.
        fold_bn (inference with running statistics): BatchNorm is folded into the weights and the bias, so the layer is
        ONE kernel: W' = W * gamma * rstd, b' = (b - mean) * gamma * rstd + beta."""
        w = self.conv.weight
        if not fold_bn and K is NativeKernels and not self.dense_small:
            plan = getattr(self, 'plan', None)
            if plan is None:                      # a step used outside a ConvStack
                plan = self.plan = PackPlan([self])
            if plan.epoch != engine.PARAM_EPOCH[0] or plan.key is None:      # full check at the stack's entry points
                plan.ensure()
            return self._pk
        key = (engine.PARAM_EPOCH[0], w._version, w.device, w.data_ptr())
        if self.conv.bias is not None:
            key += (self.conv.bias._version,)
        slot = '_packed'
        if fold_bn:
            bn = self.bn
            key += (engine.STATS_EPOCH[0],)
            key += tuple(t._version for t in (bn.running_mean, bn.running_var) if t is not None)
            key += tuple(t._version for t in (bn.weight, bn.bias) if t is not None)
            slot = '_packed_folded'
        hit = getattr(self, slot, None)
        if want_bwd is None:      # folded data-gradient weights are only needed for input gradients in eval mode (ODIN)
            want_bwd = not fold_bn
        if hit is not None and hit[0] == key and (not want_bwd or self.gemm1x1 or 'bwd' in hit[1]):
            return hit[1]
        wd = w.detach().float()
        kk = self.k * self.k
        d = {}
        b0 = self.conv.bias.detach().float() if self.conv.bias is not None else None
        if fold_bn:
            scale = (bn.running_var.float() + bn.eps).rsqrt()
            if bn.affine:
                scale = scale * bn.weight.detach().float()
            shift = -bn.running_mean.float() * scale
            if bn.affine:
                shift = shift + bn.bias.detach().float()
            wd = wd * (scale.view(1, -1, 1, 1) if self.transposed else scale.view(-1, 1, 1, 1))
            b0 = shift if b0 is None else b0 * scale + shift
        d['b'] = b0
        if self.gemm1x1:
            # Bm[(y, x, co)][ci] = W[ci][co][y][x]
            d['bm'] = wd.permute(2, 3, 1, 0).reshape(kk * self.Co, self.Ci).to(torch.bfloat16).contiguous()
            if self.Ci % 8:
                t = torch.zeros((kk * self.Co, r8(self.Ci)), dtype=torch.bfloat16, device=w.device)
                t[:, :self.Ci] = d['bm']
                d['bm'] = t[:, :self.Ci]
            d['bias'] = b0.repeat(kk).contiguous() if b0 is not None else None
        else:
            if self.transposed:     # W (Ci, Co, k, k)
                g_f = wd.permute(1, 2, 3, 0).reshape(self.Co, kk, self.Ci)
                g_b = wd.permute(0, 2, 3, 1).reshape(self.Ci, kk, self.Co)
            else:                   # W (Co, Ci, k, k)
                g_f = wd.permute(0, 2, 3, 1).reshape(self.Co, kk, self.Ci)
                g_b = wd.permute(1, 2, 3, 0).reshape(self.Ci, kk, self.Co)
            d['fwd'] = [pack_gather_weights(g_f, op['idx'], self.Ci) for op in self.fwd_ops]
            if self.merged_fwd:
                d['fwd_all'] = pack_gather_weights(g_f, self.fwd_all_idx, self.Ci)
            if self.dense_small:     # W_eff[(q, co), (r, ci)] = W[co][ci][tap(q, r)]
                hw = self.H * self.W
                weff = torch.zeros((hw, self.Co, hw, self.Ci), dtype=torch.float32, device=w.device)
                for q, r, ty, tx in self.dense_pairs:
                    weff[q, :, r, :] = wd[:, :, ty, tx]
                d['dense'] = weff.view(hw * self.Co, hw * self.Ci).to(torch.bfloat16).contiguous()
                d['dense_bias'] = b0.repeat(hw).contiguous() if b0 is not None else None
            if self.separable:      # wd (Co, Ci, ky, kx): rows (ky, co) of the 1 x k kernel, and its transpose for the data gradient
                kq = self.k
                d['sep_fwd'] = pack_gather_weights(wd.permute(2, 0, 3, 1).reshape(kq * self.Co, kq, self.Ci),
                                                   list(range(kq)), self.Ci)
                d['sep_bwd'] = pack_gather_weights(wd.permute(1, 3, 2, 0).reshape(self.Ci, kq, kq * self.Co),
                                                   list(range(kq)), kq * self.Co)
            if want_bwd:
                d['bwd'] = [pack_gather_weights(g_b, op['idx'], self.Co) for op in self.dgrad_ops]
        setattr(self, slot, (key, d))
        return d

    # ---- forward
    def forward(self, x, st, training):
        N = x.shape[0]
        bn = self.bn
        bn_train = bn is not None and (training or not bn.track_running_stats)
        if bn is not None and not bn_train:
            return self._forward_folded(x, st)
        pk = self._pack()
        bias = self.conv.bias.detach() if self.conv.bias is not None else None
        fused_act = self.act if bn is None else 0
        y = st.pop('out', None)          # a channel slice of a dense block's buffer (DenseBlockStep)
        if y is None:
            y = K.empty((N, self.Ho, self.Wo, self.ld_y), x)
        else:
            assert bn is None and not (self.gemm1x1 or self.dense_small or self.separable or self.merged_fwd)
        stats = (st.pop('stats_buf', None) if bn_train else None)
        if bn_train and stats is None:
            stats = K.zeros((2, self.Co), x, torch.float64)
        if self.gemm1x1:
            kk = self.k * self.k
            a2 = x.view(N, x.shape[-1])
            K.gemm(nat.GEMM_NT, N, kk * self.Co, self.Ci, a2, pk['bm'], bias=pk['bias'], act=fused_act,
                   out_bf16=y.view(N, kk * self.Co))
            if bn_train:
                K.bn_stats(y, N * kk, self.Co, self.ld_y, stats)
        elif self.dense_small:
            hw = self.H * self.W
            K.gemm(nat.GEMM_NT, N, hw * self.Co, hw * self.Ci, x.view(N, hw * self.Ci), pk['dense'], bias=pk['dense_bias'],
                   act=fused_act, out_bf16=y.view(N, hw * self.Co))
            if bn_train:
                K.bn_stats(y, N * hw, self.Co, self.ld_y, stats)
        elif self.separable and not SEP_FWD_DIRECT:
            self._sep_forward(x, pk, bias, fused_act, stats, y)
        elif not self._merged_forward(x, pk, y, bias, fused_act, stats):
            for i, (op, wm) in enumerate(zip(self.fwd_ops, pk['fwd'])):
                K.gather(x, self.Ci, wm, wm.shape[0], self._taps(('f', i), op['taps']), op['in_stride'], op['Hq'], op['Wq'],
                         y, self.Co, op['out_s'], op['out_o'], bias, fused_act, stats)
        st['x'] = x
        if bn is None:
            st['a'] = y
            return y
        P = N * self.Ho * self.Wo
        a = K.empty((N, self.Ho, self.Wo, self.ld_a), x)
        save = K.empty((2, self.Co), x, torch.float32) if bn_train else None
        track = bn.track_running_stats and training
        K.bn_apply_fwd(y, P, self.Co, self.ld_y, stats, bn.weight.detach() if bn.affine else None,
                       bn.bias.detach() if bn.affine else None, bn.eps, bn.momentum if bn.momentum is not None else 0.1,
                       bn.running_mean if track or not bn_train else None, bn.running_var if track or not bn_train else None,
                       bn.num_batches_tracked if track else None, bn_train, self.act, a, self.ld_a, save)
        if track:
            engine.bump_stats()      # the kernel wrote running_mean / running_var behind the version counters
        st['y'], st['save'], st['bn_train'] = y, save, bn_train
        return a

    def _merged_forward(self, x, pk, out, bias, act, stats):
        """the four sub-pixel phases of a stride-2 ConvTranspose2d in one launch; False: run them one by one"""
        if not self.merged_fwd:
            return False
        ph = self._ctaps.get('fa')
        if ph is None:
            ph = self._ctaps['fa'] = K.phases_arg(self.fwd_ops)
        wm = pk['fwd_all']
        op = self.fwd_ops[0]
        return K.subpixel(x, self.Ci, wm, wm.shape[0], ph, op['Hq'], op['Wq'], out, self.Co, self.s, bias, act, stats)

    def _sep_forward(self, x, pk, bias, act, stats, out):
        """1 x k convolution to k * Co channels (tensor cores), then the vertical shift-and-add with bias / activation / stats.
        T stays fp32: the k vertical taps of an output pixel cancel, and rounding them to bf16 first costs the gradients of the
        head and of the layer under it an order of magnitude (measured: 25 % instead of 1.8 % on the head's weight gradient)."""
        N = x.shape[0]
        T = K.empty((N, self.H, self.W, self.sep_ld), x, torch.float32)
        wm = pk['sep_fwd']
        K.gather(x, self.Ci, wm, wm.shape[0], self._taps('sf', self.sep_fwd_taps), 1, self.H, self.W, T, self.sep_C, (1, 1),
                 (0, 0), None, nat.OUT_F32, None)
        K.vsum_rows(T, self.sep_ld, N, self.H, self.W, self.k, self.p, self.Co, bias, act | nat.IN_F32, stats, out,
                    out.shape[-1])

    def _forward_folded(self, x, st):
        """inference: conv + folded BatchNorm + activation in one kernel, no intermediate tensor"""
        N = x.shape[0]
        pk = self._pack(fold_bn=True)
        a = K.empty((N, self.Ho, self.Wo, self.ld_a), x)
        if self.gemm1x1:
            kk = self.k * self.k
            K.gemm(nat.GEMM_NT, N, kk * self.Co, self.Ci, x.view(N, x.shape[-1]), pk['bm'], bias=pk['bias'], act=self.act,
                   out_bf16=a.view(N, kk * self.Co))
        elif self.dense_small:
            hw = self.H * self.W
            K.gemm(nat.GEMM_NT, N, hw * self.Co, hw * self.Ci, x.view(N, hw * self.Ci), pk['dense'], bias=pk['dense_bias'],
                   act=self.act, out_bf16=a.view(N, hw * self.Co))
        elif self.separable and not SEP_FWD_DIRECT:
            self._sep_forward(x, pk, pk['b'], self.act, None, a)
        elif not self._merged_forward(x, pk, a, pk['b'], self.act, None):
            for i, (op, wm) in enumerate(zip(self.fwd_ops, pk['fwd'])):
                K.gather(x, self.Ci, wm, wm.shape[0], self._taps(('f', i), op['taps']), op['in_stride'], op['Hq'], op['Wq'],
                         a, self.Co, op['out_s'], op['out_o'], pk['b'], self.act, None)
        st['x'], st['a'], st['bn_train'], st['folded'] = x, a, False, True
        return a

    # ---- backward: da = dL/d(output) NHWC bf16 -> (dx or None, [param grads])
    def backward(self, da, st, need_dx, prev_bn=None):
        """prev_bn: dict describing the previous layer's train-mode BatchNorm (y, ld_y, save, gamma, beta, act, sums): its
        backward reduction is folded into this layer's data-gradient kernel when the kernel supports it; prev_bn['done']
        then tells that layer to skip its own reduction pass."""
        x = st['x']
        N = x.shape[0]
        P = N * self.Ho * self.Wo
        bn = self.bn
        grads = {}
        folded = bool(st.get('folded'))
        if folded:
            # eval-mode BatchNorm is a per-channel affine map folded into the weights: a = act(conv'(x)).  Only the input
            # gradient is produced (what ODIN differentiates, cvae.py:1648-1656); the parameters get no gradient here.
            a = st['a']
            if self.act == 0 and da.shape[-1] % 8 == 0:
                dy = da
            else:
                dy = K.zeros((N, self.Ho, self.Wo, r8(self.Co)), x, torch.bfloat16) if r8(self.Co) != self.Co \
                    else K.empty((N, self.Ho, self.Wo, self.Co), x)
                K.act_bwd(da, da.shape[-1], a, a.shape[-1], P, self.Co, self.act, dy, dy.shape[-1], None)
        elif bn is not None:
            y = st['y']
            dy = K.empty(y.shape, x)
            pre = st.get('bn_sums')            # produced by the next layer's data-gradient kernel
            sums = pre if pre is not None else K.empty((2, self.Co), x, torch.float64)
            dg = db = lg = lb = None
            if bn.affine:
                lg, lb = _live_grad(bn.weight, x), _live_grad(bn.bias, x)
                dg = lg if lg is not None else K.zeros((self.Co,), x)
                db = lb if lb is not None else K.zeros((self.Co,), x)
            K.bn_bwd(da, da.shape[-1], y, self.ld_y, P, self.Co, st['save'], bn.weight.detach() if bn.affine else None,
                     bn.bias.detach() if bn.affine else None, self.act, sums, dy, self.ld_y, dg, db,
                     **({'skip_reduce': True} if pre is not None else {}))
            grads['bn_w'], grads['bn_b'] = (None if lg is not None else dg), (None if lb is not None else db)
            # the bias of a convolution followed by train-mode BatchNorm has an exactly zero gradient
            # (BN subtracts the batch mean); the reference's autograd returns rounding noise here
            grads['b'] = K.zeros((self.Co,), x) if (self.conv.bias is not None and
                                                     _live_grad(self.conv.bias, x) is None) else None
        else:
            lbias = _live_grad(self.conv.bias, x)
            dbias = lbias if lbias is not None else (K.zeros((self.Co,), x) if self.conv.bias is not None else None)
            if self.act == 0 and da.shape[-1] % 8 == 0:
                dy = da
                if dbias is not None:
                    K.act_bwd(da, da.shape[-1], None, 0, P, self.Co, 0, None, 0, dbias)
            else:
                a = st['a']
                dy = K.zeros((N, self.Ho, self.Wo, r8(self.Co)), x, torch.bfloat16) if r8(self.Co) != self.Co \
                    else K.empty((N, self.Ho, self.Wo, self.Co), x)
                K.act_bwd(da, da.shape[-1], a, a.shape[-1], P, self.Co, self.act, dy, dy.shape[-1], dbias)
            grads['b'] = None if lbias is not None else dbias
        pk = self._pack(fold_bn=folded, want_bwd=True)
        kk = self.k * self.k
        dx = None
        if folded:
            grads = {'w': None, 'b': None, 'bn_w': None, 'bn_b': None}
        if self.gemm1x1:
            dy2 = dy.view(N, kk * self.Co)
            x2 = x.view(N, x.shape[-1])
            if not folded:
                dbm = K.empty((kk * self.Co, self.Ci), x, torch.float32)
                K.gemm(nat.GEMM_TN, kk * self.Co, self.Ci, N, dy2, x2, out_f32=dbm)
                grads['w'] = dbm.view(self.k, self.k, self.Co, self.Ci).permute(3, 2, 0, 1).contiguous()
            if need_dx:
                ldx = x.shape[-1]
                if ldx == self.Ci:
                    dx = K.empty(x.shape, x)
                    K.gemm(nat.GEMM_NN, N, self.Ci, kk * self.Co, dy2, pk['bm'], out_bf16=dx.view(N, ldx))
                else:
                    tmp = K.empty((N, self.Ci), x, torch.float32)
                    K.gemm(nat.GEMM_NN, N, self.Ci, kk * self.Co, dy2, pk['bm'], out_f32=tmp)
                    dx = K.zeros(x.shape, x, torch.bfloat16)
                    dx.view(N, ldx)[:, :self.Ci] = tmp
        elif self.dense_small:
            hw = self.H * self.W
            dy2, x2 = dy.view(N, hw * self.Co), x.view(N, hw * self.Ci)
            if not folded:
                dweff = K.empty((hw * self.Co, hw * self.Ci), x, torch.float32)
                K.gemm(nat.GEMM_TN, hw * self.Co, hw * self.Ci, N, dy2, x2, out_f32=dweff)
                dw4 = dweff.view(hw, self.Co, hw, self.Ci)
                w = self.conv.weight
                live = _live_grad(w, x)
                dw = live if live is not None else K.zeros(tuple(w.shape), x)
                for q, r, ty, tx in self.dense_pairs:          # fold the (pixel, pixel) blocks back onto their taps
                    dw[:, :, ty, tx] += dw4[q, :, r, :]
                grads['w'] = None if live is not None else dw
            if need_dx:
                dx = K.empty(x.shape, x)
                K.gemm(nat.GEMM_NN, N, hw * self.Ci, hw * self.Co, dy2, pk['dense'], out_bf16=dx.view(N, hw * self.Ci))
        elif self.separable:
            kq = self.k
            U = K.empty((N, self.H, self.W, self.sep_ld), x)      # gradient of the 1 x k stage's output
            K.vstack_rows(dy, dy.shape[-1], N, self.H, self.W, kq, self.p, self.Co, U, self.sep_ld)
            if not folded:
                dwa = K.zeros((self.sep_C, self.Ci, kq), x)        # rows (ky, co), then ci, kx
                if cblk_of(self.sep_C) < cblk_of(min(self.Ci, 64)):
                    K.wgrad(x, self.Ci, U, self.sep_C, self._taps('sb', self.sep_bwd_taps), 1, dwa, swapped=True)
                else:
                    K.wgrad(U, self.sep_C, x, self.Ci, self._taps('sf', self.sep_fwd_taps), 1, dwa)
                upd = dwa.view(kq, self.Co, self.Ci, kq).permute(1, 2, 0, 3)      # -> (co, ci, ky, kx)
                live = _live_grad(self.conv.weight, x)
                if live is not None:
                    live.add_(upd)
                grads['w'] = None if live is not None else upd.contiguous()
            if need_dx:
                dx = K.empty(x.shape, x)
                wm = pk['sep_bwd']
                K.gather(U, self.sep_C, wm, wm.shape[0], self._taps('sb', self.sep_bwd_taps), 1, self.H, self.W, dx, self.Ci,
                         (1, 1), (0, 0), None, 0, None)
        else:
            # the kernel accumulates straight into the torch layout; when the Parameter already owns a dense fp32 .grad
            # (the optimizer's flat gradient buffer, zeroed by zero_grad) it accumulates THERE and autograd gets None
            w = self.conv.weight
            if not folded:
                live = _live_grad(w, x)
                dw = live if live is not None else K.zeros(tuple(w.shape), x)
                if self.transposed:      # grid tensor = x, gathered tensor = dy   -> W.grad (Ci, Co, k, k)
                    K.wgrad(x, self.Ci, dy, self.Co, self._taps('w', self.wgrad_taps), self.s, dw.view(self.Ci, self.Co, kk))
                elif self.wgrad_swapped:  # grid tensor = x, gathered tensor = dy, negated taps -> W.grad (Co, Ci, k, k)
                    K.wgrad(x, self.Ci, dy, self.Co, self._taps('wn', self.wgrad_taps_neg), 1, dw.view(self.Co, self.Ci, kk),
                            swapped=True)
                else:                    # grid tensor = dy, gathered tensor = x   -> W.grad (Co, Ci, k, k)
                    K.wgrad(dy, self.Co, x, self.Ci, self._taps('w', self.wgrad_taps), self.s, dw.view(self.Co, self.Ci, kk))
                grads['w'] = None if live is not None else dw
            if need_dx:
                dx = K.zeros(x.shape, x, torch.bfloat16) if self.dgrad_sparse else K.empty(x.shape, x)
                fuse = FUSE_BN_REDUCE and prev_bn is not None and K is NativeKernels and \
                    prev_bn['y'].shape[:3] == dx.shape[:3]
                sums_prev = K.zeros((2, self.Ci), x, torch.float64) if fuse else None
                done = fuse
                for i, (op, wm) in enumerate(zip(self.dgrad_ops, pk['bwd'])):
                    r = K.gather(dy, self.Co, wm, wm.shape[0], self._taps(('b', i), op['taps']), op['in_stride'], op['Hq'],
                                 op['Wq'], dx, self.Ci, op['out_s'], op['out_o'], None, 0, sums_prev,
                                 **({'bn': prev_bn} if fuse else {}))
                    done = done and bool(r)
                if fuse and done:
                    prev_bn['sums'] = sums_prev
        out = [grads['w'], grads['b']]
        if bn is not None:
            out += [grads['bn_w'], grads['bn_b']]
        return dx, out


class PoolStep:
    """MaxPool2d(k, stride >= k, padding 0): non-overlapping windows (what the reference's 'M' tokens build)"""

    def __init__(self, mod, in_shape):
        ks = mod.kernel_size if isinstance(mod.kernel_size, int) else mod.kernel_size[0]
        stv = mod.stride if isinstance(mod.stride, int) else mod.stride[0]
        pad = mod.padding if isinstance(mod.padding, int) else mod.padding[0]
        if mod.ceil_mode or mod.dilation not in (1, (1, 1)) or 2 * pad > ks:
            raise NotImplementedError('MaxPool2d with ceil_mode / dilation has no native kernel')
        self.k, self.s, self.p = ks, stv, pad
        self.general = pad != 0 or stv < ks        # padded / overlapping windows (ResNet stem MaxPool2d(3, 2, 1))
        self.C, self.H, self.W = in_shape
        self.Ho, self.Wo = (self.H + 2 * pad - ks) // stv + 1, (self.W + 2 * pad - ks) // stv + 1
        self.out_shape = (self.C, self.Ho, self.Wo)

    def params(self):
        return []

    def forward(self, x, st, training):
        N, _, _, ld = x.shape
        out = st.pop('out', None)        # the first channels of a dense block's buffer (DenseBlockStep)
        if out is None:
            out = K.empty((N, self.Ho, self.Wo, ld), x)
        ldo = out.stride(2)
        if self.general:
            K.maxpool_pad_fwd(x, N, self.H, self.W, ld, ld, self.k, self.s, self.p, out, ldo)
        else:
            K.maxpool_fwd(x, N, self.H, self.W, ld, ld, self.k, self.s, out, ldo)      # padded channels are pooled as well
        st['x'] = x
        return out

    def backward(self, da, st, need_dx):
        if not need_dx:
            return None, []
        x = st['x']
        N, _, _, ld = x.shape
        dx = K.empty(x.shape, x)
        if self.general:
            K.maxpool_pad_bwd(x, N, self.H, self.W, ld, ld, self.k, self.s, self.p, da, da.shape[-1], dx, ld)
        else:
            K.maxpool_bwd(x, N, self.H, self.W, ld, ld, self.k, self.s, da, da.shape[-1], dx, ld)
        return dx, []


class AvgStep:
    """AvgPool2d(k) with stride k, or AdaptiveAvgPool2d(1) (k = H = W: the last layer of torchvision's ResNet features)"""

    def __init__(self, mod, in_shape):
        self.C, self.H, self.W = in_shape
        if isinstance(mod, nn.AdaptiveAvgPool2d):
            o = mod.output_size if isinstance(mod.output_size, (tuple, list)) else (mod.output_size, mod.output_size)
            if tuple(o) != (1, 1) or self.H != self.W:
                raise NotImplementedError('AdaptiveAvgPool2d other than (1, 1) on a square map has no native kernel')
            k = self.H
        else:
            k = mod.kernel_size if isinstance(mod.kernel_size, int) else mod.kernel_size[0]
            stv = mod.stride if isinstance(mod.stride, int) else mod.stride[0]
            pad = mod.padding if isinstance(mod.padding, int) else mod.padding[0]
            if stv != k or pad != 0 or self.H % k or self.W % k or mod.ceil_mode:
                raise NotImplementedError('AvgPool2d must tile the map (stride = kernel, no padding)')
        self.k = k
        self.out_shape = (self.C, self.H // k, self.W // k)

    def params(self):
        return []

    def forward(self, x, st, training):
        N, _, _, ld = x.shape
        out = st.pop('out', None)        # the first channels of a dense block's buffer (DenseBlockStep)
        if out is None:
            out = K.empty((N, self.H // self.k, self.W // self.k, ld), x)
        K.avgpool(x, ld, out, out.stride(2), N, self.H, self.W, ld, self.k, False)
        st['ld'] = ld
        return out

    def backward(self, da, st, need_dx):
        if not need_dx:
            return None, []
        N, ld = da.shape[0], st['ld']
        dx = K.empty((N, self.H, self.W, ld), da)
        K.avgpool(da, da.shape[-1], dx, ld, N, self.H, self.W, ld, self.k, True)
        return dx, []


def is_residual_block(m):
    """torchvision.models.resnet.BasicBlock / Bottleneck (duck-typed: the package need not be imported here)"""
    return type(m).__name__ in ('BasicBlock', 'Bottleneck') and hasattr(m, 'conv1') and hasattr(m, 'downsample')


class ResidualStep:
    """out = relu(F(x) + shortcut(x)) with F = conv-bn-relu ... conv-bn (BasicBlock: 2 convs, Bottleneck: 3) and shortcut =
    identity or downsample = conv1x1-bn (torchvision/models/resnet.py; the reference wraps these models, conv.py:247-272)"""

    def __init__(self, block, in_shape):
        names = [n for n in ('conv1', 'conv2', 'conv3') if hasattr(block, n)]
        self.chain, shape = [], tuple(in_shape)
        for i, n in enumerate(names):
            conv, bn = getattr(block, n), getattr(block, 'bn' + n[-1])
            stp = ConvStep(conv, bn, 1 if i < len(names) - 1 else 0, shape, final_dense=False)
            self.chain.append(stp)
            shape = stp.out_shape
        self.ds = None
        if block.downsample is not None:
            ds = list(block.downsample)
            if len(ds) != 2 or not isinstance(ds[0], nn.Conv2d) or not isinstance(ds[1], nn.BatchNorm2d):
                raise NotImplementedError('residual shortcut other than conv1x1 + BatchNorm')
            self.ds = ConvStep(ds[0], ds[1], 0, tuple(in_shape), final_dense=False)
            if self.ds.out_shape != shape:
                raise NotImplementedError('shortcut / residual shape mismatch')
        elif tuple(in_shape) != shape:
            raise NotImplementedError('identity shortcut with a shape change')
        self.out_shape = shape

    def params(self):
        ps = [p for s in self.chain for p in s.params()]
        if self.ds is not None:
            ps += self.ds.params()
        return ps

    def forward(self, x, st, training):
        sts, t = [], x
        for s in self.chain:
            si = {}
            t = s.forward(t, si, training)
            sts.append(si)
        st_ds, idn = None, x
        if self.ds is not None:
            st_ds = {}
            idn = self.ds.forward(x, st_ds, training)
        N, Ho, Wo, ld = t.shape
        out = K.empty(t.shape, x)
        K.add_act(t, ld, idn, idn.shape[-1], N * Ho * Wo, ld, 1, out, ld)
        st['chain'], st['ds'], st['out'] = sts, st_ds, out
        return out

    def backward(self, da, st, need_dx):
        out = st['out']
        N, Ho, Wo, ld = out.shape
        P = N * Ho * Wo
        g = K.empty(out.shape, out)
        K.act_bwd(da, da.shape[-1], out, ld, P, ld, 1, g, ld, None)        # through the final ReLU: both branches see g
        grads, gi = [], g
        for idx in range(len(self.chain) - 1, -1, -1):
            gi, pg = self.chain[idx].backward(gi, st['chain'][idx], need_dx or idx > 0)
            grads = pg + grads
        dx = None
        if self.ds is not None:
            d2, pg = self.ds.backward(g, st['ds'], need_dx)
            grads = grads + pg
        else:
            d2 = g
        if need_dx:
            dx = K.empty(gi.shape, gi)
            Nn, H, W, ldx = gi.shape
            K.add_act(gi, ldx, d2, d2.shape[-1], Nn * H * W, ldx, 0, dx, ldx)
        return dx, grads


BN_MAX_C = 2048          # csrc/norm.cu: 8 channels per thread, NORM_MAX_THREADS = 256 threads per pixel row


def is_dense_block(m):
    """torchvision.models.densenet._DenseBlock: a ModuleDict of _DenseLayers (duck-typed like is_residual_block)"""
    return type(m).__name__ == '_DenseBlock' and isinstance(m, nn.ModuleDict)


def is_transition(m):
    """torchvision.models.densenet._Transition: norm -> relu -> conv1x1 -> AvgPool2d(2, 2)"""
    return type(m).__name__ == '_Transition' and isinstance(m, nn.Sequential)


def is_densenet_features(m):
    """the `features` Sequential of a torchvision DenseNet (stem, dense blocks, transitions, norm5)"""
    return isinstance(m, nn.Sequential) and any(is_dense_block(b) for b in m)


class DenseBlockStep:
    """torchvision _DenseBlock plus the pre-activation BatchNorm that reads its output (a transition's norm + relu, or norm5).

    The block lives in ONE NHWC bf16 buffer (N, H, W, C_total): the step before it (the stem's max pool, a transition's
    average pool) writes the block input into channels [0, C0), and layer l appends its `growth` channels at [Cin_l, Cin_l +
    growth) straight from conv2's epilogue, so nothing is ever concatenated.  The batch statistics of a channel are the same
    for every consumer (same data), so they are computed ONCE, when the channel is written, into one (2, C_total) f64 array;
    each consumer's norm1 (and the tail BatchNorm) normalises its channel prefix from there with its own gamma / beta /
    running statistics (jvae_bn_preact_fwd).  norm2 / relu2 are conv1's ConvStep epilogue as everywhere else.

    Backward: an fp32 accumulator of the buffer's shape collects every consumer's data gradient (jvae_bn_preact_bwd adds
    into its channel prefix).  Going through the layers in reverse, the slice of layer l is complete when layer l is reached
    (only later layers and the tail read it), so it is cast to bf16 (jvae_cast_f32_bf16_ld) and fed to conv2 / conv1's
    backward; channels [0, C0) at the end are the block input's gradient."""

    def __init__(self, block, tail_bn, tail_act, in_shape):
        C0, H, W = in_shape
        if tail_bn is None:
            raise NotImplementedError('a DenseNet block must be followed by a BatchNorm2d (transition norm or norm5)')
        self.H, self.W, self.C0 = H, W, C0
        self.layers = []
        c = C0
        for lay in block.values():
            if getattr(lay, 'drop_rate', 0) > 0 or getattr(lay, 'memory_efficient', False):
                raise NotImplementedError('DenseNet layers with drop_rate > 0 or memory_efficient=True have no native path')
            if c % 8:
                raise NotImplementedError(f'DenseNet channel offset {c} is not a multiple of 8: the block buffer needs '
                                          '16-byte aligned channel slices (growth rate and initial features multiples of 8)')
            n1, c1, n2, c2 = lay.norm1, lay.conv1, lay.norm2, lay.conv2
            if n1.num_features != c or c1.in_channels != c or c1.kernel_size != (1, 1) or c1.stride != (1, 1):
                raise NotImplementedError('_DenseLayer other than norm1 -> relu1 -> conv1x1 -> norm2 -> relu2 -> conv')
            s1 = ConvStep(c1, n2, 1, (c, H, W), final_dense=False)
            s2 = ConvStep(c2, None, 0, s1.out_shape, final_dense=False)
            if s2.out_shape[1:] != (H, W):
                raise NotImplementedError('DenseNet layer that changes the map size')
            g = c2.out_channels
            self.layers.append((n1, s1, s2, c, g))
            c += g
        if c % 8:
            raise NotImplementedError(f'DenseNet block width {c} is not a multiple of 8')
        if tail_bn.num_features != c:
            raise NotImplementedError('BatchNorm2d after a dense block with a different channel count')
        self.C = c
        # conv2's epilogue writes whole 16-channel output tiles: with a growth rate that is not a multiple of 16, the last
        # layer's zero-filled tile padding lands in 8 spare channels instead of the next pixel's first channels
        self.ld = c + (8 if any(g % 16 for *_, g in self.layers) else 0)
        self.tail_bn, self.tail_act = tail_bn, tail_act
        self.out_shape = (c, H, W)
        self.bns = [L[0] for L in self.layers] + [tail_bn] + [L[1].bn for L in self.layers]
        self.untracked = any(not b.track_running_stats for b in self.bns)

    def convs(self):
        return [s for L in self.layers for s in L[1:3]]

    def params(self):
        ps = []
        for n1, s1, s2, _, _ in self.layers:
            ps += [n1.weight, n1.bias] + s1.params() + s2.params()
        return ps + [self.tail_bn.weight, self.tail_bn.bias]

    def new_buffer(self, N, like):
        return K.empty((N, self.H, self.W, self.ld), like)

    @staticmethod
    def _pieces(C):
        """channel ranges of at most BN_MAX_C channels (a thread of the BatchNorm kernels owns 8 channels of a 256-thread row):
        densenet161's widest BatchNorms (2160, 2208 channels) run as two launches"""
        n = -(-C // BN_MAX_C)
        w = r8(-(-C // n))
        return [(c0, min(C, c0 + w)) for c0 in range(0, C, w)]

    def _bn_fwd(self, bn, buf, P, C, stats, bt, training, act, out, save):
        track = bn.track_running_stats and training
        sl = lambda t, a, b: None if t is None else t[a:b]
        for i, (a, b) in enumerate(self._pieces(C)):
            K.bn_preact_fwd(buf[..., a:], P, b - a, self.ld, sl(stats, a, None), self.C,
                            sl(bn.weight.detach() if bn.affine else None, a, b), sl(bn.bias.detach() if bn.affine else None, a, b),
                            bn.eps, bn.momentum if bn.momentum is not None else 0.1,
                            sl(bn.running_mean if track or not bt else None, a, b),
                            sl(bn.running_var if track or not bt else None, a, b),
                            bn.num_batches_tracked if track and i == 0 else None, bt, act, out[..., a:], out.stride(2),
                            None if save is None else save[i])
        if track:
            engine.bump_stats()      # the kernel wrote running_mean / running_var behind the version counters

    def forward(self, x, st, training):
        buf = st['buf']
        assert x.data_ptr() == buf.data_ptr(), 'the block input must be written into the block buffer'
        N, H, W = buf.shape[0], self.H, self.W
        P = N * H * W
        bt = training or self.untracked          # batch statistics (train mode, or BatchNorms without running statistics)
        stats = pool = None
        off = 2 * self.C
        if bt:      # the block statistics (2, C_total) and every norm2's (2, 4 growth) from ONE zeroed allocation
            pool = K.zeros((off + sum(2 * L[1].Co for L in self.layers),), buf, torch.float64)
            stats = pool[:off]
            K.bn_stats_ld(x, P, self.C0, self.ld, stats, self.C)
        saved = []
        for n1, s1, s2, c, g in self.layers:
            h = K.empty((N, H, W, c), buf)
            save = self._save(c, buf) if bt else None
            self._bn_fwd(n1, buf, P, c, stats, bt, training, 1, h, save)
            st1 = {}
            if bt:
                st1['stats_buf'] = pool[off:off + 2 * s1.Co].view(2, s1.Co)
                off += 2 * s1.Co
            a1 = s1.forward(h, st1, training)
            st2 = {'out': buf[..., c:c + g]}
            s2.forward(a1, st2, training)
            if bt:      # the new channels' statistics, once, for every later consumer
                K.bn_stats_ld(buf[..., c:], P, g, self.ld, stats[c:], self.C)
            saved.append((h, save, st1, st2))
        out = K.empty((N, H, W, self.C), buf)
        tsave = self._save(self.C, buf) if bt else None
        self._bn_fwd(self.tail_bn, buf, P, self.C, stats, bt, training, self.tail_act, out, tsave)
        st.update(layers=saved, tail_save=tsave, bn_train=bt)
        return out

    def _save(self, C, like):
        """the per-piece (2, width) mean / rstd of a train-mode pre-activation BatchNorm"""
        return [K.empty((2, b - a), like, torch.float32) for a, b in self._pieces(C)]

    def _bn_bwd(self, bn, da, buf, P, C, save, bt, act, G):
        dg = db = lg = lb = None
        if bt and bn.affine:
            lg, lb = _live_grad(bn.weight, buf), _live_grad(bn.bias, buf)
            dg = lg if lg is not None else K.zeros((C,), buf)
            db = lb if lb is not None else K.zeros((C,), buf)
        sl = lambda t, a, b: None if t is None else t[a:b]
        for i, (a, b) in enumerate(self._pieces(C)):
            sums = K.empty((2, b - a), buf, torch.float64) if bt else None
            K.bn_preact_bwd(da[..., a:], da.stride(2), buf[..., a:], self.ld, P, b - a, None if save is None else save[i],
                            sl(bn.weight.detach() if bn.affine else None, a, b), sl(bn.bias.detach() if bn.affine else None, a, b),
                            None if bt else bn.running_mean[a:b], None if bt else bn.running_var[a:b], bn.eps, bt, act, sums,
                            G[..., a:], self.ld, sl(dg, a, b), sl(db, a, b))
        return [None if lg is not None else dg, None if lb is not None else db]

    def backward(self, da, st, need_dx):
        buf, bt = st['buf'], st['bn_train']
        N, H, W = buf.shape[0], self.H, self.W
        P = N * H * W
        G = K.zeros((N, H, W, self.ld), buf, torch.float32)
        tail = self._bn_bwd(self.tail_bn, da, buf, P, self.C, st['tail_save'], bt, self.tail_act, G)
        grads = []
        for (n1, s1, s2, c, g), (h, save, st1, st2) in zip(reversed(self.layers), reversed(st['layers'])):
            d2 = K.empty((N, H, W, g), buf)
            K.cast_f32_bf16_ld(G[..., c:], self.ld, d2, g, P, g)       # complete: only later layers and the tail read it
            da1, pg2 = s2.backward(d2, st2, True)
            dh, pg1 = s1.backward(da1, st1, True)
            pgn = self._bn_bwd(n1, dh, buf, P, c, save, bt, 1, G)
            grads = pgn + pg1 + pg2 + grads
        dx = None
        if need_dx:
            dx = K.empty((N, H, W, self.C0), buf)
            K.cast_f32_bf16_ld(G, self.ld, dx, self.C0, P, self.C0)
        return dx, grads + tail


class UpStep:
    """UpsamplingNearest2d(scale_factor=2)"""

    def __init__(self, mod, in_shape):
        if int(mod.scale_factor) != 2:
            raise NotImplementedError('only 2x nearest up-sampling has a native kernel')
        self.C, self.H, self.W = in_shape
        self.out_shape = (self.C, 2 * self.H, 2 * self.W)

    def params(self):
        return []

    def forward(self, x, st, training):
        N, _, _, ld = x.shape
        out = K.empty((N, 2 * self.H, 2 * self.W, ld), x)
        K.upsample2(x, ld, out, ld, N, self.H, self.W, ld, False)
        st['ld'] = ld
        return out

    def backward(self, da, st, need_dx):
        if not need_dx:
            return None, []
        N = da.shape[0]
        ld = st['ld']
        dx = K.empty((N, self.H, self.W, ld), da)
        K.upsample2(da, da.shape[-1], dx, ld, N, self.H, self.W, ld, True)
        return dx, []


# ------------------------------------------------------------------------------------------------ the stack
class ConvStack:
    def __init__(self, mods, in_shape, image_out):
        self.in_shape = tuple(in_shape)
        self.image_out = image_out
        steps, shape = [], tuple(in_shape)
        flat = []
        for m in mods:          # torchvision's layer1..4 are Sequentials of residual blocks
            if isinstance(m, nn.Sequential) and all(is_residual_block(b) for b in m):
                flat += list(m)
            elif is_densenet_features(m):        # DenseNet: stem, blocks, transitions (norm, relu, conv, pool), norm5
                for b in m:
                    flat += list(b) if is_transition(b) else [b]
            elif is_transition(m):
                flat += list(m)
            else:
                flat.append(m)
        mods = flat
        i, n = 0, len(mods)
        groups = []
        while i < n:
            m = mods[i]
            if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):
                bn, act = None, 0
                j = i + 1
                if j < n and isinstance(mods[j], nn.BatchNorm2d):
                    bn = mods[j]
                    j += 1
                if j < n and type(mods[j]) in _ACT_CODE:
                    act = _ACT_CODE[type(mods[j])]
                    if act == 3 and abs(mods[j].negative_slope - nat.LEAKY_SLOPE) > 1e-12:
                        raise NotImplementedError('LeakyReLU with a slope other than 0.01 has no native kernel')
                    j += 1
                groups.append(('conv', m, bn, act))
                i = j
            elif isinstance(m, nn.MaxPool2d):
                groups.append(('pool', m))
                i += 1
            elif isinstance(m, nn.AvgPool2d) and (m.kernel_size if isinstance(m.kernel_size, int) else m.kernel_size[0]) == 1:
                i += 1      # AvgPool2d(1) is the identity (the vgg specs end with it)
            elif isinstance(m, (nn.AvgPool2d, nn.AdaptiveAvgPool2d)):
                groups.append(('avg', m))
                i += 1
            elif is_residual_block(m):
                groups.append(('res', m))
                i += 1
            elif is_dense_block(m):      # + the BatchNorm (+ ReLU) that reads the block's output
                bn, act, j = None, 0, i + 1
                if j < n and isinstance(mods[j], nn.BatchNorm2d):
                    bn, j = mods[j], j + 1
                    if j < n and type(mods[j]) in (nn.ReLU, nn.Identity):
                        act, j = _ACT_CODE[type(mods[j])], j + 1
                groups.append(('dense', m, bn, act))
                i = j
            elif isinstance(m, nn.UpsamplingNearest2d):
                groups.append(('up', m))
                i += 1
            elif isinstance(m, nn.Identity):
                i += 1
            else:
                raise NotImplementedError(f'{type(m).__name__} inside a conv stack')
        for gi, g in enumerate(groups):
            last = gi == len(groups) - 1
            if g[0] == 'conv':
                stp = ConvStep(g[1], g[2], g[3], shape, final_dense=last and image_out)
            elif g[0] == 'pool':
                stp = PoolStep(g[1], shape)
            elif g[0] == 'avg':
                stp = AvgStep(g[1], shape)
            elif g[0] == 'res':
                stp = ResidualStep(g[1], shape)
            elif g[0] == 'dense':
                if not (steps and isinstance(steps[-1], (PoolStep, AvgStep))) or shape[0] % 8:
                    raise NotImplementedError('a DenseNet block must follow a pooling layer with a multiple of 8 channels '
                                              '(the pooling writes the block input into the block buffer)')
                stp = DenseBlockStep(g[1], g[2], g[3], shape)
            else:
                stp = UpStep(g[1], shape)
            steps.append(stp)
            shape = stp.out_shape
        self.steps = steps
        self.out_shape = shape
        self.parameters = [p for s in steps for p in s.params()]
        convs = []
        for stp in steps:
            if isinstance(stp, ConvStep):
                convs.append(stp)
            elif isinstance(stp, ResidualStep):
                convs += stp.chain + ([stp.ds] if stp.ds is not None else [])
            elif isinstance(stp, DenseBlockStep):
                convs += stp.convs()
        self.plan = PackPlan(convs)
        for c in convs:
            c.plan = self.plan

    def forward(self, x, training):
        """x (N, C, H, W) fp32 / bf16 NCHW -> (output tensor, saved state)"""
        C, H, W = self.in_shape
        N = x.shape[0]
        if K is NativeKernels and training:
            self.plan.ensure()
        t = K.to_nhwc(x.reshape(N, C, H, W), r8(C))
        state = []
        # the BatchNorm statistics buffers of every layer of the stack come out of ONE zeroed allocation (one fill per forward
        # instead of one per layer)
        bn_steps = [s for s in self.steps if isinstance(s, ConvStep) and s.bn is not None and
                    (training or not s.bn.track_running_stats)]
        pool, off = None, 0
        if bn_steps:
            pool = K.zeros((sum(2 * s.Co for s in bn_steps),), t, torch.float64)
        pending = None
        for i, s in enumerate(self.steps):
            st, pending = pending or {}, None
            if pool is not None and any(s is b for b in bn_steps):
                st['stats_buf'] = pool[off:off + 2 * s.Co].view(2, s.Co)
                off += 2 * s.Co
            nxt = self.steps[i + 1] if i + 1 < len(self.steps) else None
            if isinstance(nxt, DenseBlockStep):      # this step writes the block input into the block's buffer
                buf = nxt.new_buffer(N, t)
                st['out'] = buf[..., :nxt.C0]
                pending = {'buf': buf}
            t = s.forward(t, st, training)
            state.append(st)
        Co, Ho, Wo = self.out_shape
        if self.image_out and t.shape[-1] == Co:
            out = t.permute(0, 3, 1, 2)          # logical NCHW, channels_last memory, bf16
        else:
            out = K.to_nchw(t, Co)               # fp32 NCHW (feature vectors for the encoder)
        return out, state, t.shape[-1]

    def backward(self, dout, state, ld_last, need_dx):
        Co, Ho, Wo = self.out_shape
        N = dout.shape[0]
        if self.image_out and ld_last == Co:
            g = dout
            if g.dtype != K.act_dtype:
                g = g.to(K.act_dtype)
            g = g.permute(0, 2, 3, 1)
            if not g.is_contiguous():
                g = g.contiguous()
        else:
            g = K.to_nhwc(dout, ld_last)
        grads = []
        for idx in range(len(self.steps) - 1, -1, -1):
            s = self.steps[idx]
            kw = {}
            prev = self.steps[idx - 1] if idx > 0 else None
            if isinstance(s, ConvStep) and isinstance(prev, ConvStep) and prev.bn is not None and \
                    state[idx - 1].get('bn_train') and not s.gemm1x1:
                pb = prev.bn
                kw['prev_bn'] = dict(y=state[idx - 1]['y'], ld_y=prev.ld_y, save=state[idx - 1]['save'],
                                     gamma=pb.weight.detach() if pb.affine else None,
                                     beta=pb.bias.detach() if pb.affine else None, act=prev.act)
            g, pg = s.backward(g, state[idx], need_dx or idx > 0, **kw)
            if 'prev_bn' in kw and kw['prev_bn'].get('sums') is not None:
                state[idx - 1]['bn_sums'] = kw['prev_bn']['sums']
            grads = pg + grads
            if g is None:
                break
        dx = None
        if need_dx and g is not None:
            C, H, W = self.in_shape
            dx = K.to_nchw(g, C)
        return dx, grads


class _StackFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, stack, training, *params):
        out, state, ld_last = stack.forward(x.detach(), training)
        ctx.stack, ctx.state, ctx.ld_last = stack, state, ld_last
        ctx.in_shape = x.shape
        return out

    @staticmethod
    def backward(ctx, dout):
        stack = ctx.stack
        dx, grads = stack.backward(dout, ctx.state, ctx.ld_last, ctx.needs_input_grad[0])
        ctx.state = None
        if dx is not None:
            dx = dx.reshape(ctx.in_shape)
        out = []
        for p, g in zip(stack.parameters, grads):
            out.append(g if (p is not None and g is not None and p.requires_grad) else None)
        return (dx, None, None) + tuple(out)


_stacks = {}


def run(mods, x, image_out=False):
    """Executes the conv-type modules `mods` (a slice of an nn.Sequential) on x (N, C, H, W)."""
    if not x.is_cuda and K is NativeKernels:
        raise nat.NativeError('joint-vae_b200 runs on CUDA devices only (there is no CPU fallback); got a CPU tensor')
    key = (tuple(id(m) for m in mods), tuple(x.shape[1:]), bool(image_out))
    stack = _stacks.get(key)
    if stack is None:
        try:
            stack = ConvStack(list(mods), tuple(x.shape[1:]), image_out)
        except NotImplementedError as e:
            stack = e                  # remembered: every later call raises the same error
        _stacks[key] = stack
    if isinstance(stack, NotImplementedError):
        raise stack
    training = any(m.training for m in mods)
    params = [p for p in stack.parameters]
    live = [p if p is not None else torch.empty(0, device=x.device) for p in params]
    if torch.is_grad_enabled() and (x.requires_grad or any(p is not None and p.requires_grad for p in params)):
        return _StackFn.apply(x, stack, training, *live)
    out, _, _ = stack.forward(x.detach(), training)
    return out
