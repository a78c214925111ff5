"""TEST INFRASTRUCTURE ONLY: a torch (CPU) emulation of the C-ABI entry points conv_engine drives
(include/jvae_b200.h: jvae_conv_gather_gemm, jvae_conv_wgrad, jvae_gemm_bf16, jvae_bn_*, jvae_act_bwd, jvae_maxpool2_*,
jvae_upsample2), with the SAME argument meaning.  It lets the `-m "not gpu"` suite check the host logic of the native
convolution path (tap tables, sub-pixel phases, weight arrangements, BatchNorm backward algebra, layouts) against
torch.nn on a machine without a GPU.  The product never imports this file."""
import torch


def _cblk(c):
    return 64 if c > 32 else (32 if c > 16 else 16)


def _act(z, act):
    if act == 1:
        return z.clamp_min(0)
    if act == 2:
        return torch.sigmoid(z)
    if act == 3:
        return torch.where(z > 0, z, 0.01 * z)
    return z


class EmuKernels:
    launches = 0
    act_dtype = store = torch.bfloat16      # set to torch.float32 to separate logic errors from bf16 storage rounding

    @staticmethod
    def empty(shape, like, dtype=torch.bfloat16):
        if dtype == torch.bfloat16:
            dtype = EmuKernels.store
        return torch.full(shape, float('nan'), dtype=dtype) if dtype.is_floating_point else torch.zeros(shape, dtype=dtype)

    @staticmethod
    def zeros(shape, like, dtype=torch.float32):
        if dtype == torch.bfloat16:
            dtype = EmuKernels.store
        return torch.zeros(shape, dtype=dtype)

    @staticmethod
    def taps_arg(taps):
        return [t[0] for t in taps], [t[1] for t in taps]

    @staticmethod
    def to_nhwc(x, c_pad):
        n, c, h, w = x.shape
        out = torch.zeros((n, h, w, c_pad), dtype=EmuKernels.store)
        out[..., :c] = x.float().permute(0, 2, 3, 1)
        return out

    @staticmethod
    def to_nchw(t, C):
        return t[..., :C].float().permute(0, 3, 1, 2).contiguous()

    @staticmethod
    def _shifted(x, dy, dx, s, Hq, Wq):
        """x (N,H,W,C) f32 -> tile[n,qy,qx,c] = x[n, qy*s+dy, qx*s+dx, c] (0 outside)"""
        N, H, W, C = x.shape
        iy = torch.arange(Hq) * s + dy
        ix = torch.arange(Wq) * s + dx
        my = (iy >= 0) & (iy < H)
        mx = (ix >= 0) & (ix < W)
        t = x[:, iy.clamp(0, H - 1)][:, :, ix.clamp(0, W - 1)]
        return t * (my[:, None] & mx[None, :]).to(t.dtype)[None, :, :, None]

    @classmethod
    def gather(cls, x, Cin, wmat, cout_pad, taps, in_stride, Hq, Wq, out, Cout, out_s, out_o, bias, act, stats):
        cls.launches += 1
        N, H, W, ld_in = x.shape
        cb = _cblk(Cin)
        nck = (Cin + cb - 1) // cb
        T = len(taps[0])
        assert wmat.shape == (cout_pad, T * nck * cb) and cout_pad % 16 == 0 and ld_in % 8 == 0
        w = wmat.float().view(cout_pad, T, nck * cb)
        assert float(w[Cout:].abs().max() if cout_pad > Cout else 0) == 0 and float(w[:, :, Cin:].abs().sum()) == 0
        w = w[:Cout, :, :Cin]
        xin = x.float()[..., :Cin]
        assert not torch.isnan(xin).any(), 'gather read an uninitialised activation'
        acc = torch.zeros((N, Hq, Wq, Cout))
        for t in range(T):
            acc += torch.einsum('nhwc,oc->nhwo', cls._shifted(xin, taps[0][t], taps[1][t], in_stride, Hq, Wq), w[:, t])
        if bias is not None:
            acc += bias.float()
        if stats is not None:
            stats[0] += acc.sum((0, 1, 2))
            stats[1] += (acc * acc).sum((0, 1, 2))
        acc = _act(acc, act & 0xff)
        view = out[:, out_o[0]::out_s[0], out_o[1]::out_s[1]]
        assert view.shape[1] == Hq and view.shape[2] == Wq, (view.shape, Hq, Wq)
        view[..., :Cout] = acc.to(EmuKernels.store)
        view[..., Cout:] = 0

    @staticmethod
    def phases_arg(ops):
        return [(EmuKernels.taps_arg(op['taps']), op['out_o']) for op in ops]

    @classmethod
    def subpixel(cls, x, Cin, wmat, cout_pad, phases, Hq, Wq, out, Cout, out_s, bias, act, stats):
        """jvae_conv_subpixel_gemm: phase i owns the next len(taps_i) [tap] blocks of the merged weight matrix"""
        cb = _cblk(Cin)
        w = (Cin + cb - 1) // cb * cb
        first = 0
        for taps, out_o in phases:
            T = len(taps[0])
            cls.gather(x, Cin, wmat[:, first * w:(first + T) * w].contiguous(), cout_pad, taps, 1, Hq, Wq, out, Cout,
                       (out_s, out_s), out_o, bias, act, stats)
            first += T
        assert first * w == wmat.shape[1]
        cls.launches -= len(phases) - 1
        return True

    @classmethod
    def wgrad(cls, g, Cg, x, Cx, taps, in_stride, dw, swapped=False):
        cls.launches += 1
        N, Hq, Wq, _ = g.shape
        gf, xf = g.float()[..., :Cg], x.float()[..., :Cx]
        assert not torch.isnan(gf).any() and not torch.isnan(xf).any()
        assert dw.shape == ((Cx, Cg, len(taps[0])) if swapped else (Cg, Cx, len(taps[0])))
        for t in range(len(taps[0])):
            v = torch.einsum('nhwa,nhwb->ab', gf, cls._shifted(xf, taps[0][t], taps[1][t], in_stride, Hq, Wq))
            dw[:, :, t] += v.t() if swapped else v

    @classmethod
    def gemm(cls, mode, M, N, K, a, b, bias=None, act=0, out_bf16=None, out_f32=None):
        cls.launches += 1
        af, bf = a.float(), b.float()
        if mode == 0:
            d = af[:M, :K] @ bf[:N, :K].t()
        elif mode == 1:
            d = af[:M, :K] @ bf[:K, :N]
        else:
            d = af[:K, :M].t() @ bf[:K, :N]
        if bias is not None:
            d = d + bias.float()
        d = _act(d, act)
        if out_bf16 is not None:
            out_bf16[:M, :N] = d.to(EmuKernels.store)
        if out_f32 is not None:
            out_f32[:M, :N] = d

    @staticmethod
    def _flat(t, P, ld):
        return t.reshape(P, ld)

    @classmethod
    def bn_stats(cls, y, P, C, ld, stats):
        cls.launches += 1
        v = cls._flat(y, P, ld)[:, :C].float()
        stats[0] += v.sum(0)
        stats[1] += (v * v).sum(0)

    @classmethod
    def bn_apply_fwd(cls, y, P, C, ld_y, stats, gamma, beta, eps, momentum, running_mean, running_var, num_batches, training,
                     act, out, ld_out, save):
        cls.launches += 1
        v = cls._flat(y, P, ld_y)[:, :C].float()
        if training:
            mean = stats[0] / P
            var = (stats[1] / P - mean * mean).clamp_min(0)
            rstd = (var + eps).rsqrt()
            save[0], save[1] = mean, rstd
            if running_mean is not None:
                running_mean.mul_(1 - momentum).add_(momentum * mean)
                running_var.mul_(1 - momentum).add_(momentum * var * P / max(P - 1, 1))
            if num_batches is not None:
                num_batches += 1
        else:
            mean, rstd = running_mean, (running_var + eps).rsqrt()
        g = gamma if gamma is not None else torch.ones(C)
        b = beta if beta is not None else torch.zeros(C)
        scale = g * rstd
        shift = b - mean * scale
        cls._flat(out, P, ld_out)[:, :C] = _act(v * scale + shift, act).to(EmuKernels.store)

    @classmethod
    def bn_bwd(cls, da, ld_da, y, ld_y, P, C, save, gamma, beta, act, sums, dy, ld_dy, dgamma, dbeta):
        cls.launches += 2
        g = cls._flat(da, P, ld_da)[:, :C].float()
        v = cls._flat(y, P, ld_y)[:, :C].float()
        mean, rstd = save[0], save[1]
        gm = gamma if gamma is not None else torch.ones(C)
        bt = beta if beta is not None else torch.zeros(C)
        scale = gm * rstd
        z = v * scale + (bt - mean * scale)
        if act == 1:
            g = g * (z > 0)
        elif act == 2:
            s = torch.sigmoid(z)
            g = g * s * (1 - s)
        elif act == 3:
            g = torch.where(z > 0, g, 0.01 * g)
        xh = (v - mean) * rstd
        s1, s2 = g.sum(0), (g * xh).sum(0)
        sums[0], sums[1] = s1, s2
        if dgamma is not None:
            dgamma += s2
        if dbeta is not None:
            dbeta += s1
        cls._flat(dy, P, ld_dy)[:, :C] = (scale * (g - s1 / P - xh * s2 / P)).to(EmuKernels.store)

    @classmethod
    def act_bwd(cls, da, ld_da, a_out, ld_a, P, C, act, dy, ld_dy, dbias):
        cls.launches += 1
        g = cls._flat(da, P, ld_da)[:, :C].float()
        if act:
            o = cls._flat(a_out, P, ld_a)[:, :C].float()
            g = g * ((o > 0).float() if act == 1 else (torch.where(o > 0, 1.0, 0.01) if act == 3 else o * (1 - o)))
        if dy is not None:
            cls._flat(dy, P, ld_dy)[:, :C] = g.to(EmuKernels.store)
        if dbias is not None:
            dbias += g.sum(0)

    @classmethod
    def maxpool_fwd(cls, x, N, H, W, C, ld_in, k, stride, out, ld_out):
        cls.launches += 1
        v = torch.nan_to_num(x.float()[..., :C]).permute(0, 3, 1, 2)
        out[..., :C] = torch.nn.functional.max_pool2d(v, k, stride).permute(0, 2, 3, 1).to(EmuKernels.store)

    @classmethod
    def maxpool_bwd(cls, x, N, H, W, C, ld_in, k, stride, dout, ld_dout, din, ld_din):
        cls.launches += 1
        with torch.enable_grad():
            v = torch.nan_to_num(x.float()[..., :C]).permute(0, 3, 1, 2).clone().requires_grad_(True)
            o = torch.nn.functional.max_pool2d(v, k, stride)
            o.backward(torch.nan_to_num(dout.float()[..., :C]).permute(0, 3, 1, 2))
        din[..., :C] = v.grad.permute(0, 2, 3, 1).to(EmuKernels.store)

    @classmethod
    def maxpool_pad_fwd(cls, x, N, H, W, C, ld_in, k, stride, pad, out, ld_out):
        cls.launches += 1
        v = torch.nan_to_num(x.float()[..., :C]).permute(0, 3, 1, 2)
        out[..., :C] = torch.nn.functional.max_pool2d(v, k, stride, pad).permute(0, 2, 3, 1).to(EmuKernels.store)

    @classmethod
    def maxpool_pad_bwd(cls, x, N, H, W, C, ld_in, k, stride, pad, dout, ld_dout, din, ld_din):
        cls.launches += 1
        with torch.enable_grad():
            v = torch.nan_to_num(x.float()[..., :C]).permute(0, 3, 1, 2).clone().requires_grad_(True)
            o = torch.nn.functional.max_pool2d(v, k, stride, pad)
            o.backward(torch.nan_to_num(dout.float()[..., :C]).permute(0, 3, 1, 2))
        din[..., :C] = v.grad.permute(0, 2, 3, 1).to(EmuKernels.store)

    @classmethod
    def avgpool(cls, src, ld_src, dst, ld_dst, N, H, W, C, k, backward):
        cls.launches += 1
        s = torch.nan_to_num(src.float()[..., :C])
        if not backward:
            dst[..., :C] = s.view(N, H // k, k, W // k, k, C).mean((2, 4)).to(EmuKernels.store)
        else:
            dst[..., :C] = (s / (k * k)).repeat_interleave(k, 1).repeat_interleave(k, 2).to(EmuKernels.store)

    @classmethod
    def vstack_rows(cls, dy, ld_dy, N, H, W, k, pad, Co, U, ld_u):
        cls.launches += 1
        g = torch.nan_to_num(dy.float())[..., :Co]
        U.zero_()
        for ty in range(k):
            sh = ty - pad                           # U[r][ty] = dy[r - sh]
            lo, hi = max(0, sh), min(H, H + sh)
            if hi > lo:
                U[:, lo:hi, :, ty * Co:(ty + 1) * Co] = g[:, lo - sh:hi - sh].to(EmuKernels.store)

    @classmethod
    def add_act(cls, a, ld_a, b, ld_b, P, C, act, out, ld_out):
        cls.launches += 1
        v = cls._flat(a, P, ld_a)[:, :C].float() + cls._flat(b, P, ld_b)[:, :C].float()
        cls._flat(out, P, ld_out)[:, :C] = _act(v, act).to(EmuKernels.store)

    @classmethod
    def upsample2(cls, src, ld_src, dst, ld_dst, N, H, W, C, backward):
        cls.launches += 1
        s = src.float()[..., :C]
        if not backward:
            dst[..., :C] = s.repeat_interleave(2, 1).repeat_interleave(2, 2).to(EmuKernels.store)
        else:
            dst[..., :C] = s.view(N, H, 2, W, 2, C).sum((2, 4)).to(EmuKernels.store)


def emu_batch_u8_to_f32(cfg, data, index, flip, crop_ij):
    """TEST ONLY: the index map of jvae_batch_u8_to_f32 (include/jvae_b200.h) in torch, CPU.  data uint8 (n, H, W, C)."""
    H, W, C, oH, oW = cfg.H, cfg.W, cfg.C, cfg.out_H, cfg.out_W
    B = index.numel()
    oy = torch.arange(oH).view(1, oH, 1).expand(B, oH, oW)
    ox = torch.arange(oW).view(1, 1, oW).expand(B, oH, oW)
    y, x = oy + cfg.post_off_y, ox + cfg.post_off_x
    inside = (y >= 0) & (y < H) & (x >= 0) & (x < W)
    fl = (flip.bool() if flip is not None else torch.zeros(B, dtype=torch.bool)).view(B, 1, 1)
    if not cfg.flip_first:
        x = torch.where(fl, W - 1 - x, x)
    if crop_ij is not None:
        y = (y + crop_ij[:, 0].view(B, 1, 1).long() - cfg.crop_pad).clamp(0, H - 1)
        x = (x + crop_ij[:, 1].view(B, 1, 1).long() - cfg.crop_pad).clamp(0, W - 1)
    if cfg.flip_first:
        x = torch.where(fl, W - 1 - x, x)
    y, x = y.clamp(0, H - 1), x.clamp(0, W - 1)
    img = data[index.view(B, 1, 1).expand(B, oH, oW), y, x]              # (B, oH, oW, C) uint8
    out = img.to(torch.float32).div(255)
    out = torch.where(inside.unsqueeze(-1), out, torch.zeros(()))
    return out.permute(0, 3, 1, 2).contiguous()
