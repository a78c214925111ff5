"""TEST INFRASTRUCTURE ONLY: torch (CPU) emulation of the DenseNet entry points of include/jvae_b200.h (jvae_bn_stats_ld,
jvae_bn_preact_fwd, jvae_bn_preact_bwd, jvae_cast_f32_bf16_ld), with the SAME argument meaning, on top of emu_kernels.EmuKernels
(every other entry point).  tests/test_densenet_cpu.py drives conv_engine.DenseBlockStep through it on a machine without a
GPU.  The product never imports this file."""
import torch

from emu_kernels import EmuKernels, _act


class DenseEmuKernels(EmuKernels):
    # (entry point, channels read) of every statistics launch when a list: the DenseNet tests check that a block's batch
    # statistics are produced once per channel
    stats_trace = None

    @staticmethod
    def _slice(t, P, C):
        """(P, C) view of the first C channels of an NHWC tensor or channel-slice view"""
        return t[..., :C].reshape(P, C)

    @classmethod
    def bn_stats_ld(cls, y, P, C, ld, stats, stats_ld):
        cls.launches += 1
        if DenseEmuKernels.stats_trace is not None:
            DenseEmuKernels.stats_trace.append(('bn_stats_ld', C))
        v = cls._slice(y, P, C).float()
        assert not torch.isnan(v).any(), 'statistics of an unwritten channel'
        stats[:C] += v.sum(0).double()
        stats[stats_ld:stats_ld + C] += (v * v).sum(0).double()

    @classmethod
    def bn_preact_fwd(cls, y, P, C, ld_y, stats, stats_ld, gamma, beta, eps, momentum, running_mean, running_var, num_batches,
                      training, act, out, ld_out, save):
        cls.launches += 1
        assert C % 8 == 0 and C <= 2048, 'jvae_bn_preact_fwd takes C <= 8 * NORM_MAX_THREADS, a multiple of 8'
        v = cls._slice(y, P, C).float()
        if training:
            mean = stats[:C] / P
            var = (stats[stats_ld:stats_ld + C] / P - mean * mean).clamp_min(0)
            mean, var = mean.float(), var.float()
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
        out[..., :C] = _act(v * scale + (b - mean * scale), act).to(EmuKernels.store).view(out[..., :C].shape)

    @classmethod
    def bn_preact_bwd(cls, da, ld_da, y, ld_y, P, C, save, gamma, beta, running_mean, running_var, eps, training, act, sums, dx,
                      ld_dx, dgamma, dbeta):
        cls.launches += 2 if training else 1
        assert C % 8 == 0 and C <= 2048, 'jvae_bn_preact_bwd takes C <= 8 * NORM_MAX_THREADS, a multiple of 8'
        g = cls._slice(da, P, C).float()
        v = cls._slice(y, P, C).float()
        if training:
            mean, rstd = save[0], save[1]
        else:
            mean, rstd = running_mean, (running_var + eps).rsqrt()
        gm = gamma if gamma is not None else torch.ones(C)
        bt = beta if beta is not None else torch.zeros(C)
        scale = gm * rstd
        z = v * scale + (bt - mean * scale)
        if act == 1:
            g = g * (z > 0)
        xh = (v - mean) * rstd
        if training:
            s1, s2 = g.sum(0), (g * xh).sum(0)
            sums[0], sums[1] = s1, s2
            if dgamma is not None:
                dgamma += s2
            if dbeta is not None:
                dbeta += s1
            d = scale * (g - s1 / P - xh * s2 / P)
        else:
            d = scale * g
        dx[..., :C] += d.view(dx[..., :C].shape)

    @classmethod
    def cast_f32_bf16_ld(cls, src, ld_src, dst, ld_dst, P, C):
        cls.launches += 1
        assert src.dtype == torch.float32
        dst[..., :C] = src[..., :C].to(EmuKernels.store)
