"""TEST INFRASTRUCTURE ONLY: torch (CPU) emulation of the spec-grammar entry points of include/jvae_b200.h
(jvae_upsample_nearest, jvae_avgpool_pad), with the SAME argument meaning, on top of emu_kernels.EmuKernels (every other entry
point; its gather / wgrad emulation already takes any input and output stride).  tests/test_spec_layers_cpu.py drives the
conv engine through it on a machine without a GPU.  The product never imports this file."""
import torch

from emu_kernels import EmuKernels


class SpecEmuKernels(EmuKernels):

    @classmethod
    def upsample_nearest(cls, src, ld_src, dst, ld_dst, N, H, W, C, s, backward):
        cls.launches += 1
        assert s >= 1
        v = src.float()[..., :C]
        assert not torch.isnan(v).any(), 'up-sampling read an uninitialised activation'
        if not backward:
            dst[..., :C] = v.repeat_interleave(s, 1).repeat_interleave(s, 2).to(EmuKernels.store)
        else:
            dst[..., :C] = v.reshape(N, H, s, W, s, C).sum((2, 4)).to(EmuKernels.store)

    @classmethod
    def avgpool_pad(cls, src, ld_src, dst, ld_dst, N, H, W, C, kh, kw, sh, sw, ph, pw, backward):
        cls.launches += 1
        assert 2 * ph <= kh and 2 * pw <= kw
        pool = lambda t: torch.nn.functional.avg_pool2d(t, (kh, kw), (sh, sw), (ph, pw), ceil_mode=False,
                                                        count_include_pad=True)
        if not backward:
            v = src.float()[..., :C]
            assert not torch.isnan(v).any(), 'pooling read an uninitialised activation'
            dst[..., :C] = pool(v.permute(0, 3, 1, 2)).permute(0, 2, 3, 1).to(EmuKernels.store)
        else:
            g = src.float()[..., :C]
            with torch.enable_grad():
                x = torch.zeros(N, C, H, W, requires_grad=True)
                pool(x).backward(g.permute(0, 3, 1, 2))
            dst[..., :C] = x.grad.permute(0, 2, 3, 1).to(EmuKernels.store)
