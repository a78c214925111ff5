"""The spec-grammar layers beyond strides 1 / 2, 2x up-sampling and tiling pools, one layer at a time on one GPU, forward and
backward, native (conv_engine steps on NHWC bf16 tensors: the layer's own launches, no layout conversion) against torch /
cuDNN in bf16 (channels_last, autocast) on the same shapes:

  (a) 'x4+0:4' Conv2d(64, 128, 4, stride 4) + ReLU at c2's B = 512 on 32 x 32 maps (the tap-box kernels, stride 4);
  (b) its transposed mirror ConvTranspose2d(128, 64, 4, stride 4) + ReLU, 8 x 8 -> 32 x 32, on (L+1)*B = 8704 images (16
      sub-pixel phases of one tap each, output stride 4; weight gradient on the tap-box kernel at stride 4);
  (c) 'U:4' UpsamplingNearest2d(4), 64 channels, 8 x 8 -> 32 x 32, on 8704 images (jvae_upsample_nearest);
  (d) 'Ax3+1:2' AvgPool2d(3, 2, 1) and 'A3+1:2' (the grammar's default pooling kernel 5: AvgPool2d(5, 2, 1)), 64 channels,
      32 x 32, B = 512 (jvae_avgpool_pad).

Convolutions: TFLOP/s of the direct algorithm (2 N Ho Wo Co Ci k^2 per pass; the backward is the data and the weight gradient).
Streaming kernels: GB/s of the algorithmic bytes (every input element read once, every output element written once, bf16).
Every working set but (d)'s is larger than the 126 MB L2.  Every time is the median of REPEATS measurements, each the mean over
ITERS calls after warm-up.  Usage: python tools/bench_spec_layers.py [--out FILE]"""
import argparse
import copy
import os
import statistics
import subprocess
import sys

import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

REPEATS, ITERS, WARMUP = 5, 20, 5
DEV = 'cuda:0'


def _time(fn, warmup=WARMUP, iters=ITERS, repeats=REPEATS):
    """median over `repeats` of the mean time of `iters` calls, in ms"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return statistics.median(out)


def _native_step(ce, mods, shape, N):
    """(forward, forward + backward) closures of the stack's single step on NHWC bf16 tensors"""
    stack = ce.ConvStack([copy.deepcopy(m).to(DEV) for m in mods], shape, False)
    assert len(stack.steps) == 1
    step = stack.steps[0]
    C, H, W = shape
    x = torch.randn(N, H, W, ce.r8(C), device=DEV).to(torch.bfloat16)
    y = step.forward(x, {}, True)
    da = torch.randn(y.shape, device=DEV).to(torch.bfloat16)

    def fwd():
        step.forward(x, {}, True)

    def fwd_bwd():
        st = {}
        step.forward(x, st, True)
        step.backward(da, st, True)
    return fwd, fwd_bwd


def _torch_step(mods, shape, N):
    m = nn.Sequential(*[copy.deepcopy(q) for q in mods]).to(DEV).to(memory_format=torch.channels_last)
    x = torch.randn(N, *shape, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    with torch.autocast('cuda', dtype=torch.bfloat16):
        g = torch.randn_like(m(x))

    def fwd():
        with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
            m(x)

    def fwd_bwd():
        with torch.autocast('cuda', dtype=torch.bfloat16):
            y = m(x)
        y.backward(g)
    return fwd, fwd_bwd


def conv_case(ce, lines, title, mods, shape, N, flops_pass):
    nf, nfb = _native_step(ce, mods, shape, N)
    tf, tfb = _torch_step(mods, shape, N)
    t = {k: _time(f) for k, f in (('nf', nf), ('nfb', nfb), ('tf', tf), ('tfb', tfb))}
    lines.append(f'{title}')
    lines.append(f'  native  forward {t["nf"]:8.3f} ms ({flops_pass / t["nf"] / 1e9:6.1f} TFLOP/s)   forward+backward '
                 f'{t["nfb"]:8.3f} ms ({3 * flops_pass / t["nfb"] / 1e9:6.1f} TFLOP/s)')
    lines.append(f'  cuDNN   forward {t["tf"]:8.3f} ms ({flops_pass / t["tf"] / 1e9:6.1f} TFLOP/s)   forward+backward '
                 f'{t["tfb"]:8.3f} ms ({3 * flops_pass / t["tfb"] / 1e9:6.1f} TFLOP/s)')


def stream_case(ce, lines, title, mods, shape, N, bytes_fwd, bytes_bwd):
    nf, nfb = _native_step(ce, mods, shape, N)
    tf, tfb = _torch_step(mods, shape, N)
    t = {k: _time(f) for k, f in (('nf', nf), ('nfb', nfb), ('tf', tf), ('tfb', tfb))}
    nb, tb = t['nfb'] - t['nf'], t['tfb'] - t['tf']
    lines.append(f'{title}')
    lines.append(f'  native  forward {t["nf"]:8.3f} ms ({bytes_fwd / t["nf"] / 1e6:6.0f} GB/s)   backward {nb:8.3f} ms '
                 f'({bytes_bwd / nb / 1e6:6.0f} GB/s)')
    lines.append(f'  torch   forward {t["tf"]:8.3f} ms ({bytes_fwd / t["tf"] / 1e6:6.0f} GB/s)   backward {tb:8.3f} ms '
                 f'({bytes_bwd / tb / 1e6:6.0f} GB/s)   (backward = forward+backward - forward)')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device: nothing is measured without one')
    import __graft_entry__ as g
    pkg = g.load()
    from jointvae_b200 import conv_engine as ce
    lines = []
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:       # noqa: BLE001 -- the report says so instead
        q = f'nvidia-smi unavailable ({type(e).__name__})'
    lines.append(f'GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q}')
    lines.append(f'torch {torch.__version__}, CUDA {torch.version.cuda}, cuDNN {torch.backends.cudnn.version()}; CUDA-event '
                 f'timings, median of {REPEATS} repeats of the mean over {ITERS} calls')
    torch.manual_seed(0)
    B, NI = 512, 8704
    conv_case(ce, lines, f"(a) Conv2d(64, 128, 4, stride=4) + ReLU, B = {B}, 64 x 32 x 32 -> 128 x 8 x 8",
              [nn.Conv2d(64, 128, 4, stride=4), nn.ReLU()], (64, 32, 32), B, 2.0 * B * 8 * 8 * 128 * 64 * 16)
    conv_case(ce, lines, f"(b) ConvTranspose2d(128, 64, 4, stride=4) + ReLU, N = {NI}, 128 x 8 x 8 -> 64 x 32 x 32",
              [nn.ConvTranspose2d(128, 64, 4, stride=4), nn.ReLU()], (128, 8, 8), NI, 2.0 * NI * 8 * 8 * 128 * 64 * 16)
    small, big = NI * 8 * 8 * 64 * 2, NI * 32 * 32 * 64 * 2
    stream_case(ce, lines, f"(c) UpsamplingNearest2d(scale_factor=4), N = {NI}, 64 x 8 x 8 -> 64 x 32 x 32 "
                f"(algorithmic bytes: forward {(small + big) / 1e9:.2f} GB, backward the same)",
                [nn.UpsamplingNearest2d(scale_factor=4)], (64, 8, 8), NI, small + big, small + big)
    for k, tok in ((3, 'Ax3+1:2'), (5, 'A3+1:2')):
        Ho = (32 + 2 - k) // 2 + 1
        byt = B * 64 * (32 * 32 + Ho * Ho) * 2
        stream_case(ce, lines, f"(d) '{tok}' AvgPool2d({k}, 2, 1), B = {B}, 64 x 32 x 32 -> 64 x {Ho} x {Ho} "
                    f"(algorithmic bytes: {byt / 1e6:.0f} MB each way)",
                    [nn.AvgPool2d(k, 2, 1)], (64, 32, 32), B, byt, byt)
    text = '\n'.join(lines)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
