"""DenseNet features on the native engine, measured with CUDA events on one GPU:

  (a) the densenet121 `features` stack, forward + backward (input and parameter gradients), at B = 128 x 3 x 64 x 64 and
      B = 512 x 3 x 32 x 32: the native dense-block steps against torchvision's own module under torch.autocast(bfloat16),
      channels_last, eager, on the same GPU, same weights;
  (b) train_step(graph=True) images/s of the c4-shaped cvae with densenet121 features (upsampler ivgg, 3 x 64 x 64, K = 256,
      L = 8, C = 20, B = 128, BatchNorm both);
  (c) native kernel launches of one training step (the library's launch counter).

Usage: python tools/bench_densenet.py [--out FILE]   (prints the report; --out also writes it)"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.dont_write_bytecode = True


def _offline_densenets():
    """the features wrapper defaults to pretrained=True (a download): build the torchvision DenseNets without weights"""
    import torchvision.models as tvm
    for name in ('densenet121', 'densenet161', 'densenet169', 'densenet201'):
        orig = getattr(tvm, name)
        setattr(tvm, name, lambda *a, _orig=orig, **k: _orig(weights=None))


def _time(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def features_fwd_bwd(pkg, B, S, lines, warmup=3, iters=10):
    import copy
    import full_cases as fc
    from jointvae_b200 import conv_engine as ce
    from jointvae_b200.module.vae_layers.conv import ResOrDenseNetFeatures
    dev = 'cuda:0'
    torch.manual_seed(0)
    seq = fc.fill_state_(ResOrDenseNetFeatures('densenet121', (3, S, S), pretrained=False)).to(dev).train()
    lib = copy.deepcopy(seq).to(memory_format=torch.channels_last).train()
    x = torch.randn(B, 3, S, S, device=dev)
    go = torch.randn(B, 1024, S // 32, S // 32, device=dev)
    xn = x.clone().requires_grad_(True)
    xl = x.clone().contiguous(memory_format=torch.channels_last).requires_grad_(True)

    def native():
        out = ce.run(list(seq), xn)
        out.backward(go)

    def torch_bf16():
        with torch.autocast(device_type='cuda', dtype=torch.bfloat16):
            out = lib(xl)
        out.backward(go.to(out.dtype))

    # the parameter .grad buffers exist before timing (native kernels then accumulate into them, torch adds to them)
    native()
    torch_bf16()
    t_nat = _time(native, warmup, iters)
    t_lib = _time(torch_bf16, warmup, iters)
    t_nat2 = _time(native, 1, iters)           # repeated after the torch run: spread between two measurements
    n0 = pkg._native.launch_count()
    native()
    torch.cuda.synchronize()
    launches = pkg._native.launch_count() - n0
    lines.append(f'(a) densenet121 features fwd+bwd B={B} 3x{S}x{S}: native {t_nat:.3f} ms (repeat {t_nat2:.3f} ms, '
                 f'{launches} native launches), torch bf16 autocast channels_last eager {t_lib:.3f} ms, '
                 f'native / torch = {min(t_nat, t_nat2) / t_lib:.3f}')
    # per-step-type breakdown of the native run: CUDA events around every step of the stack
    stack = next(s for k, s in ce._stacks.items() if not isinstance(s, Exception) and k[1] == (3, S, S))
    ev = []
    orig = {}
    for s in stack.steps:
        cls = type(s)
        if cls in orig:
            continue
        orig[cls] = (cls.forward, cls.backward)

        def wrap(f, tag):
            def g(self, *a, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = f(self, *a, **k)
                e1.record()
                ev.append((type(self).__name__ + '.' + tag, e0, e1))
                return r
            return g
        cls.forward, cls.backward = wrap(cls.forward, 'forward'), wrap(cls.backward, 'backward')
    try:
        native()
        torch.cuda.synchronize()
    finally:
        for cls, (f, b) in orig.items():
            cls.forward, cls.backward = f, b
    tot = {}
    for tag, e0, e1 in ev:
        tot[tag] = tot.get(tag, 0.0) + e0.elapsed_time(e1)
    lines.append('    native breakdown (ms, one step): ' + ', '.join(f'{k} {v:.3f}' for k, v in sorted(tot.items())))


def cvae_train_step(pkg, lines, B=128, warmup=8, iters=30):
    import full_cases as fc
    dev = 'cuda:0'
    kw = fc._conv(20, 256, features='densenet121', upsampler='ivgg', shape=(3, 64, 64), L=8)
    kw['input_shape'] = tuple(kw['input_shape'])
    kw['prior'] = dict(fc.PRIOR)
    torch.manual_seed(0)
    net = pkg.ClassificationVariationalNetwork(**kw)
    fc.fill_state_(net)
    net = net.to(dev).train()
    g = torch.Generator().manual_seed(1)
    xs = [torch.rand(B, 3, 64, 64, generator=g).to(dev) for _ in range(4)]
    ys = [torch.randint(0, 20, (B,), generator=g).to(dev) for _ in range(4)]
    n0 = pkg._native.launch_count()
    net.train_step(xs[0], ys[0])
    torch.cuda.synchronize()
    launches = pkg._native.launch_count() - n0
    it = [0]

    def step(graph):
        i = it[0] = it[0] + 1
        net.train_step(xs[i % 4], ys[i % 4], graph=graph)

    t_eager = _time(lambda: step(False), 3, 10)
    t_graph = _time(lambda: step(True), warmup, iters)
    t_graph2 = _time(lambda: step(True), 2, iters)
    lines.append(f'(b) cvae densenet121 + ivgg, 3x64x64, K=256 L=8 C=20 B={B}, BatchNorm both: train_step(graph=True) '
                 f'{t_graph:.3f} ms/step = {B / t_graph * 1e3:.0f} img/s (repeat {t_graph2:.3f} ms = '
                 f'{B / t_graph2 * 1e3:.0f} img/s); eager {t_eager:.3f} ms/step = {B / t_eager * 1e3:.0f} img/s')
    lines.append(f'(c) native launches per training step (eager, counted by the library): {launches}')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_densenet.py measures on a CUDA device; none is visible')
    _offline_densenets()
    import __graft_entry__ as ge
    pkg = ge.load()
    lines = []
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:       # noqa: BLE001 -- the report says so instead
        q = f'nvidia-smi unavailable ({type(e).__name__})'
    lines.append(f'GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q}')
    lines.append(f'torch {torch.__version__}, CUDA {torch.version.cuda}; CUDA-event timings, means over the timed iterations')
    features_fwd_bwd(pkg, 128, 64, lines)
    features_fwd_bwd(pkg, 512, 32, lines)
    cvae_train_step(pkg, lines)
    text = '\n'.join(lines) + '\n'
    print(text, end='')
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
