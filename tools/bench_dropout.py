"""Dense-layer dropout (jvae_gemm_bf16_dropout, jvae_act_dropout_bwd), measured with CUDA events on one GPU:

  (a) Linear 1024 -> 4096 + ReLU + Dropout(0.2) on 8704 rows (the decoder rows of B = 512, L = 16), forward and forward +
      backward: the fused dropout GEMM against the plain native GEMM + ReLU (no dropout), and against torch
      Linear + ReLU + Dropout under bf16 autocast; the backward kernel alone with its algorithmic bytes (da, the saved output
      and dz, bf16: 6 B per element) and GB/s;
  (b) the c1-shaped MLP cvae training step (784-512-256 -> K = 16 -> 256-512-784, L = 1, B = 128) with dropout=0.2 against
      dropout=False, eager and train_step(graph=True).

Every time is the median of REPEATS measurements, each the mean over ITERS calls after warm-up.  In (a) one bf16 activation
is 71 MB and the forward + backward touches several of them, so the working set does not stay in the 126 MB of L2.
Usage: python tools/bench_dropout.py [--out FILE]   (prints the report; --out also writes it)"""
import argparse
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
P = 0.2


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


def dense_layer(pkg, lines, M=8704, K=1024, N=4096):
    from jointvae_b200 import engine
    nat = pkg._native
    dev = 'cuda:0'
    torch.manual_seed(0)
    lin = nn.Linear(K, N).to(dev)
    x = torch.randn(M, K, device=dev).to(torch.bfloat16).requires_grad_(True)
    go = torch.randn(M, N, device=dev).to(torch.bfloat16)
    flops = 2.0 * M * N * K
    lines.append(f'(a) Linear {K} -> {N} + ReLU + Dropout({P}) on {M} rows; forward {flops / 1e9:.1f} GFLOP, '
                 f'forward + backward {3 * flops / 1e9:.1f} GFLOP')

    def native(p):
        return lambda: engine.linear(x, lin.weight, lin.bias, act='relu', dropout=p)

    def native_fb(p):
        def run():
            y = engine.linear(x, lin.weight, lin.bias, act='relu', dropout=p)
            torch.autograd.grad(y, (x, lin.weight, lin.bias), go)
        return run
    drop = nn.Dropout(P).train()

    def torch_fwd():
        with torch.autocast('cuda', dtype=torch.bfloat16):
            return drop(torch.relu(lin(x)))

    def torch_fb():
        y = torch_fwd()
        torch.autograd.grad(y, (x, lin.weight, lin.bias), go)
    rows = [('native GEMM + ReLU + dropout (fused epilogue)', native(P), native_fb(P)),
            ('native GEMM + ReLU, no dropout', native(None), native_fb(None)),
            ('torch Linear + ReLU + Dropout, bf16 autocast', torch_fwd, torch_fb)]
    for name, f, fb in rows:
        with torch.no_grad():
            t_f = _time(f)
        t_fb = _time(fb)
        lines.append(f'    {name:47s} forward {t_f:7.3f} ms ({flops / t_f / 1e9:6.0f} TFLOP/s); forward + backward '
                     f'{t_fb:7.3f} ms ({3 * flops / t_fb / 1e9:6.0f} TFLOP/s)')
    # the backward kernel alone: dz = da * keep / (1 - p) * relu'(a_out), dbias
    a_out = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
    nat.gemm_bf16_dropout(M, N, K, x.detach(), K, engine._weight_bf16(lin.weight), K, p=P, seed=1, bias=lin.bias.detach(),
                          act=nat.ACT['relu'], out_bf16=a_out, ldd=N)
    dz = torch.empty_like(a_out)
    db = torch.empty(N, device=dev)
    t_b = _time(lambda: nat.act_dropout_bwd(go, N, a_out, N, M, N, nat.ACT['relu'], P, 1, 0, None, dz, N, db))
    lines.append(f'    jvae_act_dropout_bwd alone (dz and the bias gradient): {t_b * 1e3:.1f} us = '
                 f'{6.0 * M * N / t_b / 1e6:.0f} GB/s of algorithmic bytes (6 B per element)')


def c1_steps(pkg, lines, B=128):
    dev = 'cuda:0'
    g = torch.Generator().manual_seed(1)
    xs = [torch.rand(B, 1, 28, 28, generator=g).to(dev) for _ in range(4)]
    ys = [torch.randint(0, 10, (B,), generator=g).to(dev) for _ in range(4)]
    lines.append(f'(b) c1-shaped MLP cvae training step (784-512-256 -> K=16 -> 256-512-784, L=1, C=10, B={B})')
    for dropout in (P, False):
        torch.manual_seed(0)
        net = pkg.ClassificationVariationalNetwork(
            (1, 28, 28), 10, type='cvae', encoder=[512, 256], decoder=[256, 512], classifier=[], latent_dim=16,
            latent_sampling=1, test_latent_sampling=1, gamma=0, beta=1.0, output_activation='sigmoid',
            sigma={'value': 0.1}, prior={'init_mean': 1.0, 'learned_means': True, 'var_dim': 'scalar', 'seed': 1},
            dropout=dropout, optimizer={'optim_type': 'adam', 'lr': 1e-3, 'weight_decay': 3e-5, 'grad_clipping': 100})
        net = net.to(dev).train()
        it = [0]

        def step(graph):
            i = it[0] = it[0] + 1
            net.train_step(xs[i % 4], ys[i % 4], graph=graph)
        t_eager = _time(lambda: step(False), 5, 50, 5)
        t_graph = _time(lambda: step(True), 8, 100, 5)
        captured = any('graph' in st for st in getattr(net, '_graphs', {}).values())
        lines.append(f'    dropout={str(dropout):5s} eager {t_eager:6.3f} ms/step = {B / t_eager * 1e3:7.0f} img/s; '
                     f'train_step(graph=True) {t_graph:6.3f} ms/step = {B / t_graph * 1e3:7.0f} img/s '
                     f'(step captured in a CUDA graph: {captured})')
        del net
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_dropout.py measures on a CUDA device; none is visible')
    import __graft_entry__ as ge
    pkg = ge.load()
    lines = []
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:       # noqa: BLE001 -- the report says so instead
        q = f'nvidia-smi unavailable ({type(e).__name__})'
    lines.append(f'GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q}')
    lines.append(f'torch {torch.__version__}, CUDA {torch.version.cuda}; CUDA-event timings, median of {REPEATS} repeats '
                 f'of the mean over the timed calls')
    dense_layer(pkg, lines)
    c1_steps(pkg, lines)
    text = '\n'.join(lines) + '\n'
    print(text, end='')
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
