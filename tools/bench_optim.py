"""The fused optimizer kernels (csrc/optim.cu) and the c2 training step per optimizer, measured with CUDA events on one GPU:

  (a) the update kernels alone over the c2 model's flat buffer (vgg19 + deconv32, K = 128, L = 16, C = 10: its trainable
      parameters with every slice padded to JVAE_OPT_CHUNK), with an fp32 and a bf16 gradient bucket: grad_sqnorm, each
      update (Adam, AMSGrad, SGD, SGD with momentum, Nesterov) and the pair, in microseconds, with the update's algorithmic
      bytes (fp32 p, buf, m, v, vmax read and written, g read once) and GB/s; beside them, the same update through
      clip_grad_norm_(foreach=True) + torch.optim.{Adam, SGD}(fused=True) on the same parameter shapes;
  (b) the c2 training step (B = 512) with Adam and with SGD (momentum 0.9, Nesterov), eager and train_step(graph=True), in
      ms/step and images/s.

Every time is the median of REPEATS measurements, each the mean over ITERS calls after warm-up.  At c2 one fp32 flat buffer
is 84 MB, so what an update touches (p and g at least) does not fit the 126 MB of L2: the kernels stream from HBM.
Usage: python tools/bench_optim.py [--out FILE]   (prints the report; --out also writes it)"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.dont_write_bytecode = True

REPEATS, ITERS, WARMUP = 5, 50, 10
SGD_OPT = {'optim_type': 'sgd', 'lr': 1e-2, 'momentum': 0.9, 'nesterov': True, 'weight_decay': 3e-5, 'grad_clipping': 100}
ADAM_OPT = {'optim_type': 'adam', 'lr': 1e-3, 'weight_decay': 3e-5, 'grad_clipping': 100}


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


def _c2_net(pkg, optimizer):
    import full_cases as fc
    kw = fc._conv(10, 128)
    kw['input_shape'] = tuple(kw['input_shape'])
    kw['prior'] = dict(fc.PRIOR)
    kw['optimizer'] = dict(optimizer)
    torch.manual_seed(0)
    net = pkg.ClassificationVariationalNetwork(**kw)
    fc.fill_state_(net)
    return net


def update_kernels(pkg, lines):
    nat = pkg._native
    dev = 'cuda:0'
    shapes = [p.shape for p in _c2_net(pkg, ADAM_OPT).parameters() if p.requires_grad]
    CH = nat.OPT_CHUNK
    sizes = [(s.numel() + CH - 1) // CH * CH for s in shapes]
    n, nseg = sum(sizes), len(sizes)
    lines.append(f'(a) update kernels over the c2 flat buffer: {len(shapes)} trainable parameters, '
                 f'{sum(s.numel() for s in shapes) / 1e6:.2f} M elements, {n / 1e6:.2f} M with the JVAE_OPT_CHUNK padding')
    chunk_seg = torch.repeat_interleave(torch.arange(nseg, dtype=torch.int32), torch.tensor([q // CH for q in sizes])).to(dev)
    aux = torch.zeros(1 + nseg, device=dev)
    norm2, seg_active = aux[:1], aux[1:].view(torch.int32)
    seg_step, seg_bc = torch.zeros(nseg, dtype=torch.int32, device=dev), torch.zeros(2 * nseg, device=dev)
    torch.manual_seed(0)
    g = torch.randn(n, device=dev) * 1e-3
    p, m, v, vmax, buf = (torch.zeros(n, device=dev) for _ in range(5))
    p.normal_()
    tab = dict(chunk_seg=chunk_seg, seg_active=seg_active, seg_step=seg_step)
    adam = dict(max_norm=100.0, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=3e-5, seg_bc=seg_bc, **tab)
    sgd = dict(max_norm=100.0, lr=1e-5, weight_decay=3e-5, dampening=0.0, **tab)
    variants = [
        ('Adam', 28, lambda gq: nat.adam_step(p, m, v, gq, norm2, **adam)),
        ('AMSGrad', 36, lambda gq: nat.adam_amsgrad_step(p, m, v, vmax, gq, norm2, **adam)),
        ('SGD', 12, lambda gq: nat.sgd_step(p, None, gq, norm2, momentum=0.0, nesterov=False, **sgd)),
        ('SGD momentum 0.9', 20, lambda gq: nat.sgd_step(p, buf, gq, norm2, momentum=0.9, nesterov=False, **sgd)),
        ('SGD Nesterov 0.9', 20, lambda gq: nat.sgd_step(p, buf, gq, norm2, momentum=0.9, nesterov=True, **sgd)),
    ]
    for gname, gq in (('fp32', g), ('bf16', nat.cast_f32_bf16(g))):
        gb = gq.element_size()
        aux.zero_()
        nat.grad_sqnorm(gq, norm2, chunk_seg, seg_active)

        def sq():
            aux.zero_()
            nat.grad_sqnorm(gq, norm2, chunk_seg, seg_active)
        t_sq = _time(sq)
        lines.append(f'    {gname} bucket: grad_sqnorm {t_sq * 1e3:.1f} us = {gb * n / t_sq / 1e6:.0f} GB/s ({gb} B/param)')
        for name, b32, upd in variants:
            by = b32 - 4 + gb                                      # the bucket's gradient element instead of an fp32 one
            t_up = _time(lambda: upd(gq))
            t_pair = _time(lambda: (sq(), upd(gq)))
            lines.append(f'      {name:17s} update {t_up * 1e3:6.1f} us = {by * n / t_up / 1e6:5.0f} GB/s ({by} B/param); '
                         f'grad_sqnorm + update {t_pair * 1e3:6.1f} us')
    # torch: foreach clip + fused optimizer on the same shapes (fp32 gradients)
    ps = [torch.nn.Parameter(torch.randn(s, device=dev)) for s in shapes]
    for q in ps:
        q.grad = torch.randn_like(q) * 1e-3
    for name, b32, opt in (('Adam', 28, torch.optim.Adam(ps, lr=1e-3, weight_decay=3e-5, fused=True)),
                           ('AMSGrad', 36, torch.optim.Adam(ps, lr=1e-3, weight_decay=3e-5, amsgrad=True, fused=True)),
                           ('SGD', 12, torch.optim.SGD(ps, lr=1e-5, weight_decay=3e-5, fused=True)),
                           ('SGD momentum 0.9', 20, torch.optim.SGD(ps, lr=1e-5, momentum=0.9, weight_decay=3e-5, fused=True)),
                           ('SGD Nesterov 0.9', 20, torch.optim.SGD(ps, lr=1e-5, momentum=0.9, nesterov=True, weight_decay=3e-5,
                                                                    fused=True))):
        def step():
            torch.nn.utils.clip_grad_norm_(ps, 100.0, foreach=True)
            opt.step()
        t = _time(step)
        lines.append(f'    torch clip_grad_norm_(foreach) + {name:17s} (fused), fp32 grads: {t * 1e3:6.1f} us '
                     f'(update bytes {b32} B/param: {b32 * n / t / 1e6:5.0f} GB/s over the whole pair)')
        opt.state.clear()


def train_steps(pkg, lines, B=512):
    dev = 'cuda:0'
    g = torch.Generator().manual_seed(1)
    xs = [torch.rand(B, 3, 32, 32, generator=g).to(dev) for _ in range(4)]
    ys = [torch.randint(0, 10, (B,), generator=g).to(dev) for _ in range(4)]
    lines.append(f'(b) c2 training step (vgg19 + deconv32, K=128, L=16, C=10, B={B}, BatchNorm both)')
    for name, oc in (('Adam', ADAM_OPT), ('SGD momentum 0.9 Nesterov', SGD_OPT)):
        net = _c2_net(pkg, oc).to(dev).train()
        it = [0]

        def step(graph):
            i = it[0] = it[0] + 1
            net.train_step(xs[i % 4], ys[i % 4], graph=graph)
        t_eager = _time(lambda: step(False), 3, 10, 3)
        t_graph = _time(lambda: step(True), 8, 20, 3)
        captured = any('graph' in st for st in getattr(net, '_graphs', {}).values())
        lines.append(f'    {name:26s} eager {t_eager:6.3f} ms/step = {B / t_eager * 1e3:6.0f} img/s; train_step(graph=True) '
                     f'{t_graph:6.3f} ms/step = {B / t_graph * 1e3:6.0f} img/s (step captured in a CUDA graph: {captured})')
        del net
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_optim.py measures on a CUDA device; none is visible')
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
    update_kernels(pkg, lines)
    train_steps(pkg, lines)
    text = '\n'.join(lines) + '\n'
    print(text, end='')
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text)


if __name__ == '__main__':
    main()
