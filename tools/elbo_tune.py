"""Times the fused ELBO kernels alone (CUDA events, L2 flushed between launches) at the c2 / c5 shapes.
Usage: python tools/elbo_tune.py"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as g

pkg = g.build()
nat = pkg._native
dev = 'cuda:0'
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def bench(fn, n=20):
    ts = []
    for i in range(n + 3):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        if i >= 3:
            ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def bench_graph(make, nbuf=6, n=10):
    """steady-state time per launch: nbuf launches on rotating reconstruction buffers (together larger than L2) replayed from
    a CUDA graph, so neither the CPU launch path nor the event pair is in the figure"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(nbuf): make(i)()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for i in range(nbuf): make(i)()
    ts = []
    for i in range(n + 2):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); g.replay(); b.record()
        torch.cuda.synchronize()
        if i >= 2: ts.append(a.elapsed_time(b) * 1e3 / nbuf)
    ts.sort()
    return ts[len(ts) // 2]


for (B, L, K, C, D) in [(512, 16, 128, 10, 3072), (512, 16, 256, 100, 3072), (512, 16, 256, 1000, 3072), (2048, 16, 128, 10, 3072)]:
    x = torch.rand(B, D, device=dev)
    xr = torch.rand(L + 1, B, D, device=dev).bfloat16()
    mu, lv = torch.randn(B, K, device=dev), torch.randn(B, K, device=dev) * 0.1
    z = torch.randn(L + 1, B, K, device=dev)
    en = torch.rand(L, B, device=dev) * K
    y = torch.randint(0, C, (B,), device=dev)
    means, T = torch.randn(C, K, device=dev), torch.ones(C, device=dev)
    sig = torch.zeros(1, device=dev)
    cfg = nat.make_cfg(B=B, L=L, K=K, C=C, D=D, x_reco=xr, logits=None, var_dim='scalar', prior_kind='gaussian',
                       conditional=True, sigma_is_log=True, sigma_is_rmse=False, beta=1.0, gamma_w=0.0, var_w=1.0)
    nat.elbo_prior_stats(cfg, means, T)
    cfg.prior_stats_ready = 1          # time the loss kernel alone (the prologue runs before the network in the model)
    out = nat.elbo_train_fwd(cfg, x, xr, mu, lv, None, y, means, T, sig)
    gvec = torch.full((B,), 1.0 / B, device=dev)
    bytes_fwd = B * (D * 4 + L * D * 2 + 2 * K * 4 + 8 + 32)
    t_f = bench(lambda: nat.elbo_train_fwd(cfg, x, xr, mu, lv, None, y, means, T, sig))
    t_b = bench(lambda: nat.elbo_train_bwd(cfg, gvec, x, xr, mu, lv, None, y, means, T, sig, out['wmse']))
    t_e = bench(lambda: nat.elbo_eval_fwd(cfg, x, xr, mu, lv, z, en, None, means, T, sig))
    nat.profile_drain(); nat.profile_native(True)
    for fn in (lambda: nat.elbo_train_fwd(cfg, x, xr, mu, lv, None, y, means, T, sig),
               lambda: nat.elbo_train_bwd(cfg, gvec, x, xr, mu, lv, None, y, means, T, sig, out['wmse']),
               lambda: nat.elbo_eval_fwd(cfg, x, xr, mu, lv, z, en, None, means, T, sig)):
        for i in range(12):
            flush.zero_(); fn()
    nat.profile_native(False)
    pr = {k: sorted(v)[len(v) // 2] * 1e3 for k, v in nat.profile_drain().items() if k != 'conv_launches' and v}
    print('   events inside the library (L2 flushed): ' + ' | '.join(f'{k} {v:.1f} us' for k, v in pr.items()), flush=True)
    xrs = [torch.rand(L + 1, B, D, device=dev).bfloat16() for _ in range(6)]
    dxs = [torch.empty(L + 1, B, D, device=dev, dtype=torch.bfloat16) for _ in range(6)]
    g_f = bench_graph(lambda i: (lambda: nat.elbo_train_fwd(cfg, x, xrs[i], mu, lv, None, y, means, T, sig)))
    g_e = bench_graph(lambda i: (lambda: nat.elbo_eval_fwd(cfg, x, xrs[i], mu, lv, z, en, None, means, T, sig)))
    print(f'   graph-replayed, rotating buffers: fwd {g_f:.2f} us = {bytes_fwd / g_f / 1e3:.0f} GB/s | eval {g_e:.2f} us = '
          f'{(bytes_fwd + B * L * K * 4) / g_e / 1e3:.0f} GB/s', flush=True)
    print(f'B={B} L={L} K={K} C={C}: fwd {t_f[0]:.1f} us (min {t_f[1]:.1f}) = '
          f'{bytes_fwd / t_f[0] / 1e3:.0f} GB/s | bwd {t_b[0]:.1f} us = {(bytes_fwd + B * L * D * 2) / t_b[0] / 1e3:.0f} GB/s | '
          f'eval {t_e[0]:.1f} us = {(bytes_fwd + B * L * K * 4) / t_e[0] / 1e3:.0f} GB/s', flush=True)
