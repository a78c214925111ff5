#!/usr/bin/env python
"""Benchmark of the joint-VAE hot path on B200 (BASELINE.json metric: train images/s on the CIFAR-10-shaped conv
joint-VAE, K=128, L=16, C=10, batch 512 per GPU, bf16 GEMMs; plus OOD-scoring samples/s and the fused-ELBO HBM GB/s).

  python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                    the reference's algorithm (oracle port) on the host cores
  python bench.py ... --dump-outputs DIR                  also writes the last timed step's outputs as DIR/<name>.npy

A "step" is one full optimisation step of the path: zero_grad, weight re-pack, features/encoder/sampler/decoder/classifier
forward, fused ELBO forward + backward, network backward, gradient all-reduce (N > 1), global-norm clip, Adam.
Prints ONE JSON line on rank 0.  Sub-results: `workloads` (BASELINE configs[2], [3]: c3 and c4 train steps with their own
ms_per_step) and `scoring_c5` (configs[4]: 1 Mi samples sharded over the ranks, per-class evaluate + 11 OOD scores +
predictions per batch, ONE final gather over NCCL, device ROC tables on rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree, which may be read-only

OPT = {'optim_type': 'adam', 'lr': 1e-3, 'weight_decay': 3e-5, 'grad_clipping': 100}


def _conv(C, K, features='vgg19', upsampler='deconv32', shape=(3, 32, 32), L=16):
    return dict(input_shape=shape, num_labels=C, type='cvae', features=features, upsampler=upsampler, encoder=[], decoder=[],
                classifier=[], batch_norm='both', latent_dim=K, latent_sampling=L, test_latent_sampling=L, gamma=0, beta=1.0,
                output_activation='linear', sigma={'value': 1.0, 'learned': True}, optimizer=dict(OPT))


WORKLOADS = {
    # BASELINE.json configs[1]: conv joint-VAE on synthetic 3x32x32, VGG-style encoder, K=128, L=16, C=10, B=512/GPU
    'c2': dict(ctor=_conv(10, 128), batch=512, fwd_gflop_per_img=2.903,
               name='conv joint-VAE 3x32x32 vgg19+deconv32 BN K=128 L=16 C=10 B=512/GPU'),
    # configs[2]: CIFAR-100 shape, wider per-class contraction
    'c3': dict(ctor=_conv(100, 256), batch=512, fwd_gflop_per_img=2.921,
               name='conv joint-VAE 3x32x32 vgg19+deconv32 BN K=256 L=16 C=100 B=512/GPU'),
    # configs[3]: ResNet-style, imagenet20-subset shape, data parallel at 2/4/8 GPUs
    'c4': dict(ctor=_conv(20, 256, features='resnet18', upsampler='ivgg', shape=(3, 64, 64), L=8), batch=128,
               fwd_gflop_per_img=None, name='ResNet joint-VAE 3x64x64 resnet18+ivgg BN K=256 L=8 C=20 B=128/GPU'),
    # configs[0]: the reference's CPU-runnable case
    'c1': dict(ctor=dict(input_shape=(1, 28, 28), num_labels=10, type='cvae', encoder=[512, 256], decoder=[256, 512],
                         classifier=[], latent_dim=16, latent_sampling=1, test_latent_sampling=1, gamma=0, beta=1.0,
                         output_activation='sigmoid', sigma={'value': 0.1}, optimizer=dict(OPT)),
               batch=128, fwd_gflop_per_img=0.0032, name='MLP joint-VAE 1x28x28 K=16 L=1 C=10 B=128'),
}
PRIOR = {'init_mean': 1.0, 'learned_means': True, 'var_dim': 'scalar', 'seed': 1}
C5_SAMPLES = 1 << 20          # configs[4]: 1 Mi synthetic test samples (half of them drawn as the OOD set)
PREROLL_STEPS = 48            # untimed steps right before the timed region (run_native)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('hbm_gbs', 6650.0), d.get('bf16_tflops_sustained', 1400.0), 'measured'
    return 6650.0, 1400.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)"""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc = [], None
        self.timed = False         # rows read while the timed region runs are kept apart (mark(True) / mark(False))
        self.rows_timed = []
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            row = [c.strip() for c in line.split(',')]
            self.rows.append(row)
            if self.timed:
                self.rows_timed.append(row)

    def mark(self, on):
        self.timed = on

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        # the timed region of a short run (10 steps = 0.13 s) can fall between two 100 ms samples: then the samples of the
        # identical warm-up steps right before it (the sampler starts with them) stand in, and the window says so
        rows, window = (self.rows_timed, 'timed region') if self.rows_timed else (self.rows[-3:], 'warm-up steps + timed region')
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith('active') for r in rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm), 'window': window}


def make_ctor(wl, **over):
    kw = json.loads(json.dumps(wl['ctor']))
    kw['input_shape'] = tuple(kw['input_shape'])
    kw['prior'] = dict(PRIOR)
    kw.update(over)
    return kw


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def _oracle_net(wl, **over):
    """The reference's algorithm for the path (oracle/torch_model.py + oracle/elbo_numpy.py, fp32 restatements of cvae.py's
    train / eval step pinned against the unmodified reference by tests/golden/, including at these configurations)."""
    import torch
    import __graft_entry__ as g
    from oracle.torch_model import OracleNet, describe_model
    pkg = g.load_package()
    torch.manual_seed(0)
    model = pkg.ClassificationVariationalNetwork(**make_ctor(wl, **over))          # layer containers only (CPU, no compute)
    cfg, arch = describe_model(model)
    net = OracleNet(cfg, arch)
    net.load_state_dict(model.state_dict())
    return net


def cpu_train_run(wl, steps, warmup, batch, threads):
    import torch
    from oracle.torch_model import train_step
    torch.set_num_threads(threads)
    net = _oracle_net(wl)
    net.train()
    oc = wl['ctor']['optimizer']
    opt = torch.optim.Adam(net.parameters(), lr=oc['lr'], weight_decay=oc['weight_decay'])
    B, L, K, C = batch, wl['ctor']['latent_sampling'], wl['ctor']['latent_dim'], wl['ctor']['num_labels']
    gen = torch.Generator().manual_seed(0)
    x = torch.rand(B, *wl['ctor']['input_shape'], generator=gen)
    y = torch.randint(0, C, (B,), generator=gen)
    times = []
    for i in range(warmup + steps):
        eps = torch.randn(L + 1, B, K, generator=gen)
        t0 = time.perf_counter()
        train_step(net, opt, x, y, eps, beta=wl['ctor']['beta'], gamma=wl['ctor']['gamma'] or 0.0, clip=oc['grad_clipping'])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return B / dt, dt


def cpu_score_run(wl, steps, warmup, batch, threads, **over):
    """the reference's scoring step (cvae.py:1629-1687): evaluate(x) per class + batch_dist_measures + predict_after_evaluate"""
    import numpy as np
    import torch
    from oracle import elbo_numpy as on
    torch.set_num_threads(threads)
    net = _oracle_net(wl, **over)
    net.eval()
    kw = make_ctor(wl, **over)
    B, L, K, C = batch, kw['test_latent_sampling'], kw['latent_dim'], kw['num_labels']
    gen = torch.Generator().manual_seed(0)
    x = torch.rand(B, *kw['input_shape'], generator=gen)
    n = lambda t: None if t is None else t.detach().numpy()
    prior = on.Prior(n(net.encoder.prior.mean), n(net.encoder.prior._var_parameter), var_dim='scalar', conditional=True)
    methods = ['iws-2s', 'iws-a-1-1', 'iws-a-4-1', 'iws', 'mse', 'elbo', 'soft', 'elbo-2s', 'elbo-a-1-1', 'elbo-a-4-1', 'zdist']
    times = []
    for i in range(warmup + steps):
        eps = torch.randn(L + 1, B, K, generator=gen)
        t0 = time.perf_counter()
        with torch.no_grad():
            xr, ye, mu, lv, z, en = net(x, eps)
        losses, logits = on.evaluate(n(x), n(xr), n(ye), n(mu), n(lv), n(z), n(en), prior, y=None, training=False,
                                     type='cvae', sigma_value=float(net.sigma.detach()[0]), sigma_is_log=bool(net.arch['sigma']['is_log']),
                                     y_is_decoded=bool(net.arch['y_is_decoded']))
        on.batch_dist_measures(logits, losses, methods, type='cvae', num_labels=C)
        on.predict_after_evaluate(logits, losses, 'iws')
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return B / dt, dt


def run_reference(args, wl):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    # torch.distributed.run exports OMP_NUM_THREADS=1 to every rank: the CPU arm takes all host cores explicitly
    cores = os.cpu_count() or 1
    v_small, _ = cpu_train_run(wl, max(1, args.steps // 3), 1, 32, cores)
    v, dt = cpu_train_run(wl, args.steps, args.warmup, args.cpu_batch, cores)
    v_one, _ = cpu_train_run(wl, 1, 1, 16, 1)
    vs, _ = cpu_score_run(wl, 2, 1, 32, cores)
    world = args.gpus
    line = {'impl': 'reference', 'metric': 'train_images_per_sec', 'value': v, 'unit': 'images/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': wl['name'], 'global_batch': world * wl['batch'], 'parallelism': f'dp{world}',
                       'sample_batch': args.cpu_batch},
            'cpu_baseline': {'value': v, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                             'sample': f'{args.steps} full train steps at batch {args.cpu_batch} of the configured {wl["batch"]} '
                                       f'(the step is linear in the batch: {v_small:.1f} images/s at batch 32), oracle/torch_model.py fp32',
                             'images_per_s_at_batch_32': v_small, 'images_per_s_one_thread': v_one,
                             'scoring_samples_per_s': vs, 'host_cores': cores,
                             'why_port': 'the reference is Python on /root/reference, which does not exist on the GPU box; the port '
                                         'is pinned to it by tests/golden (incl. this configuration: tests/golden/full_c2.npz)'},
            'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ native arm (GPU)
def run_native(args, wl):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: the hot path has no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    pkg = g.load()
    nat = pkg._native

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, before_last=None):
        """CUDA-event time of `steps` calls bracketed by barrier + synchronize, max over ranks (ms); `before_last` is enqueued
        ahead of the last call and its device time is left out"""
        barrier()
        a, b, c, d = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        a.record()
        for i in range(steps):
            if before_last is not None and i == steps - 1:
                c.record()
                before_last()
                d.record()
            fn(i)
        b.record()
        barrier()
        ms = a.elapsed_time(b) - (c.elapsed_time(d) if before_last is not None else 0.0)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def build_net(w, **over):
        torch.manual_seed(0)
        net = pkg.ClassificationVariationalNetwork(**make_ctor(w, **over)).to(dev)
        if world > 1:
            pkg.distributed.attach(net, bf16_bucket=True)
        return net

    def train_inputs(w, B, npool=4):
        gen = torch.Generator().manual_seed(1 + rank)
        shape, C = tuple(w['ctor']['input_shape']), w['ctor']['num_labels']
        xs_h = [torch.rand(B, *shape, generator=gen).pin_memory() for _ in range(npool)]
        ys_h = [torch.randint(0, C, (B,), generator=gen).pin_memory() for _ in range(npool)]
        return xs_h, ys_h, [t.to(dev) for t in xs_h], [t.to(dev) for t in ys_h]

    # ================================================================ headline workload: train step
    net = build_net(wl)
    net.train()
    # the seeded initial state, restored ahead of the last timed step: the training trajectory is not bit-reproducible (fp32
    # atomics in the weight-gradient reductions, amplified by Adam), so only a step that starts from these parameters computes
    # the same outputs from the same batch and noise in every run (--dump-outputs)
    initial = {k: v.detach().clone() for k, v in net.state_dict().items()}

    def restore_initial():
        with torch.no_grad():
            for k, v in net.state_dict().items():
                v.copy_(initial[k])
        pkg.engine.bump_params()
        pkg.engine.bump_stats()
    B = args.batch or wl['batch']
    C = wl['ctor']['num_labels']
    shape = tuple(wl['ctor']['input_shape'])
    npool = 4
    xs_h, ys_h, xs, ys = train_inputs(wl, B, npool)
    use_graph = args.graph                     # N > 1: the NCCL all-reduce is a node of the captured step
    step_eager = lambda i: net.train_step(xs[i % npool], ys[i % npool])
    last = {}           # what the latest step returned: the last timed step's losses / measures for --dump-outputs

    def step_dev(i):
        last['out'] = net.train_step(xs[i % npool], ys[i % npool], graph=use_graph)

    def step_e2e(i):
        x = xs_h[i % npool].to(dev, non_blocking=True)
        y = ys_h[i % npool].to(dev, non_blocking=True)
        losses, _ = net.train_step(x, y, graph=use_graph)
        return float(losses['total'].mean().item())          # device -> host read of the step's result

    for i in range(args.warmup):
        step_dev(i)
    # ---- device-resident timing (value); per-launch CUDA events around the fused ELBO kernels and every convolution launch
    # (eager steps: per-launch events cannot be recorded inside a replayed graph)
    for i in range(2):          # the capture above emptied the caching allocator: let the eager pools settle again
        step_eager(i)
    nat.profile_drain()
    nat.CONV_FLOPS = []             # algorithmic FLOPs of every convolution call, in call order (paired with the native records)
    nat.profile_native(True)        # events recorded inside the library right around each fused-ELBO / convolution launch
    n0 = nat.launch_count()
    ms_eager = timed(step_eager, args.steps)
    launches = nat.launch_count() - n0
    nat.profile_native(False)
    prof = nat.profile_drain()
    conv_launches, conv_flops = prof.pop('conv_launches'), nat.CONV_FLOPS
    nat.CONV_FLOPS = None
    conv_prof = {}
    if len(conv_launches) == len(conv_flops):
        for (kname, t_ms), flops in zip(conv_launches, conv_flops):
            e = conv_prof.setdefault(kname, [0.0, 0.0, 0])
            e[0] += t_ms * 1e-3
            e[1] += flops
            e[2] += 1
    # the published value: the same steps without per-launch events, through the public train_step (CUDA-graph replays when
    # --graph, the default on one GPU: same kernels, same arithmetic, no per-launch host cost)
    clocks = ClockSampler(local)        # started ahead of the timed region: nvidia-smi needs ~0.1-0.3 s for its first row
    # the same steps, untimed, while the sampler starts (~0.5 s of c2 at batch 512); a fixed count rather than a time, so every
    # rank runs the same number of data-parallel steps and the last timed step draws the same noise in every run
    for i in range(PREROLL_STEPS):
        step_dev(i)
    torch.cuda.synchronize()
    clocks.mark(True)
    ms = timed(step_dev, args.steps, before_last=restore_initial)
    clocks.mark(False)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last['out'])      # before later steps overwrite the graph's output buffers
    ms_plain = ms_eager
    # ---- end-to-end timing through the public API with host buffers
    step_e2e(0)
    ms_e2e = timed(step_e2e, args.steps)
    # ---- the same, fed by the uint8 input pipeline (utils/batch_loader.py): dataset in pinned HOST memory, per step one
    # uint8 batch copy + gather / flip / random-crop / ToTensor kernel on a side stream, train step, loss read back
    ms_loader = None
    if len(shape) == 3:
        from jointvae_b200.utils.batch_loader import DeviceBatchLoader
        gen = torch.Generator().manual_seed(7 + rank)
        u8 = torch.randint(0, 256, ((args.steps + 2) * B, shape[1], shape[2], shape[0]), dtype=torch.uint8, generator=gen)
        tg = torch.randint(0, C, (u8.shape[0],), generator=gen)
        loader = DeviceBatchLoader(u8, tg, B, device=dev, data_augmentation=['flip', 'crop'], resident=False, seed=rank)
        it = iter(loader)
        step_loader = lambda i: float(net.train_step(*next(it), graph=use_graph)[0]['total'].mean().item())
        step_loader(0)
        ms_loader = timed(step_loader, args.steps)
        del loader, u8

    # ================================================================ BASELINE configs[4]: sharded scoring with one final gather
    scoring = None
    if args.c5:
        scoring = []
        for C_ in (10, 100, 1000):
            scoring.append(run_c5(pkg, wl, C_, 128 if C_ == 10 else 256, dev, world, rank, timed, B, args))
    del net, xs, ys
    torch.cuda.empty_cache()

    # ================================================================ BASELINE configs[2], [3]: c3 / c4 train steps
    extra = {}
    if args.extra:
        for name in ('c3', 'c4'):
            if name == args.workload:
                continue
            w = WORKLOADS[name]
            n2 = build_net(w)
            n2.train()
            _, _, xs2, ys2 = train_inputs(w, w['batch'])
            f = lambda i: n2.train_step(xs2[i % len(xs2)], ys2[i % len(xs2)], graph=use_graph)
            for i in range(max(3, args.warmup)):
                f(i)
            ms2 = timed(f, args.steps)
            extra[name] = {'workload': w['name'], 'value': world * w['batch'] * args.steps / (ms2 * 1e-3), 'unit': 'images/s',
                           'ms_per_step': ms2 / args.steps, 'global_batch': world * w['batch'], 'steps': args.steps}
            if w['fwd_gflop_per_img']:
                extra[name]['tensor_tflops'] = 3 * w['fwd_gflop_per_img'] * 1e9 * w['batch'] * args.steps / (ms2 * 1e-3) / 1e12
            del n2, xs2, ys2
            torch.cuda.empty_cache()

    if rank != 0:
        _finish(world)
        return
    hbm, tf, which = peaks()
    L, K, D = wl['ctor']['latent_sampling'], wl['ctor']['latent_dim'], int(torch.tensor(shape).prod())
    # algorithmic bytes of the fused ELBO train forward per sample (SURVEY.md 8d): x f32 + L reconstructions (bf16)
    # + mu/log_var f32 + label + 8 outputs (logits only when a classifier exists: gamma=0 here)
    bytes_fwd = B * (D * 4 + L * D * 2 + 2 * K * 4 + 8 + 8 * 4)
    t_fwd = sum(prof['elbo_train_fwd']) / max(1, len(prof['elbo_train_fwd'])) * 1e-3
    achieved = bytes_fwd / t_fwd / 1e9 if t_fwd > 0 else None
    value = world * B * args.steps / (ms * 1e-3)
    e2e = world * B * args.steps / (ms_e2e * 1e-3)
    flops = 3 * (wl['fwd_gflop_per_img'] or 0.0) * 1e9 * B * args.steps / (ms * 1e-3)
    # dominant kernel of the step = the convolution kernel with the largest summed CUDA-event time
    dom = max(conv_prof.items(), key=lambda kv: kv[1][0]) if conv_prof else None
    roofline = None
    if dom is not None:
        kname, (t_s, fl, nl) = dom
        ach = fl / t_s / 1e12
        roofline = {'kernel': kname, 'bound': 'tensor', 'achieved': ach, 'peak': tf, 'unit': 'TFLOP/s', 'frac': ach / tf,
                    # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel, average over the launches of one
                    # step in the committed ncu --set full capture (profiles/, r02): null until re-captured for a new kernel
                    'traffic': args.traffic if args.traffic is not None else
                    (1097.1e6 if (kname == 'conv_halo_kernel' and args.workload == 'c2' and B == 512) else None),
                    'traffic_of': 'largest launch of the kernel (32 -> 32 k5 forward on 8704 x 32 x 32, 456.3 GFLOP, 1140.9 MB '
                                  'algorithmic): profiles/r02_conv_halo_ncu_full.txt; achieved / us_per_launch average all launches',
                    'peak_source': which + ' (MEASURED_PEAKS.json bf16_tflops_sustained)',
                    'launches_per_step': nl / args.steps, 'us_per_launch': t_s / nl * 1e6, 'flop_per_launch': fl / nl,
                    'share_of_step': t_s / (ms_plain * 1e-3) if ms_plain else None,
                    'by_kernel': {k: {'ms_per_step': v[0] / args.steps * 1e3, 'tflops': v[1] / v[0] / 1e12,
                                      'launches_per_step': v[2] / args.steps} for k, v in conv_prof.items()}}
    line = {
        'metric': 'train_images_per_sec', 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': {'workload': wl['name'], 'global_batch': world * B, 'parallelism': f'dp{world}',
                   'l2': 'per-step working set (activations, 53 MB x_reco alone) exceeds L2; 4 rotating input batches',
                   'launch': 'cuda graph replay' if use_graph else 'eager', 'eager_ms_per_step': ms_eager / args.steps},
        'clocks': clk,
        'e2e': {'value': e2e, 'unit': 'images/s', 'h2d_bytes_per_step': B * D * 4 + B * 8, 'd2h_bytes_per_step': 4,
                'ms_per_step': ms_e2e / args.steps},
        'e2e_uint8_loader': None if ms_loader is None else {
            'value': world * B * args.steps / (ms_loader * 1e-3), 'unit': 'images/s', 'h2d_bytes_per_step': B * D + B * 25,
            'd2h_bytes_per_step': 4, 'note': 'uint8 dataset in pinned host memory, flip + crop + ToTensor on the device'},
        'gpu_launches': int(launches),
        'roofline': roofline,
        'elbo_roofline': {'kernel': 'elbo_train_fwd_kernel (fused prior/ELBO forward)', 'bound': 'hbm', 'achieved': achieved,
                          'peak': hbm, 'unit': 'GB/s', 'frac': (achieved / hbm) if achieved else None,
                          'traffic': 57.59e6 if (args.workload == 'c2' and B == 512) else None,
                          'peak_source': which + ' (MEASURED_PEAKS.json hbm_gbs)', 'bytes_per_launch': bytes_fwd,
                          'us_per_launch': t_fwd * 1e6,
                          'bwd_us_per_launch': sum(prof['elbo_train_bwd']) / max(1, len(prof['elbo_train_bwd'])) * 1e3},
        'gemm_roofline': None if not wl['fwd_gflop_per_img'] else {
            'bound': 'tensor', 'achieved': flops / 1e12, 'peak': tf, 'unit': 'TFLOP/s', 'frac': flops / 1e12 / tf,
            'note': 'whole step: 3 x forward GEMM/conv FLOPs / step time'},
        'workloads': extra,
        'scoring_c5': scoring,
    }
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        v, dt = cpu_train_run(wl, 2, 1, args.cpu_batch if args.cpu_batch <= 64 else 64, cores)
        vs, _ = cpu_score_run(wl, 2, 1, 32, cores)
        line['cpu_baseline'] = {'value': v, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                                'sample': '2 full train steps at batch 64 after 1 warm-up, oracle/torch_model.py fp32, all host cores',
                                'scoring_samples_per_s': vs}
    print(json.dumps(line))
    _finish(world)


def dump_outputs(path, losses, measures):
    """What a caller of train_step receives from the last timed step, as <path>/<name>.npy: the per-sample losses
    (`loss.<key>`, float32) and the running measures (`measure.<key>`, float64 scalars).  That step starts from the seeded
    initial parameters, and its batch and noise follow from the seeds and the arguments alone, so two builds run with the
    same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {'loss.' + k: v.detach().float().cpu().numpy() for k, v in losses.items()}
    arrays.update({'measure.' + k: np.float64(float(v)) for k, v in measures.items()})
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def _finish(world):
    """End of a rank.  With N > 1 the captured data-parallel steps hold NCCL kernels inside CUDA graphs; tearing the communicator
    down under them can block, so the rank synchronises, meets the others at a barrier and leaves without the teardown."""
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


def run_c5(pkg, wl, C_, K_, dev, world, rank, timed, B, args):
    """BASELINE configs[4]: C5_SAMPLES synthetic samples, sample-sharded over the ranks (contiguous shards, no per-batch
    communication).  Per batch: per-class evaluate (BatchNorm folded) + the 11 OOD scores + the predictions, written into
    device buffers; then ONE gather of the scores to rank 0 (NCCL all_gather) and the device ROC table of every method
    (in-distribution half against the OOD half).  samples/s = all samples / max-over-ranks device time of the whole thing."""
    import torch
    import torch.distributed as dist
    from jointvae_b200.utils.roc_curves import roc_curve
    nat = pkg._native
    torch.manual_seed(0)
    m = pkg.ClassificationVariationalNetwork(**make_ctor(wl, num_labels=C_, latent_dim=K_)).to(dev)
    m.eval()
    shape = tuple(wl['ctor']['input_shape'])
    n_total = args.c5_samples
    lo, hi = pkg.distributed.shard_range(n_total, rank, world)
    nb = (hi - lo) // B
    gen = torch.Generator().manual_seed(11 + rank)
    pool_in = [torch.rand(B, *shape, generator=gen).to(dev) for _ in range(4)]
    # the "OOD" half: blocky images (8 x 8 constant patches), a different distribution for the ROC tables to separate
    pool_out = [torch.rand(B, shape[0], 4, 4, generator=gen).repeat_interleave(shape[1] // 4, 2)
                .repeat_interleave(shape[2] // 4, 3).to(dev) for _ in range(4)]
    methods = [mm for mm in m.ood_methods if not mm.startswith('odin')]
    base = sorted(set(mm[:-3] if mm.endswith('-2s') else mm.split('-a-')[0] for mm in methods))
    pm = m.predict_methods[0]
    buf = torch.empty((len(base), nb * B), dtype=torch.float32, device=dev)
    preds = torch.empty(nb * B, dtype=torch.int64, device=dev)
    out = {}

    def whole(_):
        with torch.no_grad():
            for i in range(nb):
                x = (pool_in if i < nb // 2 else pool_out)[i % 4]
                _, lg, ls, _ = m.evaluate(x)
                sc = m.batch_dist_measures(lg, ls, base)
                buf[:, i * B:(i + 1) * B] = torch.stack([sc[k] for k in base])
                preds[i * B:(i + 1) * B] = m.predict_after_evaluate(lg, ls, method=pm)
            local_scores = {k: buf[j] for j, k in enumerate(base)}
            full = pkg.distributed.gather_scores(local_scores, n_total) if world > 1 else local_scores
            if rank == 0:
                # shard r holds [in-distribution half | OOD half] of its own samples
                per = n_total // world
                res = {}
                for mm in methods:
                    k = mm[:-3] if mm.endswith('-2s') else mm.split('-a-')[0]
                    v = full[k].view(world, per)
                    ind, ood = v[:, :per // 2].reshape(-1), v[:, per // 2:].reshape(-1)
                    two = 'around-mean' if mm.endswith('-2s') else (tuple(int(t) for t in mm.split('-')[-2:]) if '-a-' in mm else False)
                    auc, fpr, tpr, _ = roc_curve(ind, ood, *[pc / 100 for pc in range(90, 100)], two_sided=two)
                    res[mm] = (auc, float(fpr[5]))
                out['roc'] = res

    with torch.no_grad():
        for i in range(6):          # settle the caching allocator for this model's shapes
            m.evaluate(pool_in[i % 4])
    nat.profile_drain()
    nat.profile_native(True)
    ms = timed(whole, 1)
    nat.profile_native(False)
    ev = nat.profile_drain().get('elbo_eval_fwd', [])
    L, D = wl['ctor']['test_latent_sampling'], int(torch.tensor(shape).prod())
    # algorithmic bytes of the eval kernel per sample (SURVEY 8d): x, L reconstructions (bf16), mu / log_var, z, |eps|^2,
    # outputs (5C + 3) + C logits + 16 scores + 4 predictions
    bytes_eval = D * 4 + L * D * 2 + 2 * K_ * 4 + (L + 1) * K_ * 4 + L * 4 + ((5 * C_ + 3) + C_ + 16 + 4) * 4
    us = sum(ev) / max(1, len(ev)) * 1e3
    r = {'C': C_, 'K': K_, 'L': L, 'samples': n_total, 'samples_per_s': n_total / (ms * 1e-3), 'seconds': ms * 1e-3,
         'includes': 'per-batch evaluate + scores + predictions, final gather (NCCL all_gather when N > 1), device ROC of 11 methods',
         'eval_kernel_us': us, 'eval_kernel_gbs': bytes_eval * B / (us * 1e-6) / 1e9 if us else None}
    if rank == 0 and 'roc' in out:
        r['auc_iws'] = out['roc'].get('iws', (None,))[0]
    del m, buf, preds
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=0)
    ap.add_argument('--cpu-batch', type=int, default=128)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-graph', dest='graph', action='store_false', help='eager launches instead of CUDA-graph replays')
    ap.add_argument('--no-c5', dest='c5', action='store_false', help='skip the 1 Mi-sample sharded scoring run (configs[4])')
    ap.add_argument('--c5-samples', type=int, default=C5_SAMPLES)
    ap.add_argument('--no-extra', dest='extra', action='store_false', help='skip the c3 / c4 train-step sub-results')
    ap.add_argument('--traffic', type=float, default=None, help='ncu dram bytes per launch of the dominant kernel (from profiles/)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the losses and measures of the last timed train step (rank 0's) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'native':
        ap.error('--dump-outputs writes the outputs of the native path')
    wl = WORKLOADS[args.workload]
    if args.impl == 'reference':
        run_reference(args, wl)
    else:
        run_native(args, wl)


if __name__ == '__main__':
    main()
