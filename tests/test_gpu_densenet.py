"""torchvision DenseNet features on the B200 (conv_engine.DenseBlockStep: one concatenation buffer per block, batch statistics
once per channel, fp32 gradient accumulator; csrc/norm.cu: jvae_bn_stats_ld / jvae_bn_preact_fwd / jvae_bn_preact_bwd /
jvae_cast_f32_bf16_ld), against torch fp32 on the same device, with cuDNN's bf16 path on the same modules as the noise floor of
bf16 activations; and a c4-shaped cvae with densenet121 features against the fp32 oracle run live."""
import copy

import numpy as np
import pytest
import torch

import full_cases as fc

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 2e-2


@pytest.fixture()
def offline_weights(monkeypatch):
    """the wrapper's default pretrained=True would try a download: build the torchvision DenseNets without weights"""
    import torchvision.models as tvm
    for name in ('densenet121', 'densenet161', 'densenet169', 'densenet201'):
        orig = getattr(tvm, name)
        monkeypatch.setattr(tvm, name, lambda *a, _orig=orig, **k: _orig(weights=None))


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / max(1e-12, float(b.norm())))


def _bns(seq):
    return [m for m in seq.modules() if isinstance(m, torch.nn.BatchNorm2d)]


def _features(pkg, name, shape):
    from jointvae_b200.module.vae_layers.conv import ResOrDenseNetFeatures
    torch.manual_seed(0)
    seq = ResOrDenseNetFeatures(name, shape, pretrained=False)
    fc.fill_state_(seq)              # well-conditioned BatchNorm parameters (scale 0.25..0.75, shift 0.5..1)
    for m in seq.modules():
        if isinstance(m, torch.nn.Conv2d):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()
    return seq.to(DEV)


@pytest.mark.parametrize('name,shape,N', [('densenet121', (3, 64, 64), 16), ('densenet121', (3, 32, 32), 32),
                                          ('densenet161', (3, 32, 32), 32)])
def test_features_train_match_torch_fp32(pkg, name, shape, N):
    from jointvae_b200 import conv_engine as ce
    seq = _features(pkg, name, shape)
    ref, lib = copy.deepcopy(seq), copy.deepcopy(seq)
    seq.train(), ref.train(), lib.train()
    x = torch.randn(N, *shape, device=DEV, generator=torch.Generator(DEV).manual_seed(1)).to(torch.bfloat16).float()
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    xin = x.clone().requires_grad_(True)
    n0 = pkg._native.launch_count()
    got = ce.run(list(seq), xin)
    assert pkg._native.launch_count() > n0
    assert tuple(got.shape) == tuple(want.shape)
    xl = x.clone().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    with torch.autocast(device_type='cuda', dtype=torch.bfloat16):
        lo = lib(xl)
    ef, ef_lib = _rel(got, want), _rel(lo.float(), want)
    print(f'{name} {shape} N={N} forward: native {ef:.2e}, cudnn-bf16 {ef_lib:.2e}')
    assert ef < max(2e-2, 1.5 * ef_lib), (ef, ef_lib)
    go = torch.randn_like(want)
    want.backward(go)
    lo.backward(go.to(lo.dtype))
    got.backward(go)
    ex, ex_lib = _rel(xin.grad, xr.grad), _rel(xl.grad, xr.grad)
    print(f'{name} input gradient: native {ex:.2e}, cudnn-bf16 {ex_lib:.2e}')
    assert ex < max(2e-2, 1.5 * ex_lib), (ex, ex_lib)
    gmax = max(float(p.grad.norm()) for p in ref.parameters())
    report = []
    for (k, p), (_, q), (_, l) in zip(seq.named_parameters(), ref.named_parameters(), lib.named_parameters()):
        assert p.grad is not None and torch.isfinite(p.grad).all(), k
        err = float((p.grad.double() - q.grad.double()).norm())
        err_lib = float((l.grad.double() - q.grad.double()).norm())
        report.append((k, err, err_lib, float(q.grad.norm())))
    worst = sorted(report, key=lambda r: r[1] / max(1e-12, r[3]), reverse=True)[:8]
    print(f'{name} worst parameter gradients (name, native, cudnn-bf16, |ref|):',
          [(k, f'{e:.3e}', f'{el:.3e}', f'{nr:.3e}') for k, e, el, nr in worst])
    print(f'{name} median relative gradient error: native {np.median([e / max(1e-12, nr) for _, e, _, nr in report]):.2e}, '
          f'cudnn-bf16 {np.median([el / max(1e-12, nr) for _, _, el, nr in report]):.2e}')
    for k, err, err_lib, nr in report:
        assert err <= max(2e-2 * nr + 1e-3 * gmax, 2.0 * err_lib), (k, err, err_lib, nr)
    for m, r in zip(_bns(seq), _bns(ref)):
        assert float((m.running_mean - r.running_mean).abs().max()) < 2e-2 * max(1.0, float(r.running_mean.abs().max()))
        assert _rel(m.running_var, r.running_var) < 2e-2
        assert int(m.num_batches_tracked) == 1


def test_features_eval_forward_and_input_gradient(pkg):
    """eval mode (ODIN): norm1 / tail BatchNorms with their own running statistics, norm2 folded into conv1"""
    from jointvae_b200 import conv_engine as ce
    seq = _features(pkg, 'densenet121', (3, 32, 32))
    seq.eval()
    ref, lib = copy.deepcopy(seq), copy.deepcopy(seq)
    x = torch.randn(32, 3, 32, 32, device=DEV, generator=torch.Generator(DEV).manual_seed(2)).to(torch.bfloat16).float()
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    go = torch.randn_like(want)
    want.backward(go)
    xl = x.clone().requires_grad_(True)
    with torch.autocast(device_type='cuda', dtype=torch.bfloat16):
        lo = lib(xl)
    lo.backward(go.to(lo.dtype))
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin)
    got.backward(go)
    ef, ef_lib = _rel(got, want), _rel(lo.float(), want)
    ex, ex_lib = _rel(xin.grad, xr.grad), _rel(xl.grad, xr.grad)
    print(f'eval densenet121: forward native {ef:.2e} cudnn-bf16 {ef_lib:.2e}; input gradient native {ex:.2e} '
          f'cudnn-bf16 {ex_lib:.2e}')
    assert ef < max(2e-2, 1.5 * ef_lib) and ex < max(2e-2, 1.5 * ex_lib), (ef, ef_lib, ex, ex_lib)
    assert all(int(m.num_batches_tracked) == 0 for m in _bns(seq))


CASE = 'full_c4_densenet121'


@pytest.fixture()
def densenet_case(monkeypatch, offline_weights):
    monkeypatch.setitem(fc.CASES, CASE, (fc._conv(20, 256, features='densenet121', upsampler='ivgg', shape=(3, 64, 64), L=8),
                                         16))
    return CASE


def _net(pkg, name):
    torch.manual_seed(0)
    net = pkg.ClassificationVariationalNetwork(**fc.ctor_kwargs(name))
    fc.fill_state_(net)
    return net.to(DEV)


def _relmax(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(1e-6, np.abs(b).max()))


def _n(t):
    return t.detach().float().cpu().numpy()


def test_densenet_cvae_matches_oracle(pkg, densenet_case):
    """the c4 architecture with densenet121 features at B = 16 against the fp32 oracle (torchvision modules in fp32, what the
    reference runs): eval losses / logits / predictions, training losses and every parameter gradient; gradient tolerance 2e-2
    or 1.5 x the error of a generic bf16 pipeline on the same network (tests/test_gpu_baseline_configs.py)"""
    import os
    name = densenet_case
    torch.set_num_threads(max(1, min(16, os.cpu_count() or 1)))
    out = fc.oracle_outputs(pkg, name)
    floor = fc.oracle_outputs(pkg, name, bf16_operands=True)['train']
    net = _net(pkg, name)
    x, y, eps_tr, eps_te = [t.to(DEV) for t in fc.inputs(name)]
    net.eval()
    net.encoder.sampling.injected_eps = eps_te
    with torch.no_grad():
        xr, logits, losses, _, mu, lv, z = net.evaluate(x, z_output=True)
    ev = out['eval']
    for k, v in ev['losses'].items():
        if k in losses:
            e = _relmax(_n(losses[k]), v)
            print(f'eval loss {k}: {e:.2e}')
            assert e < TOL, (k, e)
    assert _relmax(_n(logits), ev['logits']) < TOL
    assert _relmax(_n(mu), ev['mu']) < TOL
    # predictions (loss method): equal wherever the oracle's own decision margin clears the tolerance
    ref_tot = np.asarray(ev['losses']['total'], np.float64)
    srt = np.sort(ref_tot, axis=0)
    clear = (srt[1] - srt[0]) > 2 * TOL * np.maximum(1.0, np.abs(ref_tot - ref_tot.mean(0)).max(0))
    got_pred = net.predict_after_evaluate(logits, losses, method='loss').cpu().numpy()
    assert (got_pred[clear] == ref_tot.argmin(0)[clear]).all()
    print(f'predictions: {clear.mean():.3f} of the samples clear the margin')

    tr = out['train']
    net.train()
    net.encoder.sampling.injected_eps = eps_tr
    net.optimizer.zero_grad()
    n0 = pkg._native.launch_count()
    xr, logits, losses, meas, mu, lv, z = net.evaluate(x, y, with_beta=True, z_output=True)
    assert pkg._native.launch_count() > n0
    for k, v in tr['losses'].items():
        if k in losses:
            e = _relmax(_n(losses[k]), v)
            print(f'train loss {k}: {e:.2e}')
            assert e < TOL, (k, e)
    losses['total'].mean().backward()
    rows = []
    for k, p in net.named_parameters():
        if k not in tr['grads'] or p.grad is None:
            continue
        g_ref = tr['grads'][k].astype(np.float64)
        nr = np.linalg.norm(g_ref)
        if nr == 0:
            continue
        e = np.linalg.norm(_n(p.grad) - g_ref) / nr
        fl = np.linalg.norm(floor['grads'][k] - g_ref) / nr
        rows.append((k, e, fl))
    rows.sort(key=lambda r: r[1] / max(TOL, 1.5 * r[2]), reverse=True)
    print('worst gradients (name, native, generic-bf16 floor):', [(k, f'{e:.2e}', f'{f:.2e}') for k, e, f in rows[:8]])
    assert len(rows) > 300
    for k, e, fl in rows:
        assert e < max(TOL, 1.5 * fl), (k, e, fl)


def test_densenet_cvae_graph_replays_equal_eager(pkg, densenet_case):
    """train_step(graph=True) on the DenseNet cvae: the replayed steps equal the eager ones, and every eager step runs native
    kernels.  As in tests/test_gpu_graph.py, two eager runs of the same seed already differ (fp32 atomics in the weight
    gradients, amplified by the bf16 roundings of the following steps); this network has 120 BatchNorms and 15.8 k-sized losses,
    so the bound is that run-to-run spread measured here (a second eager run), not a fixed relative tolerance."""
    g = torch.Generator().manual_seed(3)
    B = 16
    xs = [torch.rand(B, 3, 64, 64, generator=g).to(DEV) for _ in range(5)]
    ys = [torch.randint(0, 20, (B,), generator=g).to(DEV) for _ in range(5)]
    out = {}
    for mode in ('eager', 'eager2', 'graph'):
        net = _net(pkg, densenet_case)
        net.train()
        for c in pkg.engine._rng_counters.values():
            c.zero_()
        losses, cur = [], {}
        for i, (x, y) in enumerate(zip(xs, ys)):
            n0 = pkg._native.launch_count()
            ls, cur = net.train_step(x, y, batch=i, current_measures=cur, graph=(mode == 'graph'))
            torch.cuda.synchronize()
            assert pkg._native.launch_count() > n0 or mode == 'graph'
            losses.append(ls['total'].detach().clone())
        if mode == 'graph':
            assert any('graph' in st for st in net._graphs.values()), 'the step was never captured'
        out[mode] = losses
    for i, (a, a2, b) in enumerate(zip(out['eager'], out['eager2'], out['graph'])):
        spread = float((a - a2).abs().max())
        err = float((a - b).abs().max())
        print(f'step {i}: graph - eager {err:.3e}, eager - eager {spread:.3e}, |loss| {float(a.abs().max()):.1f}')
        assert err <= max(2e-4 * float(a.abs().max()) + 1e-3, 2.0 * spread), (i, err, spread)
