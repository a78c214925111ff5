"""GPU checks of the layers the conv-spec grammar builds beyond strides 1 / 2, 2x up-sampling and tiling average pools:
convolutions and transposed convolutions of stride 3..8 (tap-box kernels for the strided gathers, halo or tap-box kernels for
the s*s sub-pixel phases), jvae_upsample_nearest and jvae_avgpool_pad.  Stacks follow tests/test_gpu_conv.py's protocol
(torch fp32 on the same device, with cuDNN in bf16 beside it as the noise floor of bf16 activations); a cvae built on such
specs trains from a captured CUDA graph like the eager steps (tests/test_gpu_graph.py's protocol), matches the fp32 oracle
in eval mode and produces ODIN scores."""
import numpy as np
import pytest
import torch

import full_cases as fc
import test_gpu_conv as tgc

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


STACKS = [
    # (where, spec, input shape, batch, batch_norm, output_activation)
    ('input', '[x3+1]32x4+0:4-64:3-Ax3+1:2', (3, 32, 32), 64, True, None),      # strides 4, 3 (Wq = 3: tap-box), padded pool
    ('input', '[x3+1]64x4+0:4-128:3-A3+1:2', (3, 64, 64), 32, True, None),      # wide: 128 channels at stride 3
    ('input', '32x8+0:8-160x3+1', (3, 64, 64), 32, True, None),                  # stride 8, then 160 channels
    ('input', '16x5+2:3-24x7+3:4', (3, 47, 45), 16, False, None),                # odd maps, k 5 / 7
    ('input', '8x3+0:4-16', (5, 31, 31), 16, True, None),                        # kernel < stride
    ('input', '16-Ax2-32-A2', (3, 29, 29), 16, True, None),                      # non-tiling pools
    ('output', '[x3+1]32x4+0:4-!32x3+1-U:4-!3x3+1', (64, 2, 2), 64, True, 'linear'),      # transposed stride 4, U:4
    ('output', '[x4+0]128x4+0:4-64x3+0:3++1-!3x3+1', (64, 2, 2), 16, True, 'sigmoid'),   # wide stride 4, stride 3 + op
    ('output', '[x8+0]32x8+0:8-!3x3+1', (16, 3, 3), 16, False, 'linear'),                 # transposed stride 8
    ('output', '[x3+1]16-U:3-!16x3+1-U:4-!3x3+1', (16, 3, 3), 16, True, 'linear'),        # U:3, U:4
]


@pytest.mark.parametrize('where,spec,shape,N,bn,out_act', STACKS)
def test_spec_stack_matches_torch_fp32(pkg, where, spec, shape, N, bn, out_act):
    tgc.test_stack_matches_torch_fp32(pkg, where, spec, shape, N, bn, out_act)


def _nhwc(t, ld):
    n, c, h, w = t.shape
    out = torch.zeros(n, h, w, ld, dtype=torch.bfloat16, device=DEV)
    out[..., :c] = t.permute(0, 2, 3, 1)
    return out


@pytest.mark.parametrize('s,C,ld', [(3, 64, 64), (4, 3, 8), (4, 32, 40), (1, 16, 16), (5, 128, 128)])
def test_upsample_nearest(pkg, s, C, ld):
    nat = pkg._native
    torch.manual_seed(s)
    N, H, W = 5, 7, 6
    x = torch.randn(N, C, H, W, device=DEV).to(torch.bfloat16)
    src = _nhwc(x, ld)
    out = torch.full((N, s * H, s * W, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    nat.upsample_nearest(src, ld, out, ld, N, H, W, ld, s)
    want = torch.nn.functional.interpolate(x, scale_factor=s, mode='nearest')
    assert torch.equal(out[..., :C].permute(0, 3, 1, 2), want)       # a copy: bit-equal
    g = torch.randn(N, C, s * H, s * W, device=DEV).to(torch.bfloat16)
    xr = x.float().requires_grad_(True)
    torch.nn.functional.interpolate(xr, scale_factor=s, mode='nearest').backward(g.float())
    gs = _nhwc(g, ld)
    d1 = torch.full((N, H, W, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    d2 = d1.clone()
    nat.upsample_nearest(gs, ld, d1, ld, N, H, W, ld, s, backward=True)
    nat.upsample_nearest(gs, ld, d2, ld, N, H, W, ld, s, backward=True)
    assert torch.equal(d1, d2), 'the block sums are not reproducible'
    got = d1[..., :C].permute(0, 3, 1, 2).float()
    assert float((got - xr.grad).abs().max()) <= 8e-3 * float(xr.grad.abs().max())      # one bf16 rounding of an fp32 sum


@pytest.mark.parametrize('win,H,W,C,ld', [((3, 3, 2, 2, 1, 1), 32, 32, 64, 64), ((3, 3, 2, 2, 0, 0), 15, 15, 24, 24),
                                          ((2, 2, 2, 2, 0, 0), 7, 7, 3, 8), ((5, 5, 2, 2, 1, 1), 13, 13, 64, 64),
                                          ((3, 5, 3, 5, 0, 0), 3, 5, 512, 512), ((4, 4, 3, 3, 2, 2), 17, 11, 32, 32)])
def test_avgpool_pad(pkg, win, H, W, C, ld):
    nat = pkg._native
    kh, kw, sh, sw, ph, pw = win
    torch.manual_seed(H + kh)
    N = 6
    x = torch.randn(N, C, H, W, device=DEV).to(torch.bfloat16)
    xr = x.float().requires_grad_(True)
    want = torch.nn.functional.avg_pool2d(xr, (kh, kw), (sh, sw), (ph, pw))
    Ho, Wo = want.shape[-2:]
    out = torch.full((N, Ho, Wo, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    nat.avgpool_pad(_nhwc(x, ld), ld, out, ld, N, H, W, ld, kh, kw, sh, sw, ph, pw)
    wd = want.detach()
    assert float((out[..., :C].permute(0, 3, 1, 2).float() - wd).abs().max()) <= 8e-3 * float(wd.abs().max())
    g = torch.randn(N, C, Ho, Wo, device=DEV).to(torch.bfloat16)
    want.backward(g.float())
    gs = _nhwc(g, ld)
    d1 = torch.full((N, H, W, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
    d2 = d1.clone()
    nat.avgpool_pad(gs, ld, d1, ld, N, H, W, ld, kh, kw, sh, sw, ph, pw, backward=True)
    nat.avgpool_pad(gs, ld, d2, ld, N, H, W, ld, kh, kw, sh, sw, ph, pw, backward=True)
    assert torch.equal(d1, d2), 'the window sums are not reproducible'
    got = d1[..., :C].permute(0, 3, 1, 2).float()
    assert float((got - xr.grad).abs().max()) <= 8e-3 * float(xr.grad.abs().max())


# ------------------------------------------------------------------------------------------------ a cvae on such specs
# ('!' convolutions of an upsampler spec default to padding 0, so the example head '!32-...-!3' would shrink the map by 4
# pixels a layer: with '!32x3+1' / '!3x3+1' the imager maps 2 x 2 to 32 x 32)
FEATURES = '[x3+1]32x4+0:4-64:3-A3+1:2'
UPSAMPLER = '[x3+1]32x4+0:4-!32x3+1-U:4-!3x3+1'
CASE = 'spec_layers_cvae'
TOL = 3e-2


@pytest.fixture()
def spec_case(monkeypatch):
    kw = fc._conv(10, 32, features=FEATURES, upsampler=UPSAMPLER, shape=(3, 32, 32), L=4)
    kw['decoder'] = [256]
    monkeypatch.setitem(fc.CASES, CASE, (kw, 32))
    return CASE


def _net(pkg, name, **over):
    torch.manual_seed(0)
    kw = fc.ctor_kwargs(name)
    kw.update(over)
    net = pkg.ClassificationVariationalNetwork(**kw)
    fc.fill_state_(net)
    return net.to(DEV)


def test_spec_cvae_graph_steps_equal_eager_steps(pkg, spec_case):
    g = torch.Generator().manual_seed(3)
    xs = [torch.rand(32, 3, 32, 32, generator=g).to(DEV) for _ in range(7)]
    ys = [torch.randint(0, 10, (32,), generator=g).to(DEV) for _ in range(7)]
    opt = {'optim_type': 'adam', 'lr': 1e-2, 'eps': 1.0, 'weight_decay': 3e-5, 'grad_clipping': 100}
    out = {}
    for mode in ('eager', 'graph'):
        net = _net(pkg, spec_case, optimizer=opt)
        net.train()
        for c in pkg.engine._rng_counters.values():
            c.zero_()
        losses, cur = [], {}
        for i, (x, y) in enumerate(zip(xs, ys)):
            ls, cur = net.train_step(x, y, batch=i, current_measures=cur, graph=(mode == 'graph'))
            losses.append(ls['total'].detach().clone())
        if mode == 'graph':
            assert any('graph' in st for st in net._graphs.values()), 'the step was never captured'
        out[mode] = (losses, {k: v.detach().clone() for k, v in net.state_dict().items()})
    (la, sa), (lb, sb) = out['eager'], out['graph']
    for i, (a, b) in enumerate(zip(la, lb)):
        assert torch.isfinite(a).all()
        rtol = 2e-4 if i < 4 else 5e-3          # steps 2, 3 are the first replays
        assert torch.allclose(a, b, rtol=rtol, atol=1e-3), (i, float((a - b).abs().max()))
    for k in sa:
        assert torch.allclose(sa[k].float(), sb[k].float(), rtol=1e-2, atol=2e-3), (k, float((sa[k].float() - sb[k].float()).abs().max()))


def _relmax(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(1e-6, np.abs(b).max()))


def test_spec_cvae_eval_matches_oracle_and_scores_odin(pkg, spec_case):
    """eval-mode losses / logits of the native network against the same state_dict run in fp32 by oracle/torch_model.py
    (which builds the strided convolutions, padded pools and U:4 from its layer schema), then ODIN scores"""
    out = fc.oracle_outputs(pkg, spec_case, train_backward=False)['eval']
    net = _net(pkg, spec_case)
    x, _, _, eps_te = [t.to(DEV) for t in fc.inputs(spec_case)]
    net.eval()
    net.encoder.sampling.injected_eps = eps_te
    n0 = pkg._native.launch_count()
    with torch.no_grad():
        _, logits, losses, _, mu, _, _ = net.evaluate(x, z_output=True)
    assert pkg._native.launch_count() > n0
    n = lambda t: t.detach().float().cpu().numpy()
    checked = 0
    for k, v in out['losses'].items():
        if k in losses:
            e = _relmax(n(losses[k]), v)
            print(f'eval loss {k}: {e:.2e}')
            assert e < TOL, (k, e)
            checked += 1
    assert checked >= 4
    assert _relmax(n(mu), out['mu']) < TOL
    net.encoder.sampling.injected_eps = None
    scores = net.odin_softmax(x, temps=[1, 1000], eps=[0.0, 0.004])
    assert len(scores) == 4
    for k, v in scores.items():
        assert v.shape == (32,) and torch.isfinite(v).all(), k
