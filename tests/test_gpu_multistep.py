"""Multi-step training against the UNMODIFIED reference (tests/golden/make_multistep_golden.py: the body of cvae.py:2424-2461
driven for 3 batches with the reference's own Adam, then eval, one more step, eval).  Every step must read the parameters the
previous optimizer step wrote -- the fused Adam updates the flat buffer through a raw pointer, so the bf16 weight arrangements
and the BatchNorm-folded inference weights are re-derived under explicit epochs (engine.PARAM_EPOCH / STATS_EPOCH).

Two detectors of stale derived weights:
  * parity with the reference's trajectory (per-sample losses of steps 2..4, eval after training);
  * self-consistency: a network built from the live state_dict right before a step (all copies fresh by construction)
    computes the same forward as the live network in that step, to fp32 round-off.
test_stale_weights_would_be_caught shows both are sensitive: with the epoch bump disabled they break."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.abs(a - b).max() / max(1e-6, np.abs(b).max()))


def _load(name):
    """the golden as a dict; the torch.rand inputs (multiples of 2^-24) are stored as their 24-bit integers, three
    little-endian bytes per value (tests/golden/make_multistep_golden.py), and decode exactly to the float32 inputs"""
    d = dict(np.load(os.path.join(GOLDEN, name + '.npz')))
    for k in [k for k in d if k.endswith('.u24')]:
        b = d.pop(k).astype(np.uint32)
        d[k[:-4]] = (b[..., 0] | b[..., 1] << 8 | b[..., 2] << 16).astype(np.float32) * np.float32(2 ** -24)
    return d


def _build(pkg, cfg_json, sd):
    kw = json.loads(cfg_json)
    kw['input_shape'] = tuple(kw['input_shape'])
    net = pkg.ClassificationVariationalNetwork(**kw)
    net.load_state_dict(sd)
    return net.to(DEV)


def _drive(pkg, name):
    d = _load(name)
    cfg = str(d['cfg'])
    net = _build(pkg, cfg, {k[3:]: torch.from_numpy(np.asarray(d[k])) for k in d if k.startswith('sd.')})
    T = int(d['steps'])
    t = lambda k: torch.from_numpy(d[k]).to(DEV)
    out = {'d': d, 'errs': [], 'meas': [], 'twin': {}}

    def step(i, batch, current):
        net.encoder.sampling.injected_eps = t(f'eps.{i}')
        losses, measures = net.train_step(t(f'x.{i}'), t(f'y.{i}'), batch=batch, current_measures=current)
        out['errs'].append({k: rel(v.detach().cpu().numpy(), d[f'step{i}.loss.{k}']) for k, v in losses.items()})
        pre = f'step{i}.measure.'
        out['meas'].append({k[len(pre):]: (float(measures[k[len(pre):]]), float(d[k])) for k in d if k.startswith(pre)})
        return losses, measures

    def evaluate(tag):
        net.eval()
        net.encoder.sampling.injected_eps = t('eps_eval')
        with torch.no_grad():
            _, logits, losses, _ = net.evaluate(t('x_eval'))
            e = {k: rel(v.cpu().numpy(), d[f'{tag}.loss.{k}']) for k, v in losses.items()}
            e['logits'] = float(np.abs(logits.float().cpu().numpy() - d[f'{tag}.logits']).max() /
                                max(1.0, np.abs(d[f'{tag}.logits']).max()))
            preds = {m: net.predict_after_evaluate(logits, losses, method=m).cpu().numpy() for m in ('iws', 'closest')}
            # the same evaluation by a network built from the live state (fresh folded weights by construction)
            twin = _build(pkg, cfg, {k: v.detach().clone() for k, v in net.state_dict().items()})
            twin.eval()
            twin.encoder.sampling.injected_eps = t('eps_eval')
            _, _, tl, _ = twin.evaluate(t('x_eval'))
            out['twin'][tag] = max(rel(tl[k].cpu().numpy(), losses[k].cpu().numpy()) for k in ('total', 'kl', 'iws'))
        return e, preds

    net.train()
    cur = {}
    for i in range(T):
        if i == T - 1:
            twin = _build(pkg, cfg, {k: v.detach().clone() for k, v in net.state_dict().items()})
            twin.train()
            twin.encoder.sampling.injected_eps = t(f'eps.{i}')
            _, _, tl, _ = twin.evaluate(t(f'x.{i}'), t(f'y.{i}'), with_beta=True)
            tl = {k: v.detach().cpu().numpy() for k, v in tl.items()}
        losses, cur = step(i, i, cur)
        if i == T - 1:
            out['twin']['train'] = max(rel(losses[k].detach().cpu().numpy(), tl[k]) for k in tl)
    out['sd'] = {k: v.detach().float().cpu().numpy() for k, v in net.state_dict().items()}
    out['eval_a'] = evaluate('eval_a')
    net.train()
    step(T, 0, {})
    out['eval_b'] = evaluate('eval_b')
    return out


@pytest.mark.parametrize('name', ['multistep_conv_cvae_bn', 'multistep_mlp_cvae'])
def test_adam_steps_then_eval_match_reference(pkg, name):
    o = _drive(pkg, name)
    d = o['d']
    # north_star tolerance for bf16 GEMMs on the loss terms of every step; var_kl (a small difference of sums of exp(log_var))
    # carries the bf16 noise of the log-variance head amplified, so it gets 5e-2
    # (later steps inherit the divergence of the parameters, which compounds: 3e-2 from the third step on)
    for i, e in enumerate(o['errs']):
        for k, v in e.items():
            assert v < (5e-2 if k == 'var_kl' else (2e-2 if i < 2 else 3e-2)), (f'step {i}', k, v, e)
    # running measures chained through current_measures / batch index as the reference does (cvae.py:2441-2449); sigma and
    # the dictionary measures are the values BEFORE the step's optimizer update
    for i, m in enumerate(o['meas']):
        for k, (got, want) in m.items():
            assert abs(got - want) <= 2e-2 * max(1.0, abs(want)), (f'step {i}', k, got, want)
    # self-consistency to fp32 round-off (same kernels, same weights -> same sums up to atomics ordering in BN statistics)
    assert o['twin']['train'] < 1e-4, o['twin']
    assert o['twin']['eval_a'] < 1e-4 and o['twin']['eval_b'] < 1e-4, o['twin']
    # parameters after 3 steps moved like the reference's (error judged against the distance travelled); conv biases in front
    # of a train-mode BatchNorm are excluded: their gradient is exactly zero here and rounding noise in the reference
    moved = 0
    for k, v in o['sd'].items():
        want, start = d['sd_after.' + k].astype(np.float64), d['sd.' + k].astype(np.float64)
        if want.dtype.kind != 'f' or 'num_batches' in k:
            continue
        travelled = np.linalg.norm(want - start)
        if travelled < 1e-4 * max(1.0, np.linalg.norm(start)):
            continue
        moved += 1
        assert np.linalg.norm(v - want) <= 0.35 * travelled + 1e-5, (k, np.linalg.norm(v - want), travelled)
    assert moved >= 8
    # evaluation with the BatchNorm running statistics and weights of the moment
    for tag in ('eval_a', 'eval_b'):
        e, preds = o[tag]
        for k, v in e.items():
            assert v < (8e-2 if k == 'var_kl' else (5e-2 if k == 'wmse' else 2e-2)), (tag, k, v)
        # predictions exact wherever the reference's decision margin exceeds the tolerance
        for m, got in preds.items():
            ref = d[f'{tag}.loss.' + ('iws' if m == 'iws' else 'zdist')].astype(np.float64)
            srt = np.sort(ref if m == 'closest' else -ref, axis=0)
            r = ref if m == 'closest' else -ref
            # margin against the part of the loss that differs between classes (the reconstruction term is common to all)
            clear = (srt[1] - srt[0]) > 2 * 5e-2 * np.maximum(1.0, np.abs(r - r.mean(0)).max(0))
            assert clear.mean() > 0.1, clear.mean()
            assert (got[clear] == d[f'{tag}.pred.{m}'][clear]).all(), (tag, m)


def test_stale_weights_would_be_caught(pkg, monkeypatch):
    """the same drive with the epoch bumps disabled = the packed bf16 weights of step 1 and the folded inference weights of
    the first evaluation reused later: both detectors must fire"""
    from jointvae_b200 import conv_engine
    monkeypatch.setattr(pkg.engine, 'bump_params', lambda: None)
    monkeypatch.setattr(pkg.engine, 'bump_stats', lambda: None)
    conv_engine._stacks.clear()
    try:
        o = _drive(pkg, 'multistep_conv_cvae_bn')
    finally:
        conv_engine._stacks.clear()
    assert o['twin']['train'] > 1e-3, o['twin']
    assert max(v for e in o['errs'][1:] for v in e.values()) > 5e-2, o['errs']
