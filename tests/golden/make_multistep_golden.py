"""Multi-step training golden from the UNMODIFIED reference (build container only):

    python tests/golden/make_multistep_golden.py

The body of the reference's batch loop (cvae.py:2424-2461) -- zero_grad, evaluate(x, y, batch=i, with_beta=True,
current_measures=...), total.mean().backward(), optimizer.clip, optimizer.step -- is driven for 3 batches on a conv + BatchNorm
cvae with its own Optimizer (Adam, L2 weight decay, clipping), then eval, then one more train step, then eval again.  Every
step re-reads the live parameters (and, in eval, the BatchNorm running statistics the training steps moved), so a product
whose packed / folded weight copies go stale after the first optimizer step cannot match.  The learning rates make the
steps matter (the loss falls by a third in three steps).  The conv case runs Adam with eps = 1 (a keyword the reference's
Optimizer forwards to torch.optim.Adam, optimizers.py:44): updates are then proportional to the gradient, so the trajectory is
a well-conditioned function of the gradients; with the default eps the first Adam steps are sign(g) * lr per element, which turns
bf16-level gradient noise on near-zero elements into full-size steps (the MLP case keeps the default eps).

Stored: per step the per-sample losses, the chained running measures and the batch-mean losses; the state_dict after step 3;
the per-class eval losses / logits after step 3 and after step 4.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from make_golden import CASES, import_reference, injected_noise, t2n  # noqa: E402

STEPS = 3
OPT = {'optim_type': 'adam', 'lr': 1e-2, 'weight_decay': 3e-5, 'grad_clipping': 100}


def run(cvae_mod, base, name, B, opt=None):
    kw = json.loads(json.dumps(CASES[base]))
    kw['optimizer'] = dict(opt or OPT)
    ctor = json.loads(json.dumps(kw))
    ctor['input_shape'] = tuple(ctor['input_shape'])
    torch.manual_seed(4321)
    model = cvae_mod.ClassificationVariationalNetwork(**ctor)
    C, K = kw['num_labels'], kw['latent_dim']
    Ltr, Lte = kw['latent_sampling'], kw['test_latent_sampling']
    g = torch.Generator().manual_seed(7)
    out = {'cfg': np.array(json.dumps(kw)), 'steps': np.array(STEPS)}
    for k, v in model.state_dict().items():
        out['sd.' + k] = t2n(v)
    xs = [torch.rand(B, *ctor['input_shape'], generator=g) for _ in range(STEPS + 1)]
    ys = [torch.randint(0, C, (B,), generator=g) for _ in range(STEPS + 1)]
    eps = [torch.randn(Ltr + 1, B, K, generator=g) for _ in range(STEPS + 1)]
    eps_te = torch.randn(Lte + 1, B, K, generator=g)
    x_te = torch.rand(B, *ctor['input_shape'], generator=g)
    out['x_eval'], out['eps_eval'] = t2n(x_te), t2n(eps_te)
    opt = model.optimizer
    current = {}

    def train_step(i, batch_index):
        nonlocal current
        out[f'x.{i}'], out[f'y.{i}'], out[f'eps.{i}'] = t2n(xs[i]), t2n(ys[i]), t2n(eps[i])
        opt.zero_grad()
        with injected_noise(eps[i]):
            _, _, losses, measures = model.evaluate(xs[i], ys[i], batch=batch_index, with_beta=True, kl_var_weighting=1.0,
                                                    gamma_weighting=1.0, current_measures=current)
        current = measures
        for k, v in losses.items():
            out[f'step{i}.loss.{k}'] = t2n(v)
        for k, v in measures.items():
            out[f'step{i}.measure.{k}'] = np.array(float(v))
        losses['total'].mean().backward()
        opt.clip(model.parameters())
        opt.step()

    def evaluate(tag):
        model.eval()
        with torch.no_grad(), injected_noise(eps_te):
            _, logits, losses, _ = model.evaluate(x_te)
        for k, v in losses.items():
            out[f'{tag}.loss.{k}'] = t2n(v)
        out[f'{tag}.logits'] = t2n(logits)
        out[f'{tag}.pred.iws'] = t2n(model.predict_after_evaluate(logits, losses, method='iws'))
        out[f'{tag}.pred.closest'] = t2n(model.predict_after_evaluate(logits, losses, method='closest'))

    model.train()
    for i in range(STEPS):
        train_step(i, i)
    for k, v in model.state_dict().items():
        out['sd_after.' + k] = t2n(v)
    evaluate('eval_a')
    model.train()
    current = {}
    train_step(STEPS, 0)
    evaluate('eval_b')
    # torch.rand draws are multiples of 2^-24: each input value is stored exactly as its 24-bit integer in three
    # little-endian bytes, which keeps the conv case's file under 1 MB (tests/test_gpu_multistep.py decodes them)
    for k in [k for k in out if k.startswith('x.') or k == 'x_eval']:
        u = np.round(out.pop(k).astype(np.float64) * 2 ** 24).astype('<u4')
        out[k + '.u24'] = u[..., None].view(np.uint8)[..., :3].copy()
    path = os.path.join(HERE, name + '.npz')
    np.savez_compressed(path, **out)
    print(name, 'ok', '%.1f KB' % (os.path.getsize(path) / 1024),
          [float(out[f'step{i}.loss.total'].mean()) for i in range(STEPS + 1)])


if __name__ == '__main__':
    os.chdir('/tmp')
    mod = import_reference()
    torch.set_num_threads(1)
    run(mod, 'conv_cvae_bn', 'multistep_conv_cvae_bn', 64, opt=dict(OPT, eps=1.0))
    run(mod, 'mlp_cvae', 'multistep_mlp_cvae', 32)
