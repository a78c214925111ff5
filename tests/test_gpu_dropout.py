"""Dense-layer dropout on the B200: the keep-mask of jvae_gemm_bf16_dropout against the numpy restatement (tests/philox_ref.py)
element by element, its values and the gradients of jvae_act_dropout_bwd + the two GEMMs against torch fp32 with that mask as
a constant, run-to-run bit equality at a fixed stream position and fresh masks at the next one, and a c1-shaped MLP cvae built
with dropout: eval mode bit-identical to the same weights without dropout, no torch RNG on the training path, a falling loss,
and CUDA-graph replays that follow tests/test_gpu_graph.py's protocol.

Operands are bf16-exact, so the forward differs from torch fp32 only by the bf16 rounding of the stored output (the 4e-3
norm tolerance of tests/test_gpu_layers.py).  The backward stores dz = dy * keep / (1 - p) * act' in bf16 before the two
GEMMs, as the dense backward without dropout does, so its gradients carry one such rounding too: 4e-3 for all three."""
import functools

import numpy as np
import pytest
import torch
from torch import nn
import torch.nn.functional as F

import philox_ref

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
SHAPES = [(128, 512), (2176, 36), (300, 4096), (8704, 1000)]
ACTS = ['linear', 'relu', 'sigmoid', 'leaky']
K_IN = 256
SEED = 0x0123456789ABCDEF


@functools.lru_cache(maxsize=8)
def _words(seed, pos, M, N):
    return philox_ref.dropout_words(seed, pos, np.arange(M), np.arange(N))


def _keep(seed, pos, M, N, p):
    return torch.from_numpy(philox_ref.keep_of(_words(seed, pos, M, N), p)).to(DEV)


def _act(z, act):
    return {'linear': lambda t: t, 'relu': F.relu, 'sigmoid': torch.sigmoid,
            'leaky': lambda t: F.leaky_relu(t, 0.01)}[act](z)


def _operands(M, N, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(M, K_IN, device=DEV, generator=g).to(torch.bfloat16)
    w = (torch.randn(N, K_IN, device=DEV, generator=g) * K_IN ** -0.5).to(torch.bfloat16)
    b = torch.randn(N, device=DEV, generator=g) * 0.5
    return x, w, b


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.mark.parametrize('p', [0.1, 0.5, 0.9])
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('M,N', SHAPES)
def test_forward_mask_is_exact(pkg, M, N, act, p):
    nat = pkg._native
    x, w, b = _operands(M, N)
    pos = 41
    dev_pos = torch.tensor([3], dtype=torch.int64, device=DEV)        # position = host offset + device word
    out = torch.full((M, N), float('nan'), dtype=torch.bfloat16, device=DEV)
    nat.gemm_bf16_dropout(M, N, K_IN, x, K_IN, w, K_IN, p=p, seed=SEED, offset=pos - 3, offset_dev=dev_pos, bias=b,
                          act=nat.ACT[act], out_bf16=out, ldd=N)
    keep = _keep(SEED, pos, M, N, p)
    assert abs(float(keep.float().mean()) - (1 - p)) < 0.05
    assert bool((out[~keep] == 0).all()), 'a dropped element is not zero'
    want = _act(x.float() @ w.float().t() + b, act) / (1 - p)
    e = _rel(out.float()[keep], want[keep])
    print(f'{M}x{N} {act} p={p}: kept {float(keep.float().mean()):.3f}, forward {e:.5f}')
    assert e < 4e-3, e


@pytest.mark.parametrize('M,N', SHAPES)
def test_p_one_gives_zeros(pkg, M, N):
    nat = pkg._native
    x, w, b = _operands(M, N)
    out = torch.full((M, N), 7.0, dtype=torch.bfloat16, device=DEV)
    nat.gemm_bf16_dropout(M, N, K_IN, x, K_IN, w, K_IN, p=1.0, seed=SEED, bias=b, act=nat.ACT['relu'], out_bf16=out, ldd=N)
    assert bool((out == 0).all())
    from jointvae_b200 import engine
    xin = x.float().requires_grad_(True)
    wp, bp = nn.Parameter(w.float()), nn.Parameter(b.clone())
    y = engine._LinearFn.apply(xin, wp, bp, 'sigmoid', torch.bfloat16, 1.0)
    gx, gw, gb = torch.autograd.grad(y, (xin, wp, bp), torch.ones_like(y))
    assert bool((y == 0).all()) and bool((gx == 0).all()) and bool((gw == 0).all()) and bool((gb == 0).all())


def _fwd_bwd(engine, x, w, b, act, p, go, pos):
    engine._rng_counter(torch.device(DEV)).fill_(pos)
    xin = x.float().requires_grad_(True)
    wp, bp = nn.Parameter(w.float()), nn.Parameter(b.clone())
    y = engine._LinearFn.apply(xin, wp, bp, act, torch.bfloat16, p)
    gx, gw, gb = torch.autograd.grad(y, (xin, wp, bp), go)
    return y, gx, gw, gb


@pytest.mark.parametrize('p', [0.1, 0.5])
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('M,N', SHAPES)
def test_backward_matches_torch_with_the_same_mask(pkg, M, N, act, p):
    from jointvae_b200 import engine
    torch.manual_seed(5)
    seed = torch.initial_seed()
    x, w, b = _operands(M, N, seed=1)
    go = torch.randn(M, N, device=DEV).to(torch.bfloat16)
    pos = 1000
    n0 = pkg._native.launch_count()
    y, gx, gw, gb = _fwd_bwd(engine, x, w, b, act, p, go, pos)
    assert pkg._native.launch_count() > n0
    assert int(engine._rng_counter(torch.device(DEV))[0]) == pos + 1
    keep = _keep(seed, pos, M, N, p).float()
    xr = x.float().requires_grad_(True)
    wr, br = w.float().requires_grad_(True), b.clone().requires_grad_(True)
    yr = _act(xr @ wr.t() + br, act) * keep / (1 - p)
    gxr, gwr, gbr = torch.autograd.grad(yr, (xr, wr, br), go.float())
    e = [_rel(y.float(), yr), _rel(gx, gxr), _rel(gw, gwr), _rel(gb, gbr)]
    print(f'{M}x{N} {act} p={p}: forward {e[0]:.5f} dx {e[1]:.5f} dW {e[2]:.5f} db {e[3]:.5f}')
    assert max(e) < 4e-3, e


@pytest.mark.parametrize('M,N', [(2176, 36), (8704, 1000)])
def test_same_position_is_bit_identical_next_position_is_fresh(pkg, M, N):
    from jointvae_b200 import engine
    torch.manual_seed(9)
    seed = torch.initial_seed()
    x, w, b = _operands(M, N, seed=2)
    go = torch.randn(M, N, device=DEV).to(torch.bfloat16)
    a = _fwd_bwd(engine, x, w, b, 'relu', 0.3, go, 77)
    c = _fwd_bwd(engine, x, w, b, 'relu', 0.3, go, 77)
    for u, v in zip(a, c):
        assert torch.equal(u, v)
    # consecutive calls: the counter moved on, so the second call draws the mask of position 78
    engine._rng_counter(torch.device(DEV)).fill_(77)
    xin = x.float()
    wp, bp = nn.Parameter(w.float()), nn.Parameter(b.clone())
    y1 = engine._LinearFn.apply(xin, wp, bp, 'sigmoid', torch.bfloat16, 0.3)
    y2 = engine._LinearFn.apply(xin, wp, bp, 'sigmoid', torch.bfloat16, 0.3)
    assert torch.equal(y1 != 0, _keep(seed, 77, M, N, 0.3)) and torch.equal(y2 != 0, _keep(seed, 78, M, N, 0.3))
    assert float((y1 != 0).ne(y2 != 0).float().mean()) > 0.3


# ------------------------------------------------------------------------------------------------ a c1-shaped cvae with dropout
PRIOR = {'init_mean': 1.0, 'learned_means': True, 'var_dim': 'scalar', 'seed': 1}


def _c1(pkg, dropout, lr=1e-3, eps=1e-8):
    torch.manual_seed(0)
    return pkg.ClassificationVariationalNetwork(
        (1, 28, 28), 10, type='cvae', encoder=[512, 256], decoder=[256, 512], classifier=[], latent_dim=16,
        latent_sampling=1, test_latent_sampling=1, gamma=0, beta=1.0, output_activation='sigmoid', sigma={'value': 0.1},
        prior=dict(PRIOR), dropout=dropout,
        optimizer={'optim_type': 'adam', 'lr': lr, 'eps': eps, 'weight_decay': 3e-5, 'grad_clipping': 100}).to(DEV)


def _batches(n, B=128, seed=3):
    g = torch.Generator().manual_seed(seed)
    return ([torch.rand(B, 1, 28, 28, generator=g).to(DEV) for _ in range(n)],
            [torch.randint(0, 10, (B,), generator=g).to(DEV) for _ in range(n)])


def _zero_positions(engine):
    for c in engine._rng_counters.values():
        c.zero_()


def test_c1_eval_is_bit_identical_to_no_dropout(pkg):
    from jointvae_b200 import engine
    net_d, net_p = _c1(pkg, 0.3), _c1(pkg, False)
    assert sum(isinstance(m, nn.Dropout) for m in net_d.modules()) == 4
    with torch.no_grad():
        sd_d = net_d.state_dict()
        for k, v in net_p.state_dict().items():      # prior, sigma and the imager / heads keep their names
            if k in sd_d:
                v.copy_(sd_d[k])
        lin_d = [m for m in net_d.modules() if isinstance(m, nn.Linear)]
        lin_p = [m for m in net_p.modules() if isinstance(m, nn.Linear)]
        assert [m.weight.shape for m in lin_d] == [m.weight.shape for m in lin_p]
        for a, c in zip(lin_d, lin_p):               # the Sequential indices differ: copy layer by layer
            c.weight.copy_(a.weight)
            c.bias.copy_(a.bias)
    engine.bump_params()
    (x,), _ = _batches(1)
    res = []
    for net in (net_d, net_p):
        net.eval()
        _zero_positions(engine)
        with torch.no_grad():
            xr, logits, losses, _ = net.evaluate(x)
        res.append((xr, losses))
    (xa, la), (xb, lb) = res
    assert torch.equal(xa, xb)
    for k in la:
        if torch.is_tensor(la[k]):
            assert torch.equal(la[k], lb[k]), k


def test_c1_training_uses_no_torch_rng_and_learns(pkg):
    from jointvae_b200 import engine
    net = _c1(pkg, 0.3)
    net.train()
    xs, ys = _batches(1)
    x, y = xs[0], ys[0]
    losses = []
    for i in range(20):
        rng = torch.cuda.get_rng_state()
        n0 = pkg._native.launch_count()
        ls, _ = net.train_step(x, y, batch=i)
        assert pkg._native.launch_count() > n0
        assert torch.equal(torch.cuda.get_rng_state(), rng), 'a torch RNG draw on the training path'
        losses.append(float(ls['total'].detach().mean()))
    print('c1 dropout=0.3 losses:', ' '.join(f'{v:.1f}' for v in losses))
    assert np.isfinite(losses).all()
    # uniform noise images: most of the loss is the irreducible 1/12 pixel variance over sigma^2, so it falls by a few percent
    # (measured on the B200: 2255 -> 2180 over the 20 steps, every step lower than the one before)
    assert np.mean(losses[-3:]) < 0.99 * np.mean(losses[:3]), losses


def test_c1_graph_replays_match_eager_steps(pkg):
    """tests/test_gpu_graph.py's protocol on the dropout model: two identical networks from the same Philox position, one
    stepping eagerly, one through the graph; the replays draw the masks of the positions the eager steps draw.  lr 1e-3:
    at that file's 1e-2 two EAGER runs of this model already differ by up to 4.6e-4 relative at step 3 (measured on the
    B200, with and without dropout), more than the protocol allows the first replays; at 1e-3 the first replay is
    bit-identical to the eager step and the later ones differ by at most 5.4e-4."""
    from jointvae_b200 import engine
    xs, ys = _batches(7, seed=4)
    out = {}
    for mode in ('eager', 'graph'):
        net = _c1(pkg, 0.3, lr=1e-3, eps=1.0)
        net.train()
        _zero_positions(engine)
        losses, cur = [], {}
        for i, (x, y) in enumerate(zip(xs, ys)):
            ls, cur = net.train_step(x, y, batch=i, current_measures=cur, graph=(mode == 'graph'))
            losses.append(ls['total'].detach().clone())
            meas = dict(cur)
        if mode == 'graph':
            assert any('graph' in st for st in net._graphs.values()), 'the step was never captured'
        pos = int(engine._rng_counter(torch.device(DEV))[0])
        net.eval()
        with torch.no_grad():
            net.encoder.sampling.injected_eps = torch.zeros(2, 128, 16, device=DEV)
            _, _, ev, _ = net.evaluate(xs[0])
        out[mode] = (losses, {k: v.detach().clone() for k, v in net.state_dict().items()}, meas, ev['total'].clone(), pos)
    (la, sa, ma, ea, pa), (lb, sb, mb, eb, pb) = out['eager'], out['graph']
    assert pa == pb and pa > 0          # every replay advanced the device position as the eager step did
    for i, (a, b) in enumerate(zip(la, lb)):
        rtol = 2e-4 if i < 4 else 5e-3          # steps 2, 3 are the first replays
        assert torch.allclose(a, b, rtol=rtol, atol=1e-3), (i, float((a - b).abs().max()))
    for k in sa:
        assert torch.allclose(sa[k].float(), sb[k].float(), rtol=1e-2, atol=2e-3), (k, float((sa[k].float() - sb[k].float()).abs().max()))
    for k in ma:
        assert abs(ma[k] - mb[k]) <= 5e-3 * max(1.0, abs(ma[k])), (k, ma[k], mb[k])
    assert torch.allclose(ea, eb, rtol=5e-3, atol=1e-2)
