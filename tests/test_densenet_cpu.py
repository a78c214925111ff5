"""torchvision DenseNet features on the native conv engine without a GPU: the dense-block step (one concatenation buffer,
batch statistics computed once per channel, fp32 gradient accumulator) driven through tests/emu_densenet.py with fp32
storage, against torch.nn running the same torchvision modules in fp32.  The CUDA kernels themselves are checked on the GPU
(tests/test_gpu_densenet.py)."""
import copy

import pytest
import torch

from emu_densenet import DenseEmuKernels
from emu_kernels import EmuKernels


@pytest.fixture()
def ce(pkg, monkeypatch):
    from jointvae_b200 import conv_engine
    monkeypatch.setattr(conv_engine, 'K', DenseEmuKernels)
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    conv_engine._stacks.clear()
    yield conv_engine
    conv_engine._stacks.clear()


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


def _features(name, shape, seed):
    from jointvae_b200.module.vae_layers.conv import ResOrDenseNetFeatures
    torch.manual_seed(seed)
    seq = ResOrDenseNetFeatures(name, shape, pretrained=False)
    for m in seq.modules():
        if isinstance(m, torch.nn.Conv2d):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()      # bf16-exact weights: packing does not round
        elif isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.uniform_(0.25, 0.75)
            m.bias.data.uniform_(0.5, 1.0)
    return seq


def _bns(seq):
    return [(k, m) for k, m in seq.named_modules() if isinstance(m, torch.nn.BatchNorm2d)]


@pytest.mark.parametrize('name,shape', [('densenet121', (3, 32, 32)), ('densenet121', (3, 64, 64)),
                                        ('densenet161', (3, 32, 32))])
def test_densenet_train_forward_and_gradients(pkg, ce, name, shape):
    seq = _features(name, shape, 0)
    ref = copy.deepcopy(seq)
    seq.train(), ref.train()
    # at 32 x 32 the last block runs on 1 x 1 maps: with N = 2 every BatchNorm there normalises two values, and channels whose
    # two values nearly agree make torch's own fp32 result depend on the summation order (measured: 0.2 relative between
    # sum-of-squares and two-pass variances at N = 2, 2e-6 at N = 4), so that size uses N = 4
    N = 2 if shape[1] >= 64 else 4
    # inputs from a fixed seed: at N = 2 the BatchNorms of the small maps see 8 to 32 values per channel, and an input that puts
    # one channel next to a ReLU kink or at a near-zero variance moves torch's fp32 gradient itself at the 1e-2 level
    # (measured on four input seeds at 64 x 64: 6e-6 relative on every gradient for three, 1.1e-2 on one conv1 for the fourth)
    x = torch.randn(N, *shape, generator=torch.Generator().manual_seed(5))
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin)
    C = 2208 if name == 'densenet161' else 1024
    assert tuple(got.shape) == tuple(want.shape) == (N, C, shape[1] // 32, shape[2] // 32)
    assert _rel(got, want) < 1e-3, _rel(got, want)
    go = torch.randn_like(want)
    want.backward(go)
    got.backward(go)
    gmax = max(float(p.grad.norm()) for p in ref.parameters())
    for (k, p), (_, q) in zip(seq.named_parameters(), ref.named_parameters()):
        assert p.grad is not None, k
        err = float((p.grad.double() - q.grad.double()).norm())
        assert err <= 5e-3 * float(q.grad.norm()) + 5e-4 * gmax, (k, err, float(q.grad.norm()))
    assert _rel(xin.grad, xr.grad) < 5e-3, _rel(xin.grad, xr.grad)
    # every norm* (each consumer of the shared block statistics) follows torch's running-statistics update
    for (k, m), (_, r) in zip(_bns(seq), _bns(ref)):
        assert float((m.running_mean - r.running_mean).abs().max()) < 1e-4 * (1 + float(r.running_mean.abs().max())), k
        assert float((m.running_var - r.running_var).abs().max()) < 1e-4 * (1 + float(r.running_var.abs().max())), k
        assert int(m.num_batches_tracked) == int(r.num_batches_tracked) == 1, k


def test_densenet_eval_forward_and_input_gradient(pkg, ce):
    """eval mode with randomised running statistics: each norm1 uses its own running statistics, norm2 is folded into conv1
    (bf16 folded weights), and the input gradient (ODIN) goes back through every pre-activation BatchNorm"""
    seq = _features('densenet121', (3, 32, 32), 1)
    for _, m in _bns(seq):
        m.running_mean.uniform_(-0.2, 0.2)
        m.running_var.uniform_(0.5, 1.5)
    seq.eval()
    x = torch.randn(4, 3, 32, 32)
    xr = x.clone().requires_grad_(True)
    want = seq(xr)
    go = torch.randn_like(want)
    want.backward(go)
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin)
    # only the folded conv1 weights are rounded to bf16 (the torch side keeps fp32): 58 of them along the path
    assert _rel(got, want) < 3e-2, _rel(got, want)
    got.backward(go)
    assert xin.grad is not None and _rel(xin.grad, xr.grad) < 0.1, _rel(xin.grad, xr.grad)
    assert all(int(m.num_batches_tracked) == 0 for _, m in _bns(seq))


def test_block_statistics_computed_once_per_channel(pkg, ce, monkeypatch):
    """every statistics launch of a block reads only the channels just written: the block input, then each layer's
    growth channels; no consumer recomputes statistics over its prefix"""
    trace = []
    monkeypatch.setattr(DenseEmuKernels, 'stats_trace', trace)
    seq = _features('densenet121', (3, 32, 32), 2)
    seq.train()
    ce.run(list(seq), torch.randn(2, 3, 32, 32))
    want = []
    for C0 in (64, 128, 256, 512):
        nl = {64: 6, 128: 12, 256: 24, 512: 16}[C0]
        want += [('bn_stats_ld', C0)] + [('bn_stats_ld', 32)] * nl
    assert trace == want


def test_build_routes_densenet_names(pkg, offline_weights):
    from jointvae_b200.module.vae_layers.conv import ResOrDenseNetFeatures
    build = pkg.module.vae_layers.build_de_conv_layers
    f = build((3, 64, 64), 'densenet121', where='input')
    assert isinstance(f, ResOrDenseNetFeatures) and f.output_shape == (1024, 2, 2)
    assert build((3, 32, 32), 'densenet161', where='input').output_shape == (2208, 1, 1)
    assert build((3, 64, 64), 'densenet169', where='input').output_shape == (1664, 2, 2)
    assert build((3, 64, 64), 'densenet201', where='input').output_shape == (1920, 2, 2)


def test_cvae_with_densenet_features_has_torchvision_keys(pkg, offline_weights):
    import torchvision
    from full_cases import _conv, PRIOR
    kw = _conv(20, 256, features='densenet121', upsampler='ivgg', shape=(3, 64, 64), L=8)
    kw['input_shape'] = tuple(kw['input_shape'])
    kw['prior'] = dict(PRIOR)
    net = pkg.ClassificationVariationalNetwork(**kw)
    sd = net.state_dict()
    tv = torchvision.models.densenet121(weights=None).features.state_dict()
    feats = {k[len('features.0.'):]: v.shape for k, v in sd.items() if k.startswith('features.')}
    assert feats == {k: v.shape for k, v in tv.items()}
    assert 'features.0.denseblock1.denselayer1.norm1.weight' in sd
    assert net.encoder.input_shape == (1024, 2, 2) or tuple(net.features.output_shape) == (1024, 2, 2)


def test_densenet_with_unaligned_channel_offsets_raises(pkg, ce):
    from torchvision.models import DenseNet
    net = DenseNet(growth_rate=12, block_config=(2, 2), num_init_features=24)
    with pytest.raises(NotImplementedError, match='multiple of 8'):
        ce.run([net.features], torch.randn(1, 3, 32, 32))


def test_densenet_with_dropout_raises(pkg, ce):
    from torchvision.models import DenseNet
    net = DenseNet(growth_rate=32, block_config=(2, 2), num_init_features=64, drop_rate=0.2)
    with pytest.raises(NotImplementedError, match='drop_rate'):
        ce.run([net.features], torch.randn(1, 3, 32, 32))
