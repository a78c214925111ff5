"""Host logic of the native convolution path (joint-vae_b200/conv_engine.py) without a GPU: the stack compiler, tap
tables, sub-pixel phases of strided transposed convolutions, weight arrangements, BatchNorm forward / backward algebra
and layouts are driven through tests/emu_kernels.py (a torch emulation of the C-ABI entry points, same arguments) and
compared with torch.nn running the same nn.Sequential in fp32.  The CUDA kernels themselves are checked on the GPU
(tests/test_gpu_conv.py, jvae_selftest)."""
import copy

import numpy as np
import pytest
import torch

from emu_kernels import EmuKernels


@pytest.fixture()
def ce(pkg, monkeypatch):
    from jointvae_b200 import conv_engine
    monkeypatch.setattr(conv_engine, 'K', EmuKernels)
    conv_engine._stacks.clear()
    return conv_engine


def _rel(a, b):
    a, b = a.detach().float().double(), b.detach().float().double()
    return float((a - b).norm() / max(1e-9, float(b.norm())))


CASES = [
    # (where, spec, input shape, batch_norm, output_activation)
    ('input', '[x3-Mx2]8-M-16-16-M-Ax1', (3, 8, 8), True, None),
    ('input', '[x3-Mx2]8-M-24', (3, 12, 12), False, None),
    ('input', '[x5+2]8-8:2-16-16:2-20x2+0', (3, 8, 8), True, None),
    ('input', '16x3+1:2-8x5+2', (5, 9, 9), False, None),            # odd sizes through a stride-2 conv
    ('output', '[x5+2]16x4+0-16-16:2++1-8-!3x5+2', (12, 1, 1), True, 'linear'),
    ('output', '[x5+2]16x4+0-8:2++1-!3x5+2', (12, 1, 1), False, 'sigmoid'),
    ('output', '[x3+1]8-8:2++1-!2x3+1', (6, 3, 3), True, 'sigmoid'),
    ('output', '[!x3+1-U:2]U-!8-U-!3', (4, 2, 2), True, 'linear'),
    ('output', '[x4+1]8x4+1:2-!3x3+1', (6, 3, 3), False, 'linear'),  # even kernel, stride 2, no output padding
    ('output', '[x3+1]24x4+0-!3x3+1', (12, 1, 1), False, 'linear'),   # 24 -> 3 image head: role-swapped weight gradient
    ('output', '[x5+2]24x4+0-24-!3x5+2', (12, 1, 1), True, 'sigmoid'),
    ('output', '[x5+2]40x4+0-24-!3x5+2', (12, 1, 1), True, 'linear'),    # 40 -> 24 stride-1 deconv (64- / 32-channel blocks)
    # activation = leaky (config.ini:113 of the reference), with and without BatchNorm
    ('input/leaky', '[x5+2]8-8:2-16', (3, 8, 8), True, None),
    ('input/leaky', '[x3-Mx2]8-M-24', (3, 12, 12), False, None),
    ('output/leaky', '[x5+2]16x4+0-16:2++1-!3x5+2', (12, 1, 1), True, 'linear'),
    ('output/leaky', '[x5+2]16x4+0-8:2++1-!3x5+2', (12, 1, 1), False, 'sigmoid'),
]


# fp32 storage in the emulation isolates the host logic (only the bf16 weight packing rounds): tight tolerance.
# bf16 storage is what the kernels do: at these tiny batch sizes BatchNorm backward and max-pool routing amplify the
# activation rounding (the error shrinks with the number of pixels per channel), so the tolerance is loose.
@pytest.mark.parametrize('store,tol_f,tol_g', [(torch.float32, 1e-4, 1e-3), (torch.bfloat16, 2e-2, 0.25)])
@pytest.mark.parametrize('where,spec,shape,bn,out_act', CASES)
def test_stack_matches_torch(pkg, ce, monkeypatch, where, spec, shape, bn, out_act, store, tol_f, tol_g):
    monkeypatch.setattr(EmuKernels, 'store', store)
    monkeypatch.setattr(EmuKernels, 'act_dtype', store)
    torch.manual_seed(0)
    build = pkg.module.vae_layers.build_de_conv_layers
    where, _, act = where.partition('/')
    kw = dict(output_activation=out_act) if where == 'output' else {}
    seq = build(shape, spec, batch_norm=bn, where=where, activation=act or 'relu', **kw)
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
        elif hasattr(m, 'weight'):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()      # bf16-exact weights: packing does not round
    ref = copy.deepcopy(seq)
    seq.train(), ref.train()
    N = 3
    x = torch.randn(N, *shape)
    x = x.to(torch.bfloat16).float()          # the native path stores activations in bf16
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    xin = x.clone().requires_grad_(where == 'output')
    got = ce.run(list(seq), xin, image_out=(where == 'output'))
    assert tuple(got.shape) == tuple(want.shape)
    assert _rel(got, want) < tol_f, _rel(got, want)
    go = torch.randn_like(want)
    want.backward(go)
    if where == 'output':
        g = go.to(store).contiguous(memory_format=torch.channels_last)
        assert got.dtype == store and got.is_contiguous(memory_format=torch.channels_last)
    else:
        g = go
    got.backward(g)
    names = dict(ref.named_parameters())
    gmax = max(float(p.grad.norm()) for p in names.values())
    for (k, p), (_, q) in zip(seq.named_parameters(), ref.named_parameters()):
        assert p.grad is not None, k
        err = float((p.grad.double() - q.grad.double()).norm())
        assert err <= tol_g * float(q.grad.norm()) + 0.1 * tol_g * gmax, (k, err, float(q.grad.norm()))
    if where == 'output':
        assert _rel(xin.grad, xr.grad) < tol_g
    # BatchNorm running statistics follow torch's update rule
    for m, r in zip(seq, ref):
        if isinstance(m, torch.nn.BatchNorm2d):
            assert _rel(m.running_mean, r.running_mean) < 2e-2 or float((m.running_mean - r.running_mean).abs().max()) < 2e-3
            assert _rel(m.running_var, r.running_var) < 2e-2
            assert int(m.num_batches_tracked) == int(r.num_batches_tracked) == 1


def test_eval_mode_uses_running_stats(pkg, ce):
    torch.manual_seed(1)
    seq = pkg.module.vae_layers.build_de_conv_layers((3, 8, 8), '[x3-Mx2]8-M-16', batch_norm=True, where='input')
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.uniform_(-0.2, 0.2)
            m.running_var.uniform_(0.5, 1.5)
    seq.eval()
    x = torch.randn(2, 3, 8, 8).to(torch.bfloat16).float()
    with torch.no_grad():
        want = seq(x)
        got = ce.run(list(seq), x)
    assert _rel(got, want) < 2e-2


def test_phase_tables_cover_every_tap_once(pkg):
    from jointvae_b200 import conv_engine as c
    for k, p, s in [(5, 2, 2), (4, 1, 2), (3, 1, 2), (5, 2, 1), (8, 0, 1)]:
        ops = c.deconv_form(k, p, s, 16, 16)
        idx = sorted(i for op in ops for i in op['idx'])
        assert idx == list(range(k * k))
        assert len(ops) == s * s


def test_unsupported_layers_raise(pkg, ce):
    seq = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 3, padding=1), torch.nn.LeakyReLU(0.2))
    with pytest.raises(NotImplementedError):
        ce.run(list(seq), torch.randn(1, 3, 4, 4))


@pytest.mark.parametrize('spec,shape,act', [('[x3-Mx2]8-M-16', (3, 8, 8), 'relu'), ('[x5+2]8-8:2-16', (3, 8, 8), 'leaky'),
                                            ('[x3+1]8-8-M-16:2-16', (3, 16, 16), 'relu')])
def test_input_gradient_in_eval_mode(pkg, ce, monkeypatch, spec, shape, act):
    """ODIN (cvae.py:1648-1656) differentiates the eval-mode network w.r.t. its input: BatchNorm with running statistics
    is folded into the weights, the backward produces the input gradient only."""
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    torch.manual_seed(2)
    seq = pkg.module.vae_layers.build_de_conv_layers(shape, spec, batch_norm=True, where='input', activation=act)
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.uniform_(-0.2, 0.2)
            m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
    seq.eval()
    # the torch reference runs the folded bf16 weights the kernels see (W' = W gamma rstd rounded to bf16, b' likewise in f32):
    # otherwise a ReLU / max-pool decision flipped by the weight rounding dominates the comparison at this tiny size
    ref = copy.deepcopy(seq)
    mods = list(ref)
    for i, m in enumerate(mods):
        if isinstance(m, torch.nn.Conv2d) and i + 1 < len(mods) and isinstance(mods[i + 1], torch.nn.BatchNorm2d):
            bn = mods[i + 1]
            scale = (bn.running_var + bn.eps).rsqrt() * bn.weight.data
            m.weight.data = (m.weight.data * scale.view(-1, 1, 1, 1)).to(torch.bfloat16).float()
            m.bias.data = (m.bias.data - bn.running_mean) * scale + bn.bias.data
            bn.running_mean.zero_(); bn.running_var.fill_(1 - bn.eps); bn.weight.data.fill_(1); bn.bias.data.zero_()
    x = torch.randn(3, *shape)
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    go = torch.randn_like(want)
    want.backward(go)
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin)
    assert _rel(got, want) < 2e-2
    got.backward(go)
    assert xin.grad is not None and _rel(xin.grad, xr.grad) < 3e-2, _rel(xin.grad, xr.grad)
    # the running statistics are untouched
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            assert int(m.num_batches_tracked) == 0


def test_resnet18_features_native_stack(pkg, ce, monkeypatch):
    """torchvision resnet18 minus fc (the reference's ResOrDenseNetFeatures, conv.py:247-272): 7x7 stride-2 stem,
    padded overlapping max pool, BasicBlocks with identity and conv1x1 shortcuts, global average pool -- one native stack,
    forward and every gradient against torch fp32"""
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    torch.manual_seed(0)
    from jointvae_b200.module.vae_layers.conv import ResOrDenseNetFeatures
    seq = ResOrDenseNetFeatures('resnet18', (3, 64, 64), pretrained=False)
    for m in seq.modules():
        if isinstance(m, torch.nn.Conv2d):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()
    ref = copy.deepcopy(seq)
    seq.train(), ref.train()
    x = torch.randn(2, 3, 64, 64).to(torch.bfloat16).float()
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    xin = x.clone().requires_grad_(True)
    n0 = EmuKernels.launches
    got = ce.run(list(seq), xin)
    assert EmuKernels.launches - n0 >= 40
    assert tuple(got.shape) == tuple(want.shape) == (2, 512, 1, 1)
    assert _rel(got, want) < 1e-3, _rel(got, want)
    go = torch.randn_like(want)
    want.backward(go)
    got.backward(go)
    gmax = max(float(p.grad.norm()) for p in ref.parameters())
    for (k, p), (_, q) in zip(seq.named_parameters(), ref.named_parameters()):
        assert p.grad is not None, k
        err = float((p.grad.double() - q.grad.double()).norm())
        assert err <= 5e-3 * float(q.grad.norm()) + 5e-4 * gmax, (k, err, float(q.grad.norm()))
    assert _rel(xin.grad, xr.grad) < 5e-3


def test_resnet18_eval_mode_forward_and_input_gradient(pkg, ce, monkeypatch):
    """eval mode (running statistics folded into every conv of the residual blocks and shortcuts): forward against torch, and
    the input gradient ODIN needs, through the residual joins"""
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    torch.manual_seed(1)
    from jointvae_b200.module.vae_layers.conv import ResOrDenseNetFeatures
    seq = ResOrDenseNetFeatures('resnet18', (3, 32, 32), pretrained=False)
    for m in seq.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.uniform_(-0.2, 0.2)
            m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
    seq.eval()
    x = torch.randn(2, 3, 32, 32).to(torch.bfloat16).float()
    xr = x.clone().requires_grad_(True)
    want = seq(xr)
    go = torch.randn_like(want)
    want.backward(go)
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin)
    # folded weights are rounded to bf16 (the torch side keeps fp32 weights): 20 layers deep
    assert _rel(got, want) < 3e-2, _rel(got, want)
    got.backward(go)
    assert xin.grad is not None and _rel(xin.grad, xr.grad) < 0.15, _rel(xin.grad, xr.grad)
    assert all(int(m.num_batches_tracked) == 0 for m in seq.modules() if isinstance(m, torch.nn.BatchNorm2d))


@pytest.mark.parametrize('kind', ['basic', 'basic_down', 'bottleneck', 'bottleneck_proj', 'bottleneck_down'])
def test_residual_blocks_exact(pkg, ce, monkeypatch, kind):
    """torchvision BasicBlock / Bottleneck (identity, conv1x1 projection, conv1x1 stride-2 shortcut) as ResidualStep: with
    fp32 storage in the emulation forward, input gradient and every parameter gradient equal torch's to rounding"""
    from torchvision.models.resnet import BasicBlock, Bottleneck
    nn = torch.nn
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    torch.manual_seed(0)
    if kind == 'basic':
        block, shape = BasicBlock(16, 16), (16, 8, 8)
    elif kind == 'basic_down':
        block = BasicBlock(16, 32, stride=2, downsample=nn.Sequential(nn.Conv2d(16, 32, 1, stride=2, bias=False), nn.BatchNorm2d(32)))
        shape = (16, 8, 8)
    elif kind == 'bottleneck':
        block, shape = Bottleneck(64, 16), (64, 6, 6)
    elif kind == 'bottleneck_proj':
        block = Bottleneck(16, 16, downsample=nn.Sequential(nn.Conv2d(16, 64, 1, bias=False), nn.BatchNorm2d(64)))
        shape = (16, 6, 6)
    else:
        block = Bottleneck(32, 16, stride=2, downsample=nn.Sequential(nn.Conv2d(32, 64, 1, stride=2, bias=False), nn.BatchNorm2d(64)))
        shape = (32, 8, 8)
    for m in block.modules():
        if isinstance(m, nn.Conv2d):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()
        elif isinstance(m, nn.BatchNorm2d):
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
    seq = nn.Sequential(block)
    ref = copy.deepcopy(seq)
    seq.train(), ref.train()
    x = torch.randn(6, *shape).to(torch.bfloat16).float()
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    go = torch.randn_like(want)
    want.backward(go)
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin)
    assert _rel(got, want) < 1e-5
    got.backward(go)
    assert _rel(xin.grad, xr.grad) < 1e-4
    for (k, p), (_, q) in zip(seq.named_parameters(), ref.named_parameters()):
        assert p.grad is not None and _rel(p.grad, q.grad) < 1e-4, (k, _rel(p.grad, q.grad))


@pytest.mark.parametrize('shape,spec', [((16, 2, 2), '[x3+1]16-24'), ((8, 1, 2), '[x3+1]16'), ((16, 2, 1), '[x5+2]8-8')])
def test_small_map_same_convolutions(pkg, ce, monkeypatch, shape, spec):
    """'same' convolutions on maps of at most 2x2 pixels (the vgg19 tail), where most taps read padding: forward, input
    gradient and parameter gradients equal torch's with fp32 storage, in train and eval mode"""
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    torch.manual_seed(0)
    seq = pkg.module.vae_layers.build_de_conv_layers(shape, spec, batch_norm=True, where='input')
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
        elif hasattr(m, 'weight'):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()
    ref = copy.deepcopy(seq)
    for mode in ('train', 'eval'):
        getattr(seq, mode)(), getattr(ref, mode)()
        x = torch.randn(6, *shape).to(torch.bfloat16).float()
        xr = x.clone().requires_grad_(True)
        want = ref(xr)
        go = torch.randn_like(want)
        want.backward(go)
        xin = x.clone().requires_grad_(True)
        ce._stacks.clear()
        got = ce.run(list(seq), xin)
        tol = 1e-4 if mode == 'train' else 2e-2        # eval folds BatchNorm into bf16 weights
        assert _rel(got, want) < tol
        for p in seq.parameters():
            p.grad = None
        got.backward(go)
        assert _rel(xin.grad, xr.grad) < max(tol, 1e-3)
        if mode == 'train':
            gmax = max(float(q.grad.norm()) for q in ref.parameters())
            for (k, p), (_, q) in zip(seq.named_parameters(), ref.named_parameters()):
                # a conv bias in front of train-mode BatchNorm has an exactly zero gradient here, rounding noise in autograd
                err = float((p.grad.double() - q.grad.double()).norm())
                assert p.grad is not None and err <= 1e-3 * float(q.grad.norm()) + 1e-4 * gmax, (k, err)
        for q in ref.parameters():
            q.grad = None


def test_c2_stack_plan(pkg, ce):
    """which execution form every layer of the flagship stacks takes (BASELINE configs[1]: vgg19 features, deconv32 imager)"""
    build = pkg.module.vae_layers.build_de_conv_layers
    imager = build((128, 1, 1), 'deconv32', batch_norm=True, where='output', output_activation='linear')
    st = ce.ConvStack(list(imager), (128, 1, 1), True)
    convs = [s for s in st.steps if isinstance(s, ce.ConvStep)]
    assert [s.gemm1x1 for s in convs] == [True] + [False] * 6             # ConvTranspose2d on the 1x1 latent map is a plain GEMM
    assert [s.separable for s in convs] == [False] * 6 + [True]           # 32 -> 3 k5 head: separable backward
    assert convs[-1].wgrad_swapped and not any(s.wgrad_swapped for s in convs[:-1])
    assert [len(s.fwd_ops) if s.fwd_ops else 0 for s in convs] == [0, 1, 4, 1, 4, 1, 1]      # stride-2 deconvs: 4 sub-pixel phases
    assert [s.merged_fwd for s in convs] == [False, False, True, False, True, False, False]    # ... issued as ONE merged launch
    assert st.out_shape == (3, 32, 32)
    feats = build((3, 32, 32), 'vgg19', batch_norm=True, where='input')
    sf = ce.ConvStack(list(feats), (3, 32, 32), False)
    fconvs = [s for s in sf.steps if isinstance(s, ce.ConvStep)]
    assert len(fconvs) == 16 and len([s for s in sf.steps if isinstance(s, ce.PoolStep)]) == 5
    assert not any(s.separable or s.gemm1x1 or s.dgrad_sparse for s in fconvs)
    assert sf.out_shape == (512, 1, 1)


@pytest.mark.parametrize('where,spec,shape,bn,out_act', CASES)
def test_pack_specs_equal_torch_packing(pkg, ce, where, spec, shape, bn, out_act):
    """The job table of the native weight re-pack (csrc/pack.cu, one launch per stack and step) describes exactly the
    arrangements ConvStep._pack builds with torch ops: every job, executed by its torch definition (run_pack_spec), is
    bit-equal to the torch-packed tensor.  The CUDA kernel is checked against run_pack_spec on the GPU."""
    torch.manual_seed(1)
    where, _, act = where.partition('/')
    kw = dict(output_activation=out_act) if where == 'output' else {}
    seq = pkg.module.vae_layers.build_de_conv_layers(shape, spec, batch_norm=bn, where=where, activation=act or 'relu', **kw)
    stack = ce.ConvStack(list(seq), shape, where == 'output')
    n = 0
    for stp in stack.plan.steps:
        want = stp._pack()                      # torch formulation (K is the emulation here)
        for sp in stp.pack_specs():
            src = stp.conv.weight if sp['src'] == 'w' else stp.conv.bias
            got = stp.pack_view(sp, ce.run_pack_spec(sp, src))
            ref = want[sp['name']] if sp['index'] is None else want[sp['name']][sp['index']]
            assert got.shape == ref.shape and got.dtype == ref.dtype, (sp['name'], got.shape, ref.shape)
            assert torch.equal(got, ref), sp['name']
            n += 1
    assert n >= 2
