"""GPU parity of the native convolution path (csrc/conv.cu, csrc/norm.cu through conv_engine) against torch.nn running
the same layers in fp32 on the same device.  Activations are stored in bf16 between layers, so forward results are
compared at 2e-2 relative (north_star's bf16 tolerance) and gradients per tensor relative to the tensor's norm."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _rel(a, b):
    a, b = a.detach().float().double(), b.detach().float().double()
    return float((a - b).norm() / max(1e-9, float(b.norm())))


CASES = [
    # (where, spec, input shape, batch, batch_norm, output_activation)
    ('input', 'vgg11', (3, 32, 32), 16, True, None),
    ('input', 'conv32', (3, 32, 32), 32, True, None),
    ('input', 'conv32', (3, 32, 32), 8, False, None),
    ('input', '[x3-Mx2]8-M-24-M-40', (3, 28, 28), 5, False, None),
    ('input', '16x3+1:2-8x5+2', (5, 9, 9), 7, False, None),
    ('output', 'deconv32', (128, 1, 1), 48, True, 'linear'),
    ('output', 'deconv32', (64, 1, 1), 8, False, 'sigmoid'),
    ('output', 'deconv32+', (32, 1, 1), 8, True, 'sigmoid'),
    ('output', 'ivgg', (16, 2, 2), 6, True, 'linear'),
    ('output', '[x4+1]8x4+1:2-!3x3+1', (6, 3, 3), 9, False, 'linear'),
    # activation = leaky (config.ini:113 of the reference)
    ('input/leaky', 'conv32', (3, 32, 32), 16, True, None),
    ('input/leaky', 'conv32', (3, 32, 32), 8, False, None),
    ('output/leaky', 'deconv32', (64, 1, 1), 16, True, 'linear'),
    ('output/leaky', 'deconv32', (64, 1, 1), 8, False, 'sigmoid'),
    # torchvision ResNet features (conv.py:247-272; BASELINE configs[3]): 7x7 stride-2 stem, padded overlapping max pool,
    # residual blocks with identity / conv1x1 stride-2 shortcuts, global average pool
    ('input', 'resnet18', (3, 64, 64), 16, True, None),
]


@pytest.mark.parametrize('where,spec,shape,N,bn,out_act', CASES)
def test_stack_matches_torch_fp32(pkg, where, spec, shape, N, bn, out_act):
    from jointvae_b200 import conv_engine as ce
    torch.manual_seed(0)
    where, _, act = where.partition('/')
    kw = dict(output_activation=out_act) if where == 'output' else {}
    seq = pkg.module.vae_layers.build_de_conv_layers(shape, spec, batch_norm=bn, where=where, activation=act or 'relu',
                                                     **kw).to(DEV)
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
        elif hasattr(m, 'weight'):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()
    ref = copy.deepcopy(seq)
    lib = copy.deepcopy(seq)          # the same layers through cuDNN in bf16: the noise floor of bf16 activations
    seq.train(), ref.train(), lib.train()
    x = torch.randn(N, *shape, device=DEV).to(torch.bfloat16).float()
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    xin = x.clone().requires_grad_(True)      # 'input' stacks: the gradient w.r.t. the image (ODIN differentiates it)
    n0 = pkg._native.launch_count()
    got = ce.run(list(seq), xin, image_out=(where == 'output'))
    assert pkg._native.launch_count() > n0
    assert tuple(got.shape) == tuple(want.shape)
    assert torch.isfinite(got.float()).all()
    with torch.autocast(device_type='cuda', dtype=torch.bfloat16):
        lo = lib(x.contiguous(memory_format=torch.channels_last))
    # 2e-2 (north_star's bf16 tolerance), or the cuDNN-bf16 noise floor for deep stacks (resnet18: 20 BatchNorm layers)
    assert _rel(got, want) < max(2e-2, 1.5 * _rel(lo.float(), want)), (_rel(got, want), _rel(lo.float(), want))
    go = torch.randn_like(want)
    want.backward(go)
    lo.backward(go.to(lo.dtype))
    g = go.to(torch.bfloat16).contiguous(memory_format=torch.channels_last) if where == 'output' else go
    got.backward(g)
    gmax = max(float(p.grad.norm()) for p in ref.parameters())
    report = []
    for (k, p), (_, q), (_, l) in zip(seq.named_parameters(), ref.named_parameters(), lib.named_parameters()):
        assert p.grad is not None, k
        assert torch.isfinite(p.grad).all(), k
        err = float((p.grad.double() - q.grad.double()).norm())
        err_lib = float((l.grad.double() - q.grad.double()).norm())
        report.append((k, round(err, 4), round(err_lib, 4), round(float(q.grad.norm()), 4)))
    print('grad errors (name, native, cudnn-bf16, |ref|):', report)
    for k, err, err_lib, nr in report:
        # within 12 % of the fp32 gradient, or no worse than twice what cuDNN's bf16 path does on the same layers
        # (BatchNorm over few pixels and max-pool routing amplify bf16 activation rounding)
        assert err <= max(0.12 * nr + 0.01 * gmax, 2.0 * err_lib), (k, err, err_lib, nr)
    if True:
        xl = x.clone().requires_grad_(True)
        lib2 = copy.deepcopy(ref).train()
        with torch.autocast(device_type='cuda', dtype=torch.bfloat16):
            lo2 = lib2(xl)
        lo2.backward(go.to(lo2.dtype))
        assert _rel(xin.grad, xr.grad) < max(0.12, 2.0 * _rel(xl.grad, xr.grad)), (_rel(xin.grad, xr.grad), _rel(xl.grad, xr.grad))
    for m, r in zip(seq, ref):
        if isinstance(m, torch.nn.BatchNorm2d):
            assert float((m.running_mean - r.running_mean).abs().max()) < 2e-2 * max(1.0, float(r.running_mean.abs().max()))
            assert _rel(m.running_var, r.running_var) < 2e-2
            assert int(m.num_batches_tracked) == 1


@pytest.mark.parametrize('C,ld', [(32, 32), (64, 64), (512, 512), (3, 8), (5, 8), (200, 200), (24, 24)])
def test_batchnorm_kernels(pkg, C, ld):
    """csrc/norm.cu against torch.nn.functional.batch_norm (+ relu) and its autograd"""
    nat = pkg._native
    torch.manual_seed(1)
    P = 3000
    y = (torch.randn(P, C, device=DEV) * 2 + 0.5).to(torch.bfloat16)
    buf = torch.zeros(P, ld, dtype=torch.bfloat16, device=DEV)
    buf[:, :C] = y
    gamma = torch.rand(C, device=DEV) + 0.5
    beta = torch.randn(C, device=DEV) * 0.2
    stats = torch.zeros(2, C, device=DEV, dtype=torch.float64)
    nat.bn_stats(buf, P, C, ld, stats)
    yf = y.float()
    assert _rel(stats[0], yf.sum(0)) < 1e-4 and _rel(stats[1], (yf * yf).sum(0)) < 1e-4
    rm, rv = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    nb = torch.zeros((), dtype=torch.long, device=DEV)
    out = torch.zeros(P, ld, dtype=torch.bfloat16, device=DEV)
    save = torch.empty(2, C, device=DEV)
    nat.bn_apply_fwd(buf, P, C, ld, stats, gamma, beta, 1e-5, 0.1, rm, rv, nb, True, 1, out, ld, save)
    yr = yf.clone().requires_grad_(True)
    rm2, rv2 = torch.zeros(C, device=DEV), torch.ones(C, device=DEV)
    g2, b2 = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    want = torch.relu(torch.nn.functional.batch_norm(yr, rm2, rv2, g2, b2, True, 0.1, 1e-5))
    assert _rel(out[:, :C], want) < 6e-3
    assert _rel(rm, rm2) < 1e-4 and _rel(rv, rv2) < 1e-4 and int(nb) == 1
    da = torch.randn(P, C, device=DEV).to(torch.bfloat16)
    dab = torch.zeros(P, ld, dtype=torch.bfloat16, device=DEV)
    dab[:, :C] = da
    want.backward(da.float())
    dy = torch.zeros(P, ld, dtype=torch.bfloat16, device=DEV)
    sums = torch.empty(2, C, device=DEV, dtype=torch.float64)
    dg, db = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
    nat.bn_bwd(dab, ld, buf, ld, P, C, save, gamma, beta, 1, sums, dy, ld, dg, db)
    assert _rel(dy[:, :C], yr.grad) < 1e-2
    assert _rel(dg, g2.grad) < 1e-3 and _rel(db, b2.grad) < 1e-3
    if C < 8:      # the image head: the loss gradient arrives dense (ld_da = C), y / dy in padded rows (thread-per-pixel kernels)
        dy2 = torch.full((P, ld), float('nan'), dtype=torch.bfloat16, device=DEV)
        dg2, db2 = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
        nat.bn_bwd(da.contiguous(), C, buf, ld, P, C, save, gamma, beta, 1, sums, dy2, ld, dg2, db2)
        assert torch.equal(dy2, dy) and torch.equal(dg2, dg) and torch.equal(db2, db)
        assert float(dy2[:, C:].float().abs().max()) == 0


@pytest.mark.parametrize('C', [8, 64, 3])
def test_pool_upsample_act_kernels(pkg, C):
    nat = pkg._native
    torch.manual_seed(2)
    N, H, W = 3, 8, 6
    ld = (C + 7) // 8 * 8
    x = torch.zeros(N, H, W, ld, dtype=torch.bfloat16, device=DEV)
    x[..., :C] = torch.randn(N, H, W, C, device=DEV).clamp_min(0)       # relu-like: exact ties at zero
    for k, s in ((2, 2), (3, 3), (2, 3), (5, 5)):
        Ho, Wo = (H - k) // s + 1, (W - k) // s + 1
        out = torch.zeros(N, Ho, Wo, ld, dtype=torch.bfloat16, device=DEV)
        nat.maxpool_fwd(x, N, H, W, C, ld, k, s, out, ld)
        xr = x[..., :C].float().permute(0, 3, 1, 2).clone().requires_grad_(True)
        want = torch.nn.functional.max_pool2d(xr, k, s)
        assert torch.equal(out[..., :C].float().permute(0, 3, 1, 2), want)
        go = torch.randn_like(want).to(torch.bfloat16)
        want.backward(go.float())
        gob = torch.zeros(N, Ho, Wo, ld, dtype=torch.bfloat16, device=DEV)
        gob[..., :C] = go.permute(0, 2, 3, 1)
        din = torch.full_like(x, 7.0)
        nat.maxpool_bwd(x, N, H, W, C, ld, k, s, gob, ld, din, ld)
        assert torch.equal(din[..., :C].float().permute(0, 3, 1, 2), xr.grad), (k, s)
    up = torch.zeros(N, 2 * H, 2 * W, ld, dtype=torch.bfloat16, device=DEV)
    nat.upsample2(x, ld, up, ld, N, H, W, C, False)
    assert torch.equal(up[..., :C], x[..., :C].repeat_interleave(2, 1).repeat_interleave(2, 2))
    dn = torch.zeros_like(x)
    nat.upsample2(up, ld, dn, ld, N, H, W, C, True)
    assert _rel(dn[..., :C], 4 * x[..., :C].float()) < 1e-2
    # activation backward + bias gradient
    P = N * H * W
    da = torch.zeros(P, ld, dtype=torch.bfloat16, device=DEV)
    da[:, :C] = torch.randn(P, C, device=DEV)
    dy = torch.zeros(P, ld, dtype=torch.bfloat16, device=DEV)
    dbias = torch.zeros(C, device=DEV)
    nat.act_bwd(da, ld, x, ld, P, C, 1, dy, ld, dbias)
    wantd = da[:, :C].float() * (x.view(P, ld)[:, :C] > 0)
    assert _rel(dy[:, :C], wantd) < 1e-6 or float(wantd.norm()) == 0
    assert _rel(dbias, wantd.sum(0)) < 1e-3


@pytest.mark.parametrize('spec,shape,N,act', [('[x3-Mx2]8-M-16', (3, 8, 8), 6, 'relu'), ('[x5+2]8-8:2-16', (3, 8, 8), 6, 'leaky'),
                                              ('[x3+1]8-8-M-16:2-16', (3, 16, 16), 6, 'relu'), ('vgg11', (3, 32, 32), 16, 'relu'),
                                              ('conv32', (3, 32, 32), 32, 'relu')])
def test_input_gradient_in_eval_mode(pkg, spec, shape, N, act):
    """eval-mode stack (BatchNorm folded into the weights) differentiated w.r.t. its input, as ODIN does
    (cvae.py:1648-1656), against torch fp32 running the same folded bf16 weights; cuDNN-bf16 gives the noise floor"""
    from jointvae_b200 import conv_engine as ce
    torch.manual_seed(2)
    seq = pkg.module.vae_layers.build_de_conv_layers(shape, spec, batch_norm=True, where='input', activation=act).to(DEV)
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.uniform_(-0.2, 0.2)
            m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
    seq.eval()
    ref = copy.deepcopy(seq)
    mods = list(ref)
    for i, m in enumerate(mods):
        if isinstance(m, torch.nn.Conv2d) and i + 1 < len(mods) and isinstance(mods[i + 1], torch.nn.BatchNorm2d):
            bn = mods[i + 1]
            scale = (bn.running_var + bn.eps).rsqrt() * bn.weight.data
            m.weight.data = (m.weight.data * scale.view(-1, 1, 1, 1)).to(torch.bfloat16).float()
            m.bias.data = (m.bias.data - bn.running_mean) * scale + bn.bias.data
            bn.running_mean.zero_(); bn.running_var.fill_(1 - bn.eps); bn.weight.data.fill_(1); bn.bias.data.zero_()
    lib = copy.deepcopy(ref)
    x = torch.randn(N, *shape, device=DEV).to(torch.bfloat16).float()
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
    assert _rel(got, want) < 2e-2
    got.backward(go)
    e, e_lib = _rel(xin.grad, xr.grad), _rel(xl.grad, xr.grad)
    print('input-gradient error: native', e, 'cudnn-bf16', e_lib)
    assert e < max(0.05, 2.0 * e_lib), (e, e_lib)
    assert all(int(m.num_batches_tracked) == 0 for m in seq if isinstance(m, torch.nn.BatchNorm2d))


@pytest.mark.parametrize('C,H,W,k,s,p', [(64, 32, 32, 3, 2, 1), (8, 9, 7, 3, 2, 1), (3, 8, 8, 2, 1, 0), (16, 6, 6, 3, 1, 1)])
def test_padded_overlapping_maxpool(pkg, C, H, W, k, s, p):
    """jvae_maxpool_pad_fwd / bwd against torch (ResNet stem MaxPool2d(3, 2, 1) and other padded / overlapping windows),
    with ties: bf16 inputs on a coarse grid make equal maxima common, the first one in scan order must get the gradient"""
    nat = pkg._native
    torch.manual_seed(0)
    N, ld = 5, (C + 7) // 8 * 8
    x = (torch.randint(-3, 4, (N, H, W, ld), device=DEV).float() / 2).to(torch.bfloat16)
    Ho, Wo = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
    out = torch.empty(N, Ho, Wo, ld, dtype=torch.bfloat16, device=DEV)
    nat.maxpool_pad_fwd(x, N, H, W, C, ld, k, s, p, out, ld)
    xr = x[..., :C].float().permute(0, 3, 1, 2).clone().requires_grad_(True)
    want = torch.nn.functional.max_pool2d(xr, k, s, p)
    assert torch.equal(out[..., :C].float().permute(0, 3, 1, 2), want)
    go = torch.randn(N, Ho, Wo, ld, device=DEV).to(torch.bfloat16)
    want.backward(go[..., :C].float().permute(0, 3, 1, 2))
    din = torch.empty_like(x)
    nat.maxpool_pad_bwd(x, N, H, W, C, ld, k, s, p, go, ld, din, ld)
    got = din[..., :C].float().permute(0, 3, 1, 2)
    assert float((got - xr.grad).abs().max()) <= 2e-2 * float(xr.grad.abs().max())      # sums of up to 4 bf16 gradients


@pytest.mark.parametrize('C,H,k', [(512, 2, 2), (64, 8, 4), (3, 6, 3), (16, 1, 1)])
def test_avgpool_and_residual_join(pkg, C, H, k):
    nat = pkg._native
    torch.manual_seed(1)
    N, ld = 4, (C + 7) // 8 * 8
    x = torch.randn(N, H, H, ld, device=DEV).to(torch.bfloat16)
    out = torch.empty(N, H // k, H // k, ld, dtype=torch.bfloat16, device=DEV)
    nat.avgpool(x, ld, out, ld, N, H, H, C, k, False)
    want = torch.nn.functional.avg_pool2d(x[..., :C].float().permute(0, 3, 1, 2), k)
    assert torch.allclose(out[..., :C].float().permute(0, 3, 1, 2), want, rtol=1e-2, atol=1e-2)
    g = torch.randn_like(out)
    dx = torch.empty_like(x)
    nat.avgpool(g, ld, dx, ld, N, H, H, C, k, True)
    wantg = (g[..., :C].float() / (k * k)).repeat_interleave(k, 1).repeat_interleave(k, 2)
    assert torch.allclose(dx[..., :C].float(), wantg, rtol=1e-2, atol=1e-3)
    a, b = torch.randn_like(x), torch.randn_like(x)
    o = torch.empty_like(x)
    for act, fn in ((1, torch.relu), (0, lambda t: t)):
        nat.add_act(a, ld, b, ld, N * H * H, C, act, o, ld)
        assert torch.allclose(o[..., :C].float(), fn(a[..., :C].float() + b[..., :C].float()), rtol=1e-2, atol=1e-2)


@pytest.mark.parametrize('k,Co,ld_t,ld_y,H,W', [(5, 3, 16, 8, 32, 32), (5, 3, 16, 3, 9, 8), (3, 4, 16, 8, 8, 8), (3, 1, 8, 8, 10, 12),
                                                (7, 2, 16, 2, 8, 8), (3, 3, 16, 8, 16, 16), (5, 1, 16, 8, 28, 28),
                                                (3, 1, 16, 8, 8, 24)])
def test_separable_head_vstack_rows(pkg, k, Co, ld_t, ld_y, H, W):
    """jvae_vstack_rows (backward of the vertical stage of the separable narrow-output convolution), vectorised and generic
    layouts, against the index arithmetic written out in torch, and adjoint to the vertical shift-and-add"""
    nat = pkg._native
    torch.manual_seed(0)
    N, p = 3, (k - 1) // 2
    T = torch.randn(N, H, W, ld_t, device=DEV).to(torch.bfloat16)
    acc = torch.zeros(N, H, W, Co, device=DEV)          # the vertical shift-and-add of T
    for ty in range(k):
        sh = ty - p
        lo, hi = max(0, -sh), min(H, H - sh)
        acc[:, lo:hi] += T.float()[:, lo + sh:hi + sh, :, ty * Co:(ty + 1) * Co]
    dy = torch.randn(N, H, W, ld_y, device=DEV).to(torch.bfloat16)
    U = torch.full((N, H, W, ld_t), 7.0, dtype=torch.bfloat16, device=DEV)
    nat.vstack_rows(dy, ld_y, N, H, W, k, p, Co, U, ld_t)
    want = torch.zeros(N, H, W, ld_t, device=DEV)
    for ty in range(k):
        sh = ty - p
        lo, hi = max(0, sh), min(H, H + sh)
        want[:, lo:hi, :, ty * Co:(ty + 1) * Co] = dy.float()[:, lo - sh:hi - sh, :, :Co]
    assert torch.equal(U.float(), want)
    # adjointness: <vsum(T), dy> = <T, vstack(dy)> over the k * Co real channels
    lhs = (acc * dy.float()[..., :Co]).sum()
    rhs = (T.float()[..., :k * Co] * want[..., :k * Co]).sum()
    assert abs(float(lhs - rhs)) <= 1e-3 * max(1.0, abs(float(lhs)))


@pytest.mark.parametrize('k,stride,H,C', [(3, 1, 4, 64), (3, 1, 2, 136), (5, 1, 3, 8), (2, 2, 4, 16), (1, 1, 2, 8)])
def test_im2col_matches_unfold(pkg, k, stride, H, C):
    """jvae_im2col_bf16 (patch matrix of the small-map weight gradient) against torch's unfold: same (Cin, kh, kw) column order"""
    import torch.nn.functional as F
    nat = pkg._native
    N, pad = 5, (k // 2 if stride == 1 else 0)
    ld = C + 8
    x = torch.randn(N, H, H, ld, device=DEV).to(torch.bfloat16)
    Hq = (H + 2 * pad - k) // stride + 1
    taps = nat.taps_arg([(ky - pad, kx - pad) for ky in range(k) for kx in range(k)])
    out = torch.full((N * Hq * Hq, C * k * k + 8), 7.0, dtype=torch.bfloat16, device=DEV)
    nat.im2col(x, N, H, H, C, ld, taps, stride, Hq, Hq, out)
    want = F.unfold(x[..., :C].permute(0, 3, 1, 2).float(), k, padding=pad, stride=stride)      # (N, C k k, Hq Hq)
    want = want.permute(0, 2, 1).reshape(N * Hq * Hq, C * k * k)
    assert torch.equal(out[:, :C * k * k].float(), want)
    assert (out[:, C * k * k:] == 7.0).all()          # columns past C * T are left alone


def test_im2col_tap_major_and_split_k_gemm(pkg):
    """the ResNet-stem form of the weight gradient: patch matrix with (tap, channel) columns for a 7 x 7 stride-2 window on a
    3-channel (padded to 8) image + the TN GEMM with its reduction split over the grid (fp32 atomics), against torch"""
    import torch.nn.functional as F
    nat = pkg._native
    N, H, C, k, pad, stride, Co = 6, 20, 3, 7, 3, 2, 24
    x = torch.zeros(N, H, H, 8, device=DEV, dtype=torch.bfloat16)
    x[..., :C] = torch.randn(N, H, H, C, device=DEV).to(torch.bfloat16)
    Hq = (H + 2 * pad - k) // stride + 1
    taps = nat.taps_arg([(ky - pad, kx - pad) for ky in range(k) for kx in range(k)])
    T = k * k
    cols = torch.empty((N * Hq * Hq, 8 * T), dtype=torch.bfloat16, device=DEV)
    nat.im2col(x, N, H, H, 8, 8, taps, stride, Hq, Hq, cols, tap_major=True)
    want = F.unfold(x.permute(0, 3, 1, 2).float(), k, padding=pad, stride=stride)              # (N, 8 T, P) in (ci, tap) order
    want = want.view(N, 8, T, -1).permute(0, 3, 2, 1).reshape(N * Hq * Hq, T * 8)
    assert torch.equal(cols.float(), want)
    g = torch.randn(N * Hq * Hq, Co + 8, device=DEV).to(torch.bfloat16)
    ref = g[:, :Co].float().t() @ cols.float()
    for ks in (1, 2, 5):
        out = torch.ones((Co, 8 * T), dtype=torch.float32, device=DEV)
        nat.gemm_bf16(2, Co, 8 * T, N * Hq * Hq, g, g.stride(0), cols, 8 * T, out_f32=out, ldd=8 * T, accumulate=ks if ks > 1 else True)
        assert torch.allclose(out - 1, ref, rtol=1e-4, atol=1e-3), (ks, float((out - 1 - ref).abs().max()))


@pytest.mark.parametrize('N,H,W,Ci,Co,k,p', [(33, 8, 8, 64, 64, 5, 2), (17, 16, 16, 32, 32, 5, 2), (5, 12, 20, 16, 24, 4, 1),
                                             (3, 40, 16, 8, 3, 3, 1)])
def test_merged_subpixel_launch_equals_phase_launches(pkg, N, H, W, Ci, Co, k, p):
    """jvae_conv_subpixel_gemm (all four sub-pixel phases of a stride-2 ConvTranspose2d in one launch) against one
    jvae_conv_gather_gemm per phase on the same tensors: outputs within bf16 rounding of each other, BatchNorm sums equal
    (module/vae_layers/conv.py:189-219; conv-models.ini:25 deconv32)"""
    from jointvae_b200 import conv_engine as ce
    K = ce.NativeKernels
    torch.manual_seed(N)
    Ho, Wo = 2 * H, 2 * W
    ops = ce.deconv_form(k, p, 2, Ho, Wo)
    g = (torch.randn(Co, k * k, Ci, device=DEV) * 0.2)
    x = torch.zeros(N, H, W, ce.r8(Ci), device=DEV, dtype=torch.bfloat16)
    x[..., :Ci] = torch.randn(N, H, W, Ci, device=DEV)
    bias = torch.randn(Co, device=DEV)
    w_all = ce.pack_gather_weights(g, [i for op in ops for i in op['idx']], Ci)
    out_m = torch.full((N, Ho, Wo, ce.r8(Co)), float('nan'), device=DEV, dtype=torch.bfloat16)
    st_m = torch.zeros(2, Co, device=DEV, dtype=torch.float64)
    ok = K.subpixel(x, Ci, w_all, w_all.shape[0], K.phases_arg(ops), H, W, out_m, Co, 2, bias, 0, st_m)
    assert ok, 'geometry expected to be covered by the merged kernel'
    out_p = torch.full_like(out_m, float('nan'))
    st_p = torch.zeros_like(st_m)
    for op in ops:
        wm = ce.pack_gather_weights(g, op['idx'], Ci)
        K.gather(x, Ci, wm, wm.shape[0], K.taps_arg(op['taps']), 1, H, W, out_p, Co, op['out_s'], op['out_o'], bias, 0, st_p)
    torch.cuda.synchronize()
    assert not torch.isnan(out_m.float()).any() and not torch.isnan(out_p.float()).any()
    scale = float(out_p.float().abs().max())
    assert float((out_m.float() - out_p.float()).abs().max()) <= 2e-2 * scale
    assert float((out_m[..., Co:].float()).abs().max() if out_m.shape[-1] > Co else 0) == 0
    assert torch.allclose(st_m, st_p, rtol=1e-4, atol=1e-3 * float(st_p.abs().max()))


def test_merged_subpixel_launch_declines_wide_layers(pkg):
    """more than 64 channels: JVAE_NOT_COVERED, nothing launched, the caller runs the phases one by one"""
    from jointvae_b200 import conv_engine as ce
    K = ce.NativeKernels
    ops = ce.deconv_form(3, 1, 2, 16, 16)
    g = torch.randn(128, 9, 128, device=DEV)
    x = torch.randn(2, 8, 8, 128, device=DEV).to(torch.bfloat16)
    w_all = ce.pack_gather_weights(g, [i for op in ops for i in op['idx']], 128)
    out = torch.zeros(2, 16, 16, 128, device=DEV, dtype=torch.bfloat16)
    n0 = pkg._native.launch_count()
    assert K.subpixel(x, 128, w_all, w_all.shape[0], K.phases_arg(ops), 8, 8, out, 128, 2, None, 0, None) is False
    assert pkg._native.launch_count() == n0 and float(out.float().abs().max()) == 0
