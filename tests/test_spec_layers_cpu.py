"""The layers the conv-spec grammar builds beyond strides 1 / 2, 2x up-sampling and tiling average pools (convolutions and
transposed convolutions of stride 3..8, 'U:s' nearest up-sampling, overlapping / padded / non-tiling 'A' pools), without a
GPU: the conv engine runs build_de_conv_layers stacks through tests/emu_spec_layers.py (a torch emulation of the C-ABI entry
points, same arguments) against torch.nn in fp32; the halo planners' emulators show which geometries the halo kernels take;
the argument checks of the C ABI return before any launch.  The CUDA kernels are checked on the GPU
(tests/test_gpu_spec_layers.py)."""
import copy
import ctypes

import pytest
import torch

from emu_kernels import EmuKernels
from emu_spec_layers import SpecEmuKernels

JVAE_ERR_INVALID = -1      # include/jvae_b200.h


@pytest.fixture()
def ce(pkg, monkeypatch):
    from jointvae_b200 import conv_engine
    monkeypatch.setattr(conv_engine, 'K', SpecEmuKernels)
    conv_engine._stacks.clear()
    yield conv_engine
    conv_engine._stacks.clear()


def _rel(a, b):
    a, b = a.detach().float().double(), b.detach().float().double()
    return float((a - b).norm() / max(1e-9, float(b.norm())))


CASES = [
    # (where, spec, input shape, batch_norm, output_activation)
    ('input', '[x3+1]32x4+0:4-64:3-A3+1:2', (3, 32, 32), True, None),        # patchify stride 4, stride 3, padded pool
    ('input', '16x3+1-Ax3+1:2-Ax3:2', (3, 17, 17), False, None),              # AvgPool2d(3, 2, 1), AvgPool2d(3, 2)
    ('input', '8x4+0:4-16x3+1:3', (3, 19, 19), False, None),                  # odd map, strides 4 and 3
    ('input', '8x8+0:8-16', (3, 33, 35), True, None),                          # k = s = 8 on an odd, non-square map
    ('input', '8x5+2:3-12x7+3:4', (3, 23, 21), True, None),                    # k 5 / 7, strides 3 / 4
    ('input', '8x6+1:5-16x3+1', (3, 27, 26), False, None),                     # k 6, stride 5
    ('input', '8x3+0:4-16', (5, 15, 15), True, None),                          # kernel < stride: empty gradient phases
    ('input', '[x3+1]8-A3:2-16-A3+1:2', (3, 15, 15), True, None),              # overlapping pools, unpadded and padded
    ('input', '8-Ax2', (3, 7, 7), False, None),                                # AvgPool2d(2) on a 7 x 7 map: does not tile
    ('input', '8-A2', (3, 13, 13), False, None),                               # 'A2': kernel 5, stride 2
    ('output', '[x3+1]32x4+0:4-!32-U:4-!3', (6, 2, 2), True, 'linear'),        # transposed patchify, 4x up-sampling
    ('output', '[x4+0]16x4+0:4-8x3+0:3++1-!3x3+1', (6, 2, 2), False, 'sigmoid'),   # transposed strides 4 and 3, output padding
    ('output', '[x5+1]12x5+1:3++2-!3x3+1', (8, 3, 4), True, 'linear'),         # transposed stride 3, output padding 2
    ('output', '[x3+1]8-U:3-!8-U:4-!3', (6, 2, 2), False, 'linear'),           # U:3 then U:4
]


# the tolerances of tests/test_conv_engine_cpu.py::test_stack_matches_torch: fp32 storage isolates the host logic, bf16
# storage is what the kernels do
@pytest.mark.parametrize('store,tol_f,tol_g', [(torch.float32, 1e-4, 1e-3), (torch.bfloat16, 2e-2, 0.25)])
@pytest.mark.parametrize('where,spec,shape,bn,out_act', CASES)
def test_spec_stack_matches_torch(pkg, ce, monkeypatch, where, spec, shape, bn, out_act, store, tol_f, tol_g):
    monkeypatch.setattr(EmuKernels, 'store', store)
    monkeypatch.setattr(EmuKernels, 'act_dtype', store)
    torch.manual_seed(0)
    kw = dict(output_activation=out_act) if where == 'output' else {}
    seq = pkg.module.vae_layers.build_de_conv_layers(shape, spec, batch_norm=bn, where=where, **kw)
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
        elif hasattr(m, 'weight'):
            m.weight.data = m.weight.data.to(torch.bfloat16).float()      # bf16-exact weights: packing does not round
    ref = copy.deepcopy(seq)
    seq.train(), ref.train()
    x = torch.randn(3, *shape).to(torch.bfloat16).float()
    xr = x.clone().requires_grad_(True)
    want = ref(xr)
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin, image_out=(where == 'output'))
    assert tuple(got.shape) == tuple(want.shape) == (3, *seq.output_shape)
    assert _rel(got, want) < tol_f, _rel(got, want)
    go = torch.randn_like(want)
    want.backward(go)
    got.backward(go.to(store).contiguous(memory_format=torch.channels_last) if where == 'output' else go)
    gmax = max(float(p.grad.norm()) for p in ref.parameters())
    for (k, p), (_, q) in zip(seq.named_parameters(), ref.named_parameters()):
        assert p.grad is not None, k
        err = float((p.grad.double() - q.grad.double()).norm())
        assert err <= tol_g * float(q.grad.norm()) + 0.1 * tol_g * gmax, (k, err, float(q.grad.norm()))
    assert _rel(xin.grad, xr.grad) < tol_g, _rel(xin.grad, xr.grad)
    for m, r in zip(seq, ref):
        if isinstance(m, torch.nn.BatchNorm2d):
            assert _rel(m.running_mean, r.running_mean) < 2e-2 or float((m.running_mean - r.running_mean).abs().max()) < 2e-3
            assert _rel(m.running_var, r.running_var) < 2e-2
            assert int(m.num_batches_tracked) == int(r.num_batches_tracked) == 1


def test_spec_layers_take_their_native_form(pkg, ce):
    """which step each spec layer becomes: strided convolutions keep their stride, ConvTranspose2d stride s runs s*s phases,
    U:s keeps its factor, and only non-tiling average pools leave jvae_avgpool"""
    build = pkg.module.vae_layers.build_de_conv_layers
    st = ce.ConvStack(list(build((3, 32, 32), '[x3+1]32x4+0:4-64:3-A3+1:2', where='input')), (3, 32, 32), False)
    convs = [s for s in st.steps if isinstance(s, ce.ConvStep)]
    assert [s.s for s in convs] == [4, 3] and [len(s.dgrad_ops) for s in convs] == [16, 9]
    avg = [s for s in st.steps if isinstance(s, ce.AvgStep)]
    # 'A3+1:2' sets no 'x' field: the grammar's default pooling kernel 5, padding 1, stride 2 on the 3 x 3 map
    assert len(avg) == 1 and not avg[0].tiling and avg[0].win == (5, 5, 2, 2, 1, 1) and st.out_shape == (64, 1, 1)
    # ('!' convolutions of an upsampler spec default to padding 0: '!32x3+1' keeps the map size)
    up = ce.ConvStack(list(build((6, 2, 2), '[x3+1]32x4+0:4-!32x3+1-U:4-!3x3+1', where='output')), (6, 2, 2), True)
    assert [len(s.fwd_ops) for s in up.steps if isinstance(s, ce.ConvStep)] == [16, 1, 1]
    assert not any(s.merged_fwd for s in up.steps if isinstance(s, ce.ConvStep))
    assert [s.s for s in up.steps if isinstance(s, ce.UpStep)] == [4] and up.out_shape == (3, 32, 32)
    # the tiling pool and the global pool of a square map keep jvae_avgpool
    assert ce.AvgStep(torch.nn.AvgPool2d(2), (8, 8, 8)).tiling
    assert ce.AvgStep(torch.nn.AdaptiveAvgPool2d(1), (8, 4, 4)).tiling
    assert not ce.AvgStep(torch.nn.AdaptiveAvgPool2d(1), (8, 4, 6)).tiling


def test_global_average_pool_of_a_non_square_map(pkg, ce, monkeypatch):
    """AdaptiveAvgPool2d((1, 1)) on a 3 x 5 map (ResNet features of a non-square input): forward and input gradient"""
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    seq = torch.nn.Sequential(torch.nn.Conv2d(3, 16, 3, padding=1), torch.nn.ReLU(), torch.nn.AdaptiveAvgPool2d((1, 1)))
    x = torch.randn(2, 3, 3, 5)
    xr = x.clone().requires_grad_(True)
    want = seq(xr)
    xin = x.clone().requires_grad_(True)
    got = ce.run(list(seq), xin)
    assert _rel(got, want) < 1e-2
    go = torch.randn_like(want)
    want.backward(go)
    got.backward(go)
    assert _rel(xin.grad, xr.grad) < 1e-2


@pytest.mark.parametrize('spec,shape', [('[x3+1]8x4+0:4-16:3-A3+1:2', (3, 32, 32)), ('8x5+2:3-16x4+0:4', (3, 25, 25))])
def test_input_gradient_in_eval_mode_strided(pkg, ce, monkeypatch, spec, shape):
    """ODIN differentiates the eval-mode network w.r.t. its input: strided convolutions with BatchNorm folded into the weights,
    their data gradient through the s*s phases, and the padded average pool's backward"""
    monkeypatch.setattr(EmuKernels, 'store', torch.float32)
    monkeypatch.setattr(EmuKernels, 'act_dtype', torch.float32)
    torch.manual_seed(2)
    seq = pkg.module.vae_layers.build_de_conv_layers(shape, spec, batch_norm=True, where='input')
    for m in seq:
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.uniform_(-0.2, 0.2)
            m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.3, 0.3)
    seq.eval()
    # the reference runs the folded bf16 weights the kernels see (as tests/test_conv_engine_cpu.py does)
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
    assert all(int(m.num_batches_tracked) == 0 for m in seq if isinstance(m, torch.nn.BatchNorm2d))


@pytest.mark.parametrize('s', [3, 4, 8])
def test_phase_tables_cover_every_tap_once_large_strides(pkg, s):
    from jointvae_b200 import conv_engine as c
    for k in range(s, 9):
        for p in range(0, k // 2 + 1):
            ops = c.deconv_form(k, p, s, 4 * s + 1, 3 * s + 2)
            idx = sorted(i for op in ops for i in op['idx'])
            assert idx == list(range(k * k)), (k, p, s)
            assert len(ops) == s * s
            assert all(op['in_stride'] == 1 and op['out_s'] == (s, s) for op in ops)


@pytest.mark.parametrize('k,s', [(2, 3), (3, 4)])
def test_transposed_kernel_smaller_than_stride_still_raises(pkg, ce, k, s):
    seq = torch.nn.Sequential(torch.nn.ConvTranspose2d(8, 8, k, stride=s))
    with pytest.raises(NotImplementedError, match='kernel smaller than its stride'):
        ce.run(list(seq), torch.randn(1, 8, 3, 3))


@pytest.mark.parametrize('mods,match', [
    ([torch.nn.Conv2d(3, 8, 9, stride=3)], 'larger than 8x8'),
    ([torch.nn.Conv2d(3, 8, 3, stride=9)], 'stride > 8'),
    ([torch.nn.Conv2d(3, 8, 3, dilation=2)], 'dilated'),
    ([torch.nn.Conv2d(3, 8, 3), torch.nn.MaxPool2d(2, ceil_mode=True)], 'ceil_mode'),
    ([torch.nn.Conv2d(3, 8, 3), torch.nn.AvgPool2d(3, 2, ceil_mode=True)], 'ceil_mode'),
    ([torch.nn.Conv2d(3, 8, 3), torch.nn.AvgPool2d(3, 2, 1, count_include_pad=False)], 'count_include_pad'),
    ([torch.nn.Conv2d(3, 8, 3), torch.nn.AdaptiveAvgPool2d((2, 2))], 'output size'),
    ([torch.nn.Conv2d(3, 8, 3), torch.nn.UpsamplingNearest2d(scale_factor=1.5)], 'non-integer'),
    ([torch.nn.Conv2d(3, 8, 3), torch.nn.UpsamplingNearest2d(size=(20, 20))], 'output size'),
])
def test_out_of_scope_layers_raise_with_a_reason(pkg, ce, mods, match):
    with pytest.raises(NotImplementedError, match=match):
        ce.run(mods, torch.randn(1, 3, 16, 16))


def _nhwc(x, ld):
    n, c, h, w = x.shape
    t = torch.zeros(n, h, w, ld)
    t[..., :c] = x.permute(0, 2, 3, 1)
    return t.contiguous()


@pytest.mark.parametrize('s', [3, 4, 8])
def test_halo_planners_leave_large_strides_to_the_tap_box_kernels(pkg, ce, s):
    nat = pkg._native
    N, H, W, Ci, Co, k = 2, 8 * s, 8 * s, 16, 16, 3
    taps = nat.taps_arg([(i - 1, j - 1) for i in range(k) for j in range(k)])
    Hq = (H + 2 - k) // s + 1
    x = torch.randn(N, H, W, Ci)
    wm = torch.zeros(Co, k * k * Ci)
    out = torch.zeros(N, Hq, Hq, Co)
    assert Hq >= 6
    assert nat.conv_halo_emulate(x, Ci, wm, Co, taps, s, Hq, Hq, out, Co) is None
    dw = torch.zeros(Co, Ci, k * k)
    assert nat.conv_wgrad_emulate(torch.randn(N, Hq, Hq, Co), Co, x, Ci, taps, s, dw, 1, Ci * k * k, k * k) is None


@pytest.mark.parametrize('N,H,W,Cin,Cout,k,p,s,op', [
    (3, 8, 8, 32, 32, 4, 0, 4, 0),       # transposed patchify: one tap per phase
    (2, 7, 9, 16, 24, 5, 1, 3, 2),       # stride 3, output padding 2, ragged phases
    (2, 6, 6, 64, 16, 8, 0, 8, 0),       # stride 8: 64 single-tap phases
])
def test_halo_phases_with_output_stride_above_two(pkg, ce, N, H, W, Cin, Cout, k, p, s, op):
    """The sub-pixel phases of a stride-s ConvTranspose2d are stride-1 gathers written with output stride s: where the halo
    planner takes one, its epilogue (block table, phase offsets, bounds) writes exactly that phase's pixels; all phases
    together give torch's result"""
    nat = pkg._native
    torch.manual_seed(s * 7 + k)
    conv = torch.nn.ConvTranspose2d(Cin, Cout, k, stride=s, padding=p, output_padding=op)
    conv.weight.data = conv.weight.data.to(torch.bfloat16).float()
    x = torch.randn(N, Cin, H, W)
    ref = conv(x).detach()
    Ho, Wo = ref.shape[-2:]
    g_f = conv.weight.detach().permute(1, 2, 3, 0).reshape(Cout, k * k, Cin)
    out = torch.full((N, Ho, Wo, ce.r8(Cout)), float('nan'))
    covered = 0
    for o in ce.deconv_form(k, p, s, Ho, Wo):
        wm = ce.pack_gather_weights(g_f, o['idx'], Cin).float().contiguous()
        info = nat.conv_halo_emulate(_nhwc(x, ce.r8(Cin)), Cin, wm, wm.shape[0], nat.taps_arg(o['taps']), 1, o['Hq'], o['Wq'], out,
                                     Cout, o['out_s'], o['out_o'], conv.bias.detach().contiguous(), 0)
        if info is None:      # Wq < 6: the tap-box kernel, whose epilogue addresses q * out_s + out_o directly
            view = out[:, o['out_o'][0]::s, o['out_o'][1]::s]
            assert view.shape[1:3] == (o['Hq'], o['Wq'])
            sel = ref[:, :, o['out_o'][0]::s, o['out_o'][1]::s].permute(0, 2, 3, 1)
            view[..., :Cout] = sel
            view[..., Cout:] = 0
        else:
            covered += 1
    assert covered >= 1
    assert not torch.isnan(out).any(), 'a pixel no phase wrote, or a leftover in a live row'
    assert float((out[..., :Cout].permute(0, 3, 1, 2) - ref).abs().max()) < 1e-4


# ------------------------------------------------------------------------------------------------ C ABI argument checks
P, c_int, I16P = ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int16)
A = 0x7f0000100000      # 16-byte aligned stand-ins: every case returns at an argument check, before any access


def _lib(pkg):
    L = ctypes.CDLL(pkg._native.LIB_PATH)
    L.jvae_last_error.restype = ctypes.c_char_p
    L.jvae_conv_gather_gemm.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, I16P, I16P, c_int,
                                        c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, P, P]
    L.jvae_conv_wgrad.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, I16P, I16P,
                                  c_int, P, c_int, c_int, c_int, P]
    L.jvae_upsample_nearest.argtypes = [P, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]
    L.jvae_avgpool_pad.argtypes = [P, c_int, P, c_int] + [c_int] * 11 + [P]
    return L


@pytest.mark.parametrize('stride', [0, 9, -1])
def test_conv_entry_points_reject_bad_strides(pkg, stride):
    L = _lib(pkg)
    dy, dx = pkg._native.taps_arg([(0, 0)] * 9)
    rc = L.jvae_conv_gather_gemm(A, 2, 16, 16, 16, 16, A + 0x10000, 16, 9 * 16, 9, dy, dx, stride, 8, 8, A + 0x20000, 8, 8, 16,
                                 16, 1, 1, 0, 0, None, 0, None, None)
    assert rc == JVAE_ERR_INVALID and b'input stride 1..8' in L.jvae_last_error()
    rc = L.jvae_conv_wgrad(A, 2, 8, 8, 16, 16, A + 0x10000, 16, 16, 16, 16, 9, dy, dx, stride, A + 0x20000, 1, 144, 9, None)
    assert rc == JVAE_ERR_INVALID and b'input stride 1..8' in L.jvae_last_error()
    nat = pkg._native
    x, wm, out = torch.zeros(2, 16, 16, 16), torch.zeros(16, 144), torch.zeros(2, 8, 8, 16)
    with pytest.raises(nat.NativeError, match='input stride 1..8'):
        nat.conv_halo_emulate(x, 16, wm, 16, (dy, dx), stride, 8, 8, out, 16)
    with pytest.raises(nat.NativeError, match='input stride 1..8'):
        nat.conv_wgrad_emulate(out.clone(), 16, x, 16, (dy, dx), stride, torch.zeros(16, 16, 9), 1, 144, 9)


@pytest.mark.parametrize('s', [0, -2])
def test_upsample_nearest_rejects_bad_factor(pkg, s):
    L = _lib(pkg)
    assert L.jvae_upsample_nearest(A, 16, A + 0x10000, 16, 2, 4, 4, 16, s, 0, None) == JVAE_ERR_INVALID
    assert b'up-sampling factor' in L.jvae_last_error()


@pytest.mark.parametrize('win,what', [((3, 3, 2, 2, 2, 1), 'padding'), ((3, 3, 2, 2, 1, 2), 'padding'),
                                      ((2, 2, 0, 2, 0, 0), 'bad window'), ((20, 3, 1, 1, 0, 0), 'larger than the padded map')])
def test_avgpool_pad_rejects_bad_windows(pkg, win, what):
    L = _lib(pkg)
    assert L.jvae_avgpool_pad(A, 16, A + 0x10000, 16, 2, 8, 8, 16, *win, 0, None) == JVAE_ERR_INVALID
    assert what.encode() in L.jvae_last_error()
