"""CPU-side checks of the SGD / AMSGrad optimizer path: constructor validation as torch.optim.SGD / Adam does it, torch's
state_dict layout before the first step, and the argument checks of jvae_sgd_step / jvae_adam_amsgrad_step through the C ABI
(every case returns before a kernel launch, so no GPU is needed)."""
import ctypes

import pytest
import torch

c_float, c_int, c_size_t, P = ctypes.c_float, ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p
JVAE_ERR_INVALID = -1      # include/jvae_b200.h


def _opt(pkg, **kw):
    return pkg.module.optimizers.Optimizer([torch.nn.Parameter(torch.randn(3, 4)), torch.nn.Parameter(torch.randn(5))], **kw)


@pytest.mark.parametrize('kw', [dict(nesterov=True), dict(nesterov=True, momentum=0.9, dampening=0.1),
                                dict(lr=-0.1), dict(momentum=-0.5), dict(weight_decay=-1e-4)])
def test_sgd_rejects_what_torch_rejects(pkg, kw):
    with pytest.raises(ValueError):
        torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], **{'lr': 0.01, **kw})
    with pytest.raises(ValueError):
        _opt(pkg, optim_type='sgd', **kw)


def test_optimizer_options(pkg):
    for t in ('sgd', 'adam'):
        with pytest.raises(NotImplementedError):
            _opt(pkg, optim_type=t, maximize=True)
    o = _opt(pkg, optim_type='sgd', momentum=0.9, nesterov=True, foreach=True, fused=False, differentiable=False)
    assert o._opt is None and o.lr == 0.01
    with pytest.raises(TypeError):
        _opt(pkg, optim_type='sgd', betas=(0.9, 0.99))
    o = _opt(pkg, optim_type='adam', amsgrad=True, capturable=True)
    assert o._opt is None and o.amsgrad
    assert o.state_dict()['param_groups'][0]['amsgrad'] is True


def test_sgd_state_dict_before_first_step_loads_into_torch(pkg):
    ps = [torch.nn.Parameter(torch.randn(3, 4)), torch.nn.Parameter(torch.randn(5))]
    o = pkg.module.optimizers.Optimizer(ps, optim_type='sgd', lr=0.05, momentum=0.9, nesterov=True, weight_decay=1e-4)
    sd = o.state_dict()
    ref = torch.optim.SGD(ps, lr=0.05, momentum=0.9, nesterov=True, weight_decay=1e-4).state_dict()
    assert sd == ref
    t = torch.optim.SGD(ps, lr=0.01)
    t.load_state_dict(sd)
    assert t.param_groups[0]['momentum'] == 0.9 and t.param_groups[0]['lr'] == 0.05
    o.load_state_dict(ref)
    assert o.lr == 0.05


def _lib(pkg):
    L = ctypes.CDLL(pkg._native.LIB_PATH)
    L.jvae_last_error.restype = ctypes.c_char_p
    L.jvae_sgd_step.argtypes = [P, P, P, c_int, c_size_t, P, c_float, c_float, c_float, c_float, c_int, c_float, c_int,
                                P, P, P, c_float, P]
    L.jvae_adam_amsgrad_step.argtypes = [P, P, P, P, P, c_int, c_size_t, P, c_float, c_float, c_float, c_float, c_float,
                                         c_float, c_int, P, P, P, P, c_float, P]
    return L


# stand-in device addresses: 16-byte aligned and never dereferenced, the checks reject the call before any launch
A, B, G, T = 0x10000, 0x20000, 0x30000, 0x40000


@pytest.mark.parametrize('case,args', [
    ('null p', dict(p=None)),
    ('null grad', dict(grad=None)),
    ('momentum without buf', dict(buf=None, momentum=0.9)),
    ('buf without momentum', dict(momentum=0.0)),
    ('no parameter table', dict(chunk_seg=None)),
    ('n not a whole number of chunks', dict(n=256 * 3 + 4)),
])
def test_sgd_step_argument_checks(pkg, case, args):
    L = _lib(pkg)
    a = dict(p=A, buf=B, grad=G, n=256 * 3, momentum=0.9, chunk_seg=T)
    a.update(args)
    rc = L.jvae_sgd_step(a['p'], a['buf'], a['grad'], 0, a['n'], None, 0.0, 0.01, a['momentum'], 0.0, 0, 0.0, 3,
                         a['chunk_seg'], T, T, 1.0, None)
    assert rc == JVAE_ERR_INVALID, case
    assert b'invalid argument' in L.jvae_last_error(), case


@pytest.mark.parametrize('case,args', [
    ('null p', dict(p=None)),
    ('null vmax', dict(vmax=None)),
    ('no bias-correction scratch', dict(seg_bc=None)),
    ('n not a whole number of chunks', dict(n=100)),
    ('misaligned vmax', dict(vmax=B + 4)),
])
def test_adam_amsgrad_step_argument_checks(pkg, case, args):
    L = _lib(pkg)
    a = dict(p=A, vmax=B, n=256 * 3, seg_bc=T)
    a.update(args)
    rc = L.jvae_adam_amsgrad_step(a['p'], A + 0x1000, A + 0x2000, a['vmax'], G, 0, a['n'], None, 0.0, 1e-3, 0.9, 0.999, 1e-8,
                                  0.0, 3, T, T, T, a['seg_bc'], 1.0, None)
    assert rc == JVAE_ERR_INVALID, case
    assert b'invalid argument' in L.jvae_last_error(), case
