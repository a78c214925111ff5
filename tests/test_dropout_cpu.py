"""Dense-layer dropout without a GPU: the numpy restatement of the Philox keep-mask (tests/philox_ref.py) against the Random123
known-answer vectors and the binomial keep rate, the argument checks of jvae_gemm_bf16_dropout / jvae_act_dropout_bwd through
the C ABI (they return before any launch), and the host routing -- which modules run_sequential folds into the dropout GEMM,
and what _LinearFn hands the bindings forward and backward -- with the bindings replaced by recorders.  The kernels themselves
are checked on the GPU (tests/test_gpu_dropout.py)."""
import ctypes

import numpy as np
import pytest
import torch
from torch import nn

import philox_ref

JVAE_ERR_INVALID = -1      # include/jvae_b200.h


# ------------------------------------------------------------------------------------------------ the mask
@pytest.mark.parametrize('ctr,key,want', [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert tuple(int(x) for x in philox_ref.philox4x32_10(ctr, key)) == want


@pytest.mark.parametrize('p', [0.1, 0.5, 0.9])
def test_keep_rate_is_binomial(p):
    n_rows, n_cols = 1000, 1000
    keep = philox_ref.dropout_keep(0x1234_5678_9abc_def0, 3, np.arange(n_rows), np.arange(n_cols), p)
    n = keep.size
    sigma = np.sqrt(n * p * (1 - p))
    assert abs(int(keep.sum()) - n * (1 - p)) < 5 * sigma, (keep.mean(), 1 - p)


def test_mask_depends_on_position_row_and_column_only():
    a = philox_ref.dropout_keep(7, 11, np.arange(64), np.arange(40), 0.5)
    # a sub-block regenerated on its own is the same slice of the mask (the tiling of a kernel cannot matter)
    assert (philox_ref.dropout_keep(7, 11, np.arange(30, 50), np.arange(13, 37), 0.5) == a[30:50, 13:37]).all()
    assert (philox_ref.dropout_keep(7, 12, np.arange(64), np.arange(40), 0.5) != a).mean() > 0.4
    assert not philox_ref.dropout_keep(7, 11, np.arange(8), np.arange(8), 1.0).any()
    assert philox_ref.dropout_keep(7, 11, np.arange(8), np.arange(8), 0.0).all()


# ------------------------------------------------------------------------------------------------ C ABI argument checks
P, c_int, c_float, c_u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_uint64
A, B, D, Z = 0x10000, 0x20000, 0x30000, 0x40000      # 16-byte aligned stand-ins, never dereferenced


def _lib(pkg):
    L = ctypes.CDLL(pkg._native.LIB_PATH)
    L.jvae_last_error.restype = ctypes.c_char_p
    L.jvae_gemm_bf16_dropout.argtypes = [c_int, c_int, c_int, c_int, P, c_int, P, c_int, P, c_int, P, P, c_int, P, c_int,
                                         c_float, c_u64, c_u64, P, P]
    L.jvae_act_dropout_bwd.argtypes = [P, c_int, P, c_int, c_int, c_int, c_int, c_float, c_u64, c_u64, P, P, c_int, P, P]
    return L


@pytest.mark.parametrize('case,args,what', [
    ('p < 0', dict(p=-0.1), b'p must be in [0, 1]'),
    ('p > 1', dict(p=1.5), b'p must be in [0, 1]'),
    ('p nan', dict(p=float('nan')), b'p must be in [0, 1]'),
    ('accumulate', dict(accumulate=1), b'does not accumulate'),
    ('split-K', dict(accumulate=4), b'does not accumulate'),
    ('col_stats', dict(col_stats=B + 0x8000), b'col_stats'),
    ('dgrad mode', dict(mode=1), b'mode NT'),
    ('no output', dict(out=None), b'one output'),
    ('no operand', dict(a=None), b'one output'),
])
def test_gemm_dropout_argument_checks(pkg, case, args, what):
    L = _lib(pkg)
    a = dict(mode=0, a=A, out=D, col_stats=None, accumulate=0, p=0.3)
    a.update(args)
    rc = L.jvae_gemm_bf16_dropout(a['mode'], 256, 128, 64, a['a'], 64, B, 64, None, 1, a['out'], None, 128, a['col_stats'],
                                  a['accumulate'], a['p'], 1, 0, None, None)
    assert rc == JVAE_ERR_INVALID, case
    assert what in L.jvae_last_error(), (case, L.jvae_last_error())


@pytest.mark.parametrize('case,args,what', [
    ('p < 0', dict(p=-1e-3), b'p must be in [0, 1]'),
    ('p > 1', dict(p=2.0), b'p must be in [0, 1]'),
    ('no gradient', dict(da=None), b'bad arguments'),
    ('relu without its output', dict(a_out=None), b'activation output missing'),
    ('no output', dict(dz=None, dbias=None), b'nothing to compute'),
    ('short ld_dz', dict(ld_dz=100), b'ld_dz < N'),
    ('empty', dict(M=0), b'bad arguments'),
])
def test_act_dropout_bwd_argument_checks(pkg, case, args, what):
    L = _lib(pkg)
    a = dict(da=A, a_out=B, dz=D, dbias=Z, p=0.3, ld_dz=1000, M=64)
    a.update(args)
    rc = L.jvae_act_dropout_bwd(a['da'], 1000, a['a_out'], 1000, a['M'], 1000, 1, a['p'], 1, 0, None, a['dz'], a['ld_dz'],
                                a['dbias'], None)
    assert rc == JVAE_ERR_INVALID, case
    assert what in L.jvae_last_error(), (case, L.jvae_last_error())


# ------------------------------------------------------------------------------------------------ host routing
@pytest.fixture()
def engine(pkg):
    from jointvae_b200 import engine
    return engine


@pytest.fixture()
def linear_calls(engine, monkeypatch):
    """engine.linear replaced by a recorder: (in features, out features, act, dropout, out dtype) per call"""
    calls = []

    def rec(x, w, b, act='linear', out_dtype=torch.bfloat16, dropout=None):
        calls.append((w.shape[1], w.shape[0], act, dropout, out_dtype))
        return torch.zeros(x.shape[0], w.shape[0], dtype=out_dtype)
    monkeypatch.setattr(engine, 'linear', rec)
    return calls


def test_reference_mlp_folds_dropout_when_training(pkg, engine, linear_calls):
    net = pkg.ClassificationVariationalNetwork((3, 32, 32), 10, type='cvae', encoder=[512, 256], decoder=[256, 512],
                                               latent_dim=16, latent_sampling=1, dropout=0.3)
    assert sum(isinstance(m, nn.Dropout) for m in net.modules()) == 4
    net.train()
    engine.run_sequential(net.encoder.dense_projs, torch.zeros(4, 3072))
    engine.run_sequential(net.decoder, torch.zeros(4, 16))
    assert linear_calls == [(3072, 512, 'relu', 0.3, torch.bfloat16), (512, 256, 'relu', 0.3, torch.bfloat16),
                            (16, 256, 'relu', 0.3, torch.bfloat16), (256, 512, 'relu', 0.3, torch.bfloat16)]
    linear_calls.clear()
    net.train(False)
    engine.run_sequential(net.encoder.dense_projs, torch.zeros(4, 3072))
    engine.run_sequential(net.decoder, torch.zeros(4, 16))
    assert [c[3] for c in linear_calls] == [None] * 4        # eval: the Dropout is skipped, the GEMM is the plain one
    assert [c[2] for c in linear_calls] == ['relu'] * 4


def test_dropout_without_activation_and_fp32_tail(engine, linear_calls):
    seq = nn.Sequential(nn.Linear(8, 16), nn.Dropout(0.25), nn.Linear(16, 8), nn.Sigmoid(), nn.Dropout(0.5))
    out = engine.run_sequential(seq, torch.zeros(3, 8), out_dtype=torch.float32)
    # a dropout GEMM writes bf16; the container's fp32 output is a cast of it
    assert linear_calls == [(8, 16, 'linear', 0.25, torch.bfloat16), (16, 8, 'sigmoid', 0.5, torch.bfloat16)]
    assert out.dtype == torch.float32
    linear_calls.clear()
    seq.eval()
    engine.run_sequential(seq, torch.zeros(3, 8), out_dtype=torch.float32)
    assert linear_calls == [(8, 16, 'linear', None, torch.bfloat16), (16, 8, 'sigmoid', None, torch.float32)]


@pytest.mark.parametrize('training', [True, False])
@pytest.mark.parametrize('mods', [
    lambda: [nn.Dropout(0.1), nn.Linear(8, 8)],                           # before any Linear
    lambda: [nn.Linear(8, 8), nn.ReLU(), nn.Dropout(0.1), nn.Dropout(0.1)],  # a second Dropout
    lambda: [nn.Linear(8, 8), nn.ReLU(), nn.Identity(), nn.Dropout(0.1)],   # not right after the activation
])
def test_stray_dropout_raises(engine, linear_calls, mods, training):
    seq = nn.Sequential(*mods()).train(training)
    with pytest.raises(NotImplementedError, match='Dropout'):
        engine.run_sequential(seq, torch.zeros(2, 8))


def test_linear_fn_draws_then_regenerates_at_the_same_position(engine, monkeypatch):
    """forward: jvae_gemm_bf16_dropout at the counter's position, counter advanced by one per call; backward:
    jvae_act_dropout_bwd at the position its forward read (a device snapshot), then the two GEMMs on its dz"""
    nat = engine.nat
    calls = []

    def gemm(mode, M, N, K, a, lda, b, ldb, *, out_bf16=None, out_f32=None, **kw):
        calls.append(('gemm', mode, M, N, K))
        (out_bf16 if out_bf16 is not None else out_f32).fill_(0.0)

    def gemm_dropout(M, N, K, a, lda, b, ldb, *, p, seed, offset=0, offset_dev=None, act=0, out_bf16=None, **kw):
        calls.append(('gemm_dropout', p, seed, offset + int(offset_dev[0]), act))
        out_bf16.fill_(1.0)

    def bwd(da, ld_da, a_out, ld_a, M, N, act, p, seed, offset, offset_dev, dz, ld_dz, dbias):
        calls.append(('act_dropout_bwd', act, p, seed, offset + int(offset_dev[0]), a_out is not None, dbias is not None))
        assert ld_dz % 8 == 0 and dz.shape == (M, N)
        dz.fill_(0.5)
        if dbias is not None:
            dbias.fill_(2.0)
    monkeypatch.setattr(nat, 'gemm_bf16', gemm)
    monkeypatch.setattr(nat, 'gemm_bf16_dropout', gemm_dropout)
    monkeypatch.setattr(nat, 'act_dropout_bwd', bwd)
    monkeypatch.setattr(nat, 'cast_f32_bf16', lambda t: t.to(torch.bfloat16))
    dev = torch.device('cpu')
    monkeypatch.setitem(engine._rng_counters, dev, torch.tensor([5], dtype=torch.int64))
    torch.manual_seed(123)
    seed = torch.initial_seed()
    x = torch.randn(4, 16, requires_grad=True)
    w1, b1 = nn.Parameter(torch.randn(12, 16)), nn.Parameter(torch.randn(12))
    w2, b2 = nn.Parameter(torch.randn(8, 12)), nn.Parameter(torch.randn(8))
    h = engine._LinearFn.apply(x, w1, b1, 'relu', torch.bfloat16, 0.2)
    y = engine._LinearFn.apply(h, w2, b2, 'sigmoid', torch.bfloat16, 0.4)
    assert int(engine._rng_counters[dev][0]) == 7
    assert calls == [('gemm_dropout', 0.2, seed, 5, nat.ACT['relu']), ('gemm_dropout', 0.4, seed, 6, nat.ACT['sigmoid'])]
    calls.clear()
    y.float().sum().backward()
    assert calls == [('act_dropout_bwd', nat.ACT['sigmoid'], 0.4, seed, 6, True, True),
                     ('gemm', nat.GEMM_NN, 4, 12, 8), ('gemm', nat.GEMM_TN, 8, 12, 4),
                     ('act_dropout_bwd', nat.ACT['relu'], 0.2, seed, 5, True, True),
                     ('gemm', nat.GEMM_NN, 4, 16, 12), ('gemm', nat.GEMM_TN, 12, 16, 4)]
    assert torch.equal(b1.grad, torch.full((12,), 2.0)) and torch.equal(b2.grad, torch.full((8,), 2.0))
    calls.clear()
    engine._LinearFn.apply(x, w1, b1, 'relu', torch.bfloat16, None)      # no dropout: the plain GEMM, the counter stays
    assert [c[0] for c in calls] == ['gemm'] and int(engine._rng_counters[dev][0]) == 7
