"""Execution engine: maps the reference's layer containers and loss step onto libjvae_sm100.so.

Everything here is host plumbing (PyTorch owns tensors, autograd graph and streams); the arithmetic is in
csrc/*.cu, reached through _native (ctypes, C ABI).  There is ONE execution path: a layer without a native sm_100a
kernel raises NotImplementedError (no vendor-library or eager fallback, no backend switch).
"""
import weakref

import torch
from torch import nn

from . import _native as nat

_rng_counters = {}      # device -> int64[1]: position of the Philox stream of the sampler and the dense-layer dropout


def _rng_counter(device):
    ctr = _rng_counters.get(device)
    if ctr is None:
        ctr = _rng_counters[device] = torch.zeros(1, dtype=torch.int64, device=device)
    return ctr

# Parameter epochs.  The fused Adam (csrc/optim.cu) and the BatchNorm kernels (running statistics) write parameters and
# buffers through raw pointers, which autograd's version counters never see.  Every cache of derived weights (bf16
# operand arrangements, BatchNorm-folded inference weights) therefore keys on these explicit counters as well:
# bump_params() after anything that rewrites parameters in place (Optimizer.step, broadcasts on .data),
# bump_stats() after a train-mode BatchNorm pass updated its running statistics.
PARAM_EPOCH = [0]
STATS_EPOCH = [0]


def bump_params():
    PARAM_EPOCH[0] += 1


def bump_stats():
    STATS_EPOCH[0] += 1



def _r8(n):
    return (n + 7) & ~7


def _bf16_ld8(t):
    """2-D tensor -> bf16 tensor whose row stride is a multiple of 8 elements (TMA needs 16-byte strides)."""
    M, N = t.shape
    if N % 8 == 0:
        if t.dtype == torch.bfloat16 and t.is_contiguous():
            return t
        if t.dtype == torch.float32 and t.is_contiguous():
            return nat.cast_f32_bf16(t)
        return t.to(torch.bfloat16).contiguous()
    buf = torch.zeros((M, _r8(N)), dtype=torch.bfloat16, device=t.device)
    buf[:, :N].copy_(t)
    return buf[:, :N]


def _ld(t):
    return t.stride(0)


# --------------------------------------------------------------------------------------------- dense layers
_wcache = {}


def _weight_bf16(w):
    """bf16 copy of a weight, cached per Parameter object (weak reference: a recycled id() never hits a stale entry)"""
    key = id(w)
    hit = _wcache.get(key)
    ver = (PARAM_EPOCH[0], w._version, w.data_ptr())
    if hit is not None and hit[2]() is w and hit[0] == ver and hit[1].device == w.device:
        return hit[1]
    if len(_wcache) > 256:       # temporaries (the concatenated head weights) leave dead entries behind
        for k in [k for k, v in _wcache.items() if v[2]() is None]:
            del _wcache[k]
    wb = _bf16_ld8(w.detach())
    _wcache[key] = (ver, wb, weakref.ref(w))
    return wb


class _LinearFn(torch.autograd.Function):
    """y = act(x W^T + b) on tcgen05 (csrc/gemm.cu); dgrad / wgrad reuse the same kernel with MN-major operands.
    dropout = p (training-mode nn.Dropout after the activation): the GEMM epilogue multiplies by a Philox keep-mask / (1 - p)
    drawn at the device-side stream position (advanced after the call, like the sampler's), and the backward regenerates
    the mask from a device copy of that position (jvae_act_dropout_bwd) instead of keeping it."""

    @staticmethod
    def forward(ctx, x, w, b, act, out_dtype, dropout):
        M, K = x.shape
        N = w.shape[0]
        xb = _bf16_ld8(x.detach())
        wb = _weight_bf16(w)
        out = torch.empty((M, N), dtype=out_dtype, device=x.device)
        bias = b.detach() if b is not None else None
        pos = None
        if dropout is None:
            nat.gemm_bf16(nat.GEMM_NT, M, N, K, xb, _ld(xb), wb, _ld(wb), bias=bias, act=nat.ACT[act],
                          out_bf16=out if out_dtype == torch.bfloat16 else None,
                          out_f32=out if out_dtype == torch.float32 else None, ldd=N)
        else:
            if out_dtype != torch.bfloat16:
                raise NotImplementedError('the dropout GEMM writes bf16 activations')
            ctr = _rng_counter(x.device)
            pos = ctr.clone()           # the position this call draws at (the counter moves on before the backward)
            ctx.seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
            nat.gemm_bf16_dropout(M, N, K, xb, _ld(xb), wb, _ld(wb), p=dropout, seed=ctx.seed, offset_dev=ctr, bias=bias,
                                  act=nat.ACT[act], out_bf16=out, ldd=N)
            ctr.add_(1)
        ctx.act = act
        ctx.dropout = dropout
        ctx.has_bias = b is not None
        ctx.x_dtype = x.dtype
        ctx.save_for_backward(xb, wb, out if act in ('relu', 'sigmoid', 'leaky') else None, pos)
        return out

    @staticmethod
    def backward(ctx, dy):
        xb, wb, out, pos = ctx.saved_tensors
        M, K = xb.shape
        N = wb.shape[0]
        db = None
        if ctx.dropout is not None:     # dz = dy * keep / (1 - p) * act' and the bias gradient, one launch
            da = dy.to(torch.bfloat16).contiguous()
            dzb = torch.empty((M, _r8(N)), dtype=torch.bfloat16, device=dy.device)[:, :N]
            if ctx.has_bias and ctx.needs_input_grad[2]:
                db = torch.empty(N, dtype=torch.float32, device=dy.device)
            nat.act_dropout_bwd(da, _ld(da), out, N, M, N, nat.ACT[ctx.act], ctx.dropout, ctx.seed, 0, pos, dzb, _ld(dzb), db)
        elif ctx.act == 'relu':
            dy = dy * (out > 0)
        elif ctx.act == 'sigmoid':
            o = out.float()
            dy = dy.float() * o * (1 - o)
        elif ctx.act == 'leaky':        # the output keeps the sign of the pre-activation
            dy = torch.where(out > 0, dy, dy * nat.LEAKY_SLOPE)
        if ctx.dropout is None:
            dzb = _bf16_ld8(dy)
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty((M, K), dtype=ctx.x_dtype, device=dy.device)
            nat.gemm_bf16(nat.GEMM_NN, M, K, N, dzb, _ld(dzb), wb, _ld(wb),
                          out_bf16=dx if dx.dtype == torch.bfloat16 else None,
                          out_f32=dx if dx.dtype == torch.float32 else None, ldd=K)
        if ctx.needs_input_grad[1]:
            dw = torch.empty((N, K), dtype=torch.float32, device=dy.device)
            nat.gemm_bf16(nat.GEMM_TN, N, K, M, dzb, _ld(dzb), xb, _ld(xb), out_f32=dw, ldd=K)
        if ctx.has_bias and ctx.needs_input_grad[2] and ctx.dropout is None:
            db = dy.float().sum(0)
        return dx, dw, db, None, None, None


def linear(x, w, b, act='linear', out_dtype=torch.bfloat16, dropout=None):
    """x (M,K) -> act(x W^T + b) (M,N).  act in linear|relu|sigmoid|leaky.  dropout = p: followed by a training-mode
    Dropout(p) (bf16 output only)."""
    if not x.is_cuda:
        raise nat.NativeError('joint-vae_b200 runs on CUDA devices only (there is no CPU fallback); got a CPU tensor')
    return _LinearFn.apply(x, w, b, act, out_dtype, dropout)


_ACT_OF = {nn.ReLU: 'relu', nn.Sigmoid: 'sigmoid', nn.Identity: 'linear', nn.LeakyReLU: 'leaky'}


def _act_name(m):
    """name of the fused activation a module maps to, or None (LeakyReLU: only the default slope has a kernel)"""
    name = _ACT_OF.get(type(m))
    if name == 'leaky' and abs(m.negative_slope - nat.LEAKY_SLOPE) > 1e-12:
        return None
    return name
_CONV_TYPES = (nn.Conv2d, nn.ConvTranspose2d, nn.BatchNorm2d, nn.MaxPool2d, nn.AvgPool2d, nn.AdaptiveAvgPool2d,
               nn.UpsamplingNearest2d)


def _is_conv_type(m):
    """layers the native conv engine executes, including torchvision's residual blocks and Sequentials of them, and the
    `features` Sequential of torchvision's DenseNets (stem, dense blocks, transitions, norm5)"""
    from .conv_engine import is_residual_block, is_densenet_features
    return isinstance(m, _CONV_TYPES) or is_residual_block(m) or \
        (isinstance(m, nn.Sequential) and len(m) > 0 and all(is_residual_block(b) for b in m)) or is_densenet_features(m)


def run_sequential(seq, x, out_dtype=None, image_out=False):
    """Executes an nn.Sequential container built by the reference-style constructors.
    Linear(+ReLU/Sigmoid/Identity)(+Dropout) runs become one fused GEMM: the Dropout is applied in the GEMM epilogue when the
    container is training and skipped in eval mode; a Dropout anywhere else raises NotImplementedError.  Conv-type runs go to
    run_conv_stack.
    image_out: a conv stack that ends the container returns its result as a channels_last bf16 tensor (the layout the
    fused ELBO kernel reads) instead of fp32 NCHW."""
    mods = list(seq)
    i = 0
    n = len(mods)
    if n == 0:
        return x
    while i < n:
        m = mods[i]
        last_linear = isinstance(m, nn.Linear) and not any(isinstance(k, nn.Linear) for k in mods[i + 1:])
        if isinstance(m, nn.Linear):
            act = 'linear'
            if i + 1 < n and _act_name(mods[i + 1]) is not None:
                act = _act_name(mods[i + 1])
                i += 1
            p = None
            if i + 1 < n and isinstance(mods[i + 1], nn.Dropout):
                if seq.training:
                    p = float(mods[i + 1].p)
                i += 1
            dt = out_dtype if (last_linear and out_dtype is not None and p is None) else torch.bfloat16
            x = linear(x, m.weight, m.bias, act=act, out_dtype=dt, dropout=p)
        elif _is_conv_type(m):
            j = i
            while j < n and (_is_conv_type(mods[j]) or type(mods[j]) in _ACT_OF):
                j += 1
            # a trailing Reshape (categorical imager: channels -> (256, C), conv.py:228-230) is a view of the channels_last image
            tail_is_view = all(type(k).__name__ == 'Reshape' for k in mods[j:])
            x = run_conv_stack(mods[i:j], x, image_out=image_out and (j == n or tail_is_view))
            i = j - 1
        elif isinstance(m, nn.Dropout):
            raise NotImplementedError(f'{type(m).__name__} at index {i} of the container: dropout has a native kernel only '
                                      'after a Linear (+ activation)')
        elif type(m) in _ACT_OF:
            x = m(x)
        elif any(True for _ in m.parameters()):
            raise NotImplementedError(f'{type(m).__name__} has parameters but no native kernel (there is no library path)')
        else:
            x = m(x)     # Reshape, pooling and other parameter-free modules
        i += 1
    if out_dtype is not None and x.dtype != out_dtype:
        x = x.to(out_dtype)
    return x


def run_conv_stack(mods, x, image_out=False):
    """x NCHW through the tcgen05 implicit-GEMM kernels of csrc/conv.cu + csrc/norm.cu (conv_engine).  A layer type
    without a native kernel (MaxPool2d with ceil_mode, DenseNets with dropout or channel offsets that are not multiples of
    8, ...) raises NotImplementedError."""
    from . import conv_engine
    return conv_engine.run(mods, x, image_out=image_out)


# --------------------------------------------------------------------------------------------- sampler
class _SampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, head, eps_in, L, is_sampled, uniform, seed, offset):
        K = head.shape[1] // 2
        head = nat.f32c(head.detach())
        ctr = None
        if eps_in is None:      # Philox stream position on the device, advanced after every draw (graph replays stay fresh)
            ctr = _rng_counter(head.device)
        mu, lv, z, _, eps, en = nat.sample_fwd(head, L, K, eps_in=nat.f32c(eps_in), seed=seed, offset=offset,
                                               is_sampled=is_sampled, uniform=uniform, offset_dev=ctr)
        if ctr is not None:
            ctr.add_(1)
        ctx.save_for_backward(head, lv, eps)
        ctx.dims = (L, K, is_sampled)
        ctx.mark_non_differentiable(eps, en)
        ctx.set_materialize_grads(False)
        return mu, lv, z, eps, en

    @staticmethod
    def backward(ctx, d_mu, d_lv, dz, _de, _den):
        head, lv, eps = ctx.saved_tensors
        L, K, is_sampled = ctx.dims
        if dz is not None and dz.dtype not in (torch.float32, torch.bfloat16):
            dz = dz.float()
        d_head = nat.sample_bwd(head, lv, eps, dz.contiguous() if dz is not None else None, nat.f32c(d_mu),
                                nat.f32c(d_lv), L, K, is_sampled)
        return d_head, None, None, None, None, None, None


def sample(head, L, eps_in=None, is_sampled=True, uniform=False):
    """head (B,2K) = [mean | raw log_var] -> mean, clip(log_var), z (L+1,B,K), eps (L,B,K), |eps|^2 (L,B).
    csrc/sampler.cu; eps_in (L+1,B,K) injects the noise, else Philox4x32-10 keyed by torch's seed."""
    if not head.is_cuda:
        raise nat.NativeError('joint-vae_b200 runs on CUDA devices only (there is no CPU fallback); got a CPU tensor')
    seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
    return _SampleFn.apply(head, eps_in, L, is_sampled, uniform, seed, 0)


# --------------------------------------------------------------------------------------------- fused ELBO
class _ElboTrainFn(torch.autograd.Function):
    """Forward: jvae_elbo_train_fwd; backward of `total` only (what the reference differentiates, cvae.py:2450)."""

    @staticmethod
    def forward(ctx, x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma, cfg):
        out = nat.elbo_train_fwd(cfg, x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma)
        ctx.cfg = cfg
        # the backward kernel recovers the per-sample sigma^2 of sigma=rmse from cross_x (include/jvae_b200.h)
        ctx.save_for_backward(x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma,
                              out['cross_x'] if cfg.sigma_is_rmse else out['wmse'])
        ctx.set_materialize_grads(False)
        names = ('kl', 'zdist', 'var_kl', 'wmse', 'cross_x', 'cross_y', 'total', 'dzdist')
        ctx.mark_non_differentiable(out['finite'])
        return tuple(out[k] for k in names) + (out['finite'],)

    @staticmethod
    def backward(ctx, *grads):
        g_total = grads[6]
        if any(g is not None for i, g in enumerate(grads) if i != 6):
            raise NotImplementedError('the fused ELBO differentiates `total` only (as the reference trains on '
                                      'total.mean()); detach the other loss terms')
        x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma, wmse = ctx.saved_tensors
        cfg = ctx.cfg
        need_it = ctx.needs_input_grad[7] and cfg.var_dim in (nat.VAR_DIM['diag'], nat.VAR_DIM['full'])
        d_xr, d_mu, d_lv, d_lg, d_means, d_it, d_sigma = nat.elbo_train_bwd(
            cfg, g_total.contiguous(), x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma, wmse,
            need_inv_trans=need_it)
        if ctx.needs_input_grad[7] and not need_it and inv_trans.requires_grad:
            raise NotImplementedError('a scalar prior variance is not a learned parameter (priors.py:79)')
        ng = ctx.needs_input_grad
        return (None, d_xr if ng[1] else None, d_mu if ng[2] else None, d_lv if ng[3] else None,
                d_lg if ng[4] else None, None, d_means if ng[6] else None, d_it if ng[7] else None,
                d_sigma.view_as(sigma) if (ng[8] and d_sigma is not None) else None, None)


def elbo_train(cfg, x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma):
    return _ElboTrainFn.apply(x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma, cfg)


def elbo_eval(cfg, x, x_reco, mu, log_var, z, eps_norm, logits, means, inv_trans, sigma, **kw):
    return nat.elbo_eval_fwd(cfg, x, x_reco, mu, log_var, z, eps_norm, logits, means, inv_trans, sigma, **kw)
