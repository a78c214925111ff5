"""ctypes binding of libjvae_sm100.so (the C ABI declared in include/jvae_b200.h).

The host side of this package is PyTorch (device memory, streams, torch.distributed); every arithmetic
step of the hot path goes through this module.  There is no CPU / eager fallback: if the library cannot
be loaded, or a tensor is not on a CUDA device, calls raise.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libjvae_sm100.so')

F32, BF16 = 0, 1
VAR_DIM = {'scalar': 0, 'diag': 1, 'full': 2}
PRIOR_KIND = {'gaussian': 0, 'tilted': 1, 'uniform': 2}
ACT = {'none': 0, 'linear': 0, 'relu': 1, 'sigmoid': 2, 'leaky': 3}
OUT_F32, IN_F32 = 0x100, 0x200      # include/jvae_b200.h: JVAE_OUT_F32 / JVAE_IN_F32 flags of the `act` argument
LEAKY_SLOPE = 0.01      # JVAE_LEAKY_SLOPE: nn.LeakyReLU() default, the only slope the reference builds (misc.py:27)
NSCORES, NPRED = 16, 4
SCORE_INDEX = {'elbo': 0, 'max': 0, 'sum': 1, 'mean': 2, 'iws': 3, 'soft': 4, 'softkl': 4, 'zdist': 5, 'kl': 6,
               'mse': 7, 'wmse': 8, 'logits': 9, 'baseline': 10, 'hyz': 11, 'std': 12, 'softiws': 13}
PRED_INDEX = {'loss': 0, 'esty': 1, 'closest': 2, 'iws': 3}

c_void_p, c_int, c_float, c_size_t = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
c_u64, c_i64 = ctypes.c_uint64, ctypes.c_int64


class ElboCfg(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ('B', 'L', 'K', 'C', 'D', 'xreco_dtype', 'logits_dtype', 'var_dim', 'prior_kind', 'conditional',
                 'has_xreco', 'has_logits', 'sigma_is_log', 'sigma_is_rmse')] + \
               [(n, ctypes.c_float) for n in ('beta', 'gamma_w', 'var_w', 'tau', 'alpha')] + \
               [(n, ctypes.c_int32) for n in ('prior_stats_ready', 'categorical', 'cat_group', 'sigma_per_sample')]


class BnReduce(ctypes.Structure):
    """include/jvae_b200.h: jvae_bn_reduce"""
    _fields_ = [('y', ctypes.c_void_p), ('ld_y', ctypes.c_int32), ('save_mean_rstd', ctypes.c_void_p),
                ('gamma', ctypes.c_void_p), ('beta', ctypes.c_void_p), ('act', ctypes.c_int32)]


class BatchCfg(ctypes.Structure):          # include/jvae_b200.h: jvae_batch_cfg
    _fields_ = [(n, ctypes.c_int32) for n in ('H', 'W', 'C', 'out_H', 'out_W', 'crop_pad', 'flip_first', 'post_off_y',
                                              'post_off_x')]


class PackJob(ctypes.Structure):          # include/jvae_b200.h: jvae_pack_job
    _fields_ = [('src', ctypes.c_void_p), ('dst', ctypes.c_void_p)] + \
               [(n, ctypes.c_int64) for n in ('s_r1', 's_r0', 's_t', 's_c1', 's_c0')] + \
               [(n, ctypes.c_int32) for n in ('rows', 'rows_pad', 'R0', 'T', 'tap_off', 'cols', 'cols_pad', 'C0', 'dst_f32',
                                              'first_block')]


class NativeError(RuntimeError):
    pass


_lib = None


def lib():
    """Loads the library once; raises if it is missing (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(f'{LIB_PATH} is not built: run `python -c "import __graft_entry__ as g; g.build()"` '
                          'in a container with nvcc; there is no CPU fallback')
    L = ctypes.CDLL(LIB_PATH)
    L.jvae_last_error.restype = ctypes.c_char_p
    L.jvae_abi_version.restype = c_int
    L.jvae_launch_count.restype = c_i64
    L.jvae_device_info.argtypes = [c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int), ctypes.POINTER(c_int)]
    L.jvae_elbo_workspace_bytes.restype = c_size_t
    L.jvae_elbo_workspace_bytes.argtypes = [ctypes.POINTER(ElboCfg)]
    P = c_void_p
    L.jvae_elbo_train_fwd.argtypes = [ctypes.POINTER(ElboCfg)] + [P] * 19 + [c_size_t, P]
    L.jvae_elbo_train_bwd.argtypes = [ctypes.POINTER(ElboCfg)] + [P] * 19 + [c_size_t, P]
    L.jvae_elbo_eval_fwd.argtypes = [ctypes.POINTER(ElboCfg)] + [P] * 23 + [c_size_t, P]
    L.jvae_sample_fwd.argtypes = [c_int, c_int, c_int, P, P, c_u64, c_u64, P, c_int, c_int, P, P, P, P, P, P, P]
    L.jvae_sample_bwd.argtypes = [c_int, c_int, c_int, P, P, P, P, c_int, P, P, c_int, P, P]
    L.jvae_cast_f32_bf16.argtypes = [P, P, c_size_t, P]
    L.jvae_cast_bf16_f32.argtypes = [P, P, c_size_t, P]
    L.jvae_nchw_to_nhwc_bf16.argtypes = [P, P, c_int, c_int, c_int, c_int, c_int, P]
    L.jvae_nhwc_bf16_to_nchw.argtypes = [P, P, c_int, c_int, c_int, c_int, c_int, P]
    L.jvae_grad_sqnorm.argtypes = [P, c_int, c_size_t, P, P, P, P]
    L.jvae_adam_step.argtypes = [P, P, P, P, c_int, c_size_t, P, c_float, c_float, c_float, c_float, c_float,
                                 c_float, c_int, P, P, P, P, c_float, P]
    for name in ('jvae_gemm_bf16', 'jvae_selftest'):
        if not hasattr(L, name):
            raise NativeError(f'{LIB_PATH} does not export {name}: stale build')
    L.jvae_gemm_bf16.argtypes = [c_int, c_int, c_int, c_int, P, c_int, P, c_int, P, c_int, P, P, c_int, P, c_int, P]
    L.jvae_selftest.argtypes = [c_int]
    L.jvae_probe_descriptors.argtypes = [c_int]
    L.jvae_probe_poison.argtypes = [ctypes.c_uint, P]
    L.jvae_profile_enable.argtypes = [c_int]
    L.jvae_im2col_bf16.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(ctypes.c_int16), ctypes.POINTER(ctypes.c_int16), c_int, c_int, c_int, P, c_int, c_int, P]
    L.jvae_profile_drain.argtypes = [P, P, c_int]
    I16P = ctypes.POINTER(ctypes.c_int16)
    L.jvae_conv_gather_gemm.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, I16P, I16P, c_int,
                                        c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int,
                                        P, P]
    L.jvae_conv_gather_gemm_bn.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, I16P, I16P, c_int,
                                           c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P,
                                           c_int, P, ctypes.POINTER(BnReduce), ctypes.POINTER(c_int), P]
    L.jvae_conv_wgrad.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, I16P, I16P,
                                  c_int, P, c_int, c_int, c_int, P]
    L.jvae_conv_subpixel_gemm.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, I16P, I16P, I16P, I16P,
                                          I16P, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, P, c_int, P, P]
    L.jvae_conv_wgrad_emulate.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, I16P, I16P,
                                          c_int, P, c_int, c_int, c_int, ctypes.POINTER(c_int)]
    L.jvae_conv_halo_emulate.argtypes = [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, I16P, I16P, I16P, c_int,
                                         I16P, I16P, c_int, c_int, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                         c_int, P, c_int, ctypes.POINTER(c_int)]
    L.jvae_bn_stats.argtypes = [P, c_size_t, c_int, c_int, P, P]
    L.jvae_bn_apply_fwd.argtypes = [P, c_size_t, c_int, c_int, P, P, P, c_float, c_float, P, P, P, c_int, c_int, P, c_int,
                                    P, P]
    L.jvae_bn_bwd.argtypes = [P, c_int, P, c_int, c_size_t, c_int, P, P, P, c_int, P, P, c_int, P, P, c_int, P]
    L.jvae_act_bwd.argtypes = [P, c_int, P, c_int, c_size_t, c_int, c_int, P, c_int, P, P]
    L.jvae_bn_stats_ld.argtypes = [P, c_size_t, c_int, c_int, P, c_int, P]
    L.jvae_bn_preact_fwd.argtypes = [P, c_size_t, c_int, c_int, P, c_int, P, P, c_float, c_float, P, P, P, c_int, c_int, P,
                                     c_int, P, P]
    L.jvae_bn_preact_bwd.argtypes = [P, c_int, P, c_int, c_size_t, c_int, P, P, P, P, P, c_float, c_int, c_int, P, P, c_int,
                                     P, P, P]
    L.jvae_cast_f32_bf16_ld.argtypes = [P, c_int, P, c_int, c_size_t, c_int, P]
    L.jvae_maxpool_fwd.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, P]
    L.jvae_maxpool_bwd.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, P, c_int, P]
    L.jvae_upsample2.argtypes = [P, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, P]
    L.jvae_maxpool_pad_fwd.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, P]
    L.jvae_maxpool_pad_bwd.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, P, c_int, P]
    L.jvae_avgpool.argtypes = [P, c_int, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]
    L.jvae_add_act.argtypes = [P, c_int, P, c_int, c_size_t, c_int, c_int, P, c_int, P]
    L.jvae_vsum_rows.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, P, P, c_int, P]
    L.jvae_vstack_rows.argtypes = [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, P]
    L.jvae_elbo_prior_stats.argtypes = [ctypes.POINTER(ElboCfg), P, P, P, c_size_t, P]
    L.jvae_batch_u8_to_f32.argtypes = [ctypes.POINTER(BatchCfg), P, ctypes.c_longlong, P, c_int, P, P, P, P]
    L.jvae_last_conv_kernel.restype = c_int
    L.jvae_pack_job_blocks.argtypes = [ctypes.c_longlong, c_int, c_int]
    L.jvae_pack_weights.argtypes = [P, c_int, P, c_int, P]
    if L.jvae_abi_version() != 16:
        raise NativeError('ABI version mismatch between _native.py and libjvae_sm100.so')
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise NativeError(lib().jvae_last_error().decode() + f' (status {rc})')


def launch_count():
    return int(lib().jvae_launch_count())


def ptr(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeError('libjvae_sm100 works on CUDA tensors only (got a CPU tensor); there is no CPU fallback')
    if not (t.is_contiguous() or (t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last))):
        raise NativeError('non-dense tensor passed to the native library')
    return c_void_p(t.data_ptr())


def ptr2d(t):
    """2-D operand of the GEMM: unit inner stride, any 16-byte aligned row stride"""
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeError('libjvae_sm100 works on CUDA tensors only (got a CPU tensor); there is no CPU fallback')
    if t.dim() != 2 or t.stride(1) != 1:
        raise NativeError('GEMM operands must be 2-D with unit inner stride')
    return c_void_p(t.data_ptr())


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def dtype_code(t):
    if t is None or t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise NativeError(f'unsupported dtype {t.dtype}')


def f32c(t):
    """contiguous float32 view/copy of t (None passes through)"""
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


_ws_cache = {}

# bench.py sets PROFILE = {'elbo_train_fwd': [], ...}: CUDA event pairs recorded on the launching stream around the
# named entry point (the roofline's per-launch duration is measured live inside the timed region)
PROFILE = None


PROF_TAGS = {1: 'elbo_train_fwd', 2: 'elbo_train_bwd', 3: 'elbo_eval_fwd', 4: 'conv_halo_kernel', 5: 'conv_gather_gemm_kernel',
             6: 'conv_wgrad_halo_kernel', 7: 'conv_wgrad_kernel'}
CONV_TAGS = (4, 5, 6, 7)


def profile_native(on):
    """per-launch events recorded INSIDE the library around the fused ELBO kernels (include/jvae_b200.h: jvae_profile_enable)"""
    check(lib().jvae_profile_enable(int(bool(on))))


def profile_drain(max_records=1 << 16):
    """-> {entry point: [ms per launch]} of the launches profiled since the last drain (synchronises)"""
    tags = (ctypes.c_int32 * max_records)()
    ms = (ctypes.c_float * max_records)()
    n = lib().jvae_profile_drain(tags, ms, max_records)
    out = {}
    conv = []
    for i in range(n):
        out.setdefault(PROF_TAGS.get(tags[i], str(tags[i])), []).append(float(ms[i]))
        if tags[i] in CONV_TAGS:
            conv.append((PROF_TAGS[tags[i]], float(ms[i])))
    # convolution launches in call order: bench.py pairs them with the algorithmic FLOPs the Python side noted per call
    out['conv_launches'] = conv
    return out


class _timed:
    def __init__(self, name):
        self.on = PROFILE is not None and name in PROFILE
        self.name = name

    def __enter__(self):
        if self.on:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if self.on:
            self.b.record()
            PROFILE[self.name].append((self.a, self.b))


CONV_KERNELS = {1: 'conv_halo_kernel', 2: 'conv_gather_gemm_kernel', 3: 'conv_wgrad_halo_kernel', 4: 'conv_wgrad_kernel'}


CONV_FLOPS = None      # bench.py sets a list: algorithmic FLOPs of every convolution entry-point call, in call order


class _timed_conv:
    """PROFILE['conv']: (start event, stop event, algorithmic FLOPs, kernel name) per convolution launch"""

    def __init__(self, flops):
        self.on = PROFILE is not None and 'conv' in PROFILE
        self.flops = flops

    def __enter__(self):
        if CONV_FLOPS is not None:
            CONV_FLOPS.append(self.flops)
            self.n0 = launch_count()
        if self.on:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def cancel(self):
        """the entry point launched nothing (JVAE_NOT_COVERED): no record"""
        if CONV_FLOPS is not None:
            CONV_FLOPS.pop()
        self.on = False
        self.cancelled = True

    def __exit__(self, *exc):
        if CONV_FLOPS is not None and not getattr(self, 'cancelled', False):
            # an entry point that launched several kernels (stride-2 weight gradients, one launch per parity plane) left one
            # native record per launch: the call's FLOPs are spread over them
            n = launch_count() - self.n0
            if n > 1:
                CONV_FLOPS.pop()
                CONV_FLOPS.extend([self.flops / n] * n)
        if self.on:
            self.b.record()
            PROFILE['conv'].append((self.a, self.b, self.flops, CONV_KERNELS.get(int(lib().jvae_last_conv_kernel()), '?')))


def workspace(cfg, device):
    """Scratch buffer of the ELBO entry points.  ONE buffer per workspace layout (the layout depends on B, L, K and the
    number of priors): the kernels keep their arrival counters zero between launches only within a layout, so a buffer
    is never shared between two layouts (train and eval steps of different L or batch size get their own)."""
    n = int(lib().jvae_elbo_workspace_bytes(ctypes.byref(cfg)))
    key = (device, torch.cuda.current_stream().cuda_stream, cfg.B, cfg.L, cfg.K, cfg.C if cfg.conditional else 1,
           cfg.var_dim == VAR_DIM['full'])
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < n:
        if len(_ws_cache) > 64:
            _ws_cache.clear()
        ws = torch.zeros(max(n, 1 << 12), dtype=torch.uint8, device=device)    # counters start at zero
        _ws_cache[key] = ws
    return ws, n


def make_cfg(*, B, L, K, C, D, x_reco, logits, var_dim, prior_kind, conditional, sigma_is_log, sigma_is_rmse,
             beta, gamma_w, var_w, tau=0.0, alpha=0.0, prior_stats_ready=False, categorical=False, cat_group=0,
             sigma_per_sample=False):
    return ElboCfg(categorical=int(bool(categorical)), cat_group=int(cat_group), sigma_per_sample=int(bool(sigma_per_sample)), prior_stats_ready=int(bool(prior_stats_ready)), B=B, L=L, K=K, C=C, D=D, xreco_dtype=dtype_code(x_reco), logits_dtype=dtype_code(logits),
                   var_dim=VAR_DIM[var_dim], prior_kind=PRIOR_KIND[prior_kind], conditional=int(bool(conditional)),
                   has_xreco=int(x_reco is not None), has_logits=int(logits is not None),
                   sigma_is_log=int(bool(sigma_is_log)), sigma_is_rmse=int(bool(sigma_is_rmse)),
                   beta=float(beta), gamma_w=float(gamma_w or 0.0), var_w=float(var_w), tau=float(tau or 0.0),
                   alpha=float(alpha or 0.0))


def elbo_prior_stats(cfg, means, inv_trans):
    """include/jvae_b200.h: jvae_elbo_prior_stats (run early; then pass prior_stats_ready=True to make_cfg)"""
    ws, n = workspace(cfg, means.device)
    check(lib().jvae_elbo_prior_stats(ctypes.byref(cfg), ptr(means), ptr(inv_trans), ptr(ws), n, stream()))


def elbo_train_fwd(cfg, x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma):
    """-> dict of (B,) f32 tensors + 'finite' int32 flag tensor.  include/jvae_b200.h: jvae_elbo_train_fwd"""
    dev = mu.device
    B = cfg.B
    out = torch.empty((8, B), dtype=torch.float32, device=dev)
    flag = torch.ones(1, dtype=torch.int32, device=dev)       # the kernel clears it on a non-finite total
    ws, n = workspace(cfg, dev)
    with _timed('elbo_train_fwd'):
        check(lib().jvae_elbo_train_fwd(ctypes.byref(cfg), ptr(x), ptr(x_reco), ptr(mu), ptr(log_var), ptr(logits),
                                        ptr(y), ptr(means), ptr(inv_trans), ptr(sigma),
                                        *[c_void_p(out[i].data_ptr()) for i in range(8)], ptr(flag), ptr(ws), n, stream()))
    names = ('kl', 'zdist', 'var_kl', 'wmse', 'cross_x', 'cross_y', 'total', 'dzdist')
    res = {k: out[i] for i, k in enumerate(names)}
    res['finite'] = flag
    return res


def elbo_train_bwd(cfg, g, x, x_reco, mu, log_var, logits, y, means, inv_trans, sigma, wmse, need_inv_trans=False):
    dev = mu.device
    d_xr = torch.empty_like(x_reco) if x_reco is not None else None
    d_mu = torch.empty_like(mu)
    d_lv = torch.empty_like(log_var)
    d_logits = torch.empty_like(logits) if logits is not None else None
    d_means = torch.empty_like(means)
    d_it = torch.empty_like(inv_trans) if need_inv_trans else None
    d_sigma = torch.empty(cfg.B if cfg.sigma_per_sample else 1, dtype=torch.float32, device=dev) if x_reco is not None else None
    ws, n = workspace(cfg, dev) if cfg.var_dim == VAR_DIM['full'] else (None, 0)
    with _timed('elbo_train_bwd'):
        check(lib().jvae_elbo_train_bwd(ctypes.byref(cfg), ptr(g), ptr(x), ptr(x_reco), ptr(mu), ptr(log_var),
                                        ptr(logits), ptr(y), ptr(means), ptr(inv_trans), ptr(sigma), ptr(wmse), ptr(d_xr),
                                        ptr(d_mu), ptr(d_lv), ptr(d_logits), ptr(d_means), ptr(d_it), ptr(d_sigma),
                                        ptr(ws), n, stream()))
    return d_xr, d_mu, d_lv, d_logits, d_means, d_it, d_sigma


def elbo_eval_fwd(cfg, x, x_reco, mu, log_var, z, eps_norm, logits, means, inv_trans, sigma, *, want_iws=True,
                  want_scores=True):
    """-> dict: per-class (Cp,B) kl zdist var_kl iws, total (nT,B), cross_y (C,B), per-sample wmse cross_x dzdist,
    logits (B,C), scores (B,16), preds (B,4).  include/jvae_b200.h: jvae_elbo_eval_fwd"""
    dev = mu.device
    B, C = cfg.B, cfg.C
    Cp = C if cfg.conditional else 1
    add_cy = bool(cfg.has_logits) and cfg.gamma_w != 0.0
    nT = Cp if Cp > 1 else (C if add_cy else 1)
    f = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
    kl, zdist, var_kl = f(Cp, B), f(Cp, B), f(Cp, B)
    total = f(nT, B)
    iws = f(Cp, B) if (want_iws and cfg.has_xreco and z is not None and eps_norm is not None) else None
    cross_y = f(C, B) if cfg.has_logits else None
    logits_out = f(B, C) if cfg.has_logits else None
    wmse = f(B) if cfg.has_xreco else None
    cross_x = f(B) if cfg.has_xreco else None
    dzdist = f(B) if cfg.conditional else None
    scores = f(B, NSCORES) if want_scores else None
    preds = torch.empty((B, NPRED), dtype=torch.int32, device=dev) if want_scores else None
    ws, n = workspace(cfg, dev)
    with _timed('elbo_eval_fwd'):
      check(lib().jvae_elbo_eval_fwd(ctypes.byref(cfg), ptr(x), ptr(x_reco), ptr(mu), ptr(log_var),
                                   ptr(z) if iws is not None else None, ptr(eps_norm) if iws is not None else None,
                                   ptr(logits), ptr(means), ptr(inv_trans), ptr(sigma),
                                   ptr(kl), ptr(zdist), ptr(var_kl), ptr(total), ptr(iws), ptr(cross_y), ptr(wmse),
                                   ptr(cross_x), ptr(dzdist), ptr(logits_out), ptr(scores), ptr(preds), ptr(ws), n,
                                   stream()))
    return dict(kl=kl, zdist=zdist, var_kl=var_kl, total=total, iws=iws, cross_y=cross_y, wmse=wmse, cross_x=cross_x,
                dzdist=dzdist, logits=logits_out, scores=scores, preds=preds)


def sample_fwd(head, L, K, eps_in=None, seed=0, offset=0, is_sampled=True, uniform=False, want_bf16=False, offset_dev=None):
    """head (B,2K) f32 -> mu, log_var (B,K), z (L+1,B,K), z_bf16|None, eps (L,B,K), eps_norm (L,B)"""
    dev = head.device
    B = head.shape[0]
    f = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
    mu, lv, z, eps, en = f(B, K), f(B, K), f(L + 1, B, K), f(L, B, K), f(L, B)
    z16 = torch.empty((L + 1, B, K), dtype=torch.bfloat16, device=dev) if want_bf16 else None
    check(lib().jvae_sample_fwd(B, L, K, ptr(head), ptr(eps_in), seed, offset, ptr(offset_dev), int(is_sampled), int(uniform), ptr(mu),
                                ptr(lv), ptr(z), ptr(z16), ptr(eps), ptr(en), stream()))
    return mu, lv, z, z16, eps, en


def sample_bwd(head, log_var, eps, dz, d_mu, d_lv, L, K, is_sampled=True):
    B = head.shape[0]
    d_head = torch.empty_like(head)
    check(lib().jvae_sample_bwd(B, L, K, ptr(head), ptr(log_var), ptr(eps), ptr(dz), dtype_code(dz), ptr(d_mu),
                                ptr(d_lv), int(is_sampled), ptr(d_head), stream()))
    return d_head


def cast_f32_bf16(src, dst=None):
    if dst is None:
        dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    check(lib().jvae_cast_f32_bf16(ptr(src), ptr(dst), src.numel(), stream()))
    return dst


def cast_bf16_f32(src, dst=None):
    if dst is None:
        dst = torch.empty(src.shape, dtype=torch.float32, device=src.device)
    check(lib().jvae_cast_bf16_f32(ptr(src), ptr(dst), src.numel(), stream()))
    return dst


def nchw_to_nhwc_bf16(src, c_pad=None):
    n, c, h, w = src.shape
    c_pad = c_pad or c
    dst = torch.empty((n, h, w, c_pad), dtype=torch.bfloat16, device=src.device)
    check(lib().jvae_nchw_to_nhwc_bf16(ptr(src), ptr(dst), n, c, h, w, c_pad, stream()))
    return dst


def nhwc_bf16_to_nchw(src, c=None):
    n, h, w, c_pad = src.shape
    c = c or c_pad
    dst = torch.empty((n, c, h, w), dtype=torch.float32, device=src.device)
    check(lib().jvae_nhwc_bf16_to_nchw(ptr(src), ptr(dst), n, c, h, w, c_pad, stream()))
    return dst


def batch_u8_to_f32(cfg, src, index, flip, crop_ij, out):
    """src uint8 (n, H, W, C) on the device; index (B) int64; flip (B) uint8 or None; crop_ij (B, 2) int32 or None"""
    check(lib().jvae_batch_u8_to_f32(ctypes.byref(cfg), ptr(src), src.shape[0], ptr(index), index.numel(), ptr(flip),
                                     ptr(crop_ij), ptr(out), stream()))
    return out


def pack_job_blocks(rows_pad, T, cols_pad):
    return int(lib().jvae_pack_job_blocks(rows_pad, T, cols_pad))


def pack_weights(jobs_dev, n_jobs, taps_dev, total_blocks):
    """include/jvae_b200.h: jvae_pack_weights (job table and tap table are device tensors built by conv_engine.PackPlan)"""
    check(lib().jvae_pack_weights(rawptr(jobs_dev), n_jobs, rawptr(taps_dev), total_blocks, stream()))


OPT_CHUNK = 256      # include/jvae_b200.h: JVAE_OPT_CHUNK


def grad_sqnorm(grad, out, chunk_seg=None, seg_active=None):
    check(lib().jvae_grad_sqnorm(ptr(grad), dtype_code(grad), grad.numel(), ptr(out), ptr(chunk_seg), ptr(seg_active), stream()))


def adam_step(p, m, v, grad, norm2, *, max_norm, lr, beta1, beta2, eps, weight_decay, chunk_seg, seg_active, seg_step, seg_bc,
              grad_scale=1.0):
    """include/jvae_b200.h: jvae_adam_step (per-parameter step counts on the device; gradient-less parameters are skipped)"""
    check(lib().jvae_adam_step(ptr(p), ptr(m), ptr(v), ptr(grad), dtype_code(grad), p.numel(), ptr(norm2),
                               float(max_norm or 0.0), lr, beta1, beta2, eps, weight_decay, seg_active.numel(), ptr(chunk_seg),
                               ptr(seg_active), ptr(seg_step), ptr(seg_bc), grad_scale, stream()))


GEMM_NT, GEMM_NN, GEMM_TN = 0, 1, 2


def gemm_bf16(mode, M, N, K, a, lda, b, ldb, *, bias=None, act=0, out_bf16=None, out_f32=None, ldd=None,
              col_stats=None, accumulate=False):
    check(lib().jvae_gemm_bf16(mode, M, N, K, ptr2d(a), lda, ptr2d(b), ldb, ptr(bias), act, ptr(out_bf16), ptr(out_f32),
                               ldd if ldd is not None else N, ptr(col_stats), int(accumulate), stream()))     # accumulate: 0 / 1 / n >= 2 (split-K)


def rawptr(t):
    """device pointer of a tensor the caller has laid out itself (NHWC activations with padded channel strides)"""
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeError('libjvae_sm100 works on CUDA tensors only (got a CPU tensor); there is no CPU fallback')
    return c_void_p(t.data_ptr())


_sm_count = {}


def sm_count():
    dev = torch.cuda.current_device()
    if dev not in _sm_count:
        _sm_count[dev] = torch.cuda.get_device_properties(dev).multi_processor_count
    return _sm_count[dev]


def im2col(x, N, H, W, C, ld_x, taps, in_stride, Hq, Wq, out, tap_major=False):
    """include/jvae_b200.h: jvae_im2col_bf16; out (N*Hq*Wq, >= C*T) bf16; columns ci * T + t, or t * C + ci when tap_major"""
    check(lib().jvae_im2col_bf16(rawptr(x), N, H, W, C, ld_x, len(taps[0]), taps[0], taps[1], in_stride, Hq, Wq, rawptr(out),
                                 out.stride(0), int(tap_major), stream()))


def taps_arg(taps):
    """list of (dy, dx) -> two ctypes int16 arrays"""
    n = len(taps)
    A = ctypes.c_int16 * n
    return A(*[int(t[0]) for t in taps]), A(*[int(t[1]) for t in taps])


def conv_gather_gemm(inp, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, taps, in_stride, Hq, Wq, out, Ho, Wo, Cout, ld_out,
                     out_s=(1, 1), out_o=(0, 0), bias=None, act=0, stats=None, bn=None):
    """include/jvae_b200.h: jvae_conv_gather_gemm[_bn].  taps = (dy_array, dx_array) from taps_arg.
    bn = dict(y, ld_y, save, gamma, beta, act): fold the previous layer's BatchNorm-backward reduction into this
    data-gradient launch (sums go to `stats`); returns True when the launched kernel did it."""
    if bn is None:
        with _timed_conv(2.0 * N * Hq * Wq * len(taps[0]) * Cin * Cout):
            check(lib().jvae_conv_gather_gemm(rawptr(inp), N, H, W, Cin, ld_in, rawptr(wmat), Cout_pad, ldw, len(taps[0]),
                                              taps[0], taps[1], in_stride, Hq, Wq, rawptr(out), Ho, Wo, Cout, ld_out,
                                              out_s[0], out_s[1], out_o[0], out_o[1], rawptr(bias), act, rawptr(stats),
                                              stream()))
        return False
    d = BnReduce(y=bn['y'].data_ptr(), ld_y=bn['ld_y'], save_mean_rstd=bn['save'].data_ptr(),
                 gamma=bn['gamma'].data_ptr() if bn['gamma'] is not None else None,
                 beta=bn['beta'].data_ptr() if bn['beta'] is not None else None, act=bn['act'])
    fused = c_int(0)
    check(lib().jvae_conv_gather_gemm_bn(rawptr(inp), N, H, W, Cin, ld_in, rawptr(wmat), Cout_pad, ldw, len(taps[0]),
                                         taps[0], taps[1], in_stride, Hq, Wq, rawptr(out), Ho, Wo, Cout, ld_out, out_s[0],
                                         out_s[1], out_o[0], out_o[1], rawptr(bias), act, rawptr(stats), ctypes.byref(d),
                                         ctypes.byref(fused), stream()))
    return bool(fused.value)


NOT_COVERED = 1


def phases_arg(ops):
    """gather-op dicts of the sub-pixel phases (conv_engine.deconv_form) -> the tables of jvae_conv_subpixel_gemm:
    (taps per phase, phase_oy, phase_ox, tap_dy, tap_dx, total taps) with the taps concatenated phase by phase"""
    A = ctypes.c_int16 * len(ops)
    taps = [t for op in ops for t in op['taps']]
    dy, dx = taps_arg(taps)
    return (A(*[len(op['taps']) for op in ops]), A(*[int(op['out_o'][0]) for op in ops]), A(*[int(op['out_o'][1]) for op in ops]),
            dy, dx, len(taps))


def conv_subpixel_gemm(inp, N, H, W, Cin, ld_in, wmat, Cout_pad, ldw, phases, Hq, Wq, out, Ho, Wo, Cout, ld_out, out_s,
                       bias=None, act=0, stats=None):
    """include/jvae_b200.h: jvae_conv_subpixel_gemm.  phases = phases_arg(ops).  Returns False (nothing launched) when the
    merged kernel does not cover the geometry: the caller then launches the phases one by one."""
    pn, poy, pox, dy, dx, T = phases
    with _timed_conv(2.0 * N * Hq * Wq * T * Cin * Cout) as tc:
        rc = lib().jvae_conv_subpixel_gemm(rawptr(inp), N, H, W, Cin, ld_in, rawptr(wmat), Cout_pad, ldw, len(pn), pn, poy, pox,
                                           dy, dx, Hq, Wq, rawptr(out), Ho, Wo, Cout, ld_out, out_s, rawptr(bias), act,
                                           rawptr(stats), stream())
        if rc == NOT_COVERED:
            tc.cancel()
    if rc == NOT_COVERED:
        return False
    check(rc)
    return True


def conv_halo_emulate(inp, Cin, wmat, Cout_pad, taps, in_stride, Hq, Wq, out, Cout, out_s=(1, 1), out_o=(0, 0), bias=None,
                      act=0, phases=None):
    """include/jvae_b200.h: jvae_conv_halo_emulate (HOST tensors, fp32; test aid).  inp (N,H,W,ld_in), wmat (Cout_pad, ldw),
    out (N,Ho,Wo,ld_out) CPU float32.  Returns the info list, or None when the halo kernel does not take the geometry."""
    for t in (inp, wmat, out):
        assert t.device.type == 'cpu' and t.dtype == torch.float32 and t.is_contiguous()
    N, H, W, ld_in = inp.shape
    _, Ho, Wo, ld_out = out.shape
    hp = lambda t: None if t is None else c_void_p(t.data_ptr())
    info = (c_int * 8)()
    if phases is not None:
        pn, poy, pox, dy, dx, T = phases
        nph = len(pn)
    else:
        pn = poy = pox = None
        dy, dx = taps
        T, nph = len(dy), 0
    rc = lib().jvae_conv_halo_emulate(hp(inp), N, H, W, Cin, ld_in, hp(wmat), Cout_pad, wmat.shape[1], nph, pn, poy, pox, T, dy, dx,
                                      in_stride, Hq, Wq, hp(out), Ho, Wo, Cout, ld_out, out_s[0], out_s[1], out_o[0], out_o[1],
                                      hp(bias), act, info)
    if rc == NOT_COVERED:
        return None
    check(rc)
    return list(info)


def conv_wgrad_emulate(dy, Cout, x, Cin, taps, in_stride, dw, dw_ld_tap, dw_ld_co, dw_ld_ci=1):
    """include/jvae_b200.h: jvae_conv_wgrad_emulate (HOST tensors, fp32; test aid).  dy (N,Hq,Wq,ld_dy), x (N,H,W,ld_x), dw fp32
    accumulated in place.  Returns the number of launches the plan stands for, or None when the tap-box kernel would run."""
    for t in (dy, x, dw):
        assert t.device.type == 'cpu' and t.dtype == torch.float32 and t.is_contiguous()
    N, Hq, Wq, ld_dy = dy.shape
    _, H, W, ld_x = x.shape
    n = c_int(0)
    rc = lib().jvae_conv_wgrad_emulate(c_void_p(dy.data_ptr()), N, Hq, Wq, Cout, ld_dy, c_void_p(x.data_ptr()), H, W, Cin, ld_x,
                                       len(taps[0]), taps[0], taps[1], in_stride, c_void_p(dw.data_ptr()), dw_ld_tap, dw_ld_co,
                                       dw_ld_ci, ctypes.byref(n))
    if rc == NOT_COVERED:
        return None
    check(rc)
    return n.value


def conv_wgrad(dy, N, Hq, Wq, Cout, ld_dy, x, H, W, Cin, ld_x, taps, in_stride, dw, dw_ld_tap, dw_ld_co, dw_ld_ci=1):
    with _timed_conv(2.0 * N * Hq * Wq * len(taps[0]) * Cin * Cout):
        check(lib().jvae_conv_wgrad(rawptr(dy), N, Hq, Wq, Cout, ld_dy, rawptr(x), H, W, Cin, ld_x, len(taps[0]), taps[0],
                                    taps[1], in_stride, rawptr(dw), dw_ld_tap, dw_ld_co, dw_ld_ci, stream()))


def bn_stats(y, P, C, ld, stats):
    check(lib().jvae_bn_stats(rawptr(y), P, C, ld, rawptr(stats), stream()))


def bn_apply_fwd(y, P, C, ld_y, stats, gamma, beta, eps, momentum, running_mean, running_var, num_batches, training, act,
                 out, ld_out, save):
    check(lib().jvae_bn_apply_fwd(rawptr(y), P, C, ld_y, rawptr(stats), rawptr(gamma), rawptr(beta), float(eps),
                                  float(momentum), rawptr(running_mean), rawptr(running_var), rawptr(num_batches),
                                  int(training), act, rawptr(out), ld_out, rawptr(save), stream()))


def bn_bwd(da, ld_da, y, ld_y, P, C, save, gamma, beta, act, sums, dy, ld_dy, dgamma, dbeta, skip_reduce=False):
    check(lib().jvae_bn_bwd(rawptr(da), ld_da, rawptr(y), ld_y, P, C, rawptr(save), rawptr(gamma), rawptr(beta), act,
                            rawptr(sums), rawptr(dy), ld_dy, rawptr(dgamma), rawptr(dbeta), int(skip_reduce), stream()))


def bn_stats_ld(y, P, C, ld, stats, stats_ld):
    """y: (N, H, W, >= C) view whose first channel is the slice's; stats: flat f64 view starting at the slice's channel"""
    check(lib().jvae_bn_stats_ld(rawptr(y), P, C, ld, rawptr(stats), stats_ld, stream()))


def bn_preact_fwd(y, P, C, ld_y, stats, stats_ld, gamma, beta, eps, momentum, running_mean, running_var, num_batches, training,
                  act, out, ld_out, save):
    check(lib().jvae_bn_preact_fwd(rawptr(y), P, C, ld_y, rawptr(stats), stats_ld, rawptr(gamma), rawptr(beta), float(eps),
                                   float(momentum), rawptr(running_mean), rawptr(running_var), rawptr(num_batches),
                                   int(training), act, rawptr(out), ld_out, rawptr(save), stream()))


def bn_preact_bwd(da, ld_da, y, ld_y, P, C, save, gamma, beta, running_mean, running_var, eps, training, act, sums, dx, ld_dx,
                  dgamma, dbeta):
    check(lib().jvae_bn_preact_bwd(rawptr(da), ld_da, rawptr(y), ld_y, P, C, rawptr(save), rawptr(gamma), rawptr(beta),
                                   rawptr(running_mean), rawptr(running_var), float(eps), int(training), act, rawptr(sums),
                                   rawptr(dx), ld_dx, rawptr(dgamma), rawptr(dbeta), stream()))


def cast_f32_bf16_ld(src, ld_src, dst, ld_dst, P, C):
    check(lib().jvae_cast_f32_bf16_ld(rawptr(src), ld_src, rawptr(dst), ld_dst, P, C, stream()))


def act_bwd(da, ld_da, a_out, ld_a, P, C, act, dy, ld_dy, dbias):
    check(lib().jvae_act_bwd(rawptr(da), ld_da, rawptr(a_out), ld_a, P, C, act, rawptr(dy), ld_dy, rawptr(dbias), stream()))


def maxpool_fwd(inp, N, H, W, C, ld_in, k, stride, out, ld_out):
    check(lib().jvae_maxpool_fwd(rawptr(inp), N, H, W, C, ld_in, k, stride, rawptr(out), ld_out, stream()))


def maxpool_bwd(inp, N, H, W, C, ld_in, k, stride, dout, ld_dout, din, ld_din):
    check(lib().jvae_maxpool_bwd(rawptr(inp), N, H, W, C, ld_in, k, stride, rawptr(dout), ld_dout, rawptr(din), ld_din,
                                 stream()))


def upsample2(src, ld_src, dst, ld_dst, N, H, W, C, backward=False):
    check(lib().jvae_upsample2(rawptr(src), ld_src, rawptr(dst), ld_dst, N, H, W, C, int(backward), stream()))


def maxpool_pad_fwd(inp, N, H, W, C, ld_in, k, stride, pad, out, ld_out):
    check(lib().jvae_maxpool_pad_fwd(rawptr(inp), N, H, W, C, ld_in, k, stride, pad, rawptr(out), ld_out, stream()))


def maxpool_pad_bwd(inp, N, H, W, C, ld_in, k, stride, pad, dout, ld_dout, din, ld_din):
    check(lib().jvae_maxpool_pad_bwd(rawptr(inp), N, H, W, C, ld_in, k, stride, pad, rawptr(dout), ld_dout, rawptr(din),
                                     ld_din, stream()))


def avgpool(src, ld_src, dst, ld_dst, N, H, W, C, k, backward=False):
    check(lib().jvae_avgpool(rawptr(src), ld_src, rawptr(dst), ld_dst, N, H, W, C, k, int(backward), stream()))


def vsum_rows(T, ld_t, N, H, W, k, pad, Co, bias, act, stats, out, ld_out):
    check(lib().jvae_vsum_rows(rawptr(T), ld_t, N, H, W, k, pad, Co, rawptr(bias), act, rawptr(stats), rawptr(out), ld_out,
                               stream()))


def vstack_rows(dy, ld_dy, N, H, W, k, pad, Co, U, ld_u):
    check(lib().jvae_vstack_rows(rawptr(dy), ld_dy, N, H, W, k, pad, Co, rawptr(U), ld_u, stream()))


def add_act(a, ld_a, b, ld_b, P, C, act, out, ld_out):
    check(lib().jvae_add_act(rawptr(a), ld_a, rawptr(b), ld_b, P, C, act, rawptr(out), ld_out, stream()))


def selftest(verbose=1):
    return int(lib().jvae_selftest(verbose))
