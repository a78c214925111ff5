"""Optimizer wrapper with the reference's interface (module/optimizers.py:14-133): Adam (L2 weight decay in the
gradient, not AdamW; optionally AMSGrad) or SGD (momentum, dampening, Nesterov), global-norm clipping, exponential lr decay
per epoch.

Both run as native kernels over a flat fp32 parameter buffer (csrc/optim.cu): the trainable parameters are re-pointed to
views of that buffer, their .grad to views of a flat gradient buffer, so that the data-parallel all-reduce, the global norm
and the update each touch one contiguous array.  The clip coefficient and the per-parameter step counts live on the device,
so a step replays from a CUDA graph.  As with torch.optim, a parameter without a gradient is skipped (no update, no step
count, no state); here that is a parameter whose slice of the zeroed flat gradient stayed all zero, for SGD as for Adam.
state_dict() / load_state_dict() use torch.optim.Adam's and torch.optim.SGD's layouts.
"""
import logging

import torch

from .. import _native as nat
from .. import engine

default_lr = {'sgd': 0.01, 'adam': 0.001}
params_by_type = {'sgd': ('momentum', 'nesterov', 'weight_decay'), 'adam': ('betas', 'weight_decay', 'amsgrad')}
# keyword arguments of torch.optim.SGD / Adam that only choose torch's implementation: accepted and ignored
_IMPL_KW = ('foreach', 'fused', 'capturable', 'differentiable')


class Optimizer:

    def __init__(self, parameters, optim_type='adam', lr=0, lr_decay=0, weight_decay=0, grad_clipping=None, epoch=0,
                 **kw):
        self.kind = optim_type
        lr = lr or default_lr[optim_type]
        self.params = {'optim_type': optim_type, 'lr': lr, 'lr_decay': lr_decay, 'weight_decay': weight_decay,
                       'grad_clipping': grad_clipping}
        self.params.update(kw)
        self.grad_clipping = grad_clipping
        self.init_lr = lr
        self.lr_decay = lr_decay
        self.weight_decay = weight_decay
        self._params = list(parameters)
        self._lr = lr
        self._clip_now = False
        self.grad_dtype = torch.float32      # torch.bfloat16: the DP bucket is reduced and consumed in bf16
        self.allreduce = None                # set by distributed.DataParallel: callable(flat_grad) -> flat_grad
        if kw.get('maximize'):
            raise NotImplementedError('maximize is not implemented by the fused optimizer kernels')
        if optim_type == 'adam':
            self.betas = tuple(kw.get('betas', (0.9, 0.999)))
            self.eps = kw.get('eps', 1e-8)
            self.amsgrad = bool(kw.get('amsgrad', False))
            # flat state buffer -> torch.optim.Adam's state key
            self._state_keys = {'m': 'exp_avg', 'v': 'exp_avg_sq'}
            if self.amsgrad:
                self._state_keys['vmax'] = 'max_exp_avg_sq'
        elif optim_type == 'sgd':
            unknown = set(kw) - {'momentum', 'dampening', 'nesterov', 'maximize'} - set(_IMPL_KW)
            if unknown:
                raise TypeError(f'unexpected SGD arguments: {sorted(unknown)}')
            self.momentum = kw.get('momentum', 0)
            self.dampening = kw.get('dampening', 0)
            self.nesterov = bool(kw.get('nesterov', False))
            if lr < 0:
                raise ValueError(f'Invalid learning rate: {lr}')
            if self.momentum < 0:
                raise ValueError(f'Invalid momentum value: {self.momentum}')
            if weight_decay < 0:
                raise ValueError(f'Invalid weight_decay value: {weight_decay}')
            if self.nesterov and (self.momentum <= 0 or self.dampening != 0):
                raise ValueError('Nesterov momentum requires a momentum and zero dampening')
            self._state_keys = {'buf': 'momentum_buffer'} if self.momentum != 0 else {}
        else:
            raise ValueError(optim_type)
        self._opt = None                      # no library optimizer: cvae._graph_ok relies on it
        self._flat = None
        self._pending_state = {}              # id(param) -> loaded torch.optim state waiting for the flat buffers

    # ------------------------------------------------------------------ flat buffers
    def _trainable(self):
        return [p for p in self._params if p.requires_grad]

    def _flatten(self):
        """Re-point the trainable parameters (and their .grad) to slices of flat buffers; every slice starts on a multiple of
        JVAE_OPT_CHUNK elements so that a chunk belongs to one parameter (include/jvae_b200.h: chunk_seg).  Only the state
        the configuration updates is allocated (Adam: m, v and, with amsgrad, vmax; SGD: the momentum buffer iff
        momentum != 0); it and the step counts carry over from the previous flat buffers or from load_state_dict."""
        ps = self._trainable()
        if not ps:
            raise RuntimeError('no trainable parameter')
        dev = ps[0].device
        if dev.type != 'cuda':
            raise nat.NativeError('the fused optimizer kernels need the parameters on a CUDA device (no CPU fallback)')
        old = self._flat
        CH = nat.OPT_CHUNK
        sizes = [(p.numel() + CH - 1) // CH * CH for p in ps]
        n, nseg = sum(sizes), len(ps)
        aux = torch.zeros(1 + nseg, device=dev)                  # [norm2 | seg_active (int32 view)]: one zero_() per step
        f = {'ids': [id(p) for p in ps], 'n': n, 'p': torch.zeros(n, device=dev), 'g': torch.zeros(n, device=dev),
             'aux': aux, 'norm2': aux[:1], 'seg_active': aux[1:].view(torch.int32),
             'seg_step': torch.zeros(nseg, dtype=torch.int32, device=dev), 'seg_bc': torch.zeros(2 * nseg, device=dev),
             'views': {}, 'seg': {}}
        for k in self._state_keys:
            f[k] = torch.zeros(n, device=dev)
        f['chunk_seg'] = torch.repeat_interleave(torch.arange(nseg, dtype=torch.int32),
                                                 torch.tensor([sz // CH for sz in sizes])).to(dev)
        off = 0
        steps = [0] * nseg
        for i, (p, sz) in enumerate(zip(ps, sizes)):
            sl = slice(off, off + p.numel())
            f['p'][sl].copy_(p.data.reshape(-1))
            if id(p) in self._pending_state:                      # torch.optim state from load_state_dict
                st = self._pending_state.pop(id(p))
                loaded = [k for k, tk in self._state_keys.items() if st.get(tk) is not None]
                for k in loaded:
                    f[k][sl].copy_(st[self._state_keys[k]].reshape(-1))
                # torch.optim.SGD keeps no step count: a parameter with a momentum buffer has been updated before
                steps[i] = int(st['step']) if 'step' in st else int(bool(loaded))
            elif old is not None and id(p) in old['views']:
                osl = old['views'][id(p)]
                for k in self._state_keys:
                    if k in old:
                        f[k][sl].copy_(old[k][osl])
                steps[i] = int(old['seg_step'][old['seg'][id(p)]])
            if p.grad is not None:
                f['g'][sl].copy_(p.grad.reshape(-1))
            p.data = f['p'][sl].view(p.shape)
            p.grad = f['g'][sl].view(p.shape)
            f['views'][id(p)] = sl
            f['seg'][id(p)] = i
            off += sz
        f['seg_step'].copy_(torch.tensor(steps, dtype=torch.int32))
        self._flat = f
        engine.bump_params()

    def _ensure_flat(self):
        ps = self._trainable()
        f = self._flat
        if f is None or f['ids'] != [id(p) for p in ps] or f['p'].device != ps[0].device or \
                any(p.data.data_ptr() != f['p'][f['views'][id(p)]].data_ptr() for p in ps[:1]):
            self._flatten()
        else:
            for p in ps:        # autograd may have replaced .grad by a fresh tensor
                sl = f['views'][id(p)]
                if p.grad is None:
                    p.grad = f['g'][sl].view(p.shape)
                elif p.grad.data_ptr() != f['g'][sl].data_ptr():
                    f['g'][sl].copy_(p.grad.reshape(-1))
                    p.grad = f['g'][sl].view(p.shape)

    @property
    def flat_grad(self):
        self._ensure_flat()
        return self._flat['g']

    # ------------------------------------------------------------------ reference interface
    @property
    def lr(self):
        return self._lr

    def zero_grad(self, *a, **kw):
        if self._trainable() and self._trainable()[0].is_cuda:
            self._ensure_flat()
            self._flat['g'].zero_()
        else:
            for p in self._params:
                p.grad = None

    def clip(self, parameters=None):
        """module/optimizers.py:79-81.  The norm and the clip coefficient are computed inside step() on the device; this
        call only arms them."""
        if self.grad_clipping:
            self._clip_now = True

    def step(self):
        self._ensure_flat()
        f = self._flat
        g = f['g']
        if self.grad_dtype == torch.bfloat16:
            g = nat.cast_f32_bf16(g, f.setdefault('g16', torch.empty(f['n'], dtype=torch.bfloat16, device=g.device)))
        if self.allreduce is not None:
            g = self.allreduce(g)
        max_norm = self.grad_clipping if self._clip_now else 0.0
        f['aux'].zero_()
        # one pass over the gradient: squared norm for the clip AND the per-parameter "has a gradient" flags
        nat.grad_sqnorm(g, f['norm2'], f['chunk_seg'], f['seg_active'])
        table = dict(max_norm=max_norm, lr=self._lr, weight_decay=self.weight_decay, chunk_seg=f['chunk_seg'],
                     seg_active=f['seg_active'], seg_step=f['seg_step'])
        if self.kind == 'sgd':
            nat.sgd_step(f['p'], f.get('buf'), g, f['norm2'], momentum=self.momentum, dampening=self.dampening,
                         nesterov=self.nesterov, **table)
        elif self.amsgrad:
            nat.adam_amsgrad_step(f['p'], f['m'], f['v'], f['vmax'], g, f['norm2'], beta1=self.betas[0], beta2=self.betas[1],
                                  eps=self.eps, seg_bc=f['seg_bc'], **table)
        else:
            nat.adam_step(f['p'], f['m'], f['v'], g, f['norm2'], beta1=self.betas[0], beta2=self.betas[1], eps=self.eps,
                          seg_bc=f['seg_bc'], **table)
        self._clip_now = False
        engine.bump_params()         # parameters changed in place behind autograd's version counters

    def update_lr(self):
        if self.lr_decay:
            self._lr *= 1 - self.lr_decay

    def update_scheduler_from_epoch(self, n):
        for _ in range(n):
            self.update_lr()

    def to(self, device):
        """the flat buffers follow the parameters lazily (see _ensure_flat)"""

    def state_dict(self, *a, **k):
        """torch.optim.Adam's / torch.optim.SGD's layout: `state` indexed by the position of the parameter in the FULL
        parameter list the optimizer was given (frozen ones included, as torch does), for every parameter that was ever
        updated: Adam {step, exp_avg, exp_avg_sq[, max_exp_avg_sq]}, SGD {momentum_buffer} (no state without momentum)."""
        state = {}
        if self._flat is not None:
            f = self._flat
            steps = f['seg_step'].tolist()
            for i, p in enumerate(self._params):
                if id(p) not in f['views'] or steps[f['seg'][id(p)]] == 0:
                    continue
                sl = f['views'][id(p)]
                st = {'step': torch.tensor(float(steps[f['seg'][id(p)]]))} if self.kind == 'adam' else {}
                st.update({tk: f[k][sl].view(p.shape).clone() for k, tk in self._state_keys.items()})
                if st:
                    state[i] = st
        if self.kind == 'sgd':
            group = {'lr': self._lr, 'momentum': self.momentum, 'dampening': self.dampening, 'weight_decay': self.weight_decay,
                     'nesterov': self.nesterov, 'maximize': False, 'foreach': None, 'differentiable': False, 'fused': None}
        else:
            group = {'lr': self._lr, 'betas': self.betas, 'eps': self.eps, 'weight_decay': self.weight_decay,
                     'amsgrad': self.amsgrad}
        group['params'] = list(range(len(self._params)))
        return {'state': state, 'param_groups': [group]}

    def load_state_dict(self, sd, *a, **k):
        self._lr = sd['param_groups'][0]['lr']
        self._pending_state = {id(self._params[int(i)]): st for i, st in sd['state'].items() if int(i) < len(self._params)}
        if self._pending_state and self._trainable() and self._trainable()[0].is_cuda:
            self._flatten()            # the loaded state and step counts enter the flat buffers

    def __str__(self):
        return self.__format__('10')

    def __format__(self, format_spec):
        try:
            level = int(format_spec.rstrip('x'))
        except ValueError:
            level = 0
        if not level:
            level = 10
        s = [self.kind, f'lr={self.init_lr}']
        if self.lr_decay:
            s.append(f'decay={self.lr_decay}')
        else:
            level -= 1
        if self.weight_decay:
            s.append(f'weight_decay={self.weight_decay}')
        return '--'.join(s[:level])
