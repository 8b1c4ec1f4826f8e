"""``Ranger``: the reference's Ranger optimizer (``deepsignal_plant/utils/ranger2020.py``: RAdam + Lookahead + Gradient
Centralization, lessw2020's Ranger2020) with its step fused into one CUDA kernel per parameter group
(``dsp_ranger_step``, ``csrc/optim.cu``).

The published step is a Python loop of about 15 torch ops per tensor.  Here the host keeps what the published code
computes in Python -- each tensor's step count, ``N_sma`` and ``step_size`` (``rectification``, with the published
RAdam buffer), the Lookahead schedule -- and hands the kernel one float and three flags per tensor; the kernel does
the tensor arithmetic of every tensor of the group in one launch.  Row means for the gradient centralisation are summed
in a fixed order, so a step is a pure function of its inputs: repeating it gives the same bits, and ranks that hold
the same gradients (``train_dist.py``) keep identical parameters.

State: ``state[p]`` has the published keys ``step`` (int), ``exp_avg``, ``exp_avg_sq`` and ``slow_buffer``.  The three
tensors are views into one float32 arena per parameter group, so ``state_dict()`` / ``load_state_dict()`` work through
torch's usual machinery; after a load the next step copies the loaded state into a fresh arena.

Parameters must be contiguous float32 CUDA tensors, one device per group; there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
from torch.optim.optimizer import Optimizer

from . import _native

RECTIFY, LOOKAHEAD, CENTRALIZE = 1, 2, 4          # DSP_RANGER_* (include/dsp_b200.h)


def rectification(step, betas, N_sma_threshhold=5):
    """``(N_sma, step_size)`` of RAdam at ``step`` (counted from 1), in float64 as the published step computes them:
    un-rectified (``N_sma <= N_sma_threshhold``) the step size is ``1 / (1 - beta1^t)``."""
    beta1, beta2 = betas
    beta2_t = beta2 ** step
    N_sma_max = 2 / (1 - beta2) - 1
    N_sma = N_sma_max - 2 * step * beta2_t / (1 - beta2_t)
    if N_sma > N_sma_threshhold:
        step_size = math.sqrt((1 - beta2_t) * (N_sma - 4) / (N_sma_max - 4) * (N_sma - 2) / N_sma * N_sma_max
                              / (N_sma_max - 2)) / (1 - beta1 ** step)
    else:
        step_size = 1.0 / (1 - beta1 ** step)
    return N_sma, step_size


class Ranger(Optimizer):
    """Ranger2020 with the published constructor: RAdam (``betas``, ``eps``, ``weight_decay``, rectified once
    ``N_sma > N_sma_threshhold``), Lookahead (every ``k`` steps ``slow += alpha * (p - slow)``, ``p = slow``) and
    gradient centralisation (``use_gc``; ``gc_conv_only`` limits it to tensors of more than three dimensions;
    ``gc_loc=True`` centralises ``p.grad`` in place, ``False`` the update direction instead).  Per-group ``lr``,
    ``betas``, ``eps``, ``weight_decay`` and ``k`` are honoured, so learning-rate schedulers work."""

    def __init__(self, params, lr=1e-3, alpha=0.5, k=6, N_sma_threshhold=5, betas=(.95, 0.999), eps=1e-5,
                 weight_decay=0, use_gc=True, gc_conv_only=False, gc_loc=True):
        if not 0.0 <= alpha <= 1.0:
            raise ValueError(f'Invalid slow update rate: {alpha}')
        if not 1 <= k:
            raise ValueError(f'Invalid lookahead steps: {k}')
        if not lr > 0:
            raise ValueError(f'Invalid Learning Rate: {lr}')
        if not eps > 0:
            raise ValueError(f'Invalid eps: {eps}')
        defaults = dict(lr=lr, alpha=alpha, k=k, step_counter=0, betas=betas, N_sma_threshhold=N_sma_threshhold,
                        eps=eps, weight_decay=weight_decay)
        super().__init__(params, defaults)
        # as published, these are the constructor's and not the group's
        self.N_sma_threshhold = N_sma_threshhold
        self.alpha = alpha
        self.k = k
        self.gc_loc = gc_loc
        self.use_gc = use_gc
        self.gc_conv_only = gc_conv_only
        # the published RAdam buffer: (step, N_sma, step_size) for step % 10, keyed on the step count alone
        self.radam_buffer = [[None, None, None] for _ in range(10)]
        self._arenas = {}                           # group index -> (ids of its params, arena (3, numel), offsets)

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._arenas = {}                           # the loaded tensors move into fresh arenas at the next step

    def _schedule(self, step, betas):
        buffered = self.radam_buffer[int(step % 10)]
        if step != buffered[0]:
            buffered[:] = [step, *rectification(step, betas, self.N_sma_threshhold)]
        return buffered[1], buffered[2]

    @staticmethod
    def _check(group):
        params = group['params']
        dev = params[0].device if params else None
        for p in params:
            if p.device.type != "cuda":
                raise RuntimeError("Ranger runs on the GPU only (a parameter is on %s); this library has no CPU path"
                                   % p.device)
            if p.device != dev:
                raise RuntimeError("Ranger needs every parameter of a group on one device (%s and %s)" % (dev, p.device))
            if p.dtype != torch.float32 or not p.is_contiguous():
                raise RuntimeError("Ranger needs contiguous float32 parameters (got %s, contiguous=%s)"
                                   % (p.dtype, p.is_contiguous()))
            g = p.grad
            if g is None:
                continue
            if g.is_sparse:
                raise RuntimeError('Ranger optimizer does not support sparse gradients')
            if g.dtype != torch.float32 or not g.is_contiguous() or g.device != dev or g.shape != p.shape:
                raise RuntimeError("Ranger needs contiguous float32 gradients of the parameters' shapes on %s" % dev)
        return dev

    def _arena(self, gi, group, dev):
        """The group's state arena: rows exp_avg, exp_avg_sq, slow_buffer over the group's parameters back to back.
        A new arena takes over whatever state the parameters already have (a load, or a changed group)."""
        params = group['params']
        ids = tuple(id(p) for p in params)
        a = self._arenas.get(gi)
        if a is not None and a[0] == ids:
            return a
        offs, o = [], 0
        for p in params:
            offs.append(o)
            o += p.numel()
        flat = torch.zeros(3, o, device=dev)
        for p, off in zip(params, offs):
            st = self.state.get(p)
            if not st:
                continue
            for row, key in enumerate(("exp_avg", "exp_avg_sq", "slow_buffer")):
                view = flat[row, off:off + p.numel()].view_as(p)
                view.copy_(st[key])
                st[key] = view
        a = (ids, flat, offs)
        self._arenas[gi] = a
        return a

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        devs = [self._check(group) for group in self.param_groups]       # every group before any state changes
        for gi, (group, dev) in enumerate(zip(self.param_groups, devs)):
            live = [(i, p) for i, p in enumerate(group['params']) if p.grad is not None]
            if not live:
                continue
            _, flat, offs = self._arena(gi, group, dev)
            n = len(live)
            ptrs = [(C.c_void_p * n)() for _ in range(5)]
            numel, row_len = (C.c_int64 * n)(), (C.c_int64 * n)()
            scale, flags = (C.c_float * n)(), (C.c_int32 * n)()
            for j, (i, p) in enumerate(live):
                state = self.state[p]
                if len(state) == 0:
                    o, m = offs[i], p.numel()
                    state['step'] = 0
                    state['exp_avg'] = flat[0, o:o + m].view_as(p).zero_()
                    state['exp_avg_sq'] = flat[1, o:o + m].view_as(p).zero_()
                    state['slow_buffer'] = flat[2, o:o + m].view_as(p).copy_(p)
                state['step'] += 1
                t = state['step']
                N_sma, step_size = self._schedule(t, group['betas'])
                for arr, x in zip(ptrs, (p, p.grad, state['exp_avg'], state['exp_avg_sq'], state['slow_buffer'])):
                    arr[j] = x.data_ptr()
                numel[j] = p.numel()
                row_len[j] = p.numel() // p.shape[0] if p.dim() > 1 and p.numel() > 0 else max(p.numel(), 1)
                scale[j] = -step_size * group['lr']
                flags[j] = ((RECTIFY if N_sma > self.N_sma_threshhold else 0)
                            | (LOOKAHEAD if t % group['k'] == 0 else 0)
                            | (CENTRALIZE if self.use_gc and p.dim() > (3 if self.gc_conv_only else 1) else 0))
            beta1, beta2 = group['betas']
            with torch.cuda.device(dev):
                stream = torch.cuda.current_stream(dev).cuda_stream
                _native.check(_native.lib().dsp_ranger_step(n, *ptrs, numel, row_len, scale, flags, beta1, beta2, group['eps'],
                                                group['weight_decay'], self.alpha, int(bool(self.gc_loc)), stream),
                              "dsp_ranger_step")
        return loss
