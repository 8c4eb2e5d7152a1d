"""Fused multi-tensor Adam on the CUDA kernels (SURVEY.md section 8f rank 1; reference train.py:83
``torch.optim.Adam(model.parameters(), lr=args.lr, betas=(0.9, args.beta2))``).

``FusedAdam`` is a ``torch.optim.Optimizer``: same constructor arguments, ``state_dict`` layout (``step``, ``exp_avg``,
``exp_avg_sq`` per parameter; ``weight_decay``, ``amsgrad`` and ``maximize`` per group, fixed at their defaults) and update rule
as ``torch.optim.Adam`` (no amsgrad, no weight decay), so a checkpoint of either loads into the other.  ``step()`` is ONE kernel
launch (``aero_adam_step``) per parameter group over a device table of {param, grad, exp_avg, exp_avg_sq} records instead of a
few hundred small ones; parameters whose step counts differ (one that had no gradient on an earlier step) get one launch per
distinct count, so each has its own bias correction as in ``torch.optim.Adam``.
``grad_scale`` multiplies every gradient inside the kernel (1/world_size after a sum all-reduce of a flat gradient buffer)."""
from __future__ import annotations

import ctypes as C
import struct

import torch

from . import cabi

_CHUNK = 1 << 16
# group options of torch.optim.Adam that its step() reads and this kernel does not implement: only their defaults are accepted
_FIXED = dict(weight_decay=0, amsgrad=False, maximize=False)


def _check_group(group):
    for k, v in _FIXED.items():
        if group.get(k, v) != v:
            raise ValueError(f"FusedAdam: {k}={group[k]!r} is not supported (only {v!r})")


class FusedAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False, maximize=False):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad, maximize=maximize))
        for group in self.param_groups:
            _check_group(group)
        # device chunk tables, keyed by the {param, grad, exp_avg, exp_avg_sq} pointers they hold: a re-allocated .grad or
        # moment (zero_grad(set_to_none=True), load_state_dict) gets a new table instead of writing through stale pointers
        self._tables = {}

    def _table(self, ps, tables):
        """Device chunk table over the parameters `ps` (state initialised, same step count); (table, n_chunks)."""
        sts = [self.state[p] for p in ps]
        key = tuple((p.data_ptr(), p.grad.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), p.numel())
                    for p, st in zip(ps, sts))
        hit = self._tables.get(key)
        if hit is None:
            recs = bytearray()
            n = 0
            for p, st in zip(ps, sts):
                for off in range(0, p.numel(), _CHUNK):
                    recs += struct.pack("<QQQQq", p.data_ptr() + 4 * off, p.grad.data_ptr() + 4 * off,
                                        st["exp_avg"].data_ptr() + 4 * off, st["exp_avg_sq"].data_ptr() + 4 * off,
                                        min(_CHUNK, p.numel() - off))
                    n += 1
            hit = (torch.frombuffer(recs, dtype=torch.uint8).clone().to(ps[0].device), n)
        tables[key] = hit
        return hit

    @torch.no_grad()
    def step(self, closure=None, grad_scale=1.0):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = cabi.load()
        tables = {}
        for group in self.param_groups:
            _check_group(group)
            by_step = {}
            for p in group["params"]:
                if p.grad is None:
                    continue
                if p.dtype != torch.float32 or not p.is_cuda or not p.is_contiguous() or p.grad.dtype != torch.float32 or \
                        not p.grad.is_contiguous() or p.grad.device != p.device:
                    raise TypeError("FusedAdam: contiguous fp32 CUDA parameters / gradients only")
                st = self.state[p]
                if not st:
                    st["step"] = torch.zeros((), dtype=torch.float32)
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["step"] += 1
                if p.numel():
                    by_step.setdefault(int(st["step"]), []).append(p)
            b1, b2 = group["betas"]
            for step, ps in by_step.items():
                table, n = self._table(ps, tables)
                with torch.cuda.device(ps[0].device):
                    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                    cabi.check(lib.aero_adam_step(C.c_void_p(table.data_ptr()), n, float(group["lr"]), float(b1), float(b2),
                                                  float(group["eps"]), step, float(grad_scale), stream), lib)
                # the kernel wrote through raw pointers: bump the parameters' versions as an in-place torch update would, so
                # caches keyed on them (AeroEngine's packed weights and CUDA graphs) see the step
                torch.autograd.graph.increment_version(ps)
        self._tables = tables
        return loss
