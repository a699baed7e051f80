"""Fused optimiser step for the training loops (SURVEY.md §8(f) row 1).

The reference trains with `torch.optim.Adam` followed by `model.W.clamp_(min=0)` (utilities.py:621-623): one small kernel per
parameter per elementary operation.  `Adam` here is a drop-in `torch.optim.Optimizer` whose `step()` is ONE launch of
`gpz_adam_step_*` over every parameter that has a gradient, with the non-negativity clamp of the flagged tensors applied in
the same pass.  Same update rule and operation order as torch (no weight decay, no amsgrad); there is no CPU path.
"""
from __future__ import annotations

import ctypes

import torch

from . import _cabi


class Adam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, clamp_nonneg=()):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        self._clamp_ids = {id(p) for p in clamp_nonneg}

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:
            by_dtype = {}
            for p in group["params"]:
                if p.grad is None:
                    continue
                if not p.is_cuda:
                    raise _cabi.GpzError("gpzoo_b200.optim.Adam updates CUDA parameters only (no CPU path exists)")
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                st["step"] += 1
                g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
                if not p.is_contiguous():
                    raise _cabi.GpzError("gpzoo_b200.optim.Adam needs contiguous parameters")
                by_dtype.setdefault((p.dtype, st["step"]), []).append((p, g, st))
            for (dtype, step), items in by_dtype.items():
                n = len(items)
                P = (ctypes.c_void_p * n)(*[p.data_ptr() for p, _, _ in items])
                G = (ctypes.c_void_p * n)(*[g.data_ptr() for _, g, _ in items])
                M1 = (ctypes.c_void_p * n)(*[s["exp_avg"].data_ptr() for _, _, s in items])
                M2 = (ctypes.c_void_p * n)(*[s["exp_avg_sq"].data_ptr() for _, _, s in items])
                numel = (ctypes.c_int64 * n)(*[p.numel() for p, _, _ in items])
                clamp = (ctypes.c_int * n)(*[1 if id(p) in self._clamp_ids else 0 for p, _, _ in items])
                b1, b2 = group["betas"]
                _cabi.call("adam_step", dtype, n, P, G, M1, M2, numel, clamp, float(group["lr"]), float(b1), float(b2),
                           float(group["eps"]), step)
        return loss
