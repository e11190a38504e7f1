"""PS-side optimizers that take *external* gradients.

API parity with the reference: ``SGDModified(params, lr, momentum, ...).step(grads, mode)`` and
``AdamModified(...).step(grads, mode)`` (src/optim/sgd_modified.py:5-88, src/optim/adam_modified.py:6-92), where ``grads``
is a list indexed like the parameters and ``mode`` names the aggregation that produced it (the reference only uses it
to decide whether to reshape).  Gradients may be torch tensors or numpy arrays.

These are the library-op optimizers used by the NCCL-baseline and CPU/Gloo transports; on the fused path the same SGD
arithmetic runs inside ``aggregate_update_kernel`` (csrc/cuda/aggregate_update.cu) -- ``tests/test_kernels_gpu.py``
checks the two against each other and against ``torch.optim.SGD``.
"""
from __future__ import annotations

import math
from typing import Iterable, List, Sequence

import numpy as np
import torch

_MODES = ("normal", "geometric_median", "maj_vote", "cyclic", "krum", "coord_median", "trimmed_mean", "multi_krum")


def _as_tensor(g, like: torch.Tensor) -> torch.Tensor:
    if isinstance(g, np.ndarray):
        g = torch.from_numpy(np.ascontiguousarray(g))
    return g.detach().to(device=like.device, dtype=like.dtype).reshape(like.shape)


class _External(torch.optim.Optimizer):
    def _check(self, grads: Sequence, mode: str) -> None:
        if mode not in _MODES:
            raise ValueError(f"unknown mode {mode!r}")
        n = sum(len(g["params"]) for g in self.param_groups)
        if len(grads) != n:
            raise ValueError(f"expected {n} gradients, got {len(grads)}")


class SGDModified(_External):
    """SGD with momentum / dampening / Nesterov / weight decay, torch.optim.SGD semantics."""

    def __init__(self, params: Iterable[torch.Tensor], lr: float = 0.01, momentum: float = 0.0, dampening: float = 0.0,
                 weight_decay: float = 0.0, nesterov: bool = False):
        if nesterov and (momentum <= 0 or dampening != 0):
            raise ValueError("Nesterov momentum requires a momentum and zero dampening")
        super().__init__(list(params), dict(lr=lr, momentum=momentum, dampening=dampening, weight_decay=weight_decay,
                                            nesterov=nesterov))

    @torch.no_grad()
    def step(self, grads: Sequence, mode: str = "normal", closure=None):
        loss = closure() if closure is not None else None
        self._check(grads, mode)
        i = 0
        for group in self.param_groups:
            wd, mu, damp, nest, lr = (group[k] for k in ("weight_decay", "momentum", "dampening", "nesterov", "lr"))
            for p in group["params"]:
                d_p = _as_tensor(grads[i], p)
                i += 1
                if wd != 0:
                    d_p = d_p.add(p, alpha=wd)
                if mu != 0:
                    st = self.state[p]
                    if "momentum_buffer" not in st:
                        buf = st["momentum_buffer"] = d_p.clone()
                    else:
                        buf = st["momentum_buffer"]
                        buf.mul_(mu).add_(d_p, alpha=1 - damp)
                    d_p = d_p.add(buf, alpha=mu) if nest else buf
                p.add_(d_p, alpha=-lr)
        return loss


class AdamModified(_External):
    """Adam / AMSGrad on external gradients (reference: src/optim/adam_modified.py:32-92)."""

    def __init__(self, params: Iterable[torch.Tensor], lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, amsgrad: bool = False):
        super().__init__(list(params), dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad))

    @torch.no_grad()
    def step(self, grads: Sequence, mode: str = "normal", closure=None):
        loss = closure() if closure is not None else None
        self._check(grads, mode)
        i = 0
        for group in self.param_groups:
            b1, b2 = group["betas"]
            for p in group["params"]:
                g = _as_tensor(grads[i], p)
                i += 1
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p)
                    st["exp_avg_sq"] = torch.zeros_like(p)
                    if group["amsgrad"]:
                        st["max_exp_avg_sq"] = torch.zeros_like(p)
                st["step"] += 1
                if group["weight_decay"] != 0:
                    g = g.add(p, alpha=group["weight_decay"])
                st["exp_avg"].mul_(b1).add_(g, alpha=1 - b1)
                st["exp_avg_sq"].mul_(b2).addcmul_(g, g, value=1 - b2)
                if group["amsgrad"]:
                    torch.maximum(st["max_exp_avg_sq"], st["exp_avg_sq"], out=st["max_exp_avg_sq"])
                    denom = st["max_exp_avg_sq"].sqrt().add_(group["eps"])
                else:
                    denom = st["exp_avg_sq"].sqrt().add_(group["eps"])
                bc1 = 1 - b1 ** st["step"]
                bc2 = 1 - b2 ** st["step"]
                p.addcdiv_(st["exp_avg"], denom, value=-group["lr"] * math.sqrt(bc2) / bc1)
        return loss


__all__ = ["SGDModified", "AdamModified"]
