"""The torch composition of one projected-gradient (PGD / FGSM) attack step.  TEST INFRASTRUCTURE ONLY.

csrc/ud_attack.cu mirrors these statements operation for operation in fp32 (the L-inf step bit for bit); the functions
are dtype-generic, so tests/test_attack_oracle.py checks their constraints in fp64.  eps and alpha are per-sample [N]
tensors, lo / hi the input range (the reference's Normalize(0.5, 0.5) maps images to [-1, 1]).
"""
from __future__ import annotations

from typing import Optional

import torch

Tensor = torch.Tensor


def _per_sample(v: Tensor, x: Tensor) -> Tensor:
    """[N] -> [N, 1, ...] broadcastable against x."""
    return v.reshape(-1, *([1] * (x.dim() - 1)))


def linf_step(x0: Tensor, x_adv: Tensor, g: Tensor, eps: Tensor, alpha: Tensor, lo: float, hi: float) -> Tensor:
    """x_adv = clamp(x0 + clamp((x_adv + alpha*sign(g)) - x0, -eps, eps), lo, hi)."""
    e, a = _per_sample(eps, x0), _per_sample(alpha, x0)
    d = (x_adv + a * torch.sign(g)) - x0
    d = torch.clamp(d, -e, e)
    return torch.clamp(x0 + d, lo, hi)


def l2_step(x0: Tensor, x_adv: Tensor, g: Tensor, eps: Tensor, alpha: Tensor, lo: float, hi: float) -> Tensor:
    """u = g / (||g_n|| + 1e-12); d = x_adv + alpha*u - x0; d *= min(1, eps/||d_n||) (0/0 -> 1);
    x_adv = clamp(x0 + d, lo, hi)."""
    gn = g.flatten(1).norm(dim=1)
    u = g / _per_sample(gn + 1e-12, g)
    d = x_adv + _per_sample(alpha, x0) * u - x0
    dn = d.flatten(1).norm(dim=1)
    f = torch.where(dn > eps, eps / dn, torch.ones_like(dn))
    return torch.clamp(x0 + d * _per_sample(f, d), lo, hi)


def select(loss: Tensor, best_loss: Tensor, x_adv: Tensor, x_best: Tensor):
    """Best-iterate tracking: samples whose loss strictly exceeds the best so far (a NaN loss never does) take x_adv.
    -> (best_loss, x_best, improved)."""
    imp = loss > best_loss
    return torch.where(imp, loss, best_loss), torch.where(_per_sample(imp, x_adv), x_adv, x_best), imp


def random_start_linf(x0: Tensor, eps: Tensor, lo: float, hi: float,
                      generator: Optional[torch.Generator] = None) -> Tensor:
    """Uniform in the L-inf ball: clamp(x0 + eps*U(-1, 1), lo, hi)."""
    r = torch.rand(x0.shape, generator=generator, dtype=x0.dtype, device=x0.device)
    return torch.clamp(x0 + (r * 2 - 1) * _per_sample(eps, x0), lo, hi)


def random_start_l2(x0: Tensor, eps: Tensor, lo: float, hi: float,
                    generator: Optional[torch.Generator] = None) -> Tensor:
    """A Gaussian direction scaled to radius eps*U(0, 1): clamp(x0 + z/||z_n|| * eps*r, lo, hi)."""
    z = torch.randn(x0.shape, generator=generator, dtype=x0.dtype, device=x0.device)
    r = torch.rand(x0.shape[0], generator=generator, dtype=x0.dtype, device=x0.device)
    z = z / _per_sample(z.flatten(1).norm(dim=1) + 1e-12, z)
    return torch.clamp(x0 + z * _per_sample(eps * r, x0), lo, hi)
