"""CPU restatement of the rotation trick.  TEST INFRASTRUCTURE ONLY.

NOT PINNED to the reference: the reference has no rotation trick.  This file states the contract that
`VectorQuantizer(rotation_trick=True)` and `GroupedVectorQuantizer` document (DESIGN.md §4.9), after Fifty et al.,
"Restructuring Vector Quantization with the Rotation Trick" (arXiv:2410.06424).  Per token, with y the quantizer's
view of it (F.normalize(x) under NormalizeCallback / VQKDCallback, else x) and e = W[q]:

    a = |y|, b = |e|;  a < 1e-12 or b < 1e-12: straight-through (g' = g)
    else u = y / a, ê = e / b, s = u + ê, w = s / max(|s|, 1e-12), λ = b / a
         forward value λ R y with R = I - 2 w wᵀ + 2 ê uᵀ  (= e analytically), λ, w, u, ê constants
         g' = λ Rᵀ g = λ (g - 2 w (w·g) + 2 u (ê·g))

`rotate_to` is the detach-based autograd form, `rotate_grad` the closed form of its backward, and `rotated_forward`
composes them with the pinned single-quantizer forward, `oracle.quantizer_forward`: the value of z stays the
straight-through value x + (e - x) (as in the module), its gradient to x is the rotated one.
"""
from __future__ import annotations

from typing import Sequence

import torch

from . import oracle as O

EPS = 1e-12


def _frame(y: torch.Tensor, e: torch.Tensor):
    """Per row: (fallback mask [N, 1], u, ê, w, λ), all detached."""
    y, e = y.detach(), e.detach()
    a = y.norm(dim=-1, keepdim=True)
    b = e.norm(dim=-1, keepdim=True)
    fallback = (a < EPS) | (b < EPS)
    a1, b1 = torch.where(fallback, torch.ones_like(a), a), torch.where(fallback, torch.ones_like(b), b)
    u, eh = y / a1, e / b1
    s = u + eh
    w = s / s.norm(dim=-1, keepdim=True).clamp_min(EPS)
    return fallback, u, eh, w, b1 / a1


def rotate_to(y: torch.Tensor, e: torch.Tensor) -> torch.Tensor:
    """λ R y with λ, R built from detached y and e: value e (up to rounding), gradient to y = λ Rᵀ g.  Rows with
    |y| or |e| below 1e-12 are straight-through: value y + (e - y), gradient g."""
    fallback, u, eh, w, lam = _frame(y, e)
    dot = lambda p, q: (p * q).sum(-1, keepdim=True)  # noqa: E731
    rot = lam * (y - 2 * dot(y, w) * w + 2 * dot(y, u) * eh)
    ste = y + (e - y).detach()
    return torch.where(fallback, ste, rot)


def rotate_grad(y: torch.Tensor, e: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
    """The closed form g' = λ (g - 2 w (w·g) + 2 u (ê·g)) of rotate_to's backward; g where the row falls back."""
    fallback, u, eh, w, lam = _frame(y, e)
    dot = lambda p, q: (p * q).sum(-1, keepdim=True)  # noqa: E731
    rot = lam * (g - 2 * w * dot(w, g) + 2 * u * dot(eh, g))
    return torch.where(fallback, g, rot)


def rotated_z(z_ste: torch.Tensor, y: torch.Tensor, e: torch.Tensor) -> torch.Tensor:
    """The straight-through value z_ste with rotate_to's gradient to y."""
    r = rotate_to(y, e)
    return r + (z_ste - r).detach()


def rotated_forward(spec: O.QuantizerSpec, xs_in: Sequence[torch.Tensor], weight: torch.Tensor,
                    prob: torch.Tensor | None = None) -> dict:
    """`oracle.quantizer_forward` with the rotation trick: out['z_ste'][r] keeps its value and carries the rotated
    gradient of rank r's tokens (out['x'][r], the quantizer's view y) towards e = W_used[q]."""
    out = O.quantizer_forward(spec, xs_in, weight, prob)
    out['z_ste'] = [rotated_z(zs, y, z.detach()) for zs, y, z in zip(out['z_ste'], out['x'], out['z'])]
    return out
