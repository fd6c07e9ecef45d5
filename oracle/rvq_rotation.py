"""CPU restatement of the rotation trick on a residual quantizer.  TEST INFRASTRUCTURE ONLY.

NOT PINNED to the reference: the reference has neither a residual quantizer nor the rotation trick.  This file states
the contract of `ResidualVectorQuantizer(rotation_trick=True)` (DESIGN.md §4.7, §4.9) by composing the two existing
restatements, `oracle.rvq.rvq_forward` and `oracle.rotation.rotated_z`.  The stack has ONE straight-through estimator,
z = x + sg(zhat_L - x), and the rotation trick replaces exactly that one, with the whole depth as the map x -> zhat_L:

    out = rvq_forward(spec, x, weights, probs)
    z_ste = rotated_z(z_ste, x, zhat_L)          (value unchanged: x + (zhat_L - x))

so the gradient reaching x is rotate_grad(x, zhat_L, g) plus every level's commitment terms through r_{l-1}, and
nothing else (values, indices, losses, codebook updates and codebook gradients) changes.  With L = 1 this is
`oracle.rotation.rotated_forward` on the one level.
"""
from __future__ import annotations

from typing import Sequence

import torch

from . import oracle as O
from . import rotation as R
from . import rvq


def rotated_rvq_forward(spec: O.QuantizerSpec, x: torch.Tensor, weights: Sequence[torch.Tensor],
                        probs: Sequence[torch.Tensor] | None = None) -> dict:
    """`oracle.rvq.rvq_forward` with the rotation trick over the whole depth: out['z_ste'] keeps its value and carries
    the rotated gradient of x towards zhat_L (out['zhat'])."""
    out = rvq.rvq_forward(spec, x, weights, probs)
    out['z_ste'] = R.rotated_z(out['z_ste'], x, out['zhat'].detach())
    return out
