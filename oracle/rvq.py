"""CPU restatement of residual quantization (RQ-VAE).  TEST INFRASTRUCTURE ONLY.

NOT PINNED to the reference: the reference has no residual quantizer.  This file states the semantics that
`ResidualVectorQuantizer` documents (DESIGN.md §4.7) by composing the oracle's pinned single-level forward,
`oracle.quantizer_forward`, once per level on the residuals:

    r_0 = x;   level l = quantizer_forward(spec, [r_{l-1}], W_l, prob_l)   (its own encode / update / decode / losses)
    e_l = W_l'[q_l];  zhat_l = zhat_{l-1} + e_l;  r_l = r_{l-1} - sg(e_l)      (fp32, level order)
    z = x + sg(zhat_L - x);   losses[name] = sum_l loss_{l,name}  (level order);  loss = sum over names

Autograd on the result gives the reference gradients: each level's codebook leaf (`weight_leafs[l]`) and x, which
every level's commitment term reaches through r_{l-1} (dr/dx = I).
"""
from __future__ import annotations

from typing import Sequence

import torch

from . import oracle as O


def rvq_forward(spec: O.QuantizerSpec, x: torch.Tensor, weights: Sequence[torch.Tensor],
                probs: Sequence[torch.Tensor] | None = None) -> dict:
    """x [N, D] fp32 (may require grad); weights: the L codebooks [K, D]; probs: the L `_probability` buffers
    (CVQVAECallback).  Returns dict(quant int64 [N, L], zhat, z_ste, loss, losses, levels (per-level
    quantizer_forward outputs), r (r_0 .. r_{L-1}), weights (post-step), weight_leafs, probs (post-step))."""
    r = x
    zhat = None
    levels, residuals = [], []
    losses: dict = {}
    for l, W in enumerate(weights):
        out = O.quantizer_forward(spec, [r], W, None if probs is None else probs[l])
        e = out['z'][0].detach()
        zhat = e if zhat is None else zhat + e
        for name, value in out['losses'][0].items():
            losses[name] = value if l == 0 else losses[name] + value
        levels.append(out)
        residuals.append(r)
        r = r - e
    loss = x.new_zeros([])
    for i, value in enumerate(losses.values()):
        loss = value if i == 0 else loss + value
    return dict(quant=torch.stack([o['quant'][0] for o in levels], 1), zhat=zhat, z_ste=O.ste(zhat, x), loss=loss,
                losses=losses, levels=levels, r=residuals, weights=[o['weight'] for o in levels],
                weight_leafs=[o['weight_leaf'] for o in levels], probs=[o['prob'] for o in levels])


def level_sum(weights: Sequence[torch.Tensor], quant: torch.Tensor) -> torch.Tensor:
    """sum_l W_l[quant[..., l]] in level order (fp32 adds): the decode of residual ids [..., L]."""
    z = None
    for l, W in enumerate(weights):
        e = torch.nn.functional.embedding(quant[..., l], W)
        z = e if z is None else z + e
    return z
