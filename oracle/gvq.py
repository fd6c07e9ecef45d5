"""CPU restatement of grouped (product) quantization.  TEST INFRASTRUCTURE ONLY.

NOT PINNED to the reference: the reference has no grouped quantizer.  This file states the semantics that
`GroupedVectorQuantizer` documents (DESIGN.md §4.8) by composing the oracle's pinned single-quantizer forward,
`oracle.quantizer_forward`, once per group on the column slices:

    x_g = x[:, g*Dg:(g+1)*Dg];   group g = quantizer_forward(spec, [x_g], W_g, prob_g)   (its own encode / update / losses)
    z = cat_g(z_ste_g);   losses[name] = (sum_g loss_{g,name}) / G  (fp32 adds in group order, one division);
    loss = sum over names

Autograd on the result gives the reference gradients: each group's codebook leaf (`weight_leafs[g]`) and x, whose
column slice g receives group g's straight-through and commitment gradients.
"""
from __future__ import annotations

from typing import Sequence

import torch

from . import oracle as O


def gvq_forward(spec: O.QuantizerSpec, x: torch.Tensor, weights: Sequence[torch.Tensor],
                probs: Sequence[torch.Tensor] | None = None) -> dict:
    """x [N, G*Dg] fp32 (may require grad); weights: the G codebooks [K, Dg]; probs: the G `_probability` buffers
    (CVQVAECallback).  Returns dict(quant int64 [N, G], z_ste [N, G*Dg], loss, losses, groups (per-group
    quantizer_forward outputs), weights (post-step), weight_leafs, probs (post-step))."""
    G = len(weights)
    Dg = x.shape[1] // G
    groups = []
    sums: dict = {}
    for g, W in enumerate(weights):
        out = O.quantizer_forward(spec, [x[:, g * Dg:(g + 1) * Dg]], W, None if probs is None else probs[g])
        for name, value in out['losses'][0].items():
            sums[name] = value if g == 0 else sums[name] + value
        groups.append(out)
    losses = {name: total / G for name, total in sums.items()}
    loss = x.new_zeros([])
    for i, value in enumerate(losses.values()):
        loss = value if i == 0 else loss + value
    return dict(quant=torch.stack([o['quant'][0] for o in groups], 1),
                z_ste=torch.cat([o['z_ste'][0] for o in groups], 1), loss=loss, losses=losses, groups=groups,
                weights=[o['weight'] for o in groups], weight_leafs=[o['weight_leaf'] for o in groups],
                probs=[o['prob'] for o in groups])


def group_concat(weights: Sequence[torch.Tensor], quant: torch.Tensor) -> torch.Tensor:
    """cat_g W_g[quant[..., g]]: the decode of grouped ids [..., G]."""
    return torch.cat([torch.nn.functional.embedding(quant[..., g], W) for g, W in enumerate(weights)], -1)
