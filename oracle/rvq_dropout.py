"""CPU restatement of quantizer dropout on a residual quantizer.  TEST INFRASTRUCTURE ONLY.

NOT PINNED to the reference: the reference has neither a residual quantizer nor quantizer dropout.  This file states
the contract of `ResidualVectorQuantizer(quantizer_dropout=p)` (DESIGN.md §4.10) for given per-token depths d_n in
[1, L], by composing the oracle's pinned single-level forward, `oracle.quantizer_forward`, once per level on ALL
tokens (assignment, callbacks and codebook updates do not look at the depths):

    r_0 = x;   level l = quantizer_forward(spec, [r_{l-1}], W_l, prob_l);   e_l = W_l'[q_l];   r_l = r_{l-1} - sg(e_l)
    zhat_n = sum_{l < d_n} e_l                  (fp32 adds in level order; only the active levels)
    z = x + sg(zhat - x), or the rotation x -> zhat with rotation=True (`oracle.rotation.rotated_z`)
    loss_{l,name} = the level's loss on the active tokens m_l = (l < d_n) only: every squared term times m_l, still
                    divided by N * D (mean over all elements of the masked rows)

Autograd on the result gives the contract's gradients: gx = g' + sum over active levels of the commitment terms,
gW_l only from the active tokens.  With every depth L the masks are all ones, the masked operands equal the unmasked
ones bit for bit, and the result is `oracle.rvq.rvq_forward` (or `oracle.rvq_rotation.rotated_rvq_forward`) exactly.
"""
from __future__ import annotations

from typing import Sequence

import torch
import torch.nn.functional as F

from . import oracle as O
from . import rotation as R


def _masked_mse(pred: torch.Tensor, target: torch.Tensor, m: torch.Tensor, norm: bool) -> torch.Tensor:
    """MSE over all N * D elements of the rows kept by m ([N, 1] of 0 / 1), after F.normalize with norm."""
    if norm:
        pred, target = F.normalize(pred), F.normalize(target)
    return F.mse_loss(pred * m, target * m)


def masked_losses(spec: O.QuantizerSpec, z: torch.Tensor, x: torch.Tensor, m: torch.Tensor) -> dict:
    """`oracle._losses` with every term restricted to the rows m."""
    out = {}
    for name, cfg in spec.losses.items():
        t, norm = cfg['type'], cfg.get('norm', False)
        codebook = lambda: _masked_mse(z, x.detach(), m, norm)      # noqa: E731
        commitment = lambda: _masked_mse(z.detach(), x, m, norm)    # noqa: E731
        if t == 'CodebookLoss':
            out[name] = codebook()
        elif t == 'CommitmentLoss':
            out[name] = commitment()
        elif t == 'VQGANLoss':
            out[name] = codebook() + cfg.get('beta', 0.25) * commitment()
        else:
            raise ValueError(t)
    return out


def rvq_dropout_forward(spec: O.QuantizerSpec, x: torch.Tensor, weights: Sequence[torch.Tensor],
                        depth: torch.Tensor, probs: Sequence[torch.Tensor] | None = None,
                        rotation: bool = False) -> dict:
    """x [N, D] fp32 (may require grad); weights: the L codebooks [K, D]; depth: int [N] per-token depths in [1, L];
    probs: the L `_probability` buffers (CVQVAECallback).  Returns the keys of `oracle.rvq.rvq_forward`: quant int64
    [N, L], zhat (the truncated sums), z_ste, loss, losses, levels, r, weights (post-step), weight_leafs, probs."""
    depth = depth.reshape(-1, 1).to(torch.int64)
    r = x
    zhat = None
    levels, residuals = [], []
    losses: dict = {}
    for l, W in enumerate(weights):
        out = O.quantizer_forward(spec, [r], W, None if probs is None else probs[l])
        m = (depth > l).to(x.dtype)
        e = out['z'][0]
        ed = e.detach()
        zhat = ed if zhat is None else torch.where(depth > l, zhat + ed, zhat)
        for name, value in masked_losses(spec, e, out['x'][0], m).items():
            losses[name] = value if l == 0 else losses[name] + value
        levels.append(out)
        residuals.append(r)
        r = r - ed
    loss = x.new_zeros([])
    for i, value in enumerate(losses.values()):
        loss = value if i == 0 else loss + value
    z_ste = O.ste(zhat, x)
    if rotation:
        z_ste = R.rotated_z(z_ste, x, zhat)
    return dict(quant=torch.stack([o['quant'][0] for o in levels], 1), zhat=zhat, z_ste=z_ste, loss=loss,
                losses=losses, levels=levels, r=residuals, weights=[o['weight'] for o in levels],
                weight_leafs=[o['weight_leaf'] for o in levels], probs=[o['prob'] for o in levels])
