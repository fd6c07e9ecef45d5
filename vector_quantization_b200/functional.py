"""Autograd-level operators of the quantizer hot path.  Each forward/backward is one launch of a
hand-written kernel behind the C-ABI (`ops.py`); nothing here computes on the host or in eager PyTorch.

    l2_normalize         F.normalize(x)                         normalize.py:24
    nearest_code         distance + argmin (no N x K matrix)    vq/algorithms/vq/quantizers.py:92-100
    column_nearest       d.argmin(0)                            vq/algorithms/cvqvae/anchors.py:83
    quantize_ste_loss    embedding gather + STE + MSE losses    quantizers.py:102-117, losses.py:41-62
    fsq_quantize         FSQ bound/round/pack                   vq/algorithms/fsq/quantizers.py:108-126
(paths relative to the reference root)
"""
from __future__ import annotations

import torch

from . import ops

# How an fp32 operand is fed to the bf16/fp16 tensor cores:
#   'fp32'  (default) representation error below fp32 rounding noise: the fp16 (hi, lo * 2^11) pair (22 bits, two
#           MMA terms) for a normalised codebook against one-plane bf16 tokens, three exact bf16 planes otherwise
#   'exact' always three bf16 planes (v == hi + mid + lo bit for bit; every kept product is exact)
#   'high'  two bf16 planes (16 bits), 'fast' one bf16 plane (8 bits)
PRECISION_PLANES = {'fp32': 3, 'exact': 3, 'high': 2, 'fast': 1}
DEFAULT_PRECISION = 'fp32'

# Certified one-term pass (DESIGN.md §4.2).  From this padded depth on the assignment is bound by the tensor pipe, and
# the two MMA terms of an fp16-pair codebook are run as ONE term (hi plane) + a proof: rows whose best/runner-up margin
# exceeds twice the operand error bound keep their arg-max, the others are re-run with both terms.  Results are
# identical to the two-term contraction by construction.  VQB_CERTIFIED=0 disables it.
import os as _os
FOLD_L2 = _os.environ.get('VQB_FOLD_L2', '1') != '0'   # L2 side terms in the spare operand columns (needs Dp - D >= 6: D <= 10, 17..26, ...)
CERTIFIED_MIN_DP = 128 if _os.environ.get('VQB_CERTIFIED', '1') != '0' else 1 << 30


LAST_CERTIFY = {}   # debugging / tests / bench: the device-side count tensor of the most recent certified pass


def certified_assign(a: ops.Operand, b: ops.Operand, keys: torch.Tensor, *, scale_columns: bool = False,
                     index_offset: int = 0, a_inv_norm: torch.Tensor | None = None) -> torch.Tensor:
    """arg-max of <a_i, b_j> (times the column scale) with ONE MMA term where the fp16 pair would need two.
    Exactly one of (a, b) is an 'f16x2' pair carrying `lo_norm_max`; the other is a one-plane 'f16' operand.
      pair on the b side (row arg-min: tokens x codebook): scores are <x_i, hi_j>, the bound scales with |x_i|
        (`a_inv_norm` = 1/|x_i|);
      pair on the a side (column arg-min: codebook x tokens with the 1/|x_n| column scale): the bound is delta itself.
    keys must be reset (all-ones).  Same result as ops.assign(a, b, keys, l2=False, ...)."""
    pair_is_b = b.fmt == 'f16x2'
    pair = b if pair_is_b else a
    assert pair.fmt == 'f16x2' and pair.lo_norm_max is not None and (a if pair_is_b else b).fmt == 'f16'
    hi = ops.Operand(pair.planes, pair.rows, pair.dim, 1, None, plane_rows=pair.plane_rows, inv_norm=pair.inv_norm, fmt='f16')
    second = ops.new_keys(a.rows, keys.device)
    if pair_is_b:
        ops.assign(a, hi, keys, l2=False, index_offset=index_offset, scale_columns=scale_columns, second_keys=second)
    else:
        ops.assign(hi, b, keys, l2=False, index_offset=index_offset, scale_columns=scale_columns, second_keys=second)
    row_list, count, compact = ops.certify(keys, second, a.rows, pair.lo_norm_max,
                                           row_inv_norm=a_inv_norm if pair_is_b else None)
    LAST_CERTIFY.update(count=count, rows=a.rows)
    redo = ops.gather_operand_rows(a, row_list, count)            # the uncertified rows as a compact operand
    ops.assign(redo, b, compact, l2=False, index_offset=index_offset, scale_columns=scale_columns, a_rows_dev=count)
    return ops.scatter_keys(compact, row_list, count, keys)


class _L2Normalize(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return ops.l2norm_forward(x, torch.float32)

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        return ops.l2norm_backward(gy.contiguous().float(), x)


def l2_normalize(x: torch.Tensor) -> torch.Tensor:
    """Row-wise F.normalize (fp32 result, like `norm`/`div` under the reference's autocast policy)."""
    return _L2Normalize.apply(x.contiguous())


def _planes_for(t: torch.Tensor, normalized: bool, precision: str) -> int:
    if t.dtype == torch.bfloat16 and not normalized:
        return 1  # bf16 values are exact in one plane
    return PRECISION_PLANES[precision]


def _pair_ok(W: torch.Tensor, normalize: bool, precision: str, tokens: torch.Tensor | None) -> bool:
    """fp16-pair codebook planes: normalised fp32 rows, and the tokens are bf16 (used RAW under the cosine metric,
    the arg-min does not depend on the token norm; their 8 significant bits are exact in one fp16 plane)."""
    return (precision == 'fp32' and normalize and W.dtype == torch.float32 and tokens is not None
            and tokens.dtype == torch.bfloat16)


@torch.no_grad()
def pack_codebook(W: torch.Tensor, metric: str, *, precision: str = DEFAULT_PRECISION,
                  writeback_normalized: bool = False, reset_keys: torch.Tensor | None = None,
                  tokens: torch.Tensor | None = None, zero_fill: torch.Tensor | None = None) -> ops.Operand:
    """Codebook operand: cosine -> planes of F.normalize(W) (optionally written back to W in place, which is
    NormalizeCallback's `weight.data = normalize(weight)`, normalize.py:26-28); L2 -> planes of W and 0.5|e|^2.
    `tokens`: the token tensor this codebook will be matched against (selects the plane format)."""
    cos = metric == 'Cosine'
    normalize = cos or writeback_normalized
    pair = cos and _pair_ok(W, normalize, precision, tokens)
    # small-D L2 (LlamaGen's 16384 x 8): the -0.5|e|^2 term rides in the operand's spare columns (written by the pack
    # launch itself) and the kernel's epilogue is the plain arg-max of the cosine path (half the instructions per score)
    fold = 'codes' if (not cos and FOLD_L2 and ops.can_fold_l2(W.shape[1])) else None
    return ops.pack_rows(W, normalize=normalize, planes=None if pair else _planes_for(W, normalize, precision),
                         want_half_sqnorm=not cos, writeback=W if writeback_normalized else None,
                         reset_keys=reset_keys, fmt='f16x2' if pair else 'bf16', zero_fill=zero_fill,
                         want_lo_norm=pair and ops.operand_shape(1, W.shape[1])[1] >= CERTIFIED_MIN_DP, fold=fold)


@torch.no_grad()
def nearest_code(x: torch.Tensor, codebook: ops.Operand, metric: str, *, precision: str = DEFAULT_PRECISION,
                 keys: torch.Tensor | None = None, index_offset: int = 0, normalize_tokens: bool = False,
                 tokens: ops.Operand | None = None, keys_are_reset: bool = False) -> torch.Tensor:
    """Packed (score,index) keys [N] of the nearest code of every token (row arg-min of the distance).
    Cosine arg-min is invariant to the token norm, so raw tokens are used: zero-copy for bf16 tokens
    whose D needs no padding, one exact plane otherwise.  L2 on normalised tokens (LlamaGen) packs the
    normalised planes."""
    cos = metric == 'Cosine'
    if keys is None:
        keys = torch.empty((x.shape[0],), dtype=torch.int64, device=x.device)
        keys_are_reset = False
    if tokens is None:
        if codebook.fmt != 'bf16':
            # fp16-pair codebook (cosine, bf16 tokens): the raw tokens as one fp16 plane (no bf16/fp16 mixing on
            # the tensor core); two MMA terms instead of the three of an exact bf16-plane codebook
            if not (cos and x.dtype == torch.bfloat16):
                raise ValueError('a fp16-pair codebook needs bf16 tokens and the cosine metric: '
                                 'pack the codebook with pack_codebook(..., tokens=x)')
            # D in {16, 32, 64}: zero-copy, the kernel converts the resident token tile to fp16 in shared memory;
            # otherwise one fp16 plane is packed
            tokens = ops.as_operand(x) if x.shape[1] <= 64 else None
            if tokens is None:
                tokens = ops.pack_rows(x, fmt='f16', reset_keys=None if keys_are_reset else keys)
                keys_are_reset = True
        else:
            norm = normalize_tokens and not cos
            tokens = None if (norm or codebook.folded is not None) else ops.as_operand(x)
            if tokens is None:
                tokens = ops.pack_rows(x, normalize=norm, planes=_planes_for(x, norm, precision),
                                       reset_keys=None if keys_are_reset else keys,
                                       fold='tokens' if codebook.folded is not None else None)
                keys_are_reset = True
    if codebook.folded is not None and tokens.folded is None:
        ops.fold_l2_side(tokens, 'tokens')      # the 1-columns that pick up the codes' -0.5|e|^2
    if not keys_are_reset:
        keys.fill_(-1)
    if codebook.lo_norm_max is not None and tokens.fmt == 'f16':
        # D >= 128, fp16-pair codebook: one MMA term + certificate instead of two terms
        inv = tokens.inv_norm if tokens.inv_norm is not None else ops.row_inv_norm(x, f16_rows=True)
        tokens.inv_norm = inv
        return certified_assign(tokens, codebook, keys, index_offset=index_offset, a_inv_norm=inv)
    return ops.assign(tokens, codebook, keys, l2=not cos, index_offset=index_offset)


@torch.no_grad()
def column_nearest(x: torch.Tensor, codebook: ops.Operand, metric: str, *, precision: str = DEFAULT_PRECISION,
                   index_offset: int = 0, tokens: ops.Operand | None = None, rows=None) -> torch.Tensor:
    """Packed keys [K]: for every code, the nearest token (column arg-min) — the same kernel with the
    operands swapped.  `tokens`: an already packed fmt='f16' token plane to share with `nearest_code`.  Cosine needs
    normalised token planes here (the token norm now varies along the reduced axis); L2 needs the tokens' 0.5|x|^2.
    rows = (code_list int32, count int32 [1], compact_keys): restrict the pass to the listed codes (device-side count;
    CVQ-VAE only needs the codes whose anchor gets a non-zero weight); the other entries stay all-ones."""
    cos = metric == 'Cosine'
    kw = dict(l2=False, index_offset=index_offset)
    certified = False
    if codebook.fmt != 'bf16':
        # fp16 codebook planes need fp16 token planes
        if x.dtype == torch.bfloat16:
            # raw bf16 tokens as ONE fp16 plane + the per-column 1/|x_n| scale in the epilogue: two MMA terms
            b = tokens if (tokens is not None and tokens.fmt == 'f16') else ops.pack_rows(x, fmt='f16')
            if b.inv_norm is None:
                b.inv_norm = ops.row_inv_norm(x, f16_rows=True)
            kw['scale_columns'] = True
            certified = codebook.lo_norm_max is not None
        else:
            b = ops.pack_rows(x, normalize=True, fmt='f16x2')      # normalised tokens as a pair: three terms
    else:
        b = ops.as_operand(x) if cos else None
        if b is not None:
            # bf16 tokens: ONE exact raw plane + a per-column 1/|x_n| scale in the epilogue instead of three planes
            # of the normalised tokens (halves the MMA work of this pass)
            b.inv_norm = ops.row_inv_norm(x)
            kw['scale_columns'] = True
        else:
            # folded codebook: here the tokens' -0.5|x|^2 is the term that varies along the reduced axis
            b = ops.pack_rows(x, normalize=cos, planes=_planes_for(x, cos, precision), want_half_sqnorm=not cos,
                              fold='tokens+h' if codebook.folded is not None else None)
            kw['l2'] = not cos
    keys = ops.new_keys(codebook.rows, x.device)
    if rows is not None:
        code_list, count, compact = rows
        a = ops.gather_operand_rows(codebook, code_list, count)     # the listed codes as a compact operand
        ops.assign(a, b, compact, a_rows_dev=count, **kw)
        return ops.scatter_keys(compact, code_list, count, keys)
    if certified:
        return certified_assign(codebook, b, keys, scale_columns=True, index_offset=index_offset)
    return ops.assign(codebook, b, keys, **kw)


class _DistanceMatrix(torch.autograd.Function):
    """COMPATIBILITY MODE (SURVEY.md §8f-4): the materialised [N, K] distance matrix of the reference
    (`torch.cdist(x, e)` / `1 - normalize(x) @ normalize(e).T`, vq/algorithms/vq/distances.py:28-46) for the few
    components that consume it.  Forward: the hand-written fp32 kernel `vqb_distance_matrix`.  Backward (only
    EntropyLoss differentiates through the matrix): the two [N, K] x [K, D] products are plain library GEMMs — this
    path exists for parity of rarely used components, not for speed."""

    @staticmethod
    def forward(ctx, x, W, metric):
        d = ops.distance_matrix(x, W, metric)
        ctx.save_for_backward(x, W, d)
        ctx.metric = metric
        return d

    @staticmethod
    def backward(ctx, G):
        x, W, d = ctx.saved_tensors
        G = G.contiguous().float()
        xf = x.float()
        if ctx.metric == 'Cosine':
            xn, en = ops.l2norm_forward(x), ops.l2norm_forward(W)
            gx = ops.l2norm_backward(-(G @ en), xf) if ctx.needs_input_grad[0] else None
            gW = ops.l2norm_backward(-(G.t() @ xn), W) if ctx.needs_input_grad[1] else None
        else:   # d = sqrt(|x|^2 - 2 x.e + |e|^2):  dd/dx = (x - e) / d
            H = torch.where(d > 0, G / d, torch.zeros_like(G))
            gx = (H.sum(1, keepdim=True) * xf - H @ W) if ctx.needs_input_grad[0] else None
            gW = (H.sum(0).unsqueeze(1) * W - H.t() @ xf) if ctx.needs_input_grad[1] else None
        return (None if gx is None else gx.to(x.dtype)), gW, None


def distance_matrix(x: torch.Tensor, W: torch.Tensor, metric: str) -> torch.Tensor:
    """Compatibility mode: differentiable fp32 [N, K] distance matrix (see _DistanceMatrix)."""
    return _DistanceMatrix.apply(x.contiguous(), W.contiguous(), metric)


class _EmbeddingGather(torch.autograd.Function):
    """z = W[quant] with the gradient scattered back into the codebook rows (the unfused decode of the hook-compatible
    template path; the fused forward never needs it).  Backward = the statistics scatter kernel."""

    @staticmethod
    def forward(ctx, W, quant):
        ctx.save_for_backward(quant)
        ctx.shape = W.shape
        return ops.embedding_gather(W, quant)

    @staticmethod
    def backward(ctx, g):
        (quant,) = ctx.saved_tensors
        K, D = ctx.shape
        stats = ops.scatter_stats(g.reshape(-1, D).contiguous().float(), quant.reshape(-1).contiguous(), K)
        return stats[:K * D].view(K, D), None


def embedding_lookup(W: torch.Tensor, quant: torch.Tensor) -> torch.Tensor:
    return _EmbeddingGather.apply(W, quant.contiguous())


class _TransposeLast2(torch.autograd.Function):
    """[B, R, C] -> [B, C, R]; the backward is the same kernel on the gradient."""

    @staticmethod
    def forward(ctx, x):
        return ops.transpose_last2(x)

    @staticmethod
    def backward(ctx, g):
        return ops.transpose_last2(g.contiguous())


def nchw_to_rows(x: torch.Tensor) -> torch.Tensor:
    """einops 'b c h w -> (b h w) c' (vq/tasks/image_tokenization/models/base.py:124) as one transpose kernel."""
    b, c, h, w = x.shape
    return _TransposeLast2.apply(x.contiguous().view(b, c, h * w)).view(b * h * w, c)


def rows_to_nchw(z: torch.Tensor, b: int, c: int, h: int, w: int) -> torch.Tensor:
    """einops '(b h w) c -> b c h w' + .contiguous() (base.py:126-127) as one transpose kernel."""
    return _TransposeLast2.apply(z.contiguous().view(b, h * w, c)).view(b, c, h, w)


class CodebookRef:
    """What a pending backward holds instead of the codebook tensor: the codebook is updated IN PLACE by the
    update kernels (the reference rebinds `weight.data` to a new tensor, update.py:56, so its saved tensors stay
    intact).  `VectorQuantizer.protect_saved_codebook()` swaps in a private copy (copy-on-write) right before an
    in-place update if a backward that saved the live codebook is still pending — e.g. two training forwards
    before the first backward — and costs nothing in the usual forward/backward alternation."""
    __slots__ = ('tensor', '__weakref__')

    def __init__(self, tensor: torch.Tensor) -> None:
        self.tensor = tensor


class _QuantizeSTELoss(torch.autograd.Function):
    """Outputs the four MSE terms as SEPARATE 0-dim tensors so that autograd hands their upstream gradients
    back as four device scalars (no select_backward / stack kernels between the loss and our backward)."""

    @staticmethod
    def forward(ctx, x, W, index, index_is_keys, key_offset, normalize_x, want_norm, ref, x_nchw):
        # x_nchw: the caller's [b, c, h, w] latents of which `x` is the (detached) token-major copy: z is then written
        # straight into that layout and the backward reads / writes NCHW gradients (no transposes around the kernels)
        hw = 0 if x_nchw is None else x_nchw.shape[2] * x_nchw.shape[3]
        z, mse4, quant, xn = ops.gather_ste_loss(
            x, W, quant=None if index_is_keys else index, keys=index if index_is_keys else None,
            key_offset=key_offset, normalize_x=normalize_x, want_norm=want_norm, want_quant=index_is_keys,
            want_xnorm=normalize_x, z_hw=hw)
        if x_nchw is not None:
            z = z.view(x_nchw.shape)
        ctx.nchw = None if x_nchw is None else tuple(x_nchw.shape)
        if quant is None:
            quant = index
        ctx.save_for_backward(x, quant)
        ctx.codebook = ref if ref is not None else CodebookRef(W.detach())
        ctx.cfg = (normalize_x, want_norm)
        ctx.set_materialize_grads(False)   # unused outputs arrive as None instead of freshly zero-filled tensors
        if xn is None:
            xn = x.detach()
        ctx.mark_non_differentiable(quant, xn)
        m0, m1, m2, m3 = mse4.unbind(0)
        return z, m0, m1, m2, m3, quant, xn

    @staticmethod
    def backward(ctx, gz, g0, g1, g2, g3, _gq, _gxn):
        x, quant = ctx.saved_tensors
        W = ctx.codebook.tensor
        normalize_x, want_norm = ctx.cfg
        if gz is None:
            gz = torch.zeros(ctx.nchw or x.shape, dtype=torch.float32, device=x.device)
        g4 = [None if g is None else g.contiguous().float() for g in (g0, g1, g2, g3)]
        hw = 0 if ctx.nchw is None else ctx.nchw[2] * ctx.nchw[3]
        need_gx = ctx.needs_input_grad[0] or ctx.needs_input_grad[8]
        gx, gW = ops.quantize_backward(gz.contiguous(), x, W, quant, g4, normalize_x=normalize_x,
                                       want_norm=want_norm, need_gW=ctx.needs_input_grad[1], g_hw=hw)
        if ctx.nchw is not None:     # the gradient belongs to the NCHW latents
            return None, gW, None, None, None, None, None, None, (gx.view(ctx.nchw) if need_gx else None)
        return (gx if need_gx else None), gW, None, None, None, None, None, None, None


def quantize_ste_loss(x: torch.Tensor, W: torch.Tensor, index: torch.Tensor, want_norm: bool, *,
                      index_is_keys: bool = False, key_offset: int = 0, normalize_x: bool = False,
                      codebook_ref: CodebookRef | None = None, nchw: torch.Tensor | None = None):
    """One kernel: [x' = F.normalize(x)] -> gather W[q] -> straight-through -> MSE terms.
    -> (z_ste [N,D] fp32: value x' + (W[q] - x'), gradient to x only;
        mse4 = (codebook, commitment, codebook(norm), commitment(norm)) as four 0-dim tensors;
        quant int64 [N] (unpacked from the keys when index_is_keys);  x' (detached; x itself if not normalised))"""
    z, m0, m1, m2, m3, quant, xn = _QuantizeSTELoss.apply(x.contiguous(), W, index, bool(index_is_keys),
                                                          int(key_offset), bool(normalize_x), bool(want_norm),
                                                          codebook_ref, nchw)
    return z, (m0, m1, m2, m3), quant, xn


@torch.no_grad()
def residual_levels(levels, x: torch.Tensor, memos, want_norm: bool, *, quant_out: torch.Tensor | None = None,
                    z_out: torch.Tensor | None = None, z_hw: int = 0, compact_out: torch.Tensor | None = None,
                    track_codebooks: bool = False):
    """The level loop of a residual quantizer: level l runs its own `encode` (before_encode -> assignment ->
    after_encode, codebook updates included) on r_{l-1}, then ONE `vqb_residual_step` launch gathers W_l[q_l] from the
    codebook as that encode left it, writes the [N, L] indices, the running sum and r_l, and at the last level
    z = x + (zhat_L - x).  memos[l] becomes level l's memo (x = r_{l-1}, quant = its indices).
    compact_out: uint16 / int32 [L, N]: the compact ids of every level, straight from its packed assignment keys (every
    level must then accept packed keys: no training callback reads the indices).
    -> (mse fp32 [L, 4], [CodebookRef per level] (registered with the level when track_codebooks))"""
    N, D = x.shape
    L = len(levels)
    mse = torch.empty((L, 4), dtype=torch.float32, device=x.device)
    zhat = torch.empty((N, D), dtype=torch.float32, device=x.device) if (L > 1 and z_out is not None) else None
    refs = []
    r = x
    for l, level in enumerate(levels):
        memo = memos[l]
        lazy = level._callbacks.packed_keys_ok()
        memo['_lazy_unpack'] = lazy
        _, index, memo = level.encode(r, memo)
        W = level._weight().detach()
        ref = CodebookRef(W)
        if track_codebooks:
            level._pending.add(ref)
        refs.append(ref)
        last = l == L - 1
        if compact_out is not None:
            assert lazy, 'compact ids need the packed assignment keys'
            ops.compact_tokens(index, level.codebook_size, out=compact_out[l])
        r_out = None if last else torch.empty((N, D), dtype=torch.float32, device=x.device)
        if not (last and z_out is None and quant_out is None):
            ops.residual_step(r, x, W, mse[l], level=l, L=L, quant=None if lazy else index, keys=index if lazy else None,
                              quant_out=quant_out, zhat=zhat, r_out=r_out, z_out=z_out if last else None, z_hw=z_hw,
                              want_norm=want_norm)
        memo['x'] = r
        memo['quant'] = quant_out[:, l] if quant_out is not None else index
        r = r_out
    return mse, refs


class _ResidualQuantize(torch.autograd.Function):
    """The whole depth of a residual quantizer as ONE node: forward = the level loop (`residual_levels`), backward = one
    `vqb_residual_backward` launch for all levels (+ per-level code sort / segment sum under the deterministic flag).
    Outputs z, quant [N, L] and the 4 L MSE terms as separate 0-dim tensors (their upstream gradients arrive as
    device scalars)."""

    @staticmethod
    def forward(ctx, x, x_nchw, levels, memos, want_norm, track, *Ws):
        N, D = x.shape
        L = len(levels)
        hw = 0 if x_nchw is None else x_nchw.shape[2] * x_nchw.shape[3]
        z = torch.empty(tuple(x_nchw.shape) if x_nchw is not None else (N, D), dtype=torch.float32, device=x.device)
        quant = torch.empty((N, L), dtype=torch.int64, device=x.device)
        mse, refs = residual_levels(levels, x, memos, want_norm, quant_out=quant, z_out=z, z_hw=hw,
                                    track_codebooks=track)
        ctx.save_for_backward(x, quant)
        ctx.refs = refs
        ctx.nchw = None if x_nchw is None else tuple(x_nchw.shape)
        ctx.want_norm = want_norm
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(quant)
        return (z, quant) + tuple(mse.view(-1).unbind(0))

    @staticmethod
    def backward(ctx, gz, _gq, *g):
        x, quant = ctx.saved_tensors
        L = quant.shape[1]
        if gz is None:
            gz = torch.zeros(ctx.nchw or x.shape, dtype=torch.float32, device=x.device)
        g4s = [[None if t is None else t.contiguous().float() for t in g[4 * l:4 * l + 4]] for l in range(L)]
        need_gW = list(ctx.needs_input_grad[6:6 + L])
        hw = 0 if ctx.nchw is None else ctx.nchw[2] * ctx.nchw[3]
        gx, gWs = ops.residual_backward(gz.contiguous(), x, [r.tensor for r in ctx.refs], quant, g4s,
                                        want_norm=ctx.want_norm, need_gW=need_gW, g_hw=hw)
        if ctx.nchw is not None:     # the gradient belongs to the NCHW latents
            return (None, gx.view(ctx.nchw) if ctx.needs_input_grad[1] else None, None, None, None, None, *gWs)
        return (gx if ctx.needs_input_grad[0] else None, None, None, None, None, None, *gWs)


def residual_quantize(levels, x: torch.Tensor, memos, want_norm: bool, *, nchw: torch.Tensor | None = None):
    """Residual quantization of x [N, D] (fp32 / bf16) through `levels` (VectorQuantizer modules sharing K and D).
    -> (z fp32 [N, D] (or NCHW like `nchw`): value x + (zhat_L - x), gradient straight to x;
        quant int64 [N, L];  mse: per level the four MSE terms (codebook, commitment, codebook-norm,
        commitment-norm) of e_l against r_{l-1}, 0-dim tensors whose gradients reach W_l and, through r_{l-1}, x)"""
    Ws = [level._weight() for level in levels]
    track = torch.is_grad_enabled() and (x.requires_grad or (nchw is not None and nchw.requires_grad)
                                         or any(W.requires_grad for W in Ws))
    out = _ResidualQuantize.apply(x.contiguous(), nchw, list(levels), memos, bool(want_norm), track, *Ws)
    z, quant, flat = out[0], out[1], out[2:]
    return z, quant, [tuple(flat[4 * l:4 * l + 4]) for l in range(len(levels))]


@torch.no_grad()
def group_encode(groups, xs: torch.Tensor, memos, *, keys: torch.Tensor | None = None, track_codebooks: bool = False):
    """The group loop of a grouped quantizer: group g runs its own `encode` (before_encode -> assignment ->
    after_encode, codebook updates included) on its token slice xs[g] ([G, N, Dg] from `ops.split_groups`), its
    assignment writing the packed keys straight into row g of ONE [G, N] buffer (`keys`, whose rows must be
    contiguous; allocated when None).  memos[g] becomes group g's memo.
    -> (keys int64 [G, N], [CodebookRef per group] of the codebooks as the encodes left them (registered with the
    group when track_codebooks))"""
    G, N, _ = xs.shape
    if keys is None:
        keys = torch.empty((G, N), dtype=torch.int64, device=xs.device)
    refs = []
    for g, group in enumerate(groups):
        memo = memos[g]
        memo['_keys_out'] = keys[g]
        memo['_lazy_unpack'] = group._callbacks.packed_keys_ok()
        group.encode(xs[g], memo)     # int64 indices only when a training callback reads them; the keys stay valid
        ref = CodebookRef(group._weight().detach())
        if track_codebooks:
            group._pending.add(ref)
        refs.append(ref)
    return keys, refs


class _GroupedQuantize(torch.autograd.Function):
    """Every group of a grouped quantizer as ONE node: forward = `ops.split_groups` + the group loop (`group_encode`) +
    one `vqb_group_gather_ste_loss` launch; backward = one `vqb_group_backward` launch for all groups (+ per-group code
    sort / segment sum under the deterministic flag).  x is the tokens [N, D] or the NCHW latents [b, D, h, w]; z and
    gx have x's layout.  Outputs z, quant [N, G] and the 4 G MSE terms as separate 0-dim tensors (their upstream
    gradients arrive as device scalars); memos[g] gets 'x' (the split slice xs[g]) and 'quant' (quant[:, g])."""

    @staticmethod
    def forward(ctx, x, groups, memos, want_norm, track, *Ws):
        G = len(groups)
        nchw = x.dim() == 4
        hw = x.shape[2] * x.shape[3] if nchw else 0
        xd = x.detach()
        xs = xd.view(1, *xd.shape) if (G == 1 and not nchw) else ops.split_groups(xd, G)
        N = xs.shape[1]
        keys, refs = group_encode(groups, xs, memos, track_codebooks=track)
        z = torch.empty(tuple(x.shape), dtype=torch.float32, device=x.device)
        quant = torch.empty((N, G), dtype=torch.int64, device=x.device)
        _, mse = ops.group_gather_ste_loss(xs, [r.tensor for r in refs], keys=keys, want_norm=want_norm, quant_out=quant,
                                           z_out=z, z_hw=hw)
        for g, memo in enumerate(memos):
            memo.update(x=xs[g], quant=quant[:, g])
        ctx.save_for_backward(xs, quant)
        ctx.refs = refs
        ctx.shape = tuple(x.shape)
        ctx.hw = hw
        ctx.want_norm = want_norm
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(quant)
        return (z, quant) + tuple(mse.view(-1).unbind(0))

    @staticmethod
    def backward(ctx, gz, _gq, *g):
        xs, quant = ctx.saved_tensors
        G = xs.shape[0]
        if gz is None:
            gz = torch.zeros(ctx.shape, dtype=torch.float32, device=xs.device)
        g4s = [[None if t is None else t.contiguous().float() for t in g[4 * i:4 * i + 4]] for i in range(G)]
        need_gW = list(ctx.needs_input_grad[5:5 + G])
        gx, gWs = ops.group_backward(gz.contiguous(), xs, [r.tensor for r in ctx.refs], quant, g4s,
                                     want_norm=ctx.want_norm, need_gW=need_gW, g_hw=ctx.hw)
        return (gx if ctx.needs_input_grad[0] else None, None, None, None, None, *gWs)


def grouped_quantize(groups, x: torch.Tensor, memos, want_norm: bool):
    """Grouped quantization of x (tokens [N, D] or latents [b, D, h, w]; fp32 / bf16) through `groups` (VectorQuantizer
    modules sharing K and Dg = D / G), group g on channels [g*Dg, (g+1)*Dg).
    -> (z fp32 in x's layout: value x_g + (W_g[q_g] - x_g) per group, gradient straight to x;  quant int64 [N, G];
        mse: per group the four MSE terms (codebook, commitment, codebook-norm,
        commitment-norm) of W_g[q_g] against x_g, 0-dim tensors whose gradients reach W_g and x)"""
    Ws = [group._weight() for group in groups]
    track = torch.is_grad_enabled() and (x.requires_grad or any(W.requires_grad for W in Ws))
    out = _GroupedQuantize.apply(x.contiguous(), list(groups), memos, bool(want_norm), track, *Ws)
    z, quant, flat = out[0], out[1], out[2:]
    return z, quant, [tuple(flat[4 * i:4 * i + 4]) for i in range(len(groups))]


class _FSQ(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x, params):
        zq, idx = ops.fsq_forward(x, params)
        ctx.save_for_backward(x)
        ctx.params = params
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(idx)
        return zq, idx

    @staticmethod
    def backward(ctx, gz, _gidx):
        (x,) = ctx.saved_tensors
        if gz is None:
            return None, None
        return ops.fsq_backward(gz.contiguous(), x, ctx.params), None


def fsq_quantize(x: torch.Tensor, params):
    return _FSQ.apply(x.contiguous(), params)
