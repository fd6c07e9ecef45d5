"""Quantizer modules under the reference's registry names, config keys and forward contract
(SURVEY.md §8b):  forward(x [N, D], memo) -> (z [N, D], loss [], memo)  with
memo['x'], memo['quant'] (int64 [N]; int32 for FSQ), memo['encode'], memo['decode'], memo['loss'][name].

Reference:
    BaseQuantizer            vq/tasks/image_tokenization/models/quantizers/base.py:26-182
    VectorQuantizer          vq/algorithms/vq/quantizers.py:19-117
    VQGANQuantizer           vq/algorithms/vqgan/quantizer.py:11-21
    VQKDQuantizer            vq/algorithms/vqkd/quantizers/base.py:11-15
    ScalarQuantizer          vq/algorithms/sq/quantizers.py:9-11
    FiniteScalarQuantizer    vq/algorithms/fsq/quantizers.py:74-150
The arithmetic runs in the sm_100a kernels of libvqb200.so: tensors must live on a CUDA device and the
library must be present — there is no CPU or eager-PyTorch fallback.
"""
from __future__ import annotations

import copy
import weakref
from typing import Mapping, Sequence

import torch
from torch import nn

from . import functional as Fq
from . import ops, parallel
from ._lib import MAX_LEVELS, VQBError
from .callbacks import BaseCallback, ComposedCallback
from .distances import BaseDistance
from .registry import (Config, InitRegistry, ModelRegistry, ModuleDict, VQITQuantizerCallbackRegistry,
                       VQITQuantizerDistanceRegistry, VQITQuantizerLossRegistry, VQITQuantizerRegistry,
                       build_module_dict, get_config)

__all__ = ['BaseQuantizer', 'VectorQuantizer', 'VQGANQuantizer', 'VQKDQuantizer', 'ScalarQuantizer',
           'FiniteScalarQuantizer', 'ResidualVectorQuantizer', 'GroupedVectorQuantizer']


def get_memo(memo: dict, key: str) -> dict:
    """vq/utils/misc.py:30-38."""
    if key not in memo:
        memo[key] = dict()
    assert isinstance(memo[key], dict)
    return memo[key]


def _check_tokens(x: torch.Tensor, dim: int) -> torch.Tensor:
    if not x.is_cuda:
        raise VQBError('vector_quantization_b200 quantizers run on CUDA (sm_100a) tensors only; no CPU fallback')
    if x.dim() != 2 or x.shape[1] != dim:
        raise ValueError(f'expected tokens of shape [N, {dim}] ("b c h w -> (b h w) c"), got {tuple(x.shape)}')
    if x.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f'tokens must be float32 or bfloat16, got {x.dtype}')
    return x.contiguous()


class BaseQuantizer(nn.Module):

    def __init__(self, *args, callbacks: ComposedCallback, losses: ModuleDict, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self._callbacks = callbacks
        self._losses = losses
        self._callbacks.bind(self)

    @classmethod
    def build_pre_hook(cls, config: Mapping, registry, item) -> Mapping:
        config['callbacks'] = VQITQuantizerCallbackRegistry.build(
            Config(type='ComposedCallback', callbacks=config.get('callbacks', [])))
        config['losses'] = build_module_dict(VQITQuantizerLossRegistry, get_config(config, 'losses'))
        return config

    @property
    def embedding_dim(self) -> int:
        raise NotImplementedError

    @property
    def codebook_size(self) -> int:
        raise NotImplementedError

    @property
    def embeddings(self) -> torch.Tensor:
        raise NotImplementedError

    def _init_weights(self, config: Mapping) -> bool:
        return True

    def init_weights(self, config: Mapping) -> bool:
        config = Config(config)
        before = config.pop('before_init_weights', Config())
        after = config.pop('after_init_weights', Config())
        self._callbacks.before_init_weights(before)
        recursive = self._init_weights(config)
        return self._callbacks.after_init_weights(after, recursive)

    # -- template (reference base.py:123-182) --------------------------------------------------------
    def _encode(self, x: torch.Tensor, memo: dict):
        raise NotImplementedError

    def encode(self, x: torch.Tensor, memo: dict):
        x = self._callbacks.before_encode(x, memo)
        enc = get_memo(memo, 'encode')
        for flag in ('_normalize_codebook', '_normalize_x', '_lazy_unpack', '_zero_fill', '_keys_out'):  # requests of the callbacks / forward
            if flag in memo:
                enc[flag] = memo[flag]
        memo.pop('_normalize_codebook', None)
        memo.pop('_lazy_unpack', None)
        memo.pop('_zero_fill', None)
        memo.pop('_keys_out', None)
        quant, memo['encode'] = self._encode(x, enc)
        quant = self._callbacks.after_encode(x, quant, memo)
        memo['encode'].pop('_column_ctx', None)      # operands kept for the callbacks' column arg-min
        return x, quant, memo

    def _decode(self, quant: torch.Tensor, memo: dict):
        raise NotImplementedError

    def decode(self, quant: torch.Tensor, memo: dict):
        quant = self._callbacks.before_decode(quant, memo)
        z, memo['decode'] = self._decode(quant, get_memo(memo, 'decode'))
        z = self._callbacks.after_decode(z, memo)
        return z, memo

    def _loss(self, z: torch.Tensor, x: torch.Tensor, memo: dict):
        """reference base.py:151-160: evaluate the configured losses, record them in the (loss) memo, sum."""
        losses = self._losses(z, x, memo)
        memo.update(losses)
        loss = x.new_zeros([], dtype=torch.float32)
        for v in losses.values():
            loss = loss + v
        return loss, memo

    def loss(self, z: torch.Tensor, x: torch.Tensor, memo: dict):
        """reference base.py:162-171."""
        z, x = self._callbacks.before_loss(z, x, memo)
        loss_memo = get_memo(memo, 'loss')
        distance = memo.get('encode', {}).get('distance') if isinstance(memo.get('encode'), dict) else None
        if distance is not None:
            loss_memo.setdefault('distance', distance)     # where EntropyLoss looks it up (losses.py:142)
        loss, memo['loss'] = self._loss(z, x, loss_memo)
        memo['loss'].pop('distance', None)
        loss = self._callbacks.after_loss(loss, memo)
        return loss, memo

    def forward(self, x: torch.Tensor, memo: dict):
        """reference base.py:173-182 (the template; VectorQuantizer overrides it with the fused kernels)."""
        x, quant, memo = self.encode(x, memo)
        memo.update(x=x, quant=quant)
        z, memo = self.decode(quant, memo)
        loss, memo = self.loss(z, x, memo)
        return z, loss, memo


@VQITQuantizerRegistry.register_()
class VectorQuantizer(BaseQuantizer):
    """distance -> arg-min -> (codebook update callbacks) -> gather -> losses -> straight-through, as three
    kernel launches: pack+assign (tcgen05, no N x K matrix), [stats/update], fused gather+STE+loss.

    rotation_trick: the encoder gradient of z follows the rotation trick (Fifty et al., arXiv:2410.06424; DESIGN.md
    §4.9) instead of the straight-through estimator.  z, the losses, the indices, the codebook updates and the codebook
    gradient are unchanged; only the gradient reaching x differs.  Not available with callbacks that hook decode or
    loss (they run the unfused template)."""

    def __init__(self, *args, embedding: nn.Embedding, distance: BaseDistance, precision: str = Fq.DEFAULT_PRECISION,
                 materialize_distance: bool = False, rotation_trick: bool = False, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        if precision not in Fq.PRECISION_PLANES:
            raise ValueError(f'precision must be one of {sorted(Fq.PRECISION_PLANES)}')
        self.rotation_trick = bool(rotation_trick)
        if self.rotation_trick:
            for c in self._callbacks:
                hooks = [h for h in ('before_decode', 'after_decode', 'before_loss', 'after_loss')
                         if getattr(type(c), h) is not getattr(BaseCallback, h)]
                if hooks:
                    raise ValueError(f'{type(self).__name__}: rotation_trick is not supported with callback '
                                     f'{type(c).__name__}, which hooks {", ".join(hooks)} (the unfused template path)')
        self._embedding = embedding
        self._distance = distance
        self.precision = precision
        # COMPATIBILITY / DEBUG switch: also build the reference's memo['encode']['distance'] ([N, K], quantizers.py:98)
        # for user callbacks that read it.  Implied by an EntropyLoss or a MultinomialAnchor in the config.
        self.materialize_distance = bool(materialize_distance)
        self._pending = weakref.WeakSet()   # CodebookRef of every forward whose backward has not run yet

    def protect_saved_codebook(self) -> None:
        """Call before ANY in-place write to the codebook: pending backwards that saved the live tensor get a private
        copy first (see functional.CodebookRef)."""
        live = self._embedding.weight.data_ptr()
        shared = [r for r in self._pending if r.tensor.data_ptr() == live]
        if shared:
            snapshot = shared[0].tensor.clone()
            for r in shared:
                r.tensor = snapshot
        self._pending.clear()

    @classmethod
    def build_pre_hook(cls, config, registry, item):
        config = super().build_pre_hook(config, registry, item)
        config['embedding'] = ModelRegistry.build_or_return(config['embedding'])
        config['distance'] = VQITQuantizerDistanceRegistry.build_or_return(config['distance'])
        return config

    @property
    def embedding(self) -> nn.Embedding:
        return self._embedding

    @property
    def distance(self) -> BaseDistance:
        return self._distance

    @property
    def embedding_dim(self) -> int:
        return self._embedding.embedding_dim

    @property
    def codebook_size(self) -> int:
        return self._embedding.num_embeddings

    @property
    def embeddings(self) -> torch.Tensor:
        return self._embedding.weight.clone()

    def _init_weights(self, config) -> bool:
        if config:                      # an empty node (no `init_weights` in the config) keeps nn.Embedding's own init
            InitRegistry.build(config)(self._embedding.weight)
        return False

    def _weight(self) -> torch.Tensor:
        W = self._embedding.weight
        if W.dtype != torch.float32:
            raise TypeError('the codebook (nn.Embedding weight) must be float32, as in the reference')
        if not W.is_cuda:
            raise VQBError('the codebook must live on a CUDA device; there is no CPU fallback')
        return W

    @property
    def wants_distance(self) -> bool:
        return (self.materialize_distance or self._callbacks.needs_distance
                or any(loss.needs_distance for loss in self._losses.values()))

    def _encode(self, x: torch.Tensor, memo: dict):
        if self.wants_distance:
            # compatibility mode: the reference's differentiable [N, K] matrix against the codebook as it is BEFORE
            # this step's update (`self.embeddings` clones, quantizers.py:84-85,97-98)
            W = self._weight()
            if memo.get('_normalize_codebook', False):
                self.protect_saved_codebook()
                ops.pack_rows(W.data, normalize=True, planes=1, writeback=W.data)     # NormalizeCallback, in place
            memo['distance'] = Fq.distance_matrix(_check_tokens(x, self.embedding_dim), W.clone(), self._distance.metric)
        return self._encode_nograd(x, memo)

    @torch.no_grad()
    def _encode_nograd(self, x: torch.Tensor, memo: dict):
        """Nearest code per token.  Launches: codebook pack (normalise-in-place + operand planes + key reset),
        [token pack unless zero-copy], tcgen05 assignment, [key unpack unless deferred to the gather kernel]."""
        x = _check_tokens(x.detach(), self.embedding_dim)
        W = self._weight().data
        metric = self._distance.metric
        keys = memo.pop('_keys_out', None)      # a caller's [N] int64 buffer (GroupedVectorQuantizer: a row of [G, N])
        if keys is None:
            keys = torch.empty((x.shape[0],), dtype=torch.int64, device=x.device)
        writeback = memo.pop('_normalize_codebook', False)
        if writeback:
            self.protect_saved_codebook()   # the codebook is normalised in place
        zero_fill = memo.pop('_zero_fill', None)
        book = Fq.pack_codebook(W, metric, precision=self.precision, writeback_normalized=writeback, reset_keys=keys,
                                tokens=x, zero_fill=zero_fill)
        if zero_fill is not None:
            memo['_zeroed'] = True
        normalize_tokens = memo.pop('_normalize_x', False)
        want_columns = self.training and self._callbacks.needs_column_nearest
        tokens = None
        if want_columns and book.fmt != 'bf16' and x.dtype == torch.bfloat16:
            tokens = ops.pack_rows(x, fmt='f16')      # one fp16 token plane shared by the row and the column pass
        Fq.nearest_code(x, book, metric, precision=self.precision, keys=keys, keys_are_reset=True,
                        normalize_tokens=normalize_tokens, tokens=tokens)
        memo['keys'] = keys
        if want_columns:
            # the column arg-min (per code, the nearest token) runs when the callback asks for it: CVQVAECallback first
            # works out WHICH codes need it this step (`column_keys`)
            memo['_column_ctx'] = dict(x=x, book=book, tokens=tokens, metric=metric)
        if memo.pop('_lazy_unpack', False):
            return keys, memo            # forward(): the fused gather kernel unpacks the indices
        return ops.unpack_keys(keys), memo

    @torch.no_grad()
    def column_keys(self, enc_memo: dict, rows=None) -> torch.Tensor:
        """Packed keys [K] of the nearest token per code (NearestAnchor's `d.argmin(0)`, cvqvae/anchors.py:83), computed
        on the operands `_encode` left in its memo; `rows` restricts the pass to a device-side list of codes.  The result
        is also stored as memo['encode']['column_keys']."""
        ctx = enc_memo.pop('_column_ctx')
        x = ctx['x']
        offset = parallel.rank() * x.shape[0] if self._callbacks.column_nearest_global else 0
        keys = Fq.column_nearest(x, ctx['book'], ctx['metric'], precision=self.precision, index_offset=offset,
                                 tokens=ctx['tokens'], rows=rows)
        enc_memo['column_keys'] = keys
        return keys

    def _decode(self, quant: torch.Tensor, memo: dict):
        """`nn.Embedding` gather, any index shape (decode_from_quant).  Differentiable w.r.t. the codebook when it
        requires grad (the unfused template path); plain gather kernel otherwise."""
        W = self._weight()
        if torch.is_grad_enabled() and W.requires_grad:
            return Fq.embedding_lookup(W, quant), memo
        return ops.embedding_gather(W.data, quant.contiguous()), memo

    def _loss(self, z: torch.Tensor, x: torch.Tensor, memo: dict):
        """Standalone `loss(z, x)` of the reference template (base.py:151-160) on ARBITRARY (z, x): the fused kernel
        is reused with z as the "codebook" and the identity assignment, which yields exactly mse(z, x) with the
        codebook-role gradient routed to z and the commitment-role gradient to x."""
        x2, z2 = x.reshape(-1, x.shape[-1]), z.reshape(-1, z.shape[-1]).float()
        index = torch.arange(x2.shape[0], dtype=torch.int64, device=x2.device)
        _, mse4, _, _ = Fq.quantize_ste_loss(_check_tokens(x2, self.embedding_dim), z2.contiguous(), index,
                                             self._loss_terms())
        losses = {name: (m.from_mse4(mse4) if m.uses_mse4 else m(z, x, memo)) for name, m in self._losses.items()}
        memo.update(losses)
        loss = mse4[0].new_zeros([])
        for v in losses.values():
            loss = loss + v
        return loss, memo

    def can_fuse_nchw(self) -> bool:
        """May the caller's NCHW <-> token-major rearranges (models/base.py:124,126-127) be folded into the kernels?
        Yes when forward() takes the fused path and no callback changes the tokens it is handed in before_encode
        (NormalizeCallback defers its normalisation into the fused kernels when `lazy_normalize_ok`)."""
        from .callbacks import BaseCallback, NormalizeCallback
        hooked = any(self._callbacks.overrides(h) for h in ('before_decode', 'after_decode', 'before_loss', 'after_loss'))
        known = all(type(c).before_encode is BaseCallback.before_encode or isinstance(c, NormalizeCallback)
                    for c in self._callbacks)
        normalizes = any(isinstance(c, NormalizeCallback) for c in self._callbacks)
        lazy = self._callbacks.lazy_normalize_ok() and not self.wants_distance
        return not hooked and known and (lazy or not normalizes) and not self.wants_distance

    def _forward_template(self, x: torch.Tensor, memo: dict):
        """The reference's unfused template (base.py:173-182 + quantizers.py:110-117) for configurations whose
        callbacks hook decode / loss: every hook point is honoured; each stage is still a kernel of the C-ABI."""
        x = _check_tokens(x, self.embedding_dim)
        x, quant, memo = self.encode(x, memo)
        memo.update(x=x, quant=quant)
        z, memo = self.decode(quant, memo)
        loss, memo = self.loss(z, x, memo)
        z = x + (z - x).detach()                       # ste, utils/ste.py:9-10
        return z, loss, memo

    def _loss_terms(self):
        want_norm = False
        for loss in self._losses.values():
            want_norm = want_norm or loss.needs_norm
        return want_norm

    def forward(self, x: torch.Tensor, memo: dict):
        if any(self._callbacks.overrides(h) for h in ('before_decode', 'after_decode', 'before_loss', 'after_loss')):
            return self._forward_template(x, memo)
        x = _check_tokens(x, self.embedding_dim)
        nchw = memo.pop('_nchw', None)     # tokenizer.quantize: x is the token-major copy of these [b, c, h, w] latents
        # The packed keys go straight into the fused gather kernel, which also emits memo['quant'] — unless a callback
        # that overrides after_encode needs int64 indices first (VQKDCallback reads the keys itself).
        lazy_unpack = self._callbacks.packed_keys_ok()
        # NormalizeCallback may defer F.normalize(x) into the fused kernels only when nobody else reads x
        memo['_lazy_normalize'] = self._callbacks.lazy_normalize_ok() and not self.wants_distance
        memo['_lazy_unpack'] = lazy_unpack
        x, index, memo = self.encode(x, memo)
        memo.pop('_lazy_normalize', None)
        normalize_x = memo.pop('_normalize_x', False)
        W = self._weight()
        ref = None
        if torch.is_grad_enabled() and (x.requires_grad or W.requires_grad):
            ref = Fq.CodebookRef(W.detach())
            self._pending.add(ref)
        if nchw is not None:
            ref = ref or (Fq.CodebookRef(W.detach()) if torch.is_grad_enabled() and nchw.requires_grad else None)
            if ref is not None:
                self._pending.add(ref)
        z, mse4, quant, xn = Fq.quantize_ste_loss(x, W, index, self._loss_terms(), index_is_keys=lazy_unpack,
                                                  normalize_x=normalize_x, codebook_ref=ref, nchw=nchw,
                                                  rotate=self.rotation_trick)
        memo.update(x=xn if normalize_x else x, quant=quant)
        memo['decode'] = get_memo(memo, 'decode')
        loss_memo = get_memo(memo, 'loss')
        loss = None
        distance = memo['encode'].get('distance')
        if distance is not None:
            loss_memo['distance'] = distance              # where EntropyLoss looks it up (losses.py:142)
        for name, module in self._losses.items():
            value = module.from_mse4(mse4) if module.uses_mse4 else module(z, memo['x'], loss_memo)
            loss_memo[name] = value
            loss = value if loss is None else loss + value
        loss_memo.pop('distance', None)
        if loss is None:
            loss = mse4[0].new_zeros([])
        return z, loss, memo


@VQITQuantizerRegistry.register_()
class VQGANQuantizer(VectorQuantizer):

    def _init_weights(self, config) -> bool:
        if dict(config) == dict(type='vqgan'):
            config = Config(type='uniform_', a=-1.0 / self.codebook_size, b=1.0 / self.codebook_size)
        return super()._init_weights(config)


@VQITQuantizerRegistry.register_()
class VQKDQuantizer(VectorQuantizer):

    def _init_weights(self, config) -> bool:
        return False


@VQITQuantizerRegistry.register_()
class ScalarQuantizer(BaseQuantizer):
    pass


@VQITQuantizerRegistry.register_()
class FiniteScalarQuantizer(ScalarQuantizer):
    """tanh bound -> round (STE) -> mixed-radix index, one kernel (fsq/quantizers.py:108-126)."""

    def __init__(self, *args, eps: float = 1e-3, num_scalars_per_channel: Sequence[int], **kwargs) -> None:
        super().__init__(*args, **kwargs)
        levels = tuple(int(v) for v in num_scalars_per_channel)
        self._eps = eps
        self._levels = levels
        self._params = ops.fsq_params(levels, eps)
        max_per_digit = torch.tensor(levels, dtype=torch.int)
        cumprod = torch.tensor((1,) + levels[:-1]).cumprod(0)
        self._codebook_size = int(max_per_digit.prod().item())
        quant = torch.arange(self._codebook_size).unsqueeze(-1)
        digits = (quant // cumprod) % max_per_digit
        self.register_buffer('_embeddings', digits / (max_per_digit // 2) - 1)  # implicit codebook table, :90-93

    @property
    def embedding_dim(self) -> int:
        return len(self._levels)

    @property
    def codebook_size(self) -> int:
        return self._codebook_size

    @property
    def embeddings(self) -> torch.Tensor:
        return self.get_buffer('_embeddings')

    def _encode(self, x: torch.Tensor, memo: dict):
        x = _check_tokens(x, self.embedding_dim)
        zq, quant = Fq.fsq_quantize(x, self._params)
        memo['z'] = zq
        return quant, memo

    def _decode(self, quant: torch.Tensor, memo: dict):
        if 'z' in memo:
            return memo['z'], memo
        if not quant.is_cuda:
            raise VQBError('FSQ decode runs on CUDA tensors only; there is no CPU fallback')
        return ops.fsq_decode(quant.contiguous(), self._params), memo

    def decode(self, quant: torch.Tensor, memo: dict):
        enc, dec = get_memo(memo, 'encode'), get_memo(memo, 'decode')
        if 'z' in enc:
            dec['z'] = enc['z']
        return super().decode(quant, memo)

    def forward(self, x: torch.Tensor, memo: dict):
        x, quant, memo = self.encode(x, memo)
        memo.update(x=x, quant=quant)
        z, memo = self.decode(quant, memo)
        memo['loss'] = get_memo(memo, 'loss')
        return z, x.new_zeros([]), memo


class _ComposedQuantizer(BaseQuantizer):
    """What ResidualVectorQuantizer and GroupedVectorQuantizer share.  M ordinary VectorQuantizer / VQGANQuantizer
    members are built from ONE config node (`quantizer`) and stored as `_quantizers.{i}`; each runs its own `encode`,
    one autograd node and one backward launch serve all of them, and one launch decodes.  The base owns the members
    (their checks, properties, codebooks and memos under memo[_members]), `decode`, the gate and buffer of
    `encode_compact` and the loss memo.  A subclass decides the input layout (`_check_input`, `encode`,
    `_encode_compact`), the node and the place of the rotation key (`_quantize`), the decode kernel (`_decode_ids`) and
    the reduction of the member losses (`_loss_mean`).

    Accepted members: L2 or Cosine distance, no callback or CVQVAECallback (NearestAnchor / CachedAnchor),
    CodebookLoss / CommitmentLoss / VQGANLoss.  Everything else raises a ValueError naming the offending item: callbacks
    that rewrite the tokens, callbacks that hook decode or loss, compatibility mode, a count outside [1, 16], members
    that are not VectorQuantizer modules (FSQ, or a composed quantizer: no nesting), and callbacks or losses on the
    composed node itself.  `init_weights` is applied to every member."""

    MAX_LEVELS = MAX_LEVELS
    _members = ''               # 'levels' / 'groups': the memo key of the member memos, and the noun of the messages
    _rotation_on_node = False   # rotation_trick is a key of this node; the member config may not set it
    _loss_mean = False          # the loss of a name is the mean over the members (groups), not their sum (levels)

    def _build_members(self, quantizer: Mapping, count, count_name: str) -> nn.ModuleList:
        name = type(self).__name__
        if isinstance(count, bool) or not isinstance(count, int) or not 1 <= count <= MAX_LEVELS:
            raise ValueError(f'{name}: {count_name}={count!r} is outside [1, {MAX_LEVELS}]')
        if list(self._callbacks) or len(self._losses):
            raise ValueError(f'{name}: callbacks and losses belong to the {self._members[:-1]} config (`quantizer`), '
                             f'not to the {name} node itself')
        cls = VQITQuantizerRegistry.lookup(quantizer['type']) if isinstance(quantizer.get('type'), str) else None
        if isinstance(cls, type) and not issubclass(cls, VectorQuantizer):
            raise ValueError(f'{name}: the {self._members} must be VectorQuantizer modules, got {cls.__name__}')
        built = []
        for _ in range(count):
            cfg = Config(copy.deepcopy(dict(quantizer)))
            cfg['init_weights'] = None       # applied per member by init_weights (after the train / eval mode is set)
            built.append(VQITQuantizerRegistry.build(cfg))
        for member in built:
            self._check_member(member)
        return nn.ModuleList(built)

    def _check_member(self, member) -> None:
        from .callbacks import BaseCallback, CVQVAECallback, NormalizeCallback
        from .losses import CodebookLoss, CommitmentLoss, VQGANLoss
        owner, members, name = type(self).__name__, self._members, type(member).__name__
        if not isinstance(member, VectorQuantizer):
            raise ValueError(f'{owner}: the {members} must be VectorQuantizer modules, got {name}')
        if member.materialize_distance:
            raise ValueError(f'{owner}: materialize_distance (compatibility mode) is not supported')
        if self._rotation_on_node and member.rotation_trick:
            raise ValueError(f'{owner}: rotation_trick is not supported for residual levels (one straight-through '
                             f'estimator spans the whole depth); set rotation_trick=True on the {owner} node instead')
        for c in member._callbacks:
            cname = type(c).__name__
            if isinstance(c, NormalizeCallback):
                raise ValueError(f'{owner}: callback {cname} rewrites the tokens; normalised {members} are not supported')
            hooks = [h for h in ('before_decode', 'after_decode', 'before_loss', 'after_loss')
                     if getattr(type(c), h) is not getattr(BaseCallback, h)]
            if hooks:
                raise ValueError(f'{owner}: callback {cname} hooks {", ".join(hooks)}; callbacks that '
                                 'hook decode or loss are not supported')
            if not isinstance(c, CVQVAECallback):
                raise ValueError(f'{owner}: callback {cname} is not supported ({members} take no callback '
                                 'or CVQVAECallback)')
            if c._anchor.needs_distance:
                raise ValueError(f'{owner}: {type(c._anchor).__name__} of {cname} reads the [N, K] '
                                 'distance matrix (compatibility mode), which is not supported')
        for lname, loss in member._losses.items():
            if not isinstance(loss, (CodebookLoss, CommitmentLoss, VQGANLoss)):
                raise ValueError(f'{owner}: loss {lname!r} ({type(loss).__name__}) is not supported '
                                 '(CodebookLoss, CommitmentLoss and VQGANLoss are)')

    @property
    def quantizers(self) -> nn.ModuleList:
        return self._quantizers

    @property
    def codebook_size(self) -> int:
        """Codes per member."""
        return self._quantizers[0].codebook_size

    @property
    def embeddings(self) -> torch.Tensor:
        """[M, K, Dm] copy of the member codebooks."""
        return torch.stack([member.embedding.weight.detach() for member in self._quantizers]).clone()

    def _init_weights(self, config) -> bool:
        for member in self._quantizers:
            member.init_weights(Config(copy.deepcopy(dict(config))))
        return False

    def _weights(self) -> list:
        return [member._weight() for member in self._quantizers]

    def _want_norm(self) -> bool:
        return self._quantizers[0]._loss_terms()

    def _member_memos(self, memo: dict, count: int | None = None) -> list:
        """One fresh memo per member (the first `count` members when given)."""
        memo[self._members] = [dict() for _ in range(len(self._quantizers) if count is None else count)]
        return memo[self._members]

    def _check_input(self, x: torch.Tensor) -> torch.Tensor:
        return _check_tokens(x, self.embedding_dim)

    @torch.no_grad()
    def encode_compact(self, x: torch.Tensor, memo: dict) -> torch.Tensor:
        """Tokenise-only encode: [M, N'] uint16 (K <= 65 536) or int32 ids straight from the packed assignment keys (N' = N
        rounded up to 8; the first N columns are the ids); None when a member's training callback needs int64 indices
        (then `encode` is the way)."""
        if not all(member._callbacks.packed_keys_ok() for member in self._quantizers):
            return None
        return self._encode_compact(x, self._member_memos(memo))

    def _compact_out(self, N: int, device, count: int | None = None) -> torch.Tensor:
        # rows padded to 8 ids: every row starts 16-byte aligned, as vqb_compact_tokens reads and stores 16 bytes at a time
        return torch.empty((len(self._quantizers) if count is None else count, (N + 7) // 8 * 8),
                           dtype=torch.uint16 if self.codebook_size <= 65536 else torch.int32, device=device)

    def decode(self, quant: torch.Tensor, memo: dict):
        """quant [N, M] (or [..., M]; uint16 / int32 / int64) -> (z fp32 [..., embedding_dim], memo) in one launch (see
        `_decode_ids`).  A token with an id outside [0, codebook_size) in any member decodes to NaN."""
        if not quant.is_cuda:
            raise VQBError(f'{type(self).__name__} decodes CUDA tensors only; there is no CPU fallback')
        lead = tuple(quant.shape[:-1])
        z = self._decode_ids(quant.contiguous().view(-1, quant.shape[-1]), 1)
        get_memo(memo, 'decode')
        return z.view(*lead, self.embedding_dim), memo

    def forward(self, x: torch.Tensor, memo: dict):
        x = self._check_input(x)
        members = list(self._quantizers)
        memos = self._member_memos(memo)
        z, quant, mse = self._quantize(x, members, memos, memo)
        memo.update(x=x, quant=quant)
        loss_memo = get_memo(memo, 'loss')
        sums: dict = {}
        for m, (member, member_memo) in enumerate(zip(members, memos)):
            member_memo['decode'] = get_memo(member_memo, 'decode')
            member_loss = get_memo(member_memo, 'loss')
            for name, module in member._losses.items():
                value = module.from_mse4(mse[m])
                member_loss[name] = value
                sums[name] = value if m == 0 else sums[name] + value
        loss = None
        for name, total in sums.items():
            loss_memo[name] = total / len(members) if self._loss_mean else total
            loss = loss_memo[name] if loss is None else loss + loss_memo[name]
        if loss is None:
            loss = mse[0][0].new_zeros([])
        return z, loss, memo


@VQITQuantizerRegistry.register_()
class ResidualVectorQuantizer(_ComposedQuantizer):
    """Residual quantization (RQ-VAE): L codebooks code every token in turn, level l quantizing what the earlier levels
    left over.  Levels are ordinary VectorQuantizer / VQGANQuantizer modules built from ONE config node (`quantizer`),
    stored as `_quantizers.{l}`; level l runs its own `encode` (before_encode -> assignment -> after_encode, codebook
    update included) on its input r_{l-1}:

        r_0 = x                       (fp32 view of the tokens; x is fp32 or bf16)
        q_l = level_l.encode(r_{l-1});  e_l = W_l[q_l]   (the codebook after this step's update)
        zhat_l = e_l (l = 1) or zhat_{l-1} + e_l;  r_l = r_{l-1} - e_l        (level order, fp32, no FMA)
        z = x + (zhat_L - x)          (one straight-through estimator over the whole depth: the gradient goes to x)
        loss = sum_l sum_name loss_{l,name}(e_l, r_{l-1}),  r_{l-1} = x - sum_{j<l} sg(e_j)

    so level l's CodebookLoss trains W_l against sg(r_{l-1}) and its CommitmentLoss reaches x through r_{l-1}.  With
    L = 1 this is VectorQuantizer.forward bit for bit.  memo: 'x' (the tokens), 'quant' (int64 [N, L]), 'levels'
    (level l's own memo: x = r_{l-1}, encode, decode, loss), 'loss' (per loss name, the sum over the levels).

    rotation_trick: that one estimator follows the rotation trick from x to zhat_L (Fifty et al., arXiv:2410.06424;
    DESIGN.md §4.9): x receives lambda R^T g instead of g, plus the levels' commitment terms as before.  z, the losses,
    the indices, the codebook updates and the codebook gradients are unchanged; with L = 1 the gradient is that of a
    rotated VectorQuantizer bit for bit.  The key belongs to this node; in the level config it is rejected.

    quantizer_dropout = p in [0, 1] (SoundStream, EnCodec, DAC; DESIGN.md §4.10): in training, each forward draws a
    depth d per sample on the device (a sample is an image under `tokenizer.quantize`, a token for [N, D] input): the
    first floor(S * p) of the S samples get d uniform in {1, ..., L}, the others d = L.  A sample is then coded by its
    first d levels only: z = x + (zhat_d - x), and level l's loss terms and gradients take only the tokens with l < d
    (the loss keeps its 1 / (N * D) scale).  Every level still encodes every token, so the indices, the callbacks'
    codebook updates and their statistics are those of the same step without dropout.  memo['depth'] holds the int32
    depths of the step.  With p = 0 or in eval mode the step is the one without dropout.

    encode / encode_compact(..., num_quantizers=n) run only the first n levels (truncated codes [N, n]).

    Accepted and rejected level configurations: see `_ComposedQuantizer`, with 1 <= L <= 16 and mse.norm on or off;
    rotation_trick=True and quantizer_dropout in the level config are rejected too."""

    _members = 'levels'
    _rotation_on_node = True

    def __init__(self, *args, num_quantizers: int, quantizer: Mapping, rotation_trick: bool = False,
                 quantizer_dropout: float = 0.0, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        name = type(self).__name__
        if isinstance(quantizer_dropout, bool) or not isinstance(quantizer_dropout, (int, float)) \
                or not 0.0 <= quantizer_dropout <= 1.0:
            raise ValueError(f'{name}: quantizer_dropout={quantizer_dropout!r} must be a float in [0, 1]')
        if 'quantizer_dropout' in quantizer:
            raise ValueError(f'{name}: quantizer_dropout is not a level key; set it on the {name} node')
        self.rotation_trick = bool(rotation_trick)
        self.quantizer_dropout = float(quantizer_dropout)
        self._quantizers = self._build_members(quantizer, num_quantizers, 'num_quantizers')

    @property
    def num_quantizers(self) -> int:
        return len(self._quantizers)

    @property
    def embedding_dim(self) -> int:
        return self._quantizers[0].embedding_dim

    def num_levels(self, num_quantizers: int | None = None) -> int:
        """The depth n of truncated codes: `num_quantizers` checked against [1, L], or L when None."""
        L = self.num_quantizers
        if num_quantizers is None:
            return L
        if isinstance(num_quantizers, bool) or not isinstance(num_quantizers, int) or not 1 <= num_quantizers <= L:
            raise ValueError(f'{type(self).__name__}: num_quantizers={num_quantizers!r} is outside [1, {L}]')
        return num_quantizers

    @torch.no_grad()
    def encode(self, x: torch.Tensor, memo: dict, *, num_quantizers: int | None = None):
        """-> (x, quant int64 [N, n], memo) with n = num_quantizers (L when None): the first n levels run as in forward
        (callbacks and codebook updates included); the levels past n do not run at all."""
        n = self.num_levels(num_quantizers)
        x = self._check_input(x)
        quant = torch.empty((x.shape[0], n), dtype=torch.int64, device=x.device)
        Fq.residual_levels(list(self._quantizers)[:n], x, self._member_memos(memo, n), self._want_norm(), quant_out=quant)
        return x, quant, memo

    @torch.no_grad()
    def encode_compact(self, x: torch.Tensor, memo: dict, *, num_quantizers: int | None = None) -> torch.Tensor:
        """`_ComposedQuantizer.encode_compact` over the first n = num_quantizers levels (all L when None): [n, N']."""
        n = self.num_levels(num_quantizers)
        if not all(level._callbacks.packed_keys_ok() for level in list(self._quantizers)[:n]):
            return None
        return self._encode_compact(x, self._member_memos(memo, n))

    def _encode_compact(self, x: torch.Tensor, memos: list) -> torch.Tensor:
        """The compact ids of the first len(memos) levels."""
        x = self._check_input(x)
        out = self._compact_out(x.shape[0], x.device, len(memos))
        Fq.residual_levels(list(self._quantizers)[:len(memos)], x, memos, self._want_norm(),
                           compact_out=out[:, :x.shape[0]])
        return out

    def _decode_ids(self, ids: torch.Tensor, hw: int, dtype: torch.dtype = torch.float32, bad_count=None,
                    num_quantizers: int | None = None):
        """ids [b*h*w, n] -> sum_{l<n} W_l[id_l] in level order, [b, D, h, w] of `dtype`; n = num_quantizers (L when
        None)."""
        return ops.decode_residual_tokens(self._weights()[:self.num_levels(num_quantizers)], ids, hw, dtype, bad_count)

    def draw_depths(self, samples: int, device) -> torch.Tensor:
        """The depths of one dropout step, int32 [samples], drawn on `device` with torch's CUDA generator (no host
        synchronisation; capturable in a CUDA graph): the first floor(samples * p) uniform in {1, ..., L}, the rest L."""
        L = self.num_quantizers
        depth = torch.full((samples,), L, dtype=torch.int32, device=device)
        truncated = int(samples * self.quantizer_dropout)
        if truncated:
            depth[:truncated].random_(1, L + 1)
        return depth

    def _quantize(self, x: torch.Tensor, levels: list, memos: list, memo: dict):
        nchw = memo.pop('_nchw', None)     # tokenizer.quantize: x is the token-major copy of these [b, c, h, w] latents
        dropout = {}        # without dropout: today's call
        if self.training and self.quantizer_dropout > 0:
            dropout['depth'] = memo['depth'] = self.draw_depths(x.shape[0] if nchw is None else nchw.shape[0], x.device)
        return Fq.residual_quantize(levels, x, memos, self._want_norm(), nchw=nchw, rotate=self.rotation_trick,
                                    **dropout)

@VQITQuantizerRegistry.register_()
class GroupedVectorQuantizer(_ComposedQuantizer):
    """Grouped (product) quantization: the D channels of a token are split into G groups of Dg = D / G channels and
    group g is quantized against its own codebook of K codes, so a token gets G ids (a joint code space of K^G).  Groups
    are ordinary VectorQuantizer / VQGANQuantizer modules with embedding_dim = Dg, built from ONE config node
    (`quantizer`) and stored as `_quantizers.{g}`; group g sees the column slice x_g = x[:, g*Dg:(g+1)*Dg] and behaves
    exactly like its own VectorQuantizer on x_g.contiguous():

        q_g = group_g.encode(x_g);  e_g = W_g[q_g]     (its callbacks run, CVQ-VAE update included: W_g after the step)
        z[:, g*Dg:(g+1)*Dg] = x_g + (e_g - x_g)        (fp32 subtract, then add; no FMA)
        loss[name] = (sum_g loss_{g,name}(e_g, x_g)) / G  (fp32 adds in group order, one division)

    The unnormalised MSE terms thus average over all N * D elements, so a config's loss weights keep their meaning when a
    width-D quantizer is split into groups; with mse.norm=True each group normalises its own sub-vector.  With G = 1 this
    is VectorQuantizer.forward bit for bit.  forward / encode take tokens [N, D] or latents [b, D, h, w] (z then comes
    back NCHW).  memo: 'x' (the input as given), 'quant' (int64 [N, G]), 'groups' (group g's own memo: x = its token
    slice, encode, decode, loss), 'loss' (per loss name, the group mean).

    Accepted and rejected configurations are those of ResidualVectorQuantizer (see `_ComposedQuantizer`), with
    1 <= num_groups <= 16, except that the group config may set rotation_trick=True: every group then passes its
    encoder gradient through the rotation trick (DESIGN.md §4.9)."""

    _members = 'groups'
    _loss_mean = True

    def __init__(self, *args, num_groups: int, quantizer: Mapping, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self._quantizers = self._build_members(quantizer, num_groups, 'num_groups')

    @property
    def num_groups(self) -> int:
        return len(self._quantizers)

    @property
    def group_dim(self) -> int:
        return self._quantizers[0].embedding_dim

    @property
    def embedding_dim(self) -> int:
        return self.num_groups * self.group_dim

    def _check_input(self, x: torch.Tensor) -> torch.Tensor:
        """Tokens [N, D] or latents [b, D, h, w], fp32 / bf16 on the GPU."""
        if x.dim() != 4:
            return _check_tokens(x, self.embedding_dim)
        if not x.is_cuda:
            raise VQBError('vector_quantization_b200 quantizers run on CUDA (sm_100a) tensors only; no CPU fallback')
        if x.shape[1] != self.embedding_dim:
            raise ValueError(f'expected latents of shape [b, {self.embedding_dim}, h, w], got {tuple(x.shape)}')
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise TypeError(f'latents must be float32 or bfloat16, got {x.dtype}')
        return x.contiguous()

    def _split(self, x: torch.Tensor) -> torch.Tensor:
        x = self._check_input(x).detach()
        if self.num_groups == 1 and x.dim() == 2:
            return x.view(1, *x.shape)
        return ops.split_groups(x, self.num_groups)

    @torch.no_grad()
    def encode(self, x: torch.Tensor, memo: dict):
        """-> (x, quant int64 [N, G], memo); every group's callbacks run as in forward (codebook updates included)."""
        xs = self._split(x)
        G, N, _ = xs.shape
        memos = self._member_memos(memo)
        keys, _ = Fq.group_encode(list(self._quantizers), xs, memos)
        idx = ops.unpack_keys(keys.view(-1))
        quant = idx.view(N, G) if G == 1 else ops.transpose_last2(idx.view(1, G, N)).view(N, G)
        for g, group_memo in enumerate(memos):
            group_memo.update(x=xs[g], quant=quant[:, g])
        return x, quant, memo

    def _encode_compact(self, x: torch.Tensor, memos: list) -> torch.Tensor:
        xs = self._split(x)
        G, N, _ = xs.shape
        out = self._compact_out(N, xs.device)
        keys = torch.empty(out.shape, dtype=torch.int64, device=xs.device)[:, :N]
        Fq.group_encode(list(self._quantizers), xs, memos, keys=keys)
        for g in range(G):
            ops.compact_tokens(keys[g], self.codebook_size, out=out[g, :N])
        return out

    def _decode_ids(self, ids: torch.Tensor, hw: int, dtype: torch.dtype = torch.float32, bad_count=None):
        """ids [b*h*w, G] -> channels [g*Dg, (g+1)*Dg) = W_g[id_g], [b, D, h, w] of `dtype`."""
        return ops.decode_group_tokens(self._weights(), ids, hw, dtype, bad_count)

    def _quantize(self, x: torch.Tensor, groups: list, memos: list, memo: dict):
        return Fq.grouped_quantize(groups, x, memos, self._want_norm(), rotate=groups[0].rotation_trick)
