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
from .callbacks import ComposedCallback
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
    kernel launches: pack+assign (tcgen05, no N x K matrix), [stats/update], fused gather+STE+loss."""

    def __init__(self, *args, embedding: nn.Embedding, distance: BaseDistance, precision: str = Fq.DEFAULT_PRECISION,
                 materialize_distance: bool = False, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        if precision not in Fq.PRECISION_PLANES:
            raise ValueError(f'precision must be one of {sorted(Fq.PRECISION_PLANES)}')
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
                                                  normalize_x=normalize_x, codebook_ref=ref, nchw=nchw)
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


def _build_members(owner: BaseQuantizer, quantizer: Mapping, count, count_name: str, members: str) -> list:
    """The member quantizers of a composed quantizer (ResidualVectorQuantizer levels, GroupedVectorQuantizer groups):
    `count` copies of the `quantizer` node, each an ordinary VectorQuantizer / VQGANQuantizer.  Accepted: L2 or Cosine
    distance, no callback or CVQVAECallback (NearestAnchor / CachedAnchor), CodebookLoss / CommitmentLoss / VQGANLoss.
    Everything else raises a ValueError naming the offending item: callbacks that rewrite the tokens, callbacks that
    hook decode or loss, compatibility mode, a count outside [1, 16], members that are not VectorQuantizer modules
    (FSQ, or a composed quantizer: no nesting), and callbacks or losses on the composed node itself."""
    name = type(owner).__name__
    if isinstance(count, bool) or not isinstance(count, int) or not 1 <= count <= MAX_LEVELS:
        raise ValueError(f'{name}: {count_name}={count!r} is outside [1, {MAX_LEVELS}]')
    if list(owner._callbacks) or len(owner._losses):
        raise ValueError(f'{name}: callbacks and losses belong to the {members[:-1]} config (`quantizer`), '
                         f'not to the {name} node itself')
    cls = VQITQuantizerRegistry.lookup(quantizer['type']) if isinstance(quantizer.get('type'), str) else None
    if isinstance(cls, type) and not issubclass(cls, VectorQuantizer):
        raise ValueError(f'{name}: the {members} must be VectorQuantizer modules, got {cls.__name__}')
    built = []
    for _ in range(count):
        cfg = Config(copy.deepcopy(dict(quantizer)))
        cfg['init_weights'] = None       # applied per member by init_weights (after the train / eval mode is set)
        built.append(VQITQuantizerRegistry.build(cfg))
    for member in built:
        _check_member(name, member, members)
    return built


def _check_member(owner: str, member, members: str) -> None:
    from .callbacks import BaseCallback, CVQVAECallback, NormalizeCallback
    from .losses import CodebookLoss, CommitmentLoss, VQGANLoss
    name = type(member).__name__
    if not isinstance(member, VectorQuantizer):
        raise ValueError(f'{owner}: the {members} must be VectorQuantizer modules, got {name}')
    if member.materialize_distance:
        raise ValueError(f'{owner}: materialize_distance (compatibility mode) is not supported')
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


@VQITQuantizerRegistry.register_()
class ResidualVectorQuantizer(BaseQuantizer):
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

    Accepted: 1 <= L <= 16, L2 or Cosine distance, no callback or CVQVAECallback (NearestAnchor / CachedAnchor),
    CodebookLoss / CommitmentLoss / VQGANLoss with or without mse.norm.  Rejected with a ValueError: callbacks that
    rewrite the tokens (NormalizeCallback and its subclasses), callbacks that hook decode or loss, and compatibility
    mode (EntropyLoss, MultinomialAnchor, materialize_distance).  `init_weights` is applied to every level."""

    MAX_LEVELS = 16

    def __init__(self, *args, num_quantizers: int, quantizer: Mapping, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self._quantizers = nn.ModuleList(_build_members(self, quantizer, num_quantizers, 'num_quantizers', 'levels'))

    @property
    def quantizers(self) -> nn.ModuleList:
        return self._quantizers

    @property
    def num_quantizers(self) -> int:
        return len(self._quantizers)

    @property
    def embedding_dim(self) -> int:
        return self._quantizers[0].embedding_dim

    @property
    def codebook_size(self) -> int:
        """Codes per level."""
        return self._quantizers[0].codebook_size

    @property
    def embeddings(self) -> torch.Tensor:
        """[L, K, D] copy of the level codebooks."""
        return torch.stack([level.embedding.weight.detach() for level in self._quantizers]).clone()

    def _init_weights(self, config) -> bool:
        for level in self._quantizers:
            level.init_weights(Config(copy.deepcopy(dict(config))))
        return False

    def _weights(self) -> list:
        return [level._weight() for level in self._quantizers]

    def _want_norm(self) -> bool:
        return self._quantizers[0]._loss_terms()

    def _level_memos(self, memo: dict) -> list:
        memo['levels'] = [dict() for _ in self._quantizers]
        return memo['levels']

    @torch.no_grad()
    def encode(self, x: torch.Tensor, memo: dict):
        """-> (x, quant int64 [N, L], memo); every level's callbacks run as in forward (codebook updates included)."""
        x = _check_tokens(x, self.embedding_dim)
        quant = torch.empty((x.shape[0], self.num_quantizers), dtype=torch.int64, device=x.device)
        Fq.residual_levels(list(self._quantizers), x, self._level_memos(memo), self._want_norm(), quant_out=quant)
        return x, quant, memo

    @torch.no_grad()
    def encode_compact(self, x: torch.Tensor, memo: dict) -> torch.Tensor:
        """Tokenise-only encode: [L, N'] uint16 (K <= 65 536) or int32 ids straight from the packed assignment keys (N' = N
        rounded up to 8; the first N columns are the ids); None when a level's training callback needs int64 indices
        (then `encode` is the way)."""
        if not all(level._callbacks.packed_keys_ok() for level in self._quantizers):
            return None
        x = _check_tokens(x, self.embedding_dim)
        N = x.shape[0]
        # rows padded to 8 ids: every row starts 16-byte aligned, as vqb_compact_tokens stores 16 bytes at a time
        out = torch.empty((self.num_quantizers, (N + 7) // 8 * 8),
                          dtype=torch.uint16 if self.codebook_size <= 65536 else torch.int32, device=x.device)
        Fq.residual_levels(list(self._quantizers), x, self._level_memos(memo), self._want_norm(), compact_out=out[:, :N])
        return out

    def decode(self, quant: torch.Tensor, memo: dict):
        """quant [N, L] (or [..., L]; uint16 / int32 / int64) -> (zhat fp32 [..., D], memo): sum_l W_l[q_l] in level order,
        one launch.  A token with an id outside [0, codebook_size) at any level decodes to NaN."""
        if not quant.is_cuda:
            raise VQBError('ResidualVectorQuantizer decodes CUDA tensors only; there is no CPU fallback')
        lead = tuple(quant.shape[:-1])
        flat = quant.contiguous().view(-1, quant.shape[-1])
        z = ops.decode_residual_tokens([W.detach() for W in self._weights()], flat, 1)
        get_memo(memo, 'decode')
        return z.view(*lead, self.embedding_dim), memo

    def forward(self, x: torch.Tensor, memo: dict):
        x = _check_tokens(x, self.embedding_dim)
        nchw = memo.pop('_nchw', None)     # tokenizer.quantize: x is the token-major copy of these [b, c, h, w] latents
        levels = list(self._quantizers)
        memos = self._level_memos(memo)
        z, quant, mse = Fq.residual_quantize(levels, x, memos, self._want_norm(), nchw=nchw)
        memo.update(x=x, quant=quant)
        loss_memo = get_memo(memo, 'loss')
        loss = None
        for l, (level, level_memo) in enumerate(zip(levels, memos)):
            level_memo['decode'] = get_memo(level_memo, 'decode')
            level_loss = get_memo(level_memo, 'loss')
            for name, module in level._losses.items():
                value = module.from_mse4(mse[l])
                level_loss[name] = value
                loss_memo[name] = value if l == 0 else loss_memo[name] + value
        for name in levels[0]._losses:
            loss = loss_memo[name] if loss is None else loss + loss_memo[name]
        if loss is None:
            loss = mse[0][0].new_zeros([])
        return z, loss, memo


@VQITQuantizerRegistry.register_()
class GroupedVectorQuantizer(BaseQuantizer):
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

    Accepted and rejected configurations are those of ResidualVectorQuantizer (see `_build_members`), with
    1 <= num_groups <= 16.  `init_weights` is applied to every group."""

    def __init__(self, *args, num_groups: int, quantizer: Mapping, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self._quantizers = nn.ModuleList(_build_members(self, quantizer, num_groups, 'num_groups', 'groups'))

    @property
    def quantizers(self) -> nn.ModuleList:
        return self._quantizers

    @property
    def num_groups(self) -> int:
        return len(self._quantizers)

    @property
    def group_dim(self) -> int:
        return self._quantizers[0].embedding_dim

    @property
    def embedding_dim(self) -> int:
        return self.num_groups * self.group_dim

    @property
    def codebook_size(self) -> int:
        """Codes per group."""
        return self._quantizers[0].codebook_size

    @property
    def embeddings(self) -> torch.Tensor:
        """[G, K, Dg] copy of the group codebooks."""
        return torch.stack([group.embedding.weight.detach() for group in self._quantizers]).clone()

    def _init_weights(self, config) -> bool:
        for group in self._quantizers:
            group.init_weights(Config(copy.deepcopy(dict(config))))
        return False

    def _weights(self) -> list:
        return [group._weight() for group in self._quantizers]

    def _want_norm(self) -> bool:
        return self._quantizers[0]._loss_terms()

    def _group_memos(self, memo: dict) -> list:
        memo['groups'] = [dict() for _ in self._quantizers]
        return memo['groups']

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
        keys, _ = Fq.group_encode(list(self._quantizers), xs, self._group_memos(memo))
        idx = ops.unpack_keys(keys.view(-1))
        quant = idx.view(N, G) if G == 1 else ops.transpose_last2(idx.view(1, G, N)).view(N, G)
        for g, group_memo in enumerate(memo['groups']):
            group_memo.update(x=xs[g], quant=quant[:, g])
        return x, quant, memo

    @torch.no_grad()
    def encode_compact(self, x: torch.Tensor, memo: dict) -> torch.Tensor:
        """Tokenise-only encode: [G, N'] uint16 (K <= 65 536) or int32 ids straight from the packed assignment keys (N' = N
        rounded up to 8; the first N columns are the ids); None when a group's training callback needs int64 indices
        (then `encode` is the way)."""
        if not all(group._callbacks.packed_keys_ok() for group in self._quantizers):
            return None
        xs = self._split(x)
        G, N, _ = xs.shape
        # rows padded to 8: every row starts 16-byte aligned, as vqb_compact_tokens reads and stores 16 bytes at a time
        Np = (N + 7) // 8 * 8
        keys = torch.empty((G, Np), dtype=torch.int64, device=xs.device)[:, :N]
        out = torch.empty((G, Np), dtype=torch.uint16 if self.codebook_size <= 65536 else torch.int32, device=xs.device)
        Fq.group_encode(list(self._quantizers), xs, self._group_memos(memo), keys=keys)
        for g in range(G):
            ops.compact_tokens(keys[g], self.codebook_size, out=out[g, :N])
        return out

    def decode(self, quant: torch.Tensor, memo: dict):
        """quant [N, G] (or [..., G]; uint16 / int32 / int64) -> (z fp32 [..., D], memo): channels [g*Dg, (g+1)*Dg) =
        W_g[q_g], one launch.  A token with an id outside [0, codebook_size) in any group decodes to NaN."""
        if not quant.is_cuda:
            raise VQBError('GroupedVectorQuantizer decodes CUDA tensors only; there is no CPU fallback')
        lead = tuple(quant.shape[:-1])
        flat = quant.contiguous().view(-1, quant.shape[-1])
        z = ops.decode_group_tokens([W.detach() for W in self._weights()], flat, 1)
        get_memo(memo, 'decode')
        return z.view(*lead, self.embedding_dim), memo

    def forward(self, x: torch.Tensor, memo: dict):
        x = self._check_input(x)
        groups = list(self._quantizers)
        memos = self._group_memos(memo)
        z, quant, mse = Fq.grouped_quantize(groups, x, memos, self._want_norm())
        memo.update(x=x, quant=quant)
        loss_memo = get_memo(memo, 'loss')
        sums: dict = {}
        for g, (group, group_memo) in enumerate(zip(groups, memos)):
            group_memo['decode'] = get_memo(group_memo, 'decode')
            group_loss = get_memo(group_memo, 'loss')
            for name, module in group._losses.items():
                value = module.from_mse4(mse[g])
                group_loss[name] = value
                sums[name] = value if g == 0 else sums[name] + value
        loss = None
        for name, total in sums.items():
            loss_memo[name] = total / len(groups)
            loss = loss_memo[name] if loss is None else loss + loss_memo[name]
        if loss is None:
            loss = mse[0][0].new_zeros([])
        return z, loss, memo
