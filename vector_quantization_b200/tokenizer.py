"""The callers and data formats either side of the quantizer (SURVEY.md §8f items 1 and 3).

Reference: `BaseModel.quantize` / `encode_to_quant` (vq/tasks/image_tokenization/models/base.py:116-146) hand
the quantizer NCHW encoder features; `decode_from_quant` (vq/tasks/image_reconstruction/models.py:97-108) turns
token grids back into NCHW decoder input; `TokenizeCallback` (runners/callbacks.py:29-53) and
`tools/tokenize_llamagen.py:93-103` write the resulting token grids to disk.  The functions here take the
quantizer (not a whole tokenizer model: encoders/decoders are out of scope) and reproduce those contracts —
memo keys, shapes, dtypes, file formats — with the layout changes done by the transpose kernel of the C-ABI
and a tokenise-only path that never builds the int64 index tensor unless asked for.
"""
from __future__ import annotations

import pathlib
from typing import Any, Sequence

import torch

from . import functional as Fq
from . import ops
from ._lib import VQBError
from .quantizers import (FiniteScalarQuantizer, GroupedVectorQuantizer, ResidualVectorQuantizer, VectorQuantizer,
                         _ComposedQuantizer, get_memo)

__all__ = ['quantize', 'encode_to_quant', 'decode_from_quant', 'save_tokens', 'load_tokens', 'save_llamagen_codes', 'TokenStreamWriter']


def quantize(quantizer, x: torch.Tensor, memo: dict):
    """`BaseModel.quantize` (base.py:116-129): x [b, c, h, w] -> (z [b, c, h, w] contiguous, q_loss, memo) with
    memo['quantizer'] = the quantizer's memo (+ 'x_shape').  A ResidualVectorQuantizer always takes the fused layout: its
    last residual step writes z NCHW.  A GroupedVectorQuantizer takes the latents themselves: one split launch makes
    its group-major tokens and the group gather kernel writes z NCHW."""
    quantizer_memo = get_memo(memo, 'quantizer')
    quantizer_memo['x_shape'] = (b, c, h, w) = tuple(x.shape)
    if isinstance(quantizer, GroupedVectorQuantizer) and x.is_cuda:
        z, q_loss, memo['quantizer'] = quantizer(x, quantizer_memo)
        return z, q_loss, memo
    fusable = isinstance(quantizer, ResidualVectorQuantizer) or (isinstance(quantizer, VectorQuantizer)
                                                                  and quantizer.can_fuse_nchw())
    if fusable and x.is_cuda:
        # Layout fusion: ONE transposed copy of the latents feeds the assignment, the callbacks and the kernels' token
        # reads; z is written NCHW by the gather kernel, and the backward reads the NCHW upstream gradient and writes
        # the NCHW token gradient directly — no transpose after the quantizer, none in the backward.
        x = x.contiguous()
        rows = ops.transpose_last2(x.detach().view(b, c, h * w)).view(b * h * w, c)
        quantizer_memo['_nchw'] = x
        z, q_loss, memo['quantizer'] = quantizer(rows, quantizer_memo)
        return z, q_loss, memo
    rows = Fq.nchw_to_rows(x)
    z, q_loss, memo['quantizer'] = quantizer(rows, quantizer_memo)
    return Fq.rows_to_nchw(z, b, c, h, w), q_loss, memo


def _truncation(quantizer, num_quantizers: int | None) -> dict:
    """The keyword that truncates a ResidualVectorQuantizer's codes to its first `num_quantizers` levels ({} for None)."""
    if num_quantizers is None:
        return {}
    if not isinstance(quantizer, ResidualVectorQuantizer):
        raise ValueError(f'num_quantizers truncates ResidualVectorQuantizer codes; {type(quantizer).__name__} has none')
    return dict(num_quantizers=quantizer.num_levels(num_quantizers))


@torch.no_grad()
def encode_to_quant(quantizer, x: torch.Tensor, memo: dict, *, compact: bool = False,
                    num_quantizers: int | None = None):
    """`BaseModel.encode_to_quant` after the encoder (base.py:131-146): x [b, c, h, w] -> (quant [b, h, w], memo);
    memo['quantizer'] gets 'x_shape', 'x' (token-major, after the callbacks) and 'quant' ([b*h*w] int64).
    compact=True is the tokenise-only variant: token ids come back as uint16 (K <= 65 536) or int32 straight
    from the packed assignment keys and memo['quantizer']['quant'] holds that compact tensor.
    A ResidualVectorQuantizer gives quant [b, h, w, L] (a token's L ids contiguous); with compact=True each level's
    ids are compacted into a row of an [L, N] buffer and one transpose (none when L = 1) makes the [N, L] layout.  A
    GroupedVectorQuantizer gives quant [b, h, w, G] the same way (its encode reads the latents through one split
    launch; memo['quantizer']['x'] is then the latents).
    num_quantizers=n (ResidualVectorQuantizer only, 1 <= n <= L): truncated codes [b, h, w, n] from the first n levels;
    the levels past n do not run."""
    truncate = _truncation(quantizer, num_quantizers)
    quantizer_memo = get_memo(memo, 'quantizer')
    quantizer_memo['x_shape'] = (b, _, h, w) = tuple(x.shape)
    if isinstance(quantizer, _ComposedQuantizer):
        M = truncate.get('num_quantizers', len(quantizer.quantizers))
        # a GroupedVectorQuantizer reads the latents through one split launch; residual levels read token-major rows
        x = x if isinstance(quantizer, GroupedVectorQuantizer) else Fq.nchw_to_rows(x)
        by_member = quantizer.encode_compact(x, quantizer_memo, **truncate) if compact else None
        if by_member is not None:
            quant = by_member.view(-1, 1) if M == 1 else ops.transpose_last2(by_member.view(1, M, -1)).view(-1, M)
            quant = quant[:b * h * w]
        else:
            x, quant, _ = quantizer.encode(x, quantizer_memo, **truncate)
            if compact:
                quant = quant.to(torch.int32)
        quantizer_memo.update(x=x, quant=quant)
        return quant.view(b, h, w, M), memo
    rows = Fq.nchw_to_rows(x)
    # keep the packed keys (no int64 unpack launch) unless a training callback consumes the indices in after_encode
    lazy = compact and isinstance(quantizer, VectorQuantizer) and quantizer._callbacks.packed_keys_ok()
    if lazy:
        quantizer_memo['_lazy_unpack'] = True
    rows, quant, memo['quantizer'] = quantizer.encode(rows, quantizer_memo)
    quantizer_memo = memo['quantizer']
    if lazy:
        quant = ops.compact_tokens(quant, quantizer.codebook_size)
    elif compact and quant.dtype == torch.int64:
        quant = quant.to(torch.int32)
    quantizer_memo.update(x=rows, quant=quant)
    return quant.view(b, h, w), memo


def decode_from_quant(quantizer, quant: torch.Tensor, memo: dict, *, dtype: torch.dtype = torch.float32,
                      check: bool = True, num_quantizers: int | None = None):
    """`decode_from_quant` before the decoder (vq/tasks/image_reconstruction/models.py:97-108): token ids
    quant [b, h, w] -> (z [b, c, h, w] contiguous of `dtype`, memo) with memo['quantizer'] = the quantizer's memo as
    `quantizer.decode` leaves it.  quant is uint16, int32 or int64 on the GPU: what `encode_to_quant` (compact or not)
    and FSQ produce, or a `load_tokens` dump moved to the device.  The codebook is used as stored (no before_encode).
    A ResidualVectorQuantizer takes quant [b, h, w, L] and decodes sum_l W_l[id_l] in one launch; a
    GroupedVectorQuantizer takes quant [b, h, w, G] and decodes channel group g from W_g[id_g] in one launch.
    num_quantizers=n (ResidualVectorQuantizer only, 1 <= n <= L): truncated codes [b, h, w, n], decoded as the sum of
    the first n levels, sum_{l<n} W_l[id_l], in the same one launch.

    A VectorQuantizer or FiniteScalarQuantizer without before_decode / after_decode hooks decodes in ONE launch that
    reads the ids as they are and writes NCHW `dtype` directly.  Hooks, or a codebook that requires grad with grad
    enabled, take `quantizer.decode` (hooks honoured, differentiable gather) + the transpose + a cast instead; on
    valid ids both give the same values.

    An id outside [0, codebook_size) is an error: with check=True (one 4-byte device-to-host read) it raises
    IndexError with the number of such tokens.  check=False does not synchronise (safe inside a CUDA graph capture)
    and, on the one-launch path, decodes such tokens to NaN in every channel."""
    truncate = _truncation(quantizer, num_quantizers)
    composed = isinstance(quantizer, _ComposedQuantizer)
    M = truncate.get('num_quantizers', len(quantizer.quantizers) if composed else 1)
    if composed and (quant.dim() != 4 or quant.shape[-1] != M):
        raise ValueError(f'expected {type(quantizer).__name__} token ids of shape '
                         f'[b, h, w, {M}], got {tuple(quant.shape)}')
    if not composed and quant.dim() != 3:
        raise ValueError(f'expected token ids of shape [b, h, w], got {tuple(quant.shape)}')
    if not quant.is_cuda:
        raise VQBError('vector_quantization_b200 decodes CUDA (sm_100a) token ids only; there is no CPU fallback')
    if dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f'dtype must be float32 or bfloat16, got {dtype}')
    b, h, w = quant.shape[:3]
    quantizer_memo = get_memo(memo, 'quantizer')
    if composed:
        bad = torch.zeros(1, dtype=torch.int32, device=quant.device) if check else None
        z = quantizer._decode_ids(quant.contiguous(), h * w, dtype, bad, **truncate)
        get_memo(quantizer_memo, 'decode')
        if check:
            _raise_bad_ids(int(bad.item()), quantizer.codebook_size)
        return z, memo
    fsq = isinstance(quantizer, FiniteScalarQuantizer)
    hooked = any(quantizer._callbacks.overrides(hook) for hook in ('before_decode', 'after_decode'))
    if isinstance(quantizer, VectorQuantizer):
        W = quantizer._weight()
        fused = not hooked and not (torch.is_grad_enabled() and W.requires_grad)
    else:
        # FiniteScalarQuantizer.decode returns the encode memo's z when there is one: leave that case to it
        fused = fsq and not hooked and 'z' not in quantizer_memo.get('encode', {})
    quant = quant.contiguous()
    if fused:
        bad = torch.zeros(1, dtype=torch.int32, device=quant.device) if check else None
        if fsq:
            get_memo(quantizer_memo, 'encode')
            z = ops.fsq_decode_tokens(quant, quantizer._params, h * w, dtype, bad)
        else:
            z = ops.decode_tokens(W.detach(), quant, h * w, dtype, bad)
        get_memo(quantizer_memo, 'decode')
        if check:
            _raise_bad_ids(int(bad.item()), quantizer.codebook_size)
        return z, memo
    wide = quant.to(torch.int32) if quant.dtype == torch.uint16 else quant     # uint16 has no CUDA comparisons
    wide = wide.to(torch.int32 if fsq else torch.int64)
    if check:
        K = quantizer.codebook_size
        _raise_bad_ids(int(((wide < 0) | (wide >= K)).sum()), K)
    z, memo['quantizer'] = quantizer.decode(wide, quantizer_memo)
    z = Fq.rows_to_nchw(z, b, z.shape[-1], h, w)
    return (z if z.dtype == dtype else z.to(dtype)), memo


def _token_grid(quant: torch.Tensor, x_shape: Sequence[int]) -> tuple:
    """(b, h, w) for one id per token; (b, h, w, L) for residual or grouped ids ([b, h, w, L], or L ids per token)."""
    b, _, h, w = x_shape
    depth = quant.numel() // max(b * h * w, 1)
    return (b, h, w, depth) if (quant.dim() == 4 or depth != 1) else (b, h, w)


def _raise_bad_ids(count: int, codebook_size: int) -> None:
    if count:
        raise IndexError(f'{count} token id(s) outside [0, {codebook_size}): not in the codebook')


def save_tokens(path: str | pathlib.Path, id_: Sequence[Any], category: torch.Tensor, quant: torch.Tensor,
                x_shape: Sequence[int]) -> None:
    """`TokenizeCallback.after_run_iter` (runners/callbacks.py:40-53): torch.save of the `Tokens` dict
    {id_, category, tokens [b, h, w]}.  Compact ids are widened to int64 so that reference readers see the
    dtype they expect; pass an int64 tensor to skip the conversion.  Residual and grouped ids keep their trailing
    axis: tokens [b, h, w, L]."""
    tokens = quant.reshape(_token_grid(quant, x_shape))
    if tokens.dtype != torch.int64:
        tokens = tokens.to(torch.int32).to(torch.int64) if tokens.dtype == torch.uint16 else tokens.to(torch.int64)
    torch.save(dict(id_=id_, category=category, tokens=tokens.cpu()), str(path))


class TokenStreamWriter:
    """Streaming variant of `TokenizeCallback` (runners/callbacks.py:29-53): one `{iter}_{rank}.pth` `Tokens` file per
    iteration under `token_dir`, written WITHOUT stalling the GPU.  `write` enqueues an asynchronous device-to-host
    copy of the token ids into a pinned staging buffer on a side stream and returns; a background thread waits for
    the copy (CUDA event) and does the `torch.save`.  `depth` staging buffers bound the memory; `close()` (or
    leaving the `with` block) drains the queue.  The files are exactly what `save_tokens` writes."""

    def __init__(self, token_dir: str | pathlib.Path, rank: int = 0, depth: int = 4) -> None:
        import queue
        import threading
        self.token_dir = pathlib.Path(token_dir)
        self.token_dir.mkdir(parents=True, exist_ok=True)       # TokenizeCallback.bind
        self.rank = rank
        self._free: 'queue.Queue' = queue.Queue()
        for _ in range(depth):
            self._free.put(None)                                # staging slots, allocated lazily at the first size seen
        self._jobs: 'queue.Queue' = queue.Queue()
        self._stream = None
        self._error = None
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def _run(self) -> None:
        while True:
            job = self._jobs.get()
            if job is None:
                return
            path, id_, category, host, event, shape = job
            try:
                if event is not None:
                    event.synchronize()
                tokens = host.reshape(shape)
                if tokens.dtype != torch.int64:
                    tokens = tokens.to(torch.int32).to(torch.int64) if tokens.dtype == torch.uint16 else tokens.to(torch.int64)
                torch.save(dict(id_=id_, category=category, tokens=tokens.clone()), str(path))
            except Exception as exc:  # noqa: BLE001 - surfaced by the next write()/close()
                self._error = exc
            finally:
                self._free.put(host)

    def write(self, iter_: int, id_: Sequence[Any], category: torch.Tensor, quant: torch.Tensor,
              x_shape: Sequence[int]) -> pathlib.Path:
        if self._error is not None:
            raise self._error
        host = self._free.get()                                 # blocks only when `depth` writes are in flight
        flat = quant.reshape(-1)
        if host is None or host.numel() != flat.numel() or host.dtype != flat.dtype:
            host = torch.empty(flat.numel(), dtype=flat.dtype).pin_memory() if flat.is_cuda else torch.empty_like(flat)
        event = None
        if flat.is_cuda:
            if self._stream is None:
                self._stream = torch.cuda.Stream(device=flat.device)
            self._stream.wait_stream(torch.cuda.current_stream(flat.device))
            with torch.cuda.stream(self._stream):
                host.copy_(flat, non_blocking=True)
                flat.record_stream(self._stream)
                event = torch.cuda.Event()
                event.record(self._stream)
        else:
            host.copy_(flat)
        path = self.token_dir / f'{iter_}_{self.rank}.pth'
        self._jobs.put((path, list(id_), category.detach().cpu(), host, event, _token_grid(quant, x_shape)))
        return path

    def close(self) -> None:
        self._jobs.put(None)
        self._thread.join()
        if self._error is not None:
            raise self._error

    def __enter__(self) -> 'TokenStreamWriter':
        return self

    def __exit__(self, *exc) -> None:
        self.close()


def load_tokens(path: str | pathlib.Path) -> dict:
    return torch.load(str(path), weights_only=False)


def save_llamagen_codes(code_path: str | pathlib.Path, label_path: str | pathlib.Path, quant: torch.Tensor,
                        category: torch.Tensor) -> None:
    """tools/tokenize_llamagen.py:93-103: codes as .npy of shape (1, 10, -1) (ten-crop augmentations x tokens),
    labels as a separate .npy."""
    import numpy as np
    q = quant.reshape(1, 10, -1)
    if q.dtype == torch.uint16:
        q = q.to(torch.int32)
    np.save(str(code_path), q.to(torch.int64).cpu().numpy())
    np.save(str(label_path), category.cpu().numpy())
