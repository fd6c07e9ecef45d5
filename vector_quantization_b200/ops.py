"""Tensor-level wrappers over the C-ABI (`include/vqb200.h`).

PyTorch is used only as the owner of device memory and of the current CUDA stream: every function
here passes raw device pointers + sizes + the stream handle to `libvqb200.so`.  All inputs must be
CUDA tensors; there is no CPU path.
"""
from __future__ import annotations

import ctypes
from ctypes import c_void_p
from dataclasses import dataclass

import torch

from . import _lib
from ._lib import (BACKEND_SIMT, BACKEND_TCGEN05, MAX_LEVELS, PLANES_F16, PLANES_F16X2, VQB_BF16, VQB_F32, FSQParams,
                   ResidualLevels, check)

__all__ = [
    'Operand', 'as_operand', 'pack_rows', 'fold_l2_side', 'can_fold_l2', 'assign', 'certify', 'cvq_needy_codes', 'gather_operand_rows', 'scatter_keys', 'row_inv_norm', 'new_keys', 'unpack_keys', 'keys_flip_sign', 'gather_ste_loss',
    'quantize_backward', 'l2norm_forward', 'l2norm_backward', 'scatter_stats', 'bincount_accumulate',
    'deterministic_enabled', 'segment_chunk', 'code_sort', 'segment_sum_rows',
    'kmeans_ema_update', 'gather_rows_by_key', 'cvq_update', 'embedding_gather', 'fsq_params', 'fsq_forward', 'fsq_backward',
    'fsq_decode', 'decode_tokens', 'fsq_decode_tokens', 'residual_step', 'residual_backward', 'decode_residual_tokens',
    'split_groups', 'group_gather_ste_loss', 'group_backward', 'decode_group_tokens',
    'transpose_last2', 'compact_tokens', 'distance_matrix', 'comm_kmeans_ema_update', 'comm_cvq_update',
    'comm_allreduce_min_keys', 'comm_allreduce_sum_f32', 'BACKEND_TCGEN05', 'BACKEND_SIMT',
]


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return VQB_F32
    if t.dtype == torch.bfloat16:
        return VQB_BF16
    raise TypeError(f'vector_quantization_b200 supports float32 and bfloat16 tensors, got {t.dtype}')


def _cuda(*ts: torch.Tensor | None) -> torch.device:
    """Checks that every tensor is a contiguous CUDA tensor of ONE device and returns that device."""
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.VQBError('vector_quantization_b200 runs on CUDA (sm_100a) tensors only; there is no CPU fallback')
        if not t.is_contiguous():
            raise ValueError('expected a contiguous tensor')
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise ValueError(f'all tensors of one call must live on the same device, got {dev} and {t.device}')
    return dev


def _p(t: torch.Tensor | None):
    """Device pointer as a plain int (ctypes converts ints and None for `c_void_p` parameters; no wrapper object)."""
    return t.data_ptr() if t is not None else None


class _StreamArg:
    """Placeholder for the `stream` argument: `_call` substitutes the current stream of the tensors' device."""


_S = _StreamArg()


LAUNCHES = 0     # kernels launched through the C-ABI (bench.py reports it as gpu_launches)
PROFILE = None   # when a list: (name, start_event, end_event) per launch, on the launching stream


def _call(name: str, fn, dev: torch.device, *args) -> None:
    """One C-ABI launch on the current stream of `dev`, with `dev` as the current CUDA device for the duration of
    the call (the library launches on, and encodes TMA descriptors for, the current device)."""
    global LAUNCHES
    # (raw torch._C calls: the eager step is bound by host-side launch cost, and the `torch.cuda.device` context manager
    # plus a `Stream` object per launch were a third of it - tools/profile_eager.py)
    index = dev.index if dev.index is not None else torch._C._cuda_getDevice()
    previous = torch._C._cuda_getDevice()
    if previous != index:
        torch._C._cuda_setDevice(index)
    try:
        raw_stream = torch._C._cuda_getCurrentRawStream(index)   # plain int: 0 (the default stream) converts to NULL
        args = tuple(raw_stream if a is _S else a for a in args)
        if PROFILE is not None:
            stream = torch.cuda.current_stream(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            status = fn(*args)
            b.record(stream)
            PROFILE.append((name, a, b))
        else:
            status = fn(*args)
    finally:
        if previous != index:
            torch._C._cuda_setDevice(previous)
    LAUNCHES += 1
    check(status, name)


@dataclass
class Operand:
    """A packed K-major bf16 operand: planes [P, rows_pad, Dp] + optional fp32 0.5*||row||^2."""
    planes: torch.Tensor
    rows: int
    dim: int
    nplanes: int
    half_sqnorm: torch.Tensor | None = None
    plane_rows: int = 0  # row stride between planes; 0 = padded default, rows = zero-copy view of a bf16 tensor
    inv_norm: torch.Tensor | None = None  # fp32 [rows_pad] 1/|row| (per-column scale for raw-token column arg-min)
    lo_norm_max: torch.Tensor | None = None  # fp32 [1]: max_j |row_j - hi_j| of an 'f16x2' operand (one-term error bound)
    fmt: str = 'bf16'    # 'bf16': 1..3 bf16 planes | 'f16': one fp16 plane | 'f16x2': the fp16 (hi, lo * 2^11) pair
    folded: str | None = None   # 'tokens' | 'codes': the L2 side terms live in the spare columns (fold_l2_side)

    @property
    def pair(self) -> bool:
        return self.fmt == 'f16x2'

    @property
    def abi_planes(self) -> int:
        return {'bf16': self.nplanes, 'f16': PLANES_F16, 'f16x2': PLANES_F16X2}[self.fmt]


def operand_shape(rows: int, D: int) -> tuple[int, int]:
    lib = _lib.load()
    return int(lib.vqb_operand_rows_pad(rows)), int(lib.vqb_operand_dp(D))


def pack_rows(src: torch.Tensor, *, normalize: bool = False, planes: int | None = None,
              want_half_sqnorm: bool = False, writeback: torch.Tensor | None = None,
              reset_keys: torch.Tensor | None = None, fmt: str = 'bf16',
              zero_fill: torch.Tensor | None = None, want_lo_norm: bool = False, fold: str | None = None) -> Operand:
    """fp32/bf16 rows -> operand planes (see vqb_pack_rows).
    fmt='bf16': exact bf16 planes; `planes=None` picks the exact representation (1 plane for un-normalised bf16
                input, 3 planes otherwise).
    fmt='f16x2': the two-plane fp16 (hi, lo * 2^11) pair of NORMALISED rows: 22 significant bits, two MMA terms.
    fmt='f16':  one fp16 plane of un-normalised bf16 rows (the partner of an 'f16x2' operand)."""
    lib = _lib.load()
    dev = _cuda(src, writeback, reset_keys, zero_fill)
    assert src.dim() == 2
    zero_bytes = 0
    if zero_fill is not None:      # fused memset of e.g. the step's statistics buffer (padded to 16 bytes by the owner)
        zero_bytes = zero_fill.numel() * zero_fill.element_size()
        assert zero_bytes % 16 == 0 and zero_fill.data_ptr() % 16 == 0
    rows, D = src.shape
    if fmt == 'f16x2':
        if not normalize:
            raise ValueError("the fp16-pair plane format needs normalised rows (|v| <= 1)")
        planes, code = 2, PLANES_F16X2
    elif fmt == 'f16':
        if normalize or src.dtype != torch.bfloat16:
            raise ValueError("the one-plane fp16 format takes un-normalised bf16 rows")
        planes, code = 1, PLANES_F16
    elif fmt == 'bf16':
        if planes is None:
            planes = 1 if (src.dtype == torch.bfloat16 and not normalize) else 3
        code = planes
    else:
        raise ValueError(f'unknown plane format {fmt!r}')
    rows_pad, Dp = operand_shape(rows, D)
    dst = torch.empty((planes, rows_pad, Dp), dtype=torch.bfloat16, device=src.device)   # 16-bit storage
    h = torch.empty((rows_pad,), dtype=torch.float32, device=src.device) if want_half_sqnorm else None
    if writeback is not None:
        assert writeback.dtype == torch.float32 and writeback.shape == src.shape
    lo = torch.zeros((1,), dtype=torch.float32, device=src.device) if (want_lo_norm and fmt == 'f16x2') else None
    if fold is not None:
        # L2 side terms folded into the spare columns by the pack launch itself (vqb_pack_rows_fold): 'codes', 'tokens'
        # (row arg-min: ones only) or 'tokens+h' (column arg-min: the tokens' own term as well)
        assert fmt == 'bf16' and fold in ('codes', 'tokens', 'tokens+h')
        role = {'tokens': 0, 'codes': 1, 'tokens+h': 2}[fold]
        if role != 0 and h is None and D % 8 != 0:
            h = torch.empty((rows_pad,), dtype=torch.float32, device=src.device)
        _call('vqb_pack_rows', lib.vqb_pack_rows_fold, dev, _p(src), _dt(src), rows, D, int(normalize), code, _p(dst), _p(h),
              _p(writeback), _p(reset_keys), reset_keys.numel() if reset_keys is not None else 0, _p(zero_fill), zero_bytes,
              role, _S)
        return Operand(dst, rows, D, planes, h, fmt=fmt, folded='codes' if role == 1 else 'tokens')
    _call('vqb_pack_rows', lib.vqb_pack_rows, dev, _p(src), _dt(src), rows, D, int(normalize), code, _p(dst), _p(h),
          _p(writeback), _p(reset_keys), reset_keys.numel() if reset_keys is not None else 0, _p(zero_fill), zero_bytes,
          _p(lo), _S)
    return Operand(dst, rows, D, planes, h, fmt=fmt, lo_norm_max=lo)


L2_FOLD_COLUMNS = 6


def can_fold_l2(D: int) -> bool:
    """True when the operand width of D leaves the spare zero columns the folded L2 side terms need."""
    return operand_shape(1, D)[1] - D >= L2_FOLD_COLUMNS


def fold_l2_side(op: Operand, role: str) -> Operand:
    """vqb_fold_l2_side: write the L2 side terms into the spare columns of a packed exact-bf16 operand (in place).
    role 'codes' needs op.half_sqnorm; role 'tokens' uses it when present (column arg-min) and 1-columns only
    otherwise (row arg-min).  Both operands of an `assign(..., l2=True)` must be folded, with opposite roles; the
    kernel then runs without its per-column side term."""
    lib = _lib.load()
    assert op.fmt == 'bf16' and op.plane_rows == 0 and op.folded is None and role in ('tokens', 'codes')
    dev = _cuda(op.planes, op.half_sqnorm)
    _call('vqb_fold_l2_side', lib.vqb_fold_l2_side, dev, _p(op.planes), op.nplanes, op.rows, op.dim, _p(op.half_sqnorm),
          1 if role == 'codes' else 0, _S)
    op.folded = role
    return op


def transpose_last2(src: torch.Tensor) -> torch.Tensor:
    """[B, R, C] -> [B, C, R] contiguous (vqb_transpose_last2): the caller's NCHW <-> token-major rearranges."""
    lib = _lib.load()
    dev = _cuda(src)
    assert src.dim() == 3 and src.element_size() in (2, 4, 8)
    B, R, C = src.shape
    dst = torch.empty((B, C, R), dtype=src.dtype, device=src.device)
    _call('vqb_transpose_last2', lib.vqb_transpose_last2, dev, _p(src), src.element_size(), B, R, C, _p(dst), _S)
    return dst


def compact_tokens(keys: torch.Tensor, codebook_size: int, index_offset: int = 0,
                   out: torch.Tensor | None = None) -> torch.Tensor:
    """Packed keys -> compact token ids: uint16 for codebooks of at most 65 536 codes, int32 otherwise (written into
    `out` when given: a contiguous tensor of that dtype and the keys' size)."""
    lib = _lib.load()
    dev = _cuda(keys, out)
    assert keys.dtype == torch.int64
    small = codebook_size <= 65536
    if out is None:
        out = torch.empty(keys.shape, dtype=torch.uint16 if small else torch.int32, device=keys.device)
    assert out.dtype == (torch.uint16 if small else torch.int32) and out.numel() == keys.numel()
    _call('vqb_compact_tokens', lib.vqb_compact_tokens, dev, _p(keys), keys.numel(), index_offset, _p(out), 2 if small else 4,
          _S)
    return out


def new_keys(n: int, device) -> torch.Tensor:
    """All-ones packed keys (int64 storage of the uint64 keys)."""
    return torch.full((n,), -1, dtype=torch.int64, device=device)


def assign(a: Operand, b: Operand, keys: torch.Tensor, *, l2: bool, index_offset: int = 0,
           backend: int = BACKEND_TCGEN05, scale_columns: bool = False, second_keys: torch.Tensor | None = None,
           a_rows_dev: torch.Tensor | None = None) -> torch.Tensor:
    """keys[i] = min(keys[i], key(argmax_j score)), score = <a_i,b_j> - 0.5|b_j|^2 (l2), <a_i,b_j> * (1/|b_j|)
    (scale_columns: b holds RAW rows + `inv_norm`), or <a_i,b_j>.
    second_keys: also record the runner-up score of every row (certified one-term pass); a_rows_dev: int32 [1] device
    tensor bounding the number of valid A rows (vqb_assign_ex)."""
    lib = _lib.load()
    dev = _cuda(a.planes, b.planes, keys, second_keys, a_rows_dev)
    assert a_rows_dev is None or a_rows_dev.dtype == torch.int32
    assert second_keys is None or (second_keys.dtype == torch.int64 and second_keys.numel() >= a.rows)
    assert a.dim == b.dim and keys.dtype == torch.int64 and keys.numel() >= a.rows
    side, mode = None, 0
    assert (a.folded is None) == (b.folded is None) and (a.folded is None or a.folded != b.folded), \
        'folded L2 operands come in (tokens, codes) pairs'
    if l2 and b.folded is not None:
        pass                       # the side terms are part of the contraction
    elif l2:
        assert b.half_sqnorm is not None, 'L2 assignment needs the packed operand to carry half_sqnorm'
        side, mode = b.half_sqnorm, 1
    elif scale_columns:
        assert b.inv_norm is not None
        side, mode = b.inv_norm, 2
    if second_keys is None and a_rows_dev is None:
        _call('vqb_assign', lib.vqb_assign, dev, _p(a.planes), a.abi_planes, a.rows, a.plane_rows, _p(b.planes),
              b.abi_planes, b.rows, b.plane_rows, a.dim, _p(side), mode, index_offset, _p(keys), backend, _S)
    else:
        _call('vqb_assign', lib.vqb_assign_ex, dev, _p(a.planes), a.abi_planes, a.rows, a.plane_rows, _p(b.planes),
              b.abi_planes, b.rows, b.plane_rows, a.dim, _p(side), mode, index_offset, _p(keys), _p(second_keys),
              _p(a_rows_dev), backend, _S)
    return keys


def certify(keys: torch.Tensor, second_keys: torch.Tensor, rows: int, delta: torch.Tensor, *,
            row_inv_norm: torch.Tensor | None = None, noise: float = 2.0 ** -20,
            compact_out: torch.Tensor | None = None):
    """Rows whose best - runner-up margin does not exceed twice the one-term error bound -> (row_list int32 [rows],
    count int32 [1], compact_keys int64 [rows] with the first `count` entries reset)."""
    lib = _lib.load()
    dev = _cuda(keys, second_keys, delta, row_inv_norm)
    row_list = torch.empty((rows,), dtype=torch.int32, device=keys.device)
    count = torch.empty((1,), dtype=torch.int32, device=keys.device)
    compact = compact_out if compact_out is not None else torch.empty((rows,), dtype=torch.int64, device=keys.device)
    ws = torch.empty((int(lib.vqb_certify_workspace_bytes(rows)),), dtype=torch.uint8, device=keys.device)
    _call('vqb_certify', lib.vqb_certify, dev, _p(keys), _p(second_keys), rows, _p(row_inv_norm), _p(delta), noise,
          _p(row_list), _p(count), _p(compact), _p(ws), _S)
    return row_list, count, compact


def cvq_needy_codes(prob: torch.Tensor, counts_local: torch.Tensor, total_global: int, *, decay: float, eps: float):
    """Codes whose anchor can receive a non-zero blend weight this step (vqb_cvq_needy_codes) ->
    (code_list int32 [K], count int32 [1], compact_keys int64 [K] with the first `count` entries reset)."""
    lib = _lib.load()
    dev = _cuda(prob, counts_local)
    K = prob.numel()
    assert counts_local.dtype == torch.int64 and counts_local.numel() >= K
    code_list = torch.empty((K,), dtype=torch.int32, device=prob.device)
    count = torch.empty((1,), dtype=torch.int32, device=prob.device)
    compact = torch.empty((K,), dtype=torch.int64, device=prob.device)
    ws = torch.empty((int(lib.vqb_certify_workspace_bytes(K)),), dtype=torch.uint8, device=prob.device)
    _call('vqb_cvq_needy_codes', lib.vqb_cvq_needy_codes, dev, _p(prob), _p(counts_local), float(total_global), K,
          _f32(decay), _f32(1 - decay), _f32(eps), _p(code_list), _p(count), _p(compact), _p(ws), _S)
    return code_list, count, compact


def gather_operand_rows(src: Operand, row_list: torch.Tensor, count: torch.Tensor) -> Operand:
    """Compact copy of the listed rows of a packed operand (all planes, side vectors included); capacity = src.rows."""
    lib = _lib.load()
    dev = _cuda(src.planes, row_list, count)
    P, Dp = src.planes.shape[0] if src.planes.dim() == 3 else 1, src.planes.shape[-1]
    src_plane_rows = src.plane_rows or (src.planes.shape[1] if src.planes.dim() == 3 else src.rows)
    rows_pad = operand_shape(src.rows, src.dim)[0]
    dst = torch.empty((src.nplanes, rows_pad, Dp), dtype=torch.bfloat16, device=src.planes.device)
    _call('vqb_gather_plane_rows', lib.vqb_gather_plane_rows, dev, _p(src.planes), src.nplanes, src_plane_rows, Dp,
          _p(row_list), _p(count), src.rows, _p(dst), rows_pad, _S)
    out = Operand(dst, src.rows, src.dim, src.nplanes, None, fmt=src.fmt, folded=src.folded)
    return out


def scatter_keys(compact: torch.Tensor, row_list: torch.Tensor, count: torch.Tensor, keys: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(compact, row_list, count, keys)
    _call('vqb_scatter_keys', lib.vqb_scatter_keys, dev, _p(compact), _p(row_list), _p(count), row_list.numel(), _p(keys), _S)
    return keys


def row_inv_norm(x: torch.Tensor, f16_rows: bool = False) -> torch.Tensor:
    """1 / max(|x_r|, eps) per row (zero in the operand padding); f16_rows: for rows packed with fmt='f16'."""
    lib = _lib.load()
    dev = _cuda(x)
    rows, D = x.shape
    out = torch.empty((operand_shape(rows, D)[0],), dtype=torch.float32, device=x.device)
    _call('vqb_row_inv_norm', lib.vqb_row_inv_norm, dev, _p(x), _dt(x), rows, D, int(f16_rows), _p(out), _S)
    return out


def unpack_keys(keys: torch.Tensor, index_offset: int = 0, want_score: bool = False):
    lib = _lib.load()
    dev = _cuda(keys)
    n = keys.numel()
    idx = torch.empty((n,), dtype=torch.int64, device=keys.device)
    score = torch.empty((n,), dtype=torch.float32, device=keys.device) if want_score else None
    _call('vqb_unpack_keys', lib.vqb_unpack_keys, dev, _p(keys), n, index_offset, _p(idx), _p(score), _S)
    return (idx, score) if want_score else idx


def keys_flip_sign(keys: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(keys)
    _call('vqb_keys_flip_sign', lib.vqb_keys_flip_sign, dev, _p(keys), keys.numel(), _S)
    return keys


_WS: dict = {}


def _loss_ws(device):
    """Partials + self-resetting ticket of the deterministic loss reduction: one pair per (device, stream), so
    forwards issued concurrently on different streams of a GPU never share the ticket."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    if key not in _WS:
        lib = _lib.load()
        _WS[key] = (torch.empty((int(lib.vqb_loss_partials_count()),), dtype=torch.float32, device=device),
                    torch.zeros((1,), dtype=torch.int32, device=device))
    return _WS[key]


def as_operand(x: torch.Tensor) -> Operand | None:
    """Zero-copy one-plane operand view of a contiguous bf16 [rows, D] tensor whose D needs no padding."""
    if x.dtype == torch.bfloat16 and x.is_contiguous() and x.dim() == 2 and x.data_ptr() % 16 == 0:
        rows, D = x.shape
        if operand_shape(rows, D)[1] == D:
            return Operand(x, rows, D, 1, None, plane_rows=rows)
    return None


def gather_ste_loss(x: torch.Tensor, W: torch.Tensor, *, quant: torch.Tensor | None = None,
                    keys: torch.Tensor | None = None, key_offset: int = 0, normalize_x: bool = False,
                    want_norm: bool, want_quant: bool = False, want_xnorm: bool = False, z_hw: int = 0):
    """Fused gather + STE + loss (+ token normalisation, + key unpack) — see vqb_gather_ste_loss.
    -> (z_ste [N,D] fp32, mse4 [4], quant int64 [N] | None, x_normalised [N,D] fp32 | None)"""
    lib = _lib.load()
    dev = _cuda(x, W, quant, keys)
    assert W.dtype == torch.float32 and (quant is None) != (keys is None)
    N, D = x.shape
    z = torch.empty((N, D), dtype=torch.float32, device=x.device)
    mse4 = torch.empty((4,), dtype=torch.float32, device=x.device)
    qo = torch.empty((N,), dtype=torch.int64, device=x.device) if want_quant else None
    xn = torch.empty((N, D), dtype=torch.float32, device=x.device) if want_xnorm else None
    partials, ticket = _loss_ws(x.device)
    _call('vqb_gather_ste_loss', lib.vqb_gather_ste_loss, dev, _p(x), _dt(x), N, D, int(normalize_x), _p(W), W.shape[0],
          _p(quant), _p(keys), key_offset, _p(qo), _p(xn), _p(z), z_hw, int(want_norm), _p(mse4), _p(partials), _p(ticket),
          _S)
    return z, mse4, qo, xn


def quantize_backward(g_z: torch.Tensor, x: torch.Tensor, W: torch.Tensor, quant: torch.Tensor, g4, *,
                      normalize_x: bool = False, want_norm: bool, need_gW: bool, g_hw: int = 0,
                      deterministic: bool | None = None):
    """g4: a float32 [4] tensor or a sequence of four 0-dim device tensors / None
    (codebook, commitment, codebook-norm, commitment-norm upstream gradients).
    deterministic: None follows torch.are_deterministic_algorithms_enabled(); when on, gW is the segment sum of the
    per-token gradient rows (fixed association, see vqb_segment_sum_rows) instead of fp32 atomics.  gx is the same."""
    lib = _lib.load()
    if isinstance(g4, torch.Tensor):
        g4 = [g4[i] for i in range(4)]
    dev = _cuda(g_z, x, W, quant, *g4)
    assert all(g is None or g.dtype == torch.float32 for g in g4)
    if not (g_z.dtype == torch.float32 or (g_z.dtype == torch.bfloat16 and x.dtype == torch.bfloat16)):
        g_z = g_z.float()
    N, D = x.shape
    K = W.shape[0]
    gx = torch.empty_like(x)
    gW = torch.zeros_like(W) if need_gW else None
    if need_gW and deterministic_enabled(deterministic):
        rows = _det_ws(x.device, 'gw_rows', N * D, torch.float32)
        _call('vqb_quantize_backward_rows', lib.vqb_quantize_backward_rows, dev, _p(g_z), _dt(g_z), _p(x), _dt(x),
              int(normalize_x), _p(W), K, _p(quant), N, D, _p(g4[0]), _p(g4[1]), _p(g4[2]), _p(g4[3]), int(want_norm),
              _p(gx), _p(rows), g_hw, _S)
        order, offsets = _code_sort_ws(dev, N, K, quant, None, 0)
        _segment_sum(dev, rows, N, D, False, order, offsets, K, gW, None)
        return gx, gW
    _call('vqb_quantize_backward', lib.vqb_quantize_backward, dev, _p(g_z), _dt(g_z), _p(x), _dt(x), int(normalize_x), _p(W),
          K, _p(quant), N, D, _p(g4[0]), _p(g4[1]), _p(g4[2]), _p(g4[3]), int(want_norm), _p(gx), _p(gW),
          g_hw, _S)
    return gx, gW


def l2norm_forward(x: torch.Tensor, out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(x)
    y = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    _call('vqb_l2norm_forward', lib.vqb_l2norm_forward, dev, _p(x), _dt(x), x.shape[0], x.shape[1], _p(y), _dt(y), _S)
    return y


def l2norm_backward(gy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(gy, x)
    gx = torch.empty_like(x)
    _call('vqb_l2norm_backward', lib.vqb_l2norm_backward, dev, _p(gy), _dt(gy), _p(x), _dt(x), x.shape[0], x.shape[1], _p(gx), _dt(gx),
                                  _S)
    return gx


def scatter_stats(x: torch.Tensor, quant: torch.Tensor | None, K: int, *, normalize_x: bool = False,
                  out: torch.Tensor | None = None, keys: torch.Tensor | None = None, key_offset: int = 0,
                  deterministic: bool | None = None) -> torch.Tensor:
    """fp32 [K*D + K] = per-code feature sums followed by per-code counts (one all-reduce buffer).  The code of a
    token comes from `quant` (int64 indices) or straight from the packed `keys` of the assignment.
    deterministic: None follows torch.are_deterministic_algorithms_enabled(); when on, the sums are formed by the code
    sort + chunked segment sum (fixed association, see vqb_segment_sum_rows) instead of fp32 atomics."""
    lib = _lib.load()
    dev = _cuda(x, quant, out, keys)
    assert (quant is None) != (keys is None)
    N, D = x.shape
    stats = out if out is not None else torch.zeros((K * D + K,), dtype=torch.float32, device=x.device)
    if deterministic_enabled(deterministic):
        assert stats.dtype == torch.float32 and stats.numel() >= K * D + K
        order, offsets = _code_sort_ws(dev, N, K, quant, keys, key_offset)
        _segment_sum(dev, x, N, D, normalize_x, order, offsets, K, stats, stats[K * D:])
        return stats
    _call('vqb_scatter_stats', lib.vqb_scatter_stats, dev, _p(x), _dt(x), N, D, int(normalize_x), _p(quant), _p(keys),
          key_offset, _p(stats), K, _S)
    return stats


# ---- deterministic per-code reductions (csrc/segment.cu) ---------------------------------------------------------


def deterministic_enabled(deterministic: bool | None = None) -> bool:
    """The switch of the deterministic reductions: an explicit argument, else torch's own flag, read at call time."""
    return torch.are_deterministic_algorithms_enabled() if deterministic is None else bool(deterministic)


def segment_chunk() -> int:
    """C of the segment-sum association contract (VQB_SEGMENT_CHUNK)."""
    return int(_lib.load().vqb_segment_chunk())


_DET_WS: dict = {}
_DET_RETIRED: list = []


def _det_ws(device, name: str, numel: int, dtype: torch.dtype) -> torch.Tensor:
    """Scratch of the deterministic path, cached per (device, stream, name) like `_loss_ws`, so a captured CUDA graph
    replays the same buffers.  Grows in powers of two; an outgrown buffer stays referenced because a graph captured
    earlier may still read it."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, name)
    buf = _DET_WS.get(key)
    if buf is None or buf.numel() < numel:
        if buf is not None:
            _DET_RETIRED.append(buf)
        buf = _DET_WS[key] = torch.empty((1 << max(numel - 1, 0).bit_length(),), dtype=dtype, device=device)
    return buf[:numel]


def _code_sort_call(dev, N: int, K: int, quant, keys, key_offset: int, order, offsets) -> None:
    lib = _lib.load()
    scratch = _det_ws(dev, 'sort', int(lib.vqb_code_sort_scratch_bytes(N, K)), torch.uint8)
    _call('vqb_code_sort', lib.vqb_code_sort, dev, _p(quant), _p(keys), key_offset, N, K, _p(order), _p(offsets),
          _p(scratch), scratch.numel(), _S)


def _code_sort_ws(dev, N: int, K: int, quant, keys, key_offset: int):
    order = _det_ws(dev, 'order', N, torch.int32)
    offsets = _det_ws(dev, 'offsets', K + 1, torch.int32)
    _code_sort_call(dev, N, K, quant, keys, key_offset, order, offsets)
    return order, offsets


def _segment_sum(dev, rows, N: int, D: int, normalize: bool, order, offsets, K: int, out_sums, out_counts) -> None:
    lib = _lib.load()
    scratch = _det_ws(dev, 'segment', int(lib.vqb_segment_sum_scratch_bytes(N, K, D)), torch.uint8)
    _call('vqb_segment_sum_rows', lib.vqb_segment_sum_rows, dev, _p(rows), _dt(rows), N, D, int(normalize), _p(order),
          _p(offsets), K, _p(out_sums), _p(out_counts), _p(scratch), scratch.numel(), _S)


def code_sort(K: int, *, quant: torch.Tensor | None = None, keys: torch.Tensor | None = None,
              key_offset: int = 0) -> tuple[torch.Tensor, torch.Tensor]:
    """Stable sort of the tokens by code (vqb_code_sort) -> (order int32 [N], offsets int32 [K+1]): code k owns
    order[offsets[k]:offsets[k+1]] in ascending token order; tokens whose code is outside [0, K) come last."""
    dev = _cuda(quant, keys)
    assert (quant is None) != (keys is None)
    idx = quant if quant is not None else keys
    assert idx.dtype == torch.int64
    N = idx.numel()
    order = torch.empty((N,), dtype=torch.int32, device=idx.device)
    offsets = torch.empty((K + 1,), dtype=torch.int32, device=idx.device)
    _code_sort_call(dev, N, K, quant, keys, key_offset, order, offsets)
    return order, offsets


def segment_sum_rows(rows: torch.Tensor, order: torch.Tensor, offsets: torch.Tensor, *, normalize: bool = False,
                     out_sums: torch.Tensor | None = None, out_counts: torch.Tensor | None = None) -> torch.Tensor:
    """out_sums fp32 [K, D] (+)= the per-code sums of `rows` (fp32 / bf16 [N, D]) in the fixed association of
    vqb_segment_sum_rows; out_counts fp32 [K] (+)= the token counts.  Zero-filled outputs are allocated when omitted."""
    dev = _cuda(rows, order, offsets, out_sums, out_counts)
    assert order.dtype == torch.int32 and offsets.dtype == torch.int32 and rows.dim() == 2
    N, D = rows.shape
    K = offsets.numel() - 1
    assert order.numel() == N
    if out_sums is None:
        out_sums = torch.zeros((K, D), dtype=torch.float32, device=rows.device)
    assert out_sums.dtype == torch.float32 and out_sums.numel() == K * D
    assert out_counts is None or (out_counts.dtype == torch.float32 and out_counts.numel() == K)
    _segment_sum(dev, rows, N, D, normalize, order, offsets, K, out_sums, out_counts)
    return out_sums


def bincount_accumulate(quant: torch.Tensor, counts: torch.Tensor, K: int | None = None,
                        total_slot: bool = False) -> torch.Tensor:
    """counts[:K] += bincount(quant); with total_slot, counts has K+1 entries and counts[K] += numel."""
    lib = _lib.load()
    dev = _cuda(quant, counts)
    assert quant.dtype == torch.int64 and counts.dtype == torch.int64
    K = counts.numel() - int(total_slot) if K is None else K
    assert counts.numel() >= K + int(total_slot)
    flat = quant.reshape(-1)
    _call('vqb_bincount_accumulate', lib.vqb_bincount_accumulate, dev, _p(flat), flat.numel(), _p(counts), K, int(total_slot), _S)
    return counts


def _f32(v: float) -> float:
    return float(torch.tensor(v, dtype=torch.float32).item())


def kmeans_ema_update(stats: torch.Tensor, W: torch.Tensor, decay: float) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(stats, W)
    K, D = W.shape
    _call('vqb_kmeans_ema_update', lib.vqb_kmeans_ema_update, dev, _p(stats), _p(W), K, D, _f32(decay), _f32(1 - decay), _S)
    return W


def gather_rows_by_key(x: torch.Tensor, keys: torch.Tensor, index_offset: int = 0,
                       out: torch.Tensor | None = None) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(x, keys, out)
    N, D = x.shape
    K = keys.numel()
    if out is None:
        out = torch.empty((K, D), dtype=torch.float32, device=x.device)
    assert out.dtype == torch.float32 and out.shape == (K, D)
    _call('vqb_gather_rows_by_key', lib.vqb_gather_rows_by_key, dev, _p(x), _dt(x), N, D, _p(keys), K, index_offset, _p(out), _S)
    return out


def cvq_update(W: torch.Tensor, anchors: torch.Tensor, prob: torch.Tensor, counts: torch.Tensor,
               total: torch.Tensor, *, decay: float, eps: float, anchor_scale: float = 1.0) -> None:
    """counts: int64 [K]; total: int64 [1] device tensor (both already all-reduced)."""
    lib = _lib.load()
    dev = _cuda(W, anchors, prob, counts, total)
    assert counts.dtype == torch.int64 and total.dtype == torch.int64
    K, D = W.shape
    _call('vqb_cvq_update', lib.vqb_cvq_update, dev, _p(W), _p(anchors), anchor_scale, _p(prob), _p(counts), _p(total), K, D,
                             _f32(decay), _f32(1 - decay), _f32(eps), _S)


def embedding_gather(W: torch.Tensor, quant: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(W, quant)
    assert W.dtype == torch.float32 and quant.dtype == torch.int64
    flat = quant.reshape(-1).contiguous()
    out = torch.empty((flat.numel(), W.shape[1]), dtype=torch.float32, device=W.device)
    _call('vqb_embedding_gather', lib.vqb_embedding_gather, dev, _p(W), W.shape[0], W.shape[1], _p(flat), flat.numel(), _p(out), _S)
    return out.reshape(*quant.shape, W.shape[1])


def distance_matrix(x: torch.Tensor, W: torch.Tensor, metric: str) -> torch.Tensor:
    """Compatibility mode: the materialised fp32 [N, K] distance matrix (`torch.cdist` / `1 - cos`)."""
    lib = _lib.load()
    dev = _cuda(x, W)
    assert W.dtype == torch.float32 and x.dim() == 2 and W.dim() == 2 and x.shape[1] == W.shape[1]
    N, D = x.shape
    out = torch.empty((N, W.shape[0]), dtype=torch.float32, device=x.device)
    _call('vqb_distance_matrix', lib.vqb_distance_matrix, dev, _p(x), _dt(x), N, D, _p(W), W.shape[0],
          int(metric == 'Cosine'), _p(out), _S)
    return out


# ---- fused peer-memory exchange + codebook update (csrc/comm.cu) ------------------------------------------------
NO_KEYS = (1 << 64) - 1    # (size_t)-1: "no key buffer" (sync=False anchors)


def comm_kmeans_ema_update(region, K: int, D: int, decay: float, *, stats: str = 'stats', W: str = 'W',
                           ll_in: str = 'll_in', ll_out: str = 'll_out') -> None:
    """all_reduce(SUM) of every rank's [K*D sums | K counts] + k-means/EMA codebook update, one launch; the new rows
    land in every rank's region (`region` is a parallel.PeerRegion).  With the staging buffers `ll_in` / `ll_out`
    in the region the low-latency (flag-in-data) protocol is used, otherwise the barrier protocol."""
    lib = _lib.load()
    ll = ll_in in region.offsets and ll_out in region.offsets
    _call('vqb_comm_kmeans_ema_update', lib.vqb_comm_kmeans_ema_update, region.device, c_void_p(region.base), region.rank,
          region.world, region.offsets[stats], region.offsets[W], region.offsets[ll_in] if ll else NO_KEYS,
          region.offsets[ll_out] if ll else NO_KEYS, K, D, _f32(decay), _f32(1 - decay), _S)


def comm_ll_layout(K: int, D: int, world: int):
    """Staging buffers of the low-latency exchange: (name, shape, dtype) entries for PeerRegion.alloc."""
    per = (K + world - 1) // world
    return [('ll_in', (world * per * (D + 1),), torch.int32), ('ll_out', (K * D,), torch.int32)]


def comm_cvq_update(region, K: int, D: int, *, decay: float, eps: float, minloc: bool, counts: str = 'counts',
                    anchors: str = 'anchors', keys: str = 'keys', W: str = 'W', prob: str = 'prob') -> None:
    """Usage-count + anchor exchange fused with the CVQ-VAE probability EMA and anchor blend, one launch."""
    lib = _lib.load()
    _call('vqb_comm_cvq_update', lib.vqb_comm_cvq_update, region.device, c_void_p(region.base), region.rank, region.world,
          region.offsets[counts], region.offsets[anchors], region.offsets[keys] if minloc else NO_KEYS,
          region.offsets[W], region.offsets[prob], K, D, _f32(decay), _f32(1 - decay), _f32(eps), _S)


def comm_allreduce_min_keys(region, n: int, keys: str = 'keys') -> None:
    lib = _lib.load()
    _call('vqb_comm_allreduce_min_keys', lib.vqb_comm_allreduce_min_keys, region.device, c_void_p(region.base),
          region.rank, region.world, region.offsets[keys], n, _S)


def comm_allreduce_sum_f32(region, n: int, name: str) -> None:
    lib = _lib.load()
    _call('vqb_comm_allreduce_sum_f32', lib.vqb_comm_allreduce_sum_f32, region.device, c_void_p(region.base), region.rank,
          region.world, region.offsets[name], n, _S)


# ---- FSQ -------------------------------------------------------------------------------------


def fsq_params(levels, eps: float) -> FSQParams:
    """Per-channel constants computed with torch on the host EXACTLY as the reference computes them
    (vq/algorithms/fsq/quantizers.py:30,114-115,122), then handed to the kernels by value."""
    levels = [int(v) for v in levels]
    if not 1 <= len(levels) <= 16:
        raise ValueError('FSQ supports 1..16 channels')
    max_per_digit = torch.tensor(levels, dtype=torch.int)
    cumprod = torch.tensor((1,) + tuple(levels[:-1])).cumprod(0)
    max_int = max_per_digit - 1
    max_ = max_int * (1 - eps)
    odd = max_int % 2
    shift = torch.atanh(odd / max_)
    half = max_per_digit // 2
    p = FSQParams()
    p.D = len(levels)
    for d in range(len(levels)):
        p.max_[d] = float(max_[d])
        p.odd[d] = float(odd[d])
        p.shift[d] = float(shift[d])
        p.half[d] = float(half[d])
        p.cumprod[d] = int(cumprod[d])
        p.levels[d] = levels[d]
    return p


def fsq_forward(x: torch.Tensor, p: FSQParams, out_dtype: torch.dtype | None = None):
    lib = _lib.load()
    dev = _cuda(x)
    N, D = x.shape
    assert D == p.D
    zq = torch.empty((N, D), dtype=out_dtype or x.dtype, device=x.device)
    idx = torch.empty((N,), dtype=torch.int32, device=x.device)
    _call('vqb_fsq_forward', lib.vqb_fsq_forward, dev, _p(x), _dt(x), N, ctypes.byref(p), _p(zq), _dt(zq), _p(idx), _S)
    return zq, idx


def fsq_backward(gz: torch.Tensor, x: torch.Tensor, p: FSQParams) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(gz, x)
    gx = torch.empty_like(x)
    _call('vqb_fsq_backward', lib.vqb_fsq_backward, dev, _p(gz), _dt(gz), _p(x), _dt(x), x.shape[0], ctypes.byref(p), _p(gx), _dt(gx),
                               _S)
    return gx


def fsq_decode(index: torch.Tensor, p: FSQParams) -> torch.Tensor:
    lib = _lib.load()
    dev = _cuda(index)
    index = index.to(torch.int32) if index.dtype != torch.int32 else index
    flat = index.reshape(-1).contiguous()
    z = torch.empty((flat.numel(), p.D), dtype=torch.float32, device=index.device)
    _call('vqb_fsq_decode', lib.vqb_fsq_decode, dev, _p(flat), flat.numel(), ctypes.byref(p), _p(z), _S)
    return z.reshape(*index.shape, p.D)


# ---- token ids -> NCHW latents (csrc/layout.cu) -------------------------------------------------------------------
_ID_BYTES = {torch.uint16: 2, torch.int32: 4, torch.int64: 8}


def _decode_out(ids: torch.Tensor, hw: int, D: int, out_dtype: torch.dtype, bad_count: torch.Tensor | None):
    """Checks the ids / counter of a decode_tokens call; returns (b, id_bytes, z) with z = empty [b, D, *spatial]."""
    if ids.dtype not in _ID_BYTES:
        raise TypeError(f'token ids must be uint16, int32 or int64, got {ids.dtype}')
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f'out_dtype must be float32 or bfloat16, got {out_dtype}')
    if bad_count is not None and (bad_count.dtype != torch.int32 or bad_count.numel() != 1):
        raise TypeError('bad_count must be a one-element int32 tensor')
    n = ids.numel()
    if hw <= 0 or n % hw:
        raise ValueError(f'{n} token ids do not split into images of hw = {hw} tokens')
    b = n // hw
    spatial = tuple(ids.shape[1:]) if ids.dim() >= 2 and ids.shape[0] == b else (hw,)
    return b, _ID_BYTES[ids.dtype], torch.empty((b, D) + spatial, dtype=out_dtype, device=ids.device)


def decode_tokens(W: torch.Tensor, ids: torch.Tensor, hw: int, out_dtype: torch.dtype = torch.float32,
                  bad_count: torch.Tensor | None = None) -> torch.Tensor:
    """Token ids [b, h, w] (uint16 / int32 / int64, b * hw in all) -> z = W[ids] as [b, D, h, w] of `out_dtype`, in one
    launch (vqb_decode_tokens).  An id outside [0, K) gives a NaN row and is counted into `bad_count` (a zeroed
    one-element int32 device tensor) when one is given."""
    lib = _lib.load()
    dev = _cuda(W, ids, bad_count)
    if W.dtype != torch.float32 or W.dim() != 2:
        raise TypeError('the codebook must be a float32 [K, D] tensor')
    K, D = W.shape
    b, id_bytes, z = _decode_out(ids, hw, D, out_dtype, bad_count)
    _call('vqb_decode_tokens', lib.vqb_decode_tokens, dev, _p(ids), id_bytes, b, hw, _p(W), K, D, _p(z), _dt(z),
          _p(bad_count), _S)
    return z


def fsq_decode_tokens(ids: torch.Tensor, p: FSQParams, hw: int, out_dtype: torch.dtype = torch.float32,
                      bad_count: torch.Tensor | None = None) -> torch.Tensor:
    """decode_tokens for FSQ's implicit codebook: valid ids are [0, prod(levels)) (vqb_fsq_decode_tokens)."""
    lib = _lib.load()
    dev = _cuda(ids, bad_count)
    b, id_bytes, z = _decode_out(ids, hw, p.D, out_dtype, bad_count)
    _call('vqb_fsq_decode_tokens', lib.vqb_fsq_decode_tokens, dev, _p(ids), id_bytes, b, hw, ctypes.byref(p), _p(z),
          _dt(z), _p(bad_count), _S)
    return z


# ---- residual quantization (csrc/quantize.cu, csrc/layout.cu) ------------------------------------------------------


def _residual_levels(Ws, gWs=None, g4s=None) -> ResidualLevels:
    """The vqb_residual_levels struct (host memory, copied by value into the kernel parameters)."""
    if not 1 <= len(Ws) <= MAX_LEVELS:
        raise ValueError(f'residual quantization takes 1..{MAX_LEVELS} levels, got {len(Ws)}')
    p = ResidualLevels()
    p.L = len(Ws)
    for l, W in enumerate(Ws):
        p.W[l] = W.data_ptr()
        if gWs is not None and gWs[l] is not None:
            p.gW[l] = gWs[l].data_ptr()
        if g4s is not None:
            for k, g in enumerate(g4s[l]):
                if g is not None:
                    p.g[l][k] = g.data_ptr()
    return p


def _codebooks(Ws) -> tuple[int, int]:
    K, D = Ws[0].shape
    for W in Ws:
        if W.dtype != torch.float32 or tuple(W.shape) != (K, D):
            raise TypeError(f'every level codebook must be a float32 [{K}, {D}] tensor, got {W.dtype} {tuple(W.shape)}')
    return K, D


def residual_step(r: torch.Tensor, x: torch.Tensor, W: torch.Tensor, mse4: torch.Tensor, *, level: int, L: int,
                  quant: torch.Tensor | None = None, keys: torch.Tensor | None = None, key_offset: int = 0,
                  quant_out: torch.Tensor | None = None, zhat: torch.Tensor | None = None,
                  r_out: torch.Tensor | None = None, z_out: torch.Tensor | None = None, z_hw: int = 0,
                  want_norm: bool = False) -> None:
    """One level of the residual chain (vqb_residual_step), into the caller's buffers: quant_out int64 [N, L]
    (column `level`), zhat fp32 [N, D], r_out fp32 [N, D] (None at the last level), z_out fp32 [N, D] or NCHW
    (last level only), mse4 fp32 [4] (this level's terms).  r is x at level 0 and the previous r_out after."""
    lib = _lib.load()
    dev = _cuda(r, x, W, mse4, quant, keys, quant_out, zhat, r_out, z_out)
    assert W.dtype == torch.float32 and (quant is None) != (keys is None) and mse4.dtype == torch.float32
    assert quant_out is None or (quant_out.dtype == torch.int64 and quant_out.shape == (x.shape[0], L))
    N, D = x.shape
    partials, ticket = _loss_ws(x.device)
    _call('vqb_residual_step', lib.vqb_residual_step, dev, _p(r), _dt(r), _p(x), _dt(x), N, D, _p(W), W.shape[0],
          _p(quant), _p(keys), key_offset, _p(quant_out), L, level, _p(zhat), _p(r_out), _p(z_out), z_hw,
          int(want_norm), _p(mse4), _p(partials), _p(ticket), _S)


def residual_backward(g_z: torch.Tensor, x: torch.Tensor, Ws, quant: torch.Tensor, g4s, *, want_norm: bool,
                      need_gW, g_hw: int = 0, deterministic: bool | None = None):
    """Backward of the whole residual depth in one launch (vqb_residual_backward).  Ws: the L codebooks as used by the
    forward; quant: int64 [N, L]; g4s: per level four 0-dim fp32 device tensors / None (codebook, commitment,
    codebook-norm, commitment-norm upstream gradients); need_gW: per level bool.
    deterministic: None follows torch.are_deterministic_algorithms_enabled(); when on, each gW_l is the segment sum of
    the level's per-token rows (vqb_residual_backward_rows + vqb_code_sort + vqb_segment_sum_rows, the contract of
    quantize_backward).  -> (gx in x's dtype, [gW_l fp32 [K, D] or None])"""
    lib = _lib.load()
    L = len(Ws)
    dev = _cuda(g_z, x, quant, *Ws, *[g for g4 in g4s for g in g4])
    K, D = _codebooks(Ws)
    N = x.shape[0]
    assert x.shape[1] == D and quant.dtype == torch.int64 and quant.shape == (N, L) and len(g4s) == L
    assert all(g is None or g.dtype == torch.float32 for g4 in g4s for g in g4)
    if not (g_z.dtype == torch.float32 or (g_z.dtype == torch.bfloat16 and x.dtype == torch.bfloat16)):
        g_z = g_z.float()
    gx = torch.empty_like(x)
    gWs = [torch.zeros_like(W) if need else None for W, need in zip(Ws, need_gW)]
    if any(need_gW) and deterministic_enabled(deterministic):
        rows = _det_ws(x.device, 'gw_rows', L * N * D, torch.float32).view(L, N, D)
        p = _residual_levels(Ws, list(rows), g4s)
        _call('vqb_residual_backward_rows', lib.vqb_residual_backward_rows, dev, _p(g_z), _dt(g_z), _p(x), _dt(x),
              ctypes.byref(p), K, _p(quant), N, D, int(want_norm), _p(gx), g_hw, _S)
        by_level = quant.view(L, N) if L == 1 else transpose_last2(quant.view(1, N, L)).view(L, N)
        for l, gW in enumerate(gWs):
            if gW is not None:
                order, offsets = _code_sort_ws(dev, N, K, by_level[l], None, 0)
                _segment_sum(dev, rows[l], N, D, False, order, offsets, K, gW, None)
        return gx, gWs
    p = _residual_levels(Ws, gWs, g4s)
    _call('vqb_residual_backward', lib.vqb_residual_backward, dev, _p(g_z), _dt(g_z), _p(x), _dt(x), ctypes.byref(p), K,
          _p(quant), N, D, int(want_norm), _p(gx), g_hw, _S)
    return gx, gWs


def decode_residual_tokens(Ws, ids: torch.Tensor, hw: int, out_dtype: torch.dtype = torch.float32,
                           bad_count: torch.Tensor | None = None) -> torch.Tensor:
    """Residual token ids [b, h, w, L] (uint16 / int32 / int64; a token's L ids contiguous) -> z = sum_l W_l[id_l]
    (level order, fp32 adds) as [b, D, h, w] of `out_dtype`, in one launch (vqb_decode_residual_tokens).  A token with
    an id outside [0, K) at any level gives a NaN row and is counted once into `bad_count`."""
    lib = _lib.load()
    dev = _cuda(ids, bad_count, *Ws)
    K, D = _codebooks(Ws)
    L = len(Ws)
    if ids.dim() < 2 or ids.shape[-1] != L:
        raise ValueError(f'expected residual token ids with a trailing depth axis of {L}, got {tuple(ids.shape)}')
    b, id_bytes, z = _decode_out(ids.select(-1, 0), hw, D, out_dtype, bad_count)
    p = _residual_levels(Ws)
    _call('vqb_decode_residual_tokens', lib.vqb_decode_residual_tokens, dev, _p(ids), id_bytes, b, hw, ctypes.byref(p),
          K, D, _p(z), _dt(z), _p(bad_count), _S)
    return z


# ---- grouped (product) quantization (csrc/quantize.cu, csrc/layout.cu) ---------------------------------------------


def _group_codebooks(Ws) -> tuple[int, int]:
    if not 1 <= len(Ws) <= MAX_LEVELS:
        raise ValueError(f'grouped quantization takes 1..{MAX_LEVELS} groups, got {len(Ws)}')
    return _codebooks(Ws)


def split_groups(x: torch.Tensor, G: int) -> torch.Tensor:
    """Latents [b, G*Dg, h, w] or tokens [N, G*Dg] (fp32 / bf16) -> [G, N, Dg] in one launch (vqb_split_groups): group g
    is the contiguous token slice x_g, N = b*h*w tokens in `b h w` order."""
    lib = _lib.load()
    dev = _cuda(x)
    if x.dim() not in (2, 4):
        raise ValueError(f'expected latents [b, c, h, w] or tokens [N, c], got {tuple(x.shape)}')
    if not 1 <= G <= MAX_LEVELS or x.shape[1] % G:
        raise ValueError(f'{x.shape[1]} channels do not split into {G} groups (1 <= G <= {MAX_LEVELS})')
    b, D = x.shape[0], x.shape[1]
    hw = x.shape[2] * x.shape[3] if x.dim() == 4 else 1
    out = torch.empty((G, b * hw, D // G), dtype=x.dtype, device=x.device)
    _call('vqb_split_groups', lib.vqb_split_groups, dev, _p(x), _dt(x), b, G, D // G, hw, _p(out), _S)
    return out


def _group_loss_ws(device):
    """Per-group partials + self-resetting tickets of the loss reduction (MAX_LEVELS groups), one set per
    (device, stream) like `_loss_ws`."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, 'groups')
    if key not in _WS:
        lib = _lib.load()
        _WS[key] = (torch.empty((MAX_LEVELS * int(lib.vqb_loss_partials_count()),), dtype=torch.float32, device=device),
                    torch.zeros((MAX_LEVELS,), dtype=torch.int32, device=device))
    return _WS[key]


def group_gather_ste_loss(xs: torch.Tensor, Ws, *, quant: torch.Tensor | None = None, keys: torch.Tensor | None = None,
                          want_norm: bool, quant_out: torch.Tensor | None = None, z_out: torch.Tensor | None = None,
                          z_hw: int = 0):
    """Every group's gather + STE + loss in one launch (vqb_group_gather_ste_loss).  xs: split tokens [G, N, Dg];
    quant (int64) or keys (packed): group-major [G, N].  quant_out: optional int64 [N, G]; z_out: fp32 [N, G*Dg], or
    NCHW [b, G*Dg, h, w] with z_hw = h*w (allocated token-major when None).  -> (z, mse fp32 [G, 4])"""
    lib = _lib.load()
    dev = _cuda(xs, quant, keys, quant_out, z_out, *Ws)
    K, Dg = _group_codebooks(Ws)
    G, N = len(Ws), xs.shape[1]
    if xs.dim() != 3 or tuple(xs.shape) != (G, N, Dg):
        raise ValueError(f'expected split tokens [{G}, N, {Dg}], got {tuple(xs.shape)}')
    index = quant if quant is not None else keys
    assert (quant is None) != (keys is None) and index.dtype == torch.int64 and index.shape == (G, N)
    assert quant_out is None or (quant_out.dtype == torch.int64 and quant_out.shape == (N, G))
    if z_out is None:
        z_out = torch.empty((N, G * Dg), dtype=torch.float32, device=xs.device)
    assert z_out.dtype == torch.float32 and z_out.numel() == N * G * Dg
    mse = torch.empty((G, 4), dtype=torch.float32, device=xs.device)
    partials, tickets = _group_loss_ws(xs.device)
    p = _residual_levels(Ws)
    _call('vqb_group_gather_ste_loss', lib.vqb_group_gather_ste_loss, dev, _p(xs), _dt(xs), N, Dg, ctypes.byref(p), K,
          _p(quant), _p(keys), _p(quant_out), _p(z_out), z_hw, int(want_norm), _p(mse), _p(partials), _p(tickets), _S)
    return z_out, mse


def group_backward(g_z: torch.Tensor, xs: torch.Tensor, Ws, quant: torch.Tensor, g4s, *, want_norm: bool, need_gW,
                   g_hw: int = 0, deterministic: bool | None = None):
    """Backward of every group in one launch (vqb_group_backward).  g_z: fp32 (or bf16 with bf16 tokens) [N, G*Dg], or
    NCHW with g_hw = h*w (gx then has g_z's NCHW shape); xs: the forward's split tokens [G, N, Dg]; quant: int64 [N, G];
    g4s: per group four 0-dim fp32 device tensors / None; need_gW: per group bool.
    deterministic: None follows torch.are_deterministic_algorithms_enabled(); when on, each gW_g is the segment sum of
    the group's per-token rows (vqb_group_backward_rows + vqb_code_sort + vqb_segment_sum_rows, the contract of
    quantize_backward).  -> (gx in xs's dtype with g_z's shape, [gW_g fp32 [K, Dg] or None])"""
    lib = _lib.load()
    G = len(Ws)
    dev = _cuda(g_z, xs, quant, *Ws, *[g for g4 in g4s for g in g4])
    K, Dg = _group_codebooks(Ws)
    N = xs.shape[1]
    assert tuple(xs.shape) == (G, N, Dg) and quant.dtype == torch.int64 and quant.shape == (N, G) and len(g4s) == G
    assert g_z.numel() == N * G * Dg and all(g is None or g.dtype == torch.float32 for g4 in g4s for g in g4)
    if not (g_z.dtype == torch.float32 or (g_z.dtype == torch.bfloat16 and xs.dtype == torch.bfloat16)):
        g_z = g_z.float()
    gx = torch.empty(g_z.shape, dtype=xs.dtype, device=xs.device)
    gWs = [torch.zeros_like(W) if need else None for W, need in zip(Ws, need_gW)]
    if any(need_gW) and deterministic_enabled(deterministic):
        rows = _det_ws(xs.device, 'gw_rows', G * N * Dg, torch.float32).view(G, N, Dg)
        p = _residual_levels(Ws, list(rows), g4s)
        _call('vqb_group_backward_rows', lib.vqb_group_backward_rows, dev, _p(g_z), _dt(g_z), _p(xs), _dt(xs),
              ctypes.byref(p), K, _p(quant), N, Dg, int(want_norm), _p(gx), g_hw, _S)
        by_group = quant.view(G, N) if G == 1 else transpose_last2(quant.view(1, N, G)).view(G, N)
        for g, gW in enumerate(gWs):
            if gW is not None:
                order, offsets = _code_sort_ws(dev, N, K, by_group[g], None, 0)
                _segment_sum(dev, rows[g], N, Dg, False, order, offsets, K, gW, None)
        return gx, gWs
    p = _residual_levels(Ws, gWs, g4s)
    _call('vqb_group_backward', lib.vqb_group_backward, dev, _p(g_z), _dt(g_z), _p(xs), _dt(xs), ctypes.byref(p), K,
          _p(quant), N, Dg, int(want_norm), _p(gx), g_hw, _S)
    return gx, gWs


def decode_group_tokens(Ws, ids: torch.Tensor, hw: int, out_dtype: torch.dtype = torch.float32,
                        bad_count: torch.Tensor | None = None) -> torch.Tensor:
    """Grouped token ids [b, h, w, G] (uint16 / int32 / int64; a token's G ids contiguous) -> z with channels
    [g*Dg, (g+1)*Dg) = W_g[id_g], as [b, G*Dg, h, w] of `out_dtype`, in one launch (vqb_decode_group_tokens).  A token
    with an id outside [0, K) in any group gives a NaN row and is counted once into `bad_count`."""
    lib = _lib.load()
    dev = _cuda(ids, bad_count, *Ws)
    K, Dg = _group_codebooks(Ws)
    G = len(Ws)
    if ids.dim() < 2 or ids.shape[-1] != G:
        raise ValueError(f'expected grouped token ids with a trailing group axis of {G}, got {tuple(ids.shape)}')
    b, id_bytes, z = _decode_out(ids.select(-1, 0), hw, G * Dg, out_dtype, bad_count)
    p = _residual_levels(Ws)
    _call('vqb_decode_group_tokens', lib.vqb_decode_group_tokens, dev, _p(ids), id_bytes, b, hw, ctypes.byref(p), K, Dg,
          _p(z), _dt(z), _p(bad_count), _S)
    return z
