"""ctypes binding of the C-ABI in `include/vqb200.h` (libvqb200.so, built in-tree by
`__graft_entry__.build()` / `csrc/Makefile`).

There is no CPU implementation and no fallback: if the shared library is missing, or a call is
made with tensors that are not on a CUDA device, this module raises.
"""
from __future__ import annotations

import ctypes
import os
import pathlib
import subprocess
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int64, c_size_t, c_ubyte, c_void_p

_HERE = pathlib.Path(__file__).resolve().parent
# VQB200_LIB: developer override, e.g. to A/B two builds of the library on the same GPU box
LIB_PATH = pathlib.Path(os.environ['VQB200_LIB']) if os.environ.get('VQB200_LIB') else _HERE / 'libvqb200.so'
CSRC = _HERE / 'csrc'

ABI_VERSION = 3
VQB_F32, VQB_BF16 = 0, 1
BACKEND_TCGEN05, BACKEND_SIMT = 0, 1
PLANES_F16 = 0x11     # VQB_PLANES_F16: one fp16 plane of a bf16 source
PLANES_F16X2 = 0x12   # VQB_PLANES_F16X2: the fp16 (hi, lo * 2^11) plane pair


class VQBError(RuntimeError):
    pass


class FSQParams(Structure):
    _fields_ = [('D', c_int), ('max_', c_float * 16), ('odd', c_float * 16), ('shift', c_float * 16),
                ('half', c_float * 16), ('cumprod', c_int * 16), ('levels', c_int * 16)]


MAX_LEVELS = 16   # VQB_MAX_LEVELS


class ResidualLevels(Structure):
    """vqb_residual_levels: the per-level device pointers, passed by value into the kernels."""
    _fields_ = [('L', c_int), ('W', c_void_p * MAX_LEVELS), ('gW', c_void_p * MAX_LEVELS),
                ('g', (c_void_p * 4) * MAX_LEVELS)]


# name -> (restype, argtypes); must list EVERY symbol declared in include/vqb200.h
# (tests/test_abi.py parses the header and checks this table and the .so against it).
SIGNATURES = {
    'vqb_abi_version': (c_int, []),
    'vqb_last_error': (c_char_p, []),
    'vqb_device_info': (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    'vqb_operand_dp': (c_int64, [c_int]),
    'vqb_operand_rows_pad': (c_int64, [c_int64]),
    'vqb_operand_bytes': (c_size_t, [c_int64, c_int, c_int]),
    'vqb_pack_rows': (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    'vqb_assign_ex': (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p,
                              c_int, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    'vqb_certify_workspace_bytes': (c_int64, [c_int64]),
    'vqb_certify': (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                            c_void_p, c_void_p]),
    'vqb_cvq_needy_codes': (c_int, [c_void_p, c_void_p, c_float, c_int64, c_float, c_float, c_float, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p]),
    'vqb_gather_plane_rows': (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                      c_void_p]),
    'vqb_gather_f32': (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    'vqb_scatter_keys': (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    'vqb_assign': (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_int, c_int64, c_int64, c_int, c_void_p,
                           c_int, c_int64, c_void_p, c_int, c_void_p]),
    'vqb_row_inv_norm': (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p]),
    'vqb_fold_l2_side': (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_void_p]),
    'vqb_pack_rows_fold': (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                           c_void_p, c_int64, c_int, c_void_p]),
    'vqb_unpack_keys': (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    'vqb_compact_tokens': (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int, c_void_p]),
    'vqb_transpose_last2': (c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    'vqb_keys_flip_sign': (c_int, [c_void_p, c_int64, c_void_p]),
    'vqb_loss_partials_count': (c_int64, []),
    'vqb_gather_ste_loss': (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p,
                                    c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    'vqb_quantize_backward': (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_int64, c_int,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    'vqb_quantize_backward_rows': (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_int64,
                                           c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int64,
                                           c_void_p]),
    'vqb_quantize_backward_rotated': (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p,
                                              c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                              c_void_p, c_int64, c_void_p]),
    'vqb_quantize_backward_rotated_rows': (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p,
                                                   c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                                   c_void_p, c_void_p, c_int64, c_void_p]),
    'vqb_residual_step': (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p, c_int64, c_void_p, c_void_p,
                                  c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p,
                                  c_void_p, c_void_p, c_void_p]),
    'vqb_residual_backward': (c_int, [c_void_p, c_int, c_void_p, c_int, POINTER(ResidualLevels), c_int64, c_void_p,
                                      c_int64, c_int, c_int, c_void_p, c_int64, c_void_p]),
    'vqb_residual_backward_rows': (c_int, [c_void_p, c_int, c_void_p, c_int, POINTER(ResidualLevels), c_int64, c_void_p,
                                           c_int64, c_int, c_int, c_void_p, c_int64, c_void_p]),
    'vqb_group_gather_ste_loss': (c_int, [c_void_p, c_int, c_int64, c_int, POINTER(ResidualLevels), c_int64, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                          c_void_p]),
    'vqb_group_backward': (c_int, [c_void_p, c_int, c_void_p, c_int, POINTER(ResidualLevels), c_int64, c_void_p, c_int64,
                                   c_int, c_int, c_void_p, c_int64, c_void_p]),
    'vqb_group_backward_rows': (c_int, [c_void_p, c_int, c_void_p, c_int, POINTER(ResidualLevels), c_int64, c_void_p,
                                        c_int64, c_int, c_int, c_void_p, c_int64, c_void_p]),
    'vqb_group_backward_rotated': (c_int, [c_void_p, c_int, c_void_p, c_int, POINTER(ResidualLevels), c_int64, c_void_p,
                                           c_int64, c_int, c_int, c_void_p, c_int64, c_void_p]),
    'vqb_group_backward_rotated_rows': (c_int, [c_void_p, c_int, c_void_p, c_int, POINTER(ResidualLevels), c_int64,
                                                c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p]),
    'vqb_segment_chunk': (c_int64, []),
    'vqb_code_sort_scratch_bytes': (c_size_t, [c_int64, c_int64]),
    'vqb_code_sort': (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t,
                              c_void_p]),
    'vqb_segment_sum_scratch_bytes': (c_size_t, [c_int64, c_int64, c_int]),
    'vqb_segment_sum_rows': (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p,
                                     c_void_p, c_void_p, c_size_t, c_void_p]),
    'vqb_l2norm_forward': (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_void_p]),
    'vqb_l2norm_backward': (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_void_p]),
    'vqb_scatter_stats': (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                  c_void_p]),
    'vqb_bincount_accumulate': (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    'vqb_kmeans_ema_update': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_float, c_float, c_void_p]),
    'vqb_gather_rows_by_key': (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_int64, c_int64, c_void_p,
                                       c_void_p]),
    'vqb_cvq_update': (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_float,
                               c_float, c_float, c_void_p]),
    'vqb_embedding_gather': (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    'vqb_fsq_forward': (c_int, [c_void_p, c_int, c_int64, POINTER(FSQParams), c_void_p, c_int, c_void_p, c_void_p]),
    'vqb_fsq_backward': (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, POINTER(FSQParams), c_void_p, c_int,
                                 c_void_p]),
    'vqb_fsq_decode': (c_int, [c_void_p, c_int64, POINTER(FSQParams), c_void_p, c_void_p]),
    'vqb_decode_tokens': (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p,
                                  c_void_p]),
    'vqb_fsq_decode_tokens': (c_int, [c_void_p, c_int, c_int64, c_int64, POINTER(FSQParams), c_void_p, c_int, c_void_p,
                                      c_void_p]),
    'vqb_decode_residual_tokens': (c_int, [c_void_p, c_int, c_int64, c_int64, POINTER(ResidualLevels), c_int64, c_int,
                                           c_void_p, c_int, c_void_p, c_void_p]),
    'vqb_decode_group_tokens': (c_int, [c_void_p, c_int, c_int64, c_int64, POINTER(ResidualLevels), c_int64, c_int,
                                        c_void_p, c_int, c_void_p, c_void_p]),
    'vqb_split_groups': (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_int64, c_void_p, c_void_p]),
    'vqb_distance_matrix': (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    'vqb_comm_alloc': (c_int, [c_size_t, POINTER(c_void_p), POINTER(c_ubyte)]),
    'vqb_comm_open': (c_int, [POINTER(c_ubyte), POINTER(c_void_p)]),
    'vqb_comm_close': (c_int, [c_void_p]),
    'vqb_comm_free': (c_int, [c_void_p]),
    'vqb_comm_bind': (c_int, [c_void_p, POINTER(c_void_p), c_int, c_int]),
    'vqb_comm_kmeans_ema_update': (c_int, [c_void_p, c_int, c_int, c_size_t, c_size_t, c_size_t, c_size_t, c_int64, c_int,
                                           c_float, c_float, c_void_p]),
    'vqb_comm_cvq_update': (c_int, [c_void_p, c_int, c_int, c_size_t, c_size_t, c_size_t, c_size_t, c_size_t, c_int64,
                                    c_int, c_float, c_float, c_float, c_void_p]),
    'vqb_comm_allreduce_min_keys': (c_int, [c_void_p, c_int, c_int, c_size_t, c_int64, c_void_p]),
    'vqb_comm_allreduce_sum_f32': (c_int, [c_void_p, c_int, c_int, c_size_t, c_int64, c_void_p]),
}
COMM_HEADER_BYTES = 512
COMM_MAX_WORLD = 16
IPC_HANDLE_BYTES = 64

_lib = None


def build(force: bool = False, verbose: bool = False) -> pathlib.Path:
    """Compile libvqb200.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    if LIB_PATH.exists() and not force:
        srcs = list(CSRC.glob('*.cu')) + list(CSRC.glob('*.cuh')) + [_HERE.parent / 'include' / 'vqb200.h']
        if all(s.stat().st_mtime <= LIB_PATH.stat().st_mtime for s in srcs):
            return LIB_PATH
    cmd = ['make', '-C', str(CSRC), '-j', str(min(8, os.cpu_count() or 1))]
    res = subprocess.run(cmd, capture_output=not verbose, text=True)
    if res.returncode != 0:
        raise VQBError(f'building libvqb200.so failed:\n{res.stdout}\n{res.stderr}')
    return LIB_PATH


def load() -> ctypes.CDLL:
    """Load the library (never builds implicitly: the GPU box uses the prebuilt in-tree .so)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise VQBError(
            f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` (or '
            f'`make -C {CSRC}`).  vector_quantization_b200 has no CPU or PyTorch fallback.')
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.vqb_abi_version() != ABI_VERSION:
        raise VQBError(f'ABI version mismatch: library reports {lib.vqb_abi_version()}, binding expects {ABI_VERSION}')
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().vqb_last_error()
        raise VQBError(f'{what} failed with status {status}: {msg.decode() if msg else ""}')
