"""Host side of the deterministic reductions (no GPU needed): the switch, the contract constant and the argument checks
of the new entry points."""
import torch

from vector_quantization_b200 import _lib, ops


def test_switch_follows_torch_flag_at_call_time():
    prev = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        assert ops.deterministic_enabled() is False
        assert ops.deterministic_enabled(True) is True
        torch.use_deterministic_algorithms(True)
        assert ops.deterministic_enabled() is True
        assert ops.deterministic_enabled(False) is False
    finally:
        torch.use_deterministic_algorithms(prev)


def test_chunk_and_scratch_sizes():
    lib = _lib.load()
    assert lib.vqb_segment_chunk() == 256 == ops.segment_chunk()
    # code sort: two int32 ping-pong code arrays, one index array, 256 x tiles digit histogram (256-byte aligned)
    assert lib.vqb_code_sort_scratch_bytes(65536, 8192) == 3 * 65536 * 4 + 256 * 32 * 4
    # segment sum: (N / C + K + 1) partial rows + N inverse norms
    assert lib.vqb_segment_sum_scratch_bytes(65536, 8192, 32) == -(-(256 + 8192 + 1) * 32 * 4 // 256) * 256 + 65536 * 4
    assert lib.vqb_code_sort_scratch_bytes(0, 8) == 0


def test_entry_points_reject_bad_arguments_before_launching():
    lib = _lib.load()
    fake = 1 << 20   # never dereferenced: the checks fail first
    assert lib.vqb_code_sort(fake, None, 0, 1 << 31, 8, fake, fake, fake, 1 << 40, None) == -1
    assert b'2^31' in lib.vqb_last_error()
    assert lib.vqb_code_sort(fake, fake, 0, 10, 8, fake, fake, fake, 1 << 20, None) == -1
    assert b'exactly one' in lib.vqb_last_error()
    assert lib.vqb_code_sort(fake, None, 0, 10, 8, fake, fake, fake, 16, None) == -1
    assert b'scratch too small' in lib.vqb_last_error()
    assert lib.vqb_segment_sum_rows(fake, 0, 10, 8, 0, fake, fake, 4, fake, None, fake, 1, None) == -1
    assert b'scratch too small' in lib.vqb_last_error()
    assert lib.vqb_quantize_backward_rows(fake, 0, fake, 0, 0, fake, 4, fake, 10, 8, None, None, None, None, 0, fake,
                                          None, 0, None) == -1
    assert b'null gW_rows' in lib.vqb_last_error()
