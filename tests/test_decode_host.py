"""Host-side contract of decode_from_quant and of vqb_decode_tokens / vqb_fsq_decode_tokens (no GPU needed)."""
import ctypes

import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from tests.test_gpu_decode import model_decode_from_quant
from vector_quantization_b200 import _lib, ops, tokenizer


def _vq(K=16, D=4):
    return vqb.build_quantizer(dict(type='VectorQuantizer', distance=dict(type='L2Distance'),
                                    embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K,
                                                   embedding_dim=D)))


def test_decode_from_quant_is_exported():
    assert 'decode_from_quant' in tokenizer.__all__
    assert {'decode_tokens', 'fsq_decode_tokens'} <= set(ops.__all__)


def test_decode_from_quant_rejects_bad_rank_and_cpu_ids():
    q = _vq()
    with pytest.raises(ValueError, match=r'\[b, h, w\]'):
        tokenizer.decode_from_quant(q, torch.zeros(2, 3, dtype=torch.int64), dict())
    with pytest.raises(_lib.VQBError, match='CUDA'):
        tokenizer.decode_from_quant(q, torch.zeros(2, 3, 4, dtype=torch.int64), dict())
    with pytest.raises(_lib.VQBError, match='CUDA'):
        ops.decode_tokens(q.embedding.weight.detach(), torch.zeros(2, 3, 4, dtype=torch.int64), 12)


def test_c_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    assert lib.vqb_decode_tokens(None, 4, 1, 1, dummy, 16, 4, dummy, 0, None, None) == -1
    assert b'null pointer' in lib.vqb_last_error()
    assert lib.vqb_decode_tokens(dummy, 3, 1, 1, dummy, 16, 4, dummy, 0, None, None) == -1
    assert b'id_bytes' in lib.vqb_last_error()
    assert lib.vqb_decode_tokens(dummy, 4, 1, 1, dummy, 16, 4, dummy, 7, None, None) == -1
    assert b'out_dtype' in lib.vqb_last_error()
    assert lib.vqb_decode_tokens(dummy, 4, 1, 1, dummy, 0, 4, dummy, 0, None, None) == -1
    p = ops.fsq_params([8, 5, 5, 5], 1e-3)
    p.D = 0
    assert lib.vqb_fsq_decode_tokens(dummy, 4, 1, 1, ctypes.byref(p), dummy, 0, None, None) == -1
    assert b'D must be' in lib.vqb_last_error()


def test_decode_from_quant_restatement_is_gather_then_rearrange():
    W = torch.randn(10, 3, generator=torch.Generator().manual_seed(0))
    q = torch.tensor([[[0, 9], [4, 4]]])
    z = model_decode_from_quant(W, q)
    assert z.shape == (1, 3, 2, 2) and z.is_contiguous()
    assert torch.equal(z[0, :, 0, 1], W[9]) and torch.equal(z[0, :, 1, 0], W[4])
    fsq = O.FSQ([8, 5, 5, 5])
    ids = torch.arange(fsq.codebook_size).view(10, 10, 10)
    assert torch.equal(model_decode_from_quant(fsq, ids).permute(0, 2, 3, 1).reshape(-1, 4), fsq.embeddings)
