"""tokenizer.decode_from_quant: token ids [b, h, w] -> NCHW latents (vq/tasks/image_reconstruction/models.py:97-108)
for VQ and FSQ codebooks, in one launch that reads uint16 / int32 / int64 ids and writes fp32 or bf16.  Every expected
value is computed on the CPU; out-of-range ids never reach torch's CUDA embedding (a device-side assert)."""
import itertools
import pathlib

import einops
import pytest
import torch
import torch.nn.functional as F

import vector_quantization_b200 as vqb
from oracle import oracle as O
from vector_quantization_b200 import ops, tokenizer
from vector_quantization_b200.callbacks import BaseCallback

pytestmark = pytest.mark.gpu
GOLDEN = pathlib.Path(__file__).parent / 'golden'
DTYPES = [torch.float32, torch.bfloat16]
DT_IDS = ['fp32', 'bf16']
_QUANTIZERS = {}


def model_decode_from_quant(weight_or_fsq, quant: torch.Tensor) -> torch.Tensor:
    """CPU restatement of the caller `decode_from_quant` before the decoder (vq/tasks/image_reconstruction/models.py:
    97-108): the quantizer's decode of the token grid quant [b, h, w] (`nn.Embedding`, i.e. `F.embedding`, or the
    oracle's `FSQ.decode`), then rearrange 'b h w c -> b c h w' + contiguous.  The line range and the rearrange are
    taken from SURVEY.md §1 and the a5 row of its hot-path table; they have not been re-read against the reference
    source."""
    if isinstance(weight_or_fsq, O.FSQ):
        z = weight_or_fsq.decode(quant)
    else:
        z = F.embedding(quant, weight_or_fsq)
    return einops.rearrange(z, 'b h w c -> b c h w').contiguous()


def _vq(K, D, dev, callbacks=()):
    """A VectorQuantizer with a seeded N(0, 1) codebook (cached per shape); returns (quantizer, CPU codebook)."""
    key = (K, D, tuple(type(c).__name__ for c in callbacks))
    if key not in _QUANTIZERS:
        W = torch.randn(K, D, generator=torch.Generator().manual_seed(K + 7 * D))
        q = vqb.build_quantizer(dict(type='VectorQuantizer', distance=dict(type='L2Distance'), callbacks=list(callbacks),
                                     embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K,
                                                    embedding_dim=D))).to(dev)
        with torch.no_grad():
            q.embedding.weight.copy_(W)
        _QUANTIZERS[key] = (q, W)
    return _QUANTIZERS[key]


def _fsq(levels, dev):
    return vqb.build_quantizer(dict(type='FiniteScalarQuantizer', num_scalars_per_channel=levels)).to(dev)


def _ids(shape, K, seed):
    """int64 CPU ids in [0, K), the first 0 and the last K - 1 (for K = 70 000: an id above 65 535 in every shape)."""
    q = torch.randint(0, K, shape, generator=torch.Generator().manual_seed(seed))
    q.view(-1)[0] = 0
    q.view(-1)[-1] = K - 1
    return q


_VQ_IDS = [(K, dt) for K, dt in itertools.product([512, 8192, 70000], [torch.uint16, torch.int32, torch.int64])
           if not (dt == torch.uint16 and K > 65536)]


@pytest.mark.parametrize('out_dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('K,id_dtype', _VQ_IDS, ids=[f'K{K}-{str(dt)[6:]}' for K, dt in _VQ_IDS])
@pytest.mark.parametrize('D', [8, 32, 33, 256, 768])
@pytest.mark.parametrize('bhw', [(2, 16, 16), (3, 5, 7), (1, 1, 1), (64, 16, 16)], ids=lambda s: 'x'.join(map(str, s)))
def test_vq_decode_matches_oracle_bit_for_bit(dev, bhw, D, K, id_dtype, out_dtype):
    q, W = _vq(K, D, dev)
    ids = _ids(bhw, K, seed=D + K)
    ref = model_decode_from_quant(W, ids)
    with torch.no_grad():
        z, memo = tokenizer.decode_from_quant(q, ids.to(id_dtype).to(dev), dict(), dtype=out_dtype)
    b, h, w = bhw
    assert z.shape == (b, D, h, w) and z.dtype == out_dtype and z.is_contiguous()
    assert torch.equal(z.cpu(), ref.to(out_dtype))
    assert memo['quantizer']['decode'] == {}


_FSQ_CASES = [([8, 8, 5, 5, 5], (5, 40, 40)), ([8, 8, 5, 5, 5], (64, 5, 25)), ([8, 8, 8, 5, 5, 5], (10, 80, 80))]


@pytest.mark.parametrize('out_dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('id_dtype', [torch.uint16, torch.int32, torch.int64], ids=['uint16', 'int32', 'int64'])
@pytest.mark.parametrize('levels,bhw', _FSQ_CASES, ids=['8000-40x40', '8000-5x25', '64000-80x80'])
def test_fsq_decode_every_id_bit_for_bit(dev, levels, bhw, id_dtype, out_dtype):
    """Every id of the implicit codebook, against the oracle's FSQ.decode and against ops.fsq_decode + a permute."""
    fsq = O.FSQ(levels)
    q = _fsq(levels, dev)
    ids = torch.arange(fsq.codebook_size).view(bhw)
    with torch.no_grad():
        z, _ = tokenizer.decode_from_quant(q, ids.to(id_dtype).to(dev), dict(), dtype=out_dtype)
    assert z.shape == (bhw[0], len(levels)) + bhw[1:] and z.dtype == out_dtype
    assert torch.equal(z.cpu(), model_decode_from_quant(fsq, ids).to(out_dtype))
    rows = ops.fsq_decode(ids.to(torch.int32).to(dev), q._params)
    assert torch.equal(z, rows.permute(0, 3, 1, 2).to(out_dtype))


def test_vq_round_trip_through_a_token_dump(dev, tmp_path):
    """encode_to_quant(compact=True) -> save_tokens -> load_tokens -> decode_from_quant gives W[ids] in NCHW; the
    compact (uint16) and int64 encodings decode identically."""
    rec = torch.load(GOLDEN / 'vqgan_l2.pt', weights_only=False)
    q = vqb.build_quantizer(rec['config'], training=False).to(dev)
    q._forward_pre_hooks.clear()
    step = rec['steps'][0]
    with torch.no_grad():
        q.embedding.weight.copy_(step['W_before'])
    b, h, w, D = 2, 16, 16, rec['D']
    x = step['x'].to(dev).view(b, h, w, D).permute(0, 3, 1, 2).contiguous()
    compact, memo = tokenizer.encode_to_quant(q, x, dict(), compact=True)
    assert compact.dtype == torch.uint16
    tokenizer.save_tokens(tmp_path / '1_0.pth', ['a', 'b'], torch.tensor([3, 7]), compact, memo['quantizer']['x_shape'])
    tokens = tokenizer.load_tokens(tmp_path / '1_0.pth')['tokens']
    W = q.embedding.weight.detach().cpu()
    with torch.no_grad():
        z, _ = tokenizer.decode_from_quant(q, tokens.to(dev), dict())
        z_compact, _ = tokenizer.decode_from_quant(q, compact, dict())
    assert torch.equal(z.cpu(), W[tokens].permute(0, 3, 1, 2))
    assert torch.equal(z_compact, z)


def test_fsq_round_trip_through_a_token_dump(dev, tmp_path):
    rec = torch.load(GOLDEN / 'fsq_64000.pt', weights_only=False)
    q = _fsq(rec['levels'], dev)
    b, h, w, D = 4, 16, 16, len(rec['levels'])
    x = rec['x'].to(dev).view(b, h, w, D).permute(0, 3, 1, 2).contiguous()
    compact, memo = tokenizer.encode_to_quant(q, x, dict(), compact=True)
    assert compact.dtype == torch.int32
    tokenizer.save_tokens(tmp_path / '1_0.pth', ['a'] * b, torch.arange(b), compact, memo['quantizer']['x_shape'])
    tokens = tokenizer.load_tokens(tmp_path / '1_0.pth')['tokens']
    table = q.embeddings.cpu()                       # the implicit codebook, fsq/quantizers.py:90-93
    with torch.no_grad():
        z, _ = tokenizer.decode_from_quant(q, tokens.to(dev), dict())
        z_compact, _ = tokenizer.decode_from_quant(q, compact, dict())
    assert torch.equal(z.cpu(), table[tokens].permute(0, 3, 1, 2))
    assert torch.equal(z_compact, z)


@pytest.mark.parametrize('kind', ['vq', 'fsq'])
def test_fused_path_is_one_launch_without_transpose(dev, kind):
    if kind == 'vq':
        q, _ = _vq(8192, 256, dev)
        ids, name = _ids((4, 16, 16), 8192, seed=1).to(torch.uint16).to(dev), 'vqb_decode_tokens'
    else:
        q = _fsq([8, 8, 8, 5, 5, 5], dev)
        ids, name = _ids((4, 16, 16), 64000, seed=1).to(torch.int32).to(dev), 'vqb_fsq_decode_tokens'
    ops.PROFILE = []
    try:
        with torch.no_grad():
            tokenizer.decode_from_quant(q, ids, dict(), dtype=torch.bfloat16)
        torch.cuda.synchronize()
        names = [n for n, _, _ in ops.PROFILE]
    finally:
        ops.PROFILE = None
    assert names == [name]


class _ScaleAfterDecode(BaseCallback):
    def after_decode(self, z, memo):
        memo['scaled'] = True
        return z * 3


@pytest.mark.parametrize('out_dtype', DTYPES, ids=DT_IDS)
def test_after_decode_hook_is_honoured(dev, out_dtype):
    q, W = _vq(512, 32, dev, callbacks=(_ScaleAfterDecode(),))
    plain, _ = _vq(512, 32, dev)
    ids = _ids((3, 5, 7), 512, seed=5)
    ids_dev = ids.to(torch.int32).to(dev)
    with torch.no_grad():
        z, memo = tokenizer.decode_from_quant(q, ids_dev, dict(), dtype=out_dtype)
        rows, _ = q.decode(ids.to(dev), dict())
        z_plain, _ = tokenizer.decode_from_quant(plain, ids_dev, dict(), dtype=out_dtype)
    assert memo['quantizer']['scaled'] is True
    assert torch.equal(z, rows.permute(0, 3, 1, 2).contiguous().to(out_dtype))
    assert torch.equal(z.cpu(), (model_decode_from_quant(W, ids) * 3).to(out_dtype))
    if out_dtype == torch.float32:      # the hook's product of the one-launch rows (bf16 rounds after the hook)
        assert torch.equal(z, z_plain * 3)


@pytest.mark.parametrize('out_dtype', DTYPES, ids=DT_IDS)
def test_codebook_gradient_fallback(dev, out_dtype):
    """Grad enabled and a codebook that requires grad: the differentiable gather; dL/dW is the CPU F.embedding
    gradient, and the values equal the one-launch path."""
    q, W = _vq(512, 33, dev)
    ids = _ids((3, 5, 7), 512, seed=11)
    ids_dev = ids.to(torch.uint16).to(dev)
    q.embedding.weight.grad = None
    z, _ = tokenizer.decode_from_quant(q, ids_dev, dict(), dtype=out_dtype)
    assert z.requires_grad and z.dtype == out_dtype and z.shape == (3, 33, 5, 7)
    g = torch.randn(z.shape, generator=torch.Generator().manual_seed(2))
    (z.float() * g.to(dev)).sum().backward()
    W_ref = W.clone().requires_grad_(True)
    (model_decode_from_quant(W_ref, ids).to(out_dtype).float() * g).sum().backward()
    torch.testing.assert_close(q.embedding.weight.grad.cpu(), W_ref.grad, rtol=1e-5, atol=0)
    q.embedding.weight.grad = None
    with torch.no_grad():
        z_fused, _ = tokenizer.decode_from_quant(q, ids_dev, dict(), dtype=out_dtype)
    assert torch.equal(z.detach(), z_fused)


def _bad_ids(kind, id_dtype):
    """(quantizer args, ids int64 CPU [3, 5, 7], bad mask, codebook size)."""
    size = 512 if kind == 'vq' else 8000
    ids = _ids((3, 5, 7), size, seed=13)
    flat = ids.view(-1)
    if id_dtype == torch.uint16:
        bad = {0: 65535, 50: 65535}
    elif kind == 'vq':
        bad = {0: size, 17: size + 5, 104: -1}
    else:
        bad = {3: size, 104: -1}
    for i, v in bad.items():
        flat[i] = v
    mask = torch.zeros(flat.numel(), dtype=torch.bool)
    mask[list(bad)] = True
    return ids, mask.view(3, 5, 7), size


@pytest.mark.parametrize('kind,id_dtype', [('vq', torch.int32), ('vq', torch.int64), ('vq', torch.uint16),
                                           ('fsq', torch.int32), ('fsq', torch.int64)],
                         ids=['vq-int32', 'vq-int64', 'vq-uint16', 'fsq-int32', 'fsq-int64'])
def test_out_of_range_ids_are_reported_not_clamped(dev, kind, id_dtype):
    """check=True raises IndexError with the exact count; check=False gives NaN in every channel of exactly those
    tokens and bit-exact rows elsewhere; afterwards an ordinary decode still works."""
    ids, mask, size = _bad_ids(kind, id_dtype)
    if kind == 'vq':
        q, W = _vq(size, 32, dev)
        book = W
    else:
        q = _fsq([8, 8, 5, 5, 5], dev)
        book = O.FSQ([8, 8, 5, 5, 5])
    ids_dev = (ids.to(torch.int32).to(torch.uint16) if id_dtype == torch.uint16 else ids.to(id_dtype)).to(dev)
    n_bad = int(mask.sum())
    with torch.no_grad():
        with pytest.raises(IndexError, match=rf'^{n_bad} token id\(s\) outside \[0, {size}\)'):
            tokenizer.decode_from_quant(q, ids_dev, dict())
        z, _ = tokenizer.decode_from_quant(q, ids_dev, dict(), check=False)
    rows = z.cpu().permute(0, 2, 3, 1)                                   # [b, h, w, c]
    assert torch.isnan(rows[mask]).all()
    ref = model_decode_from_quant(book, ids.masked_fill(mask, 0)).permute(0, 2, 3, 1)
    assert not torch.isnan(rows[~mask]).any() and torch.equal(rows[~mask], ref[~mask])
    if kind == 'vq':        # the differentiable fallback checks the ids before the gather
        with pytest.raises(IndexError, match=rf'^{n_bad} token'):
            tokenizer.decode_from_quant(q, ids_dev, dict())
    good = ids.masked_fill(mask, 1)
    with torch.no_grad():
        z_good, _ = tokenizer.decode_from_quant(q, good.to(dev), dict())
    torch.cuda.synchronize()
    assert torch.equal(z_good.cpu(), model_decode_from_quant(book, good))


def test_cuda_graph_replay_matches_eager(dev):
    q, W = _vq(8192, 256, dev)
    ids = _ids((4, 16, 16), 8192, seed=21).to(torch.uint16).to(dev)
    with torch.no_grad():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                                     # warm-up outside the capture
            tokenizer.decode_from_quant(q, ids, dict(), dtype=torch.bfloat16, check=False)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            z_static, _ = tokenizer.decode_from_quant(q, ids, dict(), dtype=torch.bfloat16, check=False)
        new = _ids((4, 16, 16), 8192, seed=22)
        ids.copy_(new.to(torch.int32).to(torch.uint16).to(dev))
        graph.replay()
        torch.cuda.synchronize()
        z_eager, _ = tokenizer.decode_from_quant(q, ids, dict(), dtype=torch.bfloat16)
    assert torch.equal(z_static, z_eager)
    assert torch.equal(z_eager.cpu(), model_decode_from_quant(W, new).to(torch.bfloat16))
