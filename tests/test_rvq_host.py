"""ResidualVectorQuantizer without a GPU: config validation, state-dict layout, the C-ABI argument checks, the CPU
restatement (oracle/rvq.py) and token dumps with a trailing depth axis."""
import ctypes

import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rvq as R
from vector_quantization_b200 import _lib, ops, plugin, tokenizer

K, D = 16, 4


def _cfg(L=3, **level):
    node = dict(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D),
                losses=dict(vqgan_loss=dict(type='VQGANLoss')))
    node.update(level)
    return dict(type='ResidualVectorQuantizer', num_quantizers=L, quantizer=node)


def test_registered_and_exported():
    assert 'ResidualVectorQuantizer' in plugin.QUANTIZERS
    assert isinstance(vqb.VQITQuantizerRegistry.lookup('ResidualVectorQuantizer'), type)
    assert {'residual_step', 'residual_backward', 'decode_residual_tokens'} <= set(ops.__all__)


def test_properties_state_dict_and_init_weights_on_every_level():
    q = vqb.build_quantizer(dict(_cfg(3, callbacks=[dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'),
                                                          ema=dict())]), init_weights=dict(type='vqgan')))
    assert (q.num_quantizers, q.codebook_size, q.embedding_dim) == (3, K, D)
    assert q.embeddings.shape == (3, K, D)
    keys = set(q.state_dict())
    for l in range(3):
        assert f'_quantizers.{l}._embedding.weight' in keys and f'_quantizers.{l}._probability' in keys
        assert f'_quantizers.{l}._losses.vqgan_loss._weight._steps' in keys
    assert all(k.startswith('_quantizers.') for k in keys)
    # VQGANQuantizer's 'vqgan' init: uniform(-1/K, 1/K) on every level, independently drawn
    E = q.embeddings
    assert E.abs().max() <= 1.0 / K and not torch.equal(E[0], E[1])


@pytest.mark.parametrize('level,match', [
    (dict(callbacks=[dict(type='NormalizeCallback')]), 'NormalizeCallback rewrites the tokens'),
    (dict(callbacks=[dict(type='VQKDCallback', ema=dict())]), 'VQKDCallback rewrites the tokens'),
    (dict(callbacks=[dict(type='VQGAN_VQKDCallback', ema=dict())]), 'VQGAN_VQKDCallback rewrites the tokens'),
    (dict(callbacks=[dict(type='CVQVAECallback', anchor=dict(type='MultinomialAnchor'), ema=dict())]),
     'MultinomialAnchor'),
    (dict(losses=dict(entropy=dict(type='EntropyLoss', temperature=1.0))), 'EntropyLoss'),
    (dict(materialize_distance=True), 'materialize_distance'),
])
def test_rejected_level_configs_name_the_offending_item(level, match):
    with pytest.raises(ValueError, match=match):
        vqb.build_quantizer(_cfg(2, **level))


def test_rejects_callbacks_hooking_decode_or_loss():
    @vqb.VQITQuantizerCallbackRegistry.register_(force=True)
    class _HookDecodeForRVQTest(vqb.BaseCallback):
        def after_decode(self, z, memo):
            return z

    with pytest.raises(ValueError, match='_HookDecodeForRVQTest hooks after_decode'):
        vqb.build_quantizer(_cfg(2, callbacks=[dict(type='_HookDecodeForRVQTest')]))


@pytest.mark.parametrize('L', [0, 17, 2.0])
def test_rejects_depth_outside_1_to_16(L):
    with pytest.raises(ValueError, match='num_quantizers'):
        vqb.build_quantizer(_cfg(L))


def test_rejects_fsq_levels_and_top_level_losses():
    with pytest.raises(ValueError, match='FiniteScalarQuantizer'):
        vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=2,
                                 quantizer=dict(type='FiniteScalarQuantizer', num_scalars_per_channel=[8, 5, 5, 5])))
    with pytest.raises(ValueError, match='level config'):
        vqb.build_quantizer(dict(_cfg(2), losses=dict(c=dict(type='CodebookLoss'))))


def test_c_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    lv = ops._residual_levels([torch.zeros(K, D)] * 2)
    assert lib.vqb_residual_step(dummy, 0, dummy, 0, 8, D, dummy, K, dummy, None, 0, None, 2, 2, None, None, None, 0, 0,
                                 dummy, dummy, dummy, None) == -1
    assert b'level 2 of L=2' in lib.vqb_last_error()
    assert lib.vqb_residual_step(dummy, 0, dummy, 0, 8, D, dummy, K, dummy, None, 0, None, 2, 0, None, None, None, 0, 0,
                                 dummy, dummy, dummy, None) == -1
    assert b'r_out is required' in lib.vqb_last_error()
    lv.L = 17
    assert lib.vqb_residual_backward(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, None) == -1
    assert b'L=17' in lib.vqb_last_error()
    lv.L = 2
    assert lib.vqb_residual_backward_rows(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, None) == -1
    assert b'null gradient rows at level 0' in lib.vqb_last_error()
    assert lib.vqb_decode_residual_tokens(dummy, 3, 1, 1, ctypes.byref(lv), K, D, dummy, 0, None, None) == -1
    assert b'id_bytes' in lib.vqb_last_error()
    with pytest.raises(ValueError, match='1..16 levels'):
        ops._residual_levels([torch.zeros(K, D)] * 17)


def _restatement_inputs(L, N=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, D, generator=g)
    Ws = [torch.randn(K, D, generator=g) * 0.5 ** l for l in range(L)]
    return x, Ws


@pytest.mark.parametrize('loss', ['VQGANLoss', 'CodebookLoss', 'CommitmentLoss'])
@pytest.mark.parametrize('norm', [False, True])
@pytest.mark.parametrize('distance', ['L2', 'Cosine'])
def test_restatement_at_depth_one_is_the_single_level_oracle(distance, norm, loss):
    spec = O.QuantizerSpec(distance=distance, training=False, losses={'l': dict(type=loss, norm=norm)})
    x, Ws = _restatement_inputs(1)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    a = R.rvq_forward(spec, xa, Ws)
    b = O.quantizer_forward(spec, [xb], Ws[0])
    assert torch.equal(a['quant'][:, 0], b['quant'][0])
    assert torch.equal(a['z_ste'], b['z_ste'][0]) and torch.equal(a['loss'], b['loss'][0])
    (a['loss'] + a['z_ste'].square().sum()).backward()
    (b['loss'][0] + b['z_ste'][0].square().sum()).backward()
    ga, gb = a['weight_leafs'][0].grad, b['weight_leaf'].grad
    assert torch.equal(xa.grad, xb.grad) and ((ga is None and gb is None) or torch.equal(ga, gb))


def test_restatement_zhat_is_the_level_ordered_fp32_sum():
    spec = O.QuantizerSpec(distance='L2', training=False, losses={'l': dict(type='VQGANLoss')})
    x, Ws = _restatement_inputs(4)
    out = R.rvq_forward(spec, x, Ws)
    q = out['quant']
    acc = Ws[0][q[:, 0]]
    for l in range(1, 4):
        acc = acc + Ws[l][q[:, l]]
    assert torch.equal(out['zhat'], acc) and torch.equal(R.level_sum(Ws, q), acc)
    # every level quantizes what the earlier levels left over
    for l in range(1, 4):
        assert torch.equal(out['r'][l], out['r'][l - 1] - Ws[l - 1][q[:, l - 1]])
        assert torch.equal(q[:, l], torch.cdist(out['r'][l], Ws[l]).argmin(1))
    assert torch.equal(out['z_ste'], x + (acc - x))


def test_restatement_gradients_reach_x_through_every_residual():
    """CommitmentLoss of level l reaches x through r_{l-1} = x - sum sg(e_j): gx = sum_l 2 (r_{l-1} - e_l) / (N D)."""
    spec = O.QuantizerSpec(distance='L2', training=False, losses={'c': dict(type='CommitmentLoss')})
    x, Ws = _restatement_inputs(3)
    x.requires_grad_(True)
    out = R.rvq_forward(spec, x, Ws)
    out['loss'].backward()
    q = out['quant']
    want = sum(2 * (out['r'][l] - Ws[l][q[:, l]]) / x.numel() for l in range(3))
    torch.testing.assert_close(x.grad, want, rtol=1e-6, atol=1e-7)
    assert all(w.grad is None for w in out['weight_leafs'])


@pytest.mark.parametrize('dtype', [torch.int64, torch.int32, torch.uint16])
def test_save_and_load_tokens_keep_the_depth_axis(tmp_path, dtype):
    q = torch.randint(0, K, (2, 3, 5, 4), generator=torch.Generator().manual_seed(1))
    path = tmp_path / 'tokens.pth'
    tokenizer.save_tokens(path, ['a', 'b'], torch.tensor([1, 2]), q.to(dtype), (2, D, 3, 5))
    got = tokenizer.load_tokens(path)
    assert got['tokens'].dtype == torch.int64 and torch.equal(got['tokens'], q)
    # [N, L] ids (memo['quant'] of the forward) land in the same grid; one id per token keeps [b, h, w]
    tokenizer.save_tokens(path, ['a', 'b'], torch.tensor([1, 2]), q.view(-1, 4), (2, D, 3, 5))
    assert torch.equal(tokenizer.load_tokens(path)['tokens'], q)
    tokenizer.save_tokens(path, ['a', 'b'], torch.tensor([1, 2]), q[..., 0].reshape(-1), (2, D, 3, 5))
    assert tokenizer.load_tokens(path)['tokens'].shape == (2, 3, 5)
    with tokenizer.TokenStreamWriter(tmp_path / 'stream') as writer:
        p = writer.write(0, ['a', 'b'], torch.tensor([1, 2]), q.to(dtype), (2, D, 3, 5))
    assert torch.equal(tokenizer.load_tokens(p)['tokens'], q)
