"""GroupedVectorQuantizer without a GPU: registration, config validation, state-dict layout, the C-ABI argument checks,
the CPU restatement (oracle/gvq.py) and token dumps with a trailing group axis."""
import ctypes

import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import gvq as GV
from oracle import oracle as O
from vector_quantization_b200 import _lib, ops, plugin, tokenizer

K, DG = 16, 4


def _cfg(G=3, **group):
    node = dict(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=DG),
                losses=dict(vqgan_loss=dict(type='VQGANLoss')))
    node.update(group)
    return dict(type='GroupedVectorQuantizer', num_groups=G, quantizer=node)


def test_registered_and_exported():
    assert 'GroupedVectorQuantizer' in plugin.QUANTIZERS
    assert isinstance(vqb.VQITQuantizerRegistry.lookup('GroupedVectorQuantizer'), type)
    assert {'split_groups', 'group_gather_ste_loss', 'group_backward', 'decode_group_tokens'} <= set(ops.__all__)


def test_properties_state_dict_and_init_weights_on_every_group():
    q = vqb.build_quantizer(dict(_cfg(3, callbacks=[dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'),
                                                          ema=dict())]), init_weights=dict(type='vqgan')))
    assert (q.num_groups, q.group_dim, q.codebook_size, q.embedding_dim) == (3, DG, K, 3 * DG)
    assert q.embeddings.shape == (3, K, DG)
    keys = set(q.state_dict())
    for g in range(3):
        assert f'_quantizers.{g}._embedding.weight' in keys and f'_quantizers.{g}._probability' in keys
        assert f'_quantizers.{g}._losses.vqgan_loss._weight._steps' in keys
    assert all(k.startswith('_quantizers.') for k in keys)
    # VQGANQuantizer's 'vqgan' init: uniform(-1/K, 1/K) in every group, independently drawn
    E = q.embeddings
    assert E.abs().max() <= 1.0 / K and not torch.equal(E[0], E[1]) and not torch.equal(E[1], E[2])


@pytest.mark.parametrize('group,match', [
    (dict(callbacks=[dict(type='NormalizeCallback')]), 'NormalizeCallback rewrites the tokens'),
    (dict(callbacks=[dict(type='VQKDCallback', ema=dict())]), 'VQKDCallback rewrites the tokens'),
    (dict(callbacks=[dict(type='VQGAN_VQKDCallback', ema=dict())]), 'VQGAN_VQKDCallback rewrites the tokens'),
    (dict(callbacks=[dict(type='CVQVAECallback', anchor=dict(type='MultinomialAnchor'), ema=dict())]),
     'MultinomialAnchor'),
    (dict(losses=dict(entropy=dict(type='EntropyLoss', temperature=1.0))), 'EntropyLoss'),
    (dict(materialize_distance=True), 'materialize_distance'),
])
def test_rejected_group_configs_name_the_offending_item(group, match):
    with pytest.raises(ValueError, match=f'GroupedVectorQuantizer: .*{match}'):
        vqb.build_quantizer(_cfg(2, **group))


def test_rejects_callbacks_hooking_decode_or_loss():
    @vqb.VQITQuantizerCallbackRegistry.register_(force=True)
    class _HookLossForGVQTest(vqb.BaseCallback):
        def before_loss(self, z, x, memo):
            return z, x

    with pytest.raises(ValueError, match='_HookLossForGVQTest hooks before_loss'):
        vqb.build_quantizer(_cfg(2, callbacks=[dict(type='_HookLossForGVQTest')]))


@pytest.mark.parametrize('G', [0, 17, 2.0, True])
def test_rejects_group_count_outside_1_to_16(G):
    with pytest.raises(ValueError, match='num_groups'):
        vqb.build_quantizer(_cfg(G))


def test_rejects_fsq_and_nested_groups_and_top_level_losses():
    with pytest.raises(ValueError, match='FiniteScalarQuantizer'):
        vqb.build_quantizer(dict(type='GroupedVectorQuantizer', num_groups=2,
                                 quantizer=dict(type='FiniteScalarQuantizer', num_scalars_per_channel=[8, 5, 5, 5])))
    rvq = dict(type='ResidualVectorQuantizer', num_quantizers=2, quantizer=_cfg()['quantizer'])
    with pytest.raises(ValueError, match='got ResidualVectorQuantizer'):
        vqb.build_quantizer(dict(type='GroupedVectorQuantizer', num_groups=2, quantizer=rvq))
    with pytest.raises(ValueError, match='got GroupedVectorQuantizer'):
        vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=2, quantizer=_cfg(2)))
    with pytest.raises(ValueError, match='group config'):
        vqb.build_quantizer(dict(_cfg(2), losses=dict(c=dict(type='CodebookLoss'))))
    with pytest.raises(ValueError, match='group config'):
        vqb.build_quantizer(dict(_cfg(2), callbacks=[dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'),
                                                          ema=dict())]))


def test_c_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    lv = ops._residual_levels([torch.zeros(K, DG)] * 2)
    assert lib.vqb_split_groups(dummy, 0, 2, 17, DG, 4, ctypes.c_void_p(32), None) == -1
    assert b'G=17' in lib.vqb_last_error()
    assert lib.vqb_split_groups(dummy, 0, 2, 0, DG, 4, ctypes.c_void_p(32), None) == -1
    assert b'G=0' in lib.vqb_last_error()
    assert lib.vqb_split_groups(None, 0, 2, 2, DG, 4, dummy, None) == -1
    assert b'null pointer' in lib.vqb_last_error()
    lv.L = 17
    assert lib.vqb_group_gather_ste_loss(dummy, 0, 8, DG, ctypes.byref(lv), K, None, dummy, None, dummy, 0, 0, dummy,
                                         dummy, dummy, None) == -1
    assert b'G=17' in lib.vqb_last_error()
    lv.L = 2
    assert lib.vqb_group_gather_ste_loss(dummy, 0, 8, DG, ctypes.byref(lv), K, None, dummy, None, dummy, 3, 0, dummy,
                                         dummy, dummy, None) == -1
    assert b'z_hw must divide N' in lib.vqb_last_error()
    assert lib.vqb_group_gather_ste_loss(dummy, 0, 8, DG, ctypes.byref(lv), K, None, dummy, None, None, 0, 0, dummy,
                                         dummy, dummy, None) == -1
    assert b'null pointer' in lib.vqb_last_error()
    assert lib.vqb_group_gather_ste_loss(dummy, 0, 8, DG, ctypes.byref(lv), K, dummy, dummy, None, dummy, 0, 0, dummy,
                                         dummy, dummy, None) == -1
    assert b'exactly one of quant / keys' in lib.vqb_last_error()
    assert lib.vqb_group_backward(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, DG, 0, dummy, 3, None) == -1
    assert b'g_hw must divide N' in lib.vqb_last_error()
    lv.L = 0
    assert lib.vqb_group_backward(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, DG, 0, dummy, 0, None) == -1
    assert b'G=0' in lib.vqb_last_error()
    lv.L = 2
    assert lib.vqb_group_backward_rows(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, DG, 0, dummy, 0, None) == -1
    assert b'null gradient rows of group 0' in lib.vqb_last_error()
    assert lib.vqb_decode_group_tokens(dummy, 3, 1, 1, ctypes.byref(lv), K, DG, dummy, 0, None, None) == -1
    assert b'id_bytes' in lib.vqb_last_error()
    lv.L = 17
    assert lib.vqb_decode_group_tokens(dummy, 8, 1, 1, ctypes.byref(lv), K, DG, dummy, 0, None, None) == -1
    assert b'G=17' in lib.vqb_last_error()
    with pytest.raises(ValueError, match='1..16 groups'):
        ops._group_codebooks([torch.zeros(K, DG)] * 17)


def _restatement_inputs(G, N=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, G * DG, generator=g)
    Ws = [torch.randn(K, DG, generator=g) for _ in range(G)]
    return x, Ws


@pytest.mark.parametrize('loss', ['VQGANLoss', 'CodebookLoss', 'CommitmentLoss'])
@pytest.mark.parametrize('norm', [False, True])
@pytest.mark.parametrize('distance', ['L2', 'Cosine'])
def test_restatement_with_one_group_is_the_single_quantizer_oracle(distance, norm, loss):
    spec = O.QuantizerSpec(distance=distance, training=False, losses={'l': dict(type=loss, norm=norm)})
    x, Ws = _restatement_inputs(1)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    a = GV.gvq_forward(spec, xa, Ws)
    b = O.quantizer_forward(spec, [xb], Ws[0])
    assert torch.equal(a['quant'][:, 0], b['quant'][0])
    assert torch.equal(a['z_ste'], b['z_ste'][0]) and torch.equal(a['loss'], b['loss'][0])
    (a['loss'] + a['z_ste'].square().sum()).backward()
    (b['loss'][0] + b['z_ste'][0].square().sum()).backward()
    ga, gb = a['weight_leafs'][0].grad, b['weight_leaf'].grad
    assert torch.equal(xa.grad, xb.grad) and ((ga is None and gb is None) or torch.equal(ga, gb))


@pytest.mark.parametrize('G', [2, 4, 8])
def test_restatement_loss_is_the_full_width_mse(G):
    """Unnormalised terms: the group mean of the per-group MSEs is the MSE over all N * D elements."""
    spec = O.QuantizerSpec(distance='L2', training=False, losses={'c': dict(type='CodebookLoss'),
                                                                   'm': dict(type='CommitmentLoss')})
    x, Ws = _restatement_inputs(G, seed=G)
    out = GV.gvq_forward(spec, x, Ws)
    e = GV.group_concat(Ws, out['quant'])
    full = (e - x).square().mean()
    for name in ('c', 'm'):
        torch.testing.assert_close(out['losses'][name], full, rtol=1e-6, atol=0)
    # each group quantizes its own column slice against its own codebook
    for g in range(G):
        assert torch.equal(out['quant'][:, g], torch.cdist(x[:, g * DG:(g + 1) * DG], Ws[g]).argmin(1))
    assert torch.equal(out['z_ste'], x + (e - x))


@pytest.mark.parametrize('dtype', [torch.int64, torch.int32, torch.uint16])
def test_save_and_load_tokens_keep_the_group_axis(tmp_path, dtype):
    q = torch.randint(0, K, (2, 3, 5, 4), generator=torch.Generator().manual_seed(2))
    path = tmp_path / 'tokens.pth'
    tokenizer.save_tokens(path, ['a', 'b'], torch.tensor([1, 2]), q.to(dtype), (2, 4 * DG, 3, 5))
    got = tokenizer.load_tokens(path)
    assert got['tokens'].dtype == torch.int64 and torch.equal(got['tokens'], q)
    # [N, G] ids (memo['quant'] of the forward) land in the same grid
    tokenizer.save_tokens(path, ['a', 'b'], torch.tensor([1, 2]), q.view(-1, 4), (2, 4 * DG, 3, 5))
    assert torch.equal(tokenizer.load_tokens(path)['tokens'], q)
    with tokenizer.TokenStreamWriter(tmp_path / 'stream') as writer:
        p = writer.write(0, ['a', 'b'], torch.tensor([1, 2]), q.to(dtype), (2, 4 * DG, 3, 5))
    assert torch.equal(tokenizer.load_tokens(p)['tokens'], q)
