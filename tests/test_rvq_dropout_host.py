"""Quantizer dropout and depth-truncated codes on ResidualVectorQuantizer without a GPU: the node key and the
num_quantizers argument checks, the C-ABI entry points the ops layer selects and their argument checks, and the CPU
restatement (oracle/rvq_dropout.py) against oracle/rvq.py."""
import ctypes

import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rvq
from oracle import rvq_dropout as RD
from oracle import rvq_rotation as RR
from vector_quantization_b200 import _lib, ops
from vector_quantization_b200 import functional as Fq
from vector_quantization_b200 import quantizers as Q
from vector_quantization_b200 import tokenizer as T

K, D = 16, 8


def _node(**kw):
    node = dict(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D),
                losses=dict(vqgan_loss=dict(type='VQGANLoss')))
    node.update(kw)
    return node


def _rvq(L=3, node=None, **kw):
    return vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=L, quantizer=node or _node(), **kw))


# ---- the node key -----------------------------------------------------------------------------------------------------

def test_quantizer_dropout_defaults_off_and_adds_no_state():
    off, on = _rvq(), _rvq(quantizer_dropout=0.5)
    assert off.quantizer_dropout == 0.0 and on.quantizer_dropout == 0.5
    assert _rvq(quantizer_dropout=1).quantizer_dropout == 1.0
    assert list(off.state_dict().keys()) == list(on.state_dict().keys())


@pytest.mark.parametrize('bad', [True, False, -0.1, 1.5, float('nan'), '0.5', None])
def test_quantizer_dropout_rejects_bools_and_values_outside_the_unit_interval(bad):
    with pytest.raises(ValueError, match='quantizer_dropout='):
        _rvq(quantizer_dropout=bad)


def test_quantizer_dropout_is_not_a_level_key():
    with pytest.raises(ValueError, match='quantizer_dropout is not a level key'):
        _rvq(node=_node(quantizer_dropout=0.5))


@pytest.mark.parametrize('bad', [0, 4, -1, True, 2.0, '2'])
def test_num_quantizers_outside_the_depth_is_a_value_error(bad):
    q = _rvq(L=3)
    with pytest.raises(ValueError, match='num_quantizers='):
        q.num_levels(bad)
    with pytest.raises(ValueError, match='num_quantizers='):
        q.encode(torch.zeros(4, D), dict(), num_quantizers=bad)
    with pytest.raises(ValueError, match='num_quantizers='):
        q.encode_compact(torch.zeros(4, D), dict(), num_quantizers=bad)
    with pytest.raises(ValueError, match='num_quantizers='):
        T.encode_to_quant(q, torch.zeros(1, D, 2, 2), dict(), num_quantizers=bad)
    with pytest.raises(ValueError, match='num_quantizers='):
        T.decode_from_quant(q, torch.zeros(1, 2, 2, 3, dtype=torch.int64), dict(), num_quantizers=bad)


def test_num_quantizers_is_a_residual_argument_only():
    gvq = vqb.build_quantizer(dict(type='GroupedVectorQuantizer', num_groups=2, quantizer=_node(
        embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D // 2))))
    with pytest.raises(ValueError, match='num_quantizers truncates ResidualVectorQuantizer codes'):
        T.encode_to_quant(gvq, torch.zeros(1, D, 2, 2), dict(), num_quantizers=1)
    with pytest.raises(ValueError, match='num_quantizers truncates ResidualVectorQuantizer codes'):
        T.decode_from_quant(gvq, torch.zeros(1, 2, 2, 2, dtype=torch.int64), dict(), num_quantizers=1)


def test_decode_from_quant_checks_the_trailing_axis_against_n():
    q = _rvq(L=3)
    assert q.num_levels() == 3 and q.num_levels(2) == 2
    with pytest.raises(ValueError, match=r'\[b, h, w, 3\]'):
        T.decode_from_quant(q, torch.zeros(1, 2, 2, 2, dtype=torch.int64), dict())
    with pytest.raises(ValueError, match=r'\[b, h, w, 2\]'):
        T.decode_from_quant(q, torch.zeros(1, 2, 2, 3, dtype=torch.int64), dict(), num_quantizers=2)


@pytest.mark.parametrize('p, training, drawn', [(0.0, True, False), (0.5, False, False), (0.5, True, True)])
def test_depths_are_drawn_only_in_training_with_p_above_zero(monkeypatch, p, training, drawn):
    seen = {}

    def fake(levels, x, memos, want_norm, *, nchw=None, rotate=False, depth=None):
        seen['depth'] = depth
        L = len(levels)
        return x.float(), torch.zeros(x.shape[0], L, dtype=torch.int64), [(torch.zeros([]),) * 4] * L

    monkeypatch.setattr(Fq, 'residual_quantize', fake)
    monkeypatch.setattr(Q, '_check_tokens', lambda x, dim: x.contiguous())
    q = _rvq(quantizer_dropout=p)
    q.train(training)
    _, _, memo = q(torch.randn(40, D), dict())
    if drawn:
        d = seen['depth']
        assert d.dtype == torch.int32 and d.shape == (40,) and memo['depth'] is d
        assert (d[20:] == 3).all() and ((d[:20] >= 1) & (d[:20] <= 3)).all()
    else:
        assert seen['depth'] is None and 'depth' not in memo
        seen.clear()
        monkeypatch.setattr(Fq, 'residual_quantize', lambda levels, x, memos, want_norm, *, nchw=None, rotate=False:
                            fake(levels, x, memos, want_norm, nchw=nchw, rotate=rotate))
        q(torch.randn(40, D), dict())         # the call without dropout passes no depth keyword


def test_draw_truncates_the_first_floor_of_s_times_p_samples():
    q = _rvq(L=4, quantizer_dropout=0.3)
    torch.manual_seed(0)
    d = q.draw_depths(1000, 'cpu')
    assert (d[300:] == 4).all() and ((d[:300] >= 1) & (d[:300] <= 4)).all()
    assert set(d[:300].tolist()) == {1, 2, 3, 4}
    assert (_rvq(L=4, quantizer_dropout=0.3).draw_depths(3, 'cpu') == 4).all()       # floor(0.9) = 0


# ---- the entry points ops selects --------------------------------------------------------------------------------------

@pytest.fixture
def fake_launches(monkeypatch):
    """ops without a device: every tensor counts as on `cpu`, _call records the entry point and its arguments."""
    calls = []
    monkeypatch.setattr(ops, '_cuda', lambda *ts: torch.device('cpu'))
    monkeypatch.setattr(ops, '_call', lambda name, fn, dev, *args: calls.append((name, args)))
    monkeypatch.setattr(ops, '_det_ws', lambda dev, name, numel, dtype: torch.zeros(numel, dtype=dtype))
    monkeypatch.setattr(ops, '_segment_sum_members', lambda *a: None)
    monkeypatch.setattr(ops, '_loss_ws', lambda dev: (torch.zeros(1), torch.zeros(1, dtype=torch.int32)))
    return calls


@pytest.mark.parametrize('deterministic', [False, True])
@pytest.mark.parametrize('rotate', [False, True])
@pytest.mark.parametrize('with_depth', [False, True])
def test_ops_residual_backward_selects_the_entry_point(fake_launches, with_depth, rotate, deterministic):
    L = 3
    x, Ws = torch.randn(8, D), [torch.randn(K, D) for _ in range(L)]
    depth = torch.full((2,), 2, dtype=torch.int32) if with_depth else None
    ops.residual_backward(torch.randn(8, D), x, Ws, torch.zeros(8, L, dtype=torch.int64), [[None] * 4] * L,
                          want_norm=False, need_gW=[True] * L, deterministic=deterministic, rotate=rotate,
                          depth=depth, depth_hw=4)
    name = 'vqb_residual_backward' + ('_depth' if with_depth else '') + ('_rotated' if rotate else '') + \
        ('_rows' if deterministic else '')
    [(called, args)] = fake_launches
    assert called == name
    assert len(args) == len(_lib.SIGNATURES[name][1])
    if with_depth:
        assert args[-3:-1] == (depth.data_ptr(), 4)


@pytest.mark.parametrize('with_depth', [False, True])
def test_ops_residual_step_selects_the_entry_point(fake_launches, with_depth):
    x, W = torch.randn(8, D), torch.randn(K, D)
    depth = torch.full((8,), 1, dtype=torch.int32) if with_depth else None
    ops.residual_step(x, x, W, torch.zeros(4), level=0, L=1, keys=torch.zeros(8, dtype=torch.int64), depth=depth)
    [(called, args)] = fake_launches
    name = 'vqb_residual_step' + ('_depth' if with_depth else '')
    assert called == name and len(args) == len(_lib.SIGNATURES[name][1])


def test_ops_check_the_depth_tensor(fake_launches):
    x, W = torch.randn(8, D), torch.randn(K, D)
    step = lambda depth, hw: ops.residual_step(x, x, W, torch.zeros(4), level=0, L=1,          # noqa: E731
                                               keys=torch.zeros(8, dtype=torch.int64), depth=depth, depth_hw=hw)
    with pytest.raises(TypeError, match='int32'):
        step(torch.ones(8, dtype=torch.int64), 1)
    with pytest.raises(ValueError, match='depth has 8 entries'):
        step(torch.ones(8, dtype=torch.int32), 4)
    with pytest.raises(ValueError, match='depth_hw = 3'):
        step(torch.ones(2, dtype=torch.int32), 3)
    assert not fake_launches


# ---- C-ABI argument checks ------------------------------------------------------------------------------------------

BACKWARD_DEPTH = ('vqb_residual_backward_depth', 'vqb_residual_backward_depth_rows', 'vqb_residual_backward_depth_rotated',
                  'vqb_residual_backward_depth_rotated_rows')


def test_c_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    lv = ops._residual_levels([torch.zeros(K, D)] * 2)
    for name in BACKWARD_DEPTH:
        fn = getattr(lib, name)
        assert fn(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, None, 1, None) == -1
        assert f'{name}: null depth'.encode() in lib.vqb_last_error()
        assert fn(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, dummy, 3, None) == -1
        assert f'{name}: depth_hw must divide N'.encode() in lib.vqb_last_error()
        assert fn(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, dummy, 0, None) == -1
        assert f'{name}: depth_hw must divide N'.encode() in lib.vqb_last_error()
    step = lib.vqb_residual_step_depth
    args = [dummy, 0, dummy, 0, 8, D, dummy, K, None, dummy, 0, None, 1, 0, None, None, dummy, 0, 0, dummy, dummy, dummy]
    assert step(*args, None, 1, None) == -1
    assert b'vqb_residual_step_depth: null depth' in lib.vqb_last_error()
    assert step(*args, dummy, 5, None) == -1
    assert b'vqb_residual_step_depth: depth_hw must divide N' in lib.vqb_last_error()


# ---- the restatement --------------------------------------------------------------------------------------------------

SPEC = O.QuantizerSpec(distance='L2', training=False, losses={'vqgan_loss': dict(type='VQGANLoss'),
                                                              'commit_norm': dict(type='CommitmentLoss', norm=True)})


def _data(N, L, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, D, generator=g)
    Ws = [torch.randn(K, D, generator=g) * 0.6 ** l for l in range(L)]
    gz = torch.randn(N, D, generator=g)
    return x, Ws, gz


def _grads(out, x, gz):
    ((out['z_ste'] * gz).sum() + out['loss']).backward()
    return x.grad, [W.grad for W in out['weight_leafs']]


@pytest.mark.parametrize('rotation', [False, True])
@pytest.mark.parametrize('L', [1, 3, 8])
def test_full_depth_is_oracle_rvq_bit_for_bit(L, rotation):
    x, Ws, gz = _data(192, L, seed=L)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    a = (RR.rotated_rvq_forward if rotation else rvq.rvq_forward)(SPEC, xa, Ws)
    b = RD.rvq_dropout_forward(SPEC, xb, Ws, torch.full((192,), L), rotation=rotation)
    for key in ('quant', 'zhat', 'z_ste', 'loss'):
        assert torch.equal(a[key], b[key]), key
    assert all(torch.equal(a['losses'][k], b['losses'][k]) for k in a['losses'])
    ga, gWa = _grads(a, xa, gz)
    gb, gWb = _grads(b, xb, gz)
    assert torch.equal(ga, gb)
    assert all(torch.equal(p, q) for p, q in zip(gWa, gWb))


@pytest.mark.parametrize('n, L', [(1, 3), (2, 3), (3, 8), (5, 8)])
def test_uniform_depth_n_is_oracle_rvq_on_the_first_n_levels(n, L):
    x, Ws, gz = _data(192, L, seed=100 + n)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    a = rvq.rvq_forward(SPEC, xa, Ws[:n])
    b = RD.rvq_dropout_forward(SPEC, xb, Ws, torch.full((192,), n))
    assert torch.equal(a['quant'], b['quant'][:, :n])
    assert torch.equal(a['z_ste'], b['z_ste']) and torch.equal(a['loss'], b['loss'])
    assert all(torch.equal(a['losses'][k], b['losses'][k]) for k in a['losses'])
    ga, gWa = _grads(a, xa, gz)
    gb, gWb = _grads(b, xb, gz)
    torch.testing.assert_close(gb, ga, rtol=1e-6, atol=1e-7)
    for l in range(L):
        if l < n:
            torch.testing.assert_close(gWb[l], gWa[l], rtol=1e-6, atol=1e-7)
        else:
            assert not gWb[l].any()


def test_mixed_depths_take_each_token_from_its_own_depth():
    L, N = 4, 256
    x, Ws, gz = _data(N, L, seed=7)
    depth = torch.randint(1, L + 1, (N,), generator=torch.Generator().manual_seed(1))
    xb = x.clone().requires_grad_(True)
    b = RD.rvq_dropout_forward(SPEC, xb, Ws, depth)
    gb, _ = _grads(b, xb, gz)
    for n in range(1, L + 1):
        rows = depth == n
        xa = x.clone().requires_grad_(True)
        a = rvq.rvq_forward(SPEC, xa, Ws[:n])
        assert torch.equal(a['quant'][rows], b['quant'][rows, :n])
        assert torch.equal(a['z_ste'][rows], b['z_ste'][rows])
        ga, _ = _grads(a, xa, gz)
        torch.testing.assert_close(gb[rows], ga[rows], rtol=1e-6, atol=1e-7)   # the loss terms are per row
