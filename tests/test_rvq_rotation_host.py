"""The rotation trick on ResidualVectorQuantizer without a GPU: the node key down to the C-ABI entry point it selects,
the still-rejected level key, the argument checks of the new entry points, and the CPU restatement
(oracle/rvq_rotation.py) against the single-quantizer one and against its closed form."""
import ctypes

import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rotation as R
from oracle import rvq
from oracle import rvq_rotation as RR
from vector_quantization_b200 import _lib, ops
from vector_quantization_b200 import functional as Fq
from vector_quantization_b200 import quantizers as Q

K, D = 16, 8


def _node(**kw):
    node = dict(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D),
                losses=dict(vqgan_loss=dict(type='VQGANLoss')))
    node.update(kw)
    return node


def _rvq(L=3, **kw):
    return vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=L, quantizer=_node(), **kw))


# ---- the node key -----------------------------------------------------------------------------------------------------

def test_node_key_defaults_off_is_a_bool_and_adds_no_state():
    off, on = _rvq(), _rvq(rotation_trick=1)
    assert off.rotation_trick is False and on.rotation_trick is True
    assert list(off.state_dict().keys()) == list(on.state_dict().keys())
    assert all(level.rotation_trick is False for level in on.quantizers)


@pytest.mark.parametrize('rotation_trick', [False, True])
def test_node_key_reaches_residual_quantize(monkeypatch, rotation_trick):
    seen = {}

    def fake(levels, x, memos, want_norm, *, nchw=None, rotate=False):
        seen['rotate'] = rotate
        L = len(levels)
        return x.float(), torch.zeros(x.shape[0], L, dtype=torch.int64), [(torch.zeros([]),) * 4] * L

    monkeypatch.setattr(Fq, 'residual_quantize', fake)
    monkeypatch.setattr(Q, '_check_tokens', lambda x, dim: x.contiguous())
    q = _rvq(rotation_trick=rotation_trick)
    q(torch.randn(8, D), dict())
    assert seen['rotate'] is rotation_trick


# ---- the entry point ops.residual_backward selects --------------------------------------------------------------------

@pytest.fixture
def fake_launches(monkeypatch):
    """ops without a device: every tensor counts as on `cpu`, _call records the entry point instead of launching."""
    names = []
    monkeypatch.setattr(ops, '_cuda', lambda *ts: torch.device('cpu'))
    monkeypatch.setattr(ops, '_call', lambda name, fn, dev, *args: names.append(name))
    monkeypatch.setattr(ops, '_det_ws', lambda dev, name, numel, dtype: torch.zeros(numel, dtype=dtype))
    monkeypatch.setattr(ops, '_segment_sum_members', lambda *a: None)
    return names


@pytest.mark.parametrize('deterministic', [False, True])
@pytest.mark.parametrize('rotate', [False, True])
def test_ops_select_the_entry_point(fake_launches, rotate, deterministic):
    L = 3
    x, Ws = torch.randn(8, D), [torch.randn(K, D) for _ in range(L)]
    ops.residual_backward(torch.randn(8, D), x, Ws, torch.zeros(8, L, dtype=torch.int64), [[None] * 4] * L,
                          want_norm=False, need_gW=[True] * L, deterministic=deterministic, rotate=rotate)
    tail = ('_rotated' if rotate else '') + ('_rows' if deterministic else '')
    assert fake_launches == ['vqb_residual_backward' + tail]


# ---- the level key stays rejected -------------------------------------------------------------------------------------

def test_level_key_is_rejected_and_the_message_names_the_node_key():
    with pytest.raises(ValueError, match='ResidualVectorQuantizer: rotation_trick is not supported for residual levels'
                                         r'.*rotation_trick=True on the ResidualVectorQuantizer node'):
        vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=2, quantizer=_node(rotation_trick=True)))
    with pytest.raises(ValueError, match='not supported for residual levels'):
        vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=2, rotation_trick=True,
                                 quantizer=_node(rotation_trick=True)))


# ---- C-ABI argument checks ------------------------------------------------------------------------------------------

def test_c_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    lv = ops._residual_levels([torch.zeros(K, D)] * 2)
    for name in ('vqb_residual_backward_rotated', 'vqb_residual_backward_rotated_rows'):
        fn = getattr(lib, name)
        assert fn(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 3, None) == -1
        assert f'{name}: g_hw must divide N'.encode() in lib.vqb_last_error()
        assert fn(dummy, 0, None, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, None) == -1
        assert b'null pointer' in lib.vqb_last_error()
        lv.L = 17
        assert fn(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, None) == -1
        assert b'L=17' in lib.vqb_last_error()
        lv.L = 2
    assert lib.vqb_residual_backward_rotated_rows(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0,
                                                  None) == -1
    assert b'vqb_residual_backward_rotated_rows: null gradient rows at level 0' in lib.vqb_last_error()


# ---- the restatement --------------------------------------------------------------------------------------------------

SPEC = O.QuantizerSpec(distance='L2', training=False, losses={'vqgan_loss': dict(type='VQGANLoss'),
                                                              'commit_norm': dict(type='CommitmentLoss', norm=True)})


def _data(N, L, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, D, generator=g, dtype=torch.float64)
    Ws = [torch.randn(K, D, generator=g, dtype=torch.float64) * 0.6 ** l for l in range(L)]
    gz = torch.randn(N, D, generator=g, dtype=torch.float64)
    return x, Ws, gz


def _grad_x(out, x, gz):
    ((out['z_ste'] * gz).sum() + out['loss']).backward()
    return x.grad


def test_depth_one_is_the_rotated_single_quantizer():
    x, Ws, gz = _data(128, 1, seed=1)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    a = R.rotated_forward(SPEC, [xa], Ws[0])
    b = RR.rotated_rvq_forward(SPEC, xb, Ws)
    assert torch.equal(a['quant'][0], b['quant'][:, 0])
    assert torch.equal(a['z_ste'][0], b['z_ste']) and torch.equal(a['loss'][0], b['loss'])
    ((a['z_ste'][0] * gz).sum() + a['loss'][0]).backward()
    torch.testing.assert_close(_grad_x(b, xb, gz), xa.grad, rtol=0, atol=1e-12)


@pytest.mark.parametrize('L', [1, 2, 4, 8])
def test_values_are_the_straight_through_ones_and_the_gradient_is_the_closed_form(L):
    x, Ws, gz = _data(256, L, seed=10 + L)
    x[3] = 0                                     # a zero token keeps g
    xs, xr, xl = (x.clone().requires_grad_(True) for _ in range(3))
    ste = rvq.rvq_forward(SPEC, xs, Ws)
    rot = RR.rotated_rvq_forward(SPEC, xr, Ws)
    for key in ('quant', 'zhat', 'z_ste', 'loss'):
        assert torch.equal(ste[key], rot[key]), key
    assert all(torch.equal(ste['losses'][k], rot['losses'][k]) for k in ste['losses'])
    # the straight-through RVQ's commitment terms: the gradient of the losses alone
    only_loss = rvq.rvq_forward(SPEC, xl, Ws)
    only_loss['loss'].backward()
    want = R.rotate_grad(x, rot['zhat'], gz) + xl.grad
    got = _grad_x(rot, xr, gz)
    torch.testing.assert_close(got, want, rtol=1e-12, atol=1e-12)     # the zero token's norm term is ~1e8
    torch.testing.assert_close(got[3], gz[3] + xl.grad[3], rtol=1e-12, atol=1e-12)
    assert not torch.allclose(got, _grad_x(ste, xs, gz))
