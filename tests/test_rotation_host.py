"""The rotation trick without a GPU: the CPU restatement (oracle/rotation.py) against its closed form, the straight-
through fallback rows, the config key down to the C-ABI entry point it selects, the rejected configurations and the
argument checks of the new entry points."""
import ctypes

import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rotation as R
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


@pytest.mark.parametrize('dim', [3, 8, 32, 256])
def test_autograd_of_rotate_to_is_the_closed_form_and_its_value_is_e(dim):
    g = torch.Generator().manual_seed(dim)
    y = torch.randn(257, dim, generator=g, dtype=torch.float64).requires_grad_(True)
    e = torch.randn(257, dim, generator=g, dtype=torch.float64) * 0.3
    gz = torch.randn(257, dim, generator=g, dtype=torch.float64)
    out = R.rotate_to(y, e)
    torch.testing.assert_close(out.detach(), e, rtol=0, atol=1e-12)
    out.backward(gz)
    closed = R.rotate_grad(y.detach(), e, gz)
    torch.testing.assert_close(y.grad, closed, rtol=0, atol=1e-12)
    # lambda R^T is a scaled rotation: it keeps |g| up to the factor |e| / |y|
    lam = e.norm(dim=1) / y.detach().norm(dim=1)
    torch.testing.assert_close(closed.norm(dim=1), lam * gz.norm(dim=1), rtol=1e-12, atol=0)


def test_fallback_rows_follow_the_rule():
    g = torch.Generator().manual_seed(5)
    e = torch.randn(4, D, generator=g, dtype=torch.float64)
    y = torch.randn(4, D, generator=g, dtype=torch.float64)
    y[0] = 0                 # zero token: straight-through
    e[1] = 0                 # zero code: straight-through
    y[2] = -2.0 * e[2]       # antipodal pair: s = 0, w = 0, a finite rotation by the u -> e reflection term only
    gz = torch.randn(4, D, generator=g, dtype=torch.float64)
    yl = y.clone().requires_grad_(True)
    out = R.rotate_to(yl, e)
    out.backward(gz)
    torch.testing.assert_close(out.detach(), e, rtol=0, atol=1e-12)
    assert torch.equal(yl.grad[0], gz[0]) and torch.equal(yl.grad[1], gz[1])
    closed = R.rotate_grad(y, e, gz)
    assert torch.equal(closed[0], gz[0]) and torch.equal(closed[1], gz[1])
    u = y[2] / y[2].norm()
    eh = e[2] / e[2].norm()
    assert torch.equal(u + eh, torch.zeros(D, dtype=torch.float64))
    want = 0.5 * (gz[2] + 2 * u * (eh @ gz[2]))
    torch.testing.assert_close(closed[2], want, rtol=0, atol=1e-12)
    torch.testing.assert_close(yl.grad[2], want, rtol=0, atol=1e-12)
    assert torch.isfinite(closed).all() and torch.isfinite(yl.grad).all()
    torch.testing.assert_close(yl.grad[3], closed[3], rtol=0, atol=1e-12)


@pytest.mark.parametrize('callback', [None, 'NormalizeCallback', 'VQKDCallback'])
def test_rotated_forward_keeps_the_value_and_rotates_the_gradient_of_the_quantizers_view(callback):
    spec = O.QuantizerSpec(distance='L2' if callback is None else 'Cosine', callback=callback, training=False,
                           losses={'c': dict(type='CommitmentLoss')})
    g = torch.Generator().manual_seed(1)
    x = torch.randn(64, D, generator=g, dtype=torch.float64)
    W = torch.randn(K, D, generator=g, dtype=torch.float64)
    gz = torch.randn(64, D, generator=g, dtype=torch.float64)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    a = O.quantizer_forward(spec, [xa], W)
    b = R.rotated_forward(spec, [xb], W)
    assert torch.equal(a['quant'][0], b['quant'][0]) and torch.equal(a['z_ste'][0], b['z_ste'][0])
    (b['z_ste'][0] * gz).sum().backward()
    y = b['x'][0].detach()
    rot = R.rotate_grad(y, b['z'][0].detach(), gz)
    if callback is None:
        torch.testing.assert_close(xb.grad, rot, rtol=0, atol=1e-12)
    else:   # then through F.normalize: J_n(x)^T g'
        n = x.norm(dim=1, keepdim=True)
        want = (rot - (rot * y).sum(1, keepdim=True) * y) / n
        torch.testing.assert_close(xb.grad, want, rtol=0, atol=1e-12)


# ---- the config key down to the entry point -------------------------------------------------------------------------

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
    x, W, q = torch.randn(8, D), torch.randn(K, D), torch.zeros(8, dtype=torch.int64)
    ops.quantize_backward(torch.randn(8, D), x, W, q, [None] * 4, want_norm=False, need_gW=True,
                          deterministic=deterministic, rotate=rotate)
    xs, Ws = torch.randn(2, 8, D), [torch.randn(K, D)] * 2
    ops.group_backward(torch.randn(8, 2 * D), xs, Ws, torch.zeros(8, 2, dtype=torch.int64), [[None] * 4] * 2,
                       want_norm=False, need_gW=[True, True], deterministic=deterministic, rotate=rotate)
    tail = ('_rotated' if rotate else '') + ('_rows' if deterministic else '')
    assert fake_launches == ['vqb_quantize_backward' + tail, 'vqb_group_backward' + tail]


def _fake_encode(q, quant):
    def encode(x, memo):
        memo['encode'] = dict()
        return x, quant, memo
    q.encode = encode
    q._weight = lambda: q._embedding.weight


@pytest.mark.parametrize('rotation_trick', [False, True])
def test_config_key_reaches_the_backward_entry_point(fake_launches, monkeypatch, rotation_trick):
    monkeypatch.setattr(Q, '_check_tokens', lambda x, dim: x.contiguous())
    monkeypatch.setattr(ops, 'gather_ste_loss',
                        lambda x, W, **kw: (x.float() + 0, torch.zeros(4, device=x.device), None, None))
    quant = torch.zeros(8, dtype=torch.int64)
    for cls in ('VectorQuantizer', 'VQGANQuantizer', 'VQKDQuantizer'):
        fake_launches.clear()
        q = vqb.build_quantizer(_node(type=cls, rotation_trick=rotation_trick))
        assert q.rotation_trick is rotation_trick
        _fake_encode(q, quant)
        x = torch.randn(8, D, requires_grad=True)
        z, loss, memo = q(x, dict())
        (z.sum() + loss).backward()
        assert fake_launches == ['vqb_quantize_backward_rotated' if rotation_trick else 'vqb_quantize_backward']
        # the standalone loss on arbitrary tensors never rotates
        fake_launches.clear()
        zz = torch.randn(8, D, requires_grad=True)
        q.loss(zz, x, dict())[0].backward()
        assert fake_launches == ['vqb_quantize_backward']


@pytest.mark.parametrize('rotation_trick', [False, True])
def test_grouped_config_key_reaches_every_group(monkeypatch, rotation_trick):
    seen = {}

    def fake(groups, x, memos, want_norm, *, rotate=False):
        seen['rotate'] = rotate
        G = len(groups)
        return x.float(), torch.zeros(x.shape[0], G, dtype=torch.int64), [(torch.zeros([]),) * 4] * G

    monkeypatch.setattr(Fq, 'grouped_quantize', fake)
    monkeypatch.setattr(Q.GroupedVectorQuantizer, '_check_input', lambda self, x: x)
    q = vqb.build_quantizer(dict(type='GroupedVectorQuantizer', num_groups=4,
                                 quantizer=_node(rotation_trick=rotation_trick)))
    assert all(g.rotation_trick is rotation_trick for g in q.quantizers)
    q(torch.randn(8, 4 * D), dict())
    assert seen['rotate'] is rotation_trick


# ---- rejections -----------------------------------------------------------------------------------------------------

def test_rotation_trick_with_a_callback_hooking_decode_or_loss_is_rejected():
    @vqb.VQITQuantizerCallbackRegistry.register_(force=True)
    class _HookDecodeForRotationTest(vqb.BaseCallback):
        def after_decode(self, z, memo):
            return z

    with pytest.raises(ValueError, match='VQGANQuantizer: rotation_trick .* _HookDecodeForRotationTest, which hooks '
                                         'after_decode'):
        vqb.build_quantizer(_node(rotation_trick=True, callbacks=[dict(type='_HookDecodeForRotationTest')]))
    # without the key the template path stays available
    vqb.build_quantizer(_node(callbacks=[dict(type='_HookDecodeForRotationTest')]))


def test_rotation_trick_in_a_residual_level_is_rejected():
    with pytest.raises(ValueError, match='ResidualVectorQuantizer: rotation_trick is not supported for residual levels'):
        vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=2, quantizer=_node(rotation_trick=True)))
    vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=2, quantizer=_node(rotation_trick=False)))


def test_fsq_takes_no_rotation_key():
    with pytest.raises(TypeError, match='rotation_trick'):
        vqb.build_quantizer(dict(type='FiniteScalarQuantizer', num_scalars_per_channel=[8, 5, 5, 5],
                                 rotation_trick=True))


# ---- C-ABI argument checks ------------------------------------------------------------------------------------------

def test_c_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    for name in ('vqb_quantize_backward_rotated', 'vqb_quantize_backward_rotated_rows'):
        fn = getattr(lib, name)
        assert fn(dummy, 0, dummy, 0, 0, dummy, K, dummy, 8, D, None, None, None, None, 0, dummy, dummy, 3, None) == -1
        assert b'vqb_quantize_backward_rotated: g_hw must divide N' in lib.vqb_last_error()
        assert fn(None, 0, dummy, 0, 0, dummy, K, dummy, 8, D, None, None, None, None, 0, dummy, dummy, 0, None) == -1
        assert b'null pointer' in lib.vqb_last_error()
        assert fn(dummy, 0, dummy, 0, 0, dummy, K, dummy, 0, D, None, None, None, None, 0, dummy, dummy, 0, None) == -1
        assert b'bad shape' in lib.vqb_last_error()
        assert fn(dummy, 0, dummy, 0, 0, dummy, K, dummy, 8, 4097, None, None, None, None, 0, dummy, dummy, 0,
                  None) == -1
        assert b'D=4097 unsupported' in lib.vqb_last_error()
    assert lib.vqb_quantize_backward_rotated_rows(dummy, 0, dummy, 0, 0, dummy, K, dummy, 8, D, None, None, None, None,
                                                  0, dummy, None, 0, None) == -1
    assert b'vqb_quantize_backward_rotated_rows: null gW_rows' in lib.vqb_last_error()
    lv = ops._residual_levels([torch.zeros(K, D)] * 2)
    for name in ('vqb_group_backward_rotated', 'vqb_group_backward_rotated_rows'):
        fn = getattr(lib, name)
        assert fn(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 3, None) == -1
        assert f'{name}: g_hw must divide N'.encode() in lib.vqb_last_error()
        assert fn(dummy, 0, dummy, 0, None, K, dummy, 8, D, 0, dummy, 0, None) == -1
        assert b'null pointer' in lib.vqb_last_error()
        lv.L = 17
        assert fn(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0, None) == -1
        assert b'G=17' in lib.vqb_last_error()
        lv.L = 2
    assert lib.vqb_group_backward_rotated_rows(dummy, 0, dummy, 0, ctypes.byref(lv), K, dummy, 8, D, 0, dummy, 0,
                                               None) == -1
    assert b'null gradient rows of group 0' in lib.vqb_last_error()
