"""The rotation trick on the B200: on against off (everything but gx bit-identical), gx against the float64 restatement
(oracle/rotation.py) over the row geometries, dtypes, metrics, loss terms, layouts and the shipped configs, the
degenerate rows, the grouped quantizer against the single one, and reproducibility (run to run, CUDA-graph replay)."""
import pathlib

import einops
import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rotation as R
from vector_quantization_b200 import tokenizer

pytestmark = pytest.mark.gpu
GOLDEN = pathlib.Path(__file__).parent / 'golden'
DTYPES = [torch.float32, torch.bfloat16]
DT_IDS = ['fp32', 'bf16']
METRIC = {'L2': 'L2Distance', 'Cosine': 'CosineDistance'}
SHIPPED = ['vqgan_l2', 'llamagen_l2norm', 'vqkd_train', 'vqkd_eval', 'cvqvae_train', 'llamagen_cvq_train',
           'cluster_train']


def _node(K, D, metric='L2', norm=False, callbacks=(), rotation_trick=True, type_='VQGANQuantizer'):
    losses = dict(vqgan_loss=dict(type='VQGANLoss'))
    if norm:
        losses['commit_norm'] = dict(type='CommitmentLoss', mse=dict(norm=True))
    return dict(type=type_, distance=dict(type=METRIC[metric]), callbacks=list(callbacks), losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D),
                rotation_trick=rotation_trick)


def _spec_losses(cfg):
    out = {}
    for name, c in cfg['losses'].items():
        out[name] = dict(type=c['type'], norm=c.get('mse', {}).get('norm', False))
    return out


def _build(cfg, dev, W, training=True, prob=None):
    q = vqb.build_quantizer(cfg, training=training).to(dev)
    q._forward_pre_hooks.clear()
    with torch.no_grad():
        q.embedding.weight.copy_(W)
        if prob is not None:
            q.get_buffer('_probability').copy_(prob)
    return q


def _nchw(t, b, h, w):
    return einops.rearrange(t, '(b h w) c -> b c h w', b=b, h=h, w=w).contiguous()


def _tokens(t, b, h, w):
    return einops.rearrange(t, 'b c h w -> (b h w) c', b=b, h=h, w=w)


def _step(q, x_cpu, gz_cpu, dev, hw=None):
    """forward + backward (upstream: gz on z, 1 on the loss); z / gx come back token-major."""
    W = q.embedding.weight
    if hw is not None:
        b, h, w = hw
        x = _nchw(x_cpu, b, h, w).to(dev).requires_grad_(True)
        z, loss, memo = tokenizer.quantize(q, x, dict())
        memo = memo['quantizer']
        gx, gW = torch.autograd.grad((z, loss), (x, W), (_nchw(gz_cpu, b, h, w).to(dev), torch.ones_like(loss)),
                                     allow_unused=True)
        z, gx = _tokens(z.detach(), b, h, w), _tokens(gx, b, h, w)
    else:
        x = x_cpu.to(dev).requires_grad_(True)
        z, loss, memo = q(x, dict())
        gx, gW = torch.autograd.grad((z, loss), (x, W), (gz_cpu.to(dev), torch.ones_like(loss)), allow_unused=True)
    return dict(z=z.detach(), loss=loss.detach(), losses={k: v.detach() for k, v in memo['loss'].items()},
                quant=memo['quant'].clone(), gx=gx, gW=gW, W=W.detach().clone())


def _oracle_gx(x_cpu, W_used, quant, gz, losses, normalize):
    """float64 gx of (z * gz).sum() + loss with the rotation trick, on the kernel's own indices and codebook."""
    x = x_cpu.double().requires_grad_(True)
    y = O.normalize(x) if normalize else x
    e = W_used.double()[quant.cpu()]
    z = R.rotate_to(y, e)
    ls = O._losses(O.QuantizerSpec(losses=losses), e, y)
    ((z * gz.double()).sum() + sum(ls.values())).backward()
    return x.grad


def _check_gx(gx, want, dtype):
    gx = gx.float().cpu().double()
    scale = float(want.abs().max())
    if dtype == torch.bfloat16:     # gx comes back in the token dtype: one bf16 rounding
        torch.testing.assert_close(gx, want, rtol=2 ** -7, atol=1e-4 * scale)
    else:
        torch.testing.assert_close(gx, want, rtol=1e-4, atol=1e-5 * scale)


def _load(name):
    return torch.load(GOLDEN / f'{name}.pt', weights_only=False)


# ---- 1. on against off ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', SHIPPED)
def test_rotation_changes_only_gx(dev, name):
    rec = _load(name)
    res = []
    torch.use_deterministic_algorithms(True)      # gW through the segment sum: comparable bit for bit
    try:
        for rot in (False, True):
            q = _build(dict(rec['config'], rotation_trick=rot), dev, rec['steps'][0]['W_before'], rec['training'],
                       rec['steps'][0]['prob_before'])
            steps = []
            for step in rec['steps']:     # the codebook updates of every step (CVQ-VAE, VQ-KD k-means / EMA)
                out = _step(q, step['x'], step['gz'], dev)
                prob = dict(q.named_buffers()).get('_probability')
                if prob is not None:
                    out['prob'] = prob.clone()
                steps.append(out)
            res.append(steps)
    finally:
        torch.use_deterministic_algorithms(False)
    for s, (off, on) in enumerate(zip(*res)):
        for key in ('z', 'loss', 'quant', 'W', 'prob'):
            if key in off:
                assert torch.equal(off[key], on[key]), (name, s, key)
        assert off['losses'].keys() == on['losses'].keys()
        assert all(torch.equal(off['losses'][k], on['losses'][k]) for k in off['losses']), (name, s)
        assert (off['gW'] is None) == (on['gW'] is None)
        if off['gW'] is not None:
            assert torch.equal(off['gW'], on['gW']), (name, s)
        assert not torch.equal(off['gx'], on['gx']), (name, s)


# ---- 2. gx against the float64 restatement -----------------------------------------------------------------------------
_DS = [8, 20, 32, 64, 256, 768, 2048]    # scalar path, V = 8 with NV = 1, 2, 4, 8


@pytest.mark.parametrize('D', _DS)
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_gx_matches_the_restatement(dev, D, metric, dtype):
    i = _DS.index(D)
    norm = (i + (metric == 'Cosine')) % 2 == 1
    nchw = (i + (dtype == torch.bfloat16)) % 2 == 1
    b, h, w, K = 4, 16, 16, 512
    N = b * h * w
    x, W = O.synthetic_latents(N, K, D, seed=D)
    x = x.to(dtype)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(D + 1))
    cfg = _node(K, D, metric, norm)
    q = _build(cfg, dev, W)
    out = _step(q, x, gz, dev, hw=(b, h, w) if nchw else None)
    want = _oracle_gx(x.float(), out['W'].cpu(), out['quant'], gz, _spec_losses(cfg), normalize=False)
    _check_gx(out['gx'], want, dtype)


@pytest.mark.parametrize('name', SHIPPED)
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_gx_of_the_shipped_configs_matches_the_restatement(dev, name, dtype):
    rec = _load(name)
    step = rec['steps'][0]
    q = _build(dict(rec['config'], rotation_trick=True), dev, step['W_before'], rec['training'], step['prob_before'])
    x = step['x'].to(dtype)
    out = _step(q, x, step['gz'], dev)
    spec = rec['spec']
    normalize = spec['callback'] in ('NormalizeCallback', 'VQKDCallback') or spec['normalize']
    want = _oracle_gx(x.float(), out['W'].cpu(), out['quant'], step['gz'], spec['losses'], normalize)
    _check_gx(out['gx'], want, dtype)


@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_gx_at_full_size_matches_the_restatement(dev, dtype):
    """cfg 2 shape (65 536 tokens x 32): the half-lane row geometry of the large launches."""
    N, K, D = 65536, 8192, 32
    x, W = O.synthetic_latents(N, K, D, seed=11, normalized_codebook=True)
    x = x.to(dtype)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(12))
    cfg = _node(K, D, 'Cosine', callbacks=[dict(type='VQKDCallback', ema=dict())], type_='VQKDQuantizer')
    cfg['losses'] = dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True)))
    q = _build(cfg, dev, W, training=False)
    out = _step(q, x, gz, dev)
    want = _oracle_gx(x.float(), out['W'].cpu(), out['quant'], gz, _spec_losses(cfg), normalize=True)
    _check_gx(out['gx'], want, dtype)


# ---- 3. degenerate rows ---------------------------------------------------------------------------------------------
def test_zero_token_row_gets_the_straight_through_gradient(dev):
    N, K, D = 1024, 256, 32
    x, W = O.synthetic_latents(N, K, D, seed=21)
    x[17] = 0
    x[600] = 0
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(22))
    off = _step(_build(_node(K, D, rotation_trick=False), dev, W), x, gz, dev)
    on = _step(_build(_node(K, D), dev, W), x, gz, dev)
    assert torch.equal(off['quant'], on['quant'])
    for r in (17, 600):
        assert torch.equal(off['gx'][r], on['gx'][r]), r
    assert not torch.equal(off['gx'], on['gx'])


@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_antipodal_token_and_zero_code_are_finite_and_match_the_restatement(dev, dtype):
    D = 32
    g = torch.Generator().manual_seed(31)
    # K = 1: every token is assigned the one code; token 0 is -2 e (antipodal, s = 0), the rest random
    e = torch.randn(1, D, generator=g).to(torch.bfloat16).float()      # bf16-representable: -2e is exact in bf16
    x = torch.randn(256, D, generator=g)
    x[0] = -2 * e[0]
    x = x.to(dtype)
    gz = torch.randn(256, D, generator=g)
    cfg = _node(1, D)
    out = _step(_build(cfg, dev, e), x, gz, dev)
    assert torch.isfinite(out['gx'].float()).all()
    want = _oracle_gx(x.float(), out['W'].cpu(), out['quant'], gz, _spec_losses(cfg), normalize=False)
    _check_gx(out['gx'], want, dtype)
    # a zero code row: the tokens near the origin are assigned to it (L2) and fall back to straight-through
    W = torch.randn(4, D, generator=g) * 4
    W[2] = 0
    x = torch.randn(256, D, generator=g) * 0.05
    x[128:] = W[1] + 0.1 * torch.randn(128, D, generator=g)
    x = x.to(dtype)
    out = _step(_build(_node(4, D), dev, W), x, gz, dev)
    assert (out['quant'] == 2).sum() >= 64 and (out['quant'] == 1).sum() >= 64
    assert torch.isfinite(out['gx'].float()).all()
    want = _oracle_gx(x.float(), out['W'].cpu(), out['quant'], gz, _spec_losses(_node(4, D)), normalize=False)
    _check_gx(out['gx'], want, dtype)


# ---- 4. grouped quantizer ---------------------------------------------------------------------------------------------
def _gvq(dev, Ws, metric, rotation_trick=True):
    K, Dg = Ws[0].shape
    q = vqb.build_quantizer(dict(type='GroupedVectorQuantizer', num_groups=len(Ws),
                                 quantizer=_node(K, Dg, metric, norm=True, rotation_trick=rotation_trick))).to(dev)
    with torch.no_grad():
        for grp, W in zip(q.quantizers, Ws):
            grp.embedding.weight.copy_(W)
    return q


def _grouped_inputs(N, K, Dg, G, seed):
    xs, Ws = [], []
    for g in range(G):
        x, E = O.synthetic_latents(N, K, Dg, seed=seed + 17 * g)
        xs.append(x)
        Ws.append(E)
    return torch.cat(xs, 1), Ws


@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
def test_one_group_is_the_rotated_vector_quantizer(dev, metric, dtype):
    N, K, D = 4096, 1024, 32
    x, Ws = _grouped_inputs(N, K, D, 1, seed=41)
    x = x.to(dtype)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(42))
    torch.use_deterministic_algorithms(True)
    try:
        a = _step(_build(_node(K, D, metric, norm=True), dev, Ws[0]), x, gz, dev)
        q = _gvq(dev, Ws, metric)
        xg = x.to(dev).requires_grad_(True)
        z, loss, memo = q(xg, dict())
        W = q.quantizers[0].embedding.weight
        gx, gW = torch.autograd.grad((z, loss), (xg, W), (gz.to(dev), torch.ones_like(loss)))
    finally:
        torch.use_deterministic_algorithms(False)
    assert torch.equal(a['quant'], memo['quant'][:, 0])
    assert torch.equal(a['gx'], gx) and torch.equal(a['gW'], gW)


@pytest.mark.parametrize('G', [2, 4, 8])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_every_group_is_a_standalone_rotated_quantizer(dev, G, dtype):
    b, h, w, K, Dg = 4, 16, 16, 512, 32 if G < 8 else 8
    N = b * h * w
    x, Ws = _grouped_inputs(N, K, Dg, G, seed=50 + G)
    x = x.to(dtype)
    gz = torch.randn(N, G * Dg, generator=torch.Generator().manual_seed(G))
    res = {}
    for deterministic in (False, True):
        torch.use_deterministic_algorithms(deterministic)
        try:
            q = _gvq(dev, Ws, 'Cosine')
            xg = x.to(dev).requires_grad_(True)
            z, loss, memo = q(xg, dict())
            gx, = torch.autograd.grad((z, loss), (xg,), (gz.to(dev), torch.ones_like(loss)))
            res[deterministic] = (gx, memo['quant'])
        finally:
            torch.use_deterministic_algorithms(False)
    assert torch.equal(res[False][0], res[True][0])        # the rows variant gives the atomic variant's gx
    gx, quant = res[False]
    for g in range(G):
        sl = slice(g * Dg, (g + 1) * Dg)
        vq = _build(_node(K, Dg, 'Cosine', norm=True), dev, Ws[g])
        xs = x[:, sl].contiguous().to(dev).requires_grad_(True)
        zg, lg, mg = vq(xs, dict())
        gxs, = torch.autograd.grad((zg, lg / G), (xs,), (gz[:, sl].contiguous().to(dev), torch.ones_like(lg)))
        assert torch.equal(quant[:, g], mg['quant']), g
        assert torch.equal(gx[:, sl], gxs), g


# ---- 5. reproducibility -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('grouped', [False, True], ids=['vq', 'gvq'])
def test_gx_is_reproducible_and_graph_replay_matches_eager(dev, grouped):
    b, h, w, K, D = 16, 16, 16, 1024, 32
    x_cpu, W = O.synthetic_latents(b * h * w, K, D, seed=61)
    if grouped:
        q = _gvq(dev, [W[:, :16].contiguous(), W[:, 16:].contiguous()], 'L2')
        params = [grp.embedding.weight for grp in q.quantizers]
    else:
        q = _build(_node(K, D, 'Cosine', norm=True), dev, W)
        params = [q.embedding.weight]
    x = _nchw(x_cpu.to(torch.bfloat16), b, h, w).to(dev).requires_grad_(True)
    gz = torch.randn(b, D, h, w, generator=torch.Generator().manual_seed(62)).to(dev)
    res = {}

    def step():
        z, loss, memo = tokenizer.quantize(q, x, dict())
        grads = torch.autograd.grad((z, loss), [x] + params, (gz, torch.ones_like(loss)))
        res.update(z=z.detach(), gx=grads[0])

    def run(fn):
        fn()
        torch.cuda.synchronize()
        return {k: v.clone() for k, v in res.items()}

    eager = run(step)
    again = run(step)
    assert torch.equal(eager['gx'], again['gx']) and torch.equal(eager['z'], again['z'])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(2):
        replay = run(graph.replay)
        assert torch.equal(eager['gx'], replay['gx']) and torch.equal(eager['z'], replay['z'])
    del graph
