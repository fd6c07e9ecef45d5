"""The rotation trick over the whole depth of a ResidualVectorQuantizer on the B200: on against off (everything but gx
bit-identical), L = 1 against the rotated VQGANQuantizer (bit for bit), gx against the float64 restatement over the
depths, row geometries, dtypes, metrics and loss terms, the degenerate rows, reproducibility (deterministic variant,
run to run, CUDA-graph replay), the launch count and one full-size case."""
import re

import einops
import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rotation as R
from vector_quantization_b200 import tokenizer

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.bfloat16]
DT_IDS = ['fp32', 'bf16']
METRIC = {'L2': 'L2Distance', 'Cosine': 'CosineDistance'}
CVQ = [dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'), ema=dict())]


def _level(K, D, metric='L2', norm=False, callbacks=(), rotation_trick=False):
    losses = dict(vqgan_loss=dict(type='VQGANLoss'))
    if norm:
        losses['commit_norm'] = dict(type='CommitmentLoss', mse=dict(norm=True))
    node = dict(type='VQGANQuantizer', distance=dict(type=METRIC[metric]), callbacks=list(callbacks), losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D))
    if rotation_trick:
        node['rotation_trick'] = True
    return node


def _spec_losses(node):
    return {name: dict(type=c['type'], norm=c.get('mse', {}).get('norm', False)) for name, c in node['losses'].items()}


def _rvq(dev, Ws, metric='L2', norm=False, callbacks=(), rotation_trick=True, training=True):
    K, D = Ws[0].shape
    q = vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=len(Ws), rotation_trick=rotation_trick,
                                 quantizer=_level(K, D, metric, norm, callbacks)), training=training).to(dev)
    with torch.no_grad():
        for level, W in zip(q.quantizers, Ws):
            level.embedding.weight.copy_(W)
    return q


def _inputs(N, K, D, L, seed):
    """Clustered latents around the first codebook; deeper codebooks at the scale of what is left over."""
    x, E = O.synthetic_latents(N, K, D, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    Ws = [E] + [torch.randn(K, D, generator=g) * 0.5 * E.std() * 0.8 ** (l - 1) for l in range(1, L)]
    return x, Ws


def _nchw(t, b, h, w):
    return einops.rearrange(t, '(b h w) c -> b c h w', b=b, h=h, w=w).contiguous()


def _tokens(t, b, h, w):
    return einops.rearrange(t, 'b c h w -> (b h w) c', b=b, h=h, w=w)


def _step(q, x_cpu, gz_cpu, dev, hw=None):
    """forward + backward (upstream: gz on z, 1 on the loss) of a residual or single quantizer; z / gx come back
    token-major, quant as [N, L]."""
    params = [lv.embedding.weight for lv in q.quantizers] if hasattr(q, 'quantizers') else [q.embedding.weight]
    if hw is not None:
        b, h, w = hw
        x = _nchw(x_cpu, b, h, w).to(dev).requires_grad_(True)
        z, loss, memo = tokenizer.quantize(q, x, dict())
        memo = memo['quantizer']
        grads = torch.autograd.grad((z, loss), [x] + params, (_nchw(gz_cpu, b, h, w).to(dev), torch.ones_like(loss)))
        z, gx = _tokens(z.detach(), b, h, w), _tokens(grads[0], b, h, w)
    else:
        x = x_cpu.to(dev).requires_grad_(True)
        z, loss, memo = q(x, dict())
        grads = torch.autograd.grad((z, loss), [x] + params, (gz_cpu.to(dev), torch.ones_like(loss)))
        gx = grads[0]
    N = x_cpu.shape[0]
    return dict(z=z.detach(), loss=loss.detach(), losses={k: v.detach() for k, v in memo['loss'].items()},
                quant=memo['quant'].reshape(N, -1).clone(), gx=gx, gWs=list(grads[1:]),
                Ws=[p.detach().clone() for p in params])


def _oracle_gx(x_cpu, Ws_used, quant, gz, losses, scale=1.0):
    """float64 gx of (z * gz).sum() + scale * loss with the whole-depth rotation, on the kernel's own indices and
    codebooks: r_0 = x, e_l = W_l[q_l], r_l = r_{l-1} - e_l, zhat = sum_l e_l, z = rotate_to(x, zhat)."""
    x = x_cpu.double().requires_grad_(True)
    spec = O.QuantizerSpec(losses=losses)
    r, zhat, total = x, None, 0.0
    for l, W in enumerate(Ws_used):
        e = W.double().cpu()[quant[:, l].cpu()]
        total = total + sum(O._losses(spec, e, r).values())
        zhat = e if zhat is None else zhat + e
        r = r - e
    z = R.rotate_to(x, zhat)
    ((z * gz.double()).sum() + scale * total).backward()
    return x.grad


def _check_gx(gx, want, dtype):
    gx = gx.float().cpu().double()
    scale = float(want.abs().max())
    if dtype == torch.bfloat16:     # gx comes back in the token dtype: one bf16 rounding
        torch.testing.assert_close(gx, want, rtol=2 ** -7, atol=1e-4 * scale)
    else:
        torch.testing.assert_close(gx, want, rtol=1e-4, atol=1e-5 * scale)


# ---- 1. on against off ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nchw', [False, True], ids=['tokens', 'nchw'])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('L', [2, 4])
def test_rotation_changes_only_gx(dev, L, metric, dtype, nchw):
    b, h, w, K, D = 4, 16, 16, 512, 32
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=100 + L)
    x_cpu = x_cpu.to(dtype)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(L))
    res = []
    torch.use_deterministic_algorithms(True)      # gW through the segment sum: comparable bit for bit
    try:
        for rot in (False, True):
            q = _rvq(dev, Ws, metric, norm=True, callbacks=CVQ, rotation_trick=rot)
            out = _step(q, x_cpu, gz, dev, hw=(b, h, w) if nchw else None)
            out['probs'] = [lv._probability.clone() for lv in q.quantizers]
            res.append(out)
    finally:
        torch.use_deterministic_algorithms(False)
    off, on = res
    for key in ('z', 'loss', 'quant'):
        assert torch.equal(off[key], on[key]), key
    assert off['losses'].keys() == on['losses'].keys()
    assert all(torch.equal(off['losses'][k], on['losses'][k]) for k in off['losses'])
    for key in ('Ws', 'probs', 'gWs'):       # the codebooks after this step's CVQ-VAE update, and their gradients
        assert all(torch.equal(a, b) for a, b in zip(off[key], on[key])), key
    assert not torch.equal(off['gx'], on['gx'])


# ---- 2. L = 1 is the rotated VQGANQuantizer ---------------------------------------------------------------------------
@pytest.mark.parametrize('norm', [False, True], ids=['plain', 'norm'])
@pytest.mark.parametrize('nchw', [False, True], ids=['tokens', 'nchw'])
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_depth_one_is_the_rotated_vector_quantizer(dev, dtype, metric, nchw, norm):
    b, h, w, K, D = 4, 16, 16, 1024, 32
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, 1, seed=5)
    x_cpu = x_cpu.to(dtype)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(6))
    vq = vqb.build_quantizer(_level(K, D, metric, norm, rotation_trick=True)).to(dev)
    with torch.no_grad():
        vq.embedding.weight.copy_(Ws[0])
    torch.use_deterministic_algorithms(True)
    try:
        a = _step(vq, x_cpu, gz, dev, hw=(b, h, w) if nchw else None)
        r = _step(_rvq(dev, Ws, metric, norm), x_cpu, gz, dev, hw=(b, h, w) if nchw else None)
    finally:
        torch.use_deterministic_algorithms(False)
    assert torch.equal(a['quant'], r['quant']) and torch.equal(a['z'], r['z'])
    assert a['gx'].dtype == r['gx'].dtype == dtype and torch.equal(a['gx'], r['gx'])
    assert torch.equal(a['gWs'][0], r['gWs'][0])


# ---- 3. gx against the float64 restatement ------------------------------------------------------------------------------
# row geometries (V elements x G lanes x NV slices per lane) at N = 1024: 8 -> V8 G1 NV1, 20 -> scalar G32 NV1,
# 32 / 64 / 256 -> V8 NV1, 100 -> scalar G32 NV4, 512 -> V8 G32 NV2, 768 -> V8 G32 NV4, 2048 -> V8 G32 NV8; the
# half-lane NV = 2 geometry of large N (V8, G <= 16) is the separate full-width case below
_DS = [8, 20, 32, 64, 100, 256, 512, 768, 2048]
_LS = [2, 4, 8, 16]


def _geometry(D, N, sms):
    """(G, V, NV) of row_geom in csrc/quantize.cu."""
    V = 8 if D % 8 == 0 else 1
    slices = -(-D // V)
    G = 1
    while G < 32 and G < slices:
        G <<= 1
    NV = 1
    while NV * G < slices:
        NV <<= 1
    if V == 8 and NV == 1 and 2 <= G <= 16 and N * G > sms * 1536:
        G, NV = G >> 1, 2
    return G, V, NV


def _backward_instantiations(prof):
    """{(G, V, NV, kRotate)} of the residual_backward_kernel launches in a profile (demangled or mangled names)."""
    out = set()
    for e in prof.events():
        if 'residual_backward_kernel' not in e.name:
            continue
        m = re.search(r'residual_backward_kernel<([^<>]*)>', e.name)
        if m:
            args = [t.strip() for t in m.group(1).split(',')]
            out.add((int(args[2]), int(args[3]), int(args[4]), args[6] == 'true'))
            continue
        m = re.search(r'Li(\d+)ELi(\d+)ELi(\d+)ELb[01]ELb([01])E', e.name)
        assert m, e.name
        out.add((int(m[1]), int(m[2]), int(m[3]), m[4] == '1'))
    return out


def _rotated_step_against_the_restatement(dev, x_cpu, Ws, gz, metric, norm, dtype, hw):
    N, D = x_cpu.shape
    K = Ws[0].shape[0]
    q = _rvq(dev, Ws, metric, norm)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = _step(q, x_cpu.to(dtype), gz, dev, hw=hw)
        torch.cuda.synchronize()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    assert _backward_instantiations(prof) == {_geometry(D, N, sms) + (True,)}
    assert out['quant'].shape == (N, len(Ws))
    want = _oracle_gx(x_cpu.to(dtype).float(), out['Ws'], out['quant'], gz, _spec_losses(_level(K, D, metric, norm)))
    _check_gx(out['gx'], want, dtype)


@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('D', _DS)
def test_gx_matches_the_restatement(dev, D, metric, dtype):
    i = _DS.index(D) + (metric == 'Cosine')
    L = _LS[i % 4]
    norm = i % 2 == 1
    nchw = (i + (dtype == torch.bfloat16)) % 2 == 0
    b, h, w, K = 4, 16, 16, 512
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=7 * D + L)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(D + 1))
    _rotated_step_against_the_restatement(dev, x_cpu, Ws, gz, metric, norm, dtype, (b, h, w) if nchw else None)


@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_gx_of_the_half_lane_geometry_matches_the_restatement(dev, dtype):
    """65 536 tokens x 32 (the cfg 2 shape): N * G exceeds the resident threads, so the V = 8, NV = 1 row of four lanes
    becomes two lanes with NV = 2."""
    b, h, w, D, K, L = 256, 16, 16, 32, 1024, 4
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=131)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(132))
    bf16 = dtype == torch.bfloat16
    _rotated_step_against_the_restatement(dev, x_cpu, Ws, gz, 'Cosine' if bf16 else 'L2', bf16, dtype,
                                          (b, h, w) if bf16 else None)


# ---- 4. degenerate rows ---------------------------------------------------------------------------------------------
def test_zero_token_row_gets_the_straight_through_gradient(dev):
    N, K, D, L = 1024, 256, 32, 3
    x, Ws = _inputs(N, K, D, L, seed=21)
    x[17] = 0
    x[600] = 0
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(22))
    off = _step(_rvq(dev, Ws, rotation_trick=False), x, gz, dev)
    on = _step(_rvq(dev, Ws), x, gz, dev)
    assert torch.equal(off['quant'], on['quant'])
    for r in (17, 600):
        assert torch.equal(off['gx'][r], on['gx'][r]), r
    assert not torch.equal(off['gx'], on['gx'])


@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_zero_zhat_and_antipodal_token(dev, dtype):
    D = 32
    g = torch.Generator().manual_seed(31)
    e = torch.randn(1, D, generator=g).to(torch.bfloat16).float()      # bf16-representable, as are -e, 2e and -4e
    x = (torch.randn(256, D, generator=g) * 2).to(dtype)
    gz = torch.randn(256, D, generator=g)
    # K = 1 codebooks, W_1 = -W_0: zhat_L = 0 exactly for every token, which keeps the straight-through gradient
    off = _step(_rvq(dev, [e, -e], rotation_trick=False), x, gz, dev)
    on = _step(_rvq(dev, [e, -e]), x, gz, dev)
    assert not on['z'].any()                       # z = x + (0 - x)
    assert torch.equal(off['gx'], on['gx'])
    # W_1 = W_0: zhat_L = 2 e; token 0 is x = -2 zhat_L (antipodal: s = 0), the rest random
    x[0] = -4 * e[0]
    out = _step(_rvq(dev, [e, e]), x, gz, dev)
    assert torch.isfinite(out['gx'].float()).all()
    want = _oracle_gx(x.float(), out['Ws'], out['quant'], gz, _spec_losses(_level(1, D)))
    _check_gx(out['gx'], want, dtype)


# ---- 5. reproducibility -----------------------------------------------------------------------------------------------
def test_gx_is_reproducible_deterministic_and_graph_replay_matches_eager(dev):
    b, h, w, K, D, L = 16, 16, 16, 1024, 32, 4
    x_cpu, Ws = _inputs(b * h * w, K, D, L, seed=61)
    q = _rvq(dev, Ws, 'Cosine', norm=True)
    params = [lv.embedding.weight for lv in q.quantizers]
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
    torch.use_deterministic_algorithms(True)      # the _rows variant gives the atomic variant's gx
    try:
        det = run(step)
    finally:
        torch.use_deterministic_algorithms(False)
    assert torch.equal(eager['gx'], det['gx'])
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


# ---- 6. launch count -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('L', [1, 4, 8])
def test_one_step_launch_per_level_and_one_backward_launch(dev, L):
    N, K, D = 4096, 512, 32
    x_cpu, Ws = _inputs(N, K, D, L, seed=81)
    q = _rvq(dev, Ws)
    x = x_cpu.to(dev).requires_grad_(True)
    q(x, dict())          # warm-up
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        z, loss, _ = q(x, dict())
        torch.autograd.backward((z, loss), (torch.ones_like(z), torch.ones_like(loss)))
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert sum('residual_step_kernel' in n for n in names) == L
    assert sum('residual_backward_kernel' in n for n in names) == 1
    assert not any('quantize_backward_kernel' in n or 'quantize_forward_kernel' in n for n in names)


# ---- 7. full size ----------------------------------------------------------------------------------------------------
def test_full_size_matches_the_restatement_on_a_subset(dev):
    """[256, 256, 8, 8] latents, K 16384, L 4, L2 + VQGANLoss, through tokenizer.quantize; gx of 4096 seeded rows
    against the restatement (the loss term scaled to its share of the full mean)."""
    b, D, h, w, K, L = 256, 256, 8, 8, 16384, 4
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=91)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(92))
    q = _rvq(dev, Ws)
    out = _step(q, x_cpu, gz, dev, hw=(b, h, w))
    rows = torch.randperm(N, generator=torch.Generator().manual_seed(93))[:4096]
    want = _oracle_gx(x_cpu[rows], out['Ws'], out['quant'][rows.to(dev)], gz[rows],
                      _spec_losses(_level(K, D)), scale=rows.numel() / N)
    _check_gx(out['gx'][rows.to(dev)], want, torch.float32)
