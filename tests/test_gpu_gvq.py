"""GroupedVectorQuantizer on the B200: G = 1 against VectorQuantizer (bit for bit), every group against a standalone
VectorQuantizer on its column slice (bit for bit), the CPU restatement (oracle/gvq.py), CVQ-VAE groups in training, the
token round trip, the deterministic gradient, CUDA-graph replay and the launch count of the fused forward / backward."""
import einops
import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import gvq as GV
from oracle import oracle as O
from vector_quantization_b200 import tokenizer

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.bfloat16]
DT_IDS = ['fp32', 'bf16']
METRIC = {'L2': 'L2Distance', 'Cosine': 'CosineDistance'}
LOSSES = dict(vqgan_loss=dict(type='VQGANLoss'), commit_norm=dict(type='CommitmentLoss', mse=dict(norm=True)))
SPEC_LOSSES = {'vqgan_loss': dict(type='VQGANLoss'), 'commit_norm': dict(type='CommitmentLoss', norm=True)}


def _group(K, Dg, metric, callbacks=()):
    return dict(type='VQGANQuantizer', distance=dict(type=METRIC[metric]), callbacks=list(callbacks), losses=LOSSES,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=Dg))


def _gvq(dev, Ws, metric, callbacks=(), training=True):
    K, Dg = Ws[0].shape
    q = vqb.build_quantizer(dict(type='GroupedVectorQuantizer', num_groups=len(Ws),
                                 quantizer=_group(K, Dg, metric, callbacks)), training=training).to(dev)
    with torch.no_grad():
        for group, W in zip(q.quantizers, Ws):
            group.embedding.weight.copy_(W)
    return q


def _vq(dev, W, metric, callbacks=(), training=True):
    q = vqb.build_quantizer(_group(W.shape[0], W.shape[1], metric, callbacks), training=training).to(dev)
    with torch.no_grad():
        q.embedding.weight.copy_(W)
    return q


def _inputs(N, K, Dg, G, seed):
    """Clustered latents per group around that group's codebook."""
    xs, Ws = [], []
    for g in range(G):
        x, E = O.synthetic_latents(N, K, Dg, seed=seed + 17 * g)
        xs.append(x)
        Ws.append(E)
    return torch.cat(xs, 1), Ws


def _grads(z, loss, x, Ws, gz):
    grads = torch.autograd.grad((z, loss), [x] + list(Ws), (gz, torch.ones_like(loss)), allow_unused=True)
    return grads[0], list(grads[1:])


def _tokens(t, b, h, w):
    return einops.rearrange(t, 'b c h w -> (b h w) c', b=b, h=h, w=w)


def _nchw(t, b, h, w):
    return einops.rearrange(t, '(b h w) c -> b c h w', b=b, h=h, w=w).contiguous()


def _run_grouped(q, x_cpu, gz_cpu, dtype, nchw, b, h, w, dev):
    """forward + backward of the grouped module; z / gx come back token-major."""
    W = [g.embedding.weight for g in q.quantizers]
    if nchw:
        x = _nchw(x_cpu.to(dtype), b, h, w).to(dev).requires_grad_(True)
        z, loss, memo = tokenizer.quantize(q, x, dict())
        memo = memo['quantizer']
        gx, gWs = _grads(z, loss, x, W, _nchw(gz_cpu, b, h, w).to(dev))
        z, gx = _tokens(z.detach(), b, h, w), _tokens(gx, b, h, w)
    else:
        x = x_cpu.to(dtype).to(dev).requires_grad_(True)
        z, loss, memo = q(x, dict())
        gx, gWs = _grads(z, loss, x, W, gz_cpu.to(dev))
    return z.detach(), loss.detach(), memo, gx, gWs


# ---- 1. G = 1 is VectorQuantizer --------------------------------------------------------------------------------------
@pytest.mark.parametrize('nchw', [False, True], ids=['tokens', 'nchw'])
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_one_group_is_bit_identical_to_vector_quantizer(dev, dtype, metric, nchw):
    b, h, w, K, D = 4, 16, 16, 1024, 32
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, 1, seed=5)
    vq, gvq = _vq(dev, Ws[0], metric), _gvq(dev, Ws, metric)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(6))
    res = []
    torch.use_deterministic_algorithms(True)      # gW through the segment sum: comparable bit for bit
    try:
        for q, W in ((vq, vq.embedding.weight), (gvq, gvq.quantizers[0].embedding.weight)):
            x = x_cpu.to(dtype).to(dev)
            if nchw:
                x = _nchw(x, b, h, w).requires_grad_(True)
                z, loss, memo = tokenizer.quantize(q, x, dict())
                memo = memo['quantizer']
                g = _nchw(gz, b, h, w).to(dev)
            else:
                x.requires_grad_(True)
                z, loss, memo = q(x, dict())
                g = gz.to(dev)
            gx, (gW,) = _grads(z, loss, x, [W], g)
            res.append(dict(z=z.detach(), loss=loss.detach(), quant=memo['quant'].reshape(N, -1)[:, 0], gx=gx, gW=gW,
                            losses={k: v.detach() for k, v in memo['loss'].items()}))
    finally:
        torch.use_deterministic_algorithms(False)
    a, r = res
    for key in ('z', 'loss', 'quant', 'gx', 'gW'):
        assert a[key].dtype == r[key].dtype and a[key].shape == r[key].shape and torch.equal(a[key], r[key]), key
    assert a['losses'].keys() == r['losses'].keys() and all(torch.equal(a['losses'][k], r['losses'][k]) for k in a['losses'])


# ---- 2. every group is its own VectorQuantizer on x_g.contiguous() ------------------------------------------------------
# a seeded sweep: each G, Dg (scalar path, folded L2, zero-copy bf16, certified pass), K, metric, dtype and layout
# appears at least once
_SWEEP = [(2, 6, 512, 'L2', torch.float32, False), (4, 8, 8192, 'L2', torch.bfloat16, True),
          (8, 32, 512, 'Cosine', torch.bfloat16, False), (2, 64, 8192, 'Cosine', torch.float32, True),
          (4, 256, 512, 'Cosine', torch.bfloat16, True), (2, 256, 8192, 'L2', torch.float32, False),
          (8, 6, 8192, 'Cosine', torch.float32, True), (4, 32, 8192, 'L2', torch.bfloat16, False)]


@pytest.mark.parametrize('G,Dg,K,metric,dtype,nchw', _SWEEP,
                         ids=[f'G{G}-Dg{Dg}-K{K}-{m}-{DT_IDS[DTYPES.index(dt)]}-{"nchw" if n else "tokens"}'
                              for G, Dg, K, m, dt, n in _SWEEP])
def test_every_group_is_bit_identical_to_a_standalone_quantizer(dev, G, Dg, K, metric, dtype, nchw):
    b, h, w = 8, 16, 16
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, Dg, G, seed=G * 100 + Dg + K)
    gz = torch.randn(N, G * Dg, generator=torch.Generator().manual_seed(7))
    q = _gvq(dev, Ws, metric)
    torch.use_deterministic_algorithms(True)
    try:
        z, loss, memo, gx, gWs = _run_grouped(q, x_cpu, gz, dtype, nchw, b, h, w, dev)
        assert memo['quant'].shape == (N, G) and len(memo['groups']) == G
        for g in range(G):
            sl = slice(g * Dg, (g + 1) * Dg)
            vq = _vq(dev, Ws[g], metric)
            xg = x_cpu[:, sl].to(dtype).contiguous().to(dev).requires_grad_(True)
            zg, lg, mg = vq(xg, dict())
            gxg, (gWg,) = _grads(zg, lg / G, xg, [vq.embedding.weight], gz[:, sl].contiguous().to(dev))
            assert torch.equal(memo['quant'][:, g], mg['quant']), g
            assert torch.equal(z[:, sl], zg.detach()), g
            for name, value in mg['loss'].items():
                assert torch.equal(memo['groups'][g]['loss'][name], value), (g, name)
            assert torch.equal(gx[:, sl], gxg), g
            assert torch.equal(gWs[g], gWg), g
    finally:
        torch.use_deterministic_algorithms(False)
    want = None
    for name in LOSSES:
        total = memo['groups'][0]['loss'][name]
        for g in range(1, G):
            total = total + memo['groups'][g]['loss'][name]
        assert torch.equal(memo['loss'][name], total / G)
        want = memo['loss'][name] if want is None else want + memo['loss'][name]
    assert torch.equal(loss, want)


# ---- 3. against the restatement ---------------------------------------------------------------------------------------
@pytest.mark.parametrize('G,Dg,K,metric,dtype,nchw', _SWEEP[:6],
                         ids=[f'G{G}-Dg{Dg}-K{K}-{m}-{DT_IDS[DTYPES.index(dt)]}-{"nchw" if n else "tokens"}'
                              for G, Dg, K, m, dt, n in _SWEEP[:6]])
def test_matches_the_restatement(dev, G, Dg, K, metric, dtype, nchw):
    b, h, w = 4, 16, 16
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, Dg, G, seed=G * 10 + Dg + K)
    xt = x_cpu.to(dtype)
    gz = torch.randn(N, G * Dg, generator=torch.Generator().manual_seed(9))
    q = _gvq(dev, Ws, metric)
    z, loss, memo, gx, gWs = _run_grouped(q, xt.float(), gz, dtype, nchw, b, h, w, dev)
    spec = O.QuantizerSpec(distance=metric, training=True, losses=SPEC_LOSSES)
    xo = xt.float().requires_grad_(True)
    ref = GV.gvq_forward(spec, xo, Ws)
    (ref['loss'] + (ref['z_ste'] * gz).sum()).backward()
    qg, qr = memo['quant'].cpu(), ref['quant']
    for g in range(G):       # the near-tie index policy of DESIGN.md §5, per group
        rows = (qg[:, g] != qr[:, g]).nonzero().flatten()
        d = ref['groups'][g]['distance'][0]
        gap = d[rows, qg[rows, g]] - d[rows, qr[rows, g]]
        assert (gap.abs() < 1e-5).all(), f'group {g}: index mismatch beyond a near-tie, gaps {gap.tolist()}'
    ok = (qg == qr).all(1)
    n_bad = int((~ok).sum())
    assert n_bad <= max(2, N // 200)
    torch.testing.assert_close(z.cpu()[ok], ref['z_ste'].detach()[ok], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(loss.cpu(), ref['loss'].detach(), rtol=1e-5 + 8 * n_bad / N, atol=1e-7)
    if dtype == torch.bfloat16:
        torch.testing.assert_close(gx.float().cpu()[ok], xo.grad[ok], rtol=2 ** -7, atol=1e-6)
    else:
        torch.testing.assert_close(gx.cpu()[ok], xo.grad[ok], rtol=1e-4, atol=1e-7)
    for g in range(G):
        want = ref['weight_leafs'][g].grad
        touched = torch.zeros(K, dtype=torch.bool)
        touched[qg[~ok, g]] = True
        touched[qr[~ok, g]] = True
        torch.testing.assert_close(gWs[g].cpu()[~touched], want[~touched], rtol=1e-4,
                                   atol=1e-4 * float(want.abs().max()))


# ---- 4. CVQ-VAE in every group ----------------------------------------------------------------------------------------
def test_cvqvae_groups_train_like_standalone_quantizers(dev):
    """Two training steps, both forwards before the first backward: each group's update of step 2 must leave the
    codebook that step 1's backward saved intact (copy-on-write per group)."""
    N, K, Dg, G = 4096, 512, 32, 4
    cb = [dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'), ema=dict())]
    x1, Ws = _inputs(N, K, Dg, G, seed=31)
    x2, _ = _inputs(N, K, Dg, G, seed=32)
    gz = torch.randn(N, G * Dg, generator=torch.Generator().manual_seed(33)).to(dev)
    q = _gvq(dev, Ws, 'Cosine', callbacks=cb)
    xa = x1.to(dev).requires_grad_(True)
    za, la, _ = q(xa, dict())
    q(x2.to(dev), dict())
    (gx,) = torch.autograd.grad((za, la), (xa,), (gz, torch.ones_like(la)))
    for g in range(G):
        sl = slice(g * Dg, (g + 1) * Dg)
        vq = _vq(dev, Ws[g], 'Cosine', callbacks=cb)
        xg = x1[:, sl].contiguous().to(dev).requires_grad_(True)
        zg, lg, _ = vq(xg, dict())
        vq(x2[:, sl].contiguous().to(dev), dict())
        (gxg,) = torch.autograd.grad((zg, lg / G), (xg,), (gz[:, sl].contiguous(), torch.ones_like(lg)))
        group = q.quantizers[g]
        torch.testing.assert_close(group._probability, vq._probability, rtol=1e-5, atol=1e-7)
        torch.testing.assert_close(group.embedding.weight.detach(), vq.embedding.weight.detach(), rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(gx[:, sl], gxg, rtol=1e-4, atol=1e-7)
        assert not torch.equal(group.embedding.weight.detach().cpu(), Ws[g])     # the codebook did train


# ---- 5. token round trip ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('bhw', [(4, 8, 12), (3, 5, 7)], ids=lambda s: 'x'.join(map(str, s)))
@pytest.mark.parametrize('K,Dg', [(512, 8), (70000, 6)])
def test_encode_to_quant_then_decode_from_quant_is_the_group_concatenation(dev, K, Dg, bhw):
    (b, h, w), G = bhw, 4
    x_cpu, Ws = _inputs(b * h * w, K, Dg, G, seed=41)
    q = _gvq(dev, Ws, 'L2', training=False)
    x = _nchw(x_cpu, b, h, w).to(dev)
    with torch.no_grad():
        ids, _ = tokenizer.encode_to_quant(q, x, dict(), compact=True)
        wide, _ = tokenizer.encode_to_quant(q, x, dict())
        z, _, fmemo = tokenizer.quantize(q, x, dict())
    assert ids.shape == (b, h, w, G) and ids.dtype == (torch.uint16 if K <= 65536 else torch.int32)
    assert wide.dtype == torch.int64 and torch.equal(ids.cpu().to(torch.int32).long(), wide.cpu())
    assert torch.equal(fmemo['quantizer']['quant'].cpu(), wide.cpu().view(-1, G))
    e = GV.group_concat(Ws, wide.cpu())                                     # [b, h, w, D]
    want = einops.rearrange(e, 'b h w c -> b c h w').contiguous()
    for ids_dev in (ids, wide, wide.to(torch.int32)):
        for dtype in DTYPES:
            out, _ = tokenizer.decode_from_quant(q, ids_dev, dict(), dtype=dtype)
            assert out.shape == (b, G * Dg, h, w) and out.dtype == dtype and out.is_contiguous()
            assert torch.equal(out.cpu(), want.to(dtype))
    zt, _ = q.decode(wide.view(-1, G), dict())
    assert torch.equal(zt.cpu(), e.view(-1, G * Dg))
    assert torch.equal(z.cpu(), x.cpu() + (want - x.cpu()))


def test_bad_ids_in_any_group(dev):
    b, h, w, K, Dg, G = 2, 4, 4, 512, 16, 3
    _, Ws = _inputs(8, K, Dg, G, seed=51)
    q = _gvq(dev, Ws, 'L2', training=False)
    ids = torch.randint(0, K, (b, h, w, G), generator=torch.Generator().manual_seed(52))
    bad = ids.clone()
    bad[0, 1, 2, 0] = K
    bad[1, 3, 0, G - 1] = K + 9
    bad[1, 0, 0, 1] = -1
    mask = (bad < 0).any(-1) | (bad >= K).any(-1)
    for dt in (torch.int64, torch.int32):
        with pytest.raises(IndexError, match=rf'^3 token id\(s\) outside \[0, {K}\)'):
            tokenizer.decode_from_quant(q, bad.to(dt).to(dev), dict())
        dev_ids = bad.to(dt).to(dev)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode('error')        # check=False must not synchronise
        try:
            z, _ = tokenizer.decode_from_quant(q, dev_ids, dict(), check=False)
        finally:
            torch.cuda.set_sync_debug_mode('default')
        rows = z.cpu().permute(0, 2, 3, 1)
        assert torch.isnan(rows[mask]).all() and not torch.isnan(rows[~mask]).any()
        assert torch.equal(rows[~mask], GV.group_concat(Ws, ids)[~mask])
    with pytest.raises(ValueError, match=r'\[b, h, w, 3\]'):
        tokenizer.decode_from_quant(q, ids[..., 0].to(dev), dict())


# ---- 6. deterministic gradient ----------------------------------------------------------------------------------------
def test_deterministic_runs_are_bit_identical(dev):
    N, K, Dg, G = 16384, 512, 32, 4
    x_cpu, Ws = _inputs(N, K, Dg, G, seed=61)
    q = _gvq(dev, Ws, 'L2')
    gz = torch.randn(N, G * Dg, generator=torch.Generator().manual_seed(62)).to(dev)
    params = [grp.embedding.weight for grp in q.quantizers]

    def run():
        x = x_cpu.to(dev).requires_grad_(True)
        z, loss, _ = q(x, dict())
        return _grads(z, loss, x, params, gz)

    torch.use_deterministic_algorithms(True)
    try:
        runs = [run() for _ in range(2)]
    finally:
        torch.use_deterministic_algorithms(False)
    atomic = run()
    assert torch.equal(runs[1][0], runs[0][0]) and all(torch.equal(a, b) for a, b in zip(runs[1][1], runs[0][1]))
    assert torch.equal(atomic[0], runs[0][0])
    for a, b in zip(atomic[1], runs[0][1]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-4 * float(b.abs().max()))


# ---- 7. CUDA graph ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('deterministic', [False, True], ids=['atomic', 'deterministic'])
def test_training_step_cuda_graph_matches_eager(dev, deterministic):
    b, h, w, K, Dg, G = 32, 16, 16, 1024, 32, 4
    x_cpu, Ws = _inputs(b * h * w, K, Dg, G, seed=71)
    q = _gvq(dev, Ws, 'Cosine')
    params = [grp.embedding.weight for grp in q.quantizers]
    x = _nchw(x_cpu.to(torch.bfloat16), b, h, w).to(dev).requires_grad_(True)
    gz = torch.randn(b, G * Dg, h, w, generator=torch.Generator().manual_seed(72)).to(dev)
    res = {}

    def step():
        z, loss, memo = tokenizer.quantize(q, x, dict())
        gx, gWs = _grads(z, loss, x, params, gz)
        res.update(z=z.detach(), loss=loss.detach(), quant=memo['quantizer']['quant'], gx=gx,
                   **{f'gW{g}': t for g, t in enumerate(gWs)})

    def run(fn):
        fn()
        torch.cuda.synchronize()
        return {k: v.clone() for k, v in res.items()}

    torch.use_deterministic_algorithms(deterministic)
    try:
        eager = run(step)
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
            for k in eager:
                if k.startswith('gW') and not deterministic:
                    torch.testing.assert_close(replay[k], eager[k], rtol=1e-5, atol=1e-6 * float(eager[k].abs().max()))
                else:
                    assert torch.equal(eager[k], replay[k]), k
        del graph
    finally:
        torch.use_deterministic_algorithms(False)


# ---- 8. launch count --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('G', [2, 8])
def test_one_split_one_gather_and_one_backward_launch(dev, G):
    b, h, w, K, Dg = 16, 16, 16, 512, 16
    x_cpu, Ws = _inputs(b * h * w, K, Dg, G, seed=81)
    q = _gvq(dev, Ws, 'L2')
    x = _nchw(x_cpu, b, h, w).to(dev).requires_grad_(True)
    tokenizer.quantize(q, x, dict())          # warm-up
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        z, loss, _ = tokenizer.quantize(q, x, dict())
        torch.autograd.backward((z, loss), (torch.ones_like(z), torch.ones_like(loss)))
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert sum('split_groups' in n for n in names) == 1
    assert sum('group_forward_kernel' in n for n in names) == 1
    assert sum('group_backward_kernel' in n for n in names) == 1
    assert not any('transpose_last2' in n for n in names)
    assert not any('quantize_backward_kernel' in n or 'quantize_forward_kernel' in n for n in names)
