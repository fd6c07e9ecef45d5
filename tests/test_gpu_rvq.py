"""ResidualVectorQuantizer on the B200: L = 1 against VectorQuantizer (bit for bit), depths 2..8 against the CPU
restatement (oracle/rvq.py), CVQ-VAE levels in training, the token round trip, the deterministic gradient, CUDA-graph
replay and the launch count of the fused forward / backward."""
import itertools

import einops
import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rvq as R
from vector_quantization_b200 import tokenizer

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.bfloat16]
DT_IDS = ['fp32', 'bf16']
METRIC = {'L2': 'L2Distance', 'Cosine': 'CosineDistance'}
LOSSES = dict(vqgan_loss=dict(type='VQGANLoss'), commit_norm=dict(type='CommitmentLoss', mse=dict(norm=True)))
SPEC_LOSSES = {'vqgan_loss': dict(type='VQGANLoss'), 'commit_norm': dict(type='CommitmentLoss', norm=True)}


def _level(K, D, metric, callbacks=(), losses=LOSSES, type_='VQGANQuantizer'):
    return dict(type=type_, distance=dict(type=METRIC[metric]), callbacks=list(callbacks), losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D))


def _rvq(dev, L, Ws, metric, callbacks=(), training=True, losses=LOSSES):
    K, D = Ws[0].shape
    q = vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=L,
                                 quantizer=_level(K, D, metric, callbacks, losses)), training=training).to(dev)
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


def _grads(z, loss, x, Ws, gz):
    grads = torch.autograd.grad((z, loss), [x] + list(Ws), (gz, torch.ones_like(loss)), allow_unused=True)
    return grads[0], list(grads[1:])


# ---- 1. L = 1 is VectorQuantizer ----------------------------------------------------------------------------------
@pytest.mark.parametrize('nchw', [False, True], ids=['tokens', 'nchw'])
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_depth_one_is_bit_identical_to_vector_quantizer(dev, dtype, metric, nchw):
    b, h, w, K, D = 4, 16, 16, 1024, 32
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, 1, seed=5)
    vq = vqb.build_quantizer(_level(K, D, metric)).to(dev)
    with torch.no_grad():
        vq.embedding.weight.copy_(Ws[0])
    rvq = _rvq(dev, 1, Ws, metric)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(6)).to(dev)
    res = []
    torch.use_deterministic_algorithms(True)      # gW through the segment sum: comparable bit for bit
    try:
        for q, W in ((vq, vq.embedding.weight), (rvq, rvq.quantizers[0].embedding.weight)):
            x = x_cpu.to(dtype).to(dev)
            if nchw:
                x = einops.rearrange(x, '(b h w) c -> b c h w', b=b, h=h, w=w).contiguous().requires_grad_(True)
                z, loss, memo = tokenizer.quantize(q, x, dict())
                memo = memo['quantizer']
                g = einops.rearrange(gz, '(b h w) c -> b c h w', b=b, h=h, w=w).contiguous()
            else:
                x.requires_grad_(True)
                z, loss, memo = q(x, dict())
                g = gz
            gx, (gW,) = _grads(z, loss, x, [W], g)
            res.append(dict(z=z.detach(), loss=loss.detach(), quant=memo['quant'].reshape(N, -1)[:, 0], gx=gx, gW=gW,
                            losses={k: v.detach() for k, v in memo['loss'].items()}))
    finally:
        torch.use_deterministic_algorithms(False)
    a, r = res
    for key in ('z', 'loss', 'quant', 'gx', 'gW'):
        assert a[key].dtype == r[key].dtype and torch.equal(a[key], r[key]), key
    assert a['losses'].keys() == r['losses'].keys() and all(torch.equal(a['losses'][k], r['losses'][k]) for k in a['losses'])


# ---- 2. depth 2..8 against the restatement --------------------------------------------------------------------------
def _compare_to_restatement(q, memo, z, loss, gx, gWs, ref, xo, N, bf16):
    """Indices with the near-tie policy (a row whose level-l index differs must be a near-tie at level l, its deeper
    levels are excluded), then z / loss / gx on the agreeing rows and gW_l on the codes no excluded row touched."""
    L = len(gWs)
    qg, qr = memo['quant'].cpu(), ref['quant']
    agree_before = torch.ones(N, dtype=torch.bool)
    for l in range(L):
        rows = (agree_before & (qg[:, l] != qr[:, l])).nonzero().flatten()
        d = ref['levels'][l]['distance'][0]
        gap = d[rows, qg[rows, l]] - d[rows, qr[rows, l]]
        assert (gap.abs() < 1e-5).all(), f'level {l}: index mismatch beyond a near-tie, gaps {gap.tolist()}'
        agree_before &= qg[:, l] == qr[:, l]
    ok = agree_before
    n_bad = int((~ok).sum())
    assert n_bad <= max(2, N // 200), f'{n_bad} rows excluded after near-ties'
    torch.testing.assert_close(z.detach().cpu()[ok], ref['z_ste'].detach()[ok], rtol=1e-5, atol=1e-6)
    # an excluded row moves the mean loss by at most a few times its own share
    torch.testing.assert_close(loss.detach().cpu(), ref['loss'].detach(), rtol=1e-5 + 8 * n_bad / N, atol=1e-7)
    if bf16:
        torch.testing.assert_close(gx.float().cpu()[ok], xo.grad[ok], rtol=2 ** -7, atol=1e-6)
    else:
        torch.testing.assert_close(gx.cpu()[ok], xo.grad[ok], rtol=1e-4, atol=1e-7)
    for l in range(L):
        want = ref['weight_leafs'][l].grad
        touched = torch.zeros(want.shape[0], dtype=torch.bool)
        touched[qg[~ok, l]] = True
        touched[qr[~ok, l]] = True
        scale = float(want.abs().max())
        torch.testing.assert_close(gWs[l].cpu()[~touched], want[~touched], rtol=1e-4, atol=1e-4 * scale)


_GRID = list(itertools.product([2, 4, 8], [8, 32, 256], [512, 8192]))


@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('L,D,K', _GRID, ids=[f'L{L}-D{D}-K{K}' for L, D, K in _GRID])
def test_matches_the_restatement(dev, L, D, K, metric, dtype):
    N = 1024
    x_cpu, Ws = _inputs(N, K, D, L, seed=L * 1000 + D + K)
    xt = x_cpu.to(dtype)
    q = _rvq(dev, L, Ws, metric)
    x = xt.to(dev).requires_grad_(True)
    z, loss, memo = q(x, dict())
    gz_cpu = torch.randn(N, D, generator=torch.Generator().manual_seed(9))
    gx, gWs = _grads(z, loss, x, [lv.embedding.weight for lv in q.quantizers], gz_cpu.to(dev))
    assert z.shape == (N, D) and memo['quant'].shape == (N, L) and len(memo['levels']) == L
    assert memo['levels'][0]['x'].data_ptr() == memo['x'].data_ptr() and memo['levels'][L - 1]['x'].dtype == torch.float32
    spec = O.QuantizerSpec(distance=metric, training=True, losses=SPEC_LOSSES)
    xo = xt.float().requires_grad_(True)
    ref = R.rvq_forward(spec, xo, Ws)
    (ref['loss'] + (ref['z_ste'] * gz_cpu).sum()).backward()
    _compare_to_restatement(q, memo, z, loss, gx, gWs, ref, xo, N, dtype == torch.bfloat16)
    for name in SPEC_LOSSES:
        torch.testing.assert_close(memo['loss'][name].detach().cpu(), ref['losses'][name].detach(), rtol=1e-3, atol=1e-7)


# ---- 3. CVQ-VAE on every level --------------------------------------------------------------------------------------
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
def test_cvqvae_levels_train_like_the_restatement(dev, metric):
    """Two training steps; both forwards run before the first backward, so each level's update of step 2 must leave
    the codebook that step 1's backward saved intact (copy-on-write per level)."""
    N, K, D, L = 2048, 512, 32, 3
    cb = [dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'), ema=dict())]
    x1, Ws = _inputs(N, K, D, L, seed=31)
    x2, _ = _inputs(N, K, D, L, seed=32)
    q = _rvq(dev, L, Ws, metric, callbacks=cb)
    spec = O.QuantizerSpec(distance=metric, callback='CVQVAECallback', training=True, losses=SPEC_LOSSES)
    probs = [torch.zeros(K) for _ in range(L)]
    xa = x1.to(dev).requires_grad_(True)
    za, la, ma = q(xa, dict())
    xo = x1.clone().requires_grad_(True)
    ref1 = R.rvq_forward(spec, xo, Ws, probs)
    W_after1 = [lv.embedding.weight.detach().clone() for lv in q.quantizers]
    p_after1 = [lv._probability.clone() for lv in q.quantizers]
    zb, lb, mb = q(x2.to(dev), dict())                         # step 2 updates every codebook in place
    ref2 = R.rvq_forward(spec, x2.clone(), ref1['weights'], ref1['probs'])
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(33))
    (gx,) = torch.autograd.grad((za, la), (xa,), (gz.to(dev), torch.ones_like(la)))
    (ref1['loss'] + (ref1['z_ste'] * gz).sum()).backward()
    for memo, ref, W_gpu, p_gpu in ((ma, ref1, W_after1, p_after1),
                                    (mb, ref2, [lv.embedding.weight.detach() for lv in q.quantizers],
                                     [lv._probability for lv in q.quantizers])):
        qg, qr = memo['quant'].cpu(), ref['quant']
        ok = (qg == qr).all(1)
        assert int((~ok).sum()) <= N // 200
        for l in range(L):
            touched = torch.zeros(K, dtype=torch.bool)
            touched[qg[~ok, l]] = True
            touched[qr[~ok, l]] = True
            torch.testing.assert_close(p_gpu[l].cpu()[~touched], ref['probs'][l][~touched], rtol=1e-5, atol=1e-7)
            # the anchors: nearest tokens by the column arg-min; a near-tie there picks another token for that code
            close = torch.isclose(W_gpu[l].cpu(), ref['weights'][l], rtol=1e-5, atol=1e-6).all(1)
            assert int((~close & ~touched).sum()) <= K // 100, f'level {l}: {int((~close).sum())} codebook rows differ'
    ok = (ma['quant'].cpu() == ref1['quant']).all(1)
    torch.testing.assert_close(gx.cpu()[ok], xo.grad[ok], rtol=1e-4, atol=1e-7)


# ---- 4. token round trip --------------------------------------------------------------------------------------------
@pytest.mark.parametrize('bhw', [(4, 8, 12), (3, 5, 7)], ids=lambda s: 'x'.join(map(str, s)))
@pytest.mark.parametrize('K', [512, 70000])
def test_encode_to_quant_then_decode_from_quant_reproduces_zhat(dev, K, bhw):
    (b, h, w), D, L = bhw, 32, 4
    x_cpu, Ws = _inputs(b * h * w, K, D, L, seed=41)
    q = _rvq(dev, L, Ws, 'L2', training=False)
    x = einops.rearrange(x_cpu, '(b h w) c -> b c h w', b=b, h=h, w=w).contiguous().to(dev)
    with torch.no_grad():
        ids, memo = tokenizer.encode_to_quant(q, x, dict(), compact=True)
        wide, _ = tokenizer.encode_to_quant(q, x, dict())
        z, _, fmemo = tokenizer.quantize(q, x, dict())
    assert ids.shape == (b, h, w, L) and ids.dtype == (torch.uint16 if K <= 65536 else torch.int32)
    assert wide.dtype == torch.int64 and torch.equal(ids.cpu().to(torch.int32).long(), wide.cpu())
    assert torch.equal(fmemo['quantizer']['quant'].cpu(), wide.cpu().view(-1, L))
    zhat = R.level_sum(Ws, wide.cpu())                                        # [b, h, w, D], level-ordered fp32 sum
    want = einops.rearrange(zhat, 'b h w c -> b c h w').contiguous()
    for ids_dev in (ids, wide, wide.to(torch.int32)):
        for dtype in DTYPES:
            out, dmemo = tokenizer.decode_from_quant(q, ids_dev, dict(), dtype=dtype)
            assert out.shape == (b, D, h, w) and out.dtype == dtype and out.is_contiguous()
            assert torch.equal(out.cpu(), want.to(dtype))
    zt, _ = q.decode(wide.view(-1, L), dict())
    assert torch.equal(zt.cpu(), zhat.view(-1, D))
    # the forward's z is x + (zhat - x) on that same zhat
    torch.testing.assert_close(z.cpu(), want, rtol=1e-5, atol=1e-6)
    assert torch.equal(z.cpu(), x.cpu() + (want - x.cpu()))


def test_bad_ids_at_any_level(dev):
    b, h, w, K, D, L = 2, 4, 4, 512, 16, 3
    _, Ws = _inputs(8, K, D, L, seed=51)
    q = _rvq(dev, L, Ws, 'L2', training=False)
    ids = torch.randint(0, K, (b, h, w, L), generator=torch.Generator().manual_seed(52))
    bad = ids.clone()
    bad[0, 1, 2, 0] = K
    bad[1, 3, 0, L - 1] = K + 9
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
        assert torch.equal(rows[~mask], R.level_sum(Ws, ids)[~mask])
    with pytest.raises(ValueError, match=r'\[b, h, w, 3\]'):
        tokenizer.decode_from_quant(q, ids[..., 0].to(dev), dict())


# ---- 5. deterministic gradient --------------------------------------------------------------------------------------
def test_deterministic_codebook_gradients(dev):
    N, K, D, L = 16384, 512, 32, 4
    x_cpu, Ws = _inputs(N, K, D, L, seed=61)
    q = _rvq(dev, L, Ws, 'L2')
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(62)).to(dev)
    params = [lv.embedding.weight for lv in q.quantizers]

    def run():
        x = x_cpu.to(dev).requires_grad_(True)
        z, loss, _ = q(x, dict())
        return _grads(z, loss, x, params, gz)

    torch.use_deterministic_algorithms(True)
    try:
        runs = [run() for _ in range(3)]
    finally:
        torch.use_deterministic_algorithms(False)
    atomic = run()
    for gx, gWs in runs[1:]:
        assert torch.equal(gx, runs[0][0]) and all(torch.equal(a, b) for a, b in zip(gWs, runs[0][1]))
    assert torch.equal(atomic[0], runs[0][0])
    for a, b in zip(atomic[1], runs[0][1]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-4 * float(b.abs().max()))


# ---- 6. CUDA graph ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('deterministic', [False, True], ids=['atomic', 'deterministic'])
def test_training_step_cuda_graph_matches_eager(dev, deterministic):
    N, K, D, L = 8192, 1024, 32, 4
    x_cpu, Ws = _inputs(N, K, D, L, seed=71)
    q = _rvq(dev, L, Ws, 'Cosine')
    params = [lv.embedding.weight for lv in q.quantizers]
    x = x_cpu.to(torch.bfloat16).to(dev).requires_grad_(True)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(72)).to(dev)
    res = {}

    def step():
        z, loss, memo = q(x, dict())
        gx, gWs = _grads(z, loss, x, params, gz)
        res.update(z=z.detach(), loss=loss.detach(), quant=memo['quant'], gx=gx,
                   **{f'gW{l}': g for l, g in enumerate(gWs)})

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
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step()
        for _ in range(2):
            replay = run(g.replay)
            for k in eager:
                if k.startswith('gW') and not deterministic:
                    torch.testing.assert_close(replay[k], eager[k], rtol=1e-5, atol=1e-6 * float(eager[k].abs().max()))
                else:
                    assert torch.equal(eager[k], replay[k]), k
        del g
    finally:
        torch.use_deterministic_algorithms(False)


# ---- 7. launch count -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('L', [1, 4, 8])
def test_one_step_launch_per_level_and_one_backward_launch(dev, L):
    N, K, D = 4096, 512, 32
    x_cpu, Ws = _inputs(N, K, D, L, seed=81)
    q = _rvq(dev, L, Ws, 'L2')
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
