"""Quantizer dropout and depth-truncated codes of ResidualVectorQuantizer on the B200: the _depth kernels at full depth
against today's path (bit for bit), random per-token and per-image depths against the restatement
(oracle/rvq_dropout.py) on the kernel's own indices and codebooks, the invariant that the encodes do not see the
depths, the depth draw (seeding, the truncated share, uniformity, no synchronisation), CUDA-graph replay, the launch
count, and the truncated encode / decode."""
import einops
import pytest
import torch

import vector_quantization_b200 as vqb
from oracle import oracle as O
from oracle import rvq
from oracle import rvq_dropout as RD
from vector_quantization_b200 import ops, tokenizer

pytestmark = pytest.mark.gpu
DTYPES = [torch.float32, torch.bfloat16]
DT_IDS = ['fp32', 'bf16']
METRIC = {'L2': 'L2Distance', 'Cosine': 'CosineDistance'}
CVQ = [dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'), ema=dict())]


def _level(K, D, metric='L2', norm=False, callbacks=()):
    losses = dict(vqgan_loss=dict(type='VQGANLoss'))
    if norm:
        losses['commit_norm'] = dict(type='CommitmentLoss', mse=dict(norm=True))
    return dict(type='VQGANQuantizer', distance=dict(type=METRIC[metric]), callbacks=list(callbacks), losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D))


def _spec(node):
    return O.QuantizerSpec(training=False, losses={name: dict(type=c['type'], norm=c.get('mse', {}).get('norm', False))
                                                   for name, c in node['losses'].items()})


def _rvq(dev, Ws, metric='L2', norm=False, callbacks=(), p=0.0, rotation=False, training=True):
    K, D = Ws[0].shape
    q = vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=len(Ws), quantizer_dropout=p,
                                 rotation_trick=rotation, quantizer=_level(K, D, metric, norm, callbacks)),
                            training=training).to(dev)
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
    """forward + backward (upstream: gz on z, 1 on the loss); z / gx come back token-major, quant as [N, L], depth per
    token (None without dropout)."""
    params = [lv.embedding.weight for lv in q.quantizers]
    N = x_cpu.shape[0]
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
    depth = memo.get('depth')
    if depth is not None:
        depth = depth.repeat_interleave(N // depth.numel()).cpu()
    return dict(z=z.detach(), loss=loss.detach(), losses={k: v.detach() for k, v in memo['loss'].items()},
                quant=memo['quant'].reshape(N, -1).clone(), gx=gx, gWs=list(grads[1:]), depth=depth,
                Ws=[p.detach().clone() for p in params], probs=[lv._probability.clone() for lv in q.quantizers
                                                                if hasattr(lv, '_probability')])


def _pin_depths(monkeypatch, depth_of):
    """Replace the draw with depth_of(samples) (a CPU int tensor), so that a step runs the dropout path on known depths."""
    monkeypatch.setattr(vqb.ResidualVectorQuantizer, 'draw_depths',
                        lambda self, samples, device: depth_of(samples).to(torch.int32).to(device))


def _launches(monkeypatch):
    names = []
    call = ops._call
    monkeypatch.setattr(ops, '_call', lambda name, *a: (names.append(name), call(name, *a))[1])
    return names


# ---- 1. full depth through the _depth kernels is today's step bit for bit --------------------------------------------
@pytest.mark.parametrize('rotation', [False, True], ids=['ste', 'rot'])
@pytest.mark.parametrize('nchw', [False, True], ids=['tokens', 'nchw'])
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
def test_full_depth_is_bit_identical_to_the_step_without_dropout(dev, monkeypatch, dtype, metric, nchw, rotation):
    b, h, w, K, D, L = 4, 16, 16, 512, 32, 3
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=11)
    x_cpu = x_cpu.to(dtype)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(12))
    _pin_depths(monkeypatch, lambda S: torch.full((S,), L))
    names = _launches(monkeypatch)
    res = []
    torch.use_deterministic_algorithms(True)       # gW through the segment sum: comparable bit for bit
    try:
        for p in (0.0, 0.5):
            q = _rvq(dev, Ws, metric, norm=True, callbacks=CVQ, p=p, rotation=rotation)
            res.append(_step(q, x_cpu, gz, dev, hw=(b, h, w) if nchw else None))
    finally:
        torch.use_deterministic_algorithms(False)
    plain, dropped = res
    assert plain['depth'] is None and (dropped['depth'] == L).all()
    assert 'vqb_residual_step_depth' in names and any(n.startswith('vqb_residual_backward_depth') for n in names)
    for key in ('z', 'loss', 'quant', 'gx'):
        assert plain[key].dtype == dropped[key].dtype and torch.equal(plain[key], dropped[key]), key
    assert all(torch.equal(plain['losses'][k], dropped['losses'][k]) for k in plain['losses'])
    for key in ('gWs', 'Ws', 'probs'):
        assert all(torch.equal(a, c) for a, c in zip(plain[key], dropped[key])), key


# ---- 2. random depths against the restatement -------------------------------------------------------------------------
def _restatement(monkeypatch, node, x, out, depth, rotation, dtype=torch.float32):
    """oracle/rvq_dropout.py on the kernel's own indices (its assignment is replaced by out['quant']) and codebooks, in
    `dtype` -> (restatement output, its x leaf with the gradient of (z * gz).sum() + loss still to be formed)."""
    cols = iter(range(out['quant'].shape[1]))
    quant = out['quant'].cpu()
    xo = x.detach().to(dtype).clone().requires_grad_(True)
    with monkeypatch.context() as m:
        m.setattr(O, 'encode', lambda kind, xx, W: (quant[:, next(cols)], None))
        ref = RD.rvq_dropout_forward(_spec(node), xo, [W.cpu().to(dtype) for W in out['Ws']], depth, rotation=rotation)
    return ref, xo


def _rel_close(got, want, rtol):
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    torch.testing.assert_close(got, want, rtol=rtol, atol=rtol * max(float(want.abs().max()), 1e-30))


_CASES = [(2, 8, False, 'L2', False), (4, 32, True, 'Cosine', True), (8, 64, False, 'L2', True),
          (16, 256, True, 'L2', False), (3, 20, True, 'Cosine', False), (16, 128, False, 'Cosine', True)]


@pytest.mark.parametrize('per_image', [False, True], ids=['per-token', 'per-image'])
@pytest.mark.parametrize('dtype', DTYPES, ids=DT_IDS)
@pytest.mark.parametrize('L,D,norm,metric,rotation', _CASES, ids=[f'L{c[0]}-D{c[1]}-{"norm" if c[2] else "plain"}-'
                                                                  f'{c[3]}-{"rot" if c[4] else "ste"}' for c in _CASES])
def test_random_depths_match_the_restatement(dev, monkeypatch, L, D, norm, metric, rotation, dtype, per_image):
    b, h, w, K = 8, 16, 16, 512
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=L * 100 + D)
    x_cpu = x_cpu.to(dtype)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(D))
    node = _level(K, D, metric, norm)
    q = _rvq(dev, Ws, metric, norm, p=0.75, rotation=rotation)
    torch.manual_seed(L + D)
    out = _step(q, x_cpu, gz, dev, hw=(b, h, w) if per_image else None)
    depth = out['depth']
    assert depth is not None and depth.min() >= 1 and depth.max() <= L
    sample_depth = depth.view(b, h * w)[:, 0] if per_image else depth
    assert (sample_depth[int(sample_depth.numel() * 0.75):] == L).all()
    xf = x_cpu.float()
    ref, xo = _restatement(monkeypatch, node, xf, out, depth, rotation=False)
    ((ref['z_ste'] * gz).sum() + ref['loss']).backward()
    _rel_close(out['z'], ref['z_ste'], 1e-5)
    _rel_close(out['loss'], ref['loss'], 1e-5)
    for name, value in ref['losses'].items():
        _rel_close(out['losses'][name], value, 1e-5)
    for l in range(L):
        _rel_close(out['gWs'][l], ref['weight_leafs'][l].grad, 1e-4)
    if rotation:          # the rotated gx against the float64 restatement
        ref64, x64 = _restatement(monkeypatch, node, xf, out, depth, rotation=True, dtype=torch.float64)
        ((ref64['z_ste'] * gz.double()).sum() + ref64['loss']).backward()
        want = x64.grad
    else:
        want = xo.grad
    if dtype == torch.bfloat16:
        torch.testing.assert_close(out['gx'].float().cpu().double(), want.double(), rtol=2 ** -7,
                                   atol=1e-4 * float(want.abs().max()))
    else:
        _rel_close(out['gx'], want, 1e-4)


# ---- 3. the encodes do not see the depths -----------------------------------------------------------------------------
@pytest.mark.parametrize('nchw', [False, True], ids=['tokens', 'nchw'])
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
def test_indices_codebooks_and_statistics_are_those_of_the_step_without_dropout(dev, metric, nchw):
    b, h, w, K, D, L = 8, 16, 16, 512, 32, 4
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=41)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(42))
    res = []
    for p in (0.0, 0.5):
        q = _rvq(dev, Ws, metric, norm=True, callbacks=CVQ, p=p)
        torch.manual_seed(43)
        first = _step(q, x_cpu, gz, dev, hw=(b, h, w) if nchw else None)
        second = _step(q, x_cpu.flip(0), gz, dev, hw=(b, h, w) if nchw else None)   # from the state the first left
        res.append((first, second))
    for plain, dropped in zip(*res):
        assert dropped['depth'] is not None and (dropped['depth'] < L).any()
        assert torch.equal(plain['quant'], dropped['quant'])
        for key in ('Ws', 'probs'):
            assert len(plain[key]) == L and all(torch.equal(a, c) for a, c in zip(plain[key], dropped[key])), key
        assert not torch.equal(plain['z'], dropped['z']) and not torch.equal(plain['gx'], dropped['gx'])


# ---- 4. the draw ------------------------------------------------------------------------------------------------------
def test_same_seed_same_depths_and_the_truncated_share(dev):
    _, Ws = _inputs(64, 64, 8, 6, seed=51)
    q = _rvq(dev, Ws, p=0.3)
    x = torch.randn(1000, 8, device=dev)
    depths = []
    for seed in (5, 5, 6):
        torch.manual_seed(seed)
        depths.append(q(x, dict())[2]['depth'].clone())
    assert depths[0].dtype == torch.int32 and depths[0].shape == (1000,) and depths[0].device == x.device
    assert torch.equal(depths[0], depths[1]) and not torch.equal(depths[0], depths[2])
    d = depths[0].cpu()
    assert (d[300:] == 6).all() and d[:300].min() >= 1 and d[:300].max() <= 6 and (d[:300] < 6).any()


def test_depths_are_uniform_over_the_levels(dev):
    from scipy import stats
    L = 7
    _, Ws = _inputs(64, 64, 8, L, seed=52)
    q = _rvq(dev, Ws, p=1.0)
    torch.manual_seed(53)
    d = q.draw_depths(1 << 20, dev).cpu()
    counts = torch.bincount(d.long(), minlength=L + 1)
    assert counts[0] == 0 and counts.sum() == 1 << 20
    assert stats.chisquare(counts[1:].double().numpy()).pvalue > 1e-3


def test_the_draw_does_not_synchronise(dev):
    _, Ws = _inputs(64, 64, 8, 4, seed=54)
    q = _rvq(dev, Ws, p=0.5)
    torch.cuda.set_sync_debug_mode('error')
    try:
        d = q.draw_depths(4096, dev)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert d.is_cuda and d.shape == (4096,)


def _kernels(q, x, dev):
    q(x, dict())                       # warm-up
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        z, loss, memo = q(x, dict())
        torch.autograd.grad((z, loss), [x], (torch.ones_like(z), torch.ones_like(loss)))
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA], memo


@pytest.mark.parametrize('L', [2, 8])
def test_eval_and_zero_p_never_truncate_and_launch_what_the_step_without_dropout_launches(dev, L):
    N, K, D = 4096, 512, 32
    x_cpu, Ws = _inputs(N, K, D, L, seed=61)
    x = x_cpu.to(dev).requires_grad_(True)
    base, _ = _kernels(_rvq(dev, Ws), x, dev)
    for p, training in ((0.0, True), (0.5, False), (1.0, False)):
        names, memo = _kernels(_rvq(dev, Ws, p=p, training=training), x, dev)
        assert 'depth' not in memo and sorted(names) == sorted(base), (p, training)


@pytest.mark.parametrize('L', [1, 4, 8])
def test_dropout_adds_only_the_draw_launches(dev, L):
    N, K, D = 4096, 512, 32
    x_cpu, Ws = _inputs(N, K, D, L, seed=62)
    x = x_cpu.to(dev).requires_grad_(True)
    base, _ = _kernels(_rvq(dev, Ws), x, dev)
    names, memo = _kernels(_rvq(dev, Ws, p=0.5), x, dev)
    assert memo['depth'].shape == (N,)
    assert sum('residual_step_kernel' in n for n in names) == L
    assert sum('residual_backward_kernel' in n for n in names) == 1
    assert 0 < len(names) - len(base) <= 3


# ---- 5. CUDA graph ----------------------------------------------------------------------------------------------------
def test_graph_replays_draw_fresh_depths_and_each_matches_the_restatement(dev, monkeypatch):
    b, h, w, K, D, L = 8, 16, 16, 512, 32, 4
    N = b * h * w
    x_cpu, Ws = _inputs(N, K, D, L, seed=71)
    node = _level(K, D, norm=True)
    q = _rvq(dev, Ws, norm=True, p=1.0)
    params = [lv.embedding.weight for lv in q.quantizers]
    x = _nchw(x_cpu, b, h, w).to(dev).requires_grad_(True)
    gz_cpu = torch.randn(N, D, generator=torch.Generator().manual_seed(72))
    gz = _nchw(gz_cpu, b, h, w).to(dev)
    res = {}

    def step():
        z, loss, memo = tokenizer.quantize(q, x, dict())
        grads = torch.autograd.grad((z, loss), [x] + params, (gz, torch.ones_like(loss)))
        res.update(z=z.detach(), loss=loss.detach(), gx=grads[0], gWs=list(grads[1:]), depth=memo['quantizer']['depth'],
                   quant=memo['quantizer']['quant'])

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    seen = []
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        depth = res['depth'].cpu().repeat_interleave(h * w)
        seen.append(depth)
        out = dict(quant=res['quant'].reshape(N, L), Ws=[p.detach() for p in params])
        ref, xo = _restatement(monkeypatch, node, x_cpu, out, depth, rotation=False)
        ((ref['z_ste'] * gz_cpu).sum() + ref['loss']).backward()
        _rel_close(_tokens(res['z'], b, h, w), ref['z_ste'], 1e-5)
        _rel_close(res['loss'], ref['loss'], 1e-5)
        _rel_close(_tokens(res['gx'], b, h, w), xo.grad, 1e-4)
        for l in range(L):
            _rel_close(res['gWs'][l], ref['weight_leafs'][l].grad, 1e-4)
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])
    del graph


@pytest.mark.parametrize('rotate', [False, True])
def test_deterministic_gw_is_bit_identical_between_eager_and_replay(dev, rotate):
    N, K, D, L = 8192, 512, 32, 4
    x_cpu, Ws = _inputs(N, K, D, L, seed=81)
    x = x_cpu.to(dev)
    Wd = [W.to(dev) for W in Ws]
    g = torch.Generator().manual_seed(82)
    quant = torch.randint(0, K, (N, L), generator=g).to(dev)
    depth = torch.randint(1, L + 1, (N // 64,), generator=g, dtype=torch.int32).to(dev)
    gz = torch.randn(N, D, generator=g).to(dev)
    g4s = [[torch.tensor(1.0 + l, device=dev), torch.tensor(0.25, device=dev), None, None] for l in range(L)]
    res = {}

    def step():
        res['gx'], res['gWs'] = ops.residual_backward(gz, x, Wd, quant, g4s, want_norm=False, need_gW=[True] * L,
                                                      deterministic=True, rotate=rotate, depth=depth, depth_hw=64)

    step()
    torch.cuda.synchronize()
    eager = dict(gx=res['gx'].clone(), gWs=[t.clone() for t in res['gWs']])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(eager['gx'], res['gx'])
        assert all(torch.equal(a, c) for a, c in zip(eager['gWs'], res['gWs']))
    tok = depth.repeat_interleave(64).cpu()
    for l in range(L):      # codes used only by inactive tokens get no gradient
        used = torch.zeros(K, dtype=torch.bool)
        used[quant[:, l].cpu()[tok > l]] = True
        assert not eager['gWs'][l].cpu()[~used].any()
    del graph


# ---- 6. truncated codes -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('compact', [False, True], ids=['int64', 'compact'])
@pytest.mark.parametrize('metric', ['L2', 'Cosine'])
@pytest.mark.parametrize('L,n', [(4, 2), (8, 1), (8, 5), (3, 3)])
def test_truncated_codes_are_those_of_the_first_n_levels(dev, monkeypatch, L, n, metric, compact):
    b, h, w, K, D = 4, 16, 16, 1024, 32
    x_cpu, Ws = _inputs(b * h * w, K, D, L, seed=91 + L + n)
    x = _nchw(x_cpu, b, h, w).to(dev)
    full = _rvq(dev, Ws, metric, training=False)
    head = _rvq(dev, Ws[:n], metric, training=False)
    names = _launches(monkeypatch)
    ids, memo = tokenizer.encode_to_quant(full, x, dict(), compact=compact, num_quantizers=n)
    truncated = list(names)
    names.clear()
    want, _ = tokenizer.encode_to_quant(head, x, dict(), compact=compact)
    assert ids.shape == (b, h, w, n) and ids.dtype == want.dtype and torch.equal(ids, want)
    assert len(memo['quantizer']['levels']) == n
    assert truncated == names              # the launches of the n-level quantizer: the levels past n never run
    z, _ = tokenizer.decode_from_quant(full, ids, dict(), num_quantizers=n)
    ref = rvq.level_sum([W.to(dev) for W in Ws[:n]], ids.long())
    assert torch.equal(z, einops.rearrange(ref, 'b h w c -> b c h w').contiguous())
    zb, _ = tokenizer.decode_from_quant(full, ids, dict(), num_quantizers=n, dtype=torch.bfloat16)
    assert torch.equal(zb, z.to(torch.bfloat16))


def test_truncated_encode_runs_no_callback_past_n(dev):
    K, D, L, n = 256, 16, 4, 2
    x_cpu, Ws = _inputs(2048, K, D, L, seed=99)
    q = _rvq(dev, Ws, callbacks=CVQ)
    before = [lv.embedding.weight.detach().clone() for lv in q.quantizers]
    _, quant, memo = q.encode(x_cpu.to(dev), dict(), num_quantizers=n)
    assert quant.shape == (2048, n) and len(memo['levels']) == n
    for l, lv in enumerate(q.quantizers):
        changed = not torch.equal(before[l], lv.embedding.weight)
        assert changed == (l < n), l
