"""The deterministic reductions selected by torch.use_deterministic_algorithms(True): the stable code sort, the
chunked segment sum against a CPU restatement of its association contract, batch independence of that association,
agreement with the atomic path, and bitwise run-to-run equality of every quantizer configuration whose codebook
statistics or gradient go through them (eager, NCHW, k-means init, CUDA graph, two GPUs)."""
import os
import random
import socket
import time

import numpy as np
import pytest
import torch

import vector_quantization_b200 as vqb
from vector_quantization_b200 import ops
from tests import test_gpu_modules as M

pytestmark = pytest.mark.gpu
NO_KEY = -1          # kNoKey (all ones) in the int64 storage of the packed keys
KEY_OFFSET = 1000


@pytest.fixture
def deterministic():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _codes(N, K, dist, seed):
    rng = np.random.default_rng(seed)
    if dist == 'uniform':
        return rng.integers(0, K, N)
    if dist == 'hot':
        return np.full(N, K // 2 if K > 1 else 0, dtype=np.int64)
    return (rng.zipf(1.3, N) - 1) % K


def _expected_sort(codes, K):
    valid = (codes >= 0) & (codes < K)
    order = np.argsort(np.where(valid, codes, K), kind='stable')
    offsets = np.concatenate([[0], np.cumsum(np.bincount(codes[valid], minlength=K))])
    return order, offsets


def _restate(rows, codes, K, C):
    """The association contract on the CPU in float32: each chunk of C tokens of a code summed serially in ascending
    token order from +0, the chunk sums added serially in chunk order from +0 (np.cumsum's sequential order, written
    as one vectorised addition per step so that every chunk / code advances together)."""
    N, D = rows.shape
    order, off = _expected_sort(codes, K)
    cnt = np.diff(off)
    nch = (cnt + C - 1) // C
    first = np.cumsum(nch) - nch
    ch_code = np.repeat(np.arange(K), nch)
    ch_start = off[ch_code] + (np.arange(nch.sum()) - first[ch_code]) * C
    ch_len = np.minimum(C, off[ch_code + 1] - ch_start)
    part = np.zeros((len(ch_code), D), np.float32)
    for i in range(int(ch_len.max(initial=0))):
        m = ch_len > i
        part[m] = part[m] + rows[order[ch_start[m] + i]]
    tot = np.zeros((K, D), np.float32)
    for j in range(int(nch.max(initial=0))):
        m = nch > j
        tot[m] = tot[m] + part[first[m] + j]
    return np.float32(0) + tot, cnt.astype(np.float32)


# ---- 1. sort ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('N', [1, 1000, 65536, 262147])
@pytest.mark.parametrize('K', [1, 64, 8192, 262144])
@pytest.mark.parametrize('dist', ['uniform', 'hot', 'zipf'])
@pytest.mark.parametrize('packed', [False, True], ids=['quant', 'keys'])
def test_code_sort_matches_stable_argsort(dev, N, K, dist, packed):
    rng = np.random.default_rng(N * 7 + K)
    codes = _codes(N, K, dist, seed=N + K)
    bad = rng.random(N) < 0.01                       # out-of-range codes: below 0 and at / above K
    codes = np.where(bad, np.where(rng.random(N) < 0.5, -3, K + 7), codes)
    if packed:
        nokey = (rng.random(N) < 0.01) & ~bad        # no finite score: resolves to code 0
        score = rng.integers(0, 1 << 31, N, dtype=np.int64)
        keys = np.where(nokey, NO_KEY, (score << 32) | (codes + KEY_OFFSET))
        codes = np.where(nokey, 0, codes)
        order, offsets = ops.code_sort(K, keys=torch.from_numpy(keys).to(dev), key_offset=KEY_OFFSET)
    else:
        order, offsets = ops.code_sort(K, quant=torch.from_numpy(codes).to(dev))
    want_order, want_off = _expected_sort(codes, K)
    assert order.dtype == torch.int32 and offsets.dtype == torch.int32 and offsets.numel() == K + 1
    np.testing.assert_array_equal(offsets.cpu().numpy(), want_off)
    np.testing.assert_array_equal(order.cpu().numpy(), want_order)


# ---- 2. segment sum, bitwise against the contract ------------------------------------------------------------------
@pytest.mark.parametrize('D', [5, 8, 32, 256, 768])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=['fp32', 'bf16'])
@pytest.mark.parametrize('dist', ['uniform', 'hot', 'zipf'])
def test_segment_sum_matches_contract_bitwise(dev, D, dtype, dist):
    N, K = (20000, 512) if D >= 256 else (70000, 4096)
    codes = _codes(N, K, dist, seed=D)
    codes[::97] = K + 1                               # skipped tokens
    g = torch.Generator().manual_seed(D)
    rows = torch.randn(N, D, generator=g).to(dtype)
    order, offsets = ops.code_sort(K, quant=torch.from_numpy(codes).to(dev))
    counts = torch.zeros(K, dtype=torch.float32, device=dev)
    sums = ops.segment_sum_rows(rows.to(dev), order, offsets, out_counts=counts)
    want, want_cnt = _restate(rows.float().numpy(), codes, K, ops.segment_chunk())
    np.testing.assert_array_equal(counts.cpu().numpy(), want_cnt)
    np.testing.assert_array_equal(sums.cpu().numpy(), want)


def test_segment_chunk_is_256():
    assert ops.segment_chunk() == 256


# ---- 3. the association does not depend on the rest of the batch ---------------------------------------------------
def test_stats_independent_of_other_tokens(dev):
    K, D, n = 1024, 32, 5000
    g = torch.Generator().manual_seed(3)
    x = torch.randn(n, D, generator=g)
    q = torch.randint(0, K // 2, (n,), generator=g)
    q[: n // 3] = 7                                   # a hot code spanning several chunks
    extra_x = torch.randn(200000, D, generator=g)
    extra_q = torch.randint(K // 2, K, (200000,), generator=g)
    alone = ops.scatter_stats(x.to(dev), q.to(dev), K, normalize_x=True, deterministic=True)
    mixed = ops.scatter_stats(torch.cat([x, extra_x]).to(dev), torch.cat([q, extra_q]).to(dev), K, normalize_x=True,
                              deterministic=True)
    lo = slice(0, K // 2 * D)
    assert torch.equal(alone[lo], mixed[lo])
    assert torch.equal(alone[K * D:K * D + K // 2], mixed[K * D:K * D + K // 2])


def test_codebook_gradient_independent_of_other_tokens(dev):
    K, D, N = 1024, 64, 8192
    g = torch.Generator().manual_seed(4)
    W = torch.randn(K, D, generator=g).to(dev)
    g4 = torch.tensor([1.0, 0.25, 0.5, 0.125], device=dev)
    mine = torch.rand(N, generator=g) < 0.5          # X's positions
    xa, xb = torch.randn(N, D, generator=g), torch.randn(N, D, generator=g)
    qa = torch.where(mine, torch.randint(0, K // 2, (N,), generator=g), torch.randint(K // 2, K, (N,), generator=g))
    qb = torch.where(mine, qa, torch.randint(K // 2, K, (N,), generator=g))
    xb[mine] = xa[mine]
    gz = torch.randn(N, D, generator=g)
    outs = []
    for x, q in ((xa, qa), (xb, qb)):
        _, gW = ops.quantize_backward(gz.to(dev), x.to(dev), W, q.to(dev), g4, normalize_x=True, want_norm=True,
                                      need_gW=True, deterministic=True)
        outs.append(gW[:K // 2])
    assert torch.equal(outs[0], outs[1])


# ---- 4. against the atomic path -----------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=['fp32', 'bf16'])
@pytest.mark.parametrize('hot', [False, True], ids=['spread', 'hot'])
def test_against_atomic_path(dev, dtype, hot):
    N, K, D = 65536, 8192, 32
    g = torch.Generator().manual_seed(5)
    x = torch.randn(N, D, generator=g).to(dtype).to(dev)
    q = (torch.zeros(N, dtype=torch.int64) if hot else torch.randint(0, K, (N,), generator=g)).to(dev)
    det = ops.scatter_stats(x, q, K, normalize_x=True, deterministic=True)
    ref = ops.scatter_stats(x, q, K, normalize_x=True, deterministic=False)
    # rel 1e-5 of the largest sum: 65 536 normalised rows on one code cancel, so single elements of the hot code are
    # far smaller than the terms that formed them and an element-wise relative bar would measure that cancellation
    torch.testing.assert_close(det, ref, rtol=1e-5, atol=1e-5 * float(ref[:K * D].abs().max()))
    W = torch.randn(K, D, generator=g).to(dev)
    gz = torch.randn(N, D, generator=g).to(dev)
    g4 = torch.tensor([1.0, 0.25, 0.5, 0.125], device=dev)
    gx_d, gW_d = ops.quantize_backward(gz, x, W, q, g4, normalize_x=True, want_norm=True, need_gW=True, deterministic=True)
    gx_a, gW_a = ops.quantize_backward(gz, x, W, q, g4, normalize_x=True, want_norm=True, need_gW=True, deterministic=False)
    assert torch.equal(gx_d, gx_a)
    torch.testing.assert_close(gW_d, gW_a, rtol=1e-4, atol=1e-6)


def test_flag_selects_the_path(dev):
    """None follows torch's flag, read at call time; the flag-off result is the atomic path's own."""
    N, K, D = 4096, 256, 16
    g = torch.Generator().manual_seed(6)
    x, q = torch.randn(N, D, generator=g).to(dev), torch.randint(0, K, (N,), generator=g).to(dev)
    det = ops.scatter_stats(x, q, K, deterministic=True)
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        on = ops.scatter_stats(x, q, K)
    finally:
        torch.use_deterministic_algorithms(prev)
    assert torch.equal(on, det)


# ---- 5. modules ---------------------------------------------------------------------------------------------------
GRAD_CASES = ['vqgan_l2', 'llamagen_l2norm', 'vqkd_train', 'cvqvae_train', 'llamagen_cvq_train', 'cluster_train']


def _module_steps(rec, dev, dtype):
    q = M._build(rec, dev)
    outs = []
    for step in rec['steps']:
        with torch.no_grad():
            q.embedding.weight.copy_(step['W_before'])
            if step['prob_before'] is not None:
                q.get_buffer('_probability').copy_(step['prob_before'])
        x = step['x'].to(dtype).to(dev).requires_grad_(True)
        q.embedding.weight.grad = None
        z, loss, memo = q(x, dict())
        (loss + (z * step['gz'].to(dev)).sum()).backward()
        W_grad = q.embedding.weight.grad
        outs.append([z.detach(), loss.detach(), x.grad, None if W_grad is None else W_grad.clone(),
                     q.embedding.weight.detach().clone(),
                     q.get_buffer('_probability').clone() if step['prob_before'] is not None else None])
    return outs


def _assert_bitwise(a, b):
    for sa, sb in zip(a, b):
        for ta, tb in zip(sa, sb):
            assert (ta is None) == (tb is None)
            if ta is not None:
                assert torch.equal(ta, tb)


@pytest.mark.parametrize('name', GRAD_CASES)
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=['fp32', 'bf16'])
def test_module_steps_bitwise_reproducible(dev, deterministic, name, dtype):
    rec = M._load(name)
    _assert_bitwise(_module_steps(rec, dev, dtype), _module_steps(rec, dev, dtype))
    M.test_module_vs_reference_golden(dev, name, dtype)     # still within the golden tolerances


@pytest.mark.parametrize('name', ['vqgan_l2', 'vqkd_train'])
def test_nchw_tokenizer_bitwise_reproducible(dev, deterministic, name):
    from vector_quantization_b200 import tokenizer
    rec = M._load(name)
    step = rec['steps'][0]
    D = step['x'].shape[1]
    x_nchw = step['x'].view(-1, 16, 16, D).permute(0, 3, 1, 2).contiguous()
    runs = []
    for _ in range(2):
        q = M._build(rec, dev)
        with torch.no_grad():
            q.embedding.weight.copy_(step['W_before'])
        x = x_nchw.to(dev).requires_grad_(True)
        z, loss, memo = tokenizer.quantize(q, x, dict())
        (loss + (z * z.detach()).sum()).backward()
        W_grad = q.embedding.weight.grad
        runs.append([[z.detach(), loss.detach(), x.grad, W_grad, q.embedding.weight.detach().clone()]])
    _assert_bitwise(*runs)


def test_kmeans_lazy_init_bitwise_reproducible(dev, deterministic):
    rec = M._load('vqkd_train')
    x = torch.cat([s['x'] for s in rec['steps']]).to(dev)
    runs = []
    for _ in range(2):
        torch.manual_seed(0)
        random.seed(0)
        q = vqb.build_quantizer(rec['config'], training=True).to(dev)
        with torch.no_grad():
            q.embedding.weight.normal_()
        z, loss, memo = q(x, dict())
        runs.append([[q.embedding.weight.detach().clone(), z.detach(), loss.detach()]])
    _assert_bitwise(*runs)


# ---- 6. CUDA graph ------------------------------------------------------------------------------------------------
def test_vqkd_step_cuda_graph_matches_eager(dev, deterministic):
    from oracle import oracle as O
    N, K, D = 65536, 8192, 32
    cfg = dict(type='VQKDQuantizer', distance=dict(type='CosineDistance'), callbacks=[dict(type='VQKDCallback', ema=dict())],
               losses=dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True))),
               embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D))
    x_cpu, E = O.synthetic_latents(N, K, D, seed=11, normalized_codebook=True)
    q = vqb.build_quantizer(cfg, training=True).to(dev)
    q._forward_pre_hooks.clear()
    q.requires_grad_(False)
    W0 = E.to(dev)
    x = x_cpu.to(torch.bfloat16).to(dev).requires_grad_(True)
    gz = torch.randn(N, D, generator=torch.Generator().manual_seed(12)).to(dev)
    one = torch.ones([], device=dev)
    res = {}

    def step():
        z, loss, memo = q(x, dict())
        (gx,) = torch.autograd.grad((z, loss), (x,), (gz, one))
        res.update(z=z.detach(), loss=loss.detach(), quant=memo['quant'], gx=gx)

    def run(fn):
        with torch.no_grad():
            q.embedding.weight.copy_(W0)
        fn()
        torch.cuda.synchronize()
        return {k: v.clone() for k, v in res.items()} | {'W': q.embedding.weight.detach().clone()}

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
            assert torch.equal(eager[k], replay[k]), k
    del g


# ---- 7. two GPUs --------------------------------------------------------------------------------------------------
VQGAN = dict(type='VQGANQuantizer', distance=dict(type='L2Distance'), losses=dict(vqgan_loss=dict(type='VQGANLoss')),
             init_weights=dict(type='vqgan'))
VQKD = dict(type='VQKDQuantizer', distance=dict(type='CosineDistance'), callbacks=[dict(type='VQKDCallback', ema=dict())],
            losses=dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True))))


def _two_runs(cfg, rank, world):
    from oracle import oracle as O
    torch.use_deterministic_algorithms(True)
    dev = torch.device('cuda', rank)
    N, K, D = 4096, 1024, 32
    x_all, E = O.synthetic_latents(N * world * 2, K, D, seed=5, normalized_codebook=True)
    runs = []
    for _ in range(2):
        q = vqb.build_quantizer(dict(cfg, embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K,
                                                         embedding_dim=D)), training=True).to(dev)
        q._forward_pre_hooks.clear()
        with torch.no_grad():
            q.embedding.weight.copy_(E)
        out = []
        for s in range(2):
            x = x_all[(s * world + rank) * N:(s * world + rank + 1) * N].to(dev).requires_grad_(True)
            q.embedding.weight.grad = None
            z, loss, memo = q(x, dict())
            (loss + z.sum()).backward()
            W_grad = q.embedding.weight.grad
            out.append([loss.detach().cpu(), x.grad.cpu(), None if W_grad is None else W_grad.cpu(),
                        q.embedding.weight.detach().cpu()])
        runs.append(out)
    return runs


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, cfg, out, comm, ack):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), VQB_COMM=comm)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        out.put((rank, _two_runs(cfg, rank, world)))
        ack.wait(120)            # stay alive until the parent has read the tensors
    finally:
        dist.destroy_process_group()


def _spawn(cfg, comm, world=2):
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    out, ack, port = ctx.SimpleQueue(), ctx.Event(), _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cfg, out, comm, ack)) for r in range(world)]
    for p in procs:
        p.start()
    res, deadline = {}, time.time() + 240
    while len(res) < world:      # never block on the queue: a dead worker fails the test instead of hanging it
        if not out.empty():
            r, v = out.get()
            res[r] = v
            continue
        if any(p.exitcode not in (None, 0) for p in procs) or time.time() > deadline:
            for p in procs:
                if p.is_alive():
                    p.kill()
            raise AssertionError(f'worker(s) failed or timed out: exit codes {[p.exitcode for p in procs]}')
        time.sleep(0.05)
    ack.set()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    return [res[r] for r in range(world)]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
@pytest.mark.parametrize('comm', ['p2p', 'nccl'])
@pytest.mark.parametrize('cfg', [VQKD, VQGAN], ids=['vqkd', 'vqgan'])
def test_two_gpu_steps_bitwise_reproducible(cfg, comm):
    for first, second in _spawn(cfg, comm):
        _assert_bitwise(first, second)
