"""bench.py — quantized tokens/sec of the codebook-quantization hot path on N B200 GPUs.

Workload (BASELINE.json configs[1], the config the metric is quoted on): VQ-KD cosine quantizer,
l2-normalised 8192 x 32 codebook, batch 256 x 256 = 65 536 bf16 tokens per GPU, forward + straight-through
backward of a TRAINING step, driven through the drop-in module (`VQKDQuantizer.forward` in training mode,
reference-style config): nearest code, per-code count/sum statistics, their exchange across the GPUs
(vq/algorithms/vqkd/quantizers/callbacks.py:63-64, vq/utils.py:35), k-means/EMA codebook update, gather +
straight-through + commitment loss, backward to the tokens.  At N > 1 the statistics exchange is inside
the timed step (fused into the update kernel over NVLink peer memory; `collective` in the JSON line).
A "step" is one such forward+backward over one batch of synthetic latents.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2|cfg3]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line (rank 0).  `--impl reference` times the reference's own CPU implementation of the
path (the oracle port, pinned bit-for-bit to the reference source) on the host cores.
Only this file's cpu_baseline / `--impl reference` legs execute anything under oracle/.
`--dump-outputs DIR` writes rank 0's results of the last timed step as DIR/<name>.npy (see dump_outputs()); the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import sys
import threading
import time

import torch

ROOT = pathlib.Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

SEED = 3407  # reference default (vq/train.py:21)

WORKLOADS = {
    # BASELINE.json configs[1]
    'cfg2': dict(name='cfg2: VQ-KD cosine quantizer training step (stats exchange + EMA update), fwd + straight-through bwd',
                 N=65536, K=8192, D=32, metric='Cosine', training=True,
                 config=dict(type='VQKDQuantizer', distance=dict(type='CosineDistance'),
                             callbacks=[dict(type='VQKDCallback', ema=dict())],
                             losses=dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True)))),
                 oracle=dict(distance='Cosine', callback='VQKDCallback',
                             losses={'commitment_loss': dict(type='CommitmentLoss', norm=True)})),
    # BASELINE.json configs[2]: LlamaGen-style 16384 x 8 l2-normalised codebook + EMA update + usage stats
    'cfg3': dict(name='cfg3: l2-normalised 16384x8 codebook, k-means/EMA update + usage stats, fwd + bwd', N=65536,
                 K=16384, D=8, metric='Cosine', training=True,
                 config=dict(type='VQKDQuantizer', distance=dict(type='CosineDistance'),
                             callbacks=[dict(type='VQKDCallback', ema=dict())],
                             losses=dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True)))),
                 oracle=dict(distance='Cosine', callback='VQKDCallback',
                             losses={'commitment_loss': dict(type='CommitmentLoss', norm=True)})),
    # BASELINE.json configs[3]: CVQ-VAE training step with online anchor re-init (usage counters + EMA all-reduce)
    'cfg4': dict(name='cfg4: CVQ-VAE training step (cosine, usage-EMA, NearestAnchor re-init), fwd + bwd', N=16384,
                 K=8192, D=256, metric='Cosine', training=True,
                 config=dict(type='VQGANQuantizer', distance=dict(type='CosineDistance'),
                             callbacks=[dict(type='CVQVAECallback', ema=dict(), anchor=dict(type='NearestAnchor'))],
                             losses=dict(vqgan_loss=dict(type='VQGANLoss')), init_weights=dict(type='vqgan')),
                 oracle=dict(distance='Cosine', callback='CVQVAECallback',
                             losses={'vqgan_loss': dict(type='VQGANLoss')})),
}
# BASELINE.json configs[4] (codebook-sharded 262144 x 768 stress) is `--workload cfg5`, see run_cfg5().


def emb(K, D):
    return dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D)


def synth(N, K, D, seed):
    """Seeded synthetic latents (SURVEY.md §8d): trained-like unit-norm codebook, clustered tokens."""
    g = torch.Generator(device='cpu').manual_seed(seed)
    E = torch.nn.functional.normalize(torch.randn(K, D, generator=g))
    pi = torch.randint(0, K, (N,), generator=g)
    x = E[pi] + 0.5 * E.std() * torch.randn(N, D, generator=g)
    gz = torch.randn(N, D, generator=g)
    return x.to(torch.bfloat16), E, gz


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each tensor as out_dir/<name>.npy: floating-point results as float32, code indices as float64 (exact
    for every index).  Every workload's outputs fit DUMP_LIMIT_BYTES whole (cfg4, the largest, is ~40 MB)."""
    import numpy as np
    host = {name: (t.float() if t.is_floating_point() else t.double()).detach().cpu().numpy()
            for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_LIMIT_BYTES, f'--dump-outputs: {total} bytes exceed {DUMP_LIMIT_BYTES}'
    out = pathlib.Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in host.items():
        np.save(out / f'{name}.npy', a)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the GPU legs run."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {'hw_slowdown': getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8),
                 'hw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40),
                 'sw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20),
                 'sw_power_cap': getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4)}
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)
                util = nv.nvmlDeviceGetUtilizationRates(self._h).gpu
                self.samples.append((mhz, util))
                get = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                    nv.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = get(self._h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.02)

    def start(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        busy = sorted(m for m, u in self.samples if u > 0) or sorted(m for m, _ in self.samples)
        return dict(sm_mhz=busy[len(busy) // 2] if busy else None, sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(self.samples))


# ------------------------------------------------------------------------------------------------
def run_reference(args, wl, budget_s: float = 150.0):
    """The reference's CPU implementation of the path (oracle port) on the host cores.  Runs EXACTLY args.steps timed
    steps after args.warmup warm-ups; each step is a bounded sample of the workload: the full batch when the run fits
    the time budget, otherwise the first rows of it (stated in `sample`)."""
    from oracle import oracle as O
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    N, K, D = wl['N'], wl['K'], wl['D']
    x, E, gz = synth(N, K, D, SEED)
    spec = O.QuantizerSpec(training=wl['training'], **wl['oracle'])
    prob = torch.zeros(K) if wl['oracle'].get('callback') == 'CVQVAECallback' else None

    def step(n):
        xo = x[:n].float().requires_grad_(True)
        out = O.quantizer_forward(spec, [xo], E, prob)
        torch.autograd.backward((out['z_ste'][0], out['loss'][0]), (gz[:n], torch.ones([])))
        return dict(z=out['z_ste'][0], loss=out['loss'][0], quant=out['quant'][0], gx=xo.grad, codebook=out['weight'])

    t0 = time.perf_counter()
    step(N)                                    # untimed probe: sizes the per-step sample
    probe = time.perf_counter() - t0
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    n = N
    if probe * (steps + warmup) > budget_s:
        n = max(1024, int(N * budget_s / (probe * (steps + warmup))) // 1024 * 1024)
    for _ in range(warmup):
        step(n)
    t0 = time.perf_counter()
    for _ in range(steps):
        last = step(n)
    dt = (time.perf_counter() - t0) / steps
    value = n / dt
    sample = (f'{"full batch" if n == N else f"first {n} of {N} tokens"} of {wl["name"]} per step x {steps} timed steps '
              f'after {warmup} warm-ups, fp32, torch {torch.__version__} CPU, {threads} threads')
    return dict(value=value, ms=dt * 1e3, cores=threads, kind='port', sample=sample, steps=steps, warmup=warmup,
                outputs=last)


def run_gpu_eager(wl, dev, x0, E, gz0, autocast: bool, steps: int = 10):
    """Context, not the product: the reference's OWN op sequence (normalize -> einsum -> 1 - d -> argmin -> bincount /
    scatter_add / EMA -> embedding -> mse -> backward; the oracle restatement executed with CUDA tensors, i.e. stock
    ATen / cuBLAS kernels) on the same B200.  `autocast`: under torch.autocast(bf16) as the reference trains."""
    from oracle import oracle as O
    spec = O.QuantizerSpec(training=wl['training'], **wl['oracle'])
    x, W, gz = x0.to(dev), E.to(dev), gz0.to(dev)
    prob = torch.zeros(wl['K'], device=dev) if wl['oracle'].get('callback') == 'CVQVAECallback' else None
    one = torch.ones([], device=dev)

    def step():
        xo = (x if autocast else x.float()).detach().requires_grad_(True)
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=autocast):
            out = O.quantizer_forward(spec, [xo], W, prob)
        torch.autograd.backward((out['z_ste'][0], out['loss'][0]), (gz.to(out['z_ste'][0].dtype), one))

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return dict(value=wl['N'] / (ms * 1e-3), ms_per_step=ms)


def run_cfg5(args, rank, world, local_rank):
    """Cluster-tokenizer stress: 262144 x 768 codebook sharded by contiguous row blocks over the ranks, 65536
    CLIP-sized bf16 tokens replicated; step = normalise+pack the local shard, fused tcgen05 arg-min with global
    code indices, packed (distance, index) min-loc all-reduce, index unpack."""
    import torch.distributed as dist

    from vector_quantization_b200 import ops, parallel
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    N, K, D = 65536, 262144, 768
    lo, hi = parallel.shard_range(K, rank, world)
    g = torch.Generator(device='cpu').manual_seed(SEED)
    x = torch.randn(N, D, generator=g).to(torch.bfloat16).to(dev)
    W = torch.randn(hi - lo, D, generator=torch.Generator(device='cpu').manual_seed(SEED + 1 + rank)).to(dev)
    precision = os.environ.get('VQB_PRECISION', 'fp32')

    def step():
        return parallel.sharded_nearest_code(x, W, 'Cosine', shard_lo=lo, precision=precision)[0]

    ops.LAUNCHES = 0
    step()
    launches = ops.LAUNCHES
    for _ in range(max(args.warmup, 3)):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = args.steps
    e0.record()
    for _ in range(steps):
        quant = step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(quant=quant))
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    terms = {'fp32': 2, 'exact': 3, 'high': 2, 'fast': 1}[precision]
    fmt = 'the fp16 (hi, lo*2^11) plane pair (22 bits)' if precision == 'fp32' else f'{terms} bf16 plane(s)'
    if rank == 0:
        print(json.dumps(dict(
            metric='quantized tokens/sec', value=N / (ms * 1e-3), unit='tokens/s', n_gpus=world, steps=steps,
            warmup=max(args.warmup, 3), ms_per_step=ms, higher_is_better=True, scaling='strong', vs_baseline=None,
            dtype=f'bf16 tokens, fp32 codebook as {fmt}', data='synthetic',
            config=dict(workload='cfg5: 262144x768 codebook sharded over the ranks, 65536 tokens replicated, '
                                 'min-loc all-reduce', parallelism=f'codebook-sharded x{world}', precision=precision,
                        l2_policy='operands (shard planes >= 150 MB) exceed L2'),
            roofline=dict(bound='tensor', achieved=2.0 * N * (hi - lo) * D / (ms * 1e-3) / 1e12, unit='TFLOP/s',
                          note='per-GPU algorithmic 2*N*K_shard*D over the WHOLE step (pack + assign + all-reduce)'),
            gpu_launches=launches * steps, checksum=int(quant.sum()))))
        sys.stdout.flush()
    if world > 1:
        threading.Timer(20.0, lambda: os._exit(0)).start()
        dist.barrier()
        dist.destroy_process_group()
    os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200,
                    help='timed steps of the metric (every workload and --impl); the secondary legs time fewer: '
                         'the end-to-end leg min(K, 100) steps, the isolated assign-kernel timing min(K, 30) launches')
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS) + ['cfg5'])
    ap.add_argument('--no-graph', action='store_true', help='launch eagerly instead of replaying CUDA graphs')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--e2e-h2d-streams', type=int, default=1, choices=[1, 2],
                    help='end-to-end leg: copy the tokens and the upstream gradient on one or on two copy streams')
    ap.add_argument('--e2e-readback', default='result', choices=['result', 'all'],
                    help="end-to-end leg: 'result' reads the step's results back to the host (loss + token ids); "
                         "'all' also ships the bf16 token gradient, which in a training loop stays on the device")
    ap.add_argument('--breakdown', action='store_true',
                    help='also time CUDA graphs of step prefixes (encode only / + gather+loss / + backward)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="after the timed steps, write rank 0's results of the last one (z, loss, code indices, token "
                         'gradient, updated codebook; cfg5: code indices) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.workload == 'cfg5':
        return run_cfg5(args, rank, world, local_rank)
    wl = WORKLOADS[args.workload]
    metric, unit = 'quantized tokens/sec', 'tokens/s'
    base_cfg = dict(workload=wl['name'], tokens_per_gpu=wl['N'], codebook=f'{wl["K"]}x{wl["D"]} fp32 master',
                    token_dtype='bf16', parallelism=f'token-sharded x{world}' if world > 1 else 'single GPU')

    if args.impl == 'reference':
        if rank != 0:
            return
        r = run_reference(args, wl)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r['outputs'])
        print(json.dumps(dict(
            metric=metric, value=r['value'], unit=unit, n_gpus=args.gpus, steps=r['steps'], warmup=r['warmup'],
            ms_per_step=r['ms'], higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
            impl='reference', config=base_cfg,
            cpu_baseline=dict(value=r['value'], unit=unit, cores=r['cores'], kind=r['kind'], sample=r['sample']),
            e2e=dict(value=r['value'], unit=unit, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)))
        return

    # ---------------------------------------------------------------- B200 arm
    import torch.distributed as dist

    import vector_quantization_b200 as vqb
    from vector_quantization_b200 import ops

    assert torch.cuda.is_available(), 'bench.py --impl b200 needs a CUDA device (no CPU fallback)'
    numa, all_cpus = None, os.sched_getaffinity(0)
    try:   # run on the CPUs next to this rank's GPU, so that pinned host buffers are allocated NUMA-local
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
        numa = f'{len(os.sched_getaffinity(0))} CPUs next to GPU {local_rank}'
    except Exception as exc:  # noqa: BLE001
        numa = f'not set ({exc})'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    N, K, D = wl['N'], wl['K'], wl['D']
    cfg = dict(wl['config'], embedding=emb(K, D))
    q = vqb.build_quantizer(cfg, training=wl['training']).to(dev)
    q._forward_pre_hooks.clear()  # steady-state step (the one-off k-means init is not part of the metric)
    if args.workload in ('cfg2', 'cfg3'):
        q.requires_grad_(False)   # VQ-KD freezes the quantizer parameters (reference configs/vqkd/model.py:76-82)
    x0, E, gz0 = synth(N, K, D, SEED + rank)
    with torch.no_grad():
        q.embedding.weight.copy_(synth(N, K, D, SEED)[1])  # identical codebook on every rank
    # rotating input sets: 24 x (4 MB tokens + 8 MB upstream grad) = 288 MB > 2 x 126 MB L2
    n_sets = 24
    sets = []
    for i in range(n_sets):
        xi = x0.roll(i * 977, 0).to(dev).requires_grad_(True)
        sets.append((xi, gz0.roll(i * 977, 0).to(dev)))
    one = torch.ones([], device=dev)
    result = {}

    def step(i):
        xi, gzi = sets[i % n_sets]
        z, loss, memo = q(xi, dict())
        (gx,) = torch.autograd.grad((z, loss), (xi,), (gzi, one))  # straight-through backward to the tokens
        result.update(loss=loss.detach(), quant=memo['quant'], gx=gx, z=z.detach())

    sampler = ClockSampler(local_rank)
    sampler.start()
    ops.LAUNCHES = 0
    step(0)
    launches_per_step = ops.LAUNCHES
    for i in range(3):
        step(i)
    torch.cuda.synchronize()

    graphs = None
    if not args.no_graph:
        # one CUDA graph per input set: replaying graph i runs the whole step on set i with cold inputs
        graphs, outs = [], []
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for i in range(n_sets):
                step(i)
        torch.cuda.current_stream().wait_stream(s)
        pool = None
        for i in range(n_sets):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                step(i)
                outs.append(dict(result))
            pool = g.pool()
            graphs.append(g)

        def run(i):
            graphs[i % n_sets].replay()
            return outs[i % n_sets]
    else:
        def run(i):
            step(i)
            return result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        run(i)
    # ---- timed region: exactly K steps ----
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        last = run(i)
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:   # before any later leg runs another step (training updates the codebook)
        dump_outputs(args.dump_outputs, dict(z=last['z'], loss=last['loss'], quant=last['quant'], gx=last['gx'],
                                             codebook=q.embedding.weight))
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    value = N * world / (ms * 1e-3)

    breakdown = None
    if args.breakdown and graphs is not None and world == 1:
        # in-graph share of each stage: graphs of step PREFIXES over the same rotating input sets
        def prefix(stage):
            def fn(i):
                xi, gzi = sets[i % n_sets]
                if stage == 0:
                    with torch.no_grad():
                        q.encode(xi.detach(), dict(_lazy_unpack=True, _lazy_normalize=True))  # as in forward()
                    return
                z, loss, memo = q(xi, dict())
                if stage == 2:
                    torch.autograd.grad((z, loss), (xi,), (gzi, one))
            return fn
        breakdown = {}
        for stage, name in enumerate(('encode (packs + assign)', '+ gather/STE/loss', '+ backward')):
            fn = prefix(stage)
            gs = []
            for i in range(n_sets):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, pool=pool):
                    fn(i)
                gs.append(g)
            for i in range(10):
                gs[i % n_sets].replay()
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.steps):
                gs[i % n_sets].replay()
            e1.record()
            torch.cuda.synchronize()
            breakdown[name] = e0.elapsed_time(e1) / args.steps
            del gs

    # ---- dominant kernel (tcgen05 assignment) timed live with CUDA events on the launching stream ----
    # Same operands as inside the step (raw bf16 tokens: 1 exact plane; normalised fp32 codebook: the fp16
    # (hi, lo*2^11) pair for the default precision, 3 bf16 planes for precision='exact').
    # A 1 GiB memset before every launch flushes L2 and keeps the GPU busy while the host enqueues, so the
    # event pair brackets the kernel only (no host launch latency inside).
    from vector_quantization_b200 import functional as Fq
    flush = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    x_first = sets[0][0].detach()
    book = Fq.pack_codebook(q.embedding.weight.data, wl['metric'], precision=q.precision, writeback_normalized=True,
                            tokens=x_first)
    toks = ops.as_operand(x_first) if (D <= 64 or not book.pair) else None      # same choice as Fq.nearest_code
    if toks is None:
        toks = ops.pack_rows(x_first, fmt='f16') if book.pair else ops.pack_rows(x_first, planes=1)
    n_terms = 2 if book.pair else book.nplanes
    keys = ops.new_keys(N, dev)
    ops.PROFILE = []
    for i in range(min(args.steps, 30) + 3):
        flush.zero_()
        ops.assign(toks, book, keys, l2=wl['metric'] == 'L2')
    torch.cuda.synchronize()
    assign_ms = [a.elapsed_time(b) for name, a, b in ops.PROFILE if name == 'vqb_assign'][3:]
    # ---- every kernel of the step, timed live the same way (eager launches behind an L2-flushing memset that keeps
    # the GPU busy while the host enqueues the step): the HBM-bound kernels against the measured copy bandwidth, and
    # the statistics exchange.  All ranks run the same number of steps (the exchange is a collective).
    ops.PROFILE = []
    n_prof = 12
    for i in range(n_prof):
        flush.zero_()
        flush.zero_()          # ~0.35 ms of memset: the whole step is enqueued before the GPU gets to it
        step(i)
    torch.cuda.synchronize()
    per_kernel = {}
    for name, a, b in ops.PROFILE[len(ops.PROFILE) // n_prof * 2:]:      # skip the first two steps
        per_kernel.setdefault(name, []).append(a.elapsed_time(b))
    ops.PROFILE = None
    del flush
    assign_ms.sort()
    assign_avg = sum(assign_ms) / len(assign_ms)
    peaks = {}
    try:
        peaks = json.load(open(ROOT / 'MEASURED_PEAKS.json'))
    except Exception:  # noqa: BLE001
        pass
    peak_tf = peaks.get('bf16_tflops', 1590.0)   # the kernel is timed ALONE (event-bracketed launches) -> burst figure
    flops = 2.0 * N * K * D                              # algorithmic: contraction only, un-padded, one plane
    achieved = flops / (assign_avg * 1e-3) / 1e12
    # DRAM traffic of the same kernel from the committed `ncu --set full` capture (profiles/, per launch)
    traffic, ncu_note = None, None
    try:
        ncu = json.load(open(ROOT / 'profiles' / 'r2_assign_ncu_summary.json'))
        if args.workload == 'cfg2':
            to_b = {'byte': 1, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
            traffic = sum(float(ncu[k]['value']) * to_b[ncu[k]['unit']]
                          for k in ('dram__bytes_read.sum', 'dram__bytes_write.sum'))
            ncu_note = dict(tensor_pipe_active_pct=float(
                ncu['sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active']['value']),
                source='profiles/r2_assign_ncu_summary.json (ncu --set full capture of this kernel in this workload; per launch)')
    except Exception:  # noqa: BLE001
        pass
    roofline = dict(bound='tensor', kernel='assign_tc_kernel (tcgen05 distance GEMM + fused arg-min)',
                    achieved=achieved, peak=peak_tf, unit='TFLOP/s', frac=achieved / peak_tf,
                    peak_source='MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone)' if peaks else 'fallback 1.59 PFLOP/s (B200_PROFILING.md)',
                    frac_of_sustained=achieved / peaks.get('bf16_tflops_sustained', 1400.0),
                    kernel_ms=assign_avg, kernel_share_of_step=assign_avg / ms,
                    epilogue_gelem_per_s=N * K / (assign_avg * 1e-3) / 1e9, traffic=traffic,
                    algorithmic_bytes=N * D * 2 + K * D * 2 * book.nplanes + N * 8, ncu=ncu_note,
                    mma_terms=n_terms, mma_issued_tflops=achieved * n_terms * (book.planes.shape[-1] / D),
                    note=f'algorithmic flops 2*N*K*D (one plane); the fp32 codebook is fed as {book.nplanes} 16-bit '
                         f'planes = {n_terms} MMA terms per tile, so the tensor pipe is ~{n_terms}x busier than '
                         '`frac` (mma_issued_tflops; see ncu.tensor_pipe_active_pct)')

    hbm = peaks.get('hbm_gbs', 6650.0)
    s_x = 2                                              # bf16 tokens
    launches_of = {k: len(v) / (n_prof - 2) for k, v in per_kernel.items()}
    alg_bytes = {   # algorithmic HBM bytes per launch (DESIGN.md §4); the L2-resident codebook rows are NOT counted
        'vqb_gather_ste_loss': N * (D * (s_x + 4) + 8) + (0 if wl['training'] else N * 8),
        'vqb_quantize_backward': N * (D * (4 + s_x + s_x) + 8),
        'vqb_scatter_stats': N * (D * s_x + 8) + K * (D + 1) * 4,
        'vqb_pack_rows': K * D * (4 + 4 + 2 * book.nplanes) + N * 8,
        'vqb_unpack_keys': N * 16,
    }
    membound = []
    for name, times in sorted(per_kernel.items()):
        t = sum(times) / len(times)
        rec = dict(kernel=name, ms=t, launches_per_step=launches_of[name])
        if name in alg_bytes and launches_of[name] == 1:
            rec.update(bytes=alg_bytes[name], gbs=alg_bytes[name] / (t * 1e-3) / 1e9,
                       frac=alg_bytes[name] / (t * 1e-3) / 1e9 / hbm)
        membound.append(rec)
    roofline['membound'] = membound
    roofline['membound_note'] = (f'per-launch CUDA-event times of eager launches, L2 flushed before every step; fractions '
                                 f'of the measured copy bandwidth ({hbm:.0f} GB/s); at this batch size these launches '
                                 'move 4-25 MB in a few microseconds and are launch-ramp bound, see DESIGN.md')
    collective = None
    if wl['training']:
        cb = [c for c in q._callbacks if hasattr(c, '_region')]
        fused = bool(cb and cb[0]._region)
        key = 'vqb_comm_kmeans_ema_update' if 'vqb_comm_kmeans_ema_update' in per_kernel else 'vqb_comm_cvq_update'
        t = None
        if fused and key == 'vqb_comm_kmeans_ema_update':
            # the exchange+update launch alone: a burst of back-to-back launches on every rank (no host skew between
            # the ranks inside the burst), CUDA events, max over ranks
            region = cb[0]._region
            for _ in range(5):
                ops.comm_kmeans_ema_update(region, K, D, 0.99)
            barrier()
            e0.record()
            for _ in range(50):
                ops.comm_kmeans_ema_update(region, K, D, 0.99)
            e1.record()
            barrier()
            tt = torch.tensor([e0.elapsed_time(e1) / 50], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = [float(tt)]
        payload = (K * D + K) * 4 if args.workload in ('cfg2', 'cfg3') else (K + 1) * 8 + K * D * 4
        collective = dict(
            what='per-step exchange of the per-code statistics (reference: all_reduce, vq/utils.py:35, '
                 'vqkd/quantizers/callbacks.py:63-64, cvqvae/anchors.py:64-67)',
            bytes=payload if world > 1 else 0, world=world,
            algo=('two-shot reduce + publish over NVLink peer memory, fused into the codebook-update kernel '
                  f'({key}); no NCCL call on the data path') if fused else
                 ('torch.distributed all_reduce (NCCL)' if world > 1 else 'none (single GPU)'),
            ms=(sum(t) / len(t)) if (t and fused) else None,
            protocol=('low-latency: every fp32 word carries the exchange parity in its mantissa LSB (1x wire bytes), no barrier/fence, 2 one-way NVLink hops'
                      if fused and 'll_in' in cb[0]._region.offsets else
                      ('barrier: flag, peer reads, peer writes + fence, flag' if fused else None)),
            ms_note='one fused exchange+update launch, measured as a burst of 50 back-to-back launches on every rank '
                    '(max over ranks); inside the step the launch also absorbs the wait for the slowest rank')

    # ---- end-to-end: pinned host inputs -> device -> step -> results back to pinned host ----
    xh = x0.pin_memory()
    # The upstream gradient crosses PCIe as bf16 (what a bf16-autocast decoder backward produces: autograd only widens
    # it to z's fp32 afterwards) and is widened on the device, into the step's fp32 gradient buffer.
    gh = gz0.to(torch.bfloat16).pin_memory()
    g_stage = [torch.empty(N, D, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    loss_h = torch.empty([], dtype=torch.float32).pin_memory()
    quant_h = torch.empty(N, dtype=torch.int64).pin_memory()
    gx_h = torch.empty(N, D, dtype=torch.bfloat16).pin_memory()

    # Three streams, like a training loop with a prefetching loader: the H2D copy of step i+1 and the D2H read
    # of step i-1 overlap the kernels of step i (two copy engines + SMs).  Every step still copies ITS inputs
    # from pinned host memory and reads ITS results back inside the timed region.
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    s_in2 = torch.cuda.Stream() if args.e2e_h2d_streams == 2 else s_in   # second DMA queue for the gradient
    ev_in2 = [torch.cuda.Event() for _ in range(n_sets)]
    ev_in = [torch.cuda.Event() for _ in range(n_sets)]
    ev_run = [torch.cuda.Event() for _ in range(n_sets)]
    ev_out = [torch.cuda.Event() for _ in range(n_sets)]
    cur = torch.cuda.current_stream()
    for ev in ev_run + ev_out:
        ev.record(cur)

    read_all = args.e2e_readback == 'all'

    def e2e_step(i):
        j = i % n_sets
        xi, gzi = sets[j]
        with torch.cuda.stream(s_in), torch.no_grad():
            s_in.wait_event(ev_run[j])            # the previous step that used input set j has consumed it
            xi.copy_(xh, non_blocking=True)
            ev_in[j].record(s_in)
        with torch.cuda.stream(s_in2), torch.no_grad():
            s_in2.wait_event(ev_run[j])
            g_stage[i & 1].copy_(gh, non_blocking=True)
            gzi.copy_(g_stage[i & 1])             # bf16 -> fp32 widening on the device
            ev_in2[j].record(s_in2)
        cur.wait_event(ev_in[j])
        cur.wait_event(ev_in2[j])
        cur.wait_event(ev_out[j])                 # result buffers of graph j have been read back
        out = run(i)
        ev_run[j].record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_run[j])
            if graphs is None:                    # eager results are fresh allocations of the compute stream
                for name in ('loss', 'quant', 'gx'):
                    out[name].record_stream(s_out)
            loss_h.copy_(out['loss'], non_blocking=True)
            quant_h.copy_(out['quant'], non_blocking=True)
            if read_all:
                gx_h.copy_(out['gx'], non_blocking=True)
            ev_out[j].record(s_out)

    for i in range(3):
        e2e_step(i)
    barrier()
    k2 = min(args.steps, 100)
    e0.record()
    for i in range(k2):
        e2e_step(i)
    cur.wait_stream(s_out)                       # the last read-backs are inside the timed region
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1) / k2
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t)
    h2d = xh.numel() * 2 + gh.numel() * 2
    d2h = 4 + quant_h.numel() * 8 + (gx_h.numel() * 2 if read_all else 0)
    clocks = sampler.stop()

    cpu_baseline = gpu_eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)         # the CPU baseline uses every host core again
        try:
            gpu_eager = dict(
                what="the reference's own op sequence (normalize, einsum, argmin, bincount/scatter_add/EMA, embedding, "
                     'mse_loss, autograd backward) as stock ATen/cuBLAS kernels on this B200, same workload; context only',
                fp32=run_gpu_eager(wl, dev, x0, E, gz0, autocast=False),
                autocast_bf16=run_gpu_eager(wl, dev, x0, E, gz0, autocast=True), unit=unit)
        except Exception as exc:  # noqa: BLE001 - context only
            gpu_eager = dict(error=repr(exc))
        r = run_reference(argparse.Namespace(steps=3, warmup=1), wl, budget_s=30.0)
        cpu_baseline = dict(value=r['value'], unit=unit, cores=r['cores'], kind=r['kind'], sample=r['sample'])

    if rank == 0:
        print(json.dumps(dict(
            metric=metric, value=value, unit=unit, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
            ms_per_step=ms, higher_is_better=True, scaling='weak', vs_baseline=None,
            dtype='bf16', data='synthetic',
            config=base_cfg,
            details=dict(arithmetic='16-bit tensor-core operands, fp32 accumulation: ' + (
                            'bf16 tokens zero-copy (converted to fp16 in shared memory), the fp32 codebook as the fp16 (hi, lo*2^11) plane '
                            'pair (22 significant bits, 2 MMA terms)' if book.pair else
                            f'tokens and the fp32 codebook as exact bf16 planes ({n_terms} MMA terms)') +
                        '; z/loss fp32, token gradient in the token dtype', precision=q.precision,
                        l2_policy=f'rotating {n_sets} input sets, {n_sets * (N * D * 6) >> 20} MB > L2',
                        launch='CUDA graph replay' if graphs else 'eager', kernels_per_step=launches_per_step),
            clocks=clocks, roofline=roofline, collective=collective, cpu_baseline=cpu_baseline,
            gpu_eager_baseline=gpu_eager, breakdown_ms=breakdown,
            e2e=dict(value=N * world / (e2e_ms * 1e-3), unit=unit, ms_per_step=e2e_ms, steps=k2, h2d_bytes_per_step=h2d,
                     d2h_bytes_per_step=d2h, cpu_affinity=numa,
                     readback=args.e2e_readback,
                     note='per step: bf16 tokens + bf16 upstream gradient host->device (widened to fp32 on the device), '
                          'loss + int64 token ids' + (' + bf16 token gradient' if read_all else '') + ' device->host '
                          '(the token gradient and z stay on the device, as in a training loop, unless --e2e-readback all); '
                          'three streams, PCIe-bound'),
            gpu_launches=launches_per_step * args.steps)))
    if world > 1:
        # graphs that captured NCCL collectives must be gone before the communicator is torn down; a watchdog
        # guarantees that a stuck teardown cannot hang the launcher after the result line has been printed
        sys.stdout.flush()
        threading.Timer(20.0, lambda: os._exit(0)).start()
        graphs = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        os._exit(0)


if __name__ == '__main__':
    main()
