"""Cost of the deterministic reductions (torch.use_deterministic_algorithms(True)) on the bench.py workloads.

    python tools/bench_deterministic.py [--steps 200] [--out FILE]

For the cfg2 step (VQ-KD statistics) and the cfg4 step (CVQ-VAE, codebook gradient) it times, with bench.py's method
(CUDA events around CUDA-graph replays, one graph per rotating input set, sets together larger than the 126 MB L2):
  off         the default atomic path;
  on          the flag on, torch NaN-filling every torch.empty (torch.utils.deterministic.fill_uninitialized_memory);
  on_nofill   the flag on without that fill, which isolates the cost of the new kernels from torch's own.
It then times each launch of one eager flag-on step with CUDA events (ops.PROFILE) and counts how many distinct bit
patterns ten repeats of the atomic and of the deterministic statistics give on a hot-code input of 65 536 tokens.
Prints one JSON line (also written to --out) with the GPU name and power limit beside the numbers."""
from __future__ import annotations

import argparse
import hashlib
import json
import pathlib
import subprocess
import sys

import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (WORKLOADS, synth, emb: the same shapes and inputs as the benchmark)
import vector_quantization_b200 as vqb  # noqa: E402
from vector_quantization_b200 import ops  # noqa: E402

L2_BYTES = 126 << 20


def set_mode(mode: str) -> None:
    torch.use_deterministic_algorithms(mode != 'off')
    torch.utils.deterministic.fill_uninitialized_memory = mode != 'on_nofill'


def build(name: str, dev):
    wl = bench.WORKLOADS[name]
    N, K, D = wl['N'], wl['K'], wl['D']
    q = vqb.build_quantizer(dict(wl['config'], embedding=bench.emb(K, D)), training=True).to(dev)
    q._forward_pre_hooks.clear()
    if name == 'cfg2':
        q.requires_grad_(False)   # VQ-KD freezes the quantizer parameters (as bench.py)
    x0, E, gz0 = bench.synth(N, K, D, bench.SEED)
    with torch.no_grad():
        q.embedding.weight.copy_(E)
    per_set = x0.numel() * x0.element_size() + gz0.numel() * 4
    n_sets = max(2, -(-2 * L2_BYTES // per_set))
    sets = [(x0.roll(i * 977, 0).to(dev).requires_grad_(True), gz0.roll(i * 977, 0).to(dev)) for i in range(n_sets)]
    return q, sets


def make_step(q, sets):
    one = torch.ones([], device=sets[0][0].device)
    W = q.embedding.weight
    inputs_of = (lambda x: (x, W)) if W.requires_grad else (lambda x: (x,))

    def step(i):
        x, gz = sets[i % len(sets)]
        z, loss, memo = q(x, dict())
        torch.autograd.grad((z, loss), inputs_of(x), (gz, one))
    return step


def time_graphs(q, sets, steps: int) -> float:
    step = make_step(q, sets)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(len(sets)):
            step(i)
    torch.cuda.current_stream().wait_stream(s)
    graphs, pool = [], None
    for i in range(len(sets)):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, pool=pool):
            step(i)
        pool = g.pool()
        graphs.append(g)
    for i in range(2 * len(sets)):
        graphs[i % len(graphs)].replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for i in range(steps):
        graphs[i % len(graphs)].replay()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    del graphs
    return ms


def kernel_profile(q, sets) -> dict:
    step = make_step(q, sets)
    step(0)
    torch.cuda.synchronize()
    ops.PROFILE = []
    step(1)
    torch.cuda.synchronize()
    rec, ops.PROFILE = ops.PROFILE, None
    out = {}
    for name, a, b in rec:
        d = out.setdefault(name, dict(calls=0, ms=0.0))
        d['calls'] += 1
        d['ms'] += a.elapsed_time(b)
    return {k: dict(calls=v['calls'], ms=round(v['ms'], 5)) for k, v in out.items()}


def launches_per_step(q, sets) -> int:
    step = make_step(q, sets)
    ops.LAUNCHES = 0
    step(0)
    torch.cuda.synchronize()
    return ops.LAUNCHES


def distinct_patterns(dev, deterministic: bool, repeats: int = 10) -> int:
    N, K, D = 65536, 8192, 32
    g = torch.Generator().manual_seed(1)
    x = torch.randn(N, D, generator=g).to(dev)
    quant = torch.zeros(N, dtype=torch.int64, device=dev)   # every token on one code
    seen = set()
    for _ in range(repeats):
        stats = ops.scatter_stats(x, quant, K, normalize_x=True, deterministic=deterministic)
        torch.cuda.synchronize()
        seen.add(hashlib.sha256(stats.cpu().numpy().tobytes()).hexdigest())
    return len(seen)


def gpu_info() -> dict:
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'unavailable: {e}'
    return info


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_deterministic needs a CUDA device')
    dev = torch.device('cuda', 0)
    result = dict(gpu=gpu_info(), steps=args.steps, chunk=ops.segment_chunk(), workloads={})
    prev = (torch.are_deterministic_algorithms_enabled(), torch.utils.deterministic.fill_uninitialized_memory)
    try:
        for name in ('cfg2', 'cfg4'):
            q, sets = build(name, dev)
            rec = dict(input_sets=len(sets))
            for rep in range(2):          # the three modes interleaved, twice: the spread is part of the result
                for mode in ('off', 'on', 'on_nofill'):
                    set_mode(mode)
                    rec.setdefault(f'ms_per_step_{mode}', []).append(round(time_graphs(q, sets, args.steps), 5))
            for mode in ('off', 'on_nofill'):
                set_mode(mode)
                rec[f'launches_per_step_{mode}'] = launches_per_step(q, sets)
                rec[f'kernels_{mode}'] = kernel_profile(q, sets)
            result['workloads'][name] = rec
            del q, sets
            torch.cuda.empty_cache()
        set_mode('off')
        result['hot_code_stats_distinct_bit_patterns_of_10'] = dict(
            atomic=distinct_patterns(dev, False), deterministic=distinct_patterns(dev, True))
    finally:
        torch.use_deterministic_algorithms(prev[0])
        torch.utils.deterministic.fill_uninitialized_memory = prev[1]
    line = json.dumps(result)
    print(line)
    if args.out:
        pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(args.out).write_text(line + '\n')


if __name__ == '__main__':
    main()
