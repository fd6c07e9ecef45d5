"""The rotation trick (rotation_trick=True) against the straight-through step and against what a user builds without it.

    python tools/bench_rotation.py [--steps 30] [--warmup 5] [--rounds 3] [--out FILE]

Training step = forward + backward of the quantizer, for four single / grouped workloads (WORKLOADS), three
residual ones (RVQ_WORKLOADS: those of tools/bench_rvq.py, the rotation over the whole depth) and three paths:
  a  rotation_trick=True: the rotation runs inside the one backward launch;
  b  rotation_trick=False: the straight-through step, as before;
  c  the module with the straight-through estimator plus eager rotation glue on its output
     (z = lambda R x with lambda, R from x and z.detach(), as in oracle/rotation.py): what users write today.
Backward kernel alone: ops.quantize_backward / ops.group_backward / ops.residual_backward with rotate on and off on
the forward's saved tensors, each call between an L2 flush (a 256 MB write) and timed with CUDA events around the call only.
Timing: CUDA events around `steps` back-to-back calls after `warmup` calls, `rounds` rounds with the paths
alternating, the median round reported.  Inputs rotate over enough seeded sets to exceed the 126 MB L2.
Before timing, a and b run from the same codebooks on the same input: z, the loss and the indices must be bitwise
equal (the rotation changes only the token gradient).
Prints one JSON line (also written to --out) with the GPU name, power limit and max SM clock of the same run."""
from __future__ import annotations

import argparse
import json
import math
import pathlib
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import vector_quantization_b200 as vqb  # noqa: E402
from vector_quantization_b200 import ops, tokenizer  # noqa: E402

L2_BYTES = 126 << 20
VQGAN_LOSS = dict(vqgan_loss=dict(type='VQGANLoss'))
# name: (layout (b, c, h, w) for NCHW, or (N, D) tokens, groups, K, distance, callbacks, latent dtype, losses, quantizer)
WORKLOADS = {
    'cfg2_vqkd': ((65536, 32), 1, 8192, 'Cosine', [dict(type='VQKDCallback', ema=dict())], torch.bfloat16,
                  dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True))), 'VQKDQuantizer'),
    'vqgan': ((64, 256, 16, 16), 1, 8192, 'L2', [], torch.float32, VQGAN_LOSS, 'VQGANQuantizer'),
    'llamagen_d8': ((256, 8, 16, 16), 1, 16384, 'L2', [dict(type='NormalizeCallback')], torch.float32, VQGAN_LOSS,
                    'VQGANQuantizer'),
    'gvq_vqgan_grid': ((64, 256, 16, 16), 4, 8192, 'L2', [], torch.float32, VQGAN_LOSS, 'VQGANQuantizer'),
}
CVQ = [dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'), ema=dict())]
# ResidualVectorQuantizer(rotation_trick=...) over levels of `quantizer`; the fields of WORKLOADS with the number of
# levels L in place of the groups
RVQ_WORKLOADS = {
    'rvq_rqvae_like': ((256, 256, 8, 8), 4, 16384, 'L2', [], torch.float32, VQGAN_LOSS, 'VQGANQuantizer'),
    'rvq_vqgan_grid_cvq': ((64, 256, 16, 16), 4, 8192, 'Cosine', CVQ, torch.float32, VQGAN_LOSS, 'VQGANQuantizer'),
    'rvq_small_d': ((256, 8, 16, 16), 8, 16384, 'L2', [], torch.float32, VQGAN_LOSS, 'VQGANQuantizer'),
}


def workload(name):
    return WORKLOADS[name] if name in WORKLOADS else RVQ_WORKLOADS[name]


def gpu_info() -> dict:
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'unavailable: {e}'
    return info


def build(name, dev, rotation_trick):
    if name in RVQ_WORKLOADS:
        return build_rvq(name, dev, rotation_trick)
    shape, G, K, dist, callbacks, _, losses, kind = WORKLOADS[name]
    D = shape[1]
    node = dict(type=kind, distance=dict(type=f'{dist}Distance'), callbacks=callbacks, losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D // G),
                rotation_trick=rotation_trick)
    cfg = node if G == 1 else dict(type='GroupedVectorQuantizer', num_groups=G, quantizer=node)
    q = vqb.build_quantizer(cfg, training=True).to(dev)
    q._forward_pre_hooks.clear()     # steady state: no k-means lazy init
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for m in (q.quantizers if G > 1 else [q]):
            m.embedding.weight.copy_(torch.randn(K, D // G, generator=g))
    return q


def build_rvq(name, dev, rotation_trick):
    """The residual workloads with the codebooks of tools/bench_rvq.py (level l at scale 0.6**l)."""
    shape, L, K, dist, callbacks, _, losses, kind = RVQ_WORKLOADS[name]
    D = shape[1]
    node = dict(type=kind, distance=dict(type=f'{dist}Distance'), callbacks=callbacks, losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D))
    q = vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=L, quantizer=node,
                                 rotation_trick=rotation_trick), training=True).to(dev)
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for l, level in enumerate(q.quantizers):
            level.embedding.weight.copy_(torch.randn(K, D, generator=g) * 0.6 ** l)
    return q


def inputs(name, dev):
    shape, _, _, _, _, dtype, _, _ = workload(name)
    g = torch.Generator().manual_seed(11)
    size = math.prod(shape) * (2 if dtype == torch.bfloat16 else 4)
    sets = max(2, math.ceil(2 * L2_BYTES / size))
    xs = [torch.randn(*shape, generator=g).to(dtype).to(dev).requires_grad_(True) for _ in range(sets)]
    gz = torch.randn(*shape, generator=g).to(dev)
    return xs, gz


def forward(q, x):
    if x.dim() == 4:
        z, loss, memo = tokenizer.quantize(q, x, dict())
        return z, loss, memo['quantizer']
    return q(x, dict())


def rotate_glue(x, z, dim):
    """z's value direction with the rotation trick's gradient to x, in eager torch (~ten elementwise and reduction
    launches forward, as many backward)."""
    xf = x.float()
    e = z.detach()
    a = xf.norm(dim=dim, keepdim=True).detach().clamp_min(1e-12)
    b = e.norm(dim=dim, keepdim=True).clamp_min(1e-12)
    u = (xf / a).detach()
    eh = e / b
    w = F.normalize(u + eh, dim=dim, eps=1e-12)
    return (b / a) * (xf - 2 * (xf * w).sum(dim, keepdim=True) * w + 2 * (xf * u).sum(dim, keepdim=True) * eh)


def step(q, x, gz, glue=False):
    z, loss, memo = forward(q, x)
    if glue:
        z = rotate_glue(x, z, 1)
    torch.autograd.backward((z, loss), (gz, torch.ones_like(loss)))
    return z, loss, memo['quant']


def timed(fn, xs, steps, warmup):
    for i in range(warmup):
        fn(xs[i % len(xs)])
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        fn(xs[i % len(xs)])
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def backward_kernel_us(q, x, gz, rotate, reps, flush):
    """The backward launch alone (rotate on / off) on the forward's saved tensors, L2 flushed before each call."""
    captured = {}
    names = ('quantize_backward', 'group_backward', 'residual_backward')
    real = {n: getattr(ops, n) for n in names}

    def grab(fn):
        def call(*a, **kw):
            captured.update(fn=fn, a=a, kw=kw)
            return fn(*a, **kw)
        return call

    for n in names:
        setattr(ops, n, grab(real[n]))
    try:
        step(q, x, gz)
    finally:
        for n in names:
            setattr(ops, n, real[n])
    fn, args, kw = captured['fn'], captured['a'], dict(captured['kw'], rotate=rotate)
    times = []
    for i in range(reps + 3):
        flush.add_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(*args, **kw)
        b.record()
        b.synchronize()
        if i >= 3:
            times.append(1000 * a.elapsed_time(b))
    return statistics.median(times)


def run(name, dev, args) -> dict:
    shape, G, K, dist, callbacks, dtype, _, kind = workload(name)
    rec = dict(workload=name, shape=list(shape), K=K, distance=dist, quantizer=kind,
               callbacks=[c['type'] for c in callbacks], dtype=str(dtype).split('.')[-1])
    rec['levels' if name in RVQ_WORKLOADS else 'groups'] = G
    xs, gz = inputs(name, dev)
    rec['input_sets'] = len(xs)
    qa, qb, qc = build(name, dev, True), build(name, dev, False), build(name, dev, False)
    # same codebooks, same input: everything but the token gradient is the same (deterministic statistics, so that
    # the training-mode codebook updates agree bit for bit)
    xa, xb = xs[0].detach().clone().requires_grad_(True), xs[0].detach().clone().requires_grad_(True)
    torch.use_deterministic_algorithms(True)
    try:
        za, la, ia = step(qa, xa, gz)
        zb, lb, ib = step(qb, xb, gz)
    finally:
        torch.use_deterministic_algorithms(False)
    rec['a_vs_b'] = dict(z_bitwise_equal=bool(torch.equal(za, zb)), loss_bitwise_equal=bool(torch.equal(la, lb)),
                         indices_equal=bool(torch.equal(ia, ib)), gx_equal=bool(torch.equal(xa.grad, xb.grad)))
    if not (rec['a_vs_b']['z_bitwise_equal'] and rec['a_vs_b']['loss_bitwise_equal'] and rec['a_vs_b']['indices_equal']):
        raise SystemExit(f'{name}: rotation_trick changed the forward: {rec["a_vs_b"]}')
    paths = {'a': lambda x: step(qa, x, gz), 'b': lambda x: step(qb, x, gz), 'c': lambda x: step(qc, x, gz, glue=True)}
    times = {k: [] for k in paths}
    for _ in range(args.rounds):
        for k, fn in paths.items():
            times[k].append(timed(fn, xs, args.steps, args.warmup))
    rec['train_step_ms'] = {k: statistics.median(v) for k, v in times.items()}
    rec['train_step_ms_rounds'] = times
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
    bwd = {'rotated': [], 'straight_through': []}
    for _ in range(args.rounds):
        bwd['rotated'].append(backward_kernel_us(qb, xs[1], gz, True, args.steps, flush))
        bwd['straight_through'].append(backward_kernel_us(qb, xs[1], gz, False, args.steps, flush))
    rec['backward_kernel_us'] = {k: statistics.median(v) for k, v in bwd.items()}
    rec['backward_kernel_us_rounds'] = bwd
    return rec


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', type=str, default=None)
    ap.add_argument('--workloads', nargs='*', default=list(WORKLOADS) + list(RVQ_WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_rotation.py measures on a CUDA device; none is available')
    dev = torch.device('cuda', 0)
    out = dict(gpu=gpu_info(), steps=args.steps, warmup=args.warmup, rounds=args.rounds,
               results=[run(name, dev, args) for name in args.workloads])
    line = json.dumps(out)
    print(line)
    if args.out:
        pathlib.Path(args.out).write_text(line + '\n')


if __name__ == '__main__':
    main()
