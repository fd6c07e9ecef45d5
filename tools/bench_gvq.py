"""Grouped quantization (GroupedVectorQuantizer) against what a user builds without it.

    python tools/bench_gvq.py [--steps 30] [--warmup 5] [--rounds 3] [--out FILE]

Training step = forward + backward of the quantizer on NCHW latents, for three workloads (WORKLOADS) and three paths:
  a  the new module through tokenizer.quantize: one split launch in, one assignment per group, ONE gather launch for
     all groups writing z NCHW, ONE backward launch for all groups;
  b  G VectorQuantizer modules through eager glue, as users write it today: permute in, `x.chunk(G, 1)` plus a
     `.contiguous()` copy per group, `z_g, loss_g = vq_g(x_g)`, `torch.cat`, the group-mean loss, permute out;
     G autograd nodes in the backward;
  c  stock eager torch: per group torch.cdist / the cosine matmul, argmin, F.embedding, F.mse_loss terms and the
     same glue (no codebook update: the CVQ-VAE re-initialisation of workload 2 is not part of this path).
Decode: tokenizer.decode_from_quant on [b, h, w, G] ids against G x F.embedding + cat + permute().contiguous().
Timing: CUDA events around `steps` back-to-back calls after `warmup` calls, `rounds` rounds with the paths
alternating, the median round reported.  Inputs rotate over enough seeded sets to exceed the 126 MB L2.
Before timing, a and b run from the same codebooks on the same input; their indices must agree everywhere and z must
be bitwise equal (each group of a is its own VectorQuantizer by construction).
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
from vector_quantization_b200 import tokenizer  # noqa: E402

L2_BYTES = 126 << 20
WORKLOADS = {   # name: (b, G, Dg, h, w, K, distance, CVQ-VAE callback, latent dtype, losses)
    'vqgan_grid': (64, 4, 64, 16, 16, 8192, 'L2', False, torch.float32, dict(vqgan_loss=dict(type='VQGANLoss'))),
    'cvqvae_bf16': (64, 8, 32, 16, 16, 4096, 'Cosine', True, torch.bfloat16, dict(vqgan_loss=dict(type='VQGANLoss'))),
    'small_groups': (256, 8, 8, 16, 16, 4096, 'L2', False, torch.float32, dict(vqgan_loss=dict(type='VQGANLoss'))),
}


def gpu_info() -> dict:
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'unavailable: {e}'
    return info


def group_config(name):
    b, G, Dg, h, w, K, dist, cvq, _, losses = WORKLOADS[name]
    callbacks = [dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'), ema=dict())] if cvq else []
    return dict(type='VQGANQuantizer', distance=dict(type=f'{dist}Distance'), callbacks=callbacks, losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=Dg))


def build(name, dev):
    b, G, Dg, h, w, K, dist, cvq, dtype, losses = WORKLOADS[name]
    g = torch.Generator().manual_seed(7)
    Ws = [torch.randn(K, Dg, generator=g) for _ in range(G)]
    gvq = vqb.build_quantizer(dict(type='GroupedVectorQuantizer', num_groups=G, quantizer=group_config(name)),
                              training=True).to(dev)
    groups = [vqb.build_quantizer(group_config(name), training=True).to(dev) for _ in range(G)]
    stock = [torch.nn.Parameter(W.to(dev)) for W in Ws]
    with torch.no_grad():
        for i, W in enumerate(Ws):
            gvq.quantizers[i].embedding.weight.copy_(W)
            groups[i].embedding.weight.copy_(W)
    size = b * G * Dg * h * w * (2 if dtype == torch.bfloat16 else 4)
    sets = max(2, math.ceil(2 * L2_BYTES / size))
    xs = [torch.randn(b, G * Dg, h, w, generator=g).to(dtype).to(dev) for _ in range(sets)]
    gz = torch.randn(b, G * Dg, h, w, generator=g).to(dev)
    return gvq, groups, stock, xs, gz


def step_a(gvq, x, gz):
    z, loss, memo = tokenizer.quantize(gvq, x, dict())
    torch.autograd.backward((z, loss), (gz, torch.ones_like(loss)))
    return z, memo['quantizer']['quant']


def step_b(groups, x, gz):
    b, c, h, w = x.shape
    rows = x.permute(0, 2, 3, 1).reshape(-1, c)
    zs, loss, quants = [], None, []
    for vq, xg in zip(groups, rows.chunk(len(groups), 1)):
        z_g, loss_g, memo = vq(xg.contiguous(), dict())
        zs.append(z_g)
        quants.append(memo['quant'])
        loss = loss_g if loss is None else loss + loss_g
    z = torch.cat(zs, 1).view(b, h, w, c).permute(0, 3, 1, 2).contiguous()
    torch.autograd.backward((z, loss / len(groups)), (gz, torch.ones_like(loss)))
    return z, torch.stack(quants, 1)


def step_c(stock, metric, x, gz):
    b, c, h, w = x.shape
    rows = x.permute(0, 2, 3, 1).reshape(-1, c).float()
    zs, loss = [], None
    for W, xg in zip(stock, rows.chunk(len(stock), 1)):
        with torch.no_grad():
            if metric == 'L2':
                q = torch.cdist(xg, W).argmin(1)
            else:
                q = (1 - F.normalize(xg) @ F.normalize(W).T).argmin(1)
        e = F.embedding(q, W)
        loss_g = F.mse_loss(e, xg.detach()) + 0.25 * F.mse_loss(e.detach(), xg)
        zs.append(xg + (e - xg).detach())
        loss = loss_g if loss is None else loss + loss_g
    z = torch.cat(zs, 1).view(b, h, w, c).permute(0, 3, 1, 2).contiguous()
    torch.autograd.backward((z, loss / len(stock)), (gz, torch.ones_like(loss)))
    return z


def decode_a(gvq, ids):
    return tokenizer.decode_from_quant(gvq, ids, dict(), check=False)[0]


def decode_c(Ws, ids):
    z = torch.cat([F.embedding(ids[..., g], W) for g, W in enumerate(Ws)], -1)
    return z.permute(0, 3, 1, 2).contiguous()


def timed(fn, inputs, steps, warmup):
    for i in range(warmup):
        fn(inputs[i % len(inputs)])
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        fn(inputs[i % len(inputs)])
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def run(name, dev, args) -> dict:
    b, G, Dg, h, w, K, dist, cvq, dtype, _ = WORKLOADS[name]
    gvq, groups, stock, xs, gz = build(name, dev)
    rec = dict(workload=name, b=b, G=G, Dg=Dg, h=h, w=w, K=K, distance=dist, cvq=cvq, dtype=str(dtype).split('.')[-1],
               input_sets=len(xs))
    # same codebooks, same input: compare before any codebook update
    xa = xs[0].clone().requires_grad_(True)
    xb = xs[0].clone().requires_grad_(True)
    za, qa = step_a(gvq, xa, gz)
    zb, qb = step_b(groups, xb, gz)
    rec['a_vs_b'] = dict(indices_equal=bool(torch.equal(qa, qb)), z_bitwise_equal=bool(torch.equal(za, zb)),
                         gx_bitwise_equal=bool(torch.equal(xa.grad, xb.grad)))
    if not (rec['a_vs_b']['indices_equal'] and rec['a_vs_b']['z_bitwise_equal']):
        raise SystemExit(f'{name}: the module and the per-group VectorQuantizers disagree: {rec["a_vs_b"]}')
    inputs = [x.requires_grad_(True) for x in xs]
    paths = {'a': lambda x: step_a(gvq, x, gz), 'b': lambda x: step_b(groups, x, gz),
             'c': lambda x: step_c(stock, dist, x, gz)}
    times = {k: [] for k in paths}
    for _ in range(args.rounds):
        for k, fn in paths.items():
            times[k].append(timed(fn, inputs, args.steps, args.warmup))
    rec['train_step_ms'] = {k: statistics.median(v) for k, v in times.items()}
    rec['train_step_ms_rounds'] = times
    # decode
    ids = [torch.randint(0, K, (b, h, w, G), generator=torch.Generator().manual_seed(i)).to(dev)
           for i in range(max(2, math.ceil(2 * L2_BYTES / (b * G * Dg * h * w * 4))))]
    Ws = [grp.embedding.weight.detach() for grp in gvq.quantizers]
    with torch.no_grad():
        assert torch.equal(decode_a(gvq, ids[0]), decode_c(Ws, ids[0]))
        dec = {'a': [], 'c': []}
        for _ in range(args.rounds):
            dec['a'].append(timed(lambda i: decode_a(gvq, i), ids, args.steps * 4, args.warmup))
            dec['c'].append(timed(lambda i: decode_c(Ws, i), ids, args.steps * 4, args.warmup))
    rec['decode_us'] = {k: 1000 * statistics.median(v) for k, v in dec.items()}
    return rec


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', type=str, default=None)
    ap.add_argument('--workloads', nargs='*', default=list(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_gvq.py measures on a CUDA device; none is available')
    dev = torch.device('cuda', 0)
    out = dict(gpu=gpu_info(), steps=args.steps, warmup=args.warmup, rounds=args.rounds,
               results=[run(name, dev, args) for name in args.workloads])
    line = json.dumps(out)
    print(line)
    if args.out:
        pathlib.Path(args.out).write_text(line + '\n')


if __name__ == '__main__':
    main()
