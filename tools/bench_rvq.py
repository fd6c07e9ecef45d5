"""Residual quantization (ResidualVectorQuantizer) against what a user builds without it.

    python tools/bench_rvq.py [--steps 30] [--warmup 5] [--rounds 3] [--out FILE]

Training step = forward + backward of the quantizer on NCHW latents, for three workloads (WORKLOADS) and three paths:
  a  the new module through tokenizer.quantize: one transposed copy in, one assignment + one residual-step launch per
     level, z written NCHW by the last step, ONE backward launch for all levels;
  b  L chained VectorQuantizer modules through eager glue, as users write it today: permute in, per level
     `z_l, loss_l = vq_l(r)`, `r = r - z_l.detach()`, `zhat = zhat + z_l`, then `x + (zhat - x).detach()`, permute
     out; L autograd nodes in the backward;
  c  stock eager torch: per level torch.cdist / the cosine matmul, argmin, F.embedding, F.mse_loss terms and the
     same glue (no codebook update: the CVQ-VAE re-initialisation of workload 2 is not part of this path).
Decode: tokenizer.decode_from_quant on [b, h, w, L] ids against L x F.embedding + sum + permute().contiguous().
Timing: CUDA events around `steps` back-to-back calls after `warmup` calls, `rounds` rounds with the paths
alternating, the median round reported.  Inputs rotate over enough seeded sets to exceed the 126 MB L2.
Before timing, a and b run from the same codebooks on the same input and their indices and z are compared
(b's z_l is each level's straight-through output r + (e - r), not e, so z may differ in the last bits).
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
WORKLOADS = {   # name: (b, D, h, w, K, L, distance, CVQ-VAE callback, losses)
    'rqvae_like': (256, 256, 8, 8, 16384, 4, 'L2', False, dict(vqgan_loss=dict(type='VQGANLoss'))),
    'vqgan_grid_cvq': (64, 256, 16, 16, 8192, 4, 'Cosine', True, dict(vqgan_loss=dict(type='VQGANLoss'))),
    'small_d': (256, 8, 16, 16, 16384, 8, 'L2', False, dict(vqgan_loss=dict(type='VQGANLoss'))),
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


def level_config(name):
    b, D, h, w, K, L, dist, cvq, losses = WORKLOADS[name]
    callbacks = [dict(type='CVQVAECallback', anchor=dict(type='NearestAnchor'), ema=dict())] if cvq else []
    return dict(type='VQGANQuantizer', distance=dict(type=f'{dist}Distance'), callbacks=callbacks, losses=losses,
                embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D))


def build(name, dev):
    b, D, h, w, K, L, dist, cvq, losses = WORKLOADS[name]
    g = torch.Generator().manual_seed(7)
    Ws = [torch.randn(K, D, generator=g) * 0.6 ** l for l in range(L)]
    rvq = vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=L, quantizer=level_config(name)),
                              training=True).to(dev)
    chain = [vqb.build_quantizer(level_config(name), training=True).to(dev) for _ in range(L)]
    stock = [torch.nn.Parameter(W.to(dev)) for W in Ws]
    with torch.no_grad():
        for l, W in enumerate(Ws):
            rvq.quantizers[l].embedding.weight.copy_(W)
            chain[l].embedding.weight.copy_(W)
    size = b * D * h * w * 4
    sets = max(2, math.ceil(2 * L2_BYTES / size))
    xs = [torch.randn(b, D, h, w, generator=g).to(dev) for _ in range(sets)]
    gz = torch.randn(b, D, h, w, generator=g).to(dev)
    return rvq, chain, stock, xs, gz


def step_a(rvq, x, gz):
    z, loss, memo = tokenizer.quantize(rvq, x, dict())
    torch.autograd.backward((z, loss), (gz, torch.ones_like(loss)))
    return z, memo['quantizer']['quant']


def step_b(chain, x, gz):
    b, c, h, w = x.shape
    rows = x.permute(0, 2, 3, 1).reshape(-1, c)
    r, zhat, loss, quants = rows, None, None, []
    for vq in chain:
        z_l, loss_l, memo = vq(r, dict())
        quants.append(memo['quant'])
        r = r - z_l.detach()
        zhat = z_l if zhat is None else zhat + z_l
        loss = loss_l if loss is None else loss + loss_l
    z = rows + (zhat - rows).detach()
    z = z.view(b, h, w, c).permute(0, 3, 1, 2).contiguous()
    torch.autograd.backward((z, loss), (gz, torch.ones_like(loss)))
    return z, torch.stack(quants, 1)


def step_c(stock, metric, x, gz):
    b, c, h, w = x.shape
    rows = x.permute(0, 2, 3, 1).reshape(-1, c)
    r, zhat, loss = rows, None, None
    for W in stock:
        with torch.no_grad():
            if metric == 'L2':
                q = torch.cdist(r, W).argmin(1)
            else:
                q = (1 - F.normalize(r) @ F.normalize(W).T).argmin(1)
        e = F.embedding(q, W)
        loss_l = F.mse_loss(e, r.detach()) + 0.25 * F.mse_loss(e.detach(), r)
        r = r - e.detach()
        zhat = e if zhat is None else zhat + e
        loss = loss_l if loss is None else loss + loss_l
    z = rows + (zhat - rows).detach()
    z = z.view(b, h, w, c).permute(0, 3, 1, 2).contiguous()
    torch.autograd.backward((z, loss), (gz, torch.ones_like(loss)))
    return z


def decode_a(rvq, ids):
    return tokenizer.decode_from_quant(rvq, ids, dict(), check=False)[0]


def decode_c(Ws, ids):
    z = None
    for l, W in enumerate(Ws):
        e = F.embedding(ids[..., l], W)
        z = e if z is None else z + e
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
    b, D, h, w, K, L, dist, cvq, _ = WORKLOADS[name]
    rvq, chain, stock, xs, gz = build(name, dev)
    rec = dict(workload=name, b=b, D=D, h=h, w=w, K=K, L=L, distance=dist, cvq=cvq, input_sets=len(xs))
    # same codebooks, same input: compare before any codebook update
    xa = xs[0].clone().requires_grad_(True)
    xb = xs[0].clone().requires_grad_(True)
    za, qa = step_a(rvq, xa, gz)
    zb, qb = step_b(chain, xb, gz)
    same = (qa == qb).all(1)
    rec['a_vs_b'] = dict(rows_all_levels_equal=float(same.float().mean()),
                         level_index_agreement=[float(v) for v in (qa == qb).float().mean(0)],
                         z_max_abs_diff_on_equal_rows=float((za - zb).permute(0, 2, 3, 1).reshape(-1, D)[same].abs().max()),
                         z_bitwise_equal_rows=float((za == zb).permute(0, 2, 3, 1).reshape(-1, D).all(1).float().mean()))
    inputs = [x.requires_grad_(True) for x in xs]
    paths = {'a': lambda x: step_a(rvq, x, gz), 'b': lambda x: step_b(chain, x, gz),
             'c': lambda x: step_c(stock, dist, x, gz)}
    times = {k: [] for k in paths}
    for _ in range(args.rounds):
        for k, fn in paths.items():
            times[k].append(timed(fn, inputs, args.steps, args.warmup))
    rec['train_step_ms'] = {k: statistics.median(v) for k, v in times.items()}
    rec['train_step_ms_rounds'] = times
    # decode
    ids = [torch.randint(0, K, (b, h, w, L), generator=torch.Generator().manual_seed(i)).to(dev)
           for i in range(max(2, math.ceil(2 * L2_BYTES / (b * D * h * w * 4))))]
    Ws = [lv.embedding.weight.detach() for lv in rvq.quantizers]
    with torch.no_grad():
        assert torch.equal(decode_a(rvq, ids[0]), decode_c(Ws, ids[0]))
        dec = {'a': [], 'c': []}
        for _ in range(args.rounds):
            dec['a'].append(timed(lambda i: decode_a(rvq, i), ids, args.steps * 4, args.warmup))
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
        raise SystemExit('bench_rvq.py measures on a CUDA device; none is available')
    dev = torch.device('cuda', 0)
    out = dict(gpu=gpu_info(), steps=args.steps, warmup=args.warmup, rounds=args.rounds,
               results=[run(name, dev, args) for name in args.workloads])
    line = json.dumps(out)
    print(line)
    if args.out:
        pathlib.Path(args.out).write_text(line + '\n')


if __name__ == '__main__':
    main()
