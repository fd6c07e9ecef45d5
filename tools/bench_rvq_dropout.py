"""Quantizer dropout (ResidualVectorQuantizer(quantizer_dropout=p)) and depth-truncated codes against what a user builds
without them.

    python tools/bench_rvq_dropout.py [--steps 30] [--warmup 5] [--rounds 3] [--out FILE]

Training step = forward + backward of the quantizer on NCHW latents, for the three workloads of tools/bench_rvq.py and
three paths:
  a  quantizer_dropout=0.5 through tokenizer.quantize: the depth draw (per image), one assignment + one
     vqb_residual_step_depth launch per level, ONE vqb_residual_backward_depth launch for all levels;
  b  the same module with p = 0: today's step, so a - b is the cost of the draw and the mask;
  c  DAC-style eager glue over L VectorQuantizer modules on the same depths: per level `vq.encode(r)` (callbacks run),
     e = F.embedding(q, W), the masked codebook / commitment terms, r = r - e.detach(), zhat += mask * e.detach(), then
     x + (zhat - x).detach() (the module's one straight-through estimator).
Kernel: ops.residual_backward alone with per-image depths (half the images truncated) against the same call without.
Codes: tokenizer.encode_to_quant (compact ids) and decode_from_quant at n = L/2 against n = L, eval mode.
Timing as in tools/bench_rvq.py: CUDA events around `steps` back-to-back calls after `warmup` calls, `rounds` rounds
with the paths alternating, the median round reported; inputs rotate over enough seeded sets to exceed the 126 MB L2.
Before timing, a and c run from the same codebooks on the same input and depths, and their indices, z and gx are
compared.  Prints one JSON line (also written to --out) with the GPU name, power limit and max SM clock of the same
run."""
from __future__ import annotations

import argparse
import json
import pathlib
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tools'))

import bench_rvq as B  # noqa: E402
import vector_quantization_b200 as vqb  # noqa: E402
from vector_quantization_b200 import ops, tokenizer  # noqa: E402

P = 0.5


def build(name, dev):
    b, D, h, w, K, L, dist, cvq, losses = B.WORKLOADS[name]
    g = torch.Generator().manual_seed(7)
    Ws = [torch.randn(K, D, generator=g) * 0.6 ** l for l in range(L)]
    mods = [vqb.build_quantizer(dict(type='ResidualVectorQuantizer', num_quantizers=L, quantizer_dropout=p,
                                     quantizer=B.level_config(name)), training=True).to(dev) for p in (P, 0.0)]
    chain = [vqb.build_quantizer(B.level_config(name), training=True).to(dev) for _ in range(L)]
    with torch.no_grad():
        for l, W in enumerate(Ws):
            for m in mods:
                m.quantizers[l].embedding.weight.copy_(W)
            chain[l].embedding.weight.copy_(W)
    size = b * D * h * w * 4
    sets = max(2, -(-2 * B.L2_BYTES // size))
    xs = [torch.randn(b, D, h, w, generator=g).to(dev) for _ in range(sets)]
    gz = torch.randn(b, D, h, w, generator=g).to(dev)
    return mods, chain, xs, gz


def step_module(q, x, gz):
    z, loss, memo = tokenizer.quantize(q, x, dict())
    torch.autograd.backward((z, loss), (gz, torch.ones_like(loss)))
    return z, memo['quantizer']


def step_glue(chain, depth, x, gz):
    """DAC-style dropout glue with the module's semantics (one straight-through estimator, VQGANLoss terms masked)."""
    b, c, h, w = x.shape
    rows = x.permute(0, 2, 3, 1).reshape(-1, c)
    N = rows.shape[0]
    tok = depth.repeat_interleave(h * w)
    r, zhat, loss, quants = rows, None, None, []
    for l, vq in enumerate(chain):
        _, q, _ = vq.encode(r.detach(), dict())
        quants.append(q)
        m = (tok > l).unsqueeze(1).to(r.dtype)
        e = F.embedding(q, vq.embedding.weight)
        loss_l = ((e - r.detach()) ** 2 * m).sum() / (N * c) + 0.25 * ((e.detach() - r) ** 2 * m).sum() / (N * c)
        r = r - e.detach()
        zhat = e.detach() if zhat is None else zhat + m * e.detach()
        loss = loss_l if loss is None else loss + loss_l
    z = rows + (zhat - rows).detach()
    z = z.view(b, h, w, c).permute(0, 3, 1, 2).contiguous()
    torch.autograd.backward((z, loss), (gz, torch.ones_like(loss)))
    return z, torch.stack(quants, 1)


def compare(name, dev) -> dict:
    """a against c from the same codebooks, input and depths (before any codebook update)."""
    b, D, h, w, K, L, *_ = B.WORKLOADS[name]
    (qa, _), chain, xs, gz = build(name, dev)
    torch.manual_seed(11)
    depth = qa.draw_depths(b, dev)
    qa.draw_depths = lambda samples, device: depth
    xa = xs[0].clone().requires_grad_(True)
    xc = xs[0].clone().requires_grad_(True)
    za, memo = step_module(qa, xa, gz)
    zc, quant_c = step_glue(chain, depth, xc, gz)
    same = (memo['quant'] == quant_c).all(1)
    tok = lambda t: t.permute(0, 2, 3, 1).reshape(-1, D)[same]      # noqa: E731
    rel = lambda p, q: float((p - q).abs().max() / q.abs().max())    # noqa: E731
    rec = dict(rows_all_levels_equal=float(same.float().mean()), truncated_images=int((depth < L).sum()),
               z_rel_max_diff=rel(tok(za), tok(zc)), gx_rel_max_diff=rel(tok(xa.grad), tok(xc.grad)))
    assert rec['rows_all_levels_equal'] > 0.99 and rec['z_rel_max_diff'] <= 1e-5 and rec['gx_rel_max_diff'] <= 1e-4, rec
    return rec


def run(name, dev, args) -> dict:
    b, D, h, w, K, L, dist, cvq, _ = B.WORKLOADS[name]
    rec = dict(workload=name, b=b, D=D, h=h, w=w, K=K, L=L, distance=dist, cvq=cvq, p=P, a_vs_c=compare(name, dev))
    (qa, qb), chain, xs, gz = build(name, dev)
    rec['input_sets'] = len(xs)
    inputs = [x.requires_grad_(True) for x in xs]
    paths = {'a': lambda x: step_module(qa, x, gz), 'b': lambda x: step_module(qb, x, gz),
             'c': lambda x: step_glue(chain, qa.draw_depths(b, dev), x, gz)}
    times = {k: [] for k in paths}
    for _ in range(args.rounds):
        for k, fn in paths.items():
            times[k].append(B.timed(fn, inputs, args.steps, args.warmup))
    rec['train_step_ms'] = {k: statistics.median(v) for k, v in times.items()}
    rec['train_step_ms_rounds'] = times

    # the backward kernel alone, masked against unmasked
    N = b * h * w
    g = torch.Generator().manual_seed(3)
    Ws = [lv.embedding.weight.detach() for lv in qa.quantizers]
    quant = torch.randint(0, K, (N, L), generator=g).to(dev)
    depth = torch.where(torch.arange(b) < b // 2, torch.randint(1, L + 1, (b,), generator=g), L).to(torch.int32).to(dev)
    g4s = [[torch.tensor(1.0, device=dev), torch.tensor(0.25, device=dev), None, None] for _ in range(L)]
    rows = [x.detach().permute(0, 2, 3, 1).reshape(-1, D).contiguous() for x in xs]
    gzr = gz.permute(0, 2, 3, 1).reshape(-1, D).contiguous()
    bwd = {'masked': lambda x: ops.residual_backward(gzr, x, Ws, quant, g4s, want_norm=False, need_gW=[True] * L,
                                                     depth=depth, depth_hw=h * w),
           'unmasked': lambda x: ops.residual_backward(gzr, x, Ws, quant, g4s, want_norm=False, need_gW=[True] * L)}
    kt = {k: [] for k in bwd}
    for _ in range(args.rounds):
        for k, fn in bwd.items():
            kt[k].append(1000 * B.timed(fn, rows, args.steps * 4, args.warmup))
    rec['backward_call_us'] = {k: statistics.median(v) for k, v in kt.items()}

    # truncated codes, eval mode
    qa.eval()
    n = max(1, L // 2)
    enc = {f'n={m}': (lambda x, m=m: tokenizer.encode_to_quant(qa, x, dict(), compact=True, num_quantizers=m))
           for m in (n, L)}
    ids = {m: tokenizer.encode_to_quant(qa, xs[0], dict(), compact=True, num_quantizers=m)[0] for m in (n, L)}
    dec = {f'n={m}': (lambda _, m=m: tokenizer.decode_from_quant(qa, ids[m], dict(), check=False, num_quantizers=m))
           for m in (n, L)}
    with torch.no_grad():
        et = {k: [] for k in enc}
        dt = {k: [] for k in dec}
        for _ in range(args.rounds):
            for k, fn in enc.items():
                et[k].append(1000 * B.timed(fn, xs, args.steps, args.warmup))
            for k, fn in dec.items():
                dt[k].append(1000 * B.timed(fn, xs, args.steps * 4, args.warmup))
    rec['encode_to_quant_us'] = {k: statistics.median(v) for k, v in et.items()}
    rec['decode_from_quant_us'] = {k: statistics.median(v) for k, v in dt.items()}
    return rec


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', type=str, default=None)
    ap.add_argument('--workloads', nargs='*', default=list(B.WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_rvq_dropout.py measures on a CUDA device; none is available')
    dev = torch.device('cuda', 0)
    out = dict(gpu=B.gpu_info(), steps=args.steps, warmup=args.warmup, rounds=args.rounds,
               results=[run(name, dev, args) for name in args.workloads])
    line = json.dumps(out)
    print(line)
    if args.out:
        pathlib.Path(args.out).write_text(line + '\n')


if __name__ == '__main__':
    main()
