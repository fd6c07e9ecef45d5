"""Token ids -> NCHW decoder input (tokenizer.decode_from_quant) against the routes a user has without it.

    python tools/bench_decode.py [--steps 200] [--rounds 5] [--out FILE]

For each workload (user-sized token grids, see WORKLOADS) and each output dtype (fp32, bf16) it times
  a          decode_from_quant(check=False): one vqb_decode_tokens / vqb_fsq_decode_tokens launch;
  a_checked  decode_from_quant(check=True): the same plus the 4-byte read-back of the bad-id count;
  b          the previous route: quantizer.decode(ids widened) + functional.rows_to_nchw (+ .to(bf16));
  c          stock torch: F.embedding(ids.long(), W).permute(0, 3, 1, 2).contiguous() (+ .to(bf16)); for FSQ, W is
             the implicit codebook table.
Timing: CUDA events around `steps` back-to-back calls after a warm-up, `rounds` rounds with the paths alternating,
median reported.  The ids rotate over sets, and each output is kept alive for one rotation, so ids and outputs
together exceed the 126 MB L2; the codebook itself stays resident where it fits (it does in use: every call reads
it).  The outputs of a, b and c are compared bit for bit on every timed id set before timing.
Bytes per call = ids + output + codebook rows touched (expected distinct codes of uniform ids x D x 4; none for
FSQ), computed from the shapes; GB/s is given also as a share of the 6548 GB/s copy bandwidth of DESIGN.md §7.
Prints one JSON line (also written to --out) with the GPU name, power limit and max SM clock of the same run."""
from __future__ import annotations

import argparse
import json
import pathlib
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import vector_quantization_b200 as vqb  # noqa: E402
from vector_quantization_b200 import functional as Fq  # noqa: E402
from vector_quantization_b200 import tokenizer  # noqa: E402

L2_BYTES = 126 << 20
COPY_GBPS = 6548.0          # measured B200 copy bandwidth, DESIGN.md §7
WORKLOADS = {               # name: (b, D, h, w, K or FSQ levels, id dtype)
    'vqgan_cvqvae': (64, 256, 16, 16, 8192, torch.uint16),
    'vqkd': (256, 32, 16, 16, 8192, torch.uint16),
    'llamagen_384px': (256, 8, 24, 24, 16384, torch.uint16),
    'cluster': (64, 768, 16, 16, 262144, torch.int32),
    'fsq_64000': (256, 6, 16, 16, [8, 8, 8, 5, 5, 5], torch.int32),
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


def build(name: str, dev):
    b, D, h, w, book, id_dtype = WORKLOADS[name]
    if isinstance(book, list):
        q = vqb.build_quantizer(dict(type='FiniteScalarQuantizer', num_scalars_per_channel=book)).to(dev)
        W = q.embeddings.float().contiguous()               # the implicit codebook table, for path c
    else:
        q = vqb.build_quantizer(dict(type='VectorQuantizer', distance=dict(type='L2Distance'),
                                     embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=book,
                                                    embedding_dim=D))).to(dev)
        q.requires_grad_(False)
        W = q.embedding.weight
    return q, W, (b, D, h, w), id_dtype


def paths(q, W, shape, out_dtype):
    b, D, h, w = shape
    fsq = isinstance(q, vqb.FiniteScalarQuantizer)

    def a(ids):
        return tokenizer.decode_from_quant(q, ids, dict(), dtype=out_dtype, check=False)[0]

    def a_checked(ids):
        return tokenizer.decode_from_quant(q, ids, dict(), dtype=out_dtype)[0]

    def b_(ids):
        z, _ = q.decode(ids.int() if fsq else ids.long(), dict())
        z = Fq.rows_to_nchw(z, b, D, h, w)
        return z if out_dtype == torch.float32 else z.to(out_dtype)

    def c(ids):
        z = F.embedding(ids.long(), W).permute(0, 3, 1, 2).contiguous()
        return z if out_dtype == torch.float32 else z.to(out_dtype)
    return dict(a=a, a_checked=a_checked, b=b_, c=c)


def time_path(fn, sets, ring, steps: int) -> float:
    """us per call: CUDA events around `steps` calls rotating over the id sets, each output held for one rotation."""
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(steps):
        ring[i % len(ring)] = fn(sets[i % len(sets)])
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1e3 / steps


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_decode.py measures on a CUDA device; none found')
    dev = torch.device('cuda', 0)
    result = dict(gpu=gpu_info(), steps=args.steps, rounds=args.rounds, l2_bytes=L2_BYTES, copy_gbps=COPY_GBPS,
                  workloads={})
    with torch.no_grad():
        for name in WORKLOADS:
            q, W, shape, id_dtype = build(name, dev)
            b, D, h, w = shape
            K = W.shape[0]
            N = b * h * w
            id_bytes = torch.empty(0, dtype=id_dtype).element_size()
            g = torch.Generator().manual_seed(0)
            for out_dtype in (torch.float32, torch.bfloat16):
                out_bytes = N * D * torch.empty(0, dtype=out_dtype).element_size()
                n_sets = max(2, -(-2 * L2_BYTES // (out_bytes + N * id_bytes)))
                sets = [torch.randint(0, K, (b, h, w), generator=g).to(torch.int32).to(id_dtype).to(dev)
                        for _ in range(n_sets)]
                fns = paths(q, W, shape, out_dtype)
                for ids in sets:
                    outs = {k: f(ids) for k, f in fns.items()}
                    for k, z in outs.items():
                        if not torch.equal(z, outs['a']):
                            raise SystemExit(f'{name} {out_dtype}: path {k} differs from path a')
                ring = [None] * n_sets
                for f in fns.values():                                 # warm-up
                    time_path(f, sets, ring, n_sets)
                times = {k: [] for k in fns}
                for _ in range(args.rounds):
                    for k, f in fns.items():
                        times[k].append(time_path(f, sets, ring, args.steps))
                ring.clear()
                distinct = 0 if isinstance(q, vqb.FiniteScalarQuantizer) else K * (1 - (1 - 1 / K) ** N)
                moved = N * id_bytes + out_bytes + distinct * D * 4
                rec = dict(b=b, D=D, h=h, w=w, K=K, ids=str(id_dtype)[6:], out=str(out_dtype)[6:], id_sets=n_sets,
                           bytes_per_call=int(moved), codebook_mb=round(K * D * 4 / 2 ** 20, 1),
                           codebook_fits_l2=K * D * 4 < L2_BYTES, outputs_equal=True)
                for k, ts in times.items():
                    us = statistics.median(ts)
                    gbps = moved / us / 1e3
                    rec[k] = dict(us=round(us, 2), spread_us=[round(min(ts), 2), round(max(ts), 2)],
                                  gbps=round(gbps, 1), share_of_copy_bw=round(gbps / COPY_GBPS, 3))
                rec['speedup_a_over_b'] = round(rec['b']['us'] / rec['a']['us'], 2)
                rec['speedup_a_over_c'] = round(rec['c']['us'] / rec['a']['us'], 2)
                result['workloads'][f'{name}/{str(out_dtype)[6:]}'] = rec
                print(json.dumps({f'{name}/{str(out_dtype)[6:]}': rec}), file=sys.stderr)
            del q, W
            torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(args.out).write_text(line + '\n')


if __name__ == '__main__':
    main()
