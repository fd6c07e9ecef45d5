"""Generate the golden vectors under tests/golden/ by running the reference's OWN quantizer source
files (imported unmodified from /root/reference, see oracle/ref_loader.py) on seeded synthetic latents,
and pin the oracle restatement (oracle/oracle.py) against them BIT FOR BIT on this CPU.

Run in the dev container only:   python -m oracle.make_golden
The reference has no tests/golden vectors of its own (SURVEY.md §4); these fixtures are the pinning.
What stays unpinned: the todd-side arithmetic (`EMA`, `MSELoss`), which the shim restates.
"""
from __future__ import annotations

import pathlib
import random
import sys

import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import oracle as O  # noqa: E402
from oracle import ref_loader as R  # noqa: E402

OUT = ROOT / 'tests' / 'golden'
SEED = 3407  # the reference's default seed, vq/train.py:21


def emb(K, D):
    return dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=K, embedding_dim=D)


# name -> (reference quantizer config, oracle spec, N, K, D, normalized codebook, steps, training)
CASES = {
    # configs/vqgan/model.py:19-23 (+ configs/vq/*): VQGANQuantizer, L2, VQGANLoss
    'vqgan_l2': (dict(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                      losses=dict(vqgan_loss=dict(type='VQGANLoss')), init_weights=dict(type='vqgan')),
                 O.QuantizerSpec(distance='L2', losses={'vqgan_loss': dict(type='VQGANLoss')}),
                 512, 256, 16, False, 1, True),
    # configs/llamagen/vqgan.py:18-20: + NormalizeCallback, D=8
    'llamagen_l2norm': (dict(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                             callbacks=[dict(type='NormalizeCallback')],
                             losses=dict(vqgan_loss=dict(type='VQGANLoss')), init_weights=dict(type='vqgan')),
                        O.QuantizerSpec(distance='L2', callback='NormalizeCallback',
                                        losses={'vqgan_loss': dict(type='VQGANLoss')}),
                        512, 256, 8, False, 1, True),
    # configs/vqkd/model.py:20-26: VQKDQuantizer, Cosine, VQKDCallback(ema), CommitmentLoss(norm=True)
    'vqkd_train': (dict(type='VQKDQuantizer', distance=dict(type='CosineDistance'),
                        callbacks=[dict(type='VQKDCallback', ema=dict())],
                        losses=dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True)))),
                   O.QuantizerSpec(distance='Cosine', callback='VQKDCallback',
                                   losses={'commitment_loss': dict(type='CommitmentLoss', norm=True)}),
                   1024, 128, 32, True, 3, True),
    'vqkd_eval': (dict(type='VQKDQuantizer', distance=dict(type='CosineDistance'),
                       callbacks=[dict(type='VQKDCallback', ema=dict())],
                       losses=dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True)))),
                  O.QuantizerSpec(distance='Cosine', callback='VQKDCallback', training=False,
                                  losses={'commitment_loss': dict(type='CommitmentLoss', norm=True)}),
                  512, 128, 32, True, 1, False),
    # configs/cvqvae/quantizer.py:1-6 on the VQGAN quantizer with Cosine distance
    'cvqvae_train': (dict(type='VQGANQuantizer', distance=dict(type='CosineDistance'),
                          callbacks=[dict(type='CVQVAECallback', ema=dict(), anchor=dict(type='NearestAnchor'))],
                          losses=dict(vqgan_loss=dict(type='VQGANLoss')), init_weights=dict(type='vqgan')),
                     O.QuantizerSpec(distance='Cosine', callback='CVQVAECallback',
                                     losses={'vqgan_loss': dict(type='VQGANLoss')}),
                     768, 128, 32, False, 3, True),
    # configs/cvqvae/quantizer.py (a mixin) layered on configs/llamagen/vqgan.py: NormalizeCallback + CVQVAECallback,
    # L2 on normalised tokens — anchors and the column arg-min must see F.normalize(x)
    'llamagen_cvq_train': (dict(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                                callbacks=[dict(type='NormalizeCallback'),
                                           dict(type='CVQVAECallback', ema=dict(), anchor=dict(type='NearestAnchor'))],
                                losses=dict(vqgan_loss=dict(type='VQGANLoss')), init_weights=dict(type='vqgan')),
                           O.QuantizerSpec(distance='L2', callback='CVQVAECallback', normalize=True,
                                           losses={'vqgan_loss': dict(type='VQGANLoss')}),
                           512, 128, 8, False, 2, True),
    # configs/cluster/model.py:20-31: CodebookLoss only, NearestAnchor(sync=True)
    'cluster_train': (dict(type='VQGANQuantizer', distance=dict(type='CosineDistance'),
                           callbacks=[dict(type='CVQVAECallback', ema=dict(),
                                           anchor=dict(type='NearestAnchor', sync=True))],
                           losses=dict(vqgan_loss=dict(type='CodebookLoss')), init_weights=dict(type='vqgan')),
                      O.QuantizerSpec(distance='Cosine', callback='CVQVAECallback', anchor_sync=True,
                                      losses={'vqgan_loss': dict(type='CodebookLoss')}),
                      512, 96, 64, False, 2, True),
}


# the k-means lazy init (vqkd/quantizers/callbacks.py:77-112): seeds only, full 10 rounds, fewer tokens than codes
LAZY_INIT = {'seeds': (2048, 64, 16, 0), 'iters10': (2048, 64, 16, 10), 'small': (40, 64, 16, 10)}


def run_case(name, ref_cfg, spec, N, K, D, normalized, steps, training):
    g = torch.Generator().manual_seed(SEED)
    x_all, E0 = O.synthetic_latents(N * steps, K, D, seed=SEED, normalized_codebook=normalized)
    cfg = dict(ref_cfg, embedding=emb(K, D))
    torch.manual_seed(SEED)
    random.seed(SEED)
    q = R.build_quantizer(cfg, training=training)
    q._forward_pre_hooks.clear()  # steady-state step: the one-off k-means lazy init is covered separately
    with torch.no_grad():
        q.embedding.weight.copy_(E0)
    W = E0.clone()
    prob = q.get_buffer('_probability').clone() if '_probability' in dict(q.named_buffers()) else None
    records = []
    for s in range(steps):
        x = x_all[s * N:(s + 1) * N].clone()
        gz = torch.randn(N, D, generator=g)
        # ---- reference ----
        xr = x.clone().requires_grad_(True)
        q.embedding.weight.grad = None
        z, loss, memo = q(xr, dict())
        (loss + (z * gz).sum()).backward()
        W_after = q.embedding.weight.detach().clone()
        wgrad = q.embedding.weight.grad
        rec = dict(x=x, gz=gz, W_before=W.clone(), prob_before=None if prob is None else prob.clone(),
                   z=z.detach().clone(), loss=loss.detach().clone(),
                   losses={k: v.detach().clone() for k, v in memo['loss'].items()},
                   quant=memo['quant'].clone(), x_norm=memo['x'].detach().clone(), x_grad=xr.grad.clone(),
                   W_after=W_after, W_grad=None if wgrad is None else wgrad.clone(),
                   prob_after=q.get_buffer('_probability').clone() if prob is not None else None)
        # ---- oracle restatement, same inputs ----
        xo = x.clone().requires_grad_(True)
        out = O.quantizer_forward(spec, [xo], W, prob)
        (out['loss'][0] + (out['z_ste'][0] * gz).sum()).backward()
        checks = dict(z=torch.equal(out['z_ste'][0], rec['z']), loss=torch.equal(out['loss'][0], rec['loss']),
                      quant=torch.equal(out['quant'][0], rec['quant']), W_after=torch.equal(out['weight'], W_after),
                      x_grad=torch.equal(xo.grad, rec['x_grad']),
                      W_grad=(wgrad is None and out['weight_leaf'].grad is None) or
                      torch.equal(out['weight_leaf'].grad, wgrad),
                      prob=prob is None or torch.equal(out['prob'], rec['prob_after']))
        assert all(checks.values()), f'{name} step {s}: oracle != reference source: {checks}'
        # near-tie analysis material for the GPU tests: the reference's own top-2 distance gap per row
        d = memo['encode']['distance'].detach()
        top2 = d.topk(2, dim=1, largest=False).values
        rec['top2_gap'] = (top2[:, 1] - top2[:, 0]).clone()
        rec['d_min'] = top2[:, 0].clone()
        records.append(rec)
        W = W_after.clone()
        prob = rec['prob_after']
    return dict(name=name, config=cfg, training=training, spec=spec.__dict__, N=N, K=K, D=D, steps=records,
                state_dict_keys=list(q.state_dict().keys()))


def run_fsq(levels):
    N = 1024
    g = torch.Generator().manual_seed(SEED)
    x = 1.5 * torch.randn(N, len(levels), generator=g)
    gz = torch.randn(N, len(levels), generator=g)
    q = R.build_quantizer(dict(type='FiniteScalarQuantizer', num_scalars_per_channel=levels), training=True)
    xr = x.clone().requires_grad_(True)
    z, loss, memo = q(xr, dict())
    (z * gz).sum().backward()
    fsq = O.FSQ(levels)
    xo = x.clone().requires_grad_(True)
    zq, l0, quant, pre = fsq.forward(xo)
    (zq * gz).sum().backward()
    assert torch.equal(zq, z) and torch.equal(quant, memo['quant']) and torch.equal(xo.grad, xr.grad)
    assert float(loss) == 0.0 and memo['quant'].dtype == torch.int32
    assert torch.equal(fsq.embeddings, q.embeddings)
    dec, _ = q.decode(memo['quant'], dict())           # decode-only branch (no 'z' in memo)
    assert torch.equal(dec, fsq.decode(quant))
    return dict(levels=levels, x=x, gz=gz, z=z.detach(), quant=memo['quant'], x_grad=xr.grad, pre=pre.detach(),
                decode=dec.detach(), codebook_size=q.codebook_size, state_dict_keys=list(q.state_dict().keys()))


def run_lazy_init(N, K, D, iters):
    """The one-off k-means codebook init of VQ-KD (first training forward), reference source vs `O.vqkd_lazy_init`,
    with the same `random` seed; then the first training step on the initialised codebook."""
    x, _ = O.synthetic_latents(N, K, D, seed=SEED + N, normalized_codebook=True)
    cfg = dict(type='VQKDQuantizer', embedding=emb(K, D), distance=dict(type='CosineDistance'),
               callbacks=[dict(type='VQKDCallback', ema=dict())],
               losses=dict(commitment_loss=dict(type='CommitmentLoss', mse=dict(norm=True))),
               init_weights=dict(before_init_weights=dict(lazy_init_weights=dict(iters=iters))))
    torch.manual_seed(SEED)
    q = R.build_quantizer(cfg, training=True)
    W0 = q.embedding.weight.detach().clone()
    seen = {}

    def record(module, args):        # runs after the callback's own pre-hook (registration order)
        seen.setdefault('W_init', module.embedding.weight.detach().clone())

    q.register_forward_pre_hook(record)
    random.seed(SEED)
    z, loss, memo = q(x.clone(), dict())
    random.seed(SEED)
    W_init = O.vqkd_lazy_init(x, W0, iters)
    assert torch.equal(W_init, seen['W_init']), 'oracle k-means init != reference source'
    spec = O.QuantizerSpec(distance='Cosine', callback='VQKDCallback',
                           losses={'commitment_loss': dict(type='CommitmentLoss', norm=True)})
    out = O.quantizer_forward(spec, [x], W_init)
    assert torch.equal(out['quant'][0], memo['quant']) and torch.equal(out['weight'], q.embedding.weight.detach())
    return dict(N=N, K=K, D=D, iters=iters, seed=SEED, config=cfg, x=x, W0=W0, W_init=seen['W_init'],
                quant=memo['quant'].clone(), W_after=q.embedding.weight.detach().clone(), loss=loss.detach().clone())


ANCHOR_GOLDEN = 'anchors_entropy.pt'
CACHED_ANCHOR_SHAPES = [(200, 64), (64, 64), (40, 64)]   # N > K, N == K, N < K (cache and noise top-up)


def run_anchor_cases(ref=None):
    """CachedAnchor over three consecutive steps per (N, K), EntropyLoss and MultinomialAnchor on seeded inputs: from
    the reference's own classes when `ref` (`ref_loader.load()`) is given, else from the restatements
    (`anchors.cached_rows_and_indices`, `O.entropy_loss`, `O.multinomial_anchor`) that
    tests/test_oracle_vs_reference.py pins to those classes bit for bit."""
    from vector_quantization_b200.anchors import cached_rows_and_indices
    D = 8
    cached = {}
    for N, K in CACHED_ANCHOR_SHAPES:
        g = torch.Generator().manual_seed(N)
        ref_anchor = ref.cvqvae.anchors.CachedAnchor() if ref is not None else None
        cache = torch.empty(0)
        xs, anchors = [], []
        for step in range(3):
            x = torch.randn(N, D, generator=g)
            torch.manual_seed(100 + step)
            random.seed(100 + step)
            if ref_anchor is not None:
                got, _ = ref_anchor(x, None, torch.zeros(N, K), None, torch.zeros(K))   # only d's shape is read
            else:
                rows, idx = cached_rows_and_indices(x, K, cache)
                got = rows[idx]
            cache = got
            xs.append(x)
            anchors.append(got.clone())
        cached[(N, K)] = dict(x=xs, anchors=anchors)
    x, E = O.synthetic_latents(96, 24, 8, seed=3)
    d = O.distance('L2', x, E)
    temperature = 0.7
    if ref is not None:
        entropy = ref.vq.losses.EntropyLoss(temperature=temperature)(None, None, dict(distance=d))
        torch.manual_seed(5)
        mn_anchors, _ = ref.cvqvae.anchors.MultinomialAnchor()(x, E, d, None, torch.zeros(24))
    else:
        entropy = O.entropy_loss(d, temperature)
        torch.manual_seed(5)
        mn_anchors, _ = O.multinomial_anchor(x, d)
    source = ('reference source' if ref is not None else
              'restatements pinned bit for bit to the reference source by tests/test_oracle_vs_reference.py')
    return dict(source=source, D=D, cached_anchor=cached, x=x, E=E, d=d, temperature=temperature,
                entropy=entropy.detach().clone(), multinomial_seed=5, multinomial_anchors=mn_anchors.clone())


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    ref = R.load()
    print(f'reference loaded from {R.REF} (todd shim: {ref.todd_is_shim})')
    for name, args in CASES.items():
        rec = run_case(name, *args)
        torch.save(rec, OUT / f'{name}.pt')
        print(f'{name}: oracle == reference source bit-for-bit over {len(rec["steps"])} step(s); '
              f'keys {rec["state_dict_keys"]}')
    for levels in ([8, 8, 5, 5, 5], [8, 8, 8, 5, 5, 5]):
        rec = run_fsq(levels)
        torch.save(rec, OUT / f'fsq_{rec["codebook_size"]}.pt')
        print(f'fsq_{rec["codebook_size"]}: oracle == reference source bit-for-bit')
    for tag, args in LAZY_INIT.items():
        rec = run_lazy_init(*args)
        torch.save(rec, OUT / f'vqkd_lazy_init_{tag}.pt')
        print(f'vqkd_lazy_init_{tag}: oracle == reference source bit-for-bit (N={args[0]} K={args[1]} iters={args[3]})')
    torch.save(run_anchor_cases(ref), OUT / ANCHOR_GOLDEN)
    print(f'{ANCHOR_GOLDEN}: written from the reference source')


if __name__ == '__main__':
    if sys.argv[1:] == ['anchors']:   # that file alone, from the pinned restatements when the reference is absent
        rec = run_anchor_cases(R.load() if R.available() else None)
        torch.save(rec, OUT / ANCHOR_GOLDEN)
        print(f'{ANCHOR_GOLDEN}: written from the {rec["source"]}')
    else:
        main()
