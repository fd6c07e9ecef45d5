"""The CPU oracle against the golden vectors generated from the reference's own source
(tests/golden/*.pt <- oracle/make_golden.py).  On the machine that generated them the agreement is
bit-for-bit (asserted by make_golden.py itself and by test_oracle_vs_reference.py); on another CPU, BLAS
kernels may differ in the last bit, so this test uses the documented tolerances and the near-tie rule."""
import pathlib

import pytest
import torch

from oracle import oracle as O

GOLDEN = pathlib.Path(__file__).parent / 'golden'
CASES = ['vqgan_l2', 'llamagen_l2norm', 'vqkd_train', 'vqkd_eval', 'cvqvae_train', 'llamagen_cvq_train', 'cluster_train']


@pytest.mark.parametrize('name', CASES)
def test_oracle_matches_golden(name):
    rec = torch.load(GOLDEN / f'{name}.pt', weights_only=False)
    spec = O.QuantizerSpec(**rec['spec'])
    for step in rec['steps']:
        x = step['x'].clone().requires_grad_(True)
        out = O.quantizer_forward(spec, [x], step['W_before'], step['prob_before'])
        (out['loss'][0] + (out['z_ste'][0] * step['gz']).sum()).backward()
        diff = out['quant'][0] != step['quant']
        assert (step['top2_gap'][diff] < 1e-5).all() and diff.float().mean() < 0.01
        same = ~diff
        torch.testing.assert_close(out['z_ste'][0].detach()[same], step['z'][same], rtol=1e-6, atol=1e-7)
        torch.testing.assert_close(out['loss'][0].detach(), step['loss'], rtol=1e-5, atol=1e-8)
        if not diff.any():
            torch.testing.assert_close(out['weight'], step['W_after'], rtol=1e-5, atol=1e-7)
            torch.testing.assert_close(x.grad, step['x_grad'], rtol=1e-4, atol=1e-7)
            if step['prob_after'] is not None:
                torch.testing.assert_close(out['prob'], step['prob_after'], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize('name', ['fsq_8000', 'fsq_64000'])
def test_fsq_oracle_matches_golden(name):
    rec = torch.load(GOLDEN / f'{name}.pt', weights_only=False)
    fsq = O.FSQ(rec['levels'])
    assert fsq.codebook_size == rec['codebook_size']
    quant, zq, pre = fsq.encode(rec['x'])
    safe = ((rec['pre'] - rec['pre'].floor() - 0.5).abs() > 1e-5).all(1)
    assert torch.equal(quant[safe], rec['quant'][safe]) and torch.equal(zq[safe], rec['z'][safe])
    assert torch.equal(fsq.decode(rec['quant'])[safe], rec['decode'][safe])
    assert int(quant.max()) < fsq.codebook_size and quant.dtype == torch.int32


def test_oracle_multi_rank_statistics_are_rank_order_invariant():
    """Token-sharded semantics: summing per-rank statistics == the single-process statistics."""
    x, E = O.synthetic_latents(1024, 64, 16, normalized_codebook=True)
    q, _ = O.encode('Cosine', x, E)
    one = O.vqkd_update([x], [q], E, 0.99)
    two = O.vqkd_update([x[:512], x[512:]], [q[:512], q[512:]], E, 0.99)
    torch.testing.assert_close(one, two, rtol=1e-5, atol=1e-7)
    assert torch.equal(O.bin_count([q], 64), O.bin_count([q[:300], q[300:]], 64))


def test_usage_metrics_known_answers():
    counts = torch.tensor([4, 0, 4, 0])
    assert O.codebook_usage(counts) == 0.5
    assert abs(O.codebook_ppl(counts) - 0.6931471805599453) < 1e-6   # entropy in nats, not exp


@pytest.mark.parametrize('tag', ['seeds', 'iters10', 'small'])
def test_oracle_kmeans_lazy_init_matches_golden(tag):
    """`O.vqkd_lazy_init` vs the golden written by the reference's own `lazy_init_weights` (same `random` seed)."""
    import random
    rec = torch.load(GOLDEN / f'vqkd_lazy_init_{tag}.pt', weights_only=False)
    random.seed(rec['seed'])
    W = O.vqkd_lazy_init(rec['x'], rec['W0'], rec['iters'])
    close = torch.isclose(W, rec['W_init'], rtol=1e-5, atol=1e-6).all(1)
    assert close.float().mean() >= (0.95 if tag == 'iters10' else 1.0)


@pytest.mark.parametrize('N,K', [(200, 64), (64, 64), (40, 64)])
def test_cached_anchor_sampling_rule_matches_golden(N, K):
    """`cached_rows_and_indices` (the product's CachedAnchor rule) against the stored anchors of the reference's
    CachedAnchor under the same seeds, bit for bit, over three consecutive steps (cache top-up) for N > K, N == K and
    N < K."""
    import random
    from vector_quantization_b200.anchors import cached_rows_and_indices
    rec = torch.load(GOLDEN / 'anchors_entropy.pt', weights_only=False)['cached_anchor'][(N, K)]
    cache = torch.empty(0)
    for step, (x, want) in enumerate(zip(rec['x'], rec['anchors'])):
        torch.manual_seed(100 + step); random.seed(100 + step)
        rows, idx = cached_rows_and_indices(x, K, cache)
        cache = rows[idx]
        assert torch.equal(cache, want), step


def test_entropy_loss_and_multinomial_anchor_match_golden():
    """`O.entropy_loss` and `O.multinomial_anchor` (the oracle of the compat-mode GPU tests) against the stored outputs
    of the reference's EntropyLoss and MultinomialAnchor on the stored distance matrix.  The anchors are compared bit
    for bit under the same torch seed; the entropy to fp32 rounding, since its softmax/log reductions may be summed in
    a different order on another CPU."""
    rec = torch.load(GOLDEN / 'anchors_entropy.pt', weights_only=False)
    x, d = rec['x'], rec['d']
    torch.testing.assert_close(O.entropy_loss(d, rec['temperature']), rec['entropy'], rtol=1e-6, atol=1e-7)
    torch.manual_seed(rec['multinomial_seed'])
    anchors, _ = O.multinomial_anchor(x, d)
    assert torch.equal(anchors, rec['multinomial_anchors'])
