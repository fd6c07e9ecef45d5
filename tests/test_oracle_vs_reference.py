"""Dev-container only: the reference's OWN source files (imported unmodified from /root/reference under the
todd shim) vs the oracle restatement, bit for bit, and the committed golden files are reproducible."""
import pathlib

import pytest
import torch

from oracle import ref_loader

pytestmark = [pytest.mark.reference,
              pytest.mark.skipif(not ref_loader.available(), reason='/root/reference not present')]
GOLDEN = pathlib.Path(__file__).parent / 'golden'


def test_restatement_equals_reference_source_and_golden_is_reproducible():
    from oracle import make_golden as M
    for name, args in M.CASES.items():
        rec = M.run_case(name, *args)          # asserts oracle == reference inside
        disk = torch.load(GOLDEN / f'{name}.pt', weights_only=False)
        for a, b in zip(rec['steps'], disk['steps']):
            assert torch.equal(a['quant'], b['quant']) and torch.equal(a['z'], b['z'])
            assert torch.equal(a['W_after'], b['W_after']) and torch.equal(a['loss'], b['loss'])
    for levels in ([8, 8, 5, 5, 5], [8, 8, 8, 5, 5, 5]):
        M.run_fsq(levels)
    rec = M.run_anchor_cases(ref_loader.load())
    disk = torch.load(GOLDEN / M.ANCHOR_GOLDEN, weights_only=False)
    for key, case in rec['cached_anchor'].items():
        for a, b in zip(case['anchors'], disk['cached_anchor'][key]['anchors']):
            assert torch.equal(a, b), key
    assert torch.equal(rec['entropy'], disk['entropy'])
    assert torch.equal(rec['multinomial_anchors'], disk['multinomial_anchors'])


def test_plugin_force_registers_into_reference_registries():
    """The drop-in seam: after importing the plugin, the reference's registry builds OUR classes from a
    reference-style config (custom_imports mechanism, vq/train.py:36-37)."""
    ref = ref_loader.load()
    import importlib
    import vector_quantization_b200.plugin as plugin
    importlib.reload(plugin)
    assert plugin.registered_into_reference
    import vector_quantization_b200 as vqb
    cfg = ref.todd.Config(type='VQGANQuantizer', distance=dict(type='L2Distance'),
                          embedding=dict(type='torch_nn_modules_sparse_Embedding', num_embeddings=64, embedding_dim=8),
                          losses=dict(vqgan_loss=dict(type='VQGANLoss')))
    q = ref.VQITQuantizerRegistry.build(cfg)
    assert type(q) is vqb.VQGANQuantizer and type(q.distance) is vqb.L2Distance
    assert type(q._losses['vqgan_loss']) is vqb.VQGANLoss


@pytest.mark.parametrize('N,K', [(200, 64), (64, 64), (40, 64)])
def test_cached_anchor_sampling_rule_equals_reference_source(N, K):
    """CachedAnchor never reads the distance values: with equal seeds our sampling rule (rows + indices) yields the
    reference's anchors bit for bit, over consecutive steps (cache top-up) and for N > K, N == K and N < K."""
    import random
    ref = ref_loader.load()
    from vector_quantization_b200.anchors import cached_rows_and_indices
    D = 8
    g = torch.Generator().manual_seed(N)
    ref_anchor = ref.cvqvae.anchors.CachedAnchor()
    cache = torch.empty(0)
    for step in range(3):
        x = torch.randn(N, D, generator=g)
        d = torch.zeros(N, K)                       # only its shape is used (anchors.py:146-159)
        torch.manual_seed(100 + step); random.seed(100 + step)
        want, _ = ref_anchor(x, None, d, None, torch.zeros(K))
        torch.manual_seed(100 + step); random.seed(100 + step)
        rows, idx = cached_rows_and_indices(x, K, cache)
        got = rows[idx]
        assert torch.equal(got, want), step
        cache = got
        assert torch.equal(ref_anchor.cache, cache)


def test_entropy_loss_and_multinomial_anchor_restatements_equal_reference_source():
    """The compat-mode consumers of the distance matrix: `O.entropy_loss` vs the reference's EntropyLoss (which reads
    `memo['distance']` of the memo it is handed, losses.py:142) and `O.multinomial_anchor` vs MultinomialAnchor under
    the same torch seed."""
    from oracle import oracle as O
    ref = ref_loader.load()
    x, E = O.synthetic_latents(96, 24, 8, seed=3)
    d = O.distance('L2', x, E)
    want = ref.vq.losses.EntropyLoss(temperature=0.7)(None, None, dict(distance=d))
    assert torch.equal(O.entropy_loss(d, 0.7), want)
    anchor = ref.cvqvae.anchors.MultinomialAnchor()
    torch.manual_seed(5)
    a_ref, _ = anchor(x, E, d, None, torch.zeros(24))
    torch.manual_seed(5)
    a_or, _ = O.multinomial_anchor(x, d)
    assert torch.equal(a_ref, a_or)


def test_reference_vqgan_vqkd_callback_cannot_be_imported_upstream():
    """vq/algorithms/exp/vqgan_vqkd/quantizer_callback.py:38-42 declares
    `class VQGAN_VQKDCallback(LazyInitWeightsMixin, UpdateMixin, NormalizeCallback)`; NormalizeCallback already
    derives from UpdateMixin, so Python cannot linearise the bases: the module raises TypeError at import in the
    reference itself (experimental, not imported by any config).  Our VQGAN_VQKDCallback therefore follows the
    SOURCE TEXT (`O.vqgan_vqkd_update`); there is no executable upstream behaviour to pin against."""
    import importlib
    import sys
    import types
    from oracle import oracle as O
    ref_loader.load()
    for name, path in (('vq.algorithms.exp', 'vq/algorithms/exp'), ('vq.algorithms.exp.vqgan_vqkd', 'vq/algorithms/exp/vqgan_vqkd')):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = [str(ref_loader.REF / path)]
            sys.modules[name] = m
    with pytest.raises(TypeError, match='MRO'):
        importlib.import_module('vq.algorithms.exp.vqgan_vqkd.quantizer_callback')
    W = torch.randn(16, 8)
    out = O.vqgan_vqkd_update(W, 0.99)
    torch.testing.assert_close(out.norm(dim=1), torch.ones(16), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(out, torch.nn.functional.normalize(W * 0.99 + torch.nn.functional.normalize(W) * 0.01))
