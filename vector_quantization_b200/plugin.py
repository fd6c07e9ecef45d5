"""Drop-in seam.  List this module in a reference config's `custom_imports`
(configs/vqgan/custom_imports.py:1-3, consumed at vq/train.py:36-37) AFTER the reference's own imports:

    custom_imports = [..., 'vector_quantization_b200.plugin']

When the reference package (`vq`, which needs `todd`) is importable, every class below is force-registered
under the SAME name in the reference's own registries (`register_(force=True)`, the mechanism the reference
itself uses at tools/tokenize_llamagen.py:27,65), so existing configs build the B200 implementations
unchanged.  Without the reference, the standalone registries in `registry.py` serve the same names.
"""
from __future__ import annotations

from . import anchors, callbacks, distances, losses, quantizers, registry

QUANTIZERS = ['VectorQuantizer', 'VQGANQuantizer', 'VQKDQuantizer', 'ScalarQuantizer', 'FiniteScalarQuantizer',
              'ResidualVectorQuantizer', 'GroupedVectorQuantizer']
CALLBACKS = ['ComposedCallback', 'NormalizeCallback', 'VQKDCallback', 'VQGAN_VQKDCallback', 'CVQVAECallback']
LOSSES = ['CodebookLoss', 'CommitmentLoss', 'VQGANLoss', 'EntropyLoss']
DISTANCES = ['L2Distance', 'CosineDistance']
ANCHORS = ['NearestAnchor', 'MultinomialAnchor', 'CachedAnchor']

registered_into_reference = False


def register_into_reference() -> bool:
    """Force-register our classes into the reference registries if they can be imported."""
    global registered_into_reference
    try:
        from vq.algorithms.cvqvae.registries import AnchorRegistry as RefAnchor
        from vq.algorithms.vq.distances import VQITQuantizerDistanceRegistry as RefDistance
        from vq.tasks.image_tokenization.models import VQITQuantizerRegistry as RefQuantizer
        from vq.tasks.image_tokenization.models.quantizers import (
            VQITQuantizerCallbackRegistry as RefCallback, VQITQuantizerLossRegistry as RefLoss)
    except Exception:  # noqa: BLE001 - reference (or todd) not installed: standalone mode
        return False
    for names, module, ref, ours in (
            (QUANTIZERS, quantizers, RefQuantizer, registry.VQITQuantizerRegistry),
            (CALLBACKS, callbacks, RefCallback, registry.VQITQuantizerCallbackRegistry),
            (LOSSES, losses, RefLoss, registry.VQITQuantizerLossRegistry),
            (DISTANCES, distances, RefDistance, registry.VQITQuantizerDistanceRegistry),
            (ANCHORS, anchors, RefAnchor, registry.AnchorRegistry)):
        for name in names:
            ref.register_(name, force=True)(getattr(module, name))
        ours.add_fallback(ref)  # user-defined components registered only in the reference stay reachable
    registered_into_reference = True
    return True


register_into_reference()
