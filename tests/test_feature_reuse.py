"""Encoder-feature reuse (SURVEY.md section 8f row 2): the maps tapped during ``generator(x)`` are, bit for bit,
what ``generator.get_feature_layers(x, ids)`` returns -- for the stand-in generator, narrow and at the reference
generator's default size -- and every condition under which they would not be is a miss."""
import sys

import pytest
import torch

from standin_generator import StandInGenerator
from gan_variant_research_b200.feature_reuse import (EncoderFeatureCache, enable_encoder_feature_reuse,
                                                     logical_layer_modules)


def _same(a, b):
    return len(a) == len(b) and all(x.shape == y.shape and torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("ids", [[0, 4, 8, 12, 16], [0, 2, 3, 5, 6], [6], [1, 99], [4, 0, 4]])
def test_tapped_maps_equal_get_feature_layers(ids):
    torch.manual_seed(0)
    gen = StandInGenerator()                      # 7 logical layers: 0, 1-2, 3-5, 6-7 (7 = last up ReLU)
    cache = EncoderFeatureCache(gen, ids)
    x = torch.randn(2, 3, 32, 32)
    gen(x)
    got = cache.lookup(x, ids)
    want = gen.get_feature_layers(x, ids)
    assert got is not None and _same(got, want)
    assert all(not t.requires_grad for t in got)
    assert cache.hits == 1 and cache.misses == 0


def test_logical_numbering_covers_every_stage():
    gen = StandInGenerator(n_blocks=3)
    assert len(logical_layer_modules(gen)) == 1 + 2 + 3 + 2
    with pytest.raises(TypeError):
        logical_layer_modules(torch.nn.Linear(2, 2))


def test_every_stale_condition_is_a_miss():
    torch.manual_seed(1)
    gen = StandInGenerator()
    ids = [0, 3, 6]
    cache = enable_encoder_feature_reuse(gen, ids)
    x = torch.randn(1, 3, 32, 32)
    assert cache.lookup(x, ids) is None                              # nothing captured yet
    gen(x)
    assert cache.lookup(x.clone(), ids) is None                      # equal values, another tensor
    assert cache.lookup(x, [0, 1]) is None                           # a layer that was not tapped
    gen.get_feature_layers(torch.randn(1, 3, 32, 32), ids)           # the stacks run outside generator.__call__ ...
    got = cache.lookup(x, ids)                                       # ... and do not disturb the capture
    assert got is not None and _same(got, gen.get_feature_layers(x, ids))
    assert cache.lookup(x, ids) is None                              # released after the first hit
    gen(x); x.add_(1.0)
    assert cache.lookup(x, ids) is None                              # input changed in place
    gen(x)
    with torch.no_grad():
        next(gen.parameters()).mul_(1.01)
    assert cache.lookup(x, ids) is None                              # a parameter changed (optimiser step)
    gen(x); gen.eval()
    assert cache.lookup(x, ids) is None                              # train / eval flipped
    gen.train(); gen(x)
    with torch.autocast("cpu", dtype=torch.bfloat16):
        assert cache.lookup(x, ids) is None                          # autocast state differs
        gen(x)
        got = cache.lookup(x, ids)
        assert got is not None and got[0].dtype == torch.bfloat16 and _same(got, gen.get_feature_layers(x, ids))
    # a second enable replaces the first cache and its hooks
    cache2 = enable_encoder_feature_reuse(gen, ids)
    gen(x)
    assert cache.lookup(x, ids) is None and cache2.lookup(x, ids) is not None
    cache2.remove()
    assert not hasattr(gen, "_pnce_encoder_feature_cache")


@pytest.mark.parametrize("ids", [[0, 4, 8, 12, 16], [0, 4, 8, 12, 13]])
def test_against_the_unmodified_reference_generator(ids):
    """The reference's ``ResNetGenerator()`` at its defaults (ngf=64, 9 residual blocks, 14 logical layers), which the
    stand-in reproduces on the maps and losses frozen from the reference (tests/test_oracle_golden.py)."""
    torch.manual_seed(0)
    gen = StandInGenerator(ngf=64, n_blocks=9)
    cache = enable_encoder_feature_reuse(gen, ids)
    x = torch.randn(1, 3, 64, 64)
    fake = gen(x)                                                    # train_cutpp.py:270
    got = cache.lookup(x, ids)
    want = gen.get_feature_layers(x, ids)                            # patchnce_cut.py:138-139
    assert got is not None and len(got) == len(want) == (4 if 16 in ids else 5) and _same(got, want)
    assert fake.requires_grad and all(not t.requires_grad for t in got)


@pytest.mark.gpu
def test_compute_patchnce_loss_with_reuse_equals_without(monkeypatch):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import patchnce as pmod
    torch.manual_seed(3)
    gen = StandInGenerator(ngf=16, n_blocks=3).cuda()
    ids = [0, 2, 4, 6, 16]
    photos = torch.randn(2, 3, 64, 64, device="cuda")
    seen = []
    inner = pmod.PatchNCELoss.forward

    def spy(self, a, b, batch_size=None):
        seen.append([t.clone() for t in a])
        assert all(not t.requires_grad for t in a) and all(t.requires_grad for t in b)
        return inner(self, a, b, batch_size)

    monkeypatch.setattr(pmod.PatchNCELoss, "forward", spy)

    def g_step(reuse):
        cache = pn.enable_encoder_feature_reuse(gen, ids) if reuse else None
        gen.zero_grad(); gen.feature_passes = 0
        fake = gen(photos)                                           # train_cutpp.py:270
        torch.manual_seed(7)
        loss = pn.compute_patchnce_loss(gen, photos, fake, ids, 0.07, 64)      # :285-292
        loss.backward()
        grads = [p.grad.clone() for p in gen.parameters()]
        passes = gen.feature_passes
        if cache is not None:
            assert cache.hits == 1 and cache.misses == 0
            cache.remove()
        return loss.item(), grads, passes

    l0, g0, n0 = g_step(False)
    l1, g1, n1 = g_step(True)
    assert (n0, n1) == (2, 1)                                        # one generator pass fewer
    # cuDNN's transposed convolution is not run-to-run deterministic (2e-6 on `fake`, 1e-7 on the last map: measured,
    # scratch/exp28.py) and the randomly initialised generator amplifies a 1e-6 change of `fake` into a 3.5 % change of
    # the gradient, reuse or not -- so: source maps to rounding noise, loss to 1e-4, gradients to a connectivity check
    assert len(seen) == 2 and len(seen[0]) == len(seen[1]) == 4
    for a, b in zip(*seen):
        assert a.shape == b.shape and a.dtype == b.dtype
        assert float((a - b).abs().max()) <= 1e-5 * float(a.abs().max())
    assert l1 == pytest.approx(l0, rel=1e-4)
    for a, b in zip(g0, g1):
        assert torch.isfinite(b).all()
        if a.dim() > 1:          # biases in front of an InstanceNorm have a zero gradient: rounding noise only
            assert float((a - b).abs().max()) <= 0.3 * float(a.abs().max())


REFERENCE_SEAMS = {          # module of the reference package -> the names install_reference_shim re-points there
    "utils/io_ckpt.py": "class EMA:\n    pass\n",                                                     # train_cutpp.py:34
    "utils/amp_utils.py": "class AMPContext:\n    def step_optimizer(self, *a, **k):\n        pass\n",    # amp_utils.py:29
    "training/diffaugment.py": "class DiffAugment:\n    pass\n",                                        # train_cutpp.py:30
    "losses/adv_hinge.py": "def discriminator_hinge_loss(*a):\n    pass\n\n\ndef generator_hinge_loss(*a):\n    pass\n",
    "losses/patchnce_cut.py": "class PatchNCELoss:\n    pass\n\n\ndef compute_patchnce_loss(*a):\n    pass\n",
}


def test_shim_repoints_the_optimiser_side_seams(tmp_path):
    """On a package with the reference's module layout (GAN_Variant1/..., the seams as placeholders): the shim must
    re-point every seam a training script imports by name, and win over the on-disk patchnce_cut module."""
    import gan_variant_research_b200 as pn
    for path, body in REFERENCE_SEAMS.items():
        f = tmp_path / "GAN_Variant1" / path
        f.parent.mkdir(parents=True, exist_ok=True)
        f.write_text(body)
        for d in (f.parent, f.parent.parent):
            (d / "__init__.py").touch()
    root = str(tmp_path)
    sys.path.insert(0, root)
    saved = {k: v for k, v in sys.modules.items() if k.startswith("GAN_Variant1")}
    for k in saved:
        del sys.modules[k]
    try:
        import GAN_Variant1.utils.amp_utils as au
        import GAN_Variant1.utils.io_ckpt as ck
        keep = (ck.EMA, au.AMPContext.step_optimizer)
        import GAN_Variant1.training.diffaugment as da
        import GAN_Variant1.losses.adv_hinge as ah
        pn.install_reference_shim(optimiser_side=True, d_side=True)
        assert ck.EMA is pn.EMA and au.AMPContext.step_optimizer is pn.amp_step_optimizer
        assert da.DiffAugment is pn.DiffAugment and ah.generator_hinge_loss is pn.generator_hinge_loss
        assert ah.discriminator_hinge_loss is pn.discriminator_hinge_loss
        from GAN_Variant1.losses.patchnce_cut import compute_patchnce_loss
        assert compute_patchnce_loss is pn.compute_patchnce_loss
        ck.EMA, au.AMPContext.step_optimizer = keep
    finally:
        sys.path.remove(root)
        for k in [k for k in sys.modules if k.startswith("GAN_Variant1")]:
            del sys.modules[k]
        sys.modules.update(saved)
