"""Pins the oracle to the reference: every restatement in oracle/patchnce_oracle.py is checked
against fixtures produced by running the UNMODIFIED reference (oracle/make_golden.py)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import patchnce_oracle as orc

R4 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128)]


def _load_small(path):
    d = np.load(path)
    n = int(d["n_layers"])
    src = [d[f"src{i}"] for i in range(n)]
    tgt = [d[f"tgt{i}"] for i in range(n)]
    ids = [d[f"ids{i}"] for i in range(n)]
    grads = [d[f"grad{i}"] for i in range(n)]
    return d, src, tgt, ids, grads


SMALL = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "small_*.npz")))


@pytest.mark.parametrize("path", SMALL, ids=[os.path.basename(p)[6:-4] for p in SMALL])
def test_torch_restatement_matches_reference(path):
    d, src, tgt, ids, grads = _load_small(path)
    s = [torch.from_numpy(x) for x in src]
    t = [torch.from_numpy(x).requires_grad_() for x in tgt]
    i = [torch.from_numpy(x) for x in ids]
    loss, _ = orc.patchnce_loss_torch(s, t, float(d["tau"]), int(d["num_patches"]), ids_list=i)
    assert loss.item() == pytest.approx(float(d["loss"]), rel=1e-6, abs=1e-7)
    if loss.requires_grad:
        (loss * float(d["upstream"])).backward()
    for tt, g in zip(t, grads):
        got = tt.grad.numpy() if tt.grad is not None else np.zeros_like(g)
        np.testing.assert_allclose(got, g, rtol=1e-5, atol=1e-7 * max(1.0, np.abs(g).max()))


@pytest.mark.parametrize("path", SMALL, ids=[os.path.basename(p)[6:-4] for p in SMALL])
def test_numpy_restatement_matches_reference(path):
    """The analytic backward (the formula sheet the CUDA kernels follow) vs reference autograd."""
    d, src, tgt, ids, grads = _load_small(path)
    loss, _, g_np = orc.patchnce_loss_and_grads_np(src, tgt, ids, float(d["tau"]),
                                                   upstream=float(d["upstream"]))
    assert loss == pytest.approx(float(d["loss"]), rel=2e-6, abs=1e-6)
    for got, g in zip(g_np, grads):
        scale = max(1e-30, float(np.abs(g).max()))
        # fp32 reference vs fp64 restatement: 1e-4 of the largest entry is ample
        np.testing.assert_allclose(got, g, rtol=2e-3, atol=2e-5 * scale)


def test_ids_are_drawn_like_the_reference(golden_dir):
    """One randint per layer, in order, P = min(num_patches, HW), with replacement (:60-63)."""
    d = np.load(os.path.join(golden_dir, "small_ragged.npz"))
    shapes = [d[f"src{i}"].shape for i in range(3)]
    src = [torch.from_numpy(d[f"src{i}"]) for i in range(3)]
    tgt = [torch.from_numpy(d[f"tgt{i}"]) for i in range(3)]
    torch.manual_seed(4)
    _, ids = orc.patchnce_loss_torch(src, tgt, 0.07, 64)
    for i, sh in enumerate(shapes):
        assert ids[i].dtype == torch.int64
        assert ids[i].numel() == min(64, sh[2] * sh[3])
        np.testing.assert_array_equal(ids[i].numpy(), d[f"ids{i}"])


def test_cpu_id_law(golden_dir):
    """ids = mt19937(seed) raw 32-bit % HW, consumed layer after layer (SURVEY.md 8c)."""
    law = np.load(os.path.join(golden_dir, "cpu_id_law.npz"))
    hws = (65536, 4096, 4096, 16384, 100)
    for seed in (0, 7, 12345):
        got = orc.mt19937_ids(seed, hws, 256)
        for j in range(len(hws)):
            np.testing.assert_array_equal(got[j], law[f"s{seed}_l{j}"])


@pytest.mark.parametrize("b", [1, 2])
def test_survey_tripwire_full_size(golden_dir, b):
    """SURVEY.md 8c full-size R4 case: ids, loss, per-layer losses, grad norms, nnz, grad columns."""
    d = np.load(os.path.join(golden_dir, f"survey_r4_b{b}.npz"))
    g = torch.Generator().manual_seed(1234)
    src = [torch.randn(b, *s, generator=g).relu() for s in R4]
    tgt = [torch.randn(b, *s, generator=g).relu().requires_grad_() for s in R4]
    torch.manual_seed(7)
    loss, ids = orc.patchnce_loss_torch(src, tgt, 0.07, 256)
    loss.backward()
    assert loss.item() == pytest.approx(float(d["loss"]), rel=1e-6)
    tab = {1: 5.938309669, 2: 5.962453842}            # the digits printed in SURVEY.md 8c
    assert loss.item() == pytest.approx(tab[b], rel=1e-6)
    for i, t in enumerate(tgt):
        np.testing.assert_array_equal(ids[i].numpy(), d[f"ids{i}"])
        gr = t.grad
        assert gr.double().norm().item() == pytest.approx(float(d[f"gnorm{i}"]), rel=1e-5)
        assert int((gr != 0).sum()) == int(d[f"nnz{i}"])
        cols = gr[0].reshape(gr.shape[1], -1)[:, ids[i][:8]].numpy()
        np.testing.assert_allclose(cols, d[f"gcols{i}"], rtol=1e-4, atol=1e-9)
    if b == 1:
        # numpy analytic restatement on the two 64x64 layers (cheap) against the same goldens
        for i in (1, 2):
            _, _, gnp = orc.layer_loss_and_grad_np(src[i].numpy(), tgt[i].detach().numpy(),
                                                   ids[i].numpy(), 0.07, n_layers=4)
            assert np.linalg.norm(gnp) == pytest.approx(float(d[f"gnorm{i}"]), rel=1e-4)


def test_oracle_on_the_frozen_generator_maps(golden_dir):
    """Both restatements of the oracle against the reference's loss and gradients on the feature maps of the unmodified
    ResNetGenerator (oracle/make_golden_generator.py): dead post-ReLU patches (the g / eps branch of F.normalize's
    backward, patchnce_cut.py:77-78) and 16x16 maps sampled several times per position."""
    d = np.load(os.path.join(golden_dir, "generator_maps_b5.npz"))
    n = int(d["n_layers"])
    src = [d[f"src{i}"] for i in range(n)]
    tgt = [d[f"tgt{i}"] for i in range(n)]
    ids = [d[f"ids{i}"] for i in range(n)]
    up = float(d["upstream"])
    loss, _, grads = orc.patchnce_loss_and_grads_np(src, tgt, ids, 0.07, upstream=up)
    assert loss == pytest.approx(float(d["loss"]), rel=2e-6)
    for i in range(n):
        want = d[f"grad{i}"].astype(np.float64)
        assert np.abs(grads[i] - want).max() <= 2e-4 * np.abs(want).max()
    # the op-for-op torch port draws the same ids from the same seed
    t = [torch.from_numpy(x).requires_grad_() for x in tgt]
    torch.manual_seed(7)
    tl, tids = orc.patchnce_loss_torch([torch.from_numpy(x) for x in src], t, 0.07, 256)
    (tl * up).backward()
    assert tl.item() == pytest.approx(float(d["loss"]), rel=1e-6)
    for i in range(n):
        np.testing.assert_array_equal(tids[i].numpy(), ids[i])
        np.testing.assert_allclose(t[i].grad.numpy(), d[f"grad{i}"], rtol=1e-4, atol=1e-6 * np.abs(d[f"grad{i}"]).max())


def test_standin_generator_reproduces_the_reference_maps(golden_dir):
    """The stand-in generator, seeded and run like oracle/make_golden_generator.py ran the unmodified reference
    ``ResNetGenerator(ngf=8)``, gives the frozen maps (bit for bit where they were frozen; to rounding allowed here, as
    another CPU's convolution kernels may sum in another order): the tests that stand it in for the reference
    generator compare like with like."""
    from standin_generator import StandInGenerator
    d = np.load(os.path.join(golden_dir, "generator_maps_b5.npz"))
    torch.manual_seed(2024)
    gen = StandInGenerator(ngf=8, n_blocks=9).eval()
    photo = torch.rand(2, 3, 64, 64) * 2 - 1
    fake = torch.tanh(torch.randn(2, 3, 64, 64))
    with torch.no_grad():
        src = gen.get_feature_layers(photo, [0, 4, 8, 12, 13])
        tgt = gen.get_feature_layers(fake, [0, 4, 8, 12, 13])
    assert len(src) == len(tgt) == int(d["n_layers"])
    for i, (s, t) in enumerate(zip(src, tgt)):
        np.testing.assert_allclose(s.numpy(), d[f"src{i}"], rtol=1e-5, atol=1e-6 * np.abs(d[f"src{i}"]).max())
        np.testing.assert_allclose(t.numpy(), d[f"tgt{i}"], rtol=1e-5, atol=1e-6 * np.abs(d[f"tgt{i}"]).max())


def test_invalid_layer_ids_are_skipped_and_mean_divides_by_returned_maps(golden_dir):
    """[0,4,8,12,16] returns 4 maps (id 16 never matches) and the loss divides by 4
    (generator_resnet_attn.py:203-235, patchnce_cut.py:40).  Checked against the e2e golden, which the unmodified
    reference ``ResNetGenerator()`` produced, with the stand-in generator at the reference's default width and
    depth: it builds, initialises and runs the same layers in the same order, so the same seed gives the same
    loss and gradient (and the maps of generator_maps_b5.npz, test_standin_generator_reproduces_the_reference_maps)."""
    from standin_generator import StandInGenerator
    d = np.load(os.path.join(golden_dir, "e2e_generator.npz"))
    for tag, layers, n_maps in (("r4", [0, 4, 8, 12, 16], 4), ("b5", [0, 4, 8, 12, 13], 5)):
        torch.manual_seed(0)
        gen = StandInGenerator(ngf=64, n_blocks=9)
        x = torch.randn(1, 3, 256, 256)
        y = torch.tanh(torch.randn(1, 3, 256, 256)).requires_grad_()
        assert len(gen.get_feature_layers(x, layers)) == n_maps
        torch.manual_seed(7)
        loss = orc.compute_patchnce_loss_torch(gen, x, y, layers, 0.07, 256)
        loss.backward()
        assert loss.item() == pytest.approx(float(d[f"loss_{tag}"]), rel=1e-6)
        assert y.grad.double().norm().item() == pytest.approx(float(d[f"gnorm_{tag}"]), rel=1e-4)


def test_virtual_shard_equals_full_batch(golden_dir):
    """SURVEY.md 8e: negatives are per image, so splitting the batch into N shards with the same
    ids and averaging loss / summing grads scaled by 1/N reproduces the full-batch result."""
    d, src, tgt, ids, grads = _load_small(os.path.join(golden_dir, "small_ragged.npz"))
    full, _, gfull = orc.patchnce_loss_and_grads_np(src, tgt, ids, 0.07)
    parts = []
    gparts = [np.zeros_like(g, dtype=np.float64) for g in gfull]
    for b in range(3):
        l, _, g = orc.patchnce_loss_and_grads_np([s[b:b + 1] for s in src], [t[b:b + 1] for t in tgt],
                                                 ids, 0.07)
        parts.append(l)
        for i in range(len(g)):
            gparts[i][b:b + 1] = g[i] / 3.0
    assert np.mean(parts) == pytest.approx(full, rel=1e-12)
    for a, bb in zip(gparts, gfull):
        np.testing.assert_allclose(a, bb, rtol=1e-10, atol=1e-18)


def test_head_oracle_self_consistency():
    """netF head: PARITY UNPINNED by the reference.  Checks shapes, unit norms, k detached."""
    torch.manual_seed(0)
    c, nc = 12, 16
    w1 = torch.randn(nc, c, requires_grad=True)
    b1 = torch.zeros(nc, requires_grad=True)
    w2 = torch.randn(nc, nc, requires_grad=True)
    b2 = torch.zeros(nc, requires_grad=True)
    src = [torch.randn(2, c, 5, 5)]
    tgt = [torch.randn(2, c, 5, 5, requires_grad=True)]
    ids = [torch.randint(0, 25, (10,))]
    loss = orc.patchnce_head_loss_torch(src, tgt, ids, [(w1, b1, w2, b2)])
    loss.backward()
    assert torch.isfinite(loss) and w1.grad is not None and tgt[0].grad is not None
    y = orc.head_forward_torch(torch.randn(7, c), w1, b1, w2, b2)
    torch.testing.assert_close(y.norm(dim=1), torch.ones(7), rtol=1e-5, atol=1e-5)
