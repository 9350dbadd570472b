"""Minibatch negatives (upstream CUT's nce_includes_all_negatives_from_minibatch) without a GPU: the two oracle
restatements agree with each other, with the per-image oracle at B = 1, and with a third, independent expression;
the Python entry points default the flag to False and the reference shim forwards it; the new C entry points
reject bad arguments before touching CUDA."""
import ctypes
import glob
import inspect
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import minibatch_oracle as mbo
from oracle import patchnce_oracle as orc

SMALL = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "small_*.npz")))
IDS = [os.path.basename(p)[6:-4] for p in SMALL]


def _load(path):
    d = np.load(path)
    n = int(d["n_layers"])
    return d, [(d[f"src{i}"], d[f"tgt{i}"], d[f"ids{i}"]) for i in range(n)]


def _autograd_mb(src, tgt, ids, tau):
    """Third expression: CE of (q.view(1, -1, C) @ k.view(1, -1, C).mT) / tau, clamp, by autograd (no guard)."""
    s = torch.from_numpy(src).double()
    t = torch.from_numpy(tgt).double().requires_grad_()
    i = torch.from_numpy(ids)
    b, c = s.shape[:2]
    k = F.normalize(s.reshape(b, c, -1).transpose(1, 2)[:, i, :], dim=2, eps=orc.NORM_EPS)
    q = F.normalize(t.reshape(b, c, -1).transpose(1, 2)[:, i, :], dim=2, eps=orc.NORM_EPS)
    z = (q.reshape(1, -1, c) @ k.reshape(1, -1, c).mT) / tau
    z = z.clamp(-orc.LOGIT_CLAMP, orc.LOGIT_CLAMP)[0]
    loss = F.cross_entropy(z, torch.arange(z.shape[0]))
    loss.backward()
    return loss.item(), t.grad.numpy()


@pytest.mark.parametrize("path", SMALL, ids=IDS)
def test_torch_and_float64_minibatch_oracles_agree(path):
    d, layers = _load(path)
    tau = float(d["tau"])
    for src, tgt, ids in layers:
        t = torch.from_numpy(tgt).double().requires_grad_()
        warn = []
        lt = mbo.layer_loss_torch_mb(torch.from_numpy(src).double(), t, torch.from_numpy(ids), tau, warn)
        if lt.requires_grad:
            lt.backward()
        gt = t.grad.numpy() if t.grad is not None else np.zeros_like(tgt, dtype=np.float64)
        ln, gn = mbo.layer_loss_and_grad_np_mb(src, tgt, ids, tau)
        assert float(lt.detach()) == pytest.approx(ln, rel=1e-9, abs=1e-12)
        if warn:
            # the guarded group: its loss node is a constant, so the torch restatement has no gradient path; the
            # float64 sheet states the kernel's law -- zero, NaN on the sampled target patches that hold a NaN/Inf
            assert ln == 0.0 and np.isnan(gn).any() == (~np.isfinite(tgt)).any()
            assert (gn[~np.isnan(gn)] == 0).all()
            continue
        np.testing.assert_array_equal(np.isnan(gn), np.isnan(gt))
        fin = np.isfinite(gn)
        np.testing.assert_allclose(gt[fin], gn[fin], rtol=1e-7, atol=1e-12 * max(1.0, np.abs(gn[fin]).max(initial=0)))


@pytest.mark.parametrize("path", SMALL, ids=IDS)
def test_one_image_equals_the_per_image_oracle(path):
    d, layers = _load(path)
    tau = float(d["tau"])
    for src, tgt, ids in layers:
        for b in range(src.shape[0]):
            s1, t1 = src[b:b + 1], tgt[b:b + 1]
            lp, _, gp = orc.layer_loss_and_grad_np(s1, t1, ids, tau)
            lm, gm = mbo.layer_loss_and_grad_np_mb(s1, t1, ids, tau)
            assert lm == lp
            np.testing.assert_array_equal(gm, gp)


@pytest.mark.parametrize("path", SMALL, ids=IDS)
def test_minibatch_oracle_equals_an_independent_expression(path):
    d, layers = _load(path)
    tau = float(d["tau"])
    for src, tgt, ids in layers:
        ln, gn = mbo.layer_loss_and_grad_np_mb(src, tgt, ids, tau)
        if not np.isfinite(gn).all() or ln == 0.0:
            continue                                  # guarded group: the plain expression has no guard
        la, ga = _autograd_mb(src, tgt, ids, tau)
        assert ln == pytest.approx(la, rel=1e-10, abs=1e-12)
        np.testing.assert_allclose(gn, ga, rtol=1e-8, atol=1e-12 * max(1.0, np.abs(ga).max()))


def test_minibatch_differs_from_per_image_when_batch_is_larger_than_one():
    d, layers = _load(os.path.join(os.path.dirname(__file__), "golden", "small_basic.npz"))
    src, tgt, ids = layers[0]
    assert src.shape[0] > 1
    lp, _, _ = orc.layer_loss_and_grad_np(src, tgt, ids, float(d["tau"]))
    lm, _ = mbo.layer_loss_and_grad_np_mb(src, tgt, ids, float(d["tau"]))
    assert lm > lp                                    # more negatives, larger CE


def test_flag_defaults_to_false_on_every_entry_point():
    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import patchnce
    for fn in (pn.PatchNCELoss.__init__, pn.compute_patchnce_loss, patchnce.install_reference_shim,
               patchnce.fused_patchnce):
        p = inspect.signature(fn).parameters["nce_includes_all_negatives_from_minibatch"]
        assert p.default is False
    assert pn.PatchNCELoss().nce_includes_all_negatives_from_minibatch is False
    for fn in (patchnce.patchnce_with_head, patchnce.head_loss_and_grads):
        assert "nce_includes_all_negatives_from_minibatch" not in inspect.signature(fn).parameters


def test_reference_shim_forwards_the_flag():
    from gan_variant_research_b200 import patchnce
    saved = {k: v for k, v in sys.modules.items() if k.startswith("GAN_Variant1")}
    try:
        mod = patchnce.install_reference_shim(nce_includes_all_negatives_from_minibatch=True)
        assert mod.PatchNCELoss(0.07, 16).nce_includes_all_negatives_from_minibatch is True
        assert mod.compute_patchnce_loss.keywords["nce_includes_all_negatives_from_minibatch"] is True
        mod = patchnce.install_reference_shim()
        assert mod.PatchNCELoss(0.07, 16).nce_includes_all_negatives_from_minibatch is False
        assert mod.compute_patchnce_loss is patchnce.compute_patchnce_loss
    finally:
        for k in [k for k in sys.modules if k.startswith("GAN_Variant1")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_envelope_errors_are_raised_before_any_launch():
    from gan_variant_research_b200 import patchnce
    with pytest.raises(RuntimeError, match="tensor-core"):
        patchnce.mb_check(4, [64], [256], "simt_f32")
    with pytest.raises(RuntimeError, match="65536"):
        patchnce.mb_check(129, [64], [512], "tc_bf16x3")
    with pytest.raises(RuntimeError, match="C <= 256"):
        patchnce.mb_check(4, [512], [256], "tc_bf16x3")
    with pytest.raises(RuntimeError, match="P <= 256"):
        patchnce.mb_check(4, [64], [512], "tc_bf16x3", rows=True)
    patchnce.mb_check(64, [256], [1024], "tc_bf16")           # 65536 keys: inside


@pytest.fixture(scope="module")
def lib():
    from gan_variant_research_b200 import _lib, build
    build.build()
    return _lib.load()


def _layers(shapes, p):
    from gan_variant_research_b200 import _lib
    arr = (_lib.PnceLayer * len(shapes))()
    for i, (c, h, w) in enumerate(shapes):
        arr[i].C, arr[i].H, arr[i].W, arr[i].P = c, h, w, min(p, h * w)
    return arr


def test_c_entry_points_reject_bad_arguments_without_touching_cuda(lib):
    from gan_variant_research_b200 import _lib
    n = ctypes.c_size_t(0)
    b5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
    assert lib.pnce_mb_workspace_bytes(_layers(b5, 256), 5, 64, ctypes.byref(n)) == 0
    per_image = ctypes.c_size_t(0)
    assert lib.pnce_workspace_bytes(_layers(b5, 256), 5, 64, ctypes.byref(per_image)) == 0
    assert 0 < n.value <= per_image.value
    assert lib.pnce_mb_workspace_bytes(_layers(b5, 256), 5, 256, ctypes.byref(n)) == 0       # 256 * 256 keys
    assert lib.pnce_mb_workspace_bytes(_layers(b5, 256), 5, 257, ctypes.byref(n)) == -2      # B * Ppad > 65536
    assert lib.pnce_mb_workspace_bytes(_layers([(64, 40, 40)], 1100), 1, 2, ctypes.byref(n)) == -2   # P > 1024
    assert lib.pnce_mb_workspace_bytes(_layers([(512, 8, 8)], 64), 1, 2, ctypes.byref(n)) == -2      # C > 256
    assert lib.pnce_mb_workspace_bytes(_layers(b5, 256), 5, 0, ctypes.byref(n)) == -1
    assert lib.pnce_mb_workspace_bytes(None, 1, 1, ctypes.byref(n)) == -1
    lay = _layers([(8, 4, 4)], 16)
    # simt_f32 is refused, then NULL workspace / loss / bad dtype, all before any CUDA call
    assert lib.pnce_mb_fwd(lay, 1, 2, 0, 0, 0.07, _lib.MATH_SIMT_F32, None, 0, None, 0, None, None, None, None) == -2
    assert lib.pnce_mb_fwd(lay, 1, 2, 0, 0, 0.07, _lib.MATH_TC_BF16X3, None, 0, None, 0, None, None, None, None) == -1
    assert lib.pnce_mb_fwd(lay, 1, 2, 7, 0, 0.07, _lib.MATH_TC_BF16X3, None, 0, None, 0, None, None, None, None) == -1
    assert lib.pnce_mb_fwd(lay, 1, 2, 0, 5, 0.07, _lib.MATH_TC_BF16X3, None, 0, None, 0, None, None, None, None) == -1
    big = _layers([(8, 32, 32)], 1024)
    out = ctypes.c_float(0)
    assert lib.pnce_mb_fwd(big, 1, 65, 0, 0, 0.07, _lib.MATH_TC_BF16X3, None, 0, None, 0, None,
                           ctypes.addressof(out), None, None) == -2
    rows = (_lib.PnceRows * 1)()
    rows[0].P, rows[0].D = 256, 64
    assert lib.pnce_rows_mb_workspace_bytes(rows, 1, 256, ctypes.byref(n)) == 0 and n.value > 0
    assert lib.pnce_rows_mb_workspace_bytes(rows, 1, 257, ctypes.byref(n)) == -2
    rows[0].P = 512                                     # the row pack covers one key block per image
    assert lib.pnce_rows_mb_workspace_bytes(rows, 1, 2, ctypes.byref(n)) == -2
    rows[0].P = 256
    assert lib.pnce_rows_mb_fwd_bwd(rows, 1, 2, 0.07, _lib.MATH_SIMT_F32, None, 0, ctypes.addressof(out), None, None) == -2
    assert lib.pnce_rows_mb_fwd_bwd(rows, 1, 2, 0.07, _lib.MATH_TC_BF16, None, 0, None, None, None) == -1
    assert lib.pnce_rows_mb_fwd_bwd(rows, 0, 2, 0.07, _lib.MATH_TC_BF16, None, 0, ctypes.addressof(out), None, None) == -1
    assert lib.pnce_rows_mb_fwd_bwd(rows, 1, 2, 0.07, _lib.MATH_TC_BF16, None, 0, ctypes.addressof(out), None, None) == -3
