"""Global negatives (minibatch negatives across data-parallel ranks, ``negatives_group``) without a GPU: the float64
shard oracle reproduces the full-batch minibatch oracle (mean of the shard losses, shard gradients divided by W) and
the global guard; the Python entry points default ``negatives_group`` to None and refuse it where it does not apply;
the new C entry points reject bad arguments before touching CUDA."""
import ctypes
import glob
import inspect
import os
import sys

import numpy as np
import pytest

import global_negatives_oracle as gno
import minibatch_oracle as mbo

SMALL = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "small_*.npz")))
IDS = [os.path.basename(p)[6:-4] for p in SMALL]


def _tiled(path, batch):
    """The fixture's layers with the batch repeated cyclically to ``batch`` images (divisible by every W tested)."""
    d = np.load(path)
    out = []
    for i in range(int(d["n_layers"])):
        s, t = d[f"src{i}"], d[f"tgt{i}"]
        idx = np.arange(batch) % s.shape[0]
        out.append((s[idx], t[idx], d[f"ids{i}"]))
    return float(d["tau"]), out


def _check_shards(src, tgt, ids, tau, world):
    full_loss, full_grad = mbo.layer_loss_and_grad_np_mb(src, tgt, ids, tau)
    bl = tgt.shape[0] // world
    shards = [gno.layer_loss_and_grad_np_shard(src, tgt, ids, tau, world, r) for r in range(world)]
    assert np.mean([l for l, _ in shards]) == pytest.approx(full_loss, rel=1e-12, abs=1e-14)
    for r, (_, g) in enumerate(shards):
        ref = full_grad[r * bl:(r + 1) * bl]
        np.testing.assert_array_equal(np.isnan(g), np.isnan(ref))
        fin = np.isfinite(ref)
        np.testing.assert_allclose(g[fin] / world, ref[fin], rtol=1e-9,
                                   atol=1e-14 * max(1.0, np.abs(ref[fin]).max(initial=0)))


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("path", SMALL, ids=IDS)
def test_shard_oracle_reproduces_the_full_batch(path, world):
    tau, layers = _tiled(path, 8)
    for src, tgt, ids in layers:
        _check_shards(src, tgt, ids, tau, world)


@pytest.mark.parametrize("world", [2, 4])
def test_shard_oracle_on_random_batches(world):
    rng = np.random.default_rng(world)
    for c, h, w, p in [(16, 8, 8, 40), (24, 6, 10, 60)]:
        src = rng.standard_normal((8, c, h, w))
        tgt = 0.6 * src + 0.8 * rng.standard_normal(src.shape)
        _check_shards(src, tgt, rng.integers(0, h * w, p), 0.07, world)


def test_nan_in_one_shard_zeroes_the_layer_in_every_shard():
    rng = np.random.default_rng(3)
    src = rng.standard_normal((4, 8, 6, 6))
    tgt = rng.standard_normal((4, 8, 6, 6))
    ids = rng.permutation(36)[:16]
    tgt[3, 2, ids[5] // 6, ids[5] % 6] = np.nan                 # rank 1 of 2 (images 2, 3)
    for r in range(2):
        loss, g = gno.layer_loss_and_grad_np_shard(src, tgt, ids, 0.07, 2, r)
        assert loss == 0.0
        if r == 0:
            assert (g == 0).all()
        else:
            assert np.isnan(g[1].reshape(8, -1)[:, ids[5]]).all()
            assert np.isnan(g).sum() == 8 and (g[~np.isnan(g)] == 0).all()
    full_loss, full_grad = mbo.layer_loss_and_grad_np_mb(src, tgt, ids, 0.07)
    assert full_loss == 0.0
    np.testing.assert_array_equal(np.isnan(full_grad[2:]), np.isnan(gno.layer_loss_and_grad_np_shard(
        src, tgt, ids, 0.07, 2, 1)[1]))
    src[0, 0, ids[0] // 6, ids[0] % 6] = np.inf                 # a non-finite key guards every rank too
    tgt[3, 2, ids[5] // 6, ids[5] % 6] = 0.5
    assert all(gno.layer_loss_and_grad_np_shard(src, tgt, ids, 0.07, 2, r)[0] == 0.0 for r in range(2))


def test_negatives_group_defaults_to_none_on_every_entry_point():
    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import patchnce
    for fn in (pn.PatchNCELoss.__init__, pn.compute_patchnce_loss, patchnce.install_reference_shim,
               patchnce.fused_patchnce):
        assert inspect.signature(fn).parameters["negatives_group"].default is None
    assert pn.PatchNCELoss().negatives_group is None
    for fn in (patchnce.patchnce_with_head, patchnce.head_loss_and_grads):
        assert "negatives_group" not in inspect.signature(fn).parameters


def test_negatives_group_needs_the_flag_and_the_maps_route():
    import torch
    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import patchnce
    with pytest.raises(ValueError, match="nce_includes_all_negatives_from_minibatch"):
        pn.PatchNCELoss(negatives_group=True)
    with pytest.raises(ValueError, match="nce_includes_all_negatives_from_minibatch"):
        pn.compute_patchnce_loss(None, None, None, [0], negatives_group=True)
    x = [torch.zeros(2, 4, 4, 4)]
    with pytest.raises(ValueError, match="nce_includes_all_negatives_from_minibatch"):
        patchnce.fused_patchnce(x, x, [torch.zeros(4, dtype=torch.int64)], negatives_group=True)
    with pytest.raises(ValueError, match="nce_includes_all_negatives_from_minibatch"):
        patchnce.install_reference_shim(negatives_group=True)
    crit = pn.PatchNCELoss(nce_includes_all_negatives_from_minibatch=True, negatives_group=True)
    rows = torch.zeros(32, 8)
    with pytest.raises(RuntimeError, match="row route"):
        crit(rows, rows)
    with pytest.raises(RuntimeError, match="row route"):
        crit([rows], [rows])


def test_global_batch_envelope_raises_first():
    from gan_variant_research_b200 import patchnce
    patchnce.mb_check(8, [64, 256], [256, 256], "tc_bf16x3", world=8)            # 64 x 256 keys: inside
    with pytest.raises(RuntimeError, match="global batch=72"):
        patchnce.mb_check(9, [64], [1024], "tc_bf16x3", world=8)                # 72 x 1024 keys
    with pytest.raises(RuntimeError, match="65536"):
        patchnce.mb_check(16, [64], [256], "tc_bf16", world=32)
    with pytest.raises(RuntimeError, match="tensor-core"):
        patchnce.mb_check(8, [64], [256], "simt_f32", world=2)


def test_reference_shim_forwards_negatives_group():
    from gan_variant_research_b200 import patchnce
    saved = {k: v for k, v in sys.modules.items() if k.startswith("GAN_Variant1")}
    try:
        mod = patchnce.install_reference_shim(nce_includes_all_negatives_from_minibatch=True, negatives_group=True)
        crit = mod.PatchNCELoss(0.07, 16)
        assert crit.negatives_group is True and crit.nce_includes_all_negatives_from_minibatch is True
        assert mod.compute_patchnce_loss.keywords["negatives_group"] is True
        mod = patchnce.install_reference_shim(nce_includes_all_negatives_from_minibatch=True)
        assert mod.PatchNCELoss(0.07, 16).negatives_group is None
        assert "negatives_group" not in mod.compute_patchnce_loss.keywords
    finally:
        for k in [k for k in sys.modules if k.startswith("GAN_Variant1")]:
            del sys.modules[k]
        sys.modules.update(saved)


@pytest.fixture(scope="module")
def lib():
    from gan_variant_research_b200 import _lib, build
    build.build()
    return _lib.load()


def _layers(shapes, p, fake_ptrs=False):
    from gan_variant_research_b200 import _lib
    arr = (_lib.PnceLayer * len(shapes))()
    for i, (c, h, w) in enumerate(shapes):
        arr[i].C, arr[i].H, arr[i].W, arr[i].P = c, h, w, min(p, h * w)
        if fake_ptrs:                                   # aligned, never dereferenced: the calls stop before CUDA
            arr[i].src, arr[i].tgt, arr[i].ids = 1 << 20, 2 << 20, 3 << 20
    return arr


def test_c_entry_points_reject_bad_arguments_without_touching_cuda(lib):
    from gan_variant_research_b200 import _lib
    b5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
    n, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    mb = ctypes.c_size_t(0)
    assert lib.pnce_mb_workspace_bytes(_layers(b5, 256), 5, 8, ctypes.byref(mb)) == 0
    assert lib.pnce_mb_shard_workspace_bytes(_layers(b5, 256), 5, 8, 8, ctypes.byref(n), ctypes.byref(off),
                                             ctypes.byref(sb)) == 0
    assert off.value == mb.value and sb.value % 256 == 0 and n.value == off.value + 8 * sb.value
    # a slot holds the key blobs (hi + lo, block- and key-major) and the key sums of squares of 8 images per layer
    keys = sum(8 * 256 * c * 2 * 4 + 8 * (c // 32) * 256 * 4 for c, _, _ in b5)
    assert keys <= sb.value <= keys + 256 * (1 + 5 * 5)
    args = lambda world: (_layers(b5, 256), 5, 8, world, ctypes.byref(n), ctypes.byref(off), ctypes.byref(sb))
    assert lib.pnce_mb_shard_workspace_bytes(*args(32)) == 0                    # 256 x 256 keys: inside
    assert lib.pnce_mb_shard_workspace_bytes(*args(33)) == -2                   # global keys > 65536
    assert lib.pnce_mb_shard_workspace_bytes(*args(0)) == -1
    assert lib.pnce_mb_shard_workspace_bytes(_layers(b5, 256), 5, 8, 2, None, ctypes.byref(off), ctypes.byref(sb)) == -1
    lay = _layers([(8, 4, 4)], 16, fake_ptrs=True)
    tc, f32, nchw = _lib.MATH_TC_BF16X3, _lib.PNCE_F32, _lib.LAYOUT_NCHW

    def keys_call(world, rank, math=tc, ws=None, layers=lay, batch=2, dtype=f32, layout=nchw):
        return lib.pnce_mb_shard_keys(layers, 1, batch, dtype, layout, world, rank, math, ws, 1 << 30, None, 0, None,
                                      None)

    def loss_call(world, rank, math=tc, ws=None, out=None, tau=0.07):
        return lib.pnce_mb_shard_loss(lay, 1, 2, f32, nchw, world, rank, tau, math, ws, 1 << 30, None, 0, out,
                                      None, None)

    for call in (keys_call, loss_call):
        assert call(0, 0) == -1                                               # world < 1
        assert call(2, 2) == -1 and call(2, -1) == -1                          # rank outside [0, world)
        assert call(2, 1, math=_lib.MATH_SIMT_F32) == -2
        assert call(2, 1) == -3                                                # NULL workspace
        assert call(2, 1, ws=128) == -3                                        # misaligned workspace
    assert keys_call(2, 0, dtype=7) == -1 and keys_call(2, 0, layout=5) == -1
    assert keys_call(2, 0, layers=_layers([(8, 4, 4)], 16)) == -1               # NULL maps / ids
    big = _layers([(8, 32, 32)], 1024, fake_ptrs=True)
    assert keys_call(8, 0, layers=big, batch=9) == -2 and keys_call(16, 3, layers=big, batch=5) == -2  # > 65536 keys
    assert keys_call(4, 0, layers=big, batch=16) == -3                          # 64 x 1024 keys: inside, then no workspace
    out = ctypes.c_float(0)
    ws = 1 << 30                                                                # aligned, large enough: never touched
    assert loss_call(2, 0, ws=ws) == -1                                         # NULL loss
    assert loss_call(2, 0, ws=ws, out=ctypes.addressof(out), tau=0.0) == -1
