"""The netF head with global negatives (patchnce_with_head_global_negatives) without a GPU: the float64 shard oracle
reproduces the one-GPU head minibatch oracle on the global batch (losses, d tgt, head gradients) and its guard is
global; the new Python entry points have the documented signatures and refuse out-of-envelope calls before touching a
device or a collective; the new C entry points reject bad arguments before any CUDA call and lay out the workspace as
documented."""
import ctypes
import inspect

import pytest
import torch

import head_global_negatives_oracle as hgo
import head_minibatch_oracle as hmo

SHAPES = [(24, 8, 8), (40, 6, 10)]


def _problem(seed, b, nc, p=20, shapes=SHAPES):
    g = torch.Generator().manual_seed(seed)
    src = [torch.randn(b, *s, generator=g, dtype=torch.float64) for s in shapes]
    tgt = [0.6 * a + 0.8 * torch.randn(a.shape, generator=g, dtype=torch.float64) for a in src]
    ids = [torch.randint(0, h * w, (p,), generator=g) for _, h, w in shapes]
    heads = [(0.3 * torch.randn(nc, c, generator=g, dtype=torch.float64), 0.1 * torch.randn(nc, generator=g, dtype=torch.float64),
              0.3 * torch.randn(nc, nc, generator=g, dtype=torch.float64), 0.1 * torch.randn(nc, generator=g, dtype=torch.float64))
             for c, _, _ in shapes]
    return src, tgt, ids, heads


def _loss_and_grads(fn, src, tgt, ids, heads):
    t = [x.clone().requires_grad_() for x in tgt]
    h = [tuple(w.clone().requires_grad_() for w in hd) for hd in heads]
    warn = []
    loss = fn(src, t, ids, h, warn)
    if loss.requires_grad:
        loss.backward()
    zero = lambda x: torch.zeros_like(x) if x.grad is None else x.grad
    return loss.item(), [zero(x) for x in t], [[zero(w) for w in hd] for hd in h], warn


def _global(src, tgt, ids, heads):
    return _loss_and_grads(lambda s, t, i, h, w: hmo.head_minibatch_loss(s, t, i, h, 0.07, w), src, tgt, ids, heads)


def _shard(src, tgt, ids, heads, world, rank):
    return _loss_and_grads(lambda s, t, i, h, w: hgo.head_global_negatives_loss(s, t, i, h, world, rank, 0.07, w),
                           src, tgt, ids, heads)


def test_one_rank_is_the_head_minibatch_oracle():
    src, tgt, ids, heads = _problem(1, 3, 128)
    la, ga, ha, _ = _global(src, tgt, ids, heads)
    lb, gb, hb, _ = _shard(src, tgt, ids, heads, 1, 0)
    assert lb == la
    for a, b in zip(ga + sum(ha, []), gb + sum(hb, [])):
        assert torch.equal(a, b)


@pytest.mark.parametrize("world,nc", [(2, 128), (4, 256), (4, 128)])
def test_shards_reproduce_the_global_batch(world, nc):
    bl = 2
    src, tgt, ids, heads = _problem(world + nc, world * bl, nc)
    lg, gg, hg, _ = _global(src, tgt, ids, heads)
    shards = [_shard(src, tgt, ids, heads, world, r) for r in range(world)]
    assert sum(s[0] for s in shards) / world == pytest.approx(lg, rel=1e-12)
    for l in range(len(src)):
        for r, (_, gt, _, _) in enumerate(shards):
            sl = slice(r * bl, (r + 1) * bl)
            torch.testing.assert_close(gt[l][sl] / world, gg[l][sl], rtol=1e-12, atol=1e-15)
            others = torch.ones(world * bl, dtype=torch.bool)
            others[sl] = False
            assert (gt[l][others] == 0).all()                   # a rank's loss reaches its own images only
        for k in range(4):
            mean = sum(s[2][l][k] for s in shards) / world
            torch.testing.assert_close(mean, hg[l][k], rtol=1e-11, atol=1e-14)


@pytest.mark.parametrize("side,rank", [("tgt", 1), ("src", 0)])
def test_a_non_finite_patch_on_one_rank_guards_every_rank(side, rank):
    world, bl = 2, 2
    src, tgt, ids, heads = _problem(5, world * bl, 128)
    maps = tgt if side == "tgt" else src
    maps[1][rank * bl + 1, 3].reshape(-1)[ids[1][4]] = float("nan")    # a sampled patch of layer 1 on rank `rank`
    lg, gg, hg, wg = _global(src, tgt, ids, heads)
    assert wg == ["layer"]
    for r in range(world):
        ls, gt, hs, ws = _shard(src, tgt, ids, heads, world, r)
        assert ws == ["layer"]                                  # the same decision on every rank
        assert (gt[1] == 0).all() and all((w == 0).all() for w in hs[1])
        l0, g0, h0, _ = _loss_and_grads(lambda s, t, i, h, w: hgo.head_global_negatives_loss(s, t, i, h, world, r, 0.07, w),
                                        src[:1], tgt[:1], ids[:1], heads[:1])
        assert ls == pytest.approx(l0 / 2, rel=1e-13)          # layer 1 contributes 0 to the mean over two layers
        torch.testing.assert_close(gt[0], g0[0] / 2, rtol=1e-12, atol=0)


def test_signatures_and_defaults():
    import gan_variant_research_b200 as pn
    assert "patchnce_with_head_global_negatives" in pn.__all__ and "head_global_negatives_loss_and_grads" in pn.__all__
    a = inspect.signature(pn.patchnce_with_head_global_negatives).parameters
    assert list(a) == ["netF", "src_feats", "tgt_feats", "temperature", "num_patches", "patch_ids", "math",
                       "negatives_group", "dp_group"]
    b = inspect.signature(pn.head_global_negatives_loss_and_grads).parameters
    assert list(b) == ["netF", "src_feats", "tgt_feats", "temperature", "num_patches", "patch_ids", "math",
                       "grad_output", "negatives_group", "dp_group"]
    for p in (a, b):
        assert p["temperature"].default == 0.07 and p["num_patches"].default == 256
        assert p["patch_ids"].default is None and p["math"].default is None and p["dp_group"].default is None
        assert p["negatives_group"].default is True
    assert b["grad_output"].default is None
    for fn in (pn.patchnce_with_head_global_negatives, pn.head_global_negatives_loss_and_grads):
        assert "GradReducer" in fn.__doc__ or "patchnce_with_head_global_negatives" in fn.__doc__
    assert "GradReducer" in pn.patchnce_with_head_global_negatives.__doc__
    # the four existing head entry points keep their parameter lists
    for fn in (pn.patchnce_with_head, pn.head_loss_and_grads, pn.patchnce_with_head_minibatch,
               pn.head_minibatch_loss_and_grads):
        assert "negatives_group" not in inspect.signature(fn).parameters


def test_global_envelope_raises_before_any_device_or_collective_work(monkeypatch):
    """Eight ranks (resolve_group / get_world_size patched), CPU tensors: each error is raised before the maps are looked
    at (they would fail with "no CPU fallback"), before the key exchange and before netF is built."""
    import torch.distributed as dist
    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import dp
    group = object()
    monkeypatch.setattr(dp, "resolve_group", lambda g: group if g is not None else None)
    monkeypatch.setattr(dist, "get_world_size", lambda g=None: 8)

    def no_exchange(*a, **k):
        raise AssertionError("allgather_slots_ called")
    monkeypatch.setattr(dp, "allgather_slots_", no_exchange)
    for fn in (pn.patchnce_with_head_global_negatives, pn.head_global_negatives_loss_and_grads):
        netF = pn.PatchSampleF(use_mlp=True, nc=128)
        big = [torch.randn(9, 8, 32, 32)]                       # 8 ranks x 9 images x 1024 keys > 65536
        with pytest.raises(RuntimeError, match=r"global batch=72 \(8 ranks x 9\)"):
            fn(netF, big, big, num_patches=1024)
        inside = [torch.randn(8, 8, 32, 32)]                    # 64 x 1024 keys: the per-rank shape alone would pass
        with pytest.raises(RuntimeError, match="tensor-core"):
            fn(netF, inside, inside, num_patches=1024, math="simt_f32")
        with pytest.raises(RuntimeError, match="nc must be 128 or 256"):
            fn(pn.PatchSampleF(use_mlp=True, nc=64), inside, inside)
        assert not netF.mlp_init


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


B5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]


@pytest.mark.parametrize("nc,bl,world", [(256, 32, 2), (256, 8, 8), (128, 16, 4)])
def test_workspace_is_the_head_minibatch_prefix_then_maps_route_slots(lib, nc, bl, world):
    n, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    assert lib.pnce_head_mb_shard_workspace_bytes(_layers(B5, 256), 5, bl, world, nc, ctypes.byref(n), ctypes.byref(off),
                                                  ctypes.byref(sb)) == 0
    prefix = ctypes.c_size_t(0)
    assert lib.pnce_head_mb_workspace_bytes(_layers(B5, 256), 5, bl, nc, ctypes.byref(prefix)) == 0
    assert off.value == prefix.value                            # what pnce_head_bwd_ex reads, unchanged
    virtual = _layers([(nc, h, w) for _, h, w in B5], 256)      # the head's output: C = nc
    mn, moff, msb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    assert lib.pnce_mb_shard_workspace_bytes(virtual, 5, bl, world, ctypes.byref(mn), ctypes.byref(moff),
                                             ctypes.byref(msb)) == 0
    assert sb.value == msb.value and sb.value % 256 == 0        # the slot format of the maps route
    assert n.value == off.value + world * sb.value


def test_c_entry_points_reject_bad_arguments_without_touching_cuda(lib):
    from gan_variant_research_b200 import _lib
    n, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)

    def wsb(layers=None, nl=5, bl=8, world=8, nc=256, out=True):
        layers = _layers(B5, 256) if layers is None else layers
        ptrs = (ctypes.byref(n), ctypes.byref(off), ctypes.byref(sb)) if out else (None, None, None)
        return lib.pnce_head_mb_shard_workspace_bytes(layers, nl, bl, world, nc, *ptrs)

    assert wsb() == 0                                           # 64 x 256 keys
    assert wsb(bl=33) == -2                                     # 8 x 33 x 256 keys > 65536: the GLOBAL batch
    assert wsb(nc=64) == -2
    assert wsb(world=0) == -1
    assert wsb(bl=0) == -1
    assert wsb(out=False) == -1

    buf = ctypes.create_string_buffer(4 << 20)                  # host memory, only its address is used: 256-aligned below
    ws = (ctypes.addressof(buf) + 255) // 256 * 256
    ids = (ctypes.c_int64 * 64)()
    fake = ws + 4096                                            # aligned non-NULL map pointers (never dereferenced)
    lay = _layers([(16, 8, 8)], 64)
    lay[0].src = lay[0].tgt = fake
    lay[0].ids = ctypes.addressof(ids)
    heads = (_lib.PnceHead * 1)()
    heads[0].w1 = heads[0].b1 = heads[0].w2 = heads[0].b2 = fake
    out = ctypes.c_float(0)
    f32, nchw, x3 = _lib.PNCE_F32, _lib.LAYOUT_NCHW, _lib.MATH_TC_BF16X3
    need = ctypes.c_size_t(0)
    assert lib.pnce_head_mb_shard_workspace_bytes(lay, 1, 2, 4, 128, ctypes.byref(need), ctypes.byref(off),
                                                  ctypes.byref(sb)) == 0
    assert need.value < (4 << 20) - 256

    def keys(layers=lay, hd=heads, bl=2, dtype=f32, layout=nchw, nc=128, world=4, rank=1, math=x3, w=ws, wb=need.value):
        return lib.pnce_head_mb_shard_keys(layers, hd, 1, bl, dtype, layout, nc, world, rank, math, w, wb, None, None)

    def loss(layers=lay, hd=heads, bl=2, dtype=f32, layout=nchw, nc=128, world=4, rank=1, tau=0.07, math=x3, w=ws,
             wb=need.value, lo=ctypes.addressof(out)):
        return lib.pnce_head_mb_shard_loss(layers, hd, 1, bl, dtype, layout, nc, world, rank, tau, math, w, wb, lo, None,
                                           None)

    for fn in (keys, loss):
        assert fn(world=0, rank=0) == -1
        assert fn(rank=4) == -1 and fn(rank=-1) == -1
        assert fn(dtype=7) == -1 and fn(layout=5) == -1 and fn(math=9) == -1
        assert fn(hd=None) == -1
        nulls = (_lib.PnceHead * 1)()
        nulls[0].w1 = nulls[0].b1 = nulls[0].w2 = fake             # b2 missing
        assert fn(hd=nulls) == -1
        assert fn(math=_lib.MATH_SIMT_F32) == -2
        assert fn(nc=64) == -2
        big = _layers([(16, 32, 32)], 1024)
        big[0].src = big[0].tgt = fake
        big[0].ids = ctypes.addressof(ids)
        assert fn(layers=big, bl=9, world=8, rank=0) == -2        # 72 x 1024 keys: the global batch is outside
        assert fn(w=None) == -3
        assert fn(w=ws + 128) == -3                                # misaligned
        assert fn(wb=need.value - 1) == -3                         # short
        assert fn(bl=0) == -1
    assert loss(lo=None) == -1
    assert loss(tau=0.0) == -1
