"""Global negatives on the row route (``rows_patchnce_global_negatives``) without a GPU: the float64 shard oracle equals
an autograd restatement at W = 1, reproduces the one-group loss and gradient for W in {2, 4}, and guards globally; the
Python entry point has the documented signature and raises its envelope errors before any collective; the
``PatchNCELoss`` row route still refuses ``negatives_group``; the new C entry points reject bad arguments before any CUDA
call and lay out the workspace as documented."""
import ctypes
import inspect

import numpy as np
import pytest
import torch

import rows_global_negatives_oracle as rgo


def _rows(seed, n, d, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    k = torch.nn.functional.normalize(torch.randn(n, d, generator=g, dtype=torch.float64), dim=1)
    q = torch.nn.functional.normalize(0.6 * k + 0.8 * torch.randn(n, d, generator=g, dtype=torch.float64), dim=1)
    return (scale * q).numpy(), k.numpy()


def _autograd(q, k, tau):
    """CE of clamp(q @ k.T / tau, +-50) with diagonal labels, by autograd, with the group guard."""
    qt = torch.from_numpy(q).clone().requires_grad_()
    kt = torch.from_numpy(k)
    z = torch.clamp(qt @ kt.T / tau, -50.0, 50.0)
    loss = torch.nn.functional.cross_entropy(z, torch.arange(q.shape[0]))
    if not (torch.isfinite(loss) and np.isfinite(q).all() and np.isfinite(k).all()):
        return 0.0, np.zeros_like(q)
    loss.backward()
    return loss.item(), qt.grad.numpy()


@pytest.mark.parametrize("tau", [0.07, 0.01])
def test_one_rank_is_the_autograd_restatement(tau):
    q, k = _rows(1, 96, 40, scale=1.0 if tau > 0.05 else 3.0)      # tau = 0.01 (x3 rows): the clamp binds
    la, ga = _autograd(q, k, tau)
    lo, go = rgo.layer_loss_and_grad_rows_shard(q, k, tau, 1, 0)
    assert lo == pytest.approx(la, rel=1e-12)
    np.testing.assert_allclose(go, ga, rtol=1e-10, atol=1e-14)


@pytest.mark.parametrize("tau", [0.07, 0.01])
@pytest.mark.parametrize("world", [2, 4])
def test_shards_reproduce_the_one_group_loss(world, tau):
    bl, p = 2, 24
    q, k = _rows(world, world * bl * p, 40, scale=1.0 if tau > 0.05 else 3.0)
    full, gfull = rgo.layer_loss_and_grad_rows_shard(q, k, tau, 1, 0)
    shards = [rgo.layer_loss_and_grad_rows_shard(q, k, tau, world, r) for r in range(world)]
    assert np.mean([l for l, _ in shards]) == pytest.approx(full, rel=1e-12)
    nl = bl * p
    for r, (_, g) in enumerate(shards):
        np.testing.assert_allclose(g / world, gfull[r * nl:(r + 1) * nl], rtol=1e-10,
                                   atol=1e-12 * np.abs(gfull).max())


@pytest.mark.parametrize("where", ["query", "key"])
def test_a_non_finite_row_on_one_rank_guards_every_rank(where):
    world, nl = 2, 32
    q, k = _rows(7, world * nl, 16)
    (q if where == "query" else k)[nl + 5, 3] = np.nan          # a row of rank 1
    assert rgo.layer_loss_and_grad_rows_shard(q, k, 0.07, 1, 0)[0] == 0.0
    for r in range(world):
        loss, g = rgo.layer_loss_and_grad_rows_shard(q, k, 0.07, world, r)
        assert loss == 0.0 and (g == 0).all()
    q[nl + 5, 3] = np.inf
    assert all(rgo.layer_loss_and_grad_rows_shard(q, k, 0.07, world, r)[0] == 0.0 for r in range(world))


def test_signature_and_exports():
    import gan_variant_research_b200 as pn
    assert "rows_patchnce_global_negatives" in pn.__all__
    p = inspect.signature(pn.rows_patchnce_global_negatives).parameters
    assert list(p) == ["feat_q", "feat_k", "temperature", "num_patches", "batch_size", "math", "negatives_group"]
    assert p["temperature"].default == 0.07 and p["num_patches"].default == 256
    assert p["batch_size"].default is None and p["math"].default is None and p["negatives_group"].default is True


def test_the_patchnce_loss_row_route_still_refuses_negatives_group():
    import gan_variant_research_b200 as pn
    crit = pn.PatchNCELoss(nce_includes_all_negatives_from_minibatch=True, negatives_group=True)
    rows = torch.zeros(32, 8)
    for a in (rows, [rows]):
        with pytest.raises(RuntimeError, match="row route.*rows_patchnce_global_negatives"):
            crit(a, a)


def test_global_envelope_raises_before_any_collective(monkeypatch):
    """Eight ranks (resolve_group / get_world_size patched), CPU rows with the device check patched out: each envelope
    error is raised before the key exchange and before the library is called."""
    import torch.distributed as dist
    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import dp, patchnce
    group = object()
    monkeypatch.setattr(dp, "resolve_group", lambda g: group if g is not None else None)
    monkeypatch.setattr(dist, "get_world_size", lambda g=None: 8)
    monkeypatch.setattr(patchnce, "_require_cuda", lambda t, what: None)

    def never(*a, **k):
        raise AssertionError("collective or library call reached")
    monkeypatch.setattr(dp, "allgather_slots_", never)
    monkeypatch.setattr(patchnce._RowsLossMultiFn, "apply", never)
    fn = pn.rows_patchnce_global_negatives
    inside = torch.zeros(8 * 256, 64)                           # 8 ranks x 8 images x 256 keys = 16384: inside
    with pytest.raises(AssertionError, match="reached"):
        fn(inside, inside)                                      # the guard of the test itself
    big = torch.zeros(33 * 256, 64)                             # 8 x 33 x 256 keys > 65536; 33 x 256 alone would pass
    with pytest.raises(RuntimeError, match=r"global batch=264 \(8 ranks x 33\)"):
        fn(big, big)
    with pytest.raises(RuntimeError, match="tensor-core"):
        fn(inside, inside, math="simt_f32")
    with pytest.raises(RuntimeError, match="P <= 256"):
        fn(torch.zeros(2 * 257, 64), torch.zeros(2 * 257, 64), num_patches=257)
    with pytest.raises(RuntimeError, match="C <= 256"):
        fn(torch.zeros(512, 257), torch.zeros(512, 257))
    with pytest.raises(RuntimeError, match="one batch size"):
        fn([inside, torch.zeros(4 * 256, 64)], [inside, torch.zeros(4 * 256, 64)])
    with pytest.raises(RuntimeError, match="at most 8"):
        fn([inside] * 9, [inside] * 9)


@pytest.fixture(scope="module")
def lib():
    from gan_variant_research_b200 import _lib, build
    build.build()
    return _lib.load()


def _rows_arr(shapes, fake=0, dq=None):
    from gan_variant_research_b200 import _lib
    arr = (_lib.PnceRows * len(shapes))()
    for i, (p, d) in enumerate(shapes):
        arr[i].P, arr[i].D = p, d
        if fake:                                                # aligned, never dereferenced: the calls stop before CUDA
            arr[i].q, arr[i].k, arr[i].dq = fake, fake + (1 << 20), fake + (2 << 20) if dq is None else dq
    return arr


B5_ROWS = [(256, 64), (256, 256), (256, 256), (256, 128), (256, 64)]


@pytest.mark.parametrize("shapes,bl,world", [(B5_ROWS, 32, 2), (B5_ROWS, 8, 8), ([(200, 40), (256, 256)], 3, 4)])
def test_workspace_is_the_row_minibatch_prefix_then_maps_route_slots(lib, shapes, bl, world):
    n, off, sb, pre = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    assert lib.pnce_rows_mb_shard_workspace_bytes(_rows_arr(shapes), len(shapes), bl, world, ctypes.byref(n),
                                                  ctypes.byref(off), ctypes.byref(sb)) == 0
    assert lib.pnce_rows_mb_workspace_bytes(_rows_arr(shapes), len(shapes), bl, ctypes.byref(pre)) == 0
    assert off.value == pre.value and sb.value % 256 == 0 and n.value == off.value + world * sb.value
    # a slot: the flags, then per layer K hi, K2 hi, the key sums of squares, K lo, K2 lo of bl images (C = D)
    keys = 0
    for p, d in shapes:
        ppad, cp = (p + 127) // 128 * 128, (d + 31) // 32 * 32
        keys += bl * ppad * cp * 2 * 4 + bl * (cp // 32) * ppad * 4
    assert keys <= sb.value <= keys + 256 * (1 + 5 * len(shapes))


def test_c_entry_points_reject_bad_arguments_without_touching_cuda(lib):
    from gan_variant_research_b200 import _lib
    n, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    ws_q = lambda shapes, bl, world: lib.pnce_rows_mb_shard_workspace_bytes(
        _rows_arr(shapes), len(shapes), bl, world, ctypes.byref(n), ctypes.byref(off), ctypes.byref(sb))
    assert ws_q(B5_ROWS, 64, 4) == 0                                        # 4 x 64 x 256 = 65536 keys: inside
    assert ws_q(B5_ROWS, 64, 5) == -2                                       # global keys > 65536
    assert ws_q([(257, 64)], 2, 2) == -2 and ws_q([(256, 257)], 2, 2) == -2  # P = 257, D = 257
    assert ws_q(B5_ROWS, 8, 0) == -1 and ws_q(B5_ROWS, 0, 2) == -1 and ws_q([(0, 64)], 2, 2) == -1
    assert ws_q([(64, 64)] * 9, 2, 2) == -1                                  # more than PNCE_MAX_LAYERS
    assert lib.pnce_rows_mb_shard_workspace_bytes(_rows_arr(B5_ROWS), 5, 8, 2, None, ctypes.byref(off),
                                                  ctypes.byref(sb)) == -1
    shapes = [(100, 40)]
    assert ws_q(shapes, 2, 4) == 0
    need = n.value
    base = 1 << 30                                                          # aligned, never touched
    rows = _rows_arr(shapes, fake=base + (64 << 20))
    tc, loss = _lib.MATH_TC_BF16X3, ctypes.c_float(0)

    def keys(world=4, rank=1, math=tc, ws=base, nbytes=need, r=rows):
        return lib.pnce_rows_mb_shard_keys(r, 1, 2, world, rank, math, ws, nbytes, None)

    def loss_call(world=4, rank=1, math=tc, ws=base, nbytes=need, r=rows, out=ctypes.addressof(loss), tau=0.07):
        return lib.pnce_rows_mb_shard_loss(r, 1, 2, world, rank, tau, math, ws, nbytes, out, None, None)

    for call in (keys, loss_call):
        assert call(world=0, rank=0) == -1                                  # world < 1
        assert call(rank=4) == -1 and call(rank=-1) == -1                    # rank outside [0, world)
        assert call(math=7) == -1
        assert call(math=_lib.MATH_SIMT_F32) == -2
        assert call(r=_rows_arr([(257, 40)], fake=base)) == -2               # P = 257
        assert call(r=_rows_arr([(100, 257)], fake=base)) == -2              # D = 257
        assert call(world=64 * 128) == -2                                    # 2 x 8192 x 128 keys > 65536
        assert call(ws=None) == -3 and call(ws=base + 128) == -3             # NULL / misaligned workspace
        assert call(nbytes=need - 1) == -3                                   # short workspace
    assert keys(r=_rows_arr(shapes)) == -1                                   # NULL q / k
    assert loss_call(out=None) == -1 and loss_call(tau=0.0) == -1
    assert loss_call(r=_rows_arr(shapes, fake=base, dq=0)) == -1             # NULL dq
    assert loss_call(r=_rows_arr(shapes, fake=base, dq=base + (3 << 20) + 16)) == -5   # dq not 32-byte aligned
