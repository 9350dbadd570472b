"""The netF head with minibatch negatives (patchnce_with_head_minibatch) without a GPU: the float64 oracle equals the
per-image head oracle at B = 1 and an independent autograd expression, and grows with the batch; the guard zeroes one
layer; the new Python entry points have the documented signatures and refuse out-of-envelope calls before touching a
device; the new C entry points reject bad arguments before any CUDA call."""
import ctypes
import inspect

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import head_minibatch_oracle as hmo
from oracle import patchnce_oracle as orc

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


def _loss_and_grads(fn, src, tgt, ids, heads, tau=0.07):
    t = [x.clone().requires_grad_() for x in tgt]
    h = [tuple(w.clone().requires_grad_() for w in hd) for hd in heads]
    loss = fn(src, t, ids, h, tau)
    loss.backward()
    zero = lambda x, g: torch.zeros_like(x) if g is None else g
    return loss.item(), [zero(x, x.grad) for x in t], [[zero(w, w.grad) for w in hd] for hd in h]


def _independent(src, tgt, ids, heads, tau):
    """Third expression: per layer the (B, P, nc) head output as one (1, B*P, nc) batch, ``q.view(1, -1, nc) @
    k.view(1, -1, nc).mT / tau``, F.linear for the two layers, no guard."""
    total = 0.0
    for s, t, i, (w1, b1, w2, b2) in zip(src, tgt, ids, heads):
        b, c = s.shape[:2]

        def head(x):
            rows = x.reshape(b, c, -1).transpose(1, 2)[:, i, :]                   # (B, P, C)
            return F.normalize(F.linear(F.relu(F.linear(rows, w1, b1)), w2, b2), dim=2, eps=orc.NORM_EPS)

        nc = w2.shape[0]
        k, q = head(s).detach(), head(t)
        z = (q.view(1, -1, nc) @ k.view(1, -1, nc).mT / tau).clamp(-orc.LOGIT_CLAMP, orc.LOGIT_CLAMP)[0]
        total = total + F.cross_entropy(z, torch.arange(z.shape[0]))
    return total / len(src)


@pytest.mark.parametrize("nc", [128, 256])
def test_one_image_equals_the_per_image_head_oracle(nc):
    src, tgt, ids, heads = _problem(1, 1, nc)
    la, ga, ha = _loss_and_grads(hmo.head_minibatch_loss, src, tgt, ids, heads)
    lb, gb, hb = _loss_and_grads(orc.patchnce_head_loss_torch, src, tgt, ids, heads)
    assert la == pytest.approx(lb, rel=1e-13)
    for a, b in zip(ga + sum(ha, []), gb + sum(hb, [])):
        torch.testing.assert_close(a, b, rtol=1e-11, atol=1e-15)


@pytest.mark.parametrize("b,nc", [(3, 128), (5, 256)])
def test_oracle_equals_an_independent_expression(b, nc):
    src, tgt, ids, heads = _problem(b, b, nc)
    la, ga, ha = _loss_and_grads(hmo.head_minibatch_loss, src, tgt, ids, heads)
    lb, gb, hb = _loss_and_grads(_independent, src, tgt, ids, heads)
    assert la == pytest.approx(lb, rel=1e-12)
    for a, b_ in zip(ga + sum(ha, []), gb + sum(hb, [])):
        torch.testing.assert_close(a, b_, rtol=1e-10, atol=1e-14)
    # keys carry no gradient and the head learns through q only: d tgt is zero off the sampled positions
    for g, i in zip(ga, ids):
        off = torch.ones(g.shape[2] * g.shape[3], dtype=torch.bool)
        off[i] = False
        assert (g.reshape(g.shape[0], g.shape[1], -1)[:, :, off] == 0).all()


def test_more_images_give_a_larger_loss_than_per_image_negatives():
    src, tgt, ids, heads = _problem(7, 4, 128)
    lm = hmo.head_minibatch_loss(src, tgt, ids, heads).item()
    lp = orc.patchnce_head_loss_torch(src, tgt, ids, heads).item()
    assert lm > lp                                    # more negatives, larger CE


def test_guard_zeroes_exactly_the_non_finite_layer():
    src, tgt, ids, heads = _problem(3, 3, 128)
    tgt[1][2, 5].reshape(-1)[ids[1][0]] = float("nan")    # a sampled target patch of layer 1, image 2
    warn = []
    la, ga, ha = _loss_and_grads(lambda *a: hmo.head_minibatch_loss(*a, warn=warn), src, tgt, ids, heads)
    assert warn == ["layer"]
    l0, g0, h0 = _loss_and_grads(hmo.head_minibatch_loss, src[:1], tgt[:1], ids[:1], heads[:1])
    assert la == pytest.approx(l0 / 2, rel=1e-13)        # layer 1 contributes 0 to the mean over two layers
    assert (ga[1] == 0).all() and all((w == 0).all() for w in ha[1])
    torch.testing.assert_close(ga[0], g0[0] / 2, rtol=1e-12, atol=0)


def test_signatures_and_defaults():
    import gan_variant_research_b200 as pn
    assert "patchnce_with_head_minibatch" in pn.__all__ and "head_minibatch_loss_and_grads" in pn.__all__
    a = inspect.signature(pn.patchnce_with_head_minibatch).parameters
    assert list(a) == ["netF", "src_feats", "tgt_feats", "temperature", "num_patches", "patch_ids", "math", "dp_group"]
    b = inspect.signature(pn.head_minibatch_loss_and_grads).parameters
    assert list(b) == ["netF", "src_feats", "tgt_feats", "temperature", "num_patches", "patch_ids", "math",
                       "grad_output", "dp_group"]
    for p in (a, b):
        assert p["temperature"].default == 0.07 and p["num_patches"].default == 256
        assert p["patch_ids"].default is None and p["math"].default is None and p["dp_group"].default is None
    assert b["grad_output"].default is None
    # the per-image head keeps its signature; the new names are where minibatch negatives live
    for fn in (pn.patchnce_with_head, pn.head_loss_and_grads):
        assert "head_minibatch" in fn.__doc__ or "patchnce_with_head_minibatch" in fn.__doc__


def test_out_of_envelope_calls_raise_before_touching_a_device():
    """CPU tensors: every error below is raised before the maps are looked at (they would fail with "no CPU fallback")."""
    import gan_variant_research_b200 as pn
    for fn in (pn.patchnce_with_head_minibatch, pn.head_minibatch_loss_and_grads):
        netF = pn.PatchSampleF(use_mlp=True, nc=128)
        src = [torch.randn(4, 64, 16, 16)]
        with pytest.raises(RuntimeError, match="tensor-core"):
            fn(netF, src, src, math="simt_f32")
        big = [torch.randn(65, 8, 32, 32)]                # 65 * 1024 keys > 65536
        with pytest.raises(RuntimeError, match="65536"):
            fn(netF, big, big, num_patches=1024)
        with pytest.raises(RuntimeError, match="nc must be 128 or 256"):
            fn(pn.PatchSampleF(use_mlp=True, nc=64), src, src)
        assert not netF.mlp_init                          # nothing was built either


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
    n, per_image = ctypes.c_size_t(0), ctypes.c_size_t(0)
    b5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
    assert lib.pnce_head_mb_workspace_bytes(_layers(b5, 256), 5, 64, 256, ctypes.byref(n)) == 0
    assert lib.pnce_head_workspace_bytes(_layers(b5, 256), 5, 64, 256, ctypes.byref(per_image)) == 0
    assert per_image.value < n.value < 1.05 * per_image.value   # the per-image head's layout, then the raw patches' sums
    assert lib.pnce_head_mb_workspace_bytes(_layers(b5, 256), 5, 256, 128, ctypes.byref(n)) == 0      # 256 * 256 keys
    assert lib.pnce_head_mb_workspace_bytes(_layers(b5, 256), 5, 257, 128, ctypes.byref(n)) == -2     # B * Ppad > 65536
    assert lib.pnce_head_mb_workspace_bytes(_layers(b5, 256), 5, 64, 64, ctypes.byref(n)) == -2       # nc = 64
    assert lib.pnce_head_mb_workspace_bytes(_layers([(512, 8, 8)], 64), 1, 2, 128, ctypes.byref(n)) == -2   # C > 256
    assert lib.pnce_head_mb_workspace_bytes(_layers([(64, 40, 40)], 1100), 1, 2, 128, ctypes.byref(n)) == -2  # P > 1024
    assert lib.pnce_head_mb_workspace_bytes(_layers(b5, 256), 5, 0, 128, ctypes.byref(n)) == -1
    assert lib.pnce_head_mb_workspace_bytes(None, 1, 1, 128, ctypes.byref(n)) == -1
    assert lib.pnce_head_mb_workspace_bytes(_layers(b5, 256), 5, 2, 128, None) == -1

    buf = ctypes.create_string_buffer(1 << 20)              # host memory, only its address is used: 256-aligned below
    ws = (ctypes.addressof(buf) + 255) // 256 * 256
    ids = (ctypes.c_int64 * 64)()
    fake = ws + 4096                                        # aligned non-NULL map pointers (never dereferenced)
    lay = _layers([(16, 8, 8)], 64)
    lay[0].src = lay[0].tgt = fake
    lay[0].ids = ctypes.addressof(ids)
    heads = (_lib.PnceHead * 1)()
    heads[0].w1 = heads[0].b1 = heads[0].w2 = heads[0].b2 = fake
    out = ctypes.c_float(0)
    f32, nchw, x3 = _lib.PNCE_F32, _lib.LAYOUT_NCHW, _lib.MATH_TC_BF16X3

    def fwd(layers=lay, hd=heads, batch=2, nc=128, math=x3, w=ws, wb=1 << 16, loss=ctypes.addressof(out)):
        return lib.pnce_head_mb_fwd(layers, hd, 1, batch, f32, nchw, nc, 0.07, math, w, wb, loss, None, None)

    assert fwd(hd=None) == -1                               # NULL heads
    assert fwd(nc=64) == -2
    assert fwd(math=_lib.MATH_SIMT_F32) == -2
    assert fwd(hd=None, math=_lib.MATH_SIMT_F32) == -2      # simt_f32 is refused first
    big = _layers([(16, 32, 32)], 1024)
    big[0].src = big[0].tgt = fake
    big[0].ids = ctypes.addressof(ids)
    assert fwd(layers=big, batch=65) == -2                  # 65 * 1024 keys
    assert fwd(w=None) == -3                                # NULL workspace
    need = ctypes.c_size_t(0)
    assert lib.pnce_head_mb_workspace_bytes(lay, 1, 2, 128, ctypes.byref(need)) == 0
    assert fwd(wb=need.value - 1) == -3                     # short workspace
    assert fwd(loss=None) == -1
    assert fwd(batch=0) == -1
