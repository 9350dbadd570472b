"""The per-image PatchNCE loss and the fused netF head against float64 at the sizes bench.py runs, down to bench.py's own
timed step.

The reference is restated in float64 on the GATHERED rows only (never on a dense map): per layer the rows k = src[:, :, ids]
and q = tgt[:, :, ids] as (B, P, C), the per-image loss of patchnce_cut.py:83-103 batched with bmm, d loss / d q from
autograd, and the row gradients index_add-ed into (B, C, U) at the U unique sampled positions (ids are drawn with
replacement: duplicates accumulate).  With a head, oracle.patchnce_oracle.head_forward_torch runs on both sides' raw rows
(the k side detached) and autograd gives the head gradients.

The checker compares one (image, layer) block at a time, each against its own largest entry: under one global max a
single wrong image of 64 hides, and a dead post-ReLU patch swamps the rest (test_parity_gpu._assert_rows_close).  Every
entry of the dense gradient off the sampled positions must be exactly 0 (counted on the device) and the NaN patterns must
coincide.  tests/test_benchmarked_sizes.py pins both on the CPU."""
import gc
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import bench
from oracle.patchnce_oracle import LOGIT_CLAMP, NORM_EPS, head_forward_torch
from test_patchnce_with_head_minibatch_gpu import _head_params, _maps as _quantised_maps, _netf

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gan_variant_research_b200", "csrc")
B5 = [(c, h, w) for c, h, w, _ in bench.LAYER_SETS["b5"]]
CFG4 = [(c, 2 * h, 2 * w) for c, h, w in B5]             # BASELINE config 4: 512^2 images, P = 1024
# (loss relative, gradient max-abs over the block's own max-abs).  The suite holds tc_bf16x3 / simt_f32 to 2e-4 of a
# global max and 5x that per row on the generator maps (test_parity_gpu.MATH_TOL).  tc_bf16 rounds the operands once
# to bf16 (2^-9) and 1 / tau = 14 amplifies that in the logits; the suite's 3e-2 is of a global max on small maps.  One
# block at a time the worst of B5's 320 blocks at B = 64 reaches 3.06e-2 (NVIDIA B200, 1000 W), in a layer where the
# same maps give 9e-5 with tc_bf16x3 and 8e-6 with simt_f32: bf16 rounding, not a wrong index, hence 5e-2 per block.
TOL = {"tc_bf16x3": (2e-5, 5e-4), "simt_f32": (2e-5, 5e-4), "tc_bf16": (2e-3, 5e-2)}
# the head (test_patchnce_with_head_minibatch_gpu.TOL): loss, and d tgt per block / head gradients per tensor
HEAD_TOL = {"tc_bf16x3": (1e-3, 1e-3), "tc_bf16": (1e-2, 1.5e-1)}


def _src_const(path, name):
    with open(os.path.join(CSRC, path)) as f:
        return int(re.search(rf"constexpr int {name} = (\d+);", f.read()).group(1))


FOLD_MAX_CTAS = _src_const("gather_tc.cuh", "kFoldMaxCtas")
NHWC_ITEMS_PER_WARP = _src_const("nhwc.cuh", "kNhwcItemsPerWarp")


# ---- float64 restatement on gathered rows --------------------------------------------------------------------------
def _rows(x, ids):
    """The rows of a (B, C, H, W) map (any layout, any dtype) at flat positions ``ids`` as (B, P, C) float64.  Indexing
    H and W gathers straight from the map's storage: no dense copy, whatever its layout."""
    w = x.shape[3]
    return x.detach()[:, :, ids // w, ids % w].transpose(1, 2).double()


def restate(src, tgt, ids, tau, heads=None):
    """patchnce_cut.py:83-103 (per-image negatives) in float64 on the rows at ``ids``, backward by autograd.

    ``heads``: per layer (w1, b1, w2, b2) of a netF head, applied to both sides' raw rows before the normalisation (k
    detached), as patchnce_oracle.patchnce_head_loss_torch.  Returns ``(loss, [(positions (U,), d tgt (B, C, U))] per
    layer, [[dw1, db1, dw2, db2]] per layer or None)``; positions are the sorted unique ids."""
    qs = [_rows(t, i).requires_grad_() for t, i in zip(tgt, ids)]
    hp = None if heads is None else [[p.detach().double().requires_grad_() for p in h] for h in heads]
    total = 0.0
    for l, (s, q, i) in enumerate(zip(src, qs, ids)):
        k = _rows(s, i)
        b, p, c = k.shape
        if hp is None:
            kh, qh = F.normalize(k, dim=2, eps=NORM_EPS), F.normalize(q, dim=2, eps=NORM_EPS)
        else:
            kh = head_forward_torch(k.reshape(-1, c), *hp[l]).reshape(b, p, -1).detach()
            qh = head_forward_torch(q.reshape(-1, c), *hp[l]).reshape(b, p, -1)
        z = (torch.bmm(qh, kh.transpose(1, 2)) / tau).clamp(-LOGIT_CLAMP, LOGIT_CLAMP)
        ce = F.cross_entropy(z.reshape(b * p, p), torch.arange(p, device=z.device).repeat(b), reduction="none")
        per_image = ce.view(b, p).mean(1)
        per_image = torch.where(torch.isfinite(per_image), per_image, torch.zeros_like(per_image))    # :97-99
        total = total + per_image.mean()
    total = total / len(src)
    leaves = qs + ([] if hp is None else sum(hp, []))
    grads = torch.autograd.grad(total, leaves)
    out = []
    for q, i, g in zip(qs, ids, grads):
        pos, inv = torch.unique(i, return_inverse=True)
        acc = torch.zeros(q.shape[0], q.shape[2], pos.numel(), dtype=torch.float64, device=q.device)
        out.append((pos, acc.index_add_(2, inv, g.transpose(1, 2))))
    n = len(src)
    head_grads = None if hp is None else [list(grads[n + 4 * l:n + 4 * l + 4]) for l in range(n)]
    return total.item(), out, head_grads


# ---- the checker ---------------------------------------------------------------------------------------------------
def _ulp(want, dtype):
    """One unit in the last place of |want| on ``dtype``'s grid, subnormals included: the rounding of a gradient stored
    in a half dtype.  0 for float32, whose error is what the tolerance measures."""
    if dtype == torch.float32:
        return torch.zeros_like(want)
    fi = torch.finfo(dtype)
    return torch.exp2(torch.floor(torch.log2(want.abs().clamp(min=fi.smallest_normal)))) * fi.eps


def excess(got, want, dtype=torch.float32, allow=None):
    """|got - want| beyond the rounding of the stored value: half an ulp of ``got`` in ``dtype`` (the stored value is the
    kernel's fp32 value rounded to nearest, whose ulp is at most ``got``'s), and beyond ``allow`` (an absolute allowance
    per entry, same shape).  What is left bounds the kernel's fp32 error from below."""
    d = (got - want).abs() - 0.5 * _ulp(got, dtype)
    return (d if allow is None else d - allow).clamp(min=0.0)


def block_errors(got, want, dtype=torch.float32, allow=None):
    """(B, C, N) gradient columns against the float64 reference: per image, max ``excess`` over that image's own max
    |want|.  NaN patterns must coincide."""
    got = got.double()
    nan_w = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan_w), "NaN pattern differs"
    got, want = got.masked_fill(nan_w, 0.0), want.masked_fill(nan_w, 0.0)
    return excess(got, want, dtype, allow).amax(dim=(1, 2)) / want.abs().amax(dim=(1, 2)).clamp(min=1e-30)


def off_sample_nonzeros(grad, ids):
    """Entries of the dense (B, C, H, W) gradient that are not exactly 0 away from the sampled positions, counted on
    the gradient's device with a position mask (NaN and Inf count)."""
    h, w = grad.shape[2:]
    off = torch.ones(h * w, dtype=torch.bool, device=grad.device)
    off[ids] = False
    return int(((grad != 0) & off.view(1, 1, h, w)).sum())


def check_grads(grads, ref, ids, tol, what):
    """Dense kernel gradients against ``restate``'s columns, one (image, layer) block at a time; -> the largest block
    error."""
    worst = 0.0
    for l, (g, (pos, want), i) in enumerate(zip(grads, ref, ids)):
        n_off = off_sample_nonzeros(g, i)
        assert n_off == 0, f"{what} layer {l}: {n_off} non-zero entries off the sampled positions"
        w = g.shape[3]
        err = block_errors(g[:, :, pos // w, pos % w], want, g.dtype)
        e, b = err.max().item(), int(err.argmax())
        assert e <= tol, f"{what} layer {l} image {b}: block error {e:.3e} > {tol}"
        worst = max(worst, e)
    return worst


def check_head_grads(got, want, tol, what, allow=None):
    """The four head gradients of every layer, each as max-abs error over its own max-abs; -> the largest.  ``allow``:
    per layer an absolute allowance for (dW1, db1) (``relu_flip_allowance``)."""
    worst = 0.0
    for l, (gs, ws) in enumerate(zip(got, want)):
        al = (None, None) if allow is None else allow[l]
        for name, g, r, a in zip(("W1", "b1", "W2", "b2"), gs, ws, (*al, None, None)):
            e = (excess(g.double(), r, allow=a).max() / r.abs().max().clamp(min=1e-30)).item()
            assert e <= tol, f"{what} d{name} layer {l}: error {e:.3e} > {tol}"
            worst = max(worst, e)
    return worst


def loss_error(got, want, tol, what):
    e = abs(got - want) / abs(want)
    assert e <= tol, f"{what}: loss {got!r} vs {want!r}, relative error {e:.3e} > {tol}"
    return e


# ---- dispatch restated from csrc/pnce_api.cu -------------------------------------------------------------------------
def gather_tc_ctas(shapes, p, b):
    """pnce_api.cu gather_tc_ctas: NCHW gather CTAs of both sides, one per (side, image, 256 patch slots, 32 channels)."""
    return sum(2 * b * (((p + 127) // 128 * 128 + 255) // 256) * ((c + 31) // 32) for c, _, _ in shapes)


def gather_nhwc_ctas(shapes, p, b):
    """pnce_api.cu gather_nhwc_ctas: channels-last warp items (side, image, 8 slots, 32 channels), 8 warps per CTA."""
    per = 8 * NHWC_ITEMS_PER_WARP
    return sum((2 * b * ((p + 127) // 128 * 128 >> 3) * ((c + 31) // 32) + per - 1) // per for c, _, _ in shapes)


def map_bytes(shapes, b, elem):
    """patchnce._ShapePlan.big: from patchnce._SIDE_STREAM_MIN_BYTES on, the ids are drawn and sorted ahead on a side
    stream (pnce_plan_ids_draw, k_prep) and the forward gathers with the unfolded kernel."""
    return 2 * elem * sum(b * c * h * w for c, h, w in shapes)


def loss_schedule(sm, layers, b):
    """launch_loss_tc (P <= 256 everywhere): ``layers`` = [(C, P)] -> (items, grid, light items, rot).  k_loss_tc_p runs
    min(items, SMs) CTAs over the items B * Ppad / 128 of every layer, heaviest layer first, rotated by ``rot`` so that
    a third of the CTAs starts on the lightest layer: rot = min(light, grid / 3) rounded down to even, 0 when every
    layer has the lightest channel count."""
    items = b * sum((p + 127) // 128 for _, p in layers)
    grid = min(sm, items)
    cmin = min(c for c, _ in layers)
    light = b * sum((p + 127) // 128 for c, p in layers if c == cmin)
    rot = 0 if light == items else (light if light < grid // 3 else grid // 3) & ~1
    return items, grid, light, rot


_HEAVY_C = (64, 128, 256, 96)


def schedule_case(sm, target, kind):
    """Layers [(C, H, W, P)] and a batch whose loss items are exactly ``target`` (a float: about that many), for
    ``kind`` 'below' (two channel counts, light items < grid / 3: rot taken from the light count), 'above' (two channel
    counts, light >= grid / 3: rot = grid / 3) or 'single' (one channel count: rot = 0).  One-item layers (P = 100,
    128) and two-item layers (P = 200, 256) are mixed wherever the item count allows; fewest layers first.
    -> (B, layers, schedule) or None when no batch of <= 8 layers fits."""
    best = None
    for a1 in range(9):
        for a2 in range(9 - a1):
            for h1 in range(9 - a1 - a2):
                for h2 in range(9 - a1 - a2 - h1):
                    if a1 + a2 == 0 or (kind == "single") != (h1 + h2 == 0):
                        continue
                    k = a1 + 2 * a2 + h1 + 2 * h2
                    if isinstance(target, float):
                        b = max(2, round(target / k))
                    elif target % k == 0:
                        b = target // k
                    else:
                        continue
                    cp = [(32, 100 + 28 * (j % 2)) for j in range(a1)] + [(32, 200 + 56 * (j % 2)) for j in range(a2)]
                    cp += [(_HEAVY_C[j % 4], 128 - 28 * (j % 2)) for j in range(h1)]
                    cp += [(_HEAVY_C[(j + 1) % 4], 256 - 56 * (j % 2)) for j in range(h2)]
                    sch = loss_schedule(sm, cp, b)
                    if kind == "below" and not sch[2] < sch[1] // 3 or kind == "above" and not sch[2] >= sch[1] // 3:
                        continue
                    mixed = (a1 + h1 > 0) and (a2 + h2 > 0)
                    key = (not mixed, len(cp), b < 2)
                    if best is None or key < best[0]:
                        best = (key, b, cp, sch)
    if best is None:
        return None
    _, b, cp, sch = best
    layers = [(c, 12, 12, p) if p <= 128 else (c, 20, 20, p) for c, p in cp]
    return b, layers, sch


# ---- fixtures and drivers ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pn():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gan_variant_research_b200 as m
    from gan_variant_research_b200 import _lib
    _lib.load()
    return m


def _release():
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


@pytest.fixture(autouse=True)
def _release_device_memory():
    """The B = 64 maps and their gradients hold about 10 GB in the caching allocator: hand them back after each test."""
    yield
    _release()


def _b5_maps(b, seed, dtype=torch.float32, channels_last=False, shapes=None):
    """src ~ N(0, 1), tgt = 0.6 src + 0.8 N(0, 1) (correlated positives), ReLU-ed on the post-ReLU layers of bench's b5."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    mf = torch.channels_last if channels_last else torch.contiguous_format
    src, tgt = [], []
    for (c, h, w), (_, _, _, relu) in zip(shapes or B5, bench.LAYER_SETS["b5"]):
        s = torch.randn(b, c, h, w, device="cuda", generator=g)
        t = 0.6 * s + 0.8 * torch.randn(b, c, h, w, device="cuda", generator=g)
        if relu:
            s, t = s.relu(), t.relu()
        src.append(s.to(dtype).contiguous(memory_format=mf))
        tgt.append(t.to(dtype).contiguous(memory_format=mf))
    return src, tgt


def _assert_randint_ids(fn, tgt, p, seed):
    """Runs ``fn()`` from seed ``seed`` -> its result; the ids ``fn`` returns are torch.randint's from the same
    generator state, and the generator is left where those draws leave it."""
    dev = tgt[0].device
    gen = torch.cuda.default_generators[dev.index]
    torch.manual_seed(seed)
    off0 = gen.get_offset()
    res, ids = fn()
    off1 = gen.get_offset()
    torch.manual_seed(seed)
    ref = [torch.randint(0, t.shape[2] * t.shape[3], (min(p, t.shape[2] * t.shape[3]),), device=dev) for t in tgt]
    assert gen.get_offset() - off0 == off1 - off0
    assert all(torch.equal(a, r) for a, r in zip(ids, ref))
    return res, list(ids)


def _loss_step(pn, src, tgt, math, p, seed=123):
    """PatchNCELoss.forward (ids drawn by the module) + backward -> (loss, d tgt, ids)."""
    t = [x.detach().requires_grad_() for x in tgt]

    def run():
        crit = pn.PatchNCELoss(0.07, p, math=math)
        loss = crit(src, t)
        loss.backward()
        return loss.item(), crit.last_patch_ids

    loss, ids = _assert_randint_ids(run, tgt, p, seed)
    assert pn.poll_nonfinite_warnings(block=True) == 0
    return loss, [x.grad for x in t], ids


def _per_image_case(pn, src, tgt, math, what, p=256):
    loss, grads, ids = _loss_step(pn, src, tgt, math, p)
    ltol, gtol = TOL[math]
    rl, ref, _ = restate(src, tgt, ids, 0.07)
    le = loss_error(loss, rl, ltol, what)
    ge = check_grads(grads, ref, ids, gtol, what)
    print(f"\n[{what}] loss rel err {le:.2e}, worst (image, layer) block err {ge:.2e}")
    assert all(g.dtype == src[0].dtype for g in grads)


# ---- the per-image loss at bench.py's size ---------------------------------------------------------------------------
@pytest.mark.parametrize("b,math", [(10, "tc_bf16x3"), (11, "tc_bf16x3"), (64, "tc_bf16x3"), (64, "simt_f32"),
                                    (64, "tc_bf16")])
def test_b5_nchw_fp32(pn, b, math):
    """NCHW fp32 b5 maps, P = 256, tau = 0.07, ids drawn by PatchNCELoss.forward.
    - B = 10 / 11 straddle the id-prep fold: gather_tc_ctas is 480 <= kFoldMaxCtas (k_gather_tc_fold sorts the ids
      itself) and 528 above it (k_prep, then k_gather_tc); both below _SIDE_STREAM_MIN_BYTES, so the fold is decided
      by the CTA count alone (pnce_api.cu forward_tc, gather_tc_folds).
    - B = 64 is bench.py's headline step: pnce_plan_ids_draw (k_prep on the side stream), k_gather_tc, k_loss_tc_p
      over 640 items on one CTA per SM (rot = grid / 3 rounded to even: 48 on 148 SMs), k_dense_flat over 3.2 GB of
      compressible gradient.  simt_f32 runs the CUDA-core kernels (loss_simt.cuh) at the same size, tc_bf16 the
      single-pass bf16 tensor-core math."""
    from gan_variant_research_b200 import patchnce as pmod
    if b in (10, 11):
        assert (gather_tc_ctas(B5, 256, b) <= FOLD_MAX_CTAS) == (b == 10)
        assert map_bytes(B5, b, 4) < pmod._SIDE_STREAM_MIN_BYTES
    else:
        assert map_bytes(B5, b, 4) >= pmod._SIDE_STREAM_MIN_BYTES
    src, tgt = _b5_maps(b, 1000 + b)
    _per_image_case(pn, src, tgt, math, f"b5 NCHW fp32 B={b} {math}")


@pytest.mark.parametrize("b", [5, 6, 64])
def test_b5_channels_last_fp32(pn, b):
    """Channels-last fp32 b5 maps, P = 256, tc_bf16x3.  B = 5 / 6 straddle the fold of the channels-last gather:
    gather_nhwc_ctas is 480 <= kFoldMaxCtas (k_gather_tc_nhwc_fold) and 576 above it (k_prep, then k_gather_tc_nhwc).
    B = 64 is bench.py --layout nhwc.  The backward is k_fill_zero + k_scatter_nhwc (launch_dense_nhwc: every C a
    multiple of 4 and <= 256), and the loss kernel is k_loss_tc_p as for NCHW."""
    from gan_variant_research_b200 import patchnce as pmod
    if b in (5, 6):
        assert (gather_nhwc_ctas(B5, 256, b) <= FOLD_MAX_CTAS) == (b == 5)
        assert map_bytes(B5, b, 4) < pmod._SIDE_STREAM_MIN_BYTES
    src, tgt = _b5_maps(b, 2000 + b, channels_last=True)
    _per_image_case(pn, src, tgt, "tc_bf16x3", f"b5 channels-last fp32 B={b}")


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_b5_half_maps(pn, dtype):
    """bench.py --dtype fp16 / bf16 (the AMP regime): NCHW half maps at B = 64, P = 256, tc_bf16x3.  The gather converts
    the half values (k_gather_tc, pnce_plan_ids_draw first: the maps are 3.2 GB); the restatement runs on the same half
    values.  The gradient comes back in the map dtype (k_dense_flat<__half / __nv_bfloat16>), so one ulp of that dtype
    per entry is allowed on top of the fp32 tolerance."""
    src, tgt = _b5_maps(64, 3000, dtype)
    _per_image_case(pn, src, tgt, "tc_bf16x3", f"b5 NCHW {dtype} B=64")


SCHEDULE = [("S-2", "above"), ("S-2", "single"), ("S", "below"), ("S", "above"), ("S", "single"), ("S+2", "below"),
            ("S+2", "above"), ("S+2", "single"), ("4.3S", "below"), ("4.3S", "above"), ("4.3S", "single")]


@pytest.mark.parametrize("items,kind", SCHEDULE)
def test_persistent_loss_schedule(pn, items, kind):
    """k_loss_tc_p (launch_loss_tc: P <= 256 in every layer) with more items than CTAs: one CTA per SM (S read from the
    device) walks items = B * sum(Ppad / 128) in the heavy-first order rotated by ``rot`` (tp_decode).  Items S - 2
    (fewer than CTAs), S, S + 2 and about 4.3 S (several waves), each with two channel counts and the light items below
    grid / 3 (rot = the light count) or at / above it (rot = grid / 3), and with one channel count (rot = 0).  Layers of
    P = 100 / 128 (one item per image) and P = 200 / 256 (two) are mixed where the count allows.  S - 2 = 146 on a
    148-SM B200 factors as 2 * 73, which leaves no batch with the light items below a third: that pair is not listed.
    The maps are small: the schedule does not depend on their size."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    target = {"S-2": sm - 2, "S": sm, "S+2": sm + 2, "4.3S": 4.3 * sm}[items]
    case = schedule_case(sm, target, kind)
    assert case is not None, (sm, items, kind)
    b, layers, (n_items, grid, light, rot) = case
    assert (kind == "single") == (rot == 0)
    g = torch.Generator(device="cuda").manual_seed(n_items * 3 + len(layers))
    src = [torch.randn(b, c, h, w, device="cuda", generator=g) for c, h, w, _ in layers]
    tgt = [(0.6 * s + 0.8 * torch.randn(s.shape, device="cuda", generator=g)).requires_grad_() for s in src]
    ids = [torch.randint(0, h * w, (p,), device="cuda", generator=g) for _, h, w, p in layers]
    loss = pn.fused_patchnce(src, tgt, ids, 0.07, math="tc_bf16x3")
    loss.backward()
    assert pn.poll_nonfinite_warnings(block=True) == 0
    what = f"schedule {items} {kind}: B={b}, {len(layers)} layers, {n_items} items, grid {grid}, light {light}, rot {rot}"
    ltol, gtol = TOL["tc_bf16x3"]
    rl, ref, _ = restate(src, tgt, ids, 0.07)
    le = loss_error(loss.item(), rl, ltol, what)
    ge = check_grads([t.grad for t in tgt], ref, ids, gtol, what)
    print(f"\n[{what}] loss rel err {le:.2e}, worst block err {ge:.2e}")


def test_config4_512sq_p1024(pn):
    """BASELINE config 4: B = 8, b5 maps at 512^2, P = 1024, all five layers, tc_bf16x3.  Ppad = 1024 > 256 takes the
    non-persistent two-pass loss kernel k_loss_tc (one CTA per 128-row item, four key blocks); the 3.2 GB of maps take
    pnce_plan_ids_draw + k_gather_tc."""
    src, tgt = _b5_maps(8, 4000, shapes=CFG4)
    _per_image_case(pn, src, tgt, "tc_bf16x3", "config 4 B=8 512^2 P=1024", p=1024)


# ---- the per-image netF head at bench.py's size ----------------------------------------------------------------------
@pytest.mark.parametrize("b,nc,math,nhwc", [(64, 256, "tc_bf16x3", False), (64, 256, "tc_bf16x3", True),
                                            (64, 256, "tc_bf16", False), (11, 128, "tc_bf16x3", False)],
                         ids=["B64-nc256-bf16x3-nchw", "B64-nc256-bf16x3-nhwc", "B64-nc256-bf16-nchw",
                              "B11-nc128-bf16x3-nchw"])
def test_head_per_image(pn, b, nc, math, nhwc):
    """patchnce_with_head (fused, per-image negatives) on b5 maps, P = 256, ids drawn by the call.  The head runs
    k_gemm_tc_p (persistent, one CTA per SM) over B * Ppad / 128 row tiles per layer and side (5 x 128 at B = 64),
    k_wgrad_tc split-K over min(tiles, 8) slabs (16 tiles each at B = 64; 22 tiles in slabs of 2-3 at B = 11) and
    k_wreduce; the loss is k_loss_tc_p on the head's output.  The maps and W1, b1 are quantised like
    test_patchnce_with_head_minibatch_gpu (_maps, _netf), so that X W1^T + b1 is exact and the kernels' ReLU masks are
    the restatement's.  Checked: the loss, d tgt per (image, layer), dW1, db1, dW2, db2 per layer."""
    src, tgt = _quantised_maps(5000 + b, b, B5)
    if nhwc:
        src = [x.contiguous(memory_format=torch.channels_last) for x in src]
        tgt = [x.contiguous(memory_format=torch.channels_last) for x in tgt]
    netF = _netf(pn, nc, tgt)
    t = [x.detach().requires_grad_() for x in tgt]

    def run():
        netF.zero_grad(set_to_none=True)
        loss, ids = pn.patchnce_with_head(netF, src, t, 0.07, 256, math=math)
        loss.backward()
        return loss.item(), ids

    loss, ids = _assert_randint_ids(run, tgt, 256, 77)
    assert pn.poll_nonfinite_warnings(block=True) == 0
    heads = _head_params(netF, len(B5))
    what = f"head B={b} nc={nc} {math} {'channels-last' if nhwc else 'NCHW'}"
    ltol, gtol = HEAD_TOL[math]
    rl, ref, rh = restate(src, tgt, ids, 0.07, heads)
    le = loss_error(loss, rl, ltol, what)
    ge = check_grads([x.grad for x in t], ref, ids, gtol, what)
    he = check_head_grads([[p.grad for p in ps] for ps in heads], rh, gtol, what)
    print(f"\n[{what}] loss rel err {le:.2e}, worst d tgt block err {ge:.2e}, worst head gradient err {he:.2e}")


# ---- bench.py's own step -------------------------------------------------------------------------------------------
def relu_flip_allowance(src, tgt, ids, heads, tau):
    """Per layer, what an unquantised head's ReLU masks may move, for a head restated like ``restate``.  A (row, unit)
    whose float64 pre-activation X W1^T + b1 is within 2^-16 of its magnitude sum |x| |W1| + |b1| of zero
    (test_netf_gpu._relu_boundary) may take the other mask in the kernel.  The forward then moves by at most that
    pre-activation (negligible), but the backward gains or loses the whole term g_u = (d loss / d h)_u of that unit:
    g_u W1[u, :] in the row's d tgt, g_u x in dW1[u, :], g_u in db1[u].  Returns per layer (|those| summed over the
    row's boundary units as (B, C, P) columns at the ids, the same for dW1 (nc, C) and db1 (nc,), rows on the
    boundary)."""
    out = []
    for s, t, i, prm in zip(src, tgt, ids, heads):
        w1, b1, w2, b2 = (q.detach().double() for q in prm)
        k, x = _rows(s, i), _rows(t, i)
        b, p, c = x.shape
        kh = head_forward_torch(k.reshape(-1, c), w1, b1, w2, b2).reshape(b, p, -1)
        pre = x @ w1.t() + b1
        amb = pre.abs() <= 2.0 ** -16 * (x.abs() @ w1.abs().t() + b1.abs())                   # (B, P, nc)
        y = (pre.relu() @ w2.t() + b2).requires_grad_()
        z = (torch.bmm(F.normalize(y, dim=2, eps=NORM_EPS), kh.transpose(1, 2)) / tau).clamp(-LOGIT_CLAMP, LOGIT_CLAMP)
        loss = F.cross_entropy(z.reshape(b * p, p), torch.arange(p, device=z.device).repeat(b)) / len(src)
        gh = (torch.autograd.grad(loss, y)[0] @ w2).abs() * amb                                # |g_u| on the boundary
        out.append(((gh @ w1.abs()).transpose(1, 2), gh.reshape(-1, gh.shape[2]).t() @ x.abs().reshape(-1, c),
                    gh.sum((0, 1)), int(amb.any(-1).sum())))
    return out


def check_dump(d, shapes, ids, ref, dtype, tol, what, allow=None):
    """bench.dump_outputs' gradient files against ``restate``'s columns ``ref`` at the dumped ``ids``:
    - grad_l{l} (every image's columns at the ids, duplicates included), one (image, layer) block at a time;
    - grad_l{l}_flat at the indices dump_outputs draws (torch.Generator().manual_seed(0), layer by layer, into the
      NCHW-contiguous gradient): exactly 0 off the sampled positions, within the block tolerance on them.
    ``allow``: per layer (B, C, P) absolute allowance at the ids (``relu_flip_allowance``); those layers are also held
    to 1e-3 of the layer's max over all rows at once.  -> (worst block error, worst flat error, worst layer error)."""
    worst = flat_worst = glob = 0.0
    g = torch.Generator().manual_seed(0)
    for l, ((c, h, w), i, (pos, want)) in enumerate(zip(shapes, ids, ref)):
        b, dev = want.shape[0], want.device
        inv = torch.searchsorted(pos, i)
        cols = want[:, :, inv]                                                  # (B, C, P) at the dumped ids
        got = torch.from_numpy(d[f"grad_l{l}"]).to(dev)
        assert got.shape == cols.shape, (got.shape, cols.shape)
        allow_u = None                                                          # at the unique positions
        if allow is not None:
            allow_u = torch.zeros_like(want).index_add_(2, inv, allow[l])       # duplicate ids accumulate
        allow_c = None if allow_u is None else allow_u[:, :, inv]
        err = block_errors(got, cols, dtype, allow_c)
        e, bad = err.max().item(), int(err.argmax())
        assert e <= tol, f"{what} grad_l{l} image {bad}: block error {e:.3e} > {tol}"
        worst = max(worst, e)
        if allow is not None:
            ge = (excess(got.double(), cols, dtype, allow_c).max() / cols.abs().max()).item()
            assert ge <= 1e-3, f"{what} grad_l{l}: error {ge:.3e} > 1e-3 of the layer's max"
            glob = max(glob, ge)
        n = b * c * h * w
        flat = torch.randint(0, n, (min(bench.DUMP_FLAT, n),), generator=g).to(dev)
        fv = torch.from_numpy(d[f"grad_l{l}_flat"]).to(dev).double()
        fb, fc, fp = flat // (c * h * w), flat // (h * w) % c, flat % (h * w)
        slot = torch.searchsorted(pos, fp).clamp(max=pos.numel() - 1)
        on = pos[slot] == fp
        n_off = int((fv[~on] != 0).sum())
        assert n_off == 0, f"{what} grad_l{l}_flat: {n_off} non-zero entries off the sampled positions"
        fb, fc, slot = fb[on], fc[on], slot[on]
        fe = excess(fv[on], want[fb, fc, slot], dtype, None if allow_u is None else allow_u[fb, fc, slot])
        fe = fe / want.abs().amax(dim=(1, 2)).clamp(min=1e-30)[fb]
        fe = fe.max().item() if fe.numel() else 0.0
        assert fe <= tol, f"{what} grad_l{l}_flat: error {fe:.3e} > {tol}"
        flat_worst = max(flat_worst, fe)
    return worst, flat_worst, glob


@pytest.mark.parametrize("args", [[], ["--layout", "nhwc"], ["--dtype", "fp16"], ["--head"]],
                         ids=["nchw-fp32", "nhwc-fp32", "nchw-fp16", "head"])
def test_bench_step_outputs(pn, tmp_path, args):
    """What bench.py's product arm returns from its last timed step (--dump-outputs), run in a fresh process, against
    the restatement at the dumped ids: the step after the timed loop, with the gradients in compressible memory, the
    launches chained by PDL and the allocator in its steady state.  Checked: loss.npy; grad_l{l}.npy, every image of 64
    (the dump's budget holds them all), one (image, layer) block at a time; grad_l{l}_flat.npy at the indices
    dump_outputs draws (exactly 0 off the samples, close on them); the head_* gradients.  The --head run's weights are
    not quantised: rows on the ReLU boundary may take the other mask in the kernel, which moves whole terms of their
    gradients (observed: 3.1e-2 of the layer's max in grad_l0).  Every row stays in the per-block check and in a 1e-3
    check of each layer at once, with exactly those terms allowed (relu_flip_allowance); the boundary rows are counted."""
    _release()
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "8", "--warmup", "3", "--no-e2e",
           "--no-cpu-baseline", "--no-head-line", "--dump-outputs", str(out), *args]
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert "images_sampled" not in d
    dtype = torch.float16 if "fp16" in args else torch.float32
    head = "--head" in args
    dev = torch.device("cuda", 0)
    src, tgt = bench.make_maps(bench.LAYER_SETS["b5"], 64, dtype, dev, 1234)
    if "nhwc" in args:
        src = [x.contiguous(memory_format=torch.channels_last) for x in src]
        tgt = [x.contiguous(memory_format=torch.channels_last) for x in tgt]
    ids = []
    for l in range(len(B5)):
        a = d[f"ids_l{l}"]
        assert a.shape == (256,) and (a == np.round(a)).all()
        ids.append(torch.from_numpy(a).long().to(dev))
    heads = None
    if head:
        torch.manual_seed(11)
        netF = pn.PatchSampleF(use_mlp=True, nc=256).to(dev)
        netF.create_mlp(tgt)
        heads = _head_params(netF, len(B5))
    ltol, gtol = HEAD_TOL["tc_bf16x3"] if head else TOL["tc_bf16x3"]
    what = "bench.py " + (" ".join(args) or "(defaults)")
    rl, ref, rh = restate(src, tgt, ids, 0.07, heads)
    le = loss_error(float(d["loss"][0]), rl, ltol, what)
    flips = relu_flip_allowance(src, tgt, ids, heads, 0.07) if head else None
    worst, flat_worst, glob = check_dump(d, B5, ids, ref, dtype, gtol, what, None if flips is None else
                                         [f[0] for f in flips])
    msg = f"\n[{what}] loss rel err {le:.2e}, worst grad_l block err {worst:.2e}, flat sample err {flat_worst:.2e}"
    if head:
        hg = [[torch.from_numpy(d[f"head_mlp_{l}_{k}_{a}"]).to(dev) for k in (0, 2) for a in ("weight", "bias")]
              for l in range(len(B5))]
        he = check_head_grads(hg, rh, 1e-3, what, [(f[1], f[2]) for f in flips])
        msg += (f", worst layer err {glob:.2e}, head gradient err {he:.2e}; {sum(f[3] for f in flips)} of "
                f"{64 * 256 * len(B5)} (image, id) rows on the ReLU boundary, checked with the flip allowance")
    print(msg)
