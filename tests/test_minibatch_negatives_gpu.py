"""Minibatch negatives (nce_includes_all_negatives_from_minibatch) on the B200: k_loss_tc_mb against the float64
minibatch oracle, odd shapes, the benchmarked B5 regime, layouts and dtypes, the B = 1 identity, the row route,
the non-finite guard, CUDA graphs, the kernel list and memory."""
import glob
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import minibatch_oracle as mbo
from oracle import patchnce_oracle as orc

pytestmark = pytest.mark.gpu

SMALL = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "small_*.npz")))
IDS = [os.path.basename(p)[6:-4] for p in SMALL]
B5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
TOL = {"tc_bf16x3": (2e-5, 2e-4), "tc_bf16": (2e-3, 3e-2)}     # loss rel, gradient max-abs / max


@pytest.fixture(scope="module")
def pn():
    import gan_variant_research_b200 as pn
    return pn


def _load(path):
    d = np.load(path)
    n = int(d["n_layers"])
    return d, [(d[f"src{i}"], d[f"tgt{i}"], d[f"ids{i}"]) for i in range(n)]


def _oracle(layers, tau, upstream=1.0):
    n = len(layers)
    out = [mbo.layer_loss_and_grad_np_mb(s, t, i, tau, n, upstream) for s, t, i in layers]
    return sum(l for l, _ in out) / n, [g for _, g in out]


def _run(pn, layers, tau, math, upstream=1.0, dtype=torch.float32, channels_last=False):
    dev = torch.device("cuda")
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    src = [torch.from_numpy(s).to(dev, dtype).contiguous(memory_format=fmt) for s, _, _ in layers]
    tgt = [torch.from_numpy(t).to(dev, dtype).contiguous(memory_format=fmt).requires_grad_() for _, t, _ in layers]
    ids = [torch.from_numpy(i).to(dev) for _, _, i in layers]
    loss = pn.fused_patchnce(src, tgt, ids, tau, math, nce_includes_all_negatives_from_minibatch=True)
    (loss * upstream).backward()
    pn.poll_nonfinite_warnings(block=True)
    return loss.item(), [t.grad.float().cpu().numpy() for t in tgt]


def _kink_positions(src, tgt, ids, tau, width):
    """(image, position) of the sampled target patches whose row holds a logit within ``width`` of the +-50 clamp:
    there the single-pass bf16 rounding may flip the clamp's backward mask, a jump of the whole softmax entry."""
    b, c = tgt.shape[:2]
    k, _ = orc._normalize_np(np.asarray(src, np.float64).reshape(b, c, -1)[:, :, ids].transpose(0, 2, 1).reshape(-1, c))
    q, _ = orc._normalize_np(np.asarray(tgt, np.float64).reshape(b, c, -1)[:, :, ids].transpose(0, 2, 1).reshape(-1, c))
    with np.errstate(all="ignore"):
        near = (np.abs(np.abs(q @ k.T / tau) - orc.LOGIT_CLAMP) < width).any(axis=1)
    return [(r // len(ids), ids[r % len(ids)]) for r in np.nonzero(near)[0]]


def _check(loss, grads, ref_loss, ref_grads, layers, math, tau=0.07):
    rl, rg = TOL[math]
    kink = math == "tc_bf16" and tau < 0.05
    if kink:
        rl, rg = 2e-2, 2e-1                # as in per-image mode: 1/tau = 100 amplifies the single-pass bf16 rounding
    assert loss == pytest.approx(ref_loss, rel=rl, abs=1e-6)
    for g, r, (s, t, ids) in zip(grads, ref_grads, layers):
        np.testing.assert_array_equal(np.isnan(g), np.isnan(r))
        sampled = np.zeros(r.shape[2] * r.shape[3], bool)
        sampled[ids] = True
        off = g.reshape(g.shape[0], g.shape[1], -1)[:, :, ~sampled]
        assert (off == 0).all()                                 # exact zeros off the sampled positions
        fin = np.isfinite(r)
        if kink:
            for bi, pos in _kink_positions(s, t, ids, tau, 1.0):
                fin.reshape(fin.shape[0], fin.shape[1], -1)[bi, :, pos] = False
        scale = max(np.abs(r[fin]).max(initial=0.0), 1e-30)
        assert np.abs(g[fin] - r[fin]).max(initial=0.0) <= rg * scale


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("path", SMALL, ids=IDS)
def test_small_fixtures_match_the_float64_oracle(pn, path, math):
    d, layers = _load(path)
    tau, up = float(d["tau"]), float(d["upstream"])
    ref_loss, ref_grads = _oracle(layers, tau, up)
    loss, grads = _run(pn, layers, tau, math, up)
    _check(loss, grads, ref_loss, ref_grads, layers, math, tau)


def _random_layers(rng, b, shapes, p):
    out = []
    for c, h, w in shapes:
        s = rng.standard_normal((b, c, h, w)).astype(np.float32)
        t = (0.6 * s + 0.8 * rng.standard_normal((b, c, h, w))).astype(np.float32)
        out.append((s, t, rng.integers(0, h * w, min(p, h * w)).astype(np.int64)))
    return out


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("b,shapes,p,tau", [
    (3, [(40, 16, 16)], 200, 0.07),                  # P not a multiple of 128, C not a multiple of 32
    (2, [(64, 32, 32)], 600, 0.07),                  # P > 256: several key blocks per image
    (9, [(24, 12, 12), (96, 20, 20)], 144, 0.07),    # B = 9, padding in every image's last block
    (5, [(32, 30, 30)], 700, 0.015),                 # clamp-binding tau: the two-pass form
    (4, [(256, 16, 16), (8, 8, 8)], 64, 0.1),        # C = 256, P = 64
])
def test_odd_shapes(pn, b, shapes, p, tau, math):
    layers = _random_layers(np.random.default_rng(b * 7 + p), b, shapes, p)
    ref_loss, ref_grads = _oracle(layers, tau)
    loss, grads = _run(pn, layers, tau, math)
    _check(loss, grads, ref_loss, ref_grads, layers, math, tau)


def _restate_gpu64(src, tgt, ids, tau):
    """Upstream's formula (batch_dim_for_bmm = 1) in float64 on the GPU, autograd backward, all layers."""
    total = 0.0
    t64 = [t.detach().double().requires_grad_() for t in tgt]
    for s, t, i in zip(src, t64, ids):
        b, c = s.shape[:2]
        k = F.normalize(s.double().reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(-1, c), dim=1, eps=orc.NORM_EPS)
        q = F.normalize(t.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(-1, c), dim=1, eps=orc.NORM_EPS)
        z = (q @ k.t() / tau).clamp(-50, 50)
        total = total + F.cross_entropy(z, torch.arange(z.shape[0], device=z.device))
    total = total / len(src)
    total.backward()
    return total.item(), [t.grad for t in t64]


@pytest.mark.parametrize("batch", [16, 64])
def test_b5_full_size_against_float64_restatement(pn, batch):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(batch)
    src = [torch.randn(batch, *s, device=dev, generator=g) for s in B5]
    tgt = [(0.5 * a + torch.randn(a.shape, device=dev, generator=g)).requires_grad_() for a in src]
    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True, math="tc_bf16x3")
    gen = torch.cuda.default_generators[0]
    torch.manual_seed(123)
    off0 = gen.get_offset()
    loss = crit(src, tgt)
    loss.backward()
    ids = crit.last_patch_ids
    off1 = gen.get_offset()
    torch.manual_seed(123)
    ref_ids = [torch.randint(0, s[1] * s[2], (256,), device=dev) for s in B5]
    assert gen.get_offset() - off0 == off1 - off0
    for a, r in zip(ids, ref_ids):
        assert torch.equal(a, r)
    ref_loss, ref_grads = _restate_gpu64(src, tgt, ids, 0.07)
    assert loss.item() == pytest.approx(ref_loss, rel=1e-4)
    for t, r in zip(tgt, ref_grads):
        assert (t.grad.double() - r).abs().max().item() <= 1e-3 * r.abs().max().item()


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_maps_and_channels_last(pn, dtype):
    layers = _random_layers(np.random.default_rng(5), 6, [(64, 16, 16), (32, 24, 24)], 256)
    layers = [(s.astype(np.float32), t, i) for s, t, i in layers]
    # the oracle on the values the half maps hold
    rounded = [(torch.from_numpy(s).to(dtype).float().numpy(), torch.from_numpy(t).to(dtype).float().numpy(), i)
               for s, t, i in layers]
    ref_loss, ref_grads = _oracle(rounded, 0.07)
    loss, grads = _run(pn, layers, 0.07, "tc_bf16x3", dtype=dtype)
    assert loss == pytest.approx(ref_loss, rel=2e-5)
    for g, r in zip(grads, ref_grads):
        assert np.abs(g - r).max() <= 1e-2 * np.abs(r).max()      # gradient stored in the half dtype
    loss_cl, grads_cl = _run(pn, layers, 0.07, "tc_bf16x3", dtype=dtype, channels_last=True)
    assert loss_cl == pytest.approx(loss, rel=1e-6)
    for a, b in zip(grads, grads_cl):                  # the same fp32 values up to summation order, stored in half
        np.testing.assert_allclose(a, b, rtol=1e-2, atol=1e-3 * np.abs(a).max())


def test_batch_of_one_is_bit_identical_to_per_image_mode(pn):
    dev = torch.device("cuda")
    src = [torch.randn(1, *s, device=dev) for s in B5]
    tgt = [torch.randn(1, *s, device=dev) for s in B5]
    out = []
    for mb in (False, True):
        t = [x.clone().requires_grad_() for x in tgt]
        torch.manual_seed(7)
        loss = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=mb)(src, t)
        loss.backward()
        out.append((loss.detach(), [x.grad for x in t]))
    assert torch.equal(out[0][0], out[1][0])
    for a, b in zip(out[0][1], out[1][1]):
        assert torch.equal(a, b)


def test_module_split_route_equals_the_maps_route(pn):
    dev = torch.device("cuda")
    shapes = [(64, 32, 32), (128, 16, 16)]
    src = [torch.randn(8, *s, device=dev) for s in shapes]
    tgt = [torch.randn(8, *s, device=dev, requires_grad=True) for s in shapes]
    ids = pn.draw_patch_ids_all(src, 256)
    maps = pn.fused_patchnce(src, tgt, ids, 0.07, nce_includes_all_negatives_from_minibatch=True)
    gm = torch.autograd.grad(maps, tgt)
    netF = pn.PatchSampleF(use_mlp=False)
    fk, _ = netF(src, 256, ids)
    fq, _ = netF(tgt, 256, ids)
    rows = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True)(fq, fk)
    gr = torch.autograd.grad(rows, tgt)
    assert rows.item() == pytest.approx(maps.item(), rel=2e-5)
    for a, b in zip(gm, gr):
        assert (a - b).abs().max().item() <= 2e-4 * a.abs().max().item()


def test_module_split_with_mlp_matches_autograd(pn):
    dev = torch.device("cuda")
    torch.manual_seed(3)
    shapes = [(64, 16, 16), (32, 16, 16)]
    src = [torch.randn(4, *s, device=dev) for s in shapes]
    tgt = [torch.randn(4, *s, device=dev, requires_grad=True) for s in shapes]
    netF = pn.PatchSampleF(use_mlp=True, nc=128)
    with torch.no_grad():
        fk, ids = netF(src, 128)
    fq, _ = netF(tgt, 128, ids)
    loss = pn.PatchNCELoss(0.07, 128, nce_includes_all_negatives_from_minibatch=True)(fq, fk)
    loss.backward()
    gq = [t.grad.clone() for t in tgt]
    # torch restatement on the same head output
    total = 0.0
    t2 = [t.detach().clone().requires_grad_() for t in tgt]
    for l, (s, t, i) in enumerate(zip(src, t2, ids)):
        mlp = getattr(netF, f"mlp_{l}")
        b, c = s.shape[:2]
        k = F.normalize(mlp(s.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(-1, c)), dim=1, eps=1e-6).detach()
        h = t.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(-1, c)
        q = F.normalize(mlp(h), dim=1, eps=1e-6)
        z = (q @ k.t() / 0.07).clamp(-50, 50)
        total = total + F.cross_entropy(z, torch.arange(z.shape[0], device=dev))
    total = total / len(src)
    total.backward()
    assert loss.item() == pytest.approx(total.item(), rel=1e-3)
    for a, r in zip(gq, t2):
        assert (a - r.grad).abs().max().item() <= 1e-3 * r.grad.abs().max().item()


def test_nan_image_zeroes_exactly_its_layers(pn, capsys):
    path = os.path.join(os.path.dirname(__file__), "golden", "small_nan_image.npz")
    d, layers = _load(path)
    tau = float(d["tau"])
    bad = [not (np.isfinite(s).all() and np.isfinite(t).all()) for s, t, _ in layers]
    assert any(bad)
    capsys.readouterr()
    dev = torch.device("cuda")
    src = [torch.from_numpy(s).to(dev) for s, _, _ in layers]
    tgt = [torch.from_numpy(t).to(dev) for _, t, _ in layers]
    ids = [torch.from_numpy(i).to(dev) for _, _, i in layers]
    call_loss = pn.fused_patchnce(src, tgt, ids, tau, nce_includes_all_negatives_from_minibatch=True)
    n = pn.poll_nonfinite_warnings(block=True)
    out = capsys.readouterr().out
    assert n == sum(bad)
    assert out.count("Warning: NaN in PatchNCE loss") == sum(bad)
    ref_loss, _ = _oracle(layers, tau)
    assert call_loss.item() == pytest.approx(ref_loss, rel=2e-5)       # the oracle zeroes exactly the bad layers


def test_graph_capture_and_loss_and_grads(pn):
    g = torch.Generator().manual_seed(4)
    shapes = [(64, 32, 32), (128, 16, 16)]
    src = [torch.randn(8, *s, generator=g).cuda() for s in shapes]
    tgt = [torch.randn(8, *s, generator=g).cuda().requires_grad_() for s in shapes]
    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                      # warm-up outside the capture (lazy init, smem opt-in)
        for _ in range(2):
            for t in tgt:
                t.grad = None
            crit(src, tgt).backward()
    torch.cuda.current_stream().wait_stream(side)
    for t in tgt:
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gl = crit(src, tgt)
        gl.backward()
        ids_static = [i.clone() for i in crit.last_patch_ids]
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        gg = [t.grad.clone() for t in tgt]
        t2 = [t.detach().clone().requires_grad_() for t in tgt]
        eager = pn.fused_patchnce(src, t2, [i.clone() for i in ids_static], 0.07,
                                  nce_includes_all_negatives_from_minibatch=True)
        eager.backward()
        assert torch.equal(gl.detach(), eager.detach())
        for a, b in zip(gg, t2):
            assert torch.equal(a, b.grad)
    for t in tgt:
        t.grad = None
    # loss_and_grads = forward + backward
    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True)
    torch.manual_seed(11)
    loss = crit(src, tgt)
    gf = torch.autograd.grad(loss, tgt)
    torch.manual_seed(11)
    loss2, g2 = crit.loss_and_grads(src, [t.detach() for t in tgt])
    assert torch.equal(loss.detach(), loss2)
    for a, b in zip(gf, g2):
        assert torch.equal(a, b)


def test_kernel_list_and_memory_at_b64(pn):
    dev = torch.device("cuda")
    src = [torch.randn(64, *s, device=dev) for s in B5]
    tgt = [torch.randn(64, *s, device=dev, requires_grad=True) for s in B5]
    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True)
    loss = crit(src, tgt)
    loss.backward()                                           # warm: workspace, shape plan
    for t in tgt:
        t.grad = None
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss = crit(src, tgt)
        loss.backward()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    assert any("k_loss_tc_mb" in n for n in names), names
    banned = ("gemm", "bmm", "softmax", "cutlass", "cublas", "nvjet", "sm90_xmma", "sm100_xmma")
    assert not [n for n in names if any(b in n.lower() for b in banned)], names
    peak = torch.cuda.max_memory_allocated() - base
    grads = sum(t.numel() * 4 for t in tgt)
    ws_bytes = max(sp.ws_bytes for sp in pn.patchnce._SHAPE_PLANS.values() if sp.mb and sp.batch == 64)
    n = 64 * 256
    assert peak - grads - ws_bytes < n * n * 4, (peak, grads, ws_bytes)


def test_faster_than_the_eager_restatement_at_b16(pn):
    dev = torch.device("cuda")
    src = [torch.randn(16, *s, device=dev) for s in B5]
    tgt = [torch.randn(16, *s, device=dev, requires_grad=True) for s in B5]
    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True)

    def ours():
        crit(src, tgt).backward()

    def eager():
        ids = [torch.randint(0, s[1] * s[2], (256,), device=dev) for s in B5]
        tot = 0.0
        for s, t, i in zip(src, tgt, ids):
            b, c = s.shape[:2]
            k = F.normalize(s.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(1, -1, c), dim=2, eps=1e-6)
            q = F.normalize(t.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(1, -1, c), dim=2, eps=1e-6)
            z = (torch.bmm(q, k.transpose(2, 1)) / 0.07).clamp(-50, 50)[0]
            tot = tot + F.cross_entropy(z, torch.arange(z.shape[0], device=dev))
        (tot / len(B5)).backward()

    def timed(fn):
        for _ in range(3):
            fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / 20

    t_ours, t_eager = timed(ours), timed(eager)
    print(f"B=16 minibatch negatives: k_loss_tc_mb step {t_ours:.3f} ms, eager torch {t_eager:.3f} ms")
    assert t_ours < t_eager
