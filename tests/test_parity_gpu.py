"""Parity tests proper: the CUDA path (through the ctypes C ABI) against the golden fixtures
frozen from the unmodified reference and against the oracle on the same seeded inputs.
Tolerances: ids bit-exact; loss and gradients 1e-3 relative (north_star) -- the fp32 SIMT mode is
held to 2e-5 / 1e-4 so the gate has teeth."""
import glob
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
SMALL = sorted(glob.glob(os.path.join(HERE, "golden", "small_*.npz")))
R4 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128)]
B5 = R4 + [(64, 256, 256)]


@pytest.fixture(scope="module")
def pn():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gan_variant_research_b200 as m
    from gan_variant_research_b200 import _lib
    _lib.load()
    return m


@pytest.fixture(scope="module")
def orc():
    from oracle import patchnce_oracle
    return patchnce_oracle


def dev(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return t if dtype is None else t.to(dtype)


def assert_grad_close(got, want, rtol, what="", ids=None):
    """max-abs error relative to the largest reference entry; NaN patterns must coincide.
    With ``ids`` the dense gradient must be EXACTLY zero off the sampled positions (at a sampled
    position an analytically-zero entry may differ from 0.0 by rounding, e.g. a one-hot post-ReLU
    row, so closeness is the test there)."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want), err_msg=f"{what}: NaN pattern")
    m = ~np.isnan(want)
    scale = max(float(np.abs(want[m]).max()) if m.any() else 0.0, 1e-30)
    err = float(np.abs(got[m] - want[m]).max()) / scale if m.any() else 0.0
    assert err <= rtol, f"{what}: rel err {err:.3e} > {rtol}"
    if ids is not None:
        b, c = got.shape[:2]
        flat = got.reshape(b, c, -1)
        off = np.ones(flat.shape[2], dtype=bool)
        off[np.asarray(ids)] = False
        assert not np.any(flat[:, :, off] != 0), f"{what}: non-zero gradient off the sampled positions"


def load_small(path):
    d = np.load(path)
    n = int(d["n_layers"])
    return (d, [d[f"src{i}"] for i in range(n)], [d[f"tgt{i}"] for i in range(n)],
            [d[f"ids{i}"] for i in range(n)], [d[f"grad{i}"] for i in range(n)])


# (loss rtol, grad rtol) per contraction engine; north_star asks 1e-3 in fp32-accumulate mode
MATH_TOL = {"simt_f32": (2e-5, 1e-4), "tc_bf16x3": (2e-5, 2e-4), "tc_bf16": (2e-3, 3e-2)}


@pytest.mark.parametrize("math", list(MATH_TOL))
@pytest.mark.parametrize("path", SMALL, ids=[os.path.basename(p)[6:-4] for p in SMALL])
def test_fused_matches_reference_goldens(pn, path, math):
    d, src, tgt, ids, grads = load_small(path)
    t = [dev(x).requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([dev(x) for x in src], t, [dev(i) for i in ids], float(d["tau"]), math=math)
    (loss * float(d["upstream"])).backward()
    assert loss.dtype == torch.float32 and loss.dim() == 0 and loss.is_cuda
    ltol, gtol = MATH_TOL[math]
    if math == "tc_bf16" and float(d["tau"]) < 0.05:
        ltol, gtol = 2e-2, 2e-1            # 1/tau = 100 amplifies the single-pass bf16 rounding
    assert loss.item() == pytest.approx(float(d["loss"]), rel=ltol, abs=1e-6)
    for i, (tt, g) in enumerate(zip(t, grads)):
        assert_grad_close(tt.grad.cpu().numpy(), g, gtol, f"layer {i}", ids=ids[i])
    assert pn.poll_nonfinite_warnings(block=True) >= 0      # raises on a kernel protocol timeout


def _assert_rows_close(got, want, ids, rtol, what):
    """Gradient rows (one per sampled position, all channels) compared each against ITS OWN largest entry: a dead
    post-ReLU patch (||q|| < eps -> the g / eps branch, patchnce_cut.py:77 backward) has rows ~1e6 times larger than
    its neighbours and would hide every other row behind a single max-norm."""
    b, c = got.shape[:2]
    g = got.reshape(b, c, -1)[:, :, np.unique(ids)].astype(np.float64)
    w = want.reshape(b, c, -1)[:, :, np.unique(ids)].astype(np.float64)
    scale = np.maximum(np.abs(w).max(axis=1, keepdims=True), 1e-12 * np.abs(w).max())
    err = (np.abs(g - w) / scale).max()
    assert err <= rtol, f"{what}: row-relative err {err:.3e} > {rtol}"


@pytest.mark.parametrize("math", ["simt_f32", "tc_bf16x3"])
def test_real_generator_maps_match_the_reference(pn, math):
    """Feature maps of the unmodified reference ResNetGenerator (generator_resnet_attn.py:190-235, frozen by
    oracle/make_golden_generator.py) through the CUDA path: real post-InstanceNorm / post-ReLU / residual-sum statistics
    (dead 8-channel patches that take the g / eps branch, 16x16 maps where 256 draws hit every position several
    times).  The fixture's ids are passed in (torch's CPU and CUDA generators draw different streams; the id law is
    tested separately); loss and d loss / d tgt_feat against the reference's own."""
    d = np.load(os.path.join(HERE, "golden", "generator_maps_b5.npz"))
    n = int(d["n_layers"])
    src = [dev(d[f"src{i}"]) for i in range(n)]
    tgt = [dev(d[f"tgt{i}"]).requires_grad_() for i in range(n)]
    ids = [dev(d[f"ids{i}"]) for i in range(n)]
    loss = pn.fused_patchnce(src, tgt, ids, 0.07, math=math)
    (loss * float(d["upstream"])).backward()
    ltol, gtol = MATH_TOL[math]
    assert loss.item() == pytest.approx(float(d["loss"]), rel=ltol)
    for i in range(n):
        got, want = tgt[i].grad.cpu().numpy(), d[f"grad{i}"]
        assert_grad_close(got, want, gtol, f"layer {i}", ids=d[f"ids{i}"])
        _assert_rows_close(got, want, d[f"ids{i}"], 5 * gtol, f"layer {i}")
    assert pn.poll_nonfinite_warnings(block=True) == 0


def test_nonfinite_images_are_counted_and_reported(pn, capsys):
    d, src, tgt, ids, _ = load_small(os.path.join(HERE, "golden", "small_nan_image.npz"))
    pn.poll_nonfinite_warnings(block=True)
    loss = pn.fused_patchnce([dev(x) for x in src], [dev(x) for x in tgt], [dev(i) for i in ids], 0.07)
    assert torch.isfinite(loss)
    assert pn.poll_nonfinite_warnings(block=True) == 1
    assert "Warning: NaN in PatchNCE loss" in capsys.readouterr().out


def test_patch_ids_bit_exact_and_rng_stream_aligned(pn, orc):
    """Same generator state on the same device => identical ids per layer (int64, with
    replacement, shared by the batch, one draw per returned layer, P = min(num_patches, HW)) and
    the generator is left in the same state (SURVEY.md 3.1 RNG note)."""
    shapes = [(8, 64, 64), (4, 7, 9), (16, 128, 128), (4, 3, 3)]
    src = [torch.randn(2, *s, device="cuda") for s in shapes]
    tgt = [torch.randn(2, *s, device="cuda") for s in shapes]
    torch.manual_seed(7)
    want = [orc.draw_patch_ids(s[1] * s[2], 256, "cuda") for s in shapes]
    after_want = torch.rand(4, device="cuda")
    torch.manual_seed(7)
    mod = pn.PatchNCELoss(0.07, 256, [0, 4, 8, 12, 16])
    mod(src, tgt)
    after_got = torch.rand(4, device="cuda")
    for g, w, s in zip(mod.last_patch_ids, want, shapes):
        assert g.dtype == torch.int64 and g.numel() == min(256, s[1] * s[2])
        assert torch.equal(g, w)
    assert torch.equal(after_got, after_want)
    # PatchSampleF draws the same way
    torch.manual_seed(7)
    _, ids = pn.PatchSampleF()(tgt, 256)
    for g, w in zip(ids, want):
        assert torch.equal(g, w)
    # large problems issue the draws on a side stream: same ids, same generator state afterwards
    from gan_variant_research_b200 import patchnce as pmod
    keep = pmod._SIDE_STREAM_MIN_BYTES
    pmod._SIDE_STREAM_MIN_BYTES = 0
    try:
        torch.manual_seed(7)
        mod(src, tgt)
        after_side = torch.rand(4, device="cuda")
    finally:
        pmod._SIDE_STREAM_MIN_BYTES = keep
    for g, w in zip(mod.last_patch_ids, want):
        assert torch.equal(g, w)
    assert torch.equal(after_side, after_want)


def test_library_id_draw_follows_torch_randint_bit_for_bit(pn):
    """pnce_draw_ids / pnce_fwd_draw draw the ids inside the library: for any seed, any generator offset and any
    (H*W, P) they must be exactly what the reference's ``torch.randint(0, HW, (P,), device=...)`` calls return
    (patchnce_cut.py:63), and the generator must end up where those calls would have left it."""
    from gan_variant_research_b200 import patchnce as pmod
    dev = torch.device("cuda", torch.cuda.current_device())
    assert pmod._philox_ready(dev), "the in-library draw was rejected on this torch build (host fell back to randint)"
    cases = [(256 * 256, 256), (64 * 64, 256), (128 * 128, 256), (512 * 512, 1024), (128 * 128, 1024), (9, 9), (1, 1),
             (300, 256), (1 << 20, 4096)]
    for seed in (0, 7, 1234567891011, 2 ** 63 - 5):
        torch.manual_seed(seed)
        torch.rand(3 + seed % 5, device=dev)                       # some offset into the stream
        state = torch.cuda.get_rng_state(dev)
        want = [torch.randint(0, hw, (p,), device=dev) for hw, p in cases[:8]]
        after_want = torch.rand(5, device=dev)
        torch.cuda.set_rng_state(state, dev)
        feats = [torch.empty(1, 1, 1, hw, device=dev) for hw, _ in cases[:8]]
        got = []
        for f, (_, p) in zip(feats, cases[:8]):                    # P differs per layer: one call each
            got += pn.draw_ids([f], p)
        after_got = torch.rand(5, device=dev)
        for g, w in zip(got, want):
            assert g.dtype == torch.int64 and torch.equal(g, w)
        assert torch.equal(after_got, after_want)
        # several layers in one launch
        torch.cuda.set_rng_state(state, dev)
        want8 = [torch.randint(0, hw, (min(256, hw),), device=dev) for hw, _ in cases]
        torch.cuda.set_rng_state(state, dev)
        got8 = pn.draw_ids([torch.empty(1, 1, 1, hw, device=dev) for hw, _ in cases[:8]], 256)
        assert all(torch.equal(g, w) for g, w in zip(got8, want8))
    # P = 4096 spans 16 blocks of torch's launch
    torch.manual_seed(3)
    w = torch.randint(0, 1 << 20, (4096,), device=dev)
    torch.manual_seed(3)
    (g,) = pn.draw_ids([torch.empty(1, 1, 1024, 1024, device=dev)], 4096)
    assert torch.equal(g, w)


@pytest.mark.parametrize("math", ["simt_f32", "tc_bf16x3"])
@pytest.mark.parametrize("b", [1, 2])
def test_survey_tripwire_full_size(pn, b, math):
    """SURVEY.md 8c: full-size R4 maps, the reference's own CPU-drawn ids."""
    d = np.load(os.path.join(HERE, "golden", f"survey_r4_b{b}.npz"))
    g = torch.Generator().manual_seed(1234)
    src = [torch.randn(b, *s, generator=g).relu() for s in R4]
    tgt = [torch.randn(b, *s, generator=g).relu() for s in R4]
    ids = [dev(d[f"ids{i}"]) for i in range(4)]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, ids, 0.07, math=math)
    loss.backward()
    assert loss.item() == pytest.approx(float(d["loss"]), rel=2e-5)
    for i, tt in enumerate(t):
        gr = tt.grad
        assert gr.double().norm().item() == pytest.approx(float(d[f"gnorm{i}"]), rel=1e-4)
        assert gr.double().sum().item() == pytest.approx(float(d[f"gsum{i}"]), rel=1e-3, abs=1e-7)
        assert int((gr != 0).sum()) == int(d[f"nnz{i}"])            # = unique(ids) * C
        cols = gr[0].reshape(gr.shape[1], -1)[:, ids[i][:8]].cpu().numpy()
        assert_grad_close(cols, d[f"gcols{i}"], 1e-4, f"layer {i} columns")


def test_layer_mean_divides_by_number_of_maps(pn, orc):
    """[0,4,8,12,16] returns 4 maps and the loss divides by 4 (patchnce_cut.py:40): checked with a
    stub generator that numbers layers like generator_resnet_attn.py:203-235."""
    class StubG(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.convs = torch.nn.ModuleList(
                [torch.nn.Conv2d(3 if i == 0 else 8, 8, 3, padding=1) for i in range(14)])

        def get_feature_layers(self, x, layer_ids=None):
            feats = []
            for i, c in enumerate(self.convs):       # logical layers 0..13 only
                x = torch.relu(c(x))
                if i in layer_ids:
                    feats.append(x)
            return feats

    torch.manual_seed(0)
    gen = StubG().cuda()
    x = torch.randn(2, 3, 16, 16, device="cuda")
    y = torch.randn(2, 3, 16, 16, device="cuda", requires_grad=True)
    assert len(gen.get_feature_layers(x, [0, 4, 8, 12, 16])) == 4
    torch.manual_seed(3)
    loss = pn.compute_patchnce_loss(gen, x, y, [0, 4, 8, 12, 16], 0.07, 64)
    loss.backward()
    g_got = y.grad.clone()
    y.grad = None
    gen_cpu = StubG()
    gen_cpu.load_state_dict(gen.state_dict())
    # same ids: redraw on the device with the same seed
    torch.manual_seed(3)
    ids = [orc.draw_patch_ids(256, 64, "cuda").cpu() for _ in range(4)]
    y_cpu = y.detach().cpu().requires_grad_()
    want = orc.compute_patchnce_loss_torch(gen_cpu, x.cpu(), y_cpu, [0, 4, 8, 12, 16], 0.07, 64, ids_list=ids)
    want.backward()
    assert loss.item() == pytest.approx(want.item(), rel=1e-4)
    assert_grad_close(g_got.cpu().numpy(), y_cpu.grad.numpy(), 2e-3, "d loss / d tgt image")
    # params of the generator received gradient only through the tgt pass
    assert all(p.grad is not None for c in list(gen.convs)[:13] for p in c.parameters())


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_precision_feature_maps(pn, orc, dtype):
    """AMP regime: 16-bit maps in, fp32 math inside, dense gradient in the map dtype."""
    g = torch.Generator().manual_seed(21)
    shapes = [(32, 16, 16), (24, 8, 8)]
    src = [torch.randn(2, *s, generator=g).to(dtype) for s in shapes]
    tgt = [torch.randn(2, *s, generator=g).to(dtype) for s in shapes]
    ids = [torch.randint(0, s[1] * s[2], (min(64, s[1] * s[2]),), generator=g) for s in shapes]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07)
    loss.backward()
    want, _, gw = orc.patchnce_loss_and_grads_np([x.float().numpy() for x in src],
                                                 [x.float().numpy() for x in tgt],
                                                 [i.numpy() for i in ids], 0.07)
    assert loss.item() == pytest.approx(want, rel=2e-5)
    for tt, gg in zip(t, gw):
        assert tt.grad.dtype == dtype
        got = tt.grad.float().cpu().numpy()
        scale = np.abs(gg).max()
        assert np.abs(got - gg).max() / scale < (2e-3 if dtype == torch.float16 else 1e-2)
        np.testing.assert_array_equal(got[gg == 0], 0)


def test_patch_sample_f_rows_and_backward(pn, orc):
    g = torch.Generator().manual_seed(31)
    feats = [torch.randn(3, 20, 9, 7, generator=g), torch.randn(3, 64, 16, 16, generator=g).relu()]
    ids = [torch.randint(0, 63, (40,), generator=g), torch.randint(0, 256, (256,), generator=g)]
    fd = [f.cuda().requires_grad_() for f in feats]
    rows, rid = pn.PatchSampleF()(fd, 256, [i.cuda() for i in ids])
    upstream = [torch.randn(r.shape, generator=g) for r in rows]
    torch.autograd.backward(rows, [u.cuda() for u in upstream])
    for f, i, r, u, fdev, ri in zip(feats, ids, rows, upstream, fd, rid):
        want, _ = orc.gather_normalize_np(f.numpy(), i.numpy())
        assert r.shape == (3 * i.numel(), f.shape[1]) and r.dtype == torch.float32
        np.testing.assert_allclose(r.detach().cpu().numpy(), want, rtol=2e-6, atol=2e-7)
        assert torch.equal(ri.cpu(), i)
        fc = f.clone().requires_grad_()
        b, c = f.shape[:2]
        ref = torch.nn.functional.normalize(
            fc.reshape(b, c, -1).transpose(1, 2)[:, i, :], dim=2, eps=1e-6).reshape(-1, c)
        ref.backward(u)
        assert_grad_close(fdev.grad.cpu().numpy(), fc.grad.numpy(), 1e-5, "PatchSampleF backward")


def test_module_split_composes_to_the_reference(pn):
    """PatchSampleF (no head) + PatchNCELoss(feat_q, feat_k), summed / L, equals the fused
    reference-compat path on the same ids (SURVEY.md section 0, consequence 2)."""
    d, src, tgt, ids, grads = load_small(os.path.join(HERE, "golden", "small_ragged.npz"))
    t = [dev(x).requires_grad_() for x in tgt]
    s = [dev(x) for x in src]
    idd = [dev(i) for i in ids]
    sampler, crit = pn.PatchSampleF(), pn.PatchNCELoss(0.07, 64)
    fq, _ = sampler(t, 64, idd)
    with torch.no_grad():
        fk, _ = sampler(s, 64, idd)
    total = 0.0
    for q, k in zip(fq, fk):
        total = total + crit(q, k, batch_size=3)
    loss = total / len(fq)
    loss.backward()
    assert loss.item() == pytest.approx(float(d["loss"]), rel=2e-5)
    for i, (tt, g) in enumerate(zip(t, grads)):
        assert_grad_close(tt.grad.cpu().numpy(), g, 1e-4, f"layer {i}", ids=ids[i])


def _in_own_process(target):
    """``target(out_path)`` in a spawned process -> what it saved.  Launch lists are recorded there: in a long test
    process a profiler session can come back missing device events (CUPTI state left by earlier sessions)."""
    import multiprocessing as mp
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        out = os.path.join(d, "launches.pt")
        proc = mp.get_context("spawn").Process(target=target, args=(out,))
        proc.start()
        proc.join(timeout=600)
        if proc.is_alive():
            proc.kill()
            proc.join()
        assert proc.exitcode == 0, proc.exitcode
        return torch.load(out)


def _list_form_launches(out_path):
    """The libpnce launches of one PatchNCELoss list-form call on small_ragged's rows (after a warm call)."""
    import gan_variant_research_b200 as pn
    from torch.profiler import ProfilerActivity, profile
    _, src, tgt, ids, _ = load_small(os.path.join(HERE, "golden", "small_ragged.npz"))
    sampler = pn.PatchSampleF()
    idd = [dev(i) for i in ids]
    with torch.no_grad():
        fq, _ = sampler([dev(x) for x in tgt], 64, idd)
        fk, _ = sampler([dev(x) for x in src], 64, idd)
    pn.rows_patchnce_multi(fq, fk, 0.07, 64, batch_size=3)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pn.rows_patchnce_multi(fq, fk, 0.07, 64, batch_size=3)
        torch.cuda.synchronize()
    torch.save([e.key for e in prof.key_averages() if "pnce::" in e.key for _ in range(e.count)], out_path)


def test_module_split_list_form_is_one_call_and_composes_to_the_reference(pn):
    """PatchNCELoss(feat_q_list, feat_k_list) -- every layer of PatchSampleF's output in ONE library call -- equals the
    per-layer loop / L on the reference-frozen fixture, loss and dense gradients; a layer outside the tensor-core
    envelope (D > 256) sends the whole list through the per-layer calls with the same result."""
    d, src, tgt, ids, grads = load_small(os.path.join(HERE, "golden", "small_ragged.npz"))
    t = [dev(x).requires_grad_() for x in tgt]
    s = [dev(x) for x in src]
    idd = [dev(i) for i in ids]
    sampler, crit = pn.PatchSampleF(), pn.PatchNCELoss(0.07, 64)
    fq, _ = sampler(t, 64, idd)
    with torch.no_grad():
        fk, _ = sampler(s, 64, idd)
    loss = crit(fq, fk, batch_size=3)
    (loss * 3.0).backward()
    assert loss.item() == pytest.approx(float(d["loss"]), rel=2e-5)
    for i, (tt, g) in enumerate(zip(t, grads)):
        assert_grad_close(tt.grad.cpu().numpy() / 3.0, g, 1e-4, f"layer {i}", ids=ids[i])
    # the same rows through the per-layer calls
    q2 = [q.detach().clone().requires_grad_() for q in fq]
    total = 0.0
    for q, k in zip(q2, fk):
        total = total + crit(q, k, batch_size=3)
    per_layer = total / len(q2)
    per_layer.backward()
    q3 = [q.detach().clone().requires_grad_() for q in fq]
    fused = pn.rows_patchnce_multi(q3, fk, 0.07, 64, batch_size=3)
    fused.backward()
    assert fused.item() == pytest.approx(per_layer.item(), rel=1e-6)
    for a, b in zip(q3, q2):
        torch.testing.assert_close(a.grad, b.grad, rtol=1e-5, atol=1e-9)
    # one launch of each kernel for the whole list
    names = _in_own_process(_list_form_launches)
    assert sum("k_rows_pack" in n for n in names) == 1 and sum("k_loss_tc" in n for n in names) == 1, names
    # a wide layer (D = 320) is outside the envelope: per-layer route, same numbers as calling it layer by layer
    g = torch.Generator().manual_seed(5)
    wide_q = torch.nn.functional.normalize(torch.randn(3 * 64, 320, generator=g), dim=1).cuda()
    wide_k = torch.nn.functional.normalize(torch.randn(3 * 64, 320, generator=g), dim=1).cuda()
    mixed = pn.rows_patchnce_multi([fq[0].detach(), wide_q], [fk[0], wide_k], 0.07, 64, batch_size=3)
    want = (pn.rows_patchnce(fq[0].detach(), fk[0], 0.07, 64, 3) + pn.rows_patchnce(wide_q, wide_k, 0.07, 64, 3)) / 2
    assert mixed.item() == pytest.approx(want.item(), rel=1e-6)


def test_rows_loss_matches_torch(pn):
    g = torch.Generator().manual_seed(41)
    b, p, dd = 3, 100, 48
    q = torch.nn.functional.normalize(torch.randn(b * p, dd, generator=g), dim=1)
    k = torch.nn.functional.normalize(torch.randn(b * p, dd, generator=g), dim=1)
    qd = q.cuda().requires_grad_()
    loss = pn.rows_patchnce(qd, k.cuda(), 0.07, num_patches=p)
    (loss * 2.5).backward()
    qc = q.clone().requires_grad_()
    acc = 0.0
    for i in range(b):
        z = (qc[i * p:(i + 1) * p] @ k[i * p:(i + 1) * p].t() / 0.07).clamp(-50, 50)
        acc = acc + torch.nn.functional.cross_entropy(z, torch.arange(p))
    want = acc / b
    (want * 2.5).backward()
    assert loss.item() == pytest.approx(want.item(), rel=2e-5)
    assert_grad_close(qd.grad.cpu().numpy(), qc.grad.numpy(), 1e-4, "dq")


def test_full_size_properties_b5(pn):
    """Size-independent properties at BASELINE's full sizes (B5 layer set, B=4, P=256):
    sparsity = unique(ids)*C per image, linearity in the upstream gradient, and the virtual-shard
    law of SURVEY.md 8e (same ids, batch split in two, losses averaged, grads halved)."""
    b = 4
    g = torch.Generator(device="cuda").manual_seed(99)
    src = [torch.randn(b, *s, device="cuda", generator=g).relu() for s in B5]
    tgt = [torch.randn(b, *s, device="cuda", generator=g).relu() for s in B5]
    ids = [torch.randint(0, s[1] * s[2], (256,), device="cuda", generator=g) for s in B5]

    def run(sl, scale):
        t = [x[sl].clone().requires_grad_() for x in tgt]
        loss = pn.fused_patchnce([x[sl] for x in src], t, ids, 0.07)
        (loss * scale).backward()
        return loss.detach(), [x.grad for x in t]

    loss, grads = run(slice(0, b), 1.0)
    loss2, grads2 = run(slice(0, b), 4.0)
    assert torch.equal(loss, loss2)
    for l, (ga, gb, i) in enumerate(zip(grads, grads2, ids)):
        u = torch.unique(i).numel()
        per_image = (ga != 0).reshape(b, -1).sum(1)
        assert torch.all(per_image <= u * B5[l][0])
        assert torch.all(per_image >= u * B5[l][0] - 8)         # an exact 0.0 entry is possible, barely
        mask = torch.zeros(B5[l][1] * B5[l][2], dtype=torch.bool, device="cuda")
        mask[i] = True
        assert not (ga.reshape(b, B5[l][0], -1)[:, :, ~mask] != 0).any()
        torch.testing.assert_close(gb, ga * 4.0, rtol=1e-6, atol=0)
    la, gA = run(slice(0, 2), 1.0)
    lb, gB = run(slice(2, 4), 1.0)
    assert ((la + lb) / 2).item() == pytest.approx(loss.item(), rel=1e-6)
    for ga, g1, g2 in zip(grads, gA, gB):
        torch.testing.assert_close(torch.cat([g1, g2]) / 2, ga, rtol=1e-5, atol=1e-12)


def test_stress_config_p1024_512(pn, orc):
    """BASELINE config 4 shape class: 512^2 maps, num_patches=1024 (one 256x128x128 layer, B=2),
    checked against the float64 analytic oracle."""
    g = torch.Generator().manual_seed(77)
    s = (256, 128, 128)
    src = [torch.randn(2, *s, generator=g)]
    tgt = [torch.randn(2, *s, generator=g)]
    ids = [torch.randint(0, s[1] * s[2], (1024,), generator=g)]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07)
    loss.backward()
    want, _, gw = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                 [i.numpy() for i in ids], 0.07)
    assert loss.item() == pytest.approx(want, rel=2e-5)
    assert_grad_close(t[0].grad.cpu().numpy(), gw[0], 1e-4, "P=1024")


def test_empty_and_mismatched_inputs(pn):
    with pytest.raises(ZeroDivisionError):
        pn.PatchNCELoss()([], [])
    a = torch.randn(1, 4, 4, 4, device="cuda")
    with pytest.raises(RuntimeError):
        pn.fused_patchnce([a], [torch.randn(1, 4, 5, 4, device="cuda")], [torch.zeros(4, dtype=torch.int64, device="cuda")])
    # zip truncation: 2 src maps, 1 tgt map -> one layer computed, divided by len(src_feats) = 2 (:36-40)
    torch.manual_seed(1)
    l2 = pn.PatchNCELoss(0.07, 8)([a, a], [a.clone()])
    torch.manual_seed(1)
    l1 = pn.PatchNCELoss(0.07, 8)([a], [a.clone()])
    assert l2.item() == pytest.approx(l1.item() / 2, rel=1e-6)


def _head_problem(seed, b, shapes, p):
    g = torch.Generator().manual_seed(seed)
    src = [torch.randn(b, *s, generator=g) for s in shapes]
    tgt = [torch.randn(b, *s, generator=g) for s in shapes]
    ids = [torch.randint(0, s[1] * s[2], (min(p, s[1] * s[2]),), generator=g) for s in shapes]
    return src, tgt, ids


@pytest.mark.parametrize("nc,fused", [(64, False), (256, False), (128, True), (256, True)])
def test_netf_head_matches_the_oracle(pn, orc, nc, fused):
    """North-star PatchSampleF(use_mlp=True) + PatchNCELoss(feat_q, feat_k): loss, dense d tgt and
    the head gradients against the oracle's torch restatement (PARITY UNPINNED by the reference,
    which has no head: SURVEY.md section 8 row a13).  Tolerance 1e-3 relative (north_star)."""
    shapes = [(64, 32, 32), (128, 16, 16), (24, 20, 12)]
    src, tgt, ids = _head_problem(123, 3, shapes, 64)
    torch.manual_seed(5)
    netF = pn.PatchSampleF(use_mlp=True, nc=nc, init_gain=0.3)
    netF.create_mlp([x.cuda() for x in tgt])
    for prm in netF.parameters():                           # non-zero biases so their gradients are exercised
        if prm.dim() == 1:
            torch.nn.init.normal_(prm, 0.0, 0.1)
    t = [x.cuda().requires_grad_() for x in tgt]
    idd = [i.cuda() for i in ids]
    loss, rid = pn.patchnce_with_head(netF, [x.cuda() for x in src], t, 0.07, 64, idd, fused=fused)
    (loss * 2.0).backward()
    assert pn.poll_nonfinite_warnings(block=True) == 0      # raises on a kernel protocol timeout
    assert all(torch.equal(a, b) for a, b in zip(rid, idd))
    heads = []
    for l in range(len(shapes)):
        mlp = getattr(netF, f"mlp_{l}")
        heads.append(tuple(x.detach().cpu().clone().requires_grad_()
                           for x in (mlp[0].weight, mlp[0].bias, mlp[2].weight, mlp[2].bias)))
    tc = [x.clone().requires_grad_() for x in tgt]
    want = orc.patchnce_head_loss_torch(src, tc, ids, heads)
    (want * 2.0).backward()
    assert loss.item() == pytest.approx(want.item(), rel=1e-3)
    for l in range(len(shapes)):
        assert_grad_close(t[l].grad.cpu().numpy(), tc[l].grad.numpy(), 1e-3, f"d tgt layer {l}", ids=ids[l])
        mlp = getattr(netF, f"mlp_{l}")
        for got, w, name in zip((mlp[0].weight, mlp[0].bias, mlp[2].weight, mlp[2].bias), heads[l],
                                ("W1", "b1", "W2", "b2")):
            assert_grad_close(got.grad.cpu().numpy(), w.grad.numpy(), 1e-3, f"d{name} layer {l}")


def test_netf_head_virtual_shard_law(pn):
    """SURVEY.md 8e with the head: same ids, batch split in two, head gradients averaged over the
    'ranks' equal the full-batch gradients (what allreduce_head_grads computes across GPUs)."""
    shapes = [(32, 16, 16), (48, 8, 8)]
    src, tgt, ids = _head_problem(9, 4, shapes, 32)
    torch.manual_seed(2)
    netF = pn.PatchSampleF(use_mlp=True, nc=64, init_gain=0.3)
    idd = [i.cuda() for i in ids]

    def run(sl):
        netF.zero_grad()
        t = [x[sl].cuda().requires_grad_() for x in tgt]
        loss, _ = pn.patchnce_with_head(netF, [x[sl].cuda() for x in src], t, 0.07, 32, idd)
        loss.backward()
        return loss.detach(), [p.grad.clone() for p in netF.parameters()]

    full, gfull = run(slice(0, 4))
    la, ga = run(slice(0, 2))
    lb, gb = run(slice(2, 4))
    assert ((la + lb) / 2).item() == pytest.approx(full.item(), rel=1e-5)
    for a, b, f in zip(ga, gb, gfull):
        torch.testing.assert_close((a + b) / 2, f, rtol=2e-4, atol=1e-7)


@pytest.mark.parametrize("p,c", [(300, 24), (600, 96), (1000, 256), (1024, 64)])
@pytest.mark.parametrize("math", ["tc_bf16x3", "simt_f32"])
def test_more_than_256_patches(pn, orc, p, c, math):
    """num_patches > 256 (BASELINE config 4 asks for 1024): the tcgen05 kernel walks the keys in
    blocks of 256 (two passes, logits recomputed for dZ); checked against the float64 oracle, with
    duplicate ids (the map has 1600 positions) and a second, small layer in the same launch."""
    g = torch.Generator().manual_seed(1000 * p + c)
    shapes = [(c, 40, 40), (16, 12, 12)]
    src = [torch.randn(2, *s, generator=g) for s in shapes]
    tgt = [torch.randn(2, *s, generator=g) for s in shapes]
    ids = [torch.randint(0, s[1] * s[2], (min(p, s[1] * s[2]),), generator=g) for s in shapes]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07, math=math)
    (loss * 1.5).backward()
    assert pn.poll_nonfinite_warnings(block=True) == 0
    want, _, gw = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                 [i.numpy() for i in ids], 0.07, upstream=1.5)
    assert loss.item() == pytest.approx(want, rel=2e-5)
    for l in range(2):
        assert_grad_close(t[l].grad.cpu().numpy(), gw[l], 2e-4, f"P={p} layer {l}", ids=ids[l].numpy())


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_precision_maps_head_and_many_patches(pn, orc, dtype):
    """The AMP regime of the real training loop (fp16 features under autocast, train_cutpp.py:268) through
    the two newer kernels: the fused netF head and the key-blocked path for num_patches > 256.  The oracle
    sees the same rounded inputs; the dense gradients come back in the maps' dtype."""
    g = torch.Generator().manual_seed(77)
    # (a) head, P <= 256
    shapes = [(48, 16, 16), (128, 12, 12)]
    src = [torch.randn(2, *s, generator=g).to(dtype) for s in shapes]
    tgt = [torch.randn(2, *s, generator=g).to(dtype) for s in shapes]
    ids = [torch.randint(0, s[1] * s[2], (96,), generator=g) for s in shapes]
    torch.manual_seed(3)
    netF = pn.PatchSampleF(use_mlp=True, nc=128, init_gain=0.3)
    t = [x.cuda().requires_grad_() for x in tgt]
    loss, _ = pn.patchnce_with_head(netF, [x.cuda() for x in src], t, 0.07, 96, [i.cuda() for i in ids], fused=True)
    loss.backward()
    heads = [tuple(x.detach().cpu().clone().requires_grad_() for x in
                   (getattr(netF, f"mlp_{l}")[0].weight, getattr(netF, f"mlp_{l}")[0].bias,
                    getattr(netF, f"mlp_{l}")[2].weight, getattr(netF, f"mlp_{l}")[2].bias)) for l in range(2)]
    tc = [x.float().clone().requires_grad_() for x in tgt]
    want = orc.patchnce_head_loss_torch([x.float() for x in src], tc, ids, heads)
    want.backward()
    assert loss.item() == pytest.approx(want.item(), rel=1e-3)
    for l in range(2):
        assert t[l].grad.dtype == dtype
        assert_grad_close(t[l].grad.float().cpu().numpy(), tc[l].grad.numpy(), 1e-2, f"head d tgt {l}", ids=ids[l])
        assert_grad_close(getattr(netF, f"mlp_{l}")[2].weight.grad.cpu().numpy(), heads[l][2].grad.numpy(), 1e-3, "dW2")
    # (b) 600 patches, no head
    s = (40, 32, 32)
    src = [torch.randn(2, *s, generator=g).to(dtype)]
    tgt = [torch.randn(2, *s, generator=g).to(dtype)]
    ids = [torch.randint(0, 1024, (600,), generator=g)]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07)
    loss.backward()
    want, _, gw = orc.patchnce_loss_and_grads_np([x.float().numpy() for x in src], [x.float().numpy() for x in tgt],
                                                 [i.numpy() for i in ids], 0.07)
    assert loss.item() == pytest.approx(want, rel=2e-5)
    assert_grad_close(t[0].grad.float().cpu().numpy(), gw[0], 1e-2, "P=600 half maps", ids=ids[0].numpy())
    assert pn.poll_nonfinite_warnings(block=True) == 0


def test_cuda_graph_capture_and_replay(pn, orc):
    """include/pnce.h promises that every entry point is asynchronous, sync-free and CUDA-graph
    capturable: capture forward + backward (ids drawn inside the graph, as the reference draws them),
    replay it, and check every replay against the oracle on the ids that replay drew."""
    g = torch.Generator().manual_seed(4)
    shapes = [(32, 24, 24), (64, 16, 16)]
    src = [torch.randn(2, *s, generator=g).cuda() for s in shapes]
    tgt = [torch.randn(2, *s, generator=g).cuda().requires_grad_() for s in shapes]
    crit = pn.PatchNCELoss(0.07, 128)
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
        loss = crit(src, tgt)
        loss.backward()
        ids_static = [i.clone() for i in crit.last_patch_ids]
    seen = []
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        ids = [i.cpu() for i in ids_static]
        seen.append(ids[0].clone())
        want, _, gw = orc.patchnce_loss_and_grads_np([x.cpu().numpy() for x in src],
                                                     [x.detach().cpu().numpy() for x in tgt],
                                                     [i.numpy() for i in ids], 0.07)
        assert loss.item() == pytest.approx(want, rel=2e-5)
        for l in range(2):
            assert_grad_close(tgt[l].grad.cpu().numpy(), gw[l], 2e-4, f"replay layer {l}", ids=ids[l].numpy())
    assert not torch.equal(seen[0], seen[1])            # the RNG stream advances from replay to replay


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_pinned_host_maps_zero_copy(pn, dtype):
    """Feature maps left in pinned HOST memory and passed through ``pinned_as_device`` (the gather reads
    the sampled sectors over PCIe) give bit-identical loss and gradients to device-resident copies."""
    g = torch.Generator().manual_seed(8)
    shapes = [(2, 32, 24, 24), (2, 64, 16, 16)]
    h_src = [torch.randn(s, generator=g).to(dtype).pin_memory() for s in shapes]
    h_tgt = [torch.randn(s, generator=g).to(dtype).pin_memory() for s in shapes]
    a_src = [pn.pinned_as_device(h) for h in h_src]
    a_tgt = [pn.pinned_as_device(h).requires_grad_() for h in h_tgt]
    d_src = [h.cuda() for h in h_src]
    d_tgt = [h.cuda().requires_grad_() for h in h_tgt]
    assert a_src[0].is_cuda and a_src[0].data_ptr() == h_src[0].data_ptr() and a_src[0].dtype == dtype
    crit = pn.PatchNCELoss(0.07, 128)
    torch.manual_seed(5)
    la = crit(a_src, a_tgt)
    la.backward()
    torch.manual_seed(5)
    ld = crit(d_src, d_tgt)
    ld.backward()
    assert la.item() == ld.item()
    for x, y in zip(a_tgt, d_tgt):
        assert x.grad.is_cuda and torch.equal(x.grad, y.grad)
    with pytest.raises(RuntimeError):
        pn.pinned_as_device(torch.randn(4, 4))            # pageable memory is refused


def test_side_stream_id_plan_gives_identical_results(pn, orc):
    """Large problems draw AND sort the ids on a side stream (pnce_plan_ids / pnce_fwd_planned /
    pnce_bwd_planned); forced here on a small ragged problem: bit-identical to the in-line path, and
    right against the oracle."""
    from gan_variant_research_b200 import patchnce as pmod
    g = torch.Generator().manual_seed(17)
    shapes = [(32, 24, 24), (64, 16, 16), (8, 3, 5), (128, 40, 40)]
    src = [torch.randn(3, *s, generator=g).cuda() for s in shapes]
    tgt_a = [torch.randn(3, *s, generator=g).cuda().requires_grad_() for s in shapes]
    tgt_b = [t.detach().clone().requires_grad_() for t in tgt_a]
    crit = pn.PatchNCELoss(0.07, 256)
    torch.manual_seed(9)
    la = crit(src, tgt_a)
    la.backward()
    ids_a = [i.clone() for i in crit.last_patch_ids]
    keep = pmod._SIDE_STREAM_MIN_BYTES
    pmod._SIDE_STREAM_MIN_BYTES = 0
    try:
        torch.manual_seed(9)
        lb = crit(src, tgt_b)
        (lb * 2.0).backward()
    finally:
        pmod._SIDE_STREAM_MIN_BYTES = keep
    assert all(torch.equal(a, b) for a, b in zip(ids_a, crit.last_patch_ids))
    assert la.item() == lb.item()
    for a, b in zip(tgt_a, tgt_b):
        assert torch.equal(a.grad * 2.0, b.grad)
    want, _, gw = orc.patchnce_loss_and_grads_np([x.cpu().numpy() for x in src],
                                                 [x.detach().cpu().numpy() for x in tgt_a],
                                                 [i.cpu().numpy() for i in ids_a], 0.07)
    assert la.item() == pytest.approx(want, rel=2e-5)
    for l in range(len(shapes)):
        assert_grad_close(tgt_a[l].grad.cpu().numpy(), gw[l], 2e-4, f"layer {l}", ids=ids_a[l].cpu().numpy())
    assert pn.poll_nonfinite_warnings(block=True) == 0


@pytest.mark.parametrize("b,c,h,w,p", [(5, 200, 20, 20, 200), (1, 130, 16, 16, 129), (7, 64, 12, 12, 256),
                                       (3, 255, 17, 15, 255), (2, 32, 128, 128, 160)])
def test_odd_shapes_against_the_oracle(pn, orc, b, c, h, w, p):
    """Channel counts that are not multiples of 32, patch counts that leave the second 128-row half of the
    logits partly empty, maps whose rows are not 16-byte multiples: persistent tcgen05 kernel vs the oracle."""
    g = torch.Generator().manual_seed(b * 1000 + c)
    src = [torch.randn(b, c, h, w, generator=g)]
    tgt = [torch.randn(b, c, h, w, generator=g)]
    ids = [torch.randint(0, h * w, (min(p, h * w),), generator=g)]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07)
    (loss * 0.5).backward()
    want, _, gw = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                 [i.numpy() for i in ids], 0.07, upstream=0.5)
    assert loss.item() == pytest.approx(want, rel=2e-5)
    assert_grad_close(t[0].grad.cpu().numpy(), gw[0], 2e-4, "odd shape", ids=ids[0].numpy())
    assert pn.poll_nonfinite_warnings(block=True) == 0


def test_eight_layers_is_the_limit(pn, orc):
    g = torch.Generator().manual_seed(88)
    shapes = [(8 + 8 * l, 6 + l, 5 + l) for l in range(8)]
    src = [torch.randn(2, *s, generator=g) for s in shapes]
    tgt = [torch.randn(2, *s, generator=g) for s in shapes]
    ids = [torch.randint(0, s[1] * s[2], (min(64, s[1] * s[2]),), generator=g) for s in shapes]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07)
    loss.backward()
    want, _, gw = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                 [i.numpy() for i in ids], 0.07)
    assert loss.item() == pytest.approx(want, rel=2e-5)
    for l in range(8):
        assert_grad_close(t[l].grad.cpu().numpy(), gw[l], 2e-4, f"layer {l}", ids=ids[l].numpy())
    with pytest.raises(RuntimeError):
        pn.fused_patchnce([x.cuda() for x in src] * 2, [x.cuda() for x in tgt] * 2, [i.cuda() for i in ids] * 2, 0.07)


@pytest.mark.parametrize("tau", [0.07, 0.03])            # logits near -14 / -33 (0.02 would sit exactly on the +-50 clamp)
@pytest.mark.parametrize("p", [1, 20, 150])
def test_all_logits_very_negative_with_padding_columns(pn, orc, tau, p):
    """Every real logit of a row far below zero while the last 32-column chunk holds padding columns (P not a
    multiple of 32): the sum of exp2 must not be formed as (sum incl. padding) - (pad count) -- found by
    scratch/stress.py with P = 1 / C = 1 layers.  Target patches point away from every source patch."""
    g = torch.Generator().manual_seed(p)
    v = torch.randn(1, 16, 1, 1, generator=g)
    src = [(v + 0.01 * torch.randn(2, 16, 12, 12, generator=g))]
    tgt = [(-v + 0.01 * torch.randn(2, 16, 12, 12, generator=g))]
    ids = [torch.randint(0, 144, (p,), generator=g)]
    for math in ("tc_bf16x3", "simt_f32"):
        t = [x.cuda().requires_grad_() for x in tgt]
        loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], tau, math=math)
        loss.backward()
        want, _, gw = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                     [i.numpy() for i in ids], tau)
        assert loss.item() == pytest.approx(want, rel=1e-4, abs=2e-5), (math, loss.item(), want)
        if p > 1:
            assert_grad_close(t[0].grad.cpu().numpy(), gw[0], 2e-3, f"{math} P={p}", ids=ids[0].numpy())
    assert pn.poll_nonfinite_warnings(block=True) == 0


@pytest.mark.parametrize("b", [300, 513])
def test_more_images_than_the_finalize_has_lanes(pn, orc, b):
    """Batches above 256 images: the last-CTA finalize sums the per-image losses with every thread of the launch
    (352 in the persistent kernel = 11 warps) -- its per-warp scratch used to hold 8 warps only, which batches up
    to 256 never noticed (threads >= 256 had nothing to add)."""
    g = torch.Generator().manual_seed(b)
    src = [torch.randn(b, 8, 6, 6, generator=g)]
    tgt = [torch.randn(b, 8, 6, 6, generator=g)]
    tgt[0][b - 1, :, :, :] = float("nan")                      # a guarded image handled by a thread of a high warp
    ids = [torch.randint(0, 36, (16,), generator=g)]
    for math in ("tc_bf16x3", "simt_f32"):
        t = [x.cuda().requires_grad_() for x in tgt]
        loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07, math=math)
        loss.backward()
        assert pn.poll_nonfinite_warnings(block=True) == 1
        want, _, gw = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                     [i.numpy() for i in ids], 0.07)
        assert loss.item() == pytest.approx(want, rel=2e-5), math
        assert_grad_close(t[0].grad.cpu().numpy(), gw[0], 2e-4, f"{math} B={b}")


@pytest.mark.parametrize("b,c,h,w,p", [(2, 8, 40, 40, 1280), (2, 512, 12, 12, 64), (1, 1024, 8, 8, 33), (2, 300, 36, 36, 1100)])
def test_largest_supported_shapes(pn, orc, b, c, h, w, p):
    """Outside the tensor-core envelope (P <= 1024, C <= 256) the fp32 CUDA-core kernels take over: up to 1280 patches
    (its 32-row logits tile must fit shared memory) and up to 1024 channels."""
    g = torch.Generator().manual_seed(c + p)
    src = [torch.randn(b, c, h, w, generator=g)]
    tgt = [torch.randn(b, c, h, w, generator=g)]
    ids = [torch.randint(0, h * w, (min(p, h * w),), generator=g)]
    t = [x.cuda().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce([x.cuda() for x in src], t, [i.cuda() for i in ids], 0.07)
    loss.backward()
    want, _, gw = orc.patchnce_loss_and_grads_np([x.numpy() for x in src], [x.numpy() for x in tgt],
                                                 [i.numpy() for i in ids], 0.07)
    assert loss.item() == pytest.approx(want, rel=2e-5)
    assert_grad_close(t[0].grad.cpu().numpy(), gw[0], 2e-4, "large shape", ids=ids[0].numpy())


@pytest.mark.parametrize("c,h,w,p", [(8, 40, 40, 1500), (8, 70, 70, 4096), (1025, 4, 4, 16)])
def test_shapes_beyond_the_limits_fail_loudly(pn, c, h, w, p):
    g = torch.Generator().manual_seed(1)
    src = [torch.randn(1, c, h, w, generator=g).cuda()]
    tgt = [torch.randn(1, c, h, w, generator=g).cuda().requires_grad_()]
    ids = [torch.randint(0, h * w, (min(p, h * w),), generator=g).cuda()]
    with pytest.raises(RuntimeError, match="outside compiled limits|not supported"):
        pn.fused_patchnce(src, tgt, ids, 0.07)


def test_loss_and_grads_equals_forward_backward(pn):
    """The autograd-free entry (forward + complete backward in one call) returns what loss.backward(g) leaves in .grad --
    bit for bit: same ids from the same generator state, same kernels."""
    g = torch.Generator().manual_seed(21)
    shapes = [(32, 24, 24), (64, 16, 16), (128, 40, 40)]
    src = [torch.randn(3, *s, generator=g).cuda() for s in shapes]
    tgt = [torch.randn(3, *s, generator=g).cuda().requires_grad_() for s in shapes]
    crit = pn.PatchNCELoss(0.07, 256)
    up = torch.tensor(2.5, device="cuda")
    torch.manual_seed(4)
    la = crit(src, tgt)
    la.backward(up)
    ids_a = [i.clone() for i in crit.last_patch_ids]
    after_a = torch.rand(3, device="cuda")
    torch.manual_seed(4)
    lb, grads = crit.loss_and_grads(src, [t.detach() for t in tgt], up)
    after_b = torch.rand(3, device="cuda")
    assert la.item() == lb.item() and torch.equal(after_a, after_b)
    assert all(torch.equal(a, b) for a, b in zip(ids_a, crit.last_patch_ids))
    for t, gr in zip(tgt, grads):
        assert gr.shape == t.shape and torch.equal(t.grad, gr)
    # unit upstream gradient when none is given; a truncated layer list is scaled like the reference (:36-40)
    torch.manual_seed(4)
    lc, gc = crit.loss_and_grads(src, [t.detach() for t in tgt])
    assert lc.item() == la.item()
    for a, b in zip(grads, gc):
        assert torch.allclose(a, b * 2.5, rtol=1e-6, atol=0)
    torch.manual_seed(4)
    ld, gd = crit.loss_and_grads(src, [t.detach() for t in tgt[:2]])
    torch.manual_seed(4)
    tg2 = [t.detach().clone().requires_grad_() for t in tgt[:2]]
    le = crit(src, tg2)
    le.backward()
    assert ld.item() == pytest.approx(le.item(), rel=1e-6)
    for a, t in zip(gd, tg2):
        assert torch.allclose(a, t.grad, rtol=1e-6, atol=0)
    assert pn.poll_nonfinite_warnings(block=True) == 0


def test_layers_of_mixed_dtype_and_batch_follow_the_reference_loop(pn, orc):
    """The reference handles every layer on its own (patchnce_cut.py:36-38): a list whose layers differ in dtype or
    batch size is valid input there.  One C-ABI call carries ONE dtype and batch, so such lists take a call per
    layer -- never a reinterpretation of another layer's memory."""
    g = torch.Generator().manual_seed(33)
    specs = [(2, 32, 12, 12, torch.float32), (3, 16, 10, 10, torch.float32), (2, 64, 8, 8, torch.float16)]
    src = [torch.randn(b, c, h, w, generator=g).to(dt) for b, c, h, w, dt in specs]
    tgt = [torch.randn(b, c, h, w, generator=g).to(dt) for b, c, h, w, dt in specs]
    t = [x.cuda().requires_grad_() for x in tgt]
    crit = pn.PatchNCELoss(0.07, 64)
    torch.manual_seed(12)
    loss = crit([x.cuda() for x in src], t)
    loss.backward()
    ids = crit.last_patch_ids
    assert len(ids) == 3
    want = 0.0
    for l in range(3):
        w, _, gw = orc.patchnce_loss_and_grads_np([src[l].float().numpy()], [tgt[l].float().numpy()], [ids[l].cpu().numpy()],
                                                  0.07, upstream=1.0 / 3.0)
        want += w / 3.0
        tol = 2e-4 if specs[l][4] == torch.float32 else 2e-2
        assert_grad_close(t[l].grad.float().cpu().numpy(), gw[0], tol, f"layer {l}", ids=ids[l].cpu().numpy())
    assert loss.item() == pytest.approx(want, rel=2e-4)
    with pytest.raises(RuntimeError):
        pn.fused_patchnce([x.cuda() for x in src], t, ids[:2], 0.07)          # fewer id tensors than layers


@pytest.mark.gpu
@pytest.mark.parametrize("nhwc", [False, True])
def test_head_loss_and_grads_equals_the_autograd_route(pn, nhwc):
    """The autograd-free head entry returns / leaves in .grad what patchnce_with_head(...).backward(g) does, bit for bit
    (same ids from the same generator state, same kernels), and accumulates into existing parameter gradients."""
    g = torch.Generator().manual_seed(33)
    shapes = [(32, 24, 24), (64, 16, 16), (128, 20, 20)]
    mf = torch.channels_last if nhwc else torch.contiguous_format
    src = [torch.randn(3, *s, generator=g).cuda().contiguous(memory_format=mf) for s in shapes]
    tgt = [torch.randn(3, *s, generator=g).cuda().contiguous(memory_format=mf).requires_grad_() for s in shapes]
    torch.manual_seed(2)
    netF = pn.PatchSampleF(use_mlp=True, nc=256).cuda()
    netF.create_mlp(tgt)
    for p_ in netF.parameters():                       # non-zero biases, larger weights than the 0.02 init
        p_.data.normal_(0.0, 0.1)
    up = torch.tensor(1.75, device="cuda")
    torch.manual_seed(9)
    la, ids_a = pn.patchnce_with_head(netF, src, tgt, 0.07, 64)
    la.backward(up)
    after_a = torch.rand(3, device="cuda")
    ref_p = [p_.grad.clone() for p_ in netF.parameters()]
    for p_ in netF.parameters():
        p_.grad = None
    torch.manual_seed(9)
    lb, grads, ids_b = pn.head_loss_and_grads(netF, src, [t.detach() for t in tgt], 0.07, 64, grad_output=up)
    after_b = torch.rand(3, device="cuda")
    assert la.item() == lb.item() and torch.equal(after_a, after_b)
    assert all(torch.equal(a, b) for a, b in zip(ids_a, ids_b))
    for t, gr in zip(tgt, grads):
        assert gr.shape == t.shape and torch.equal(t.grad, gr)
        assert gr.is_contiguous(memory_format=mf)
    for p_, r in zip(netF.parameters(), ref_p):
        assert p_.grad.shape == p_.shape and torch.equal(p_.grad, r)
    # a second call accumulates into the existing gradients, like autograd
    torch.manual_seed(9)
    pn.head_loss_and_grads(netF, src, [t.detach() for t in tgt], 0.07, 64, grad_output=up)
    for p_, r in zip(netF.parameters(), ref_p):
        assert torch.allclose(p_.grad, 2 * r, rtol=1e-6, atol=0)
    # unit upstream gradient when none is given; frozen parameters get no gradient
    for p_ in netF.parameters():
        p_.grad = None
    netF.mlp_1[0].weight.requires_grad_(False)
    torch.manual_seed(9)
    lc, gc, _ = pn.head_loss_and_grads(netF, src, [t.detach() for t in tgt], 0.07, 64)
    assert lc.item() == la.item() and netF.mlp_1[0].weight.grad is None
    for a, b in zip(grads, gc):
        assert torch.allclose(a, b * 1.75, rtol=1e-6, atol=1e-12)


@pytest.mark.gpu
def test_dense_gradients_in_compressible_memory_are_the_same_gradients(pn):
    """The dense gradients of large calls are allocated from a MemPool backed by the library's compressible allocator
    (csrc/comp_alloc.cuh).  Only the allocation differs: values are bit-identical to the default pool's, on the fused path
    (NCHW and channels-last), the fused head and the module-split backward; tensors behave like any other (clone, cpu,
    in-place math, freeing and re-use across steps)."""
    from gan_variant_research_b200 import _lib, patchnce as pm
    dev_ = torch.device("cuda", torch.cuda.current_device())
    supported = _lib.load().pnce_comp_supported(dev_.index) == 1
    g = torch.Generator().manual_seed(77)
    shapes = [(32, 40, 40), (64, 16, 16), (128, 24, 24)]
    src = [torch.randn(4, *s, generator=g).cuda() for s in shapes]
    tgt0 = [torch.randn(4, *s, generator=g).cuda() for s in shapes]
    old = (pm._GRAD_COMPRESSION, pm._GRAD_COMPRESSION_MIN_BYTES)
    try:
        results = {}
        for on in (False, True):
            pn.set_gradient_compression(on, min_bytes=0)
            for layout in ("nchw", "nhwc"):
                mf = torch.channels_last if layout == "nhwc" else torch.contiguous_format
                s_ = [x.clone(memory_format=mf) for x in src]
                for rep in range(3):                               # blocks are freed and re-used across steps
                    t_ = [x.detach().clone(memory_format=mf).requires_grad_() for x in tgt0]
                    torch.manual_seed(5)
                    loss = pn.PatchNCELoss(0.07, 128)(s_, t_)
                    loss.backward(torch.tensor(3.0, device="cuda"))
                grads = [t.grad for t in t_]
                if on and supported:
                    assert all(pn.gradient_is_compressed(x) for x in grads)
                if not on:
                    assert not any(pn.gradient_is_compressed(x) for x in grads)
                for x in grads:
                    assert x.is_contiguous(memory_format=mf)
                    x.mul_(1.0)                                    # ordinary tensors: in-place math, copies
                results[(on, layout)] = (loss.item(), [x.clone().cpu() for x in grads])
            torch.manual_seed(5)
            netF = pn.PatchSampleF(use_mlp=True, nc=128).cuda()
            t_ = [x.clone().requires_grad_() for x in tgt0]
            netF.create_mlp(t_)
            torch.manual_seed(6)
            hl, _ = pn.patchnce_with_head(netF, src, t_, 0.07, 128)
            hl.backward()
            results[(on, "head")] = (hl.item(), [t.grad.clone().cpu() for t in t_])
            t_ = [x.clone().requires_grad_() for x in tgt0]
            torch.manual_seed(6)
            rows, ids = pn.PatchSampleF()(t_, 128)
            ups = [torch.randn(r.shape, generator=torch.Generator().manual_seed(40 + i)).cuda() for i, r in enumerate(rows)]
            torch.autograd.backward(rows, ups)
            results[(on, "split")] = (0.0, [t.grad.clone().cpu() for t in t_])
        for key in ("nchw", "nhwc", "head", "split"):
            a, b = results[(False, key)], results[(True, key)]
            assert a[0] == b[0]
            for x, y in zip(a[1], b[1]):
                assert torch.equal(x, y), key
        torch.cuda.empty_cache()                                   # hands the pool's blocks back through pnce_comp_free
    finally:
        pn.set_gradient_compression(*old)
