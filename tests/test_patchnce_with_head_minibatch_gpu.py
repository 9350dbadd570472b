"""The netF head with minibatch negatives (patchnce_with_head_minibatch, head_minibatch_loss_and_grads) on the B200:
loss, dense d tgt and the four head gradients per layer against the float64 oracle (tests/head_minibatch_oracle.py) at
odd shapes, the benchmarked B5 regime and BASELINE config 4; the B = 1 identity with the per-image head; the
autograd-free route; layouts and dtypes; the group guard; CUDA graphs; the kernel list and memory; two ranks."""
import contextlib
import io
import os

import pytest
import torch

import head_minibatch_oracle as hmo
from test_parity_gpu import assert_grad_close

pytestmark = pytest.mark.gpu

B5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
CFG4 = [(c, 2 * h, 2 * w) for c, h, w in B5]             # BASELINE config 4: 512^2 images, P = 1024
# loss rel, gradient max-abs / max.  tc_bf16 rounds H, Y, dY and dH once each to bf16 (8 bits) and 1 / tau = 14
# amplifies that in the logits, hence the looser bound.
TOL = {"tc_bf16x3": (1e-3, 1e-3), "tc_bf16": (1e-2, 1.5e-1)}


def _q(x, step):
    """Round to multiples of ``step`` (a power of two): the maps (1/8, |x| <= 4) and W1, b1 (1/64, 1/512) are then exact in
    bf16, and X W1^T + b1 is exact in fp32 for C <= 256.  So the kernels' ReLU masks are the oracle's: a pre-activation
    within rounding of 0 would flip a mask, a jump of a whole entry of dH (at B = 64, N nc = 4 M pre-activations per
    layer), which no tolerance on a smooth function covers."""
    return torch.round(x / step).clamp(-4 / step, 4 / step) * step


@pytest.fixture(scope="module")
def pn():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gan_variant_research_b200 as m
    from gan_variant_research_b200 import _lib
    _lib.load()
    return m


@pytest.fixture(autouse=True)
def _release_device_memory():
    """The float64 oracle at B = 64 and the 512^2 maps hold tens of GB in the caching allocator: hand them back after each
    test, so that what runs later in the process (CUPTI's buffers for a profiler session among them) finds device memory."""
    yield
    import gc
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _maps(seed, b, shapes, dev="cuda"):
    g = torch.Generator(device=dev).manual_seed(seed)
    src = [torch.randn(b, *s, device=dev, generator=g) for s in shapes]
    tgt = [_q(0.6 * a + 0.8 * torch.randn(a.shape, device=dev, generator=g), 0.125) for a in src]
    return [_q(a, 0.125) for a in src], tgt


def _netf(pn, nc, feats, seed=5):
    torch.manual_seed(seed)
    netF = pn.PatchSampleF(use_mlp=True, nc=nc, init_gain=0.3)
    netF.create_mlp(feats)
    for prm in netF.parameters():                           # non-zero biases so their gradients are exercised
        if prm.dim() == 1:
            torch.nn.init.normal_(prm, 0.0, 0.1)
    with torch.no_grad():
        for l in range(len(feats)):
            lin = getattr(netF, f"mlp_{l}")[0]
            lin.weight.copy_(_q(lin.weight, 1 / 64))
            lin.bias.copy_(_q(lin.bias, 1 / 512))
    return netF


def _head_params(netF, n):
    return [[getattr(getattr(netF, f"mlp_{l}")[k], a) for k in (0, 2) for a in ("weight", "bias")] for l in range(n)]


def _ours(pn, netF, src, tgt, ids, math="tc_bf16x3", upstream=1.0, num_patches=None, tau=0.07):
    """-> (loss, d tgt per layer, head grads per layer, ids, guarded-layer count) through autograd."""
    netF.zero_grad(set_to_none=True)
    t = [x.detach().clone().requires_grad_() for x in tgt]
    np_ = num_patches if num_patches is not None else max(i.numel() for i in ids)
    loss, rid = pn.patchnce_with_head_minibatch(netF, src, t, tau, np_, ids, math)
    (loss * upstream).backward()
    n = pn.poll_nonfinite_warnings(block=True)
    return (loss.item(), [x.grad for x in t], [[p.grad for p in ps] for ps in _head_params(netF, len(src))], rid, n)


def _oracle(netF, src, tgt, ids, upstream=1.0, dev="cpu", tau=0.07):
    """float64 oracle on ``dev``: (loss, d tgt per layer, head grads per layer); None gradients read as zeros."""
    heads = [tuple(p.detach().to(dev, torch.float64).clone().requires_grad_() for p in ps)
             for ps in _head_params(netF, len(src))]
    t = [x.detach().to(dev, torch.float64).requires_grad_() for x in tgt]
    loss = hmo.head_minibatch_loss([x.to(dev, torch.float64) for x in src], t, [i.to(dev) for i in ids], heads, tau)
    if loss.requires_grad:
        (loss * upstream).backward()
    z = lambda x: torch.zeros_like(x) if x.grad is None else x.grad
    return loss.item(), [z(x) for x in t], [[z(w) for w in h] for h in heads]


def _check(got, want, ids, tol, what=""):
    (loss, gt, gh), (rl, rt, rh) = got, want
    lt, ght = tol
    assert loss == pytest.approx(rl, rel=lt), what
    for l, (a, r) in enumerate(zip(gt, rt)):
        assert_grad_close(a.float().cpu().numpy(), r.cpu().numpy(), ght, f"{what} d tgt layer {l}", ids=ids[l].cpu().numpy())
        for name, x, y in zip(("W1", "b1", "W2", "b2"), gh[l], rh[l]):
            assert_grad_close(x.cpu().numpy(), y.cpu().numpy(), ght, f"{what} d{name} layer {l}")


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("nc,b,shapes,p", [
    (128, 3, [(64, 32, 32), (128, 16, 16), (24, 20, 12)], 64),
    (256, 2, [(40, 24, 24), (256, 20, 20)], 300),          # P not a multiple of 128: two key blocks per image
    (128, 2, [(64, 40, 40)], 1024),                         # four key blocks per image
    (256, 5, [(32, 16, 16)], 64),
])
def test_matches_the_float64_oracle(pn, nc, b, shapes, p, math):
    src, tgt = _maps(b * 31 + p, b, shapes)
    g = torch.Generator(device="cuda").manual_seed(p)
    ids = [torch.randint(0, h * w, (min(p, h * w),), device="cuda", generator=g) for _, h, w in shapes]
    netF = _netf(pn, nc, tgt)
    loss, gt, gh, rid, n = _ours(pn, netF, src, tgt, ids, math, upstream=1.5)
    assert n == 0 and all(torch.equal(a, r) for a, r in zip(rid, ids))
    _check((loss, gt, gh), _oracle(netF, src, tgt, ids, upstream=1.5), ids, TOL[math], math)


def _library_drawn(pn, netF, src, tgt, p, seed):
    """The ids the call draws are torch.randint's from the same generator state, as for the per-image head."""
    dev = torch.device("cuda")
    gen = torch.cuda.default_generators[0]
    torch.manual_seed(seed)
    off0 = gen.get_offset()
    netF.zero_grad(set_to_none=True)
    t = [x.detach().clone().requires_grad_() for x in tgt]
    loss, ids = pn.patchnce_with_head_minibatch(netF, src, t, 0.07, p)
    loss.backward()
    off1 = gen.get_offset()
    torch.manual_seed(seed)
    ref = [torch.randint(0, h * w, (min(p, h * w),), device=dev) for _, _, h, w in (x.shape for x in src)]
    assert gen.get_offset() - off0 == off1 - off0
    assert all(torch.equal(a, r) for a, r in zip(ids, ref))
    assert pn.poll_nonfinite_warnings(block=True) == 0
    return (loss.item(), [x.grad for x in t], [[q.grad for q in ps] for ps in _head_params(netF, len(src))]), ids


@pytest.mark.parametrize("batch", [16, 64])
def test_b5_full_size_with_library_drawn_ids(pn, batch):
    src, tgt = _maps(batch, batch, B5)
    netF = _netf(pn, 256, tgt)
    got, ids = _library_drawn(pn, netF, src, tgt, 256, 123)
    _check(got, _oracle(netF, src, tgt, ids, dev="cuda"), ids, TOL["tc_bf16x3"], f"B5 B={batch}")


def test_config4_512sq_p1024(pn):
    src, tgt = _maps(4, 8, CFG4)
    netF = _netf(pn, 256, tgt)
    got, ids = _library_drawn(pn, netF, src, tgt, 1024, 77)
    _check(got, _oracle(netF, src, tgt, ids, dev="cuda"), ids, TOL["tc_bf16x3"], "config 4")


def test_batch_of_one_is_bit_identical_to_the_per_image_head(pn):
    src, tgt = _maps(1, 1, B5)
    netF = _netf(pn, 256, tgt)
    out = []
    for fn in (pn.patchnce_with_head, pn.patchnce_with_head_minibatch):
        netF.zero_grad(set_to_none=True)
        t = [x.clone().requires_grad_() for x in tgt]
        torch.manual_seed(7)
        loss, ids = fn(netF, src, t, 0.07, 256)
        loss.backward(torch.tensor(1.25, device="cuda"))
        out.append((loss.detach(), ids, [x.grad for x in t], [q.grad.clone() for q in netF.parameters()]))
    (la, ia, ga, pa), (lb, ib, gb, pb) = out
    assert torch.equal(la, lb)
    for a, b in zip(ia + ga + pa, ib + gb + pb):
        assert torch.equal(a, b)


@pytest.mark.parametrize("nhwc", [False, True])
def test_autograd_free_route_equals_autograd_bit_for_bit(pn, nhwc):
    mf = torch.channels_last if nhwc else torch.contiguous_format
    src, tgt = _maps(33, 6, [(32, 24, 24), (64, 16, 16), (128, 20, 20)])
    src = [x.contiguous(memory_format=mf) for x in src]
    tgt = [x.contiguous(memory_format=mf) for x in tgt]
    netF = _netf(pn, 256, tgt)
    up = torch.tensor(1.75, device="cuda")
    netF.zero_grad(set_to_none=True)
    la = []
    for k in range(2):                                   # two steps: the second accumulates into .grad
        t = [x.clone().requires_grad_() for x in tgt]
        torch.manual_seed(9)
        loss, ids_a = pn.patchnce_with_head_minibatch(netF, src, t, 0.07, 64)
        loss.backward(up)
        la.append(loss.detach())
        if k == 0:
            one = [q.grad.clone() for q in netF.parameters()]
            tg = [x.grad for x in t]
    after_a = torch.rand(3, device="cuda")
    ref = [q.grad.clone() for q in netF.parameters()]
    netF.zero_grad(set_to_none=True)
    for k in range(2):
        torch.manual_seed(9)
        lb, grads, ids_b = pn.head_minibatch_loss_and_grads(netF, src, tgt, 0.07, 64, grad_output=up)
        assert torch.equal(lb, la[k]) and all(torch.equal(a, b) for a, b in zip(ids_a, ids_b))
        if k == 0:
            for q, r in zip(netF.parameters(), one):
                assert torch.equal(q.grad, r)
            for x, r in zip(grads, tg):
                assert torch.equal(x, r) and x.is_contiguous(memory_format=mf)
    after_b = torch.rand(3, device="cuda")
    assert torch.equal(after_a, after_b)
    for q, r in zip(netF.parameters(), ref):
        assert torch.equal(q.grad, r)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_channels_last_and_half_maps(pn, dtype):
    shapes = [(64, 16, 16), (32, 24, 24)]
    src, tgt = _maps(5, 6, shapes)
    src, tgt = [x.to(dtype) for x in src], [x.to(dtype) for x in tgt]
    netF = _netf(pn, 128, [x.float() for x in tgt])
    g = torch.Generator(device="cuda").manual_seed(3)
    ids = [torch.randint(0, h * w, (200,), device="cuda", generator=g) for _, h, w in shapes]
    res = []
    for fmt in (torch.contiguous_format, torch.channels_last):
        res.append(_ours(pn, netF, [x.contiguous(memory_format=fmt) for x in src],
                         [x.contiguous(memory_format=fmt) for x in tgt], ids))
        assert res[-1][4] == 0
    (la, ga, ha, _, _), (lb, gb, hb, _, _) = res
    assert lb == pytest.approx(la, rel=1e-6)
    for a, b in zip(ga, gb):
        assert b.is_contiguous(memory_format=torch.channels_last) and b.dtype == dtype
        torch.testing.assert_close(b.float(), a.float(), rtol=1e-2 if dtype != torch.float32 else 1e-5,
                                   atol=1e-3 * a.float().abs().max().item())
    for x, y in zip(sum(ha, []), sum(hb, [])):
        torch.testing.assert_close(y, x, rtol=1e-5, atol=1e-6 * x.abs().max().item())
    # against the oracle on the values the half maps hold (the oracle casts to float64)
    tol = TOL["tc_bf16x3"] if dtype == torch.float32 else (1e-3, 1e-2)    # gradients stored in the half dtype
    _check((la, ga, ha), _oracle(netF, src, tgt, ids), ids, tol, str(dtype))


def test_nan_in_one_layer_zeroes_that_layer_only(pn, capsys):
    shapes = [(64, 32, 32), (128, 16, 16), (24, 20, 12)]
    src, tgt = _maps(8, 3, shapes)
    g = torch.Generator(device="cuda").manual_seed(8)
    ids = [torch.randint(0, h * w, (64,), device="cuda", generator=g) for _, h, w in shapes]
    pos = ids[1][5].item()
    tgt[1][2, 7].view(-1)[pos] = float("nan")              # one element of a sampled target patch, layer 1, image 2
    netF = _netf(pn, 128, tgt)
    capsys.readouterr()
    loss, gt, gh, _, n = _ours(pn, netF, src, tgt, ids)
    out = capsys.readouterr().out
    assert n == 1 and out.count("Warning: NaN in PatchNCE loss (minibatch negatives)") == 1
    assert (gt[1] == 0).all() and all((x == 0).all() for x in gh[1])
    want = _oracle(netF, src, tgt, ids)
    assert want[0] != 0.0 and (want[1][1] == 0).all()
    _check((loss, gt, gh), want, ids, TOL["tc_bf16x3"], "nan")
    # a NaN on the key side guards the layer as well
    src[2][0, 3].view(-1)[ids[2][0].item()] = float("inf")
    tgt[1][2, 7].view(-1)[pos] = 0.0
    loss2, gt2, gh2, _, n2 = _ours(pn, netF, src, tgt, ids)
    assert n2 == 1 and (gt2[2] == 0).all() and all((x == 0).all() for x in gh2[2])
    _check((loss2, gt2, gh2), _oracle(netF, src, tgt, ids), ids, TOL["tc_bf16x3"], "inf key")
    capsys.readouterr()


def test_cuda_graph_replay_equals_eager(pn):
    shapes = [(64, 32, 32), (128, 16, 16)]
    src, tgt = _maps(4, 8, shapes)
    tgt = [x.requires_grad_() for x in tgt]
    netF = _netf(pn, 256, tgt)
    g = torch.Generator(device="cuda").manual_seed(4)
    ids = [torch.randint(0, h * w, (256,), device="cuda", generator=g) for _, h, w in shapes]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                          # warm-up outside the capture (lazy init, smem opt-in)
        for _ in range(2):
            netF.zero_grad(set_to_none=True)
            for t in tgt:
                t.grad = None
            pn.patchnce_with_head_minibatch(netF, src, tgt, 0.07, 256, ids)[0].backward()
    torch.cuda.current_stream().wait_stream(side)
    for t in tgt:
        t.grad = None
    netF.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gl, _ = pn.patchnce_with_head_minibatch(netF, src, tgt, 0.07, 256, ids)
        gl.backward()
    gg = [t.grad for t in tgt]                             # the buffers every replay writes
    gp = [q.grad for q in netF.parameters()]
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        loss, gt, gh, _, _ = _ours(pn, netF, src, tgt, ids)
        assert gl.item() == loss
        for a, b in zip(gg + gp, gt + sum(gh, [])):
            assert torch.equal(a, b)


def _launch_list_worker(out_path):
    """The kernels of one forward at B = 64 (B5, nc = 256), written to ``out_path``.  Run in a process of its own: the
    profiler session then leaves no CUPTI state behind in the test process, whose later tests profile their own
    launches."""
    import gan_variant_research_b200 as pn
    from torch.profiler import ProfilerActivity, profile
    src, tgt = _maps(2, 64, B5)
    netF = _netf(pn, 256, tgt)
    tgt = [x.requires_grad_() for x in tgt]
    pn.patchnce_with_head_minibatch(netF, src, tgt, 0.07, 256)[0].backward()      # warm: workspace, smem opt-in
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss, _ = pn.patchnce_with_head_minibatch(netF, src, tgt, 0.07, 256)
        torch.cuda.synchronize()
    torch.save([e.key for e in prof.key_averages() if e.device_time_total > 0], out_path)


def test_kernel_list_and_memory_at_b64(pn, tmp_path):
    import multiprocessing as mp
    proc = mp.get_context("spawn").Process(target=_launch_list_worker, args=(str(tmp_path / "names.pt"),))
    proc.start()
    proc.join(timeout=600)
    if proc.is_alive():
        proc.kill()
        proc.join()
    assert proc.exitcode == 0, proc.exitcode
    names = torch.load(str(tmp_path / "names.pt"))
    kernels = [n for n in names if "memcpy" not in n.lower() and "memset" not in n.lower()]
    assert any("k_loss_tc_mb(" in n for n in kernels), kernels
    assert not [n for n in kernels if "k_loss_tc(" in n or "k_loss_tc_p" in n or "k_loss_tc_mb_gn" in n], kernels
    # libpnce's kernels only (k_draw_ids is outside the namespace), besides torch's id draw when it takes over
    foreign = [n for n in kernels if not (n.startswith("k_") or "pnce::k_" in n)
               and "random" not in n.lower() and "distribution" not in n.lower()]
    assert not foreign, foreign
    # peak memory of a forward + backward above the inputs, the gradients and the workspace
    src, tgt = _maps(2, 64, B5)
    netF = _netf(pn, 256, tgt)
    tgt = [x.requires_grad_() for x in tgt]
    pn.patchnce_with_head_minibatch(netF, src, tgt, 0.07, 256)[0].backward()
    netF.zero_grad(set_to_none=True)
    for t in tgt:
        t.grad = None
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    pn.patchnce_with_head_minibatch(netF, src, tgt, 0.07, 256)[0].backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    grads = sum(t.numel() * 4 for t in tgt) + sum(q.numel() * 4 for q in netF.parameters())
    ws = max(v for k, v in pn.patchnce._HEAD_WS_BYTES.items() if k[4] and k[5][0][0] == 64)
    n = 64 * 256
    assert peak - grads - ws < n * n * 4, (peak, grads, ws)


# ---- two processes through the public API ----------------------------------------------------------------------------
SHAPES2 = [(64, 32, 32), (128, 16, 16), (32, 24, 24)]


def _worker(rank, world, init_file, out_dir):
    import torch.distributed as dist
    import gan_variant_research_b200 as pn
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        src, tgt = _maps(21, 8, SHAPES2)
        netF = _netf(pn, 128, tgt)
        g = torch.Generator(device="cuda").manual_seed(21)
        ids = [torch.randint(0, h * w, (128,), device="cuda", generator=g) for _, h, w in SHAPES2]
        sl = slice(rank * 4, rank * 4 + 4)
        t = [x[sl].clone().requires_grad_() for x in tgt]
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            loss, _ = pn.patchnce_with_head_minibatch(netF, [x[sl] for x in src], t, 0.07, 128, ids, dp_group=True)
            loss.backward()
            la = loss.item()
            agrad = [q.grad.clone().cpu() for q in netF.parameters()]
            netF.zero_grad(set_to_none=True)
            lb, grads, _ = pn.head_minibatch_loss_and_grads(netF, [x[sl] for x in src], [x[sl] for x in tgt], 0.07, 128,
                                                            ids, dp_group=True)
            fgrad = [q.grad.clone().cpu() for q in netF.parameters()]
        torch.save({"loss": la, "loss_free": lb.item(), "agrad": agrad, "fgrad": fgrad,
                    "dtgt": [x.grad.cpu() for x in t], "dtgt_free": [x.cpu() for x in grads]},
                   os.path.join(out_dir, f"rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_processes_on_one_gpu_gloo(pn, tmp_path):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, 2, str(tmp_path / "init"), str(tmp_path))) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    res = [torch.load(str(tmp_path / f"rank{r}.pt"), weights_only=False) for r in range(2)]
    src, tgt = _maps(21, 8, SHAPES2)
    netF = _netf(pn, 128, tgt)
    g = torch.Generator(device="cuda").manual_seed(21)
    ids = [torch.randint(0, h * w, (128,), device="cuda", generator=g) for _, h, w in SHAPES2]
    shards = [_oracle(netF, [x[r * 4:r * 4 + 4] for x in src], [x[r * 4:r * 4 + 4] for x in tgt], ids) for r in range(2)]
    mean = [(a + b) / 2 for a, b in zip(sum(shards[0][2], []), sum(shards[1][2], []))]
    for r in range(2):
        assert res[r]["loss"] == pytest.approx(shards[r][0], rel=1e-3)            # the rank's own shard as negatives
        assert res[r]["loss_free"] == res[r]["loss"]
        for k, (a, e) in enumerate(zip(res[r]["agrad"], mean)):
            assert_grad_close(a.numpy(), e.numpy(), 1e-3, f"rank {r} head grad {k}")
            assert torch.equal(a, res[r]["fgrad"][k])
        for l, (a, e) in enumerate(zip(res[r]["dtgt"], shards[r][1])):
            assert_grad_close(a.numpy(), e.numpy(), 1e-3, f"rank {r} d tgt {l}", ids=ids[l].cpu().numpy())
            assert torch.equal(a, res[r]["dtgt_free"][l])
