"""Global negatives (``negatives_group``) on the B200: W = 1 is today's minibatch call; virtual shards in one process
through the C ABI (slots exchanged by device copies) against the one-process minibatch result; two processes on one GPU
(gloo) and on two GPUs (NCCL) through the public API; the global guard; the kernel list and memory."""
import contextlib
import ctypes
import glob
import io
import os

import numpy as np
import pytest
import torch

import global_negatives_oracle as gno

pytestmark = pytest.mark.gpu

SMALL = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "small_*.npz")))
IDS = [os.path.basename(p)[6:-4] for p in SMALL]
B5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
TOL = {"tc_bf16x3": (2e-5, 2e-4), "tc_bf16": (2e-3, 3e-2)}     # vs the float64 oracle: loss rel, gradient max-abs / max
# shards vs one process: the same per-row arithmetic (an item walks the same key blocks in the same order), only the
# fp32 sums of the row losses are grouped per rank
REORDER = (1e-5, 1e-5)


@pytest.fixture(scope="module")
def pn():
    import gan_variant_research_b200 as pn
    return pn


def _layer_array(src, tgt, ids, dtgt=None):
    from gan_variant_research_b200 import _lib
    arr = (_lib.PnceLayer * len(tgt))()
    for l, (s, t, i) in enumerate(zip(src, tgt, ids)):
        arr[l].src, arr[l].tgt, arr[l].ids = s.data_ptr(), t.data_ptr(), i.data_ptr()
        arr[l].dtgt = dtgt[l].data_ptr() if dtgt is not None else None
        arr[l].C, arr[l].H, arr[l].W, arr[l].P = t.shape[1], t.shape[2], t.shape[3], i.numel()
    return arr


def _virtual_shards(src, tgt, ids, tau, math, world):
    """W ranks in one process through the C ABI: keys of every rank, the slot exchange as device copies between the W
    workspaces, then the loss and the backward of every rank.  -> ([loss_r], [[grad_l of rank r]], [nonfinite_r])."""
    from gan_variant_research_b200 import _lib
    lib = _lib.load()
    n, b = len(tgt), tgt[0].shape[0]
    bl = b // world
    dcode = {torch.float32: _lib.PNCE_F32, torch.float16: _lib.PNCE_F16, torch.bfloat16: _lib.PNCE_BF16}[tgt[0].dtype]
    mcode = {"tc_bf16x3": _lib.MATH_TC_BF16X3, "tc_bf16": _lib.MATH_TC_BF16}[math]
    nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    shard = lambda xs, r: [x[r * bl:(r + 1) * bl] for x in xs]
    _lib.check(lib.pnce_mb_shard_workspace_bytes(_layer_array(shard(src, 0), shard(tgt, 0), ids), n, bl, world,
                                                 ctypes.byref(nb), ctypes.byref(off), ctypes.byref(sb)), "ws")
    st = torch.cuda.current_stream().cuda_stream
    ws = [torch.empty(nb.value, dtype=torch.uint8, device="cuda") for _ in range(world)]
    grads = [[torch.empty_like(t) for t in shard(tgt, r)] for r in range(world)]
    arrs = [_layer_array(shard(src, r), shard(tgt, r), ids, grads[r]) for r in range(world)]
    for r in range(world):
        _lib.check(lib.pnce_mb_shard_keys(arrs[r], n, bl, dcode, _lib.LAYOUT_NCHW, world, r, mcode, ws[r].data_ptr(),
                                          nb.value, None, 0, None, st), "pnce_mb_shard_keys")
    slot = lambda w: slice(off.value + w * sb.value, off.value + (w + 1) * sb.value)
    for r in range(world):
        for w in range(world):
            if w != r:
                ws[r][slot(w)].copy_(ws[w][slot(w)])
    outs = [torch.empty(1 + n, device="cuda") for _ in range(world)]
    flags = [torch.zeros(2, dtype=torch.int32, device="cuda") for _ in range(world)]
    for r in range(world):
        _lib.check(lib.pnce_mb_shard_loss(arrs[r], n, bl, dcode, _lib.LAYOUT_NCHW, world, r, tau, mcode,
                                          ws[r].data_ptr(), nb.value, None, 0, outs[r].data_ptr(), flags[r].data_ptr(),
                                          st), "pnce_mb_shard_loss")
        _lib.check(lib.pnce_bwd_ex(arrs[r], n, bl, dcode, _lib.LAYOUT_NCHW, mcode, ws[r].data_ptr(), nb.value, None, 0,
                                   None, st), "pnce_bwd_ex")
    torch.cuda.synchronize()
    return [o[0].item() for o in outs], grads, [int(f[0].item()) for f in flags]


def _one_process(pn, src, tgt, ids, tau, math):
    t = [x.detach().clone().requires_grad_() for x in tgt]
    loss = pn.fused_patchnce(src, t, ids, tau, math, nce_includes_all_negatives_from_minibatch=True)
    loss.backward()
    return loss.item(), [x.grad for x in t]


def _compare_shards(pn, src, tgt, ids, tau, math, world):
    losses, grads, _ = _virtual_shards(src, tgt, ids, tau, math, world)
    ref_loss, ref_grads = _one_process(pn, src, tgt, ids, tau, math)
    bl = tgt[0].shape[0] // world
    assert float(np.mean(losses)) == pytest.approx(ref_loss, rel=REORDER[0], abs=1e-7)
    worst = 0.0
    for l, ref in enumerate(ref_grads):
        for r in range(world):
            a, e = grads[r][l].double() / world, ref[r * bl:(r + 1) * bl].double()
            assert torch.equal(torch.isnan(a), torch.isnan(e))
            fin = torch.isfinite(e)
            scale = max(e[fin].abs().max().item() if fin.any() else 0.0, 1e-30)
            worst = max(worst, (a[fin] - e[fin]).abs().max().item() / scale if fin.any() else 0.0)
    assert worst <= REORDER[1]
    return losses, grads, ref_loss, worst


def test_group_of_one_rank_is_todays_minibatch_call(pn):
    """negatives_group=True without a process group: the same launches and bit-identical results."""
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1)
    shapes = [(64, 32, 32), (128, 16, 16)]
    src = [torch.randn(8, *s, device=dev, generator=g) for s in shapes]
    tgt = [torch.randn(8, *s, device=dev, generator=g) for s in shapes]
    res = []
    for group in (None, True):
        crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True, negatives_group=group)
        t = [x.clone().requires_grad_() for x in tgt]
        torch.manual_seed(5)
        crit(src, t).backward()                                     # warm
        t = [x.clone().requires_grad_() for x in tgt]
        torch.manual_seed(5)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            loss = crit(src, t)
            loss.backward()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
        res.append((loss.detach(), [x.grad for x in t], names))
    assert res[0][2] == res[1][2] and any("k_loss_tc_mb" in n for n in res[0][2])
    assert torch.equal(res[0][0], res[1][0])
    for a, b in zip(res[0][1], res[1][1]):
        assert torch.equal(a, b)


def _tiled(path, batch):
    d = np.load(path)
    layers = []
    for i in range(int(d["n_layers"])):
        idx = np.arange(batch) % d[f"src{i}"].shape[0]
        layers.append((d[f"src{i}"][idx], d[f"tgt{i}"][idx], d[f"ids{i}"]))
    return float(d["tau"]), layers


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("path", SMALL, ids=IDS)
def test_virtual_shards_on_the_small_fixtures(pn, path, world, math):
    tau, layers = _tiled(path, 8)
    dev = torch.device("cuda")
    src = [torch.from_numpy(s).to(dev, torch.float32) for s, _, _ in layers]
    tgt = [torch.from_numpy(t).to(dev, torch.float32) for _, t, _ in layers]
    ids = [torch.from_numpy(i).to(dev, torch.int64) for _, _, i in layers]
    losses, grads, _, _ = _compare_shards(pn, src, tgt, ids, tau, math, world)
    # and each shard against the float64 shard oracle
    rl, rg = TOL[math]
    if math == "tc_bf16" and tau < 0.05:
        return                                   # the clamp-binding fixture: covered against one process above
    n = len(layers)
    for r in range(world):
        ref = [gno.layer_loss_and_grad_np_shard(s, t, i, tau, world, r, n) for s, t, i in layers]
        assert losses[r] == pytest.approx(sum(l for l, _ in ref) / n, rel=rl, abs=1e-6)
        for g, (_, e) in zip(grads[r], ref):
            g = g.cpu().numpy()
            np.testing.assert_array_equal(np.isnan(g), np.isnan(e))
            fin = np.isfinite(e)
            assert np.abs(g[fin] - e[fin]).max(initial=0.0) <= rg * max(np.abs(e[fin]).max(initial=0.0), 1e-30)


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("case", ["b5_16", "b5_64", "p1024_8"])
def test_virtual_shards_at_full_size(pn, case, world, math):
    dev = torch.device("cuda")
    shapes, batch, p = {"b5_16": (B5, 16, 256), "b5_64": (B5, 64, 256), "p1024_8": ([(64, 512, 512)], 8, 1024)}[case]
    g = torch.Generator(device=dev).manual_seed(batch + p + world)
    src = [torch.randn(batch, *s, device=dev, generator=g) for s in shapes]
    tgt = [0.5 * a + torch.randn(a.shape, device=dev, generator=g) for a in src]
    ids = [torch.randint(0, s[1] * s[2], (p,), device=dev, generator=g) for s in shapes]
    losses, _, ref_loss, worst = _compare_shards(pn, src, tgt, ids, 0.07, math, world)
    print(f"{case} W={world} {math}: mean shard loss {np.mean(losses):.7f} vs one process {ref_loss:.7f}, "
          f"gradient max |shard / W - one process| / max = {worst:.2e}")


def test_kernels_and_memory_of_a_shard(pn):
    """The per-rank forward and backward: k_loss_tc_mb and no ATen GEMM, bmm or softmax; peak memory above the inputs,
    the gradients and the workspace stays below one N_l x N fp32 logits buffer."""
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda")
    world, batch = 2, 64
    src = [torch.randn(batch, *s, device=dev) for s in B5]
    tgt = [torch.randn(batch, *s, device=dev) for s in B5]
    ids = [torch.randint(0, s[1] * s[2], (256,), device=dev) for s in B5]
    _virtual_shards(src, tgt, ids, 0.07, "tc_bf16x3", world)           # warm
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _virtual_shards(src, tgt, ids, 0.07, "tc_bf16x3", world)
    names = [e.key for e in prof.key_averages()]
    assert any("k_loss_tc_mb" in n for n in names), names
    banned = ("gemm", "bmm", "softmax", "cutlass", "cublas", "nvjet", "sm90_xmma", "sm100_xmma")
    assert not [n for n in names if any(b in n.lower() for b in banned)], names
    peak = torch.cuda.max_memory_allocated() - base
    from gan_variant_research_b200 import _lib
    nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    bl = batch // world
    _lib.check(_lib.load().pnce_mb_shard_workspace_bytes(_layer_array([s[:bl] for s in src], [t[:bl] for t in tgt], ids),
                                                         5, bl, world, ctypes.byref(nb), ctypes.byref(off),
                                                         ctypes.byref(sb)), "ws")
    grads = sum(t.numel() * 4 for t in tgt)                           # every rank's gradients together
    n_l, n = bl * 256, batch * 256
    assert peak - grads - world * nb.value < n_l * n * 4, (peak, grads, nb.value)


# ---- two processes through the public API ----------------------------------------------------------------------------
SHAPES2 = [(64, 32, 32), (128, 16, 16), (32, 24, 24)]


def _inputs(batch, dtype, channels_last, nan_layer=None):
    g = torch.Generator().manual_seed(21)
    src = [torch.randn(batch, *s, generator=g) for s in SHAPES2]
    tgt = [0.6 * a + 0.8 * torch.randn(a.shape, generator=g) for a in src]
    if nan_layer is not None:
        tgt[nan_layer][batch - 1, 3, 2, :] = float("nan")              # a row of the last image: rank 1's shard
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    cast = lambda xs: [x.to(dtype).contiguous(memory_format=fmt) for x in xs]
    return cast(src), cast(tgt)


def _step(pn, src, tgt, group, seed):
    """(loss, layer losses, grads via autograd, loss and grads via loss_and_grads, ids); ids drawn by the library."""
    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True, negatives_group=group)
    t = [x.clone().requires_grad_() for x in tgt]
    torch.manual_seed(seed)
    loss = crit(src, t)
    loss.backward()
    ids = [i.clone() for i in crit.last_patch_ids]
    torch.manual_seed(seed)
    loss2, g2 = crit.loss_and_grads(src, tgt)
    return loss.detach(), [x.grad for x in t], loss2, g2, ids


def _worker(rank, world, backend, init_file, out_dir, cases, nan_layer):
    import torch.distributed as dist
    import gan_variant_research_b200 as pn
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        res = {}
        for dtype, cl in cases:
            src, tgt = _inputs(8, dtype, cl, nan_layer)
            bl = 8 // world
            src = [x[rank * bl:(rank + 1) * bl].cuda() for x in src]
            tgt = [x[rank * bl:(rank + 1) * bl].cuda() for x in tgt]
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                out = _step(pn, src, tgt, True, 77)
                n = pn.poll_nonfinite_warnings(block=True)
            res[(str(dtype), cl)] = ([x.cpu() if isinstance(x, torch.Tensor) else [y.cpu() for y in x] for x in out],
                                     n, buf.getvalue())
        torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _two_processes(pn, tmp_path, backend, cases, nan_layer=None):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, 2, backend, str(tmp_path / "init"), str(tmp_path), cases, nan_layer))
             for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    return [torch.load(str(tmp_path / f"rank{r}.pt"), weights_only=False) for r in range(2)]


def _check_two(pn, res, cases, nan_layer=None):
    for dtype, cl in cases:
        src, tgt = _inputs(8, dtype, cl, nan_layer)
        src, tgt = [x.cuda() for x in src], [x.cuda() for x in tgt]
        loss, grads, loss2, g2, ids = _step(pn, src, tgt, None, 77)
        got = [r[(str(dtype), cl)] for r in res]
        for r in range(2):
            for a, b in zip(got[r][0][4], ids):                        # every rank drew the one-process ids
                assert torch.equal(a, b.cpu())
        lossf = lambda r, k: got[r][0][k].item()
        tol_l, tol_g = (1e-5, 1e-5) if dtype == torch.float32 else (1e-5, 1e-2)
        for k in (0, 2):                                               # autograd, loss_and_grads
            assert (lossf(0, k) + lossf(1, k)) / 2 == pytest.approx(loss.item(), rel=tol_l, abs=1e-7)
            for r in range(2):
                for a, e in zip(got[r][0][1 if k == 0 else 3], grads):
                    e = e[r * 4:(r + 1) * 4].cpu().double()
                    a = a.double() / 2
                    assert torch.equal(torch.isnan(a), torch.isnan(e))
                    fin = torch.isfinite(e)
                    assert (a[fin] - e[fin]).abs().max().item() <= tol_g * max(e[fin].abs().max().item(), 1e-30)
                    if cl:
                        assert got[r][0][1 if k == 0 else 3][0].is_contiguous(memory_format=torch.channels_last)
    return got


CASES = [(torch.float32, False), (torch.float32, True), (torch.bfloat16, False), (torch.bfloat16, True)]


def test_two_processes_on_one_gpu_gloo(pn, tmp_path):
    res = _two_processes(pn, tmp_path, "gloo", CASES)
    _check_two(pn, res, CASES)


def test_global_guard_zeroes_the_layer_on_every_rank(pn, tmp_path):
    cases = [(torch.float32, False)]
    res = _two_processes(pn, tmp_path, "gloo", cases, nan_layer=1)
    got = _check_two(pn, res, cases, nan_layer=1)
    for r in range(2):
        _, n, text = got[r]
        # one guarded layer in each of the two forwards of _step (autograd, loss_and_grads), reported on both ranks
        assert n >= 1 and text.count("Warning: NaN in PatchNCE loss (minibatch negatives)") == 2, (r, n, text)
        g = got[r][0][1][1]
        if r == 0:
            assert (g == 0).all()                                      # rank 0's rows are finite: zero gradient
        else:
            assert torch.isnan(g).any() and (g[~torch.isnan(g)] == 0).all()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_nccl(pn, tmp_path):
    res = _two_processes(pn, tmp_path, "nccl", CASES)
    _check_two(pn, res, CASES)
