"""The netF head with global negatives (patchnce_with_head_global_negatives, head_global_negatives_loss_and_grads) on
the B200: a group of one rank is today's head minibatch call; virtual shards in one process through the C ABI (slots
exchanged by device copies) against the one-process head minibatch result and the float64 shard oracle; two processes on
one GPU (gloo) and on two GPUs (NCCL) through the public API; the global guard; the kernels and memory of a rank's step.
Inputs, netF and tolerances are those of test_patchnce_with_head_minibatch_gpu.py."""
import contextlib
import ctypes
import io
import os

import numpy as np
import pytest
import torch

import head_global_negatives_oracle as hgo
from test_patchnce_with_head_minibatch_gpu import B5, CFG4, TOL, _check, _head_params, _maps, _netf

pytestmark = pytest.mark.gpu

# shards vs one process: the same per-row arithmetic (an item walks the same key blocks in the same order); the row
# losses and the head gradients' split-K slabs are summed per rank
REORDER = 1e-5
WARNING = "Warning: NaN in PatchNCE loss (minibatch negatives)"


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
    test."""
    yield
    import gc
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _worst(a, e):
    """max |a - e| / max |e| over the finite entries (NaN patterns must agree)."""
    a, e = a.double(), e.double()
    assert torch.equal(torch.isnan(a), torch.isnan(e))
    fin = torch.isfinite(e)
    if not fin.any():
        return 0.0
    return (a[fin] - e[fin]).abs().max().item() / max(e[fin].abs().max().item(), 1e-30)


def _one_process(pn, netF, src, tgt, ids, math="tc_bf16x3"):
    """patchnce_with_head_minibatch on the global batch: (loss, d tgt, head grads per layer, guarded layers)."""
    netF.zero_grad(set_to_none=True)
    t = [x.detach().clone().requires_grad_() for x in tgt]
    loss, _ = pn.patchnce_with_head_minibatch(netF, src, t, 0.07, max(i.numel() for i in ids), ids, math)
    loss.backward()
    n = pn.poll_nonfinite_warnings(block=True)
    z = lambda p: torch.zeros_like(p) if p.grad is None else p.grad.clone()
    return loss.item(), [x.grad for x in t], [[z(p) for p in ps] for ps in _head_params(netF, len(src))], n


def _layer_array(src, tgt, ids, dtgt):
    from gan_variant_research_b200 import _lib
    arr = (_lib.PnceLayer * len(tgt))()
    for l, (s, t, i, d) in enumerate(zip(src, tgt, ids, dtgt)):
        arr[l].src, arr[l].tgt, arr[l].ids, arr[l].dtgt = s.data_ptr(), t.data_ptr(), i.data_ptr(), d.data_ptr()
        arr[l].C, arr[l].H, arr[l].W, arr[l].P = t.shape[1], t.shape[2], t.shape[3], i.numel()
    return arr


def _virtual_shards(netF, src, tgt, ids, math, world, tau=0.07):
    """W ranks in one process through the C ABI: pnce_head_mb_shard_keys on every rank, the slot exchange as device
    copies between the W workspaces, then pnce_head_mb_shard_loss and pnce_head_bwd_ex on every rank.
    -> ([loss_r], [[d tgt_l of rank r]], [[[dW1, db1, dW2, db2] of layer l] of rank r], [guarded layers of rank r])."""
    from gan_variant_research_b200 import _lib
    lib = _lib.load()
    n, b, nc = len(tgt), tgt[0].shape[0], netF.nc
    bl = b // world
    dcode = {torch.float32: _lib.PNCE_F32, torch.float16: _lib.PNCE_F16, torch.bfloat16: _lib.PNCE_BF16}[tgt[0].dtype]
    mcode = {"tc_bf16x3": _lib.MATH_TC_BF16X3, "tc_bf16": _lib.MATH_TC_BF16}[math]
    params = [p.detach().float().contiguous() for ps in _head_params(netF, n) for p in ps]
    sizes = [p.numel() for p in params]
    shard = lambda xs, r: [x[r * bl:(r + 1) * bl] for x in xs]
    grads = [[torch.empty_like(t) for t in shard(tgt, r)] for r in range(world)]
    flats = [torch.empty(sum(sizes), device="cuda") for _ in range(world)]
    arrs = [_layer_array(shard(src, r), shard(tgt, r), ids, grads[r]) for r in range(world)]
    heads = []
    for r in range(world):
        h = (_lib.PnceHead * n)()
        ptr = flats[r].data_ptr()
        for l in range(n):
            h[l].w1, h[l].b1, h[l].w2, h[l].b2 = (params[4 * l + k].data_ptr() for k in range(4))
            dp_ = []
            for k in range(4):
                dp_.append(ptr)
                ptr += 4 * sizes[4 * l + k]
            h[l].dw1, h[l].db1, h[l].dw2, h[l].db2 = dp_
        heads.append(h)
    nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    _lib.check(lib.pnce_head_mb_shard_workspace_bytes(arrs[0], n, bl, world, nc, ctypes.byref(nb), ctypes.byref(off),
                                                      ctypes.byref(sb)), "ws")
    st = torch.cuda.current_stream().cuda_stream
    ws = [torch.empty(nb.value, dtype=torch.uint8, device="cuda") for _ in range(world)]
    flags = [torch.zeros(2, dtype=torch.int32, device="cuda") for _ in range(world)]
    for r in range(world):
        _lib.check(lib.pnce_head_mb_shard_keys(arrs[r], heads[r], n, bl, dcode, _lib.LAYOUT_NCHW, nc, world, r, mcode,
                                               ws[r].data_ptr(), nb.value, flags[r].data_ptr(), st), "keys")
    slot = lambda w: slice(off.value + w * sb.value, off.value + (w + 1) * sb.value)
    for r in range(world):
        for w in range(world):
            if w != r:
                ws[r][slot(w)].copy_(ws[w][slot(w)])
    outs = [torch.empty(1 + n, device="cuda") for _ in range(world)]
    one = torch.ones((), device="cuda")
    for r in range(world):
        _lib.check(lib.pnce_head_mb_shard_loss(arrs[r], heads[r], n, bl, dcode, _lib.LAYOUT_NCHW, nc, world, r, tau, mcode,
                                               ws[r].data_ptr(), nb.value, outs[r].data_ptr(), flags[r].data_ptr(), st),
                   "loss")
        _lib.check(lib.pnce_head_bwd_ex(arrs[r], heads[r], n, bl, dcode, _lib.LAYOUT_NCHW, 3, nc, mcode, ws[r].data_ptr(),
                                        nb.value, one.data_ptr(), st), "bwd")
    torch.cuda.synchronize()
    assert all(int(f[1].item()) == 0 for f in flags)             # no tensor-core protocol timeout
    hgrads = [[list(torch.split_with_sizes(flats[r], sizes)[4 * l:4 * l + 4]) for l in range(n)] for r in range(world)]
    hgrads = [[[g.view(p.shape) for g, p in zip(hl, params[4 * l:4 * l + 4])] for l, hl in enumerate(hr)] for hr in hgrads]
    return [o[0].item() for o in outs], grads, hgrads, [int(f[0].item()) for f in flags]


def _shard_oracle(netF, src, tgt, ids, world, rank, dev):
    """float64 shard oracle on ``dev``: (loss, d tgt of the rank's images, head grads per layer)."""
    n = len(src)
    bl = tgt[0].shape[0] // world
    heads = [tuple(p.detach().to(dev, torch.float64).clone().requires_grad_() for p in ps) for ps in _head_params(netF, n)]
    t = [x.detach().to(dev, torch.float64).requires_grad_() for x in tgt]
    loss = hgo.head_global_negatives_loss([x.to(dev, torch.float64) for x in src], t, [i.to(dev) for i in ids], heads,
                                          world, rank)
    if loss.requires_grad:
        loss.backward()
    z = lambda x: torch.zeros_like(x) if x.grad is None else x.grad
    return loss.item(), [z(x)[rank * bl:(rank + 1) * bl] for x in t], [[z(w) for w in h] for h in heads]


def _compare(pn, netF, src, tgt, ids, math, world, what, oracle_ranks):
    losses, dt, dh, nf = _virtual_shards(netF, src, tgt, ids, math, world)
    rl, rt, rh, rn = _one_process(pn, netF, src, tgt, ids, math)
    assert rn == 0 and nf == [0] * world
    bl = tgt[0].shape[0] // world
    assert float(np.mean(losses)) == pytest.approx(rl, rel=REORDER, abs=1e-7), what
    worst_t = max(_worst(dt[r][l] / world, rt[l][r * bl:(r + 1) * bl]) for l in range(len(tgt)) for r in range(world))
    worst_h = max(_worst(sum(dh[r][l][k] for r in range(world)) / world, rh[l][k])
                  for l in range(len(tgt)) for k in range(4))
    exact = all(torch.equal(dt[r][l] / world, rt[l][r * bl:(r + 1) * bl]) for l in range(len(tgt)) for r in range(world))
    print(f"{what}: mean shard loss {np.mean(losses):.7f} vs one process {rl:.7f}; max |shard / W - one process| / max: "
          f"d tgt {worst_t:.2e} (bit-identical: {exact}), head gradients {worst_h:.2e}")
    assert worst_t <= REORDER and worst_h <= REORDER, what
    for r in oracle_ranks:
        want = _shard_oracle(netF, src, tgt, ids, world, r, "cuda")
        _check((losses[r], dt[r], dh[r]), want, ids, TOL[math], f"{what} rank {r}")


def test_group_of_one_rank_is_the_head_minibatch_call(pn):
    """negatives_group=True without a process group: the same CUDA kernels and bit-identical loss, d tgt and head
    gradients as patchnce_with_head_minibatch, on both routes."""
    from torch.profiler import ProfilerActivity, profile
    shapes = [(64, 32, 32), (128, 16, 16)]
    src, tgt = _maps(3, 6, shapes)
    netF = _netf(pn, 256, tgt)
    up = torch.tensor(1.25, device="cuda")
    res = []
    for fn in (pn.patchnce_with_head_minibatch, pn.patchnce_with_head_global_negatives):
        for warm in (True, False):
            netF.zero_grad(set_to_none=True)
            t = [x.clone().requires_grad_() for x in tgt]
            torch.manual_seed(7)
            with (contextlib.nullcontext() if warm else profile(activities=[ProfilerActivity.CUDA])) as prof:
                loss, ids = fn(netF, src, t, 0.07, 256)
                loss.backward(up)
                torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
        res.append((loss.detach(), ids, [x.grad for x in t], [q.grad.clone() for q in netF.parameters()], names))
    (la, ia, ga, pa, na), (lb, ib, gb, pb, nb) = res
    assert na == nb and any("k_loss_tc_mb(" in x for x in na), (na, nb)
    assert torch.equal(la, lb)
    for a, b in zip(ia + ga + pa, ib + gb + pb):
        assert torch.equal(a, b)
    free = []
    for fn in (pn.head_minibatch_loss_and_grads, pn.head_global_negatives_loss_and_grads):
        netF.zero_grad(set_to_none=True)
        torch.manual_seed(7)
        loss, grads, ids = fn(netF, src, tgt, 0.07, 256, grad_output=up)
        free.append((loss, ids, grads, [q.grad.clone() for q in netF.parameters()]))
    (la, ia, ga, pa), (lb, ib, gb, pb) = free
    assert torch.equal(la, lb)
    for a, b in zip(ia + ga + pa, ib + gb + pb):
        assert torch.equal(a, b)


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("nc,shapes,p", [
    (256, [(40, 24, 24), (256, 20, 20)], 300),              # P not a multiple of 128: two key blocks per image
    (128, [(64, 40, 40)], 1024),                            # four key blocks per image
], ids=["nc256_p300", "nc128_p1024"])
def test_virtual_shards_on_odd_shapes(pn, nc, shapes, p, world, math):
    batch = 8                                               # W = 8: one image per rank
    src, tgt = _maps(world * 13 + p, batch, shapes)
    g = torch.Generator(device="cuda").manual_seed(p + world)
    ids = [torch.randint(0, h * w, (min(p, h * w),), device="cuda", generator=g) for _, h, w in shapes]
    netF = _netf(pn, nc, tgt)
    _compare(pn, netF, src, tgt, ids, math, world, f"{shapes} P={p} nc={nc} W={world} {math}", range(world))


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("batch", [16, 64])
def test_virtual_shards_b5(pn, batch, world):
    src, tgt = _maps(batch + world, batch, B5)
    g = torch.Generator(device="cuda").manual_seed(batch * world)
    ids = [torch.randint(0, h * w, (256,), device="cuda", generator=g) for _, h, w in B5]
    netF = _netf(pn, 256, tgt)
    _compare(pn, netF, src, tgt, ids, "tc_bf16x3", world, f"B5 B={batch} W={world}", (0, world - 1))


def test_virtual_shards_config4_one_image_per_rank(pn):
    """BASELINE config 4 (B = 8, 512^2, P = 1024) over eight ranks: B_l = 1, still minibatch negatives of 8 images."""
    src, tgt = _maps(4, 8, CFG4)
    g = torch.Generator(device="cuda").manual_seed(77)
    ids = [torch.randint(0, h * w, (1024,), device="cuda", generator=g) for _, h, w in CFG4]
    netF = _netf(pn, 256, tgt)
    _compare(pn, netF, src, tgt, ids, "tc_bf16x3", 8, "config 4 W=8", (0, 7))


def test_kernels_and_memory_of_a_rank_step(pn):
    """A rank's keys, loss and backward (W = 2, global B = 64, B5, nc = 256): k_loss_tc_mb_gn and no ATen GEMM, bmm or
    softmax; peak memory above the inputs, the gradients and the workspaces below one N_l x N fp32 logits buffer."""
    from torch.profiler import ProfilerActivity, profile
    world, batch = 2, 64
    src, tgt = _maps(2, batch, B5)
    g = torch.Generator(device="cuda").manual_seed(2)
    ids = [torch.randint(0, h * w, (256,), device="cuda", generator=g) for _, h, w in B5]
    netF = _netf(pn, 256, tgt)
    _virtual_shards(netF, src, tgt, ids, "tc_bf16x3", world)                  # warm
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _virtual_shards(netF, src, tgt, ids, "tc_bf16x3", world)
    names = [e.key for e in prof.key_averages()]
    assert any("k_loss_tc_mb_gn" in n for n in names), names
    banned = ("gemm", "bmm", "softmax", "cutlass", "cublas", "nvjet", "sm90_xmma", "sm100_xmma")
    assert not [n for n in names if any(b in n.lower() for b in banned) and "k_gemm_tc" not in n], names
    peak = torch.cuda.max_memory_allocated() - base
    from gan_variant_research_b200 import _lib
    bl = batch // world
    nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    arr = _layer_array([s[:bl] for s in src], [t[:bl] for t in tgt], ids, [t[:bl] for t in tgt])
    _lib.check(_lib.load().pnce_head_mb_shard_workspace_bytes(arr, 5, bl, world, 256, ctypes.byref(nb), ctypes.byref(off),
                                                              ctypes.byref(sb)), "ws")
    grads = sum(t.numel() * 4 for t in tgt) + world * sum(q.numel() * 4 for q in netF.parameters())
    n_l, n = bl * 256, batch * 256
    print(f"rank step W={world} B={batch}: peak {peak / 2**20:.0f} MB, workspace {nb.value / 2**20:.1f} MB "
          f"(slots from {off.value / 2**20:.1f} MB, {sb.value / 2**20:.1f} MB each)")
    assert peak - grads - world * nb.value < n_l * n * 4, (peak, grads, nb.value)


# ---- two processes through the public API ----------------------------------------------------------------------------
SHAPES2 = [(64, 32, 32), (128, 16, 16), (32, 24, 24)]
# (map dtype, channels-last, dp_group)
CASES = [(torch.float32, False, True), (torch.float32, True, True), (torch.bfloat16, False, True),
         (torch.bfloat16, True, True), (torch.float32, False, None)]
# (value, side, rank, layer).  The scaled patches stay finite through the head: at 1e18 and 1e30 the row's partial sums
# of squares overflow, at 1e36 and 1e37 its product with ordinary keys overflows fp32 as well (checked in the test).
GUARDS = [("nan", "tgt", 1, 1), ("nan", "src", 0, 2), (1e18, "tgt", 1, 0), (1e30, "tgt", 1, 0), (1e36, "tgt", 1, 0),
          (1e37, "tgt", 1, 0)]
FLT_MAX = 3.4028234663852886e38


def _inputs(dtype=torch.float32, channels_last=False, guard=None):
    """Global batch of 8 on the current device; ``guard`` = (value, side, rank, layer): one sampled patch of that rank's
    second image set to NaN (value "nan") or scaled by the value."""
    src, tgt = _maps(21, 8, SHAPES2)
    g = torch.Generator(device="cuda").manual_seed(21)
    ids = [torch.randint(0, h * w, (128,), device="cuda", generator=g) for _, h, w in SHAPES2]
    if guard is not None:
        value, side, rank, layer = guard
        maps = tgt if side == "tgt" else src
        pos = ids[layer][3].item()
        x = maps[layer][rank * 4 + 1].view(maps[layer].shape[1], -1)
        if value == "nan":
            x[2, pos] = float("nan")
        else:
            x[:, pos] *= value                                # every channel of a finite patch
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    cast = lambda xs: [x.to(dtype).contiguous(memory_format=fmt) for x in xs]
    return cast(src), cast(tgt), ids


def _step(pn, netF, src, tgt, ids, global_negatives, dp_group):
    """Both routes: (loss, d tgt, head grads) through autograd, the same through the autograd-free route, the ids the
    calls used, the guarded-layer count of the two forwards and the warnings printed.  ``ids`` None: the calls draw them
    from the seeded generator.  global_negatives=False: the one-process head minibatch."""
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        netF.zero_grad(set_to_none=True)
        t = [x.clone().requires_grad_() for x in tgt]
        torch.manual_seed(77)
        if global_negatives:
            loss, rid = pn.patchnce_with_head_global_negatives(netF, src, t, 0.07, 128, ids, negatives_group=True,
                                                               dp_group=dp_group)
        else:
            loss, rid = pn.patchnce_with_head_minibatch(netF, src, t, 0.07, 128, ids)
        loss.backward()
        z = lambda p: torch.zeros_like(p) if p.grad is None else p.grad.clone()
        auto = (loss.detach(), [x.grad for x in t], [z(q) for q in netF.parameters()])
        n = pn.poll_nonfinite_warnings(block=True)
        netF.zero_grad(set_to_none=True)
        torch.manual_seed(77)
        if global_negatives:
            lf, gf, _ = pn.head_global_negatives_loss_and_grads(netF, src, tgt, 0.07, 128, ids, negatives_group=True,
                                                                dp_group=dp_group)
        else:
            lf, gf, _ = pn.head_minibatch_loss_and_grads(netF, src, tgt, 0.07, 128, ids)
        free = (lf, gf, [z(q) for q in netF.parameters()])
        n += pn.poll_nonfinite_warnings(block=True)
    cpu = lambda r: (r[0].cpu(), [x.cpu() for x in r[1]], [x.cpu() for x in r[2]])
    return cpu(auto), cpu(free), [i.cpu() for i in rid], n, buf.getvalue()


def _worker(rank, world, backend, init_file, out_dir, job):
    import torch.distributed as dist
    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import patchnce
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        if job == "api":
            # a process that has seen many head shapes: the first call below evicts the workspace-size cache
            for i in range(len(patchnce._HEAD_WS_BYTES), 257):
                patchnce._HEAD_WS_BYTES[("another shape", i)] = 0
        res = {}
        for case in (CASES if job == "api" else GUARDS):
            dtype, cl, dp_group = case if job == "api" else (torch.float32, False, None)
            src, tgt, ids = _inputs(dtype, cl, None if job == "api" else case)
            netF = _netf(pn, 128, [x.float() for x in tgt])
            sl = slice(rank * 4, rank * 4 + 4)
            res[str(case)] = _step(pn, netF, [x[sl] for x in src], [x[sl] for x in tgt], None if job == "api" else ids,
                                   True, dp_group)
        torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _two_processes(tmp_path, backend, job):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, 2, backend, str(tmp_path / "init"), str(tmp_path), job))
             for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=900)
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    return [torch.load(str(tmp_path / f"rank{r}.pt"), weights_only=False) for r in range(2)]


def _check_api(pn, res):
    for case in CASES:
        dtype, cl, dp_group = case
        src, tgt, ids = _inputs(dtype, cl)
        netF = _netf(pn, 128, [x.float() for x in tgt])
        (rl, rt, rh), _, rid, rn, _ = _step(pn, netF, src, tgt, None, False, None)
        got = [r[str(case)] for r in res]
        tol_g = REORDER if dtype == torch.float32 else 1e-2               # d tgt stored in bf16
        for r in range(2):
            auto, free, gid, n, _ = got[r]
            assert n == 0 and rn == 0
            assert all(torch.equal(a, b) for a, b in zip(gid, rid))       # every rank drew the one-process ids
            assert not all(torch.equal(a, b.cpu()) for a, b in zip(gid, ids))   # drawn, not the fixture's
            # the autograd-free route is the autograd route, bit for bit
            assert torch.equal(auto[0], free[0])
            assert all(torch.equal(a, b) for a, b in zip(auto[1] + auto[2], free[1] + free[2]))
            for l, (a, e) in enumerate(zip(auto[1], rt)):
                assert _worst(a / 2, e[r * 4:(r + 1) * 4]) <= tol_g, (case, r, l)
                if cl:
                    assert a.is_contiguous(memory_format=torch.channels_last)
        assert (got[0][0][0].item() + got[1][0][0].item()) / 2 == pytest.approx(rl, rel=REORDER, abs=1e-7), case
        if dp_group:                                                      # averaged over the ranks already
            for k, e in enumerate(rh):
                assert torch.equal(got[0][0][2][k], got[1][0][2][k])
                assert _worst(got[0][0][2][k], e) <= REORDER, (case, k)
        else:                                                             # the caller averages
            for k, e in enumerate(rh):
                assert _worst((got[0][0][2][k] + got[1][0][2][k]) / 2, e) <= REORDER, (case, k)


def test_two_processes_on_one_gpu_gloo(pn, tmp_path):
    _check_api(pn, _two_processes(tmp_path, "gloo", "api"))


def _scaled_row_regime(netF, src, tgt, ids, case):
    """fp32 head output of the scaled query row: (all finite, largest sum of squares of a 32-channel chunk, max over the
    layer's keys of |y . k|)."""
    _, _, rank, layer = case
    seq = getattr(netF, f"mlp_{layer}")
    with torch.no_grad():
        row = tgt[layer][rank * 4 + 1].reshape(tgt[layer].shape[1], -1)[:, ids[layer][3]]
        y = seq(row[None].float())[0].double()
        keys = seq(src[layer].reshape(8, src[layer].shape[1], -1)[:, :, ids[layer]].transpose(1, 2)
                   .reshape(-1, src[layer].shape[1]).float()).double()
        return bool(torch.isfinite(y).all()), (y.view(-1, 32) ** 2).sum(1).max().item(), (keys @ y).abs().max().item()


def test_global_guard_on_every_rank(pn, tmp_path):
    """A NaN sampled tgt patch on rank 1, a NaN sampled src patch on rank 0, and a finite sampled tgt patch on rank 1
    scaled so that the head's output overflows -- its sums of squares from 1e18 on, and its fp32 products with ordinary
    keys at 1e36 and 1e37: every rank guards exactly the layers the one-GPU call on the global batch guards, with the same
    warning count; a guarded layer's d tgt and head gradients are exactly 0 on every rank, the other layers still match
    one GPU."""
    res = _two_processes(tmp_path, "gloo", "guard")
    n_layers = len(SHAPES2)
    for case in GUARDS:
        src, tgt, ids = _inputs(guard=case)
        netF = _netf(pn, 128, tgt)
        (rl, rt, rh), _, _, rn, rtext = _step(pn, netF, src, tgt, ids, False, None)
        guarded = [all((rh[4 * l + k] == 0).all() for k in range(4)) for l in range(n_layers)]
        print(f"guard case {case}: one GPU guards layers {[l for l in range(n_layers) if guarded[l]]}")
        assert rn == 2 * sum(guarded) and rtext.count(WARNING) == rn       # one per guarded layer and forward
        assert guarded[case[3]], case                                     # the modified layer is guarded on one GPU
        if case[0] != "nan":
            finite, ss, qk = _scaled_row_regime(netF, src, tgt, ids, case)
            print(f"  scaled row: finite {finite}, chunk sum of squares {ss:.2e}, max |y . k| {qk:.2e}")
            if case[0] < 1e37:                                            # 1e37 may reach Inf inside the head
                assert finite and ss > FLT_MAX                            # finite entries, squares beyond FLT_MAX
                assert (qk > FLT_MAX) == (case[0] >= 1e36)                # the q . k overflow window
        got = [r[str(case)] for r in res]
        for r in range(2):
            auto, free, _, n, text = got[r]
            assert n == rn and text.count(WARNING) == rtext.count(WARNING), (case, r, n, text)
            for l in range(n_layers):
                hz = [auto[2][4 * l + k] for k in range(4)]
                if guarded[l]:
                    assert (auto[1][l] == 0).all() and all((x == 0).all() for x in hz), (case, r, l)
                else:
                    assert not all((x == 0).all() for x in hz), (case, r, l)
                    assert _worst(auto[1][l] / 2, rt[l][r * 4:(r + 1) * 4]) <= REORDER, (case, r, l)
        for l in range(n_layers):
            if not guarded[l]:
                for k in range(4):
                    mean = (got[0][0][2][4 * l + k] + got[1][0][2][4 * l + k]) / 2
                    assert _worst(mean, rh[4 * l + k]) <= REORDER, (case, l, k)
        assert (got[0][0][0].item() + got[1][0][0].item()) / 2 == pytest.approx(rl, rel=REORDER, abs=1e-7), case


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_nccl(pn, tmp_path):
    _check_api(pn, _two_processes(tmp_path, "nccl", "api"))
