"""Global negatives on the row route (``rows_patchnce_global_negatives``) on the B200: no group is today's minibatch row
call; virtual shards in one process through the C ABI (slots exchanged by device copies) against the one-process
``PatchNCELoss(mb)(rows)`` and the float64 shard oracle; rows from ``PatchSampleF`` against the maps route and through
the head; the global guard; two processes on one GPU (gloo) and on two GPUs (NCCL) through the public function; the
kernels and memory of a rank's step."""
import contextlib
import ctypes
import io
import os

import numpy as np
import pytest
import torch

import rows_global_negatives_oracle as rgo

pytestmark = pytest.mark.gpu

TOL = {"tc_bf16x3": (2e-5, 2e-4), "tc_bf16": (2e-3, 3e-2)}     # vs the float64 oracle: loss rel, gradient max-abs / max
# shards vs one process: the same per-row arithmetic (an item walks the same key blocks in the same order), only the
# fp32 sums of the row losses are grouped per rank
REORDER = (1e-5, 1e-5)
B5_ROWS = [(256, 64), (256, 256), (256, 256), (256, 128), (256, 64)]
ODD_ROWS = [(200, 40), (72, 100), (129, 7)]


@pytest.fixture(scope="module")
def pn():
    import gan_variant_research_b200 as pn
    return pn


@pytest.fixture(autouse=True)
def _release_device_memory():
    """Hand the caching allocator's blocks back after each test, so that what runs later in the process finds device
    memory."""
    yield
    import gc
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _in_own_process(target, tmp_path):
    """Run ``target(out_path)`` in a spawned process and return what it saved.  The launch lists are recorded there: a
    profiler session leaves CUPTI state behind in its process, and in a long test process a later session can come back
    with no device events at all."""
    import multiprocessing as mp
    out = str(tmp_path / "launches.pt")
    proc = mp.get_context("spawn").Process(target=target, args=(out,))
    proc.start()
    proc.join(timeout=600)
    if proc.is_alive():
        proc.kill()
        proc.join()
    assert proc.exitcode == 0, proc.exitcode
    return torch.load(out)


def _mcode(math):
    from gan_variant_research_b200 import _lib
    return {"tc_bf16x3": _lib.MATH_TC_BF16X3, "tc_bf16": _lib.MATH_TC_BF16}[math]


def _problem(shapes, batch, seed):
    """Global rows (batch * P, D) per layer: unit keys and unit queries correlated with them, fp32 on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    qs, ks = [], []
    for p, d in shapes:
        k = torch.nn.functional.normalize(torch.randn(batch * p, d, device="cuda", generator=g), dim=1)
        q = torch.nn.functional.normalize(0.6 * k + 0.8 * torch.randn(k.shape, device="cuda", generator=g), dim=1)
        qs.append(q)
        ks.append(k)
    return qs, ks


class _Shards:
    """W ranks in one process through the C ABI, each with its rows, d q buffers, workspace and outputs."""

    def __init__(self, qs, ks, batch, world):
        from gan_variant_research_b200 import _lib
        self.lib, self.n, self.world, self.bl = _lib.load(), len(qs), world, batch // world
        self.ps = [q.shape[0] // batch for q in qs]
        sl = lambda x, p, r: x[r * self.bl * p:(r + 1) * self.bl * p]
        self.q = [[sl(q, p, r) for q, p in zip(qs, self.ps)] for r in range(world)]
        self.k = [[sl(k, p, r) for k, p in zip(ks, self.ps)] for r in range(world)]
        self.dq = [[torch.empty_like(q) for q in self.q[r]] for r in range(world)]
        self.rows = []
        for r in range(world):
            arr = (_lib.PnceRows * self.n)()
            for l in range(self.n):
                arr[l].q, arr[l].k, arr[l].dq = self.q[r][l].data_ptr(), self.k[r][l].data_ptr(), self.dq[r][l].data_ptr()
                arr[l].P, arr[l].D = self.ps[l], qs[l].shape[1]
            self.rows.append(arr)
        nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
        _lib.check(self.lib.pnce_rows_mb_shard_workspace_bytes(self.rows[0], self.n, self.bl, world, ctypes.byref(nb),
                                                               ctypes.byref(off), ctypes.byref(sb)), "ws")
        self.nbytes, self.off, self.sb = nb.value, off.value, sb.value
        self.ws = [torch.empty(self.nbytes, dtype=torch.uint8, device="cuda") for _ in range(world)]
        self.out = [torch.empty(1 + self.n, device="cuda") for _ in range(world)]
        self.flags = [torch.zeros(2, dtype=torch.int32, device="cuda") for _ in range(world)]

    def keys(self, r, math):
        from gan_variant_research_b200 import _lib
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(self.lib.pnce_rows_mb_shard_keys(self.rows[r], self.n, self.bl, self.world, r, _mcode(math),
                                                    self.ws[r].data_ptr(), self.nbytes, st), "pnce_rows_mb_shard_keys")

    def exchange(self):
        slot = lambda w: slice(self.off + w * self.sb, self.off + (w + 1) * self.sb)
        for r in range(self.world):
            for w in range(self.world):
                if w != r:
                    self.ws[r][slot(w)].copy_(self.ws[w][slot(w)])

    def loss(self, r, math, tau):
        from gan_variant_research_b200 import _lib
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(self.lib.pnce_rows_mb_shard_loss(self.rows[r], self.n, self.bl, self.world, r, tau, _mcode(math),
                                                    self.ws[r].data_ptr(), self.nbytes, self.out[r].data_ptr(),
                                                    self.flags[r].data_ptr(), st), "pnce_rows_mb_shard_loss")

    def run(self, math, tau=0.07):
        """-> ([loss_r], [[layer losses of r]], [[dq_l of r]], [nonfinite_r])."""
        for r in range(self.world):
            self.keys(r, math)
        self.exchange()
        for r in range(self.world):
            self.loss(r, math, tau)
        torch.cuda.synchronize()
        return ([o[0].item() for o in self.out], [o[1:].tolist() for o in self.out], self.dq,
                [int(f[0].item()) for f in self.flags])


def _one_process(pn, qs, ks, batch, math, tau=0.07):
    q = [x.detach().clone().requires_grad_() for x in qs]
    crit = pn.PatchNCELoss(tau, 256, nce_includes_all_negatives_from_minibatch=True, math=math)
    loss = crit(q, ks, batch_size=batch)
    loss.backward()
    return loss.item(), [x.grad for x in q]


def _worst(a, e):
    """max |a - e| / max |e| over the finite entries of e (NaN patterns must coincide)."""
    a, e = a.double(), e.double()
    assert torch.equal(torch.isnan(a), torch.isnan(e))
    fin = torch.isfinite(e)
    if not fin.any():
        return 0.0
    return (a[fin] - e[fin]).abs().max().item() / max(e[fin].abs().max().item(), 1e-30)


def _compare(pn, qs, ks, batch, math, world, oracle_ranks=None, tau=0.07):
    sh = _Shards(qs, ks, batch, world)
    losses, _, dqs, _ = sh.run(math, tau)
    ref_loss, ref_grads = _one_process(pn, qs, ks, batch, math, tau)
    assert float(np.mean(losses)) == pytest.approx(ref_loss, rel=REORDER[0], abs=1e-7)
    nl = [batch // world * p for p in sh.ps]
    worst = max(_worst(dqs[r][l] / world, ref_grads[l][r * nl[l]:(r + 1) * nl[l]])
                for r in range(world) for l in range(len(qs)))
    assert worst <= REORDER[1], worst
    rl, rg = TOL[math]
    n = len(qs)
    for r in (range(world) if oracle_ranks is None else oracle_ranks):
        ref = [rgo.layer_loss_and_grad_rows_shard(q.cpu().numpy(), k.cpu().numpy(), tau, world, r, n)
               for q, k in zip(qs, ks)]
        assert losses[r] == pytest.approx(sum(l for l, _ in ref) / n, rel=rl, abs=1e-6)
        for g, (_, e) in zip(dqs[r], ref):
            e = torch.from_numpy(e)
            assert (g.cpu().double() - e).abs().max().item() <= rg * max(e.abs().max().item(), 1e-30)
    return losses, ref_loss, worst


def _no_group_calls(pn, profiled=False):
    """PatchNCELoss(mb)(rows) and rows_patchnce_global_negatives with negatives_group None and True (no process group),
    for one tensor and for lists -> {single: [(loss, grads, CUDA launch names or None) per way]}."""
    qs, ks = _problem(ODD_ROWS[:2], 8, 1)
    out = {}
    for single in (True, False):
        a, b = (qs[0], ks[0]) if single else (qs, ks)
        res = []
        for how in ("crit", None, True):
            def leaf():
                return a.detach().clone().requires_grad_() if single else [x.detach().clone().requires_grad_() for x in a]

            def call(q):
                if how == "crit":
                    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True)
                    return crit(q, b, batch_size=8)
                return pn.rows_patchnce_global_negatives(q, b, batch_size=8, negatives_group=how)
            call(leaf()).backward()                                 # warm
            torch.cuda.synchronize()
            q = leaf()
            names = None
            if profiled:
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    loss = call(q)
                    loss.backward()
                    torch.cuda.synchronize()
                names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
            else:
                loss = call(q)
                loss.backward()
            grads = [q.grad] if single else [x.grad for x in q]
            res.append((loss.detach().cpu(), [g.cpu() for g in grads], names))
        out[single] = res
    return out


def _no_group_launches_worker(out_path):
    import gan_variant_research_b200 as pn
    torch.save({k: [r[2] for r in v] for k, v in _no_group_calls(pn, profiled=True).items()}, out_path)


def test_no_group_is_todays_minibatch_row_call(pn, tmp_path):
    """negatives_group=None and True without a process group: the same launches and bit-identical results as
    PatchNCELoss(mb)(rows), for one tensor and for lists."""
    for single, res in _no_group_calls(pn).items():
        for other in res[1:]:
            assert torch.equal(other[0], res[0][0]), (single, other[0].item(), res[0][0].item())
            for x, y in zip(other[1], res[0][1]):
                assert torch.equal(x, y), (single, (x - y).abs().max().item(), y.abs().max().item())
    for single, names in _in_own_process(_no_group_launches_worker, tmp_path).items():
        assert any("k_loss_tc_mb" in n for n in names[0]), (single, names[0])
        for other in names[1:]:
            assert other == names[0], (single, other, names[0])


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_virtual_shards_on_odd_shapes(pn, world, math):
    """P not a multiple of 128 (200, 72, 129) and D not a multiple of 32 (40, 100, 7), eight images."""
    qs, ks = _problem(ODD_ROWS, 8, world)
    _compare(pn, qs, ks, 8, math, world)


@pytest.mark.parametrize("math", ["tc_bf16x3", "tc_bf16"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_virtual_shards_b5_at_64(pn, world, math):
    """B5-shaped rows at P = 256 with D = C_l, a global batch of 64 (16384 keys per layer); the float64 oracle on the
    first and last rank at W = 8 (its N_l x N logits are 0.27 GB per layer there)."""
    qs, ks = _problem(B5_ROWS, 64, 10 + world)
    losses, ref, worst = _compare(pn, qs, ks, 64, math, world, oracle_ranks=[0, 7] if world == 8 else [])
    print(f"B5 B=64 W={world} {math}: mean shard loss {np.mean(losses):.7f} vs one process {ref:.7f}, "
          f"dq max |shard / W - one process| / max = {worst:.2e}")


def test_rows_of_patch_sample_f_match_the_maps_route(pn):
    """PatchSampleF(use_mlp=False) rows of sharded maps through the row route: the same losses as the maps route's
    shards (pnce_mb_shard_*) and, through the sampler's backward, the same d tgt."""
    import test_global_negatives_gpu as gng
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(3)
    shapes = [(64, 32, 32), (128, 16, 16), (40, 12, 12)]
    batch, world = 8, 4
    src = [torch.randn(batch, *s, device=dev, generator=g) for s in shapes]
    tgt = [0.5 * a + torch.randn(a.shape, device=dev, generator=g) for a in src]
    ids = [torch.randint(0, s[1] * s[2], (min(256, s[1] * s[2]),), device=dev, generator=g) for s in shapes]
    m_losses, m_grads, _ = gng._virtual_shards(src, tgt, ids, 0.07, "tc_bf16x3", world)
    sampler = pn.PatchSampleF(use_mlp=False)
    t = [x.detach().clone().requires_grad_() for x in tgt]
    feat_q, _ = sampler(t, 256, ids)
    with torch.no_grad():
        feat_k, _ = sampler(src, 256, ids)
    sh = _Shards([q.detach().contiguous() for q in feat_q], feat_k, batch, world)
    losses, _, dqs, _ = sh.run("tc_bf16x3")
    bl = batch // world
    for r in range(world):
        assert losses[r] == pytest.approx(m_losses[r], rel=2e-5)
    # d tgt of every rank's shard through the sampler's backward (rows of image b depend on tgt[b] only)
    torch.autograd.backward(feat_q, [torch.cat([dqs[r][l] for r in range(world)]) for l in range(len(shapes))])
    for l in range(len(shapes)):
        for r in range(world):
            assert _worst(t[l].grad[r * bl:(r + 1) * bl], m_grads[r][l]) <= 2e-4


@pytest.mark.parametrize("nc", [128, 256])
def test_rows_of_the_mlp_head_match_autograd_through_the_head(pn, nc):
    """PatchSampleF(use_mlp=True) on each rank's maps, the rank's d q pushed back through the head: the mean of the
    shard losses and of the shard head gradients is one process's PatchNCELoss(mb) on the global rows under autograd."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(nc)
    shapes = [(64, 32, 32), (128, 16, 16)]
    batch, world = 8, 2
    src = [torch.randn(batch, *s, device=dev, generator=g) for s in shapes]
    tgt = [0.5 * a + torch.randn(a.shape, device=dev, generator=g) for a in src]
    ids = [torch.randint(0, s[1] * s[2], (256,), device=dev, generator=g) for s in shapes]
    torch.manual_seed(nc)
    netF = pn.PatchSampleF(use_mlp=True, nc=nc)
    netF(tgt, 256, ids)                                             # builds the head
    params = list(netF.parameters())
    # one process on the global batch
    netF.zero_grad()
    with torch.no_grad():
        k_all, _ = netF(src, 256, ids)
    q_all, _ = netF(tgt, 256, ids)
    crit = pn.PatchNCELoss(0.07, 256, nce_includes_all_negatives_from_minibatch=True)
    ref = crit(q_all, k_all, batch_size=batch)
    ref.backward()
    ref_grads = [p.grad.clone() for p in params]
    # the ranks: netF on the rank's maps, the shard entry points, d q back through the head
    bl = batch // world
    netF.zero_grad()
    q_r, k_r = [], []
    for r in range(world):
        with torch.no_grad():
            k, _ = netF([s[r * bl:(r + 1) * bl] for s in src], 256, ids)
        q, _ = netF([t[r * bl:(r + 1) * bl] for t in tgt], 256, ids)
        q_r.append(q)
        k_r.append(k)
    sh = _Shards([torch.cat([q_r[r][l].detach() for r in range(world)]) for l in range(len(shapes))],
                 [torch.cat([k_r[r][l] for r in range(world)]) for l in range(len(shapes))], batch, world)
    losses, _, dqs, _ = sh.run("tc_bf16x3")
    for r in range(world):
        torch.autograd.backward(q_r[r], [d / world for d in dqs[r]])       # the rank-mean of the head gradients
    assert float(np.mean(losses)) == pytest.approx(ref.item(), rel=2e-5)
    for p, e in zip(params, ref_grads):
        assert _worst(p.grad, e) <= 1e-4


def test_guard_of_virtual_shards(pn):
    """A NaN / Inf query row on rank 1 and a NaN key on rank 2 zero their layers on every rank, as one GPU does; a finite
    query row scaled by 100 -- far from unit norm, outside the row route's inputs -- is the documented window where the
    owning rank guards alone (DESIGN.md 4.15)."""
    world, batch = 4, 8
    qs, ks = _problem(ODD_ROWS, batch, 5)
    nl = [batch // world * p for p, _ in ODD_ROWS]
    qs[0][1 * nl[0] + 3, 5] = float("nan")                          # layer 0: a query row of rank 1
    qs[1][1 * nl[1] + 7, 0] = float("inf")                          # layer 1: a query row of rank 1
    ks[2][2 * nl[2] + 1, 2] = float("nan")                          # layer 2: a key of rank 2
    sh = _Shards(qs, ks, batch, world)
    losses, layer_losses, dqs, bad = sh.run("tc_bf16x3")
    ref_loss, ref_grads = _one_process(pn, qs, ks, batch, "tc_bf16x3")
    assert ref_loss == 0.0 and losses == [0.0] * world and bad == [3] * world
    assert all((d == 0).all() for r in range(world) for d in dqs[r])
    assert all((g == 0).all() for g in ref_grads)
    # the window: finite but far from unit norm
    qs, ks = _problem(ODD_ROWS[:1], batch, 6)
    qs[0][nl[0] + 2] *= 100.0
    sh = _Shards(qs, ks, batch, world)
    losses, _, _, bad = sh.run("tc_bf16x3")
    ref_loss, _ = _one_process(pn, qs, ks, batch, "tc_bf16x3")
    assert ref_loss == 0.0 and bad[1] == 1 and losses[1] == 0.0
    assert bad[0] == bad[2] == bad[3] == 0 and all(np.isfinite(losses[r]) and losses[r] > 0 for r in (0, 2, 3))


def _rank_step_launches_worker(out_path):
    from torch.profiler import ProfilerActivity, profile
    qs, ks = _problem(B5_ROWS, 64, 2)
    sh = _Shards(qs, ks, 64, 4)
    sh.run("tc_bf16x3")                                             # warm; every slot filled
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sh.keys(0, "tc_bf16x3")
        sh.loss(0, "tc_bf16x3", 0.07)
        torch.cuda.synchronize()
    torch.save([e.name for e in prof.events() if e.device_type.name == "CUDA"], out_path)


def test_kernels_and_memory_of_a_rank_step(pn, tmp_path):
    """A rank's shard step (keys + loss) launches k_rows_pack, k_mb_qbad and k_loss_tc_mb_gn besides memsets, and
    allocates nothing above its inputs, outputs and workspace."""
    names = _in_own_process(_rank_step_launches_worker, tmp_path)
    kernels = [n.split("(")[0].split("::")[-1] for n in names if "memset" not in n.lower()]
    assert kernels == ["k_rows_pack", "k_mb_qbad", "k_loss_tc_mb_gn"], names
    qs, ks = _problem(B5_ROWS, 64, 2)
    sh = _Shards(qs, ks, 64, 4)
    sh.run("tc_bf16x3")                                             # warm; every slot filled
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    sh.keys(0, "tc_bf16x3")
    sh.loss(0, "tc_bf16x3", 0.07)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() == base


# ---- two processes through the public function --------------------------------------------------------------------
SHAPES2 = [(256, 64), (100, 40), (64, 256)]


def _inputs(job):
    g = torch.Generator().manual_seed(31)
    ks = [torch.nn.functional.normalize(torch.randn(8 * p, d, generator=g), dim=1) for p, d in SHAPES2]
    qs = [torch.nn.functional.normalize(0.6 * k + 0.8 * torch.randn(k.shape, generator=g), dim=1) for k in ks]
    if job == "guard":
        qs[1][4 * 100 + 9, 3] = float("inf")                        # a query row of rank 1 (images 4..7), layer 1
        ks[2][2 * 64 + 5, 0] = float("nan")                         # a key of rank 0, layer 2
    return qs, ks


def _worker(rank, world, backend, init_file, out_dir, job):
    import torch.distributed as dist
    import gan_variant_research_b200 as pn
    torch.cuda.set_device(rank if backend == "nccl" else 0)
    dist.init_process_group(backend, init_method=f"file://{init_file}", rank=rank, world_size=world)
    try:
        qs, ks = _inputs(job)
        bl = 8 // world
        q = [x[rank * bl * p:(rank + 1) * bl * p].cuda().requires_grad_() for x, (p, _) in zip(qs, SHAPES2)]
        k = [x[rank * bl * p:(rank + 1) * bl * p].cuda() for x, (p, _) in zip(ks, SHAPES2)]
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            loss = pn.rows_patchnce_global_negatives(q, k, batch_size=bl)
            loss.backward()
            q0 = q[0].detach().clone().requires_grad_()
            loss0 = pn.rows_patchnce_global_negatives(q0, k[0])       # one tensor, the batch inferred (P = 256)
            loss0.backward()
            n = pn.poll_nonfinite_warnings(block=True)
        torch.save({"loss": loss.item(), "grads": [x.grad.cpu() for x in q], "loss0": loss0.item(),
                    "grad0": q0.grad.cpu(), "n": n, "text": buf.getvalue()}, os.path.join(out_dir, f"rank{rank}.pt"))
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
        p.join(timeout=600)
    for p in procs:
        if p.is_alive():
            p.kill()
            p.join()
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    return [torch.load(str(tmp_path / f"rank{r}.pt"), weights_only=False) for r in range(2)]


def _check_api(pn, res, job):
    qs, ks = _inputs(job)
    qs, ks = [x.cuda() for x in qs], [x.cuda() for x in ks]
    ref_loss, ref_grads = _one_process(pn, qs, ks, 8, "tc_bf16x3")
    ref0, ref0_grads = _one_process(pn, qs[:1], ks[:1], 8, "tc_bf16x3")
    assert (res[0]["loss"] + res[1]["loss"]) / 2 == pytest.approx(ref_loss, rel=1e-5, abs=1e-7)
    assert (res[0]["loss0"] + res[1]["loss0"]) / 2 == pytest.approx(ref0, rel=1e-5, abs=1e-7)
    for r in range(2):
        for (p, _), a, e in zip(SHAPES2, res[r]["grads"], ref_grads):
            assert _worst(a / 2, e[r * 4 * p:(r + 1) * 4 * p].cpu()) <= 1e-5
        assert _worst(res[r]["grad0"] / 2, ref0_grads[0][r * 1024:(r + 1) * 1024].cpu()) <= 1e-5
    return ref_grads


def test_two_processes_on_one_gpu_gloo(pn, tmp_path):
    res = _two_processes(tmp_path, "gloo", "api")
    _check_api(pn, res, "api")
    assert all(r["n"] == 0 and r["text"] == "" for r in res)


def test_global_guard_on_every_rank_gloo(pn, tmp_path):
    """An Inf query row on rank 1 (layer 1) and a NaN key on rank 0 (layer 2): both layers are guarded on both ranks,
    their d q rows are zero, and poll_nonfinite_warnings reports the two layers on each rank."""
    res = _two_processes(tmp_path, "gloo", "guard")
    _check_api(pn, res, "guard")
    for r in range(2):
        assert (res[r]["grads"][1] == 0).all() and (res[r]["grads"][2] == 0).all()
        assert res[r]["grads"][0].abs().max() > 0
        assert res[r]["n"] == 2, res[r]
        assert res[r]["text"].count("Warning: NaN in PatchNCE loss (minibatch negatives)") == 2, res[r]["text"]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_nccl(pn, tmp_path):
    _check_api(pn, _two_processes(tmp_path, "nccl", "api"), "api")
