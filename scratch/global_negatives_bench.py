"""Global negatives (PatchNCELoss(..., nce_includes_all_negatives_from_minibatch=True, negatives_group=...)): one JSON line.

One GPU (default): the per-rank step of a VIRTUAL shard -- rank 0 of W holds B_l = 64 / W images and contrasts them with
the keys of all 64 -- for W in {1, 2, 4, 8}, bench.py's B5 maps, P = 256, NCHW fp32, tc_bf16x3 and tc_bf16:
  * ms per step (CUDA events, 5 warm-up, 20 timed): pnce_mb_shard_keys + pnce_mb_shard_loss + pnce_bwd_ex of rank 0,
  * the kernel split from torch.profiler (a separate pass) and peak max_memory_allocated.
The other ranks' slots are filled once before timing.  THE KEY EXCHANGE IS EXCLUDED: no collective runs on one GPU, so
these rows are the local work of a rank.  W = 1 is today's minibatch step (PatchNCELoss, pnce_mb_fwd) at B = 64.

Under torchrun with >= 2 GPUs (--torchrun): the full public-API step including the all-gather, against per-shard
negatives (negatives_group=None) on the same shard, and one GPU at the global batch (rank 0 alone).
The GPU name and power limit are read in the same run.  Usage: python scratch/global_negatives_bench.py [--out FILE]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gan_variant_research_b200 as pn  # noqa: E402
from gan_variant_research_b200 import _lib  # noqa: E402

B5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
P = 256
GLOBAL = 64


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def timed(fn, warm=5, steps=20):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def kernel_split(fn, steps=5):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_time_total > 0:
            name = e.key.split("(")[0].replace("void ", "").replace("pnce::", "")
            out[name] = round(out.get(name, 0.0) + e.device_time_total / steps / 1000.0, 4)
    return out


def layer_array(src, tgt, ids, dtgt):
    arr = (_lib.PnceLayer * len(tgt))()
    for l, (s, t, i, g) in enumerate(zip(src, tgt, ids, dtgt)):
        arr[l].src, arr[l].tgt, arr[l].ids, arr[l].dtgt = s.data_ptr(), t.data_ptr(), i.data_ptr(), g.data_ptr()
        arr[l].C, arr[l].H, arr[l].W, arr[l].P = t.shape[1], t.shape[2], t.shape[3], i.numel()
    return arr


def virtual_rank(world, math, src, tgt, ids):
    """-> step function of rank 0 of `world` (keys, loss, backward); the other slots are filled once here."""
    lib = _lib.load()
    bl, n = GLOBAL // world, len(B5)
    mcode = {"tc_bf16x3": _lib.MATH_TC_BF16X3, "tc_bf16": _lib.MATH_TC_BF16}[math]
    grads = [torch.empty_like(t[:bl]) for t in tgt]
    arrs = [layer_array([s[r * bl:(r + 1) * bl] for s in src], [t[r * bl:(r + 1) * bl] for t in tgt], ids, grads)
            for r in range(world)]
    nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    _lib.check(lib.pnce_mb_shard_workspace_bytes(arrs[0], n, bl, world, ctypes.byref(nb), ctypes.byref(off),
                                                 ctypes.byref(sb)), "ws")
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(1 + n, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for r in range(1, world):                         # every other rank's keys land in its slot of rank 0's workspace
        _lib.check(lib.pnce_mb_shard_keys(arrs[r], n, bl, _lib.PNCE_F32, _lib.LAYOUT_NCHW, world, r, mcode, ws.data_ptr(),
                                          nb.value, None, 0, None, st), "keys")

    def step():
        _lib.check(lib.pnce_mb_shard_keys(arrs[0], n, bl, _lib.PNCE_F32, _lib.LAYOUT_NCHW, world, 0, mcode, ws.data_ptr(),
                                          nb.value, None, 0, None, st), "keys")
        _lib.check(lib.pnce_mb_shard_loss(arrs[0], n, bl, _lib.PNCE_F32, _lib.LAYOUT_NCHW, world, 0, 0.07, mcode,
                                          ws.data_ptr(), nb.value, None, 0, out.data_ptr(), None, st), "loss")
        _lib.check(lib.pnce_bwd_ex(arrs[0], n, bl, _lib.PNCE_F32, _lib.LAYOUT_NCHW, mcode, ws.data_ptr(), nb.value, None,
                                   0, None, st), "bwd")
    return step, nb.value, sb.value


def one_gpu(args):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(0)
    src = [torch.randn(GLOBAL, *s, device=dev, generator=g) for s in B5]
    tgt = [torch.randn(GLOBAL, *s, device=dev, generator=g) for s in B5]
    ids = [torch.randint(0, s[1] * s[2], (P,), device=dev, generator=g) for s in B5]
    rows = []
    for world in (1, 2, 4, 8):
        bl = GLOBAL // world
        for math in ("tc_bf16x3", "tc_bf16"):
            if world == 1:
                crit = pn.PatchNCELoss(0.07, P, math=math, nce_includes_all_negatives_from_minibatch=True)
                t1 = [t.clone().requires_grad_() for t in tgt]

                def step():
                    for t in t1:
                        t.grad = None
                    crit(src, t1).backward()
                ws = slot = None
            else:
                step, ws, slot = virtual_rank(world, math, src, tgt, ids)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            ms = timed(step)
            peak = torch.cuda.max_memory_allocated() - base
            split = kernel_split(step)
            row = {"W": world, "B_local": bl, "B_global": GLOBAL, "math": math, "rank_step_ms": round(ms, 4),
                   "kernels_ms": split, "peak_alloc_above_inputs_bytes": peak, "workspace_bytes": ws,
                   "slot_bytes": slot, "exchange": "excluded (one GPU)" if world > 1 else "none",
                   "loss_flop": sum(4.0 * bl * P * GLOBAL * P * c for c, _, _ in B5)}
            rows.append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
            del step
            torch.cuda.empty_cache()
    return {"mode": "virtual_shards_one_gpu", "gpu": gpu_info(), "layers": B5, "P": P, "rows": rows,
            "multi_gpu": "not measured"}


def multi_gpu(args):
    import torch.distributed as dist
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dev = torch.device("cuda")
    bl = GLOBAL // world
    g = torch.Generator(device=dev).manual_seed(0)
    src = [torch.randn(GLOBAL, *s, device=dev, generator=g) for s in B5]
    tgt = [torch.randn(GLOBAL, *s, device=dev, generator=g) for s in B5]
    rows = []
    for math in ("tc_bf16x3", "tc_bf16"):
        for name, group, images in (("global_negatives", True, slice(rank * bl, (rank + 1) * bl)),
                                    ("per_shard_negatives", None, slice(rank * bl, (rank + 1) * bl)),
                                    ("one_gpu_global_batch", None, slice(0, GLOBAL))):
            if name == "one_gpu_global_batch" and rank != 0:
                dist.barrier()
                continue
            crit = pn.PatchNCELoss(0.07, P, math=math, nce_includes_all_negatives_from_minibatch=True,
                                   negatives_group=group)
            s = [x[images].contiguous() for x in src]
            t = [x[images].contiguous().requires_grad_() for x in tgt]

            def step():
                for x in t:
                    x.grad = None
                crit(s, t).backward()
            ms = timed(step)
            rows.append({"impl": name, "math": math, "W": world, "step_ms": round(ms, 4)})
            if name == "one_gpu_global_batch":
                dist.barrier()
    if rank == 0:
        return {"mode": "torchrun", "gpu": gpu_info(), "world": world, "rows": rows}
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--torchrun", action="store_true", help="run under torchrun on >= 2 GPUs (includes the all-gather)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    res = multi_gpu(args) if args.torchrun else one_gpu(args)
    if res is None:
        return
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
