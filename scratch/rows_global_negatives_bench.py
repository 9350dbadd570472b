"""Global negatives on the row route (rows_patchnce_global_negatives): one JSON line.

One GPU (default): the per-rank step of a VIRTUAL shard -- rank 0 of W holds B_l = 64 / W images and contrasts its query
rows with the key rows of all 64 -- for W in {1, 2, 4, 8}, B5-shaped rows at P = 256, with D = C_l (PatchSampleF without
the head) and with D = 256 (the shape after the head), tc_bf16x3 and tc_bf16:
  * ms per step (CUDA events, 5 warm-up, 20 timed): pnce_rows_mb_shard_keys + pnce_rows_mb_shard_loss of rank 0,
  * the kernel split from torch.profiler (a separate pass) and peak max_memory_allocated above the inputs.
The other ranks' slots are filled once before timing.  THE KEY EXCHANGE IS EXCLUDED: no collective runs on one GPU, so
these rows are the local work of a rank.  W = 1 is today's PatchNCELoss(nce_includes_all_negatives_from_minibatch=True)
on the rows at B = 64 (pnce_rows_mb_fwd_bwd, forward and backward under autograd).

Under torchrun with >= 2 GPUs (--torchrun): the full public-API step including the all-gather, against per-shard
negatives on the same shard, and one GPU at the global batch (rank 0 alone).
The GPU name and power limit are read in the same run.  Usage: python scratch/rows_global_negatives_bench.py [--out FILE]"""
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

B5_C = [64, 256, 256, 128, 64]
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


def rows_inputs(dims):
    g = torch.Generator(device="cuda").manual_seed(0)
    ks = [torch.nn.functional.normalize(torch.randn(GLOBAL * P, d, device="cuda", generator=g), dim=1) for d in dims]
    qs = [torch.nn.functional.normalize(0.6 * k + 0.8 * torch.randn(k.shape, device="cuda", generator=g), dim=1)
          for k in ks]
    return qs, ks


def virtual_rank(world, math, qs, ks):
    """-> step function of rank 0 of `world` (keys + loss, d q written); the other slots are filled once here."""
    lib = _lib.load()
    bl, n = GLOBAL // world, len(qs)
    mcode = {"tc_bf16x3": _lib.MATH_TC_BF16X3, "tc_bf16": _lib.MATH_TC_BF16}[math]
    dqs = [torch.empty_like(q[:bl * P]) for q in qs]
    arrs = []
    for r in range(world):
        arr = (_lib.PnceRows * n)()
        for l in range(n):
            arr[l].q = qs[l][r * bl * P:(r + 1) * bl * P].data_ptr()
            arr[l].k = ks[l][r * bl * P:(r + 1) * bl * P].data_ptr()
            arr[l].dq = dqs[l].data_ptr()
            arr[l].P, arr[l].D = P, qs[l].shape[1]
        arrs.append(arr)
    nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    _lib.check(lib.pnce_rows_mb_shard_workspace_bytes(arrs[0], n, bl, world, ctypes.byref(nb), ctypes.byref(off),
                                                      ctypes.byref(sb)), "ws")
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(1 + n, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for r in range(1, world):                         # every other rank's keys land in its slot of rank 0's workspace
        _lib.check(lib.pnce_rows_mb_shard_keys(arrs[r], n, bl, world, r, mcode, ws.data_ptr(), nb.value, st), "keys")

    def step():
        _lib.check(lib.pnce_rows_mb_shard_keys(arrs[0], n, bl, world, 0, mcode, ws.data_ptr(), nb.value, st), "keys")
        _lib.check(lib.pnce_rows_mb_shard_loss(arrs[0], n, bl, world, 0, 0.07, mcode, ws.data_ptr(), nb.value,
                                               out.data_ptr(), None, st), "loss")
    return step, nb.value, sb.value


def one_gpu(args):
    rows = []
    for dname, dims in (("D=C_l", B5_C), ("D=256", [256] * len(B5_C))):
        qs, ks = rows_inputs(dims)
        for world in (1, 2, 4, 8):
            bl = GLOBAL // world
            for math in ("tc_bf16x3", "tc_bf16"):
                if world == 1:
                    crit = pn.PatchNCELoss(0.07, P, math=math, nce_includes_all_negatives_from_minibatch=True)
                    q1 = [q.clone().requires_grad_() for q in qs]

                    def step():
                        for q in q1:
                            q.grad = None
                        crit(q1, ks).backward()
                    ws = slot = None
                else:
                    step, ws, slot = virtual_rank(world, math, qs, ks)
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                ms = timed(step)
                peak = torch.cuda.max_memory_allocated() - base
                split = kernel_split(step)
                row = {"rows": dname, "W": world, "B_local": bl, "B_global": GLOBAL, "math": math,
                       "rank_step_ms": round(ms, 4), "kernels_ms": split, "peak_alloc_above_inputs_bytes": peak,
                       "workspace_bytes": ws, "slot_bytes": slot,
                       "exchange": "excluded (one GPU)" if world > 1 else "none",
                       "loss_flop": sum(4.0 * bl * P * GLOBAL * P * d for d in dims)}
                rows.append(row)
                print(json.dumps(row), file=sys.stderr, flush=True)
                del step
                torch.cuda.empty_cache()
        del qs, ks
    return {"mode": "virtual_shards_one_gpu", "gpu": gpu_info(), "D_l": {"D=C_l": B5_C, "D=256": [256] * 5}, "P": P,
            "rows": rows, "multi_gpu": "not measured"}


def multi_gpu(args):
    import torch.distributed as dist
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    bl = GLOBAL // world
    qs, ks = rows_inputs(B5_C)
    rows = []
    for math in ("tc_bf16x3", "tc_bf16"):
        for name, images in (("global_negatives", slice(rank * bl * P, (rank + 1) * bl * P)),
                             ("per_shard_negatives", slice(rank * bl * P, (rank + 1) * bl * P)),
                             ("one_gpu_global_batch", slice(0, GLOBAL * P))):
            if name == "one_gpu_global_batch" and rank != 0:
                dist.barrier()
                continue
            q = [x[images].contiguous().requires_grad_() for x in qs]
            k = [x[images].contiguous() for x in ks]
            if name == "global_negatives":
                fn = lambda: pn.rows_patchnce_global_negatives(q, k, 0.07, P, math=math)
            else:
                crit = pn.PatchNCELoss(0.07, P, math=math, nce_includes_all_negatives_from_minibatch=True)
                fn = lambda: crit(q, k)

            def step():
                for x in q:
                    x.grad = None
                fn().backward()
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
