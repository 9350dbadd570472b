"""Minibatch negatives (nce_includes_all_negatives_from_minibatch): one JSON line with, for B in {1, 4, 16, 64}, the B5
maps (bench.py's layers), P = 256, NCHW and channels-last, tc_bf16x3 and tc_bf16:
  * ms per forward + backward step (CUDA events, 5 warm-up steps, 20 timed) and patches/s,
  * the k_loss_tc_mb kernel time from torch.profiler (a separate pass),
  * its FLOPs (4 N^2 C_l per layer, N = B P), achieved and issued (x3 for bf16x3) TFLOP/s, and the share of the
    1408.6 TFLOP/s bf16 figure bench.py uses,
  * the exp2 count (N^2 per layer) and the L2 -> SM operand bytes (B^2 Ppad^2 Cp / 16 per layer in bf16x3: every item
    re-reads its layer's K and K2 blobs, hi + lo; half that in bf16),
  * peak max_memory_allocated,
and the eager torch restatement (upstream's bmm formula, fp32) at the same sizes with its step time and peak memory.
The GPU name and power limit are read in the same run.  Usage: python scratch/minibatch_bench.py [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gan_variant_research_b200 as pn  # noqa: E402

B5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
TENSOR_TFLOPS = 1408.6
P = 256


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


def kernel_ms(fn, name, steps=5):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    tot = sum(e.device_time_total for e in prof.key_averages() if name in e.key)
    return tot / steps / 1000.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="1,4,16,64")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    dev = torch.device("cuda")
    res = {"gpu": gpu_info(), "layers": B5, "P": P, "rows": []}
    for B in [int(x) for x in args.batches.split(",")]:
        n = B * P
        flops = sum(4.0 * n * n * c for c, _, _ in B5)
        exp2 = float(n * n * len(B5))
        for layout in ("nchw", "channels_last"):
            fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
            src = [torch.randn(B, *s, device=dev).contiguous(memory_format=fmt) for s in B5]
            tgt = [torch.randn(B, *s, device=dev).contiguous(memory_format=fmt).requires_grad_() for s in B5]
            for math in ("tc_bf16x3", "tc_bf16"):
                crit = pn.PatchNCELoss(0.07, P, math=math, nce_includes_all_negatives_from_minibatch=True)

                def step():
                    for t in tgt:
                        t.grad = None
                    crit(src, tgt).backward()

                torch.cuda.reset_peak_memory_stats()
                ms = timed(step)
                peak = torch.cuda.max_memory_allocated()
                kname = "k_loss_tc_mb" if B > 1 else "k_loss_tc"
                kms = kernel_ms(step, kname)
                x3 = 3 if math == "tc_bf16x3" else 1
                l2 = sum(B * B * P * P * ((c + 31) // 32 * 32) / 16.0 * (x3 + 1) / 4 for c, _, _ in B5)
                row = {"B": B, "N": n, "layout": layout, "math": math, "step_ms": round(ms, 4),
                       "patches_per_s": round(n * len(B5) / (ms / 1000.0)), "kernel": kname,
                       "kernel_ms": round(kms, 4), "flop": flops, "exp2": exp2, "l2_to_sm_bytes": l2,
                       "peak_alloc_bytes": peak}
                if kms > 0:
                    row["achieved_tflops"] = round(flops / (kms / 1000.0) / 1e12, 2)
                    row["issued_tflops"] = round(x3 * flops / (kms / 1000.0) / 1e12, 2)
                    row["share_of_tensor_figure"] = round(x3 * flops / (kms / 1000.0) / 1e12 / TENSOR_TFLOPS, 4)
                res["rows"].append(row)
                print(json.dumps(row), file=sys.stderr, flush=True)
            del src, tgt
        # eager restatement: upstream's formula (view(1, -1, C), bmm, CE), fp32, NCHW
        src = [torch.randn(B, *s, device=dev) for s in B5]
        tgt = [torch.randn(B, *s, device=dev).requires_grad_() for s in B5]

        def eager():
            tot = 0.0
            for s, t in zip(src, tgt):
                b, c = s.shape[:2]
                i = torch.randint(0, s.shape[2] * s.shape[3], (P,), device=dev)
                k = F.normalize(s.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(1, -1, c), dim=2, eps=1e-6)
                q = F.normalize(t.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(1, -1, c), dim=2, eps=1e-6)
                z = (torch.bmm(q, k.transpose(2, 1)) / 0.07).clamp(-50, 50)[0]
                tot = tot + F.cross_entropy(z, torch.arange(z.shape[0], device=dev))
            for t in tgt:
                t.grad = None
            (tot / len(B5)).backward()

        torch.cuda.reset_peak_memory_stats()
        ms = timed(eager, warm=2, steps=5 if B == 64 else 20)
        row = {"B": B, "N": n, "impl": "eager_torch_fp32", "step_ms": round(ms, 4),
               "patches_per_s": round(n * len(B5) / (ms / 1000.0)), "peak_alloc_bytes": torch.cuda.max_memory_allocated()}
        res["rows"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del src, tgt
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
