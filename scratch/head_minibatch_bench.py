"""The netF head with minibatch negatives (patchnce_with_head_minibatch): one JSON line with, for the B5 maps
(bench.py's layers) at P = 256 and B in {1, 4, 16, 64}, and BASELINE config 4 (B = 8, 512^2 maps, P = 1024), nc = 256,
NCHW and channels-last, tc_bf16x3 and tc_bf16:
  * ms per forward + backward step (CUDA events, 5 warm-up steps, 20 timed) and patches/s,
  * the loss kernel's time from torch.profiler (a separate pass): k_loss_tc_mb, or the per-image kernel at B = 1,
  * FLOPs: 4 N^2 nc per layer in the loss (N = B P) plus the head GEMMs (forward 2 N (C_l nc + nc^2) per side, backward
    dH, dX and the two weight gradients: 8 N (C_l nc + nc^2) per layer in all), achieved TFLOP/s of the loss kernel,
  * peak max_memory_allocated,
and, at the same sizes, the module-split composition (PatchSampleF(use_mlp=True) on both sides, then
PatchNCELoss(nce_includes_all_negatives_from_minibatch=True)(feat_q, feat_k)) where it runs (P <= 256), and an eager
torch restatement (nn.Linear head, upstream's bmm formula, fp32).  The GPU name and power limit are read in the same run.
Usage: python scratch/head_minibatch_bench.py [--out FILE] [--batches 1,4,16,64]"""
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
CFG4 = [(c, 2 * h, 2 * w) for c, h, w in B5]
NC = 256


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


def kernel_ms(fn, names, steps=5):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    tot = sum(e.device_time_total for e in prof.key_averages() if any(n in e.key for n in names))
    return tot / steps / 1000.0


def flops(B, P, layers):
    n = B * P
    loss = sum(4.0 * n * n * NC for _ in layers)
    # forward: H = X W1^T, Y = H W2^T on both sides; backward (q side): dH = dY W2, dX = dH W1, dW2 = dY^T H, dW1 = dH^T X
    head = sum(2.0 * n * (2 * (c * NC + NC * NC) + 2 * NC * NC + 2 * c * NC) for c, _, _ in layers)
    return loss, head


def netf(feats):
    torch.manual_seed(0)
    m = pn.PatchSampleF(use_mlp=True, nc=NC)
    m.create_mlp(feats)
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="1,4,16,64")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    dev = torch.device("cuda")
    res = {"gpu": gpu_info(), "nc": NC, "rows": []}
    cases = [("b5", B5, B, 256) for B in (int(x) for x in args.batches.split(","))] + [("cfg4_512sq", CFG4, 8, 1024)]
    for name, layers, B, P in cases:
        n = B * P
        fl, fh = flops(B, P, layers)
        for layout in ("nchw", "channels_last"):
            fmt = torch.channels_last if layout == "channels_last" else torch.contiguous_format
            src = [torch.randn(B, *s, device=dev).contiguous(memory_format=fmt) for s in layers]
            tgt = [torch.randn(B, *s, device=dev).contiguous(memory_format=fmt).requires_grad_() for s in layers]
            net = netf(tgt)
            for math in ("tc_bf16x3", "tc_bf16"):
                def step():
                    for t in tgt:
                        t.grad = None
                    net.zero_grad(set_to_none=True)
                    pn.patchnce_with_head_minibatch(net, src, tgt, 0.07, P, math=math)[0].backward()

                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                ms = timed(step)
                peak = torch.cuda.max_memory_allocated()
                knames = ["k_loss_tc_mb("] if B > 1 else ["k_loss_tc(", "k_loss_tc_p("]
                kms = kernel_ms(step, knames)
                row = {"config": name, "B": B, "P": P, "N": n, "layout": layout, "math": math, "impl": "fused_head_mb",
                       "step_ms": round(ms, 4), "patches_per_s": round(n * len(layers) / (ms / 1000.0)),
                       "loss_kernel": knames[0].rstrip("("), "loss_kernel_ms": round(kms, 4), "loss_flop": fl,
                       "head_flop": fh, "peak_alloc_bytes": peak}
                if kms > 0:
                    row["loss_kernel_achieved_tflops"] = round(fl / (kms / 1000.0) / 1e12, 2)
                res["rows"].append(row)
                print(json.dumps(row), file=sys.stderr, flush=True)
            del src, tgt, net
            torch.cuda.empty_cache()
        src = [torch.randn(B, *s, device=dev) for s in layers]
        tgt = [torch.randn(B, *s, device=dev).requires_grad_() for s in layers]
        net = netf(tgt)
        if P <= 256:
            # module-split composition: PatchSampleF on both sides, then the minibatch row loss
            crit = pn.PatchNCELoss(0.07, P, nce_includes_all_negatives_from_minibatch=True)

            def split():
                for t in tgt:
                    t.grad = None
                net.zero_grad(set_to_none=True)
                with torch.no_grad():
                    fk, ids = net(src, P)
                fq, _ = net(tgt, P, ids)
                crit(fq, fk).backward()

            torch.cuda.reset_peak_memory_stats()
            ms = timed(split)
            row = {"config": name, "B": B, "P": P, "N": n, "layout": "nchw", "math": "tc_bf16x3", "impl": "module_split",
                   "step_ms": round(ms, 4), "patches_per_s": round(n * len(layers) / (ms / 1000.0)),
                   "peak_alloc_bytes": torch.cuda.max_memory_allocated()}
            res["rows"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)

        def eager():
            for t in tgt:
                t.grad = None
            net.zero_grad(set_to_none=True)
            tot = 0.0
            for l, (s, t) in enumerate(zip(src, tgt)):
                b, c = s.shape[:2]
                mlp = getattr(net, f"mlp_{l}")
                i = torch.randint(0, s.shape[2] * s.shape[3], (P,), device=dev)
                with torch.no_grad():
                    k = F.normalize(mlp(s.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(-1, c)), dim=1, eps=1e-6)
                q = F.normalize(mlp(t.reshape(b, c, -1)[:, :, i].transpose(1, 2).reshape(-1, c)), dim=1, eps=1e-6)
                z = (torch.bmm(q.view(1, -1, NC), k.view(1, -1, NC).transpose(2, 1)) / 0.07).clamp(-50, 50)[0]
                tot = tot + F.cross_entropy(z, torch.arange(z.shape[0], device=dev))
            (tot / len(layers)).backward()

        torch.cuda.reset_peak_memory_stats()
        ms = timed(eager, warm=2, steps=5 if n >= 8192 else 20)
        row = {"config": name, "B": B, "P": P, "N": n, "layout": "nchw", "impl": "eager_torch_fp32",
               "step_ms": round(ms, 4), "patches_per_s": round(n * len(layers) / (ms / 1000.0)),
               "peak_alloc_bytes": torch.cuda.max_memory_allocated()}
        res["rows"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del src, tgt, net
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
