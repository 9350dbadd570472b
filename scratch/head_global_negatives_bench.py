"""netF head with global negatives (patchnce_with_head_global_negatives): one JSON line.

One GPU: the per-rank step of a VIRTUAL shard -- rank 0 of W holds B_l = 64 / W images and contrasts them with the keys
of all 64 -- for W in {1, 2, 4, 8}, bench.py's B5 maps, P = 256, nc = 256, NCHW fp32, tc_bf16x3 and tc_bf16:
  * ms per step (CUDA events, 5 warm-up, 20 timed): pnce_head_mb_shard_keys + pnce_head_mb_shard_loss +
    pnce_head_bwd_ex (all phases) of rank 0,
  * the kernel split from torch.profiler (a separate pass), the loss kernel's TFLOP/s on
    4 (B_l P) (W B_l P) nc per layer, peak max_memory_allocated, workspace and slot bytes.
The other ranks' slots are filled once before timing.  THE KEY EXCHANGE IS EXCLUDED: no collective runs on one GPU, so
these rows are the local work of a rank.  W = 1 is today's head minibatch step (patchnce_with_head_minibatch) at B = 64.
The GPU name and power limit are read in the same run.  Usage: python scratch/head_global_negatives_bench.py [--out FILE]"""
import argparse
import ctypes
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gan_variant_research_b200 as pn  # noqa: E402
from gan_variant_research_b200 import _lib  # noqa: E402
from global_negatives_bench import gpu_info, kernel_split, layer_array, timed  # noqa: E402

B5 = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]
P = 256
NC = 256
GLOBAL = 64


def head_arrays(netF, n):
    """(head parameter tensors, PnceHead array with the weights and the gradient pointers into one flat buffer, flat)."""
    params = [p.detach() for p in netF.parameters()]
    sizes = [p.numel() for p in params]
    flat = torch.empty(sum(sizes), device="cuda")
    heads = (_lib.PnceHead * n)()
    ptr = flat.data_ptr()
    for l in range(n):
        heads[l].w1, heads[l].b1, heads[l].w2, heads[l].b2 = (params[4 * l + k].data_ptr() for k in range(4))
        d = []
        for k in range(4):
            d.append(ptr)
            ptr += 4 * sizes[4 * l + k]
        heads[l].dw1, heads[l].db1, heads[l].dw2, heads[l].db2 = d
    return params, heads, flat


def virtual_rank(world, math, netF, src, tgt, ids):
    """-> step function of rank 0 of `world` (keys, loss, backward); the other slots are filled once here."""
    lib = _lib.load()
    bl, n = GLOBAL // world, len(B5)
    mcode = {"tc_bf16x3": _lib.MATH_TC_BF16X3, "tc_bf16": _lib.MATH_TC_BF16}[math]
    grads = [torch.empty_like(t[:bl]) for t in tgt]
    arrs = [layer_array([s[r * bl:(r + 1) * bl] for s in src], [t[r * bl:(r + 1) * bl] for t in tgt], ids, grads)
            for r in range(world)]
    params, heads, flat = head_arrays(netF, n)
    nb, off, sb = ctypes.c_size_t(0), ctypes.c_size_t(0), ctypes.c_size_t(0)
    _lib.check(lib.pnce_head_mb_shard_workspace_bytes(arrs[0], n, bl, world, NC, ctypes.byref(nb), ctypes.byref(off),
                                                      ctypes.byref(sb)), "ws")
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(1 + n, device="cuda")
    one = torch.ones((), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    f32, nchw = _lib.PNCE_F32, _lib.LAYOUT_NCHW
    for r in range(1, world):                         # every other rank's keys land in its slot of rank 0's workspace
        _lib.check(lib.pnce_head_mb_shard_keys(arrs[r], heads, n, bl, f32, nchw, NC, world, r, mcode, ws.data_ptr(),
                                               nb.value, None, st), "keys")

    def step():
        _lib.check(lib.pnce_head_mb_shard_keys(arrs[0], heads, n, bl, f32, nchw, NC, world, 0, mcode, ws.data_ptr(),
                                               nb.value, None, st), "keys")
        _lib.check(lib.pnce_head_mb_shard_loss(arrs[0], heads, n, bl, f32, nchw, NC, world, 0, 0.07, mcode, ws.data_ptr(),
                                               nb.value, out.data_ptr(), None, st), "loss")
        _lib.check(lib.pnce_head_bwd_ex(arrs[0], heads, n, bl, f32, nchw, 3, NC, mcode, ws.data_ptr(), nb.value,
                                        one.data_ptr(), st), "bwd")
    step.keep = (grads, params, flat, ws, out, one)
    return step, nb.value, off.value, sb.value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(0)
    src = [torch.randn(GLOBAL, *s, device=dev, generator=g) for s in B5]
    tgt = [torch.randn(GLOBAL, *s, device=dev, generator=g) for s in B5]
    ids = [torch.randint(0, s[1] * s[2], (P,), device=dev, generator=g) for s in B5]
    torch.manual_seed(0)
    netF = pn.PatchSampleF(use_mlp=True, nc=NC)
    netF.create_mlp(tgt)
    rows = []
    for world in (1, 2, 4, 8):
        bl = GLOBAL // world
        for math in ("tc_bf16x3", "tc_bf16"):
            if world == 1:
                t1 = [t.clone().requires_grad_() for t in tgt]

                def step():
                    for t in t1:
                        t.grad = None
                    netF.zero_grad(set_to_none=True)
                    pn.patchnce_with_head_minibatch(netF, src, t1, 0.07, P, ids, math)[0].backward()
                ws = prefix = slot = None
            else:
                step, ws, prefix, slot = virtual_rank(world, math, netF, src, tgt, ids)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            ms = timed(step)
            peak = torch.cuda.max_memory_allocated() - base
            split = kernel_split(step)
            flop = sum(4.0 * bl * P * GLOBAL * P * NC for _ in B5)
            loss_ms = split.get("k_loss_tc_mb_gn" if world > 1 else "k_loss_tc_mb")
            row = {"W": world, "B_local": bl, "B_global": GLOBAL, "math": math, "rank_step_ms": round(ms, 4),
                   "kernels_ms": split, "loss_flop": flop,
                   "loss_tflops": round(flop / (loss_ms * 1e-3) / 1e12, 1) if loss_ms else None,
                   "peak_alloc_above_inputs_bytes": peak, "workspace_bytes": ws, "slot_offset_bytes": prefix,
                   "slot_bytes": slot, "slot_bytes_per_image": slot // bl if slot else None,
                   "exchange": "excluded (one GPU)" if world > 1 else "none"}
            rows.append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
            del step
            torch.cuda.empty_cache()
    res = {"mode": "virtual_shards_one_gpu", "gpu": gpu_info(), "layers": B5, "P": P, "nc": NC, "rows": rows,
           "multi_gpu": "not measured"}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
