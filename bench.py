#!/usr/bin/env python
"""bench.py -- PatchNCE fwd+bwd patches/s on B200 (BASELINE.json metric), one process per GPU.

    python bench.py --gpus 1 --steps K --warmup W                      # this implementation
    python bench.py --impl reference --gpus 1 --steps K --warmup W      # CPU port of the reference
    python bench.py ... --dump-outputs DIR                              # + the last timed step's outputs as DIR/*.npy
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A step = id draw + gather + normalise + logits + diagonal CE + full backward to the dense
d tgt_feat of every layer, for one batch of synthetic feature maps (SURVEY.md section 8d); the
generator passes are not part of the metric.  Prints ONE JSON line on rank 0.  Secondary objects on that line, all
measured AFTER the timed region:
  at every N : head_mode (netF head, its gradient all-reduce INSIDE the timed steps when N > 1), strong (global batch
               64 sharded over the N ranks: strong scaling), nccl_selfcheck (N > 1: data-parallel head gradients
               against the full batch on one rank), e2e
  at N = 1   : configs (B = 1, B = 16, fp16 maps: BASELINE configs 1-3 and the AMP regime), module_split, next_rows
               (the optimiser-side and D-side pieces of SURVEY.md 8f), train_step (BASELINE configs 2 / 3: the whole
               train_step order on stand-in networks, with the PatchNCE share), cpu_baseline.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# logical layer id -> (C, H, W, post_relu) at 256x256 (generator_resnet_attn.py:190-235)
LAYER_SETS = {
    "b5": [(64, 256, 256, True), (256, 64, 64, False), (256, 64, 64, False), (128, 128, 128, True),
           (64, 256, 256, True)],                       # nce_layers [0,4,8,12,13]: "5 layers"
    "r4": [(64, 256, 256, True), (256, 64, 64, False), (256, 64, 64, False), (128, 128, 128, True)],
}                                                       # what [0,4,8,12,16] really returns
METRIC = "patchnce_fwd_bwd_patches_per_s"
UNIT = "patches/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU (weak scaling)")
    ap.add_argument("--layers", default="b5", choices=sorted(LAYER_SETS))
    ap.add_argument("--patches", type=int, default=256)
    ap.add_argument("--tau", type=float, default=0.07)
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "fp16", "bf16"])
    ap.add_argument("--math", default=None)
    ap.add_argument("--layout", default="nchw", choices=["nchw", "nhwc"],
                    help="nhwc: the maps are torch.channels_last (an extension of the reference's interface: the gather "
                         "then reads contiguous rows); the default is the reference's contiguous NCHW")
    ap.add_argument("--cpu-batch", type=int, default=4, help="images in the CPU-baseline sample")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pin", action="store_true", help="N > 1: do not give every rank its own slice of the host cores")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--head", action="store_true", help="time the netF-head mode (nc=256) as the workload")
    ap.add_argument("--no-head-line", action="store_true", help="skip the secondary head-mode measurement")
    ap.add_argument("--clock-period", type=float, default=0.02, help="seconds between NVML clock samples (0: no sampling)")
    ap.add_argument("--settle", type=float, default=0.0, help="experiment: seconds to idle after the maps are created, before warm-up")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (loss, ids, gradients; rank 0) as DIR/<name>.npy")
    return ap.parse_args()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes_per_image(layers, p, elem):
    """SURVEY.md section 8d: sum_l [2*P*C_l*s (useful q,k gather bytes) + C_l*H_l*W_l*s (dense d tgt)]."""
    return sum(2 * min(p, h * w) * c * elem + c * h * w * elem for c, h, w, _ in layers)


def dense_kernel_bytes_per_image(layers, p, elem):
    """The backward kernel alone: the dense d tgt it must write + the gradient rows it reads."""
    return sum(c * h * w * elem + min(p, h * w) * c * 4 for c, h, w, _ in layers)


def make_maps(layers, batch, dtype, device, seed):
    g = torch.Generator(device=device).manual_seed(seed)
    src, tgt = [], []
    for c, h, w, relu in layers:
        for lst in (src, tgt):
            x = torch.randn(batch, c, h, w, device=device, generator=g)
            lst.append((x.relu() if relu else x).to(dtype).contiguous())
    return src, tgt


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  Reads NVML in-process (the library
    nvidia-smi is built on): spawning `nvidia-smi -lms` stalls kernel launches for tens of ms per
    poll, which is as long as the whole timed region here."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index, period=0.02):
        self.index, self.period, self.rows = index, period, []
        self.recording = False
        self.first_at = 0.0
        self.stop_flag = threading.Event()
        self.thread = None
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:                                 # noqa: BLE001
            self.err = repr(e)

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].strip().isdigit():
                return int(ids[index])
        return index

    def sample(self):
        try:
            sm = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
            mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            self.rows.append((float(sm), int(mask)))
        except Exception:                                      # noqa: BLE001
            pass

    def _loop(self):
        while not self.stop_flag.is_set():
            if self.recording and time.perf_counter() >= self.first_at:
                self.sample()
            self.stop_flag.wait(self.period)

    def begin(self, head_start=0.04):
        """Start sampling: called when the timed region starts.  An NVML query holds a driver lock that kernel
        launches need, for up to several milliseconds.  With nothing queued ahead of the host -- the first steps
        after the barrier -- that is a GPU bubble of the same length (it showed up as one 3-11 ms step in an
        otherwise flat 0.86 ms series, always the second step: step_us.max / max_at_step), so the first query
        waits until the host has built a lead (it issues a step in about half the time the GPU needs for it);
        bench takes one more sample right after the last launch, while the queue is still draining."""
        self.rows = []
        self.first_at = time.perf_counter() + head_start
        self.recording = True

    def start(self):
        if self.h is None:
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag.set()
        self.thread.join(timeout=1.0)
        sm = sorted(r[0] for r in self.rows)
        reasons = sorted({name for name, bit in self.REASONS for _, m in self.rows if m & bit})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "reasons": reasons,
                "samples": len(sm), "source": "nvml"}


def cpu_port_step(orc, src, tgt, tau, patches):
    """One fwd+bwd of the oracle's op-for-op torch port (same ATen sequence as the reference) -> (loss, ids)."""
    for t in tgt:
        t.grad = None
    loss, ids = orc.patchnce_loss_torch(src, tgt, tau, patches)
    loss.backward()
    return loss, ids


DUMP_BYTES = 64 << 20
DUMP_FLAT = 65536


def dump_outputs(out_dir, loss, tgt, ids, head=None):
    """--dump-outputs: what one step handed its caller, so that two builds can be compared file for file (the inputs
    and ids are seeded: same arguments, same step).  All float32 / float64, at most DUMP_BYTES in all:
      loss.npy                       the loss (float64, shape (1,))
      ids_l{l}.npy                   the patch positions drawn for layer l (float64)
      grad_l{l}.npy                  d loss / d tgt_feats[l] at those positions, (images, C, P) float32: every value the
                                     step can make non-zero; all images, or a fixed seeded sample of them (images_sampled.npy)
                                     when all would pass the budget
      grad_l{l}_flat.npy             a fixed seeded sample of DUMP_FLAT entries of the whole gradient map, which shows a
                                     write outside the sampled positions
      head_{name}.npy                head mode: the gradient of every netF parameter"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": np.array([float(loss.detach().double().item())])}
    if head is not None:
        for name, p in head.named_parameters():
            if p.grad is not None:
                arrays["head_" + name.replace(".", "_")] = p.grad.detach().float().cpu().numpy()
    g = torch.Generator().manual_seed(0)
    for l, (t, i) in enumerate(zip(tgt, ids)):
        arrays[f"ids_l{l}"] = i.detach().double().cpu().numpy()
        flat = torch.randint(0, t.numel(), (min(DUMP_FLAT, t.numel()),), generator=g)
        arrays[f"grad_l{l}_flat"] = t.grad.detach().contiguous().view(-1)[flat.to(t.device)].float().cpu().numpy()
    used = sum(a.nbytes for a in arrays.values())
    per_image = sum(t.shape[1] * i.numel() * 4 for t, i in zip(tgt, ids))
    batch = tgt[0].shape[0]
    n_img = min(batch, (DUMP_BYTES - used - 8 * batch) // per_image)
    if n_img <= 0:
        raise SystemExit(f"--dump-outputs: one image's gradients ({per_image} bytes) do not fit in {DUMP_BYTES} bytes")
    images = torch.arange(batch) if n_img == batch else torch.randperm(batch, generator=g)[:n_img].sort().values
    if n_img < batch:
        arrays["images_sampled"] = images.double().numpy()
    for l, (t, i) in enumerate(zip(tgt, ids)):
        cols = t.grad.detach().flatten(2)[:, :, i.to(t.device)]           # (B, C, P)
        arrays[f"grad_l{l}"] = cols[images.to(t.device)].float().cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_baseline(args, layers, seconds, min_steps=2):
    """The reference's CPU path (oracle port: /root/reference is Python and cannot travel to the
    GPU box) on this box's host cores, on a bounded sample of the workload."""
    from oracle import patchnce_oracle as orc
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    b = args.cpu_batch
    g = torch.Generator().manual_seed(1234)
    src = [torch.randn(b, c, h, w, generator=g) for c, h, w, _ in layers]
    src = [x.relu() if l[3] else x for x, l in zip(src, layers)]
    tgt = [torch.randn(b, c, h, w, generator=g) for c, h, w, _ in layers]
    tgt = [(x.relu() if l[3] else x).requires_grad_() for x, l in zip(tgt, layers)]
    torch.manual_seed(7)
    cpu_port_step(orc, src, tgt, args.tau, args.patches)            # warm-up
    times = []
    t_end = time.perf_counter() + seconds
    while len(times) < min_steps or time.perf_counter() < t_end:
        t0 = time.perf_counter()
        cpu_port_step(orc, src, tgt, args.tau, args.patches)
        times.append(time.perf_counter() - t0)
        if len(times) >= 200:
            break
    times.sort()
    med = times[len(times) // 2]
    n_patches = b * sum(min(args.patches, h * w) for _, h, w, _ in layers)
    return {"value": n_patches / med, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{len(times)} fwd+bwd steps of B={b} images, layer set {args.layers}, P={args.patches}, "
                      f"fp32, torch CPU port of patchnce_cut.py (oracle/patchnce_oracle.py), median {med * 1e3:.1f} ms"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port) as its own arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import patchnce_oracle as orc
    layers = LAYER_SETS[args.layers]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    b = args.cpu_batch
    g = torch.Generator().manual_seed(1234)
    src = [torch.randn(b, c, h, w, generator=g) for c, h, w, _ in layers]
    src = [x.relu() if l[3] else x for x, l in zip(src, layers)]
    tgt = [torch.randn(b, c, h, w, generator=g) for c, h, w, _ in layers]
    tgt = [(x.relu() if l[3] else x).requires_grad_() for x, l in zip(tgt, layers)]
    torch.manual_seed(7)
    for _ in range(max(args.warmup, 1)):
        cpu_port_step(orc, src, tgt, args.tau, args.patches)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loss, ids = cpu_port_step(orc, src, tgt, args.tau, args.patches)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, loss, tgt, ids)
    n_patches = b * sum(min(args.patches, h * w) for _, h, w, _ in layers)
    value = n_patches * args.steps / dt
    sample = (f"each step = B={b} images of the workload (reference backward is O(B^2), full B={args.batch} "
              f"would take minutes per step), all {cores} host threads, fp32; SINGLE HOST PROCESS whatever --gpus says "
              "(the reference has no distributed code, SURVEY.md 0): its value does not grow with N, so a ratio against "
              "it at N > 1 compares N GPUs with one CPU process")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, layers),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "processes": 1,
    }))


def workload_config(args, layers):
    return {
        "workload": f"PatchNCE fwd+bwd, CUT 256x256 feature maps, layer set {args.layers} "
                    f"({len(layers)} maps: " + ", ".join(f"{c}x{h}x{w}" for c, h, w, _ in layers) +
                    f"), P={args.patches}, tau={args.tau}, batch {args.batch} images per GPU "
                    "(BASELINE config 5 per-GPU batch, weak scaling), reference-exact mode (no netF head)",
        "layers": args.layers, "batch_per_gpu": args.batch, "num_patches": args.patches,
        "layout": "nchw (the reference's contiguous maps)" if args.layout == "nchw" else
                  "nhwc (torch.channels_last maps: an extension, not the reference's interface)",
        "l2_policy": "inputs larger than L2 (feature maps >> 126 MB), no explicit flush",
        "parallelism": f"dp{args.gpus} (batch sharded, identical ids, no collective in no-head mode)",
    }


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import gan_variant_research_b200 as pn
    from gan_variant_research_b200 import _lib
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    _lib.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pinned = None
    if world > 1 and not args.no_pin:
        # one slice of the box's host cores per rank (what numactl / taskset do for a multi-process job): the ranks' Python
        # threads otherwise migrate over all cores and the small-batch (host-bound) lines lose up to 1.6x at N = 8
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            mine = cores[local * per:(local + 1) * per] or cores
            os.sched_setaffinity(0, mine)
            pinned = len(mine)
        except (AttributeError, OSError):
            pinned = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    layers = LAYER_SETS[args.layers]
    tdtype = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    elem = 4 if args.dtype == "fp32" else 2
    math = args.math or pn.DEFAULT_MATH
    B = args.batch
    src, tgt = make_maps(layers, B, tdtype, dev, 1234 + rank)
    if args.layout == "nhwc":
        src = [x.contiguous(memory_format=torch.channels_last) for x in src]
        tgt = [x.contiguous(memory_format=torch.channels_last) for x in tgt]
    tgt = [t.requires_grad_() for t in tgt]
    crit = pn.PatchNCELoss(args.tau, args.patches, [0, 4, 8, 12, 13], math=math)
    netF = None
    if args.head:
        torch.manual_seed(11)      # identical head weights on every rank
        netF = pn.PatchSampleF(use_mlp=True, nc=256).to(dev)
        netF.create_mlp(tgt)
    torch.manual_seed(7)           # identical ids on every rank (SURVEY.md 8e)

    # CUDA events around the backward (the dominant kernel's launch) on every EV_STRIDE-th step of the
    # timed region: a timing event between two kernels costs a few microseconds of stream bubble, which
    # on a 0.9 ms step is worth measuring around, not paying 2x per step
    EV_STRIDE = 4
    ev_b0 = {i: torch.cuda.Event(enable_timing=True) for i in range(0, args.steps, EV_STRIDE)}
    ev_b1 = {i: torch.cuda.Event(enable_timing=True) for i in range(0, args.steps, EV_STRIDE)}
    ev_step = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]     # end of every step
    host_us = []
    head_ids = [None]

    def step(i=None):
        for t in tgt:
            t.grad = None
        if netF is None:
            loss = crit(src, tgt)
        else:
            netF.zero_grad(set_to_none=True)
            # dp_group: the head gradients leave backward() already averaged over the ranks -- the only
            # collective of the path (SURVEY.md 8e), started on a side stream under the dense kernel
            loss, head_ids[0] = pn.patchnce_with_head(netF, src, tgt, args.tau, args.patches, math=math,
                                                      dp_group=True if world > 1 else None)
        if i in ev_b0:
            ev_b0[i].record()
        loss.backward()
        if i in ev_b1:
            ev_b1[i].record()
        return loss

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local, period=args.clock_period or 1e9)
    if args.settle > 0:
        torch.cuda.synchronize()
        time.sleep(args.settle)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the cyclic garbage collector stays out of the timed region (what timeit does): a full collection over
    # torch's heap takes 3-15 ms, and it used to land on the second timed step, when nothing is queued ahead
    # of the host yet -- one long step in an otherwise flat series (step_us.max / max_at_step).  Collected and
    # switched off BEFORE the warm-up steps, so that they run in the regime of the timed ones (a collection
    # between the two also walks the whole heap through the CPU caches right before the first timed step).
    gc.collect()
    gc.disable()
    for _ in range(max(args.warmup, 3)):
        loss = step()                       # same object lifetimes as in the timed loop (the allocator's steady state)
    barrier()
    if rank == 0:
        sampler.begin()
    e0.record()
    for i in range(args.steps):
        h0 = time.perf_counter()
        loss = step(i)
        host_us.append((time.perf_counter() - h0) * 1e6)
        ev_step[i].record()
    e1.record()
    if rank == 0 and sampler.h is not None:
        sampler.sample()                    # the GPU is still working through the queued steps
    barrier()
    gc.enable()
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, loss, tgt, crit.last_patch_ids if netF is None else head_ids[0], netF)
    ms = e0.elapsed_time(e1)
    tmax = torch.tensor([ms], device=dev)
    if world > 1:
        torch.distributed.all_reduce(tmax, op=torch.distributed.ReduceOp.MAX)
    ms = float(tmax.item())
    bwd_ms = sorted(ev_b0[i].elapsed_time(ev_b1[i]) for i in ev_b0)
    bwd_med = bwd_ms[len(bwd_ms) // 2]
    patches_per_image = sum(min(args.patches, h * w) for _, h, w, _ in layers)
    value = world * B * patches_per_image * args.steps / (ms * 1e-3)
    peak, peak_src = peaks()

    dense_bytes = dense_kernel_bytes_per_image(layers, args.patches, elem) * B
    dense_name = "k_fill_zero" if args.layout == "nhwc" and not args.head else "k_dense_flat"
    roof = {"bound": "hbm", "kernel": (dense_name + " (dense d tgt_feat: zero fill + sampled values, one write per line)" if dense_name == "k_dense_flat"
                                       else "k_fill_zero + k_scatter_nhwc (dense d tgt_feat: zero fill of every map, then the sampled rows)"),
            "achieved": dense_bytes / (bwd_med * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "peak_source": peak_src, "traffic": ncu_traffic(dense_name, B, elem), "launch_ms": bwd_med}
    roof["note"] = ("write-only stream (zero fill + sampled values): it can exceed the measured peak, which is a "
                    "read+write copy (6457 GB/s); cudaMemset of the same bytes reaches ~7.3 TB/s on this GPU")
    if args.head:
        roof["note"] = "head mode: the backward events also cover the head's backward GEMMs"
    roof["frac"] = roof["achieved"] / peak
    path_bytes = algorithmic_bytes_per_image(layers, args.patches, elem) * B
    roof_path = {"bound": "hbm", "achieved": path_bytes / (ms / args.steps * 1e-3) / 1e9, "peak": peak,
                 "unit": "GB/s", "bytes_per_patch": path_bytes / (B * patches_per_image)}
    roof_path["frac"] = roof_path["achieved"] / peak

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "fp16": "f16", "bf16": "bf16"}[args.dtype],
        "math": math, "data": "synthetic", "config": workload_config(args, layers),
        "roofline": roof, "roofline_path": roof_path, "clocks": clocks,
        "gpu_launches": (10 if args.head else 4) * args.steps, "loss": float(loss.item()),
    }
    if pinned is not None:
        out["host_cores_per_rank"] = pinned
    # where the dense gradients live: compressible device memory (csrc/comp_alloc.cuh) when the device grants it -- said
    # in the line, with the same step on default-pool memory beside it (timed after the headline region, same maps)
    grads_compressed = all(pn.gradient_is_compressed(t.grad) for t in tgt if t.grad is not None)
    out["config"]["grad_memory"] = ("compressible (cuMemCreate CU_MEM_ALLOCATION_COMP_GENERIC via a torch MemPool: B200 L2/HBM "
                                    "compute-data compression; PNCE_GRAD_COMPRESSION=0 turns it off)" if grads_compressed
                                    else "default pool")
    if grads_compressed:
        if dense_name == "k_dense_flat" and ncu_traffic("k_dense_flat_compressible", B, elem) is not None:
            roof["traffic"] = ncu_traffic("k_dense_flat_compressible", B, elem)
        roof["note"] += ("; the gradients are in compressible memory: the zero lines are compressed between L2 and HBM, so "
                         "DRAM traffic (ncu) is BELOW the algorithmic bytes")
        pn.set_gradient_compression(False)
        pms = timed_steps(step, min(args.steps, 50), 3, world, dev)
        pn.set_gradient_compression(True)
        for _ in range(3):
            step()
        out["plain_alloc"] = {"ms_per_step": pms, "value": world * B * patches_per_image / (pms * 1e-3), "unit": UNIT,
                              "roofline_path_frac": path_bytes / (pms * 1e-3) / 1e9 / peak,
                              "note": "the same step with the dense gradients in torch's default pool (no compression)"}
    if rank == 0:
        # distribution of the per-step device time inside the timed region (ms_per_step is its mean): a handful of
        # slow steps means the host stalled (a busy node), a uniform shift means the kernels themselves moved
        marks = [e0] + ev_step
        raw = [marks[i].elapsed_time(marks[i + 1]) * 1e3 for i in range(args.steps)]
        slowest = max(range(args.steps), key=lambda i: raw[i])
        d = sorted(raw)
        h = sorted(host_us)
        n = len(d)
        out["step_us"] = {"p10": round(d[n // 10], 1), "p50": round(d[n // 2], 1), "p90": round(d[(9 * n) // 10], 1),
                          "max": round(d[-1], 1), "max_at_step": slowest, "host_issue_p50": round(h[n // 2], 1), "host_issue_max": round(h[-1], 1)}
        # the same path roofline on the MEDIAN step (the mean above carries the start-up step after the barrier)
        roof_path["frac_p50"] = path_bytes / (d[n // 2] * 1e-6) / 1e9 / peak
    # the per-kernel breakdowns use torch.profiler, which leaves CUPTI attached to the process (+11 % on a host-bound step,
    # measured): every TIMED secondary line below runs first, the breakdowns after them
    breakdowns = [("kernels_us", step)]
    if args.head:
        out["config"]["workload"] = out["config"]["workload"].replace(
            "reference-exact mode (no netF head)", "netF head mode (Linear-ReLU-Linear, nc=256, tcgen05)")
    elif not args.no_head_line:
        # every rank takes part (world > 1: the head-gradient all-reduce is a collective); rank 0 reports
        hm = head_line(args, pn, src, tgt, math, patches_per_image, world, dev)
        st = strong_line(args, pn, src, tgt, math, patches_per_image, world, dev, layers, elem, peak)
        nh = nhwc_line(args, pn, src, tgt, math, patches_per_image, world, dev, layers, elem, peak, breakdowns) if args.layout == "nchw" else None
        if rank == 0 and nh is not None:
            out["nhwc"] = nh
        sc = nccl_selfcheck(args, pn, layers, dev, world, rank, math) if world > 1 else None
        gr = grad_reducer_line(pn, dev, world) if world > 1 else None
        if rank == 0:
            out["head_mode"], out["strong"] = hm, st
            if sc is not None:
                out["nccl_selfcheck"] = sc
            if gr is not None:
                out["grad_reducer"] = gr
    if rank == 0 and world == 1 and not args.head and not args.no_head_line:
        out["module_split"] = module_split_line(args, pn, src, tgt, math, patches_per_image)
        out["configs"] = config_lines(args, pn, layers, dev, math, peak)
    for key, fn in breakdowns:                # on every rank: head mode's backward holds a collective
        k = kernel_breakdown(fn)
        if rank != 0:
            continue
        if key == "kernels_us":
            out["kernels_us"] = k
            if not args.head and "k_gather_tc" in k and "k_loss_tc_p" in k:
                out["roofline_other_kernels"] = other_kernel_rooflines(args, layers, B, elem, k, peak)
        elif isinstance(out.get("nhwc"), dict):
            tgt_d = out["nhwc"] if key == "nhwc" else out["nhwc"].get("head_mode")
            if isinstance(tgt_d, dict):
                tgt_d["kernels_us"] = k
    breakdowns.clear()
    if rank == 0 and world == 1 and not args.head and not args.no_head_line:
        out["next_rows"] = next_rows_line(pn, dev)
        out["train_step"] = train_step_line(pn, dev)

    # ---- e2e: same metric through the public API with HOST buffers ------------------------------
    if not args.no_e2e:
        out["e2e"] = run_e2e(args, pn, crit, layers, tdtype, elem, dev, world, rank)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args, layers, args.cpu_seconds)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        torch.distributed.destroy_process_group()


def kernel_breakdown(step, n=5):
    """Mean duration (us) of every kernel of one step, from the torch profiler over n extra steps AFTER the
    timed region (never inside it): says which launch moved when ms_per_step moves.  The library's kernels are
    chained by programmatic dependent launch (DESIGN.md 4.9): a kernel is resident -- and "running" for the profiler --
    while it still waits for its predecessor, so each of them is counted from the end of the library kernel that
    started before it and ends inside it (a side-stream id prep under the previous dense kernel fits neither way)."""
    try:
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                step()
            torch.cuda.synchronize()
        evs = []
        for e in prof.events():
            if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range.end > e.time_range.start:
                evs.append((e.name, float(e.time_range.start), float(e.time_range.end)))
        evs.sort(key=lambda t: t[1])
        ours = [(nm, a, b) for nm, a, b in evs if "pnce::" in nm or nm.startswith("k_")]
        rows = {}
        for nm, a, b in evs:
            if "pnce::" in nm or nm.startswith("k_"):
                ends = [pb for pn_, pa, pb in ours if pa < a < pb <= b]
                a = max([a] + ends)
            name = nm.split("(")[0].replace("void ", "").replace("pnce::", "").split("<")[0][:40]
            rows[name] = rows.get(name, 0.0) + (b - a) / n
        return dict(sorted(((k, round(v, 1)) for k, v in rows.items()), key=lambda kv: -kv[1])[:8])
    except Exception as e:                                     # noqa: BLE001
        return {"unavailable": repr(e)}


def other_kernel_rooflines(args, layers, B, elem, kernels, hbm_peak):
    """The two kernels beside the dominant one, timed by the profiler pass above (SURVEY.md 8d figures):
    the gather against HBM with its USEFUL bytes (and the DRAM traffic ncu measured: NCHW puts every channel of a
    patch in its own 128-byte line, so the traffic is ~19x the useful bytes -- inherent to the reference's layout),
    the logits/CE kernel against the tensor pipe with its algorithmic flops (4 P^2 C per image-layer: QK^T and
    dZ K; the bf16x3 mode issues three MMAs per product, so 'issued' is 3x 'achieved')."""
    p = args.patches
    useful = B * sum(2 * min(p, h * w) * c * elem for c, h, w, _ in layers)
    flops = B * sum(4 * min(p, h * w) ** 2 * c for c, h, w, _ in layers)
    tg, tl = kernels["k_gather_tc"] * 1e-6, kernels["k_loss_tc_p"] * 1e-6
    tensor_peak = 1408.6
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        tensor_peak = float(json.load(open(path)).get("bf16_tflops_sustained", tensor_peak))
    ach = flops / tl / 1e12
    return [
        {"kernel": "k_gather_tc", "bound": "hbm", "achieved": useful / tg / 1e9, "peak": hbm_peak, "unit": "GB/s",
         "frac": useful / tg / 1e9 / hbm_peak, "traffic": ncu_traffic("k_gather_tc", B, elem),
         "traffic_gbs": (ncu_traffic("k_gather_tc", B, elem) or 0) / tg / 1e9, "launch_ms": tg * 1e3},
        {"kernel": "k_loss_tc_p", "bound": "tensor", "achieved": ach, "issued_bf16x3": 3 * ach, "peak": tensor_peak,
         "unit": "TFLOP/s", "frac": ach / tensor_peak, "traffic": ncu_traffic("k_loss_tc_p", B, elem),
         "launch_ms": tl * 1e3},
    ]


def ncu_traffic(kernel, batch, elem):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    ncu --set full capture (profiles/traffic.json), scaled to this batch; None when never captured."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path) or elem != 4:
        return None
    d = json.load(open(path)).get(kernel)
    if not d:
        return None
    return d["dram_bytes_per_launch"] * batch / d["batch"]


def next_rows_line(pn, dev, n=30):
    """Secondary measurements, after the timed region: the pieces around the path (SURVEY.md 8f rows 3 and 4) on the
    reference generator's parameter shapes (tests/golden/model_param_shapes.json) and on 16 x 3 x 256 x 256 images.
    Device time per call in us (CUDA events around n calls); never fatal for the bench line."""
    try:
        shapes = json.load(open(os.path.join(ROOT, "tests", "golden", "model_param_shapes.json")))["generator"]
        g = torch.Generator(device=dev).manual_seed(3)
        params = [torch.nn.Parameter(torch.randn(*s, device=dev, generator=g) * 0.02) for s in shapes]
        for p in params:
            p.grad = torch.randn(p.shape, device=dev, generator=g) * 1e-4
        net = torch.nn.Module()
        net.params = torch.nn.ParameterList(params)
        opt = torch.optim.Adam(net.parameters(), lr=2e-4, betas=(0.5, 0.999))
        scaler = torch.amp.GradScaler("cuda", init_scale=1.0, growth_interval=10 ** 9)
        scaler.scale(torch.zeros((), device=dev))
        stepper, ema = pn.FusedAdamStep(opt, scaler, 10.0), pn.EMA(net, 0.999)
        aug = pn.DiffAugment(["color", "translation", "cutout"])
        x = (torch.rand(16, 3, 256, 256, device=dev, generator=g) * 2 - 1).requires_grad_()
        up = torch.randn(16, 3, 256, 256, device=dev, generator=g)

        def aug_step():
            x.grad = None
            aug(x).backward(up)

        def timed(fn):
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return round(e0.elapsed_time(e1) / n * 1e3, 1)

        return {"parameters": sum(p.numel() for p in params), "tensors": len(params),
                "amp_adam_step_us": timed(stepper.step), "ema_update_us": timed(ema.update),
                "diffaugment_fwd_bwd_b16_us": timed(aug_step),
                "note": "unscale + clip + Adam + loss-scale update in 3 launches; EMA in 1; DiffAugment colour + translation + "
                        "cutout in 2 + 2 (plus the 7 draws); DESIGN.md 7.2 - 7.5"}
    except Exception as e:  # noqa: BLE001 - a secondary line must not take the bench down
        return {"error": f"{type(e).__name__}: {e}"}


def train_step_line(pn, dev, timed=8):
    """BASELINE configs 2 and 3 (SURVEY.md 8d): the reference's whole train_step order (training/train_cutpp.py:206-331 --
    D step, G step with the adversarial hinge + PatchNCE, AMP optimiser steps, EMA) at 256 x 256 under autocast, batch 1
    with lambda_NCE = 1 and batch 16 with lambda_NCE = 10, built from this package's pieces around STAND-IN networks with
    the reference's shapes (tests/standin_generator.py: ResNet-9, ngf 64; a 70 x 70-PatchGAN-shaped discriminator -- the
    reference's own models are Python under /root/reference and do not travel to the GPU box).  `patchnce_ms` is the
    difference to the same step without the PatchNCE term: what the loss, its second feature pass and its share of the
    generator's backward cost inside the step.  After the timed region; never fatal for the bench line."""
    try:
        import torch.nn as nn
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from standin_generator import StandInGenerator
        layers = [0, 4, 8, 12, 13]

        def make_d():
            mods, ch = [nn.Conv2d(3, 64, 4, 2, 1), nn.LeakyReLU(0.2)], 64
            for s in (2, 2, 1):
                mods += [nn.Conv2d(ch, ch * 2, 4, s, 1), nn.InstanceNorm2d(ch * 2), nn.LeakyReLU(0.2)]
                ch *= 2
            return nn.Sequential(*mods, nn.Conv2d(ch, 1, 4, 1, 1))

        out = {}
        for name, b, lam in (("config2_b1", 1, 1.0), ("config3_b16_fastcut", 16, 10.0)):
            torch.manual_seed(0)
            gen, dis = StandInGenerator(ngf=64, n_blocks=9).to(dev), make_d().to(dev)
            og = torch.optim.Adam(gen.parameters(), lr=2e-4, betas=(0.5, 0.999))
            od = torch.optim.Adam(dis.parameters(), lr=2e-4, betas=(0.5, 0.999))
            scaler = torch.amp.GradScaler("cuda")
            pn.enable_encoder_feature_reuse(gen, layers)
            ema, aug = pn.EMA(gen, 0.999), pn.DiffAugment(["color", "translation", "cutout"])
            sg, sd = pn.FusedAdamStep(og, scaler, 10.0), pn.FusedAdamStep(od, scaler, 10.0)
            photos = torch.rand(b, 3, 256, 256, device=dev) * 2 - 1

            def step(with_nce):
                od.zero_grad()                                                    # D step, train_cutpp.py:229-253
                with torch.autocast("cuda"):
                    fake = gen(photos)
                    d_loss = pn.discriminator_hinge_loss(dis(aug(photos)), dis(aug(fake.detach())))
                scaler.scale(d_loss).backward()
                sd.step()
                og.zero_grad()                                                    # G step, :266-308
                with torch.autocast("cuda"):
                    fake = gen(photos)
                    g_loss = pn.generator_hinge_loss(dis(aug(fake)))
                    if with_nce:
                        g_loss = g_loss + lam * pn.compute_patchnce_loss(gen, photos, fake, nce_layers=layers,
                                                                         temperature=0.07, num_patches=256)
                scaler.scale(g_loss).backward()
                sg.step()
                ema.update()                                                      # :310-312
                return g_loss

            ms = {}
            for with_nce in (True, False, True):                                 # the first pass warms cuDNN and the allocator
                for _ in range(3):
                    step(with_nce)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(timed):
                    last = step(with_nce)
                e1.record()
                torch.cuda.synchronize()
                ms[with_nce] = e0.elapsed_time(e1) / timed
            out[name] = {"batch": b, "lambda_nce": lam, "ms_per_step": round(ms[True], 3),
                         "ms_per_step_without_patchnce": round(ms[False], 3), "patchnce_ms": round(ms[True] - ms[False], 3),
                         "patchnce_share": round((ms[True] - ms[False]) / ms[True], 4), "g_loss": float(last.item())}
            del gen, dis, og, od, ema, aug, sg, sd, photos
            torch.cuda.empty_cache()
        out["note"] = ("stand-in networks with the reference's shapes, every piece from this package (fused DiffAugment, hinge "
                       "losses, PatchNCE with encoder-feature reuse, 3-launch AMP optimiser step, 1-launch EMA), no .item() "
                       "reads inside the step; the same loop from stock torch pieces: scratch/train_step_bench.py, DESIGN.md 7.6")
        return out
    except Exception as e:  # noqa: BLE001 - a secondary line must not take the bench down
        return {"error": f"{type(e).__name__}: {e}"}


def timed_steps(step, steps, warmup, world, dev):
    """ms per step of `step` on this job: barrier + synchronize on both sides, CUDA events, max over ranks."""
    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


def head_line(args, pn, src, tgt, math, patches_per_image, world, dev, steps=20):
    """Secondary measurement at EVERY N: the same maps through the netF head (nc=256), fused tcgen05 path.  With
    N > 1 the head gradients are all-reduced (NCCL, the only collective of the path, SURVEY.md 8e) INSIDE every
    timed step: `patchnce_with_head(..., dp_group=True)` starts it on a side stream under the dense kernel."""
    torch.manual_seed(11)              # identical head weights on every rank
    netF = pn.PatchSampleF(use_mlp=True, nc=256).to(dev)
    netF.create_mlp(tgt)
    torch.manual_seed(7)               # identical ids on every rank

    def step():
        for t in tgt:
            t.grad = None
        netF.zero_grad(set_to_none=True)
        loss, _ = pn.patchnce_with_head(netF, src, tgt, args.tau, args.patches, math=math,
                                        dp_group=True if world > 1 else None)
        loss.backward()

    ms = timed_steps(step, steps, 3, world, dev)
    nparams = sum(p.numel() for p in netF.parameters())
    return {"ms_per_step": ms, "value": world * args.batch * patches_per_image / (ms * 1e-3), "unit": UNIT, "nc": 256,
            "steps": steps, "n_gpus": world, "scaling": "weak",
            "collective": (f"one flat NCCL all-reduce(AVG) of the {nparams} head gradients per step, inside the timed "
                           "region, overlapped with the dense kernel") if world > 1 else "none (single GPU)",
            "note": "netF head Linear-ReLU-Linear on tcgen05, parity unpinned by the reference"}


def strong_line(args, pn, src, tgt, math, patches_per_image, world, dev, layers, elem, peak, global_batch=64):
    """STRONG scaling (BASELINE config 5 as written: 'batch 64 ... across 2/4/8'): the global batch of 64 images is
    sharded over the N ranks, 64/N images each, reference-exact mode (no collective), through PatchNCELoss.forward
    + backward exactly like the headline -- and the same step replayed from a CUDA graph (GPU time without the
    Python host), which is what a fixed-shape training loop can do."""
    if global_batch % world or global_batch // world > args.batch:
        return {"skipped": f"global batch {global_batch} does not shard over {world} ranks of <= {args.batch} images"}
    b = global_batch // world
    s_src = [x[:b] for x in src]
    s_tgt = [x.detach()[:b].requires_grad_() for x in tgt]
    crit = pn.PatchNCELoss(args.tau, args.patches, [0, 4, 8, 12, 13], math=math)
    torch.manual_seed(7)

    def step():
        for t in s_tgt:
            t.grad = None
        crit(s_src, s_tgt).backward()

    steps = 50 if b >= 32 else 200
    ms = timed_steps(step, steps, 10, world, dev)
    path_bytes = algorithmic_bytes_per_image(layers, args.patches, elem) * b
    out = {"global_batch": global_batch, "batch_per_gpu": b, "n_gpus": world, "scaling": "strong", "steps": steps,
           "ms_per_step": ms, "value": global_batch * patches_per_image / (ms * 1e-3), "unit": UNIT,
           "roofline_path_frac": path_bytes / (ms * 1e-3) / 1e9 / peak,
           "api": "PatchNCELoss.forward + backward (eager, ids drawn inside the library)"}
    try:
        d_tgt = [t.detach() for t in s_tgt]
        dms = timed_steps(lambda: crit.loss_and_grads(s_src, d_tgt), steps, 10, world, dev)
        out["direct"] = {"ms_per_step": dms, "value": global_batch * patches_per_image / (dms * 1e-3),
                         "roofline_path_frac": path_bytes / (dms * 1e-3) / 1e9 / peak,
                         "api": "PatchNCELoss.loss_and_grads: the same forward + backward in one autograd-free call "
                                "(no engine hand-off, no ones_like of the root gradient)"}
    except Exception as e:  # noqa: BLE001 - secondary
        out["direct"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                step()
        torch.cuda.current_stream().wait_stream(side)
        with torch.cuda.graph(g):
            step()
        gms = timed_steps(g.replay, steps, 5, world, dev)
        out["graph_replay"] = {"ms_per_step": gms, "value": global_batch * patches_per_image / (gms * 1e-3),
                               "note": "the same fwd+bwd step captured once (static inputs, ids drawn by torch.randint "
                                       "inside the graph) and replayed: device time without the Python host"}
    except Exception as e:  # noqa: BLE001 - secondary
        out["graph_replay"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def nhwc_line(args, pn, src, tgt, math, patches_per_image, world, dev, layers, elem, peak, breakdowns, steps=20):
    """Secondary measurement at EVERY N: the same values stored channels-last (torch.channels_last), through the same
    PatchNCELoss.forward + backward.  NOT the reference's interface (its .view(B, C, -1) takes contiguous NCHW only):
    an extension for generators run in channels_last, reported beside the parity mode, never instead of it.  The
    path roofline uses the same algorithmic bytes (a patch is 2 P C useful bytes in either layout)."""
    try:
        cl = torch.channels_last
        s_src = [x.contiguous(memory_format=cl) for x in src]
        s_tgt = [x.detach().contiguous(memory_format=cl).requires_grad_() for x in tgt]
        crit = pn.PatchNCELoss(args.tau, args.patches, [0, 4, 8, 12, 13], math=math)
        torch.manual_seed(7)

        def step():
            for t in s_tgt:
                t.grad = None
            crit(s_src, s_tgt).backward()

        ms = timed_steps(step, steps, 5, world, dev)
        path_bytes = algorithmic_bytes_per_image(layers, args.patches, elem) * args.batch
        out = {"ms_per_step": ms, "value": world * args.batch * patches_per_image / (ms * 1e-3), "unit": UNIT,
               "steps": steps, "n_gpus": world, "scaling": "weak", "layout": "channels_last (B, H, W, C) storage",
               "roofline_path": {"bound": "hbm", "achieved": path_bytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                 "frac": path_bytes / (ms * 1e-3) / 1e9 / peak},
               "note": "extension: channels-last maps (the reference's .view rejects them); same ids / loss / gradient law"}
        b = 64 // world if 64 % world == 0 and 64 // world <= args.batch else None
        if b is not None and b < args.batch:                   # strong scaling of the global batch of 64 in this layout
            t_src = [x[:b] for x in s_src]
            t_tgt = [x.detach()[:b].requires_grad_() for x in s_tgt]

            def sstep():
                for t in t_tgt:
                    t.grad = None
                crit(t_src, t_tgt).backward()

            sms = timed_steps(sstep, 200, 10, world, dev)
            d_tgt = [t.detach() for t in t_tgt]
            dms = timed_steps(lambda: crit.loss_and_grads(t_src, d_tgt), 200, 10, world, dev)
            out["strong"] = {"global_batch": 64, "batch_per_gpu": b, "ms_per_step": sms,
                             "value": 64 * patches_per_image / (sms * 1e-3), "direct_ms_per_step": dms,
                             "direct_value": 64 * patches_per_image / (dms * 1e-3)}
        # the netF head on the same channels-last maps (collective inside the timed region when N > 1)
        torch.manual_seed(11)
        netF = pn.PatchSampleF(use_mlp=True, nc=256).to(dev)
        netF.create_mlp(s_tgt)
        torch.manual_seed(7)

        def hstep():
            for t in s_tgt:
                t.grad = None
            netF.zero_grad(set_to_none=True)
            loss, _ = pn.patchnce_with_head(netF, s_src, s_tgt, args.tau, args.patches, math=math,
                                            dp_group=True if world > 1 else None)
            loss.backward()

        hms = timed_steps(hstep, steps, 3, world, dev)
        out["head_mode"] = {"ms_per_step": hms, "value": world * args.batch * patches_per_image / (hms * 1e-3), "unit": UNIT,
                            "roofline_path_frac": path_bytes / (hms * 1e-3) / 1e9 / peak}
        breakdowns.append(("nhwc", step))          # run by main() after every timed line (the closures keep the maps alive)
        if world == 1:
            breakdowns.append(("nhwc_head", hstep))
        return out
    except Exception as e:  # noqa: BLE001 - secondary
        return {"error": f"{type(e).__name__}: {e}"}


def nccl_selfcheck(args, pn, layers, dev, world, rank, math, b=2):
    """N > 1: the data-parallel head path against the full batch on ONE rank, on this job's own NCCL communicator
    (the two-GPU pytest cases are skipped on single-GPU test boxes; this runs wherever the scaling bench runs).
    Every rank takes b images (maps seeded per rank), same ids, `dp_group=True`; rank 0 then rebuilds all N shards
    from their seeds, runs the whole batch alone and compares: loss, averaged head gradients, its own dense
    gradients."""
    import torch.distributed as dist
    try:
        torch.manual_seed(11)
        netF = pn.PatchSampleF(use_mlp=True, nc=256).to(dev)
        my_src, my_tgt = make_maps(layers, b, torch.float32, dev, 4321 + rank)
        my_tgt = [t.requires_grad_() for t in my_tgt]
        netF.create_mlp(my_tgt)
        torch.manual_seed(5)
        ids = pn.draw_ids(my_tgt, args.patches)
        loss, _ = pn.patchnce_with_head(netF, my_src, my_tgt, args.tau, args.patches, patch_ids=ids, math=math,
                                        dp_group=True)
        loss.backward()
        dp_grads = torch.cat([p.grad.reshape(-1).float() for p in netF.parameters()])
        mean_loss = loss.detach().clone()
        dist.all_reduce(mean_loss, op=dist.ReduceOp.SUM)
        mean_loss /= world
        # the same reduction through the un-overlapped helper must agree with itself across ranks
        spread = dp_grads.clone()
        dist.all_reduce(spread, op=dist.ReduceOp.MAX)
        rank_spread = float((spread - dp_grads).abs().max().item())
        res = None
        if rank == 0:
            shards = [make_maps(layers, b, torch.float32, dev, 4321 + r) for r in range(world)]
            f_src = [torch.cat([sh[0][l] for sh in shards]) for l in range(len(layers))]
            f_tgt = [torch.cat([sh[1][l] for sh in shards]).requires_grad_() for l in range(len(layers))]
            netF.zero_grad(set_to_none=True)
            full, _ = pn.patchnce_with_head(netF, f_src, f_tgt, args.tau, args.patches, patch_ids=ids, math=math)
            full.backward()
            ref = torch.cat([p.grad.reshape(-1).float() for p in netF.parameters()])
            g_err = float(((dp_grads - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item())
            l_err = abs(float(mean_loss.item()) - float(full.item())) / abs(float(full.item()))
            d_err = max(float(((f.grad[:b] * world - m.grad).abs().max() / m.grad.abs().max().clamp_min(1e-30)).item())
                        for f, m in zip(f_tgt, my_tgt))
            res = {"ranks": world, "images_per_rank": b, "head_grad_rel_err": g_err, "loss_rel_err": l_err,
                   "dense_grad_rel_err": d_err, "rank_spread_abs": rank_spread,
                   "ok": bool(g_err < 2e-3 and l_err < 1e-4 and d_err < 2e-3 and rank_spread == 0.0),
                   "what": "patchnce_with_head(dp_group=True) on N ranks vs the full batch on rank 0"}
        dist.barrier()
        return res
    except Exception as e:  # noqa: BLE001
        try:
            dist.barrier()
        except Exception:  # noqa: BLE001
            pass
        return {"ok": False, "error": f"{type(e).__name__}: {e}"} if rank == 0 else None


def grad_reducer_line(pn, dev, world, n=20):
    """N > 1, SURVEY.md 8f row 1 (BASELINE config 5: "NCCL allreduce of netF/G/D grads"): dp.GradReducer averaging the
    gradients of a parameter set shaped like the reference generator (tests/golden/model_param_shapes.json, 11.4 M
    values in 48 tensors, 45.5 MB) over the N ranks -- flat fp32 buckets all-reduced (mean) on a side stream from
    post-accumulate-grad hooks, written back at the end of backward().  The backward pass here is the cheapest
    one that reaches every parameter (loss = sum of the parameter sums), so the number is the reducer's own cost:
    hooks, bucket copies, NCCL, write-back -- not hidden under a generator backward as it is in training."""
    import torch.distributed as dist
    from gan_variant_research_b200 import dp
    try:
        shapes = json.load(open(os.path.join(ROOT, "tests", "golden", "model_param_shapes.json")))["generator"]
        torch.manual_seed(100 + dist.get_rank())
        params = [torch.randn(*s, device=dev).requires_grad_() for s in shapes]

        def backward():
            for p in params:
                p.grad = None
            total = params[0].sum()
            for p in params[1:]:
                total = total + p.sum()
            total.backward()

        def timed():
            for _ in range(5):
                backward()
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                backward()
            e1.record()
            dist.barrier()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        plain = timed()
        red = dp.GradReducer(params)
        with_red = timed()
        # averaged gradients are identical on every rank (each rank's own are all ones here: the mean is 1)
        ok = all(bool(torch.allclose(p.grad, torch.ones_like(p))) for p in params)
        red.remove()
        nbytes = 4 * sum(p.numel() for p in params)
        return {"n_gpus": world, "tensors": len(params), "bytes": nbytes, "buckets": len(red.buckets),
                "backward_ms": plain, "backward_with_reducer_ms": with_red, "reducer_ms": with_red - plain,
                "allreduce_gbs": nbytes / max(with_red - plain, 1e-9) / 1e6, "averaged_ok": ok,
                "what": "dp.GradReducer on reference-generator-shaped parameters, NCCL all-reduce(mean) per bucket"}
    except Exception as e:  # noqa: BLE001 - secondary
        return {"error": f"{type(e).__name__}: {e}"}


def config_lines(args, pn, layers, dev, math, peak):
    """N = 1: the other BASELINE configurations of the loss on one GPU -- B = 1 (configs 1 and 2) and B = 16 (config 3)
    in fp32, and fp16 maps at the headline batch (the AMP regime train_cutpp.py:268 runs in) -- each through
    PatchNCELoss.forward + backward with its own path roofline."""
    rows = []
    ppi = sum(min(args.patches, h * w) for _, h, w, _ in layers)
    for name, b, tdtype, elem in (("b1_fp32", 1, torch.float32, 4), ("b16_fp32", 16, torch.float32, 4),
                                  (f"b{args.batch}_fp16", args.batch, torch.float16, 2),
                                  ("b1_fp32_channels_last", 1, torch.float32, 4), ("b16_fp32_channels_last", 16, torch.float32, 4),
                                  (f"b{args.batch}_fp16_channels_last", args.batch, torch.float16, 2)):
        try:
            src, tgt = make_maps(layers, b, tdtype, dev, 99)
            if name.endswith("channels_last"):                # the extension of DESIGN.md 4.7, not the reference's layout
                src = [x.contiguous(memory_format=torch.channels_last) for x in src]
                tgt = [x.contiguous(memory_format=torch.channels_last) for x in tgt]
            tgt = [t.requires_grad_() for t in tgt]
            crit = pn.PatchNCELoss(args.tau, args.patches, [0, 4, 8, 12, 13], math=math)

            def step():
                for t in tgt:
                    t.grad = None
                crit(src, tgt).backward()

            steps = 200 if b <= 16 else 30
            ms = timed_steps(step, steps, 10, 1, dev)
            d_tgt = [t.detach() for t in tgt]
            dms = timed_steps(lambda: crit.loss_and_grads(src, d_tgt), steps, 10, 1, dev)
            pb = algorithmic_bytes_per_image(layers, args.patches, elem) * b
            rows.append({"config": name, "batch": b, "dtype": str(tdtype).replace("torch.", ""), "steps": steps,
                         "ms_per_step": ms, "value": b * ppi / (ms * 1e-3), "unit": UNIT,
                         "direct_ms_per_step": dms,
                         "roofline_path": {"bound": "hbm", "achieved": pb / (ms * 1e-3) / 1e9, "peak": peak,
                                           "unit": "GB/s", "frac": pb / (ms * 1e-3) / 1e9 / peak}})
            del src, tgt
        except Exception as e:  # noqa: BLE001
            rows.append({"config": name, "error": f"{type(e).__name__}: {e}"})
    # BASELINE config 4: 512^2 images (every HW x 4), P = 1024, B = 8 -- the key-blocked tcgen05 kernel (k_loss_tc)
    try:
        big = [(c, 2 * h, 2 * w, relu) for c, h, w, relu in layers]
        src, tgt = make_maps(big, 8, torch.float32, dev, 99)
        tgt = [t.requires_grad_() for t in tgt]
        crit4 = pn.PatchNCELoss(args.tau, 1024, [0, 4, 8, 12, 13], math=math)

        def step4():
            for t in tgt:
                t.grad = None
            crit4(src, tgt).backward()

        ms = timed_steps(step4, 50, 10, 1, dev)
        ppi4 = sum(min(1024, h * w) for _, h, w, _ in big)
        pb = algorithmic_bytes_per_image(big, 1024, 4) * 8
        rows.append({"config": "cfg4_b8_512sq_p1024", "batch": 8, "dtype": "float32", "num_patches": 1024, "steps": 50,
                     "ms_per_step": ms, "value": 8 * ppi4 / (ms * 1e-3), "unit": UNIT,
                     "roofline_path": {"bound": "hbm", "achieved": pb / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                       "frac": pb / (ms * 1e-3) / 1e9 / peak}})
        del src, tgt
    except Exception as e:  # noqa: BLE001
        rows.append({"config": "cfg4_b8_512sq_p1024", "error": f"{type(e).__name__}: {e}"})
    torch.cuda.empty_cache()
    # the north-star shape (netF head, dim 256) at the batches the reference trains with: the fused head through autograd
    # (patchnce_with_head + backward) and through the autograd-free entry (head_loss_and_grads)
    for name, b in (("b1_fp32_head", 1), ("b16_fp32_head", 16)):
        try:
            src, tgt = make_maps(layers, b, torch.float32, dev, 99)
            tgt = [t.requires_grad_() for t in tgt]
            torch.manual_seed(3)
            netF = pn.PatchSampleF(use_mlp=True, nc=256).to(dev)
            netF.create_mlp(tgt)
            hp = list(netF.parameters())

            def hstep():
                for t in tgt:
                    t.grad = None
                for q in hp:
                    q.grad = None
                loss, _ = pn.patchnce_with_head(netF, src, tgt, args.tau, args.patches, math=math)
                loss.backward()

            d_tgt = [t.detach() for t in tgt]

            def dstep():
                for q in hp:
                    q.grad = None
                pn.head_loss_and_grads(netF, src, d_tgt, args.tau, args.patches, math=math)

            ms = timed_steps(hstep, 200, 10, 1, dev)
            dms = timed_steps(dstep, 200, 10, 1, dev)
            pb = algorithmic_bytes_per_image(layers, args.patches, 4) * b
            rows.append({"config": name, "batch": b, "dtype": "float32", "nc": 256, "steps": 200, "ms_per_step": ms,
                         "value": b * ppi / (ms * 1e-3), "unit": UNIT, "direct_ms_per_step": dms,
                         "direct_value": b * ppi / (dms * 1e-3),
                         "roofline_path": {"bound": "hbm", "achieved": pb / (ms * 1e-3) / 1e9, "peak": peak,
                                           "unit": "GB/s", "frac": pb / (ms * 1e-3) / 1e9 / peak,
                                           "frac_direct": pb / (dms * 1e-3) / 1e9 / peak},
                         "note": "netF head Linear-ReLU-Linear on tcgen05, parity unpinned by the reference"})
            del src, tgt, netF
        except Exception as e:  # noqa: BLE001
            rows.append({"config": name, "error": f"{type(e).__name__}: {e}"})
    torch.cuda.empty_cache()
    return rows


def module_split_line(args, pn, src, tgt, math, patches_per_image, steps=20):
    """Secondary measurement: the same maps through the north-star module signatures, composed in Python the way
    upstream CUT does -- feat_k, ids = PatchSampleF(src); feat_q, _ = PatchSampleF(tgt, ids); mean over layers of
    PatchNCELoss(feat_q_l, feat_k_l) -- instead of the fused all-layer call."""
    samp = pn.PatchSampleF(use_mlp=False)
    crit = pn.PatchNCELoss(args.tau, args.patches, math=math)
    batch = tgt[0].shape[0]

    def step():
        for t in tgt:
            t.grad = None
        with torch.no_grad():
            feat_k, ids = samp(src, args.patches, None)
        feat_q, _ = samp(tgt, args.patches, ids)
        loss = sum(crit(q, k, batch_size=batch) for q, k in zip(feat_q, feat_k)) / len(feat_q)
        loss.backward()

    for _ in range(3):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps

    def step_list():
        for t in tgt:
            t.grad = None
        with torch.no_grad():
            feat_k, ids = samp(src, args.patches, None)
        feat_q, _ = samp(tgt, args.patches, ids)
        crit(feat_q, feat_k, batch_size=batch).backward()

    lms = timed_steps(step_list, steps, 3, 1, tgt[0].device)
    return {"ms_per_step": ms, "value": args.batch * patches_per_image / (ms * 1e-3), "unit": UNIT, "steps": steps,
            "note": "PatchSampleF.forward(feats, num_patches, patch_ids) + per-layer PatchNCELoss(feat_q, feat_k)",
            "list_form": {"ms_per_step": lms, "value": args.batch * patches_per_image / (lms * 1e-3), "unit": UNIT,
                          "note": "the same composition with PatchNCELoss(feat_q_list, feat_k_list): every layer's rows "
                                  "loss in one library call (pnce_rows_loss_multi_fwd_bwd)"}}


def run_e2e(args, pn, crit, layers, tdtype, elem, dev, world, rank):
    """The same metric through the public API with HOST buffers.  The feature maps of every step live
    in pinned host memory and are handed to ``PatchNCELoss.forward`` through ``pinned_as_device`` (a
    zero-copy device view): the gather kernel pulls exactly the sampled 32-byte sectors over PCIe
    inside the timed region -- that IS the step's host->device transfer -- and the step's result, the
    loss, is read back (D2H).  The dense gradients stay on the device, where the generator's backward
    consumes them in the training loop (train_cutpp.py:300-308).  ``bulk_copy`` repeats the
    measurement the naive way (whole maps copied H2D every step, then the device path)."""
    B = args.batch
    shapes = [(B, c, h, w) for c, h, w, _ in layers]
    h_src = [torch.randn(s, dtype=torch.float32).to(tdtype).pin_memory() for s in shapes]
    h_tgt = [torch.randn(s, dtype=torch.float32).to(tdtype).pin_memory() for s in shapes]
    h_loss = torch.empty((), dtype=torch.float32).pin_memory()
    a_src = [pn.pinned_as_device(h, dev) for h in h_src]
    a_tgt = [pn.pinned_as_device(h, dev).requires_grad_() for h in h_tgt]
    d_src = [torch.empty(s, dtype=tdtype, device=dev) for s in shapes]
    d_tgt = [torch.empty(s, dtype=tdtype, device=dev).requires_grad_() for s in shapes]

    def step_zero_copy():
        for t in a_tgt:
            t.grad = None
        loss = crit(a_src, a_tgt)
        loss.backward()
        h_loss.copy_(loss.detach(), non_blocking=True)

    def step_bulk():
        for d, h in zip(d_src, h_src):
            d.copy_(h, non_blocking=True)
        for d, h in zip(d_tgt, h_tgt):
            d.grad = None
            d.detach().copy_(h, non_blocking=True)
        loss = crit(d_src, d_tgt)
        loss.backward()
        h_loss.copy_(loss.detach(), non_blocking=True)

    def timed(fn, n):
        fn()
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            torch.distributed.all_reduce(dt, op=torch.distributed.ReduceOp.MAX)
        return float(dt.item())

    patches_per_image = sum(min(args.patches, h * w) for _, h, w, _ in layers)
    n_elem = sum(c * h * w for c, h, w, _ in layers) * B
    sampled = 2 * B * sum(min(args.patches, h * w) * c for c, h, w, _ in layers)      # elements read, src + tgt
    dt = timed(step_zero_copy, args.e2e_steps)
    loss_zc = float(h_loss.item())
    bulk_steps = max(2, args.e2e_steps // 2)
    dt_bulk = timed(step_bulk, bulk_steps)
    # the other end of the claim: the dense gradients are ALSO brought back to the host every step (a caller whose
    # generator backward does not run on this GPU) -- 3.2 GB of D2H per step at B=64, PCIe-bound
    h_grads = [torch.empty(s, dtype=tdtype).pin_memory() for s in shapes]

    def step_grads_d2h():
        step_zero_copy()
        for h, t in zip(h_grads, a_tgt):
            h.copy_(t.grad, non_blocking=True)

    gd_steps = max(2, args.e2e_steps // 3)
    dt_gd = timed(step_grads_d2h, gd_steps)
    # the same zero-copy step on CHANNELS-LAST host maps (the extension of DESIGN.md 4.7; the same pinned bytes re-read
    # as (B, H, W, C) storage -- the values are random either way): a sampled patch is one contiguous row, so the gather
    # pulls the useful bytes over PCIe instead of one 32-byte sector per element
    nhwc = None
    try:
        def cl_view(h, s):
            b, c, hh, ww = s
            return h.view(-1).view(b, hh, ww, c).permute(0, 3, 1, 2)
        c_src = [pn.pinned_as_device(cl_view(h, s), dev) for h, s in zip(h_src, shapes)]
        c_tgt = [pn.pinned_as_device(cl_view(h, s), dev).requires_grad_() for h, s in zip(h_tgt, shapes)]

        def step_zero_copy_cl():
            for t in c_tgt:
                t.grad = None
            loss = crit(c_src, c_tgt)
            loss.backward()
            h_loss.copy_(loss.detach(), non_blocking=True)

        dt_cl = timed(step_zero_copy_cl, args.e2e_steps)
        nhwc = {"value": world * B * patches_per_image * args.e2e_steps / dt_cl, "unit": UNIT,
                "h2d_bytes_per_step": sampled * elem, "d2h_bytes_per_step": 4, "steps": args.e2e_steps,
                "note": "channels-last pinned host maps (extension, not the reference's layout): each sampled patch is one "
                        "contiguous row over PCIe"}
    except Exception as e:  # noqa: BLE001 - secondary
        nhwc = {"error": f"{type(e).__name__}: {e}"}
    with_grads = {"value": world * B * patches_per_image * gd_steps / dt_gd, "unit": UNIT,
                  "h2d_bytes_per_step": sampled * 32, "d2h_bytes_per_step": 4 + n_elem * elem, "steps": gd_steps,
                  "note": "zero-copy inputs as in the headline e2e, plus every dense d tgt_feat copied to pinned host "
                          "memory inside the timed region"}
    return {"value": world * B * patches_per_image * args.e2e_steps / dt, "unit": UNIT,
            "h2d_bytes_per_step": sampled * 32, "d2h_bytes_per_step": 4,
            "steps": args.e2e_steps, "loss": loss_zc,
            "api": "PatchNCELoss.forward + backward on pinned host maps via pinned_as_device (zero-copy: the gather "
                   "reads one 32-byte sector per sampled element over PCIe; h2d_bytes counts those sectors, "
                   f"useful bytes = {sampled * elem})",
            "n_gpus": world,
            "scaling_note": "per-rank host memory and PCIe are shared on one box: this number scales worse than the "
                            "device-resident one (0.63 efficiency at N=8 in round 1)",
            "with_grads_d2h": with_grads,
            "channels_last": nhwc,
            "bulk_copy": {"value": world * B * patches_per_image * bulk_steps / dt_bulk, "unit": UNIT,
                          "h2d_bytes_per_step": 2 * n_elem * elem, "steps": bulk_steps,
                          "note": "whole maps copied H2D every step, then the device path (PCIe-bound)"}}


if __name__ == "__main__":
    main()
