"""Host side of the B200 PatchNCE path: the reference's Python seam over the libpnce C ABI.

Mirrors ``GAN_Variant1/losses/patchnce_cut.py`` of the reference (same names, arguments and
return values) so ``training/train_cutpp.py:285-292`` runs unchanged:

* ``compute_patchnce_loss(generator, src_images, tgt_images, nce_layers, temperature, num_patches)``
  -- patchnce_cut.py:113-149
* ``PatchNCELoss(temperature, num_patches, nce_layers).forward(src_feats, tgt_feats)``
  -- patchnce_cut.py:7-110

and adds the north-star module split underneath (SURVEY.md section 8b):

* ``PatchSampleF(use_mlp=False, nc=256).forward(feats, num_patches, patch_ids)``
* ``PatchNCELoss(...).forward(feat_q, feat_k)`` on (B*P, D) rows.

torch is plumbing here (device memory, streams, autograd glue); every FLOP and byte of the path
runs in the hand-written sm_100a kernels of ``csrc/``.  There is no CPU or eager fallback: CPU
tensors or a missing ``libpnce.so`` raise.
"""
from __future__ import annotations

import ctypes
import os
import sys
import threading
from typing import List, Optional, Sequence

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib

_DTYPES = {torch.float32: _lib.PNCE_F32, torch.float16: _lib.PNCE_F16, torch.bfloat16: _lib.PNCE_BF16}
_MATH = {"simt_f32": _lib.MATH_SIMT_F32, "tc_bf16x3": _lib.MATH_TC_BF16X3, "tc_bf16": _lib.MATH_TC_BF16}

#: contraction engine used when a module does not choose one
DEFAULT_MATH = "tc_bf16x3"
NORM_EPS = 1e-6          # F.normalize(..., eps=1e-6)   patchnce_cut.py:77-78


def _stream_ptr(device) -> int:
    # the raw cudaStream_t of torch's current stream (torch.cuda.current_stream(device).cuda_stream, without building
    # the Stream object: 0.2 us instead of 2.2 us, on a path that small batches are bound by)
    return torch._C._cuda_getCurrentRawStream(device.index)


class _NullCtx:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NULL_CTX = _NullCtx()


def _on_device(dev):
    """``torch.cuda.device(dev)``, or nothing when ``dev`` already is the current device (the usual case:
    the context manager costs ~10 us of host time per use, which matters at the reference's batch of 1)."""
    return _NULL_CTX if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(
            f"{what} is on {t.device}: the B200 PatchNCE path has no CPU fallback "
            "(use the reference implementation or oracle/ for CPU checks)")


def patch_count(num_patches: int, hw: int) -> int:
    """P = min(num_patches, H*W) -- patchnce_cut.py:60"""
    return min(int(num_patches), int(hw))


def draw_patch_ids(feat: torch.Tensor, num_patches: int) -> torch.Tensor:
    """The reference's id draw, issued exactly as it issues it (shape, range, device, one call per
    layer) so the ids are bit-identical and the device RNG stream stays aligned with the rest of
    ``train_step`` -- patchnce_cut.py:60-63, SURVEY.md section 3.1 RNG note."""
    hw = feat.shape[2] * feat.shape[3]
    return torch.randint(0, hw, (patch_count(num_patches, hw),), device=feat.device)


_ID_STREAMS = {}         # device index -> side stream the id draw + sort are issued on
# The side-stream route costs ~120 us more HOST time per step than the in-line one (stream switch, two allocations on
# the side pool, event hand-over, record_stream) and takes the 8 us id sort off the GPU's critical path: it pays once a step's
# GPU time is comfortably above the host's ~0.3 ms, i.e. from ~2.5 GB of feature maps (B >= 25 at the CUT shapes in fp32;
# at B = 16 -- 1.6 GB, 0.25 ms of GPU work -- it made the step host-bound: 0.31 vs 0.26 ms)
_SIDE_STREAM_MIN_BYTES = 5 << 29


def _id_stream(dev) -> "torch.cuda.Stream":
    side = _ID_STREAMS.get(dev.index)
    if side is None:
        # high priority: its few small CTAs take the first slots that free up under a kernel that fills the GPU
        # (at equal priority they wait until that kernel's whole grid has been dispatched)
        side = _ID_STREAMS[dev.index] = torch.cuda.Stream(device=dev, priority=-1)
    return side


def draw_patch_ids_all(feats, num_patches: int) -> List[torch.Tensor]:
    """One ``draw_patch_ids`` per layer, in layer order (patchnce_cut.py:36-38, :63): the torch.randint
    path, used while a CUDA graph is being captured (torch's graph-safe generator state), on the fp32
    CUDA-core path and whenever the in-library draw has not been validated (``_philox_ready``)."""
    return [draw_patch_ids(f, num_patches) for f in feats]


# ------------------------------------------------------------------------------------------------
# the id draw inside the library (pnce_fwd_draw / pnce_plan_ids_draw / pnce_draw_ids, include/pnce.h)
# ------------------------------------------------------------------------------------------------
_PHILOX_OK = {}          # device index -> True (validated against torch.randint) / False (disabled)


def _philox_ready(dev) -> bool:
    """True when the library may draw the ids itself on ``dev``.  Checked ONCE per device and process: a handful
    of ``torch.randint`` calls (sizes that exercise one- and multi-block launches) against ``pnce_draw_ids`` at the
    same generator state, and the generator's offset bookkeeping (+4 per call).  The generator is left exactly as
    it was found.  Any mismatch -- another torch build with another sampling law -- switches the library draw off
    for good and the host keeps calling ``torch.randint`` like the reference does (ids stay bit-exact either way)."""
    ok = _PHILOX_OK.get(dev.index)
    if ok is not None:
        return ok
    if torch.cuda.is_current_stream_capturing():
        return False                                  # decide later, outside the capture
    ok = False
    try:
        gen = torch.cuda.default_generators[dev.index]
        state = gen.get_state()
        probes = [(256 * 256, 256), (64 * 64, 256), (128 * 128, 1024), (100, 100), (7, 7), (512 * 512, 300)]
        ref = [torch.randint(0, hw, (p,), device=dev) for hw, p in probes]
        end = gen.get_offset()
        gen.set_state(state)
        seed, off = gen.initial_seed(), gen.get_offset()
        ours = [torch.empty(p, dtype=torch.int64, device=dev) for _, p in probes]
        arr = (_lib.PnceLayer * len(probes))()
        for l, ((hw, p), o) in enumerate(zip(probes, ours)):
            arr[l].ids, arr[l].C, arr[l].H, arr[l].W, arr[l].P = o.data_ptr(), 1, 1, hw, p
        with _on_device(dev):
            _lib.check(_lib.load().pnce_draw_ids(arr, len(probes), seed, off, _stream_ptr(dev)), "pnce_draw_ids")
        ok = end == off + 4 * len(probes) and all(torch.equal(a, b) for a, b in zip(ref, ours))
        gen.set_state(state)
        if not ok:
            print("gan_variant_research_b200: torch.randint does not follow the Philox law the library draws ids "
                  "with on this torch build; falling back to torch.randint calls (ids stay bit-exact).", file=sys.stderr)
    except Exception as e:  # noqa: BLE001 - an unexpected generator API: stay on torch.randint
        print(f"gan_variant_research_b200: in-library id draw disabled ({type(e).__name__}: {e})", file=sys.stderr)
        ok = False
    _PHILOX_OK[dev.index] = ok
    return ok


def draw_ids(feats, num_patches: int) -> List[torch.Tensor]:
    """The reference's id draws for a list of maps (one per layer, layer order, patchnce_cut.py:60-63) in ONE
    launch of the library (``pnce_draw_ids``) when the in-library draw is validated on this device, else the
    ``torch.randint`` calls themselves.  Same ids, same generator state afterwards, either way."""
    feats = list(feats)
    if not feats:
        return []
    dev = feats[0].device
    if (not feats[0].is_cuda or any(f.device != dev for f in feats) or len(feats) > _lib.MAX_LAYERS
            or torch.cuda.is_current_stream_capturing() or not _philox_ready(dev)):
        return draw_patch_ids_all(feats, num_patches)
    n = len(feats)
    hw = [f.shape[2] * f.shape[3] for f in feats]
    p_list = [patch_count(num_patches, x) for x in hw]
    arr = (_lib.PnceLayer * n)()
    with _on_device(dev):
        ids_all = torch.empty(sum(p_list), dtype=torch.int64, device=dev)
        ptr = ids_all.data_ptr()
        for l in range(n):
            arr[l].ids, arr[l].C, arr[l].H, arr[l].W, arr[l].P = ptr, 1, 1, hw[l], p_list[l]
            ptr += 8 * p_list[l]
        seed, off = _philox_take(dev, n)
        _lib.check(_lib.load().pnce_draw_ids(arr, n, seed, off, _stream_ptr(dev)), "pnce_draw_ids")
    return list(ids_all.split(p_list))


def _philox_take(dev, n_draws: int):
    """(seed, offset) of the device's default CUDA generator, which is advanced by what ``n_draws`` randint calls
    consume (4 each) -- the RNG stream stays aligned with the reference's training step (SURVEY.md 3.1)."""
    gen = torch.cuda.default_generators[dev.index]
    off = gen.get_offset()
    gen.set_offset(off + 4 * n_draws)
    return gen.initial_seed(), off


class _PinnedAlias:
    """``__cuda_array_interface__`` view of a pinned host tensor (unified addressing: a pinned
    allocation is addressable from the device under the same pointer)."""

    def __init__(self, t: torch.Tensor):
        typestr = {torch.float32: "<f4", torch.float16: "<f2", torch.int64: "<i8"}.get(t.dtype)
        if typestr is None:
            raise RuntimeError(f"pinned_as_device: unsupported dtype {t.dtype}")
        self.__cuda_array_interface__ = {"shape": tuple(t.shape), "typestr": typestr,
                                         "data": (t.data_ptr(), False), "version": 2, "strides": None}


def pinned_as_device(t: torch.Tensor, device=None) -> torch.Tensor:
    """Device-side view of a PINNED, contiguous host tensor -- no copy.  Feature maps that live in host
    memory can be handed to ``PatchNCELoss`` / ``PatchSampleF`` through this view: the gather kernel
    then pulls exactly the sampled 32-byte sectors over PCIe (2*B*P*C of them per layer) instead of
    the caller copying whole maps to the device first (B*C*H*W elements each) -- 8x fewer bytes on
    the bus at the CUT shapes (bench.py ``e2e``).  The view shares storage with ``t``; keep ``t`` alive.
    The returned tensor is a CUDA tensor as far as autograd is concerned (gradients are device
    tensors), so ``pinned_as_device(h).requires_grad_()`` works as a target map."""
    if t.is_cuda:
        return t
    if t.dim() == 4 and not t.is_contiguous() and t.is_contiguous(memory_format=torch.channels_last) and t.is_pinned():
        # channels-last host maps: alias the dense (B, H, W, C) storage, hand back the (B, C, H, W) view -- the gather then
        # pulls each sampled patch as ONE contiguous row over PCIe (DESIGN.md 4.7)
        return pinned_as_device(t.permute(0, 2, 3, 1), device).permute(0, 3, 1, 2)
    if not t.is_pinned() or not t.is_contiguous():
        raise RuntimeError("pinned_as_device needs a pinned, contiguous host tensor (tensor.pin_memory())")
    if t.dtype == torch.bfloat16:            # no typestr for bf16: alias the bits as int16, then view
        alias = torch.as_tensor(_PinnedAlias(t.view(torch.float16)),
                                device=device or torch.device("cuda", torch.cuda.current_device()))
        out = alias.view(torch.bfloat16)
    else:
        out = torch.as_tensor(_PinnedAlias(t), device=device or torch.device("cuda", torch.cuda.current_device()))
    out._pnce_host_owner = t                  # keeps the pinned storage alive as long as the view
    return out


# ------------------------------------------------------------------------------------------------
# lazy non-finite warnings (the reference prints from inside the loop after a host sync, :97-98;
# here the flag is copied to pinned memory asynchronously and reported on a later call)
# ------------------------------------------------------------------------------------------------
class _WarnQueue:
    """The kernels write their two status words (guarded-image count, protocol-timeout flag) STRAIGHT
    INTO PINNED HOST MEMORY (zero-copy over PCIe: pinned allocations are device-addressable under
    unified addressing), so no D2H memcpy sits on the stream between the forward and the backward
    kernels -- and no CUDA event either: the host stores -1 into word 0 before the launch and the loss
    kernel's last CTA overwrites it with the count (>= 0) when the forward is done, so "word 0 >= 0" IS the
    completion test (an event record + query per step cost ~8 us of host time, which small batches are bound
    by).  A ring of 64 slots, one queue per device; a lock makes it safe to call from several threads (the
    autograd engine's threads never touch it: only forwards do)."""
    SLOTS = 64

    def __init__(self):
        self.pending = []            # slots in launch order
        self.host = None
        self.words = None            # numpy view of the pinned buffer: plain loads and stores, no tensor indexing
        self.free = []
        self.mb = [False] * self.SLOTS       # slot -> minibatch-negatives launch (the count is of layers)
        self.lock = threading.Lock()

    def acquire(self, mb: bool = False):
        """-> (slot, device-usable pointer to int32[2]) or (None, 0) while a CUDA graph is being captured
        (then the failure of a launch shows in-band: the loss is NaN, include/pnce.h).  ``mb``: a minibatch-negatives
        launch, whose count is of guarded layers."""
        if torch.cuda.is_current_stream_capturing():
            return None, 0
        with self.lock:
            if self.host is None:
                self.host = torch.zeros(self.SLOTS, 2, dtype=torch.int32).pin_memory()
                self.words = self.host.numpy()
                self.base = self.host.data_ptr()
                self.free = list(range(self.SLOTS))
            if not self.free:
                self._poll(False)
                if not self.free:                    # 64 launches in flight un-polled: drain the device
                    torch.cuda.synchronize()
                    self._poll(True)
            slot = self.free.pop()
            self.mb[slot] = mb
            self.words[slot, 0] = -1                 # "in flight"; word 1 is cleared by the sequence's first kernel
            self.words[slot, 1] = 0
            self.pending.append(slot)
        return slot, self.base + 8 * slot

    def poll(self, block: bool = False) -> int:
        """Print the reference's warning for finished launches; returns images guarded so far."""
        if not self.pending:
            return 0
        if block:
            if torch.cuda.is_current_stream_capturing():
                return 0
            torch.cuda.synchronize()
        with self.lock:
            return self._poll(block)

    def _poll(self, drained: bool) -> int:
        total, keep, proto_err = 0, [], False
        w = self.words
        for slot in self.pending:
            n = int(w[slot, 0])
            if n >= 0 or drained:
                self.free.append(slot)
                proto_err = proto_err or bool(w[slot, 1])
                if n > 0:
                    if self.mb[slot]:
                        for _ in range(n):
                            print("Warning: NaN in PatchNCE loss (minibatch negatives). A layer's loss replaced by 0.")
                    else:
                        print(f"Warning: NaN in PatchNCE loss. {n} (layer, image) loss(es) replaced by 0.")
                    total += n
            else:
                keep.append(slot)
        self.pending = keep
        if proto_err:
            raise _lib.PnceError("libpnce kernel protocol timeout (tcgen05 pipeline stalled)")
        return total


_WARN_QUEUES = {}        # device index -> _WarnQueue


def _warn_queue(dev) -> _WarnQueue:
    q = _WARN_QUEUES.get(dev.index)
    if q is None:
        q = _WARN_QUEUES.setdefault(dev.index, _WarnQueue())
    return q


def poll_nonfinite_warnings(block: bool = False) -> int:
    total = sum(q.poll(block) for q in list(_WARN_QUEUES.values()))
    if block and not torch.cuda.is_current_stream_capturing():
        for t in list(_NETF_STATUS.values()):
            if int(t.item()) != 0:
                t.zero_()
                raise _lib.PnceError("libpnce kernel protocol timeout (tcgen05 pipeline stalled, netF head)")
    return total


# ------------------------------------------------------------------------------------------------
# fused path: all layers, forward = 3 launches (id draw + sort | gather | logits/CE/dQ), backward = 1
# ------------------------------------------------------------------------------------------------
class _ShapePlan:
    """Everything a fused call needs that depends only on the problem SHAPE (device, dtype, batch, layer
    geometry, patch counts, math mode) -- built once and reused by every step of a training loop, so that the
    host side of a step is a handful of pointer stores and one C call each way (small batches are bound by this
    host path, not by the GPU: DESIGN.md 4.5).  The C-ABI layer tables are owned here; the forward table and the
    backward table are separate objects because autograd runs ``backward`` on its own thread, and each is
    guarded by a lock so that two Python threads sharing a shape do not interleave their pointer stores."""

    __slots__ = ("n", "batch", "dtype", "dtype_code", "math", "math_code", "dev", "p_list", "p_total", "tc",
                 "ws_bytes", "plan_bytes", "fwd_layers", "bwd_layers", "fwd_lock", "bwd_lock", "big", "shapes", "nhwc",
                 "mb", "world", "slot_offset", "slot_bytes")

    def __init__(self, dev, dtype, shapes, p_list, math, nhwc=False, mb=False, world=1):
        if mb:
            mb_check(shapes[0][0], [s[1] for s in shapes], p_list, math, world=world)
        lib = _lib.load()
        self.mb = mb                             # minibatch negatives (pnce_mb_fwd)
        self.world = world                       # > 1: global negatives over `world` ranks (pnce_mb_shard_*)
        self.slot_offset = self.slot_bytes = 0
        self.n, self.batch, self.dtype, self.dev, self.math = len(shapes), shapes[0][0], dtype, dev, math
        self.nhwc = nhwc                         # channels-last storage (pnce_fwd_ex / pnce_bwd_ex, LAYOUT_NHWC)
        self.dtype_code, self.math_code = _DTYPES[dtype], _MATH[math]
        self.shapes = shapes
        self.p_list, self.p_total = list(p_list), sum(p_list)
        self.fwd_layers = (_lib.PnceLayer * self.n)()
        self.bwd_layers = (_lib.PnceLayer * self.n)()
        for arr in (self.fwd_layers, self.bwd_layers):
            for l, ((_, c, h, w), p) in enumerate(zip(shapes, p_list)):
                arr[l].C, arr[l].H, arr[l].W, arr[l].P = c, h, w, p
        nbytes = ctypes.c_size_t(0)
        if world > 1:
            so, sb = ctypes.c_size_t(0), ctypes.c_size_t(0)
            _lib.check(lib.pnce_mb_shard_workspace_bytes(self.fwd_layers, self.n, self.batch, world, ctypes.byref(nbytes),
                                                         ctypes.byref(so), ctypes.byref(sb)), "pnce_mb_shard_workspace_bytes")
            self.slot_offset, self.slot_bytes = so.value, sb.value
        elif mb:
            _lib.check(lib.pnce_mb_workspace_bytes(self.fwd_layers, self.n, self.batch, ctypes.byref(nbytes)),
                       "pnce_mb_workspace_bytes")
        else:
            _lib.check(lib.pnce_workspace_bytes(self.fwd_layers, self.n, self.batch, ctypes.byref(nbytes)),
                       "pnce_workspace_bytes")
        self.ws_bytes = nbytes.value
        # the tensor-core kernels' envelope (csrc/pnce_api.cu tc_shapes_ok); outside it the fp32 CUDA-core kernels run
        self.tc = tc_envelope(shapes, p_list, math)
        if nhwc and not self.tc:
            raise RuntimeError("channels-last maps need the tensor-core path (C <= 256, P <= 1024, math != simt_f32)")
        self.plan_bytes = 0
        if self.tc:
            _lib.check(lib.pnce_plan_bytes(self.fwd_layers, self.n, ctypes.byref(nbytes)), "pnce_plan_bytes")
            self.plan_bytes = nbytes.value
        # bytes of feature maps: from _SIDE_STREAM_MIN_BYTES on, the id draw + sort go to a side stream, under whatever
        # the GPU is still busy with (below, the stream switch only costs host time)
        elem = 4 if dtype == torch.float32 else 2
        self.big = 2 * elem * sum(b * c * h * w for b, c, h, w in shapes)
        self.fwd_lock, self.bwd_lock = threading.Lock(), threading.Lock()


_SHAPE_PLANS = {}


def tc_envelope(shapes, p_list, math) -> bool:
    """The tensor-core kernels' envelope (csrc/pnce_api.cu tc_shapes_ok); outside it the fp32 CUDA-core kernels run."""
    return math != "simt_f32" and all(s[1] <= 256 and p <= 1024 for s, p in zip(shapes, p_list))


MB_MAX_KEYS = 65536      # keys (B * round_up(P, 128)) per layer of the minibatch-negatives kernel (include/pnce.h)


def mb_check(batch, channels, p_list, math, rows=False, world=1):
    """The envelope of minibatch negatives (``nce_includes_all_negatives_from_minibatch``): tensor-core math, C <= 256,
    P <= 1024 per image (P <= 256 on the row route) and B * round_up(P, 128) <= 65536 per layer.  Raises RuntimeError
    outside it: there is no other implementation of this mode to fall back to.  ``world``: global negatives over that
    many equal shards of ``batch`` images each -- the key bound applies to the global batch ``world * batch``."""
    if math == "simt_f32":
        raise RuntimeError("nce_includes_all_negatives_from_minibatch needs a tensor-core math mode (tc_bf16x3 or tc_bf16), "
                           "not simt_f32")
    pmax = 256 if rows else 1024
    for c, p in zip(channels, p_list):
        if c > 256 or p > pmax:
            raise RuntimeError(f"nce_includes_all_negatives_from_minibatch supports C <= 256 and P <= {pmax} per layer "
                               f"(got C={c}, P={p})")
        if world * batch * ((p + 127) // 128 * 128) > MB_MAX_KEYS:
            got = f"batch={batch}" if world == 1 else f"global batch={world * batch} ({world} ranks x {batch})"
            raise RuntimeError(f"nce_includes_all_negatives_from_minibatch supports at most {MB_MAX_KEYS} keys per layer "
                               f"(batch * round_up(P, 128)); got {got}, P={p}")


def _is_nhwc(t) -> bool:
    """(B, C, H, W) tensor whose storage is dense (B, H, W, C): torch.channels_last (and not also plain contiguous)."""
    return t.dim() == 4 and not t.is_contiguous() and t.is_contiguous(memory_format=torch.channels_last)


def _shape_plan(tgt, p_list, math, nhwc=False, mb=False, world=1) -> _ShapePlan:
    t0 = tgt[0]
    key = (t0.device.index, t0.dtype, math, nhwc, mb, world, tuple(p_list), *[t.shape for t in tgt])
    sp = _SHAPE_PLANS.get(key)
    if sp is None:
        if len(_SHAPE_PLANS) > 256:                  # a caller cycling through many shapes: do not grow without bound
            _SHAPE_PLANS.clear()
        sp = _SHAPE_PLANS[key] = _ShapePlan(t0.device, t0.dtype, [tuple(t.shape) for t in tgt], p_list, math, nhwc, mb,
                                            world)
    return sp


class _FlatIds:
    """The ids of every layer in ONE int64 buffer (what the library's draw fills); quacks like the list of per-layer
    tensors as far as the C-ABI glue is concerned (``ids[l].data_ptr()``) without creating the views."""
    __slots__ = ("flat", "ptrs")

    class _Ptr:
        __slots__ = ("p",)

        def __init__(self, p):
            self.p = p

        def data_ptr(self):
            return self.p

    def __init__(self, flat, p_list):
        self.flat = flat
        base, self.ptrs = flat.data_ptr(), []
        for p in p_list:
            self.ptrs.append(_FlatIds._Ptr(base))
            base += 8 * p

    def __getitem__(self, l):
        return self.ptrs[l]


class _Call:
    """One fused call: the shape plan plus what is not a differentiable input."""
    __slots__ = ("sp", "src", "ids", "temperature", "rng", "idplan", "group")

    def __init__(self, sp, src, ids, temperature, rng=None, idplan=None, group=None):
        self.sp, self.src, self.ids, self.temperature = sp, src, ids, float(temperature)
        self.rng = rng            # (philox seed, offset): the library draws the ids itself (pnce_fwd_draw)
        self.idplan = idplan      # k_prep's outputs when the id draw + sort already ran on the side stream
        self.group = group        # global negatives: the process group of sp.world ranks the keys are gathered over


def _layer_array(src, tgt, dtgt, ids):
    n = len(tgt)
    arr = (_lib.PnceLayer * n)()
    for l in range(n):
        b, c, h, w = tgt[l].shape
        arr[l].src = src[l].data_ptr() if src is not None else None
        arr[l].tgt = tgt[l].data_ptr()
        arr[l].dtgt = dtgt[l].data_ptr() if dtgt is not None else None
        arr[l].ids = ids[l].data_ptr()
        arr[l].C, arr[l].H, arr[l].W, arr[l].P = c, h, w, ids[l].numel()
    return arr


def _run_fwd(call: _Call, tgt_feats):
    """The forward launches of one fused call (id draw + sort | gather | logits, CE and the gradient rows):
    -> (workspace, out) with out[0] = loss, out[1 + l] = layer losses."""
    lib = _lib.load()
    sp = call.sp
    dev = sp.dev
    n = sp.n
    with _on_device(dev):
        ws = torch.empty(sp.ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty(1 + n, dtype=torch.float32, device=dev)
        slot, flag_ptr = _warn_queue(dev).acquire(sp.mb)      # both words are written by the kernels
        st = _stream_ptr(dev)
        src, ids = call.src, call.ids
        with sp.fwd_lock:
            layers = sp.fwd_layers
            for l in range(n):
                a = layers[l]
                a.src, a.tgt, a.ids = src[l].data_ptr(), tgt_feats[l].data_ptr(), ids[l].data_ptr()
            if sp.world > 1:
                rc = _run_fwd_global(lib, call, layers, ws, out, flag_ptr, st)
            elif sp.mb:
                philox = (ctypes.c_ulonglong * 2)(call.rng[0], call.rng[1]) if call.rng is not None else None
                pl = call.idplan
                rc = lib.pnce_mb_fwd(layers, n, sp.batch, sp.dtype_code, _lib.LAYOUT_NHWC if sp.nhwc else _lib.LAYOUT_NCHW,
                                     call.temperature, sp.math_code, ws.data_ptr(), sp.ws_bytes,
                                     pl.data_ptr() if pl is not None else None, pl.numel() if pl is not None else 0, philox,
                                     out.data_ptr(), flag_ptr or None, st)
            elif sp.nhwc:
                philox = (ctypes.c_ulonglong * 2)(call.rng[0], call.rng[1]) if call.rng is not None else None
                pl = call.idplan
                rc = lib.pnce_fwd_ex(layers, n, sp.batch, sp.dtype_code, _lib.LAYOUT_NHWC, call.temperature,
                                     sp.math_code, ws.data_ptr(), sp.ws_bytes, pl.data_ptr() if pl is not None else None,
                                     pl.numel() if pl is not None else 0, philox, out.data_ptr(), flag_ptr or None, st)
            elif call.rng is not None:
                rc = lib.pnce_fwd_draw(layers, n, sp.batch, sp.dtype_code, call.temperature, sp.math_code,
                                       ws.data_ptr(), sp.ws_bytes, call.rng[0], call.rng[1], out.data_ptr(),
                                       flag_ptr or None, st)
            elif call.idplan is None:
                rc = lib.pnce_fwd(layers, n, sp.batch, sp.dtype_code, call.temperature, sp.math_code,
                                  ws.data_ptr(), sp.ws_bytes, out.data_ptr(), flag_ptr or None, st)
            else:
                rc = lib.pnce_fwd_planned(layers, n, sp.batch, sp.dtype_code, call.temperature, sp.math_code,
                                          ws.data_ptr(), sp.ws_bytes, call.idplan.data_ptr(),
                                          call.idplan.numel(), out.data_ptr(), flag_ptr or None, st)
        if rc != 0:
            _lib.check(rc, "pnce_fwd")
    return ws, out


def _run_fwd_global(lib, call: _Call, layers, ws, out, flag_ptr, st) -> int:
    """Global negatives: this rank's keys into its slot of the workspace, the all-gather of the slots (the one
    collective of the mode; keys carry no gradient, so the backward is local), then the loss over every rank's keys."""
    from . import dp
    sp = call.sp
    rank = dist.get_rank(call.group)
    layout = _lib.LAYOUT_NHWC if sp.nhwc else _lib.LAYOUT_NCHW
    philox = (ctypes.c_ulonglong * 2)(call.rng[0], call.rng[1]) if call.rng is not None else None
    pl = call.idplan
    plp, pln = (pl.data_ptr(), pl.numel()) if pl is not None else (None, 0)
    rc = lib.pnce_mb_shard_keys(layers, sp.n, sp.batch, sp.dtype_code, layout, sp.world, rank, sp.math_code,
                                ws.data_ptr(), sp.ws_bytes, plp, pln, philox, st)
    if rc != 0:
        return rc
    dp.allgather_slots_(ws[sp.slot_offset:sp.slot_offset + sp.world * sp.slot_bytes], rank, call.group)
    return lib.pnce_mb_shard_loss(layers, sp.n, sp.batch, sp.dtype_code, layout, sp.world, rank, call.temperature,
                                  sp.math_code, ws.data_ptr(), sp.ws_bytes, plp, pln, out.data_ptr(), flag_ptr or None, st)


# ---- compressible memory for the dense gradients (csrc/comp_alloc.cuh) ---------------------------------------------
# d tgt_feat is written once per step by the HBM-bound dense kernel and is zero except for one sampled float in a few
# per cent of its lines: in memory the driver compresses between L2 and HBM the same kernel is ~11 % faster (and the
# generator's backward reads the zero lines ~40 % faster).  The gradient tensors of large calls therefore come from a
# torch.cuda.MemPool backed by the library's allocator; everything else about them is an ordinary torch tensor.
# PNCE_GRAD_COMPRESSION=0 (or set_gradient_compression(False)) keeps them in the default pool.
_GRAD_COMPRESSION = os.environ.get("PNCE_GRAD_COMPRESSION", "1") not in ("0", "")
_GRAD_COMPRESSION_MIN_BYTES = 192 << 20      # below this the pool switch costs more host time than the kernel gains
_GRAD_POOLS = {}                             # device index -> (allocator, MemPool) or None when unsupported


def set_gradient_compression(enabled: bool = True, min_bytes: Optional[int] = None):
    """Switch the compressible gradient pool on or off (default: on where the device supports it, for calls whose
    dense gradients total at least ``min_bytes``)."""
    global _GRAD_COMPRESSION, _GRAD_COMPRESSION_MIN_BYTES
    _GRAD_COMPRESSION = bool(enabled)
    if min_bytes is not None:
        _GRAD_COMPRESSION_MIN_BYTES = int(min_bytes)


def _grad_pool(dev):
    entry = _GRAD_POOLS.get(dev.index, False)
    if entry is False:
        entry = None
        try:
            if _lib.load().pnce_comp_supported(dev.index) == 1:
                from torch.cuda.memory import CUDAPluggableAllocator
                alloc = CUDAPluggableAllocator(_lib.LIB_PATH, "pnce_comp_alloc", "pnce_comp_free")
                entry = (alloc, torch.cuda.MemPool(alloc.allocator()))
        except Exception:                    # noqa: BLE001 - an older torch without MemPool: the default pool it is
            entry = None
        _GRAD_POOLS[dev.index] = entry
    return entry[1] if entry is not None else None


def gradient_is_compressed(t: torch.Tensor) -> bool:
    """True when ``t`` lives in a block of the compressible pool AND the driver granted compression for it."""
    return bool(t.is_cuda and _lib.load().pnce_comp_is_compressed(t.data_ptr()) == 1)


def _grad_pool_ctx(nbytes, dev):
    """Context in which the dense gradients of a call are allocated: the compressible pool when the call is large enough
    (and nothing is being captured into a CUDA graph), else nothing."""
    if _GRAD_COMPRESSION and nbytes >= _GRAD_COMPRESSION_MIN_BYTES and not torch.cuda.is_current_stream_capturing():
        pool = _grad_pool(dev)
        if pool is not None:
            return torch.cuda.use_mem_pool(pool, dev)
    return _NULL_CTX


def _empty_grads(tgt_like, dev):
    """One uninitialised gradient tensor per map (``empty_like``: same shape, dtype and memory layout).  Caller is on
    device ``dev``."""
    nbytes = 0
    for t in tgt_like:
        nbytes += t.numel() * t.element_size()
    with _grad_pool_ctx(nbytes, dev):
        return [torch.empty_like(t) for t in tgt_like]


def _run_bwd(call: _Call, ws, grad_out, tgt_like):
    """The backward launch: dense d loss / d tgt_feat of every layer, scaled by ``grad_out`` (device scalar or None = 1)."""
    lib = _lib.load()
    sp = call.sp
    dev = sp.dev
    g = grad_out
    if g is not None and (g.dtype != torch.float32 or g.device != dev or not g.is_contiguous()):
        g = g.detach().to(device=dev, dtype=torch.float32).contiguous()
    with _on_device(dev):
        grads = _empty_grads(tgt_like, dev)
        st = _stream_ptr(dev)
        ids = call.ids
        with sp.bwd_lock:
            layers = sp.bwd_layers
            for l in range(sp.n):
                layers[l].dtgt, layers[l].ids = grads[l].data_ptr(), ids[l].data_ptr()
            gp = g.data_ptr() if g is not None else None
            if sp.nhwc or sp.mb:
                pl = call.idplan
                rc = lib.pnce_bwd_ex(layers, sp.n, sp.batch, sp.dtype_code,
                                     _lib.LAYOUT_NHWC if sp.nhwc else _lib.LAYOUT_NCHW, sp.math_code,
                                     ws.data_ptr(), sp.ws_bytes, pl.data_ptr() if pl is not None else None,
                                     pl.numel() if pl is not None else 0, gp, st)
            elif call.idplan is None:
                rc = lib.pnce_bwd(layers, sp.n, sp.batch, sp.dtype_code, sp.math_code, ws.data_ptr(),
                                  sp.ws_bytes, gp, st)
            else:
                rc = lib.pnce_bwd_planned(layers, sp.n, sp.batch, sp.dtype_code, sp.math_code, ws.data_ptr(),
                                          sp.ws_bytes, call.idplan.data_ptr(), call.idplan.numel(), gp, st)
        if rc != 0:
            _lib.check(rc, "pnce_bwd")
    return grads


class _FusedPatchNCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, call: _Call, *tgt_feats):
        ws, out = _run_fwd(call, tgt_feats)
        # the workspace goes through save_for_backward: autograd then frees it with the graph, right after
        # backward() -- kept as a plain ctx attribute it lived as long as the loss tensor did, and a caller that
        # holds on to the loss across steps (loss = step()) made every step allocate a second 0.26 GB workspace
        ctx.save_for_backward(ws)
        ctx.call = call
        ctx.tgt_keep = tgt_feats          # shapes / dtypes of the gradients to allocate
        ctx.layer_losses = out[1:]
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        (ws,) = ctx.saved_tensors
        return (None, *_run_bwd(ctx.call, ws, grad_out, ctx.tgt_keep))


def _prepare_maps(src_feats, tgt_feats, math=None, patches=None):
    """The reference's argument handling (patchnce_cut.py:25-40) plus what the C ABI needs: CUDA tensors,
    (B, C, H, W), src/tgt of equal shape, contiguous NCHW.  Returns (src, tgt, len(src_feats), uniform); ``uniform``:
    every layer shares batch size, dtype, device and memory layout, so ONE C-ABI call covers them all (the reference
    treats each layer on its own, :36-38, so mixed lists are valid input there and take one call per layer here).

    Channels-last target maps (``torch.channels_last``: an extension, the reference's ``.view`` rejects them) are
    kept as they are when the layer fits the tensor-core kernels (``math``; ``patches`` = num_patches or the list of
    id counts) -- the gather then reads each patch as one contiguous row, and the gradient comes back channels-last;
    otherwise they are re-laid out to NCHW like any other non-contiguous input."""
    n_src = len(src_feats)
    n = min(n_src, len(tgt_feats))                   # the reference zips and silently truncates (:36) ...
    if n_src == 0:
        raise ZeroDivisionError("division by zero")  # ... but divides by len(src_feats) (:40)
    if n == 0:
        raise RuntimeError("no target feature maps")
    if n > _lib.MAX_LAYERS:
        raise RuntimeError(f"at most {_lib.MAX_LAYERS} nce layers per call")
    src, tgt = [], []
    t0 = tgt_feats[0]
    b0, dt0, dev0 = (t0.shape[0] if t0.dim() else -1), t0.dtype, t0.device
    uniform = True
    nh0 = None
    for l in range(n):
        s, t = src_feats[l], tgt_feats[l]
        if s.shape != t.shape or s.dtype != t.dtype or s.device != t.device or t.dim() != 4 or not t.is_cuda:
            # off the fast path: say what is wrong, or convert what may be converted
            _require_cuda(t, "tgt_feat")
            _require_cuda(s, "src_feat")
            if t.dim() != 4 or s.dim() != 4:
                raise ValueError("not enough values to unpack (expected 4): feature maps must be (B, C, H, W)")
            if s.shape != t.shape:
                raise RuntimeError(f"src/tgt feature shapes differ: {tuple(s.shape)} vs {tuple(t.shape)}")
            if s.device != t.device:
                raise RuntimeError(f"src/tgt features on different devices: {s.device} vs {t.device}")
            s = s.to(t.dtype)
        dt = t.dtype
        if dt is not dt0 or t.shape[0] != b0 or t.device != dev0:
            uniform = False
        if dt not in _DTYPES:
            raise RuntimeError(f"unsupported feature dtype {dt}")
        if s.requires_grad:
            s = s.detach()
        nh = False
        if not t.is_contiguous() and math is not None and _is_nhwc(t):
            hw = t.shape[2] * t.shape[3]
            pl = patch_count(patches, hw) if isinstance(patches, int) else int(patches[l].numel())
            nh = tc_envelope([t.shape], [pl], math)
        if nh0 is None:
            nh0 = nh
        elif nh != nh0:
            uniform = False
        if nh:
            src.append(s if _is_nhwc(s) else s.contiguous(memory_format=torch.channels_last))
            tgt.append(t)
        else:
            src.append(s if s.is_contiguous() else s.contiguous())
            tgt.append(t if t.is_contiguous() else t.contiguous())
    return src, tgt, n_src, uniform


def _negatives_group(mb, negatives_group):
    """-> (process group, world) of global negatives, or (None, 1): minibatch negatives on this rank's batch alone."""
    if negatives_group is None:
        return None, 1
    if not mb:
        raise ValueError("negatives_group needs nce_includes_all_negatives_from_minibatch=True")
    from . import dp
    group = dp.resolve_group(negatives_group)
    return (group, dist.get_world_size(group)) if group is not None else (None, 1)


def _mb_plan(tgt, p_list, math, mb, world):
    # B = 1 on one rank: minibatch negatives ARE the per-image loss -- the per-image kernels, bit for bit
    return _shape_plan(tgt, p_list, math, _is_nhwc(tgt[0]), mb and (tgt[0].shape[0] > 1 or world > 1), world)


def _fused_call(src, tgt, ids, temperature, math, rng=None, idplan=None, mb=False, group=None, world=1):
    sp = _mb_plan(tgt, [i.numel() for i in ids], math, mb, world)
    return _FusedPatchNCE.apply(_Call(sp, src, ids, temperature, rng, idplan, group), *tgt)


def fused_patchnce(src_feats, tgt_feats, ids_list, temperature=0.07, math: Optional[str] = None,
                   denom_layers: Optional[int] = None, nce_includes_all_negatives_from_minibatch: bool = False,
                   negatives_group=None):
    """All-layer PatchNCE on dense NCHW maps with given ids.  Returns the scalar loss tensor
    (fp32, on device, differentiable w.r.t. every ``tgt_feats[l]`` that requires grad).
    ``nce_includes_all_negatives_from_minibatch``, ``negatives_group``: see ``PatchNCELoss`` (every rank passes the
    same ids)."""
    mb = bool(nce_includes_all_negatives_from_minibatch)
    group, world = _negatives_group(mb, negatives_group)
    math = math or DEFAULT_MATH
    if len(ids_list) < min(len(src_feats), len(tgt_feats)):
        raise RuntimeError(f"{len(ids_list)} id tensors for {min(len(src_feats), len(tgt_feats))} layers")
    src, tgt, n_src, uniform = _prepare_maps(src_feats, tgt_feats, math, list(ids_list))
    n = len(tgt)
    ids = []
    for i in list(ids_list)[:n]:
        _require_cuda(i, "patch_ids")
        if i.dtype != torch.int64 or not i.is_contiguous():
            i = i.to(torch.int64).contiguous()
        if i.numel() > _lib.MAX_PATCHES:
            raise RuntimeError(f"num_patches > {_lib.MAX_PATCHES} is not supported")
        ids.append(i)
    denom = n_src if denom_layers is None else denom_layers
    if uniform:
        loss = _fused_call(src, tgt, ids, temperature, math, mb=mb, group=group, world=world)
    else:
        # layers of different batch size / dtype: one call per layer, summed like the reference's loop (:36-40)
        loss = sum(_fused_call([s], [t], [i], temperature, math, mb=mb, group=group, world=world)
                   for s, t, i in zip(src, tgt, ids)) / float(n)
    if denom != n:                       # zip truncation case: kernel divided by n, reference by len(src)
        loss = loss * (float(n) / float(denom))
    return loss


class PatchNCELoss(nn.Module):
    """Drop-in for ``PatchNCELoss`` of patchnce_cut.py:7-110 -- and, on 2-D inputs, the north-star
    ``PatchNCELoss(feat_q, feat_k)``.

    ``forward(src_feats, tgt_feats)`` with two lists of (B,C,H,W) maps follows the reference: one
    id draw per zipped layer, loss = sum over layers / len(src_feats).
    ``forward(feat_q, feat_k)`` with two (B*P, D) row tensors (rows grouped per image, already
    L2-normalised, e.g. from ``PatchSampleF``) returns that layer's mean diagonal CE; the number of
    images is ``feat_q.shape[0] // min(num_patches, rows)`` unless ``batch_size`` is given.

    ``nce_includes_all_negatives_from_minibatch=True`` is upstream CUT's switch of that name (``batch_dim_for_bmm = 1``;
    the reference's config declares it, configs/train_gan_cutpp.yaml:80): each query patch of a layer is contrasted with
    the patches of ALL images of the batch, not only its own image's.  Per layer the loss is the reference's
    (:42-110) on one group of B * P rows -- logits N x N with N = B * P, diagonal positives, +-50 clamp, mean CE over the
    N rows, the non-finite guard applied to the group -- computed on the tensor cores (k_loss_tc_mb) without the N x N
    logits ever reaching memory.  At B = 1 it is the per-image loss.  Under data parallelism the negatives are the
    rank's own shard, as upstream CUT under DDP, unless ``negatives_group`` is given (below).  Tensor-core math modes only; C <= 256, P <= 1024 (<= 256 on the row
    route) and B * round_up(P, 128) <= 65536 per layer, RuntimeError otherwise.

    ``negatives_group`` (with the flag only, ValueError otherwise): global negatives under data parallelism.  ``True``
    (the default process group) or a ``ProcessGroup`` of W ranks, each holding an equal shard of B_l images in rank
    order (``dp.shard_batch``) and drawing the same ids (one seed, or ``dp.broadcast_patch_ids``): every rank's query
    rows are contrasted with the keys of all W * B_l images, which are all-gathered without gradient in the forward.
    Each rank returns the mean over its own rows, so averaging gradients over the ranks (``dp.GradReducer``, DDP)
    reproduces one GPU on the global batch; a non-finite row or key anywhere zeroes the layer on every rank.  The
    envelope above applies to the global batch.  ``None`` (default), or a group of one rank: the rank's own batch.
    Maps route only: the row route raises RuntimeError."""

    def __init__(self, temperature: float = 0.07, num_patches: int = 256,
                 nce_layers: Sequence[int] = (0, 4, 8, 12, 16), math: Optional[str] = None,
                 nce_includes_all_negatives_from_minibatch: bool = False, negatives_group=None):
        super().__init__()
        if negatives_group is not None and not nce_includes_all_negatives_from_minibatch:
            raise ValueError("negatives_group needs nce_includes_all_negatives_from_minibatch=True")
        self.temperature = temperature
        self.num_patches = num_patches
        self.nce_layers = list(nce_layers)      # stored, never used -- as in the reference (:22)
        self.math = math
        self.nce_includes_all_negatives_from_minibatch = bool(nce_includes_all_negatives_from_minibatch)
        self.negatives_group = negatives_group
        self._last_ids = None

    @property
    def last_patch_ids(self) -> Optional[List[torch.Tensor]]:
        """The ids of the most recent ``forward(src_feats, tgt_feats)``: one int64 (P_l,) tensor per layer."""
        v = self._last_ids
        if isinstance(v, tuple):                 # (flat buffer the library drew into, patch counts): split on demand
            v = self.__dict__["_last_ids"] = list(v[0].split(v[1]))
        return v

    def forward(self, a, b, batch_size: Optional[int] = None):
        mb = self.nce_includes_all_negatives_from_minibatch
        rows = (isinstance(a, torch.Tensor) and a.dim() == 2) or (not isinstance(a, torch.Tensor) and len(a) > 0
                                                                   and a[0].dim() == 2)
        if rows and self.negatives_group is not None:
            raise RuntimeError("negatives_group covers the maps route (PatchNCELoss(src_feats, tgt_feats)); global "
                               "negatives on the row route (PatchNCELoss(feat_q, feat_k)) are out of scope")
        if isinstance(a, torch.Tensor) and a.dim() == 2:
            if mb:
                return rows_patchnce_multi([a], [b], self.temperature, self.num_patches, batch_size, self.math, True)
            return rows_patchnce(a, b, self.temperature, self.num_patches, batch_size, self.math)
        if not isinstance(a, torch.Tensor) and len(a) > 0 and a[0].dim() == 2:
            # two lists of (B*P_l, D_l) rows (what PatchSampleF returns): every layer in one call, mean over layers
            return rows_patchnce_multi(a, b, self.temperature, self.num_patches, batch_size, self.math, mb)
        call, tgt, scale = self._begin(a, b)
        if call is None:
            return tgt                               # mixed layers: the per-layer composition already ran
        loss = _FusedPatchNCE.apply(call, *tgt)
        return loss if scale is None else loss * scale

    def loss_and_grads(self, src_feats, tgt_feats, grad_output: Optional[torch.Tensor] = None):
        """``forward(src_feats, tgt_feats)`` and its complete backward in ONE call, without autograd: returns
        ``(loss, [d (grad_output * loss) / d tgt_feats[l]])`` -- same ids (one draw per layer, generator advanced
        like the reference's), same kernels, same values as ``loss = forward(...); loss.backward(grad_output)``.
        For training loops that drive the generator's backward themselves (``feat.backward(grad)``) and for
        small batches, where autograd's fixed cost per backward() (engine thread hand-off, the ones_like of the
        root gradient: ~100 us of host time) is more than the whole step's GPU time (DESIGN.md 4.5)."""
        call, tgt, scale = self._begin(src_feats, tgt_feats)
        if call is None:
            raise RuntimeError("loss_and_grads needs layers of one batch size, dtype and device")
        tgt = [t.detach() for t in tgt]
        ws, out = _run_fwd(call, tgt)
        g = grad_output
        if scale is not None:
            g = torch.full((), scale, device=out.device) if g is None else g.to(torch.float32) * scale
        grads = _run_bwd(call, ws, g, tgt)
        loss = out[0]
        return (loss if scale is None else loss * scale), grads

    def _begin(self, a, b):
        """Argument handling + the id draw of one ``forward``: -> (call, tgt, scale)."""
        math = self.math or DEFAULT_MATH
        src, tgt, n_src, uniform = _prepare_maps(a, b, math, int(self.num_patches))
        n = len(tgt)
        dev = tgt[0].device
        _warn_queue(dev).poll()
        mb = self.nce_includes_all_negatives_from_minibatch
        if not uniform:
            ids = draw_patch_ids_all(src, self.num_patches)                           # :60-63
            self.__dict__["_last_ids"] = ids
            return None, fused_patchnce(src, tgt, ids, self.temperature, math, denom_layers=n_src,
                                        nce_includes_all_negatives_from_minibatch=mb,
                                        negatives_group=self.negatives_group), None
        p_list = [patch_count(self.num_patches, t.shape[2] * t.shape[3]) for t in tgt]    # :60
        if max(p_list) > _lib.MAX_PATCHES:
            raise RuntimeError(f"num_patches > {_lib.MAX_PATCHES} is not supported")
        group, world = _negatives_group(mb, self.negatives_group)
        sp = _mb_plan(tgt, p_list, math, mb, world)
        rng = idplan = None
        if sp.tc and not torch.cuda.is_current_stream_capturing() and _philox_ready(dev):
            # the library draws the ids (bit for bit torch.randint's, :63) inside its id-sort launch: no randint
            # launches, and the generator is advanced by exactly what they would have consumed
            if sp.big < _SIDE_STREAM_MIN_BYTES:
                with _on_device(dev):
                    ids_all = torch.empty(sp.p_total, dtype=torch.int64, device=dev)
                rng = _philox_take(dev, n)
            else:
                # draw + sort on a high-priority side stream: they depend on nothing but the generator state, so they
                # run under whatever the caller's stream is still busy with (in a steady loop, the previous step's
                # dense kernel) instead of at the head of this step's critical path
                main, side = torch.cuda.current_stream(dev), _id_stream(dev)
                seed, off = _philox_take(dev, n)
                with torch.cuda.stream(side):
                    ids_all = torch.empty(sp.p_total, dtype=torch.int64, device=dev)
                    idplan = torch.empty(sp.plan_bytes, dtype=torch.uint8, device=dev)
                    with sp.fwd_lock:
                        layers = sp.fwd_layers
                        ptr = ids_all.data_ptr()
                        for l in range(n):
                            layers[l].ids = ptr
                            ptr += 8 * p_list[l]
                        _lib.check(_lib.load().pnce_plan_ids_draw(layers, n, seed, off, idplan.data_ptr(), sp.plan_bytes,
                                                                  side.cuda_stream), "pnce_plan_ids_draw")
                main.wait_stream(side)
                ids_all.record_stream(main)      # allocated on the side stream's pool, consumed on the caller's
                idplan.record_stream(main)
            ids = _FlatIds(ids_all, p_list)
            self.__dict__["_last_ids"] = (ids_all, p_list)       # nn.Module.__setattr__ costs 3 us; split lazily
        else:
            ids = draw_patch_ids_all(src, self.num_patches)                           # :60-63
            self.__dict__["_last_ids"] = ids
        # zip truncation: the kernel divides by n, the reference by len(src_feats) (:40)
        return (_Call(sp, src, ids, self.temperature, rng, idplan, group), tgt,
                (None if n_src == n else float(n) / float(n_src)))


def compute_patchnce_loss(generator, src_images, tgt_images, nce_layers, temperature=0.07,
                          num_patches=256, math: Optional[str] = None,
                          nce_includes_all_negatives_from_minibatch: bool = False, negatives_group=None):
    """Drop-in for ``compute_patchnce_loss`` -- patchnce_cut.py:113-149 (call site
    training/train_cutpp.py:285-292).  ``generator`` only needs ``get_feature_layers``.  After
    ``enable_encoder_feature_reuse(generator, nce_layers)`` the source features are the activations of the
    ``generator(src_images)`` call that produced ``tgt_images`` (feature_reuse.py), not a second pass.
    ``nce_includes_all_negatives_from_minibatch``, ``negatives_group``: see ``PatchNCELoss``."""
    nce_loss_fn = PatchNCELoss(temperature, num_patches, nce_layers, math=math,                       # :135
                               nce_includes_all_negatives_from_minibatch=nce_includes_all_negatives_from_minibatch,
                               negatives_group=negatives_group)
    from .feature_reuse import cached_source_features
    src_feats = cached_source_features(generator, src_images, nce_layers)  # maps of the generator(src) just run, if tapped
    if src_feats is None:
        with torch.no_grad():                                                          # :138-139
            src_feats = generator.get_feature_layers(src_images, nce_layers)
    src_feats = [f.detach() for f in src_feats]                                        # :142
    tgt_feats = generator.get_feature_layers(tgt_images, nce_layers)                   # :145
    return nce_loss_fn(src_feats, tgt_feats)                                           # :147


# ------------------------------------------------------------------------------------------------
# module split: PatchSampleF and the rows loss
# ------------------------------------------------------------------------------------------------
class _SampleFn(torch.autograd.Function):
    """Random-patch gather (+ L2 normalisation unless ``raw``) of one NCHW map; backward = dense
    scatter with duplicate ids accumulated.  ``raw=True`` feeds the netF head."""

    @staticmethod
    def forward(ctx, feat, ids, raw=False):
        lib = _lib.load()
        f = feat.detach().contiguous()
        b, c, h, w = f.shape
        p = ids.numel()
        dev = f.device
        with torch.cuda.device(dev):
            rows = torch.empty(b * p, c, dtype=torch.float32, device=dev)
            inv = None if raw else torch.empty(b * p, dtype=torch.float32, device=dev)
            _lib.check(lib.pnce_sample_fwd(f.data_ptr(), _DTYPES[f.dtype], b, c, h, w, ids.data_ptr(), p,
                                           rows.data_ptr(), None if raw else inv.data_ptr(),
                                           _stream_ptr(dev)), "pnce_sample_fwd")
        if raw:
            ctx.save_for_backward(ids)
        else:
            ctx.save_for_backward(ids, rows, inv)
        ctx.meta = (b, c, h, w, p, f.dtype, dev, raw)
        return rows

    @staticmethod
    def backward(ctx, drows):
        lib = _lib.load()
        b, c, h, w, p, dt, dev, raw = ctx.meta
        if raw:
            (ids,) = ctx.saved_tensors
            rows = inv = None
        else:
            ids, rows, inv = ctx.saved_tensors
        g = drows.detach().to(torch.float32).contiguous()
        nbytes = ctypes.c_size_t(0)
        _lib.check(lib.pnce_sample_bwd_workspace_bytes(b, c, h, w, p, ctypes.byref(nbytes)),
                   "pnce_sample_bwd_workspace_bytes")
        with torch.cuda.device(dev):
            ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
            dfeat = torch.empty(b, c, h, w, dtype=dt, device=dev)
            _lib.check(lib.pnce_sample_bwd(g.data_ptr(), None if raw else rows.data_ptr(),
                                           None if raw else inv.data_ptr(), _DTYPES[dt],
                                           b, c, h, w, ids.data_ptr(), p, ws.data_ptr(), nbytes.value,
                                           dfeat.data_ptr(), _stream_ptr(dev)), "pnce_sample_bwd")
        return dfeat, None, None


class _SampleAllFn(torch.autograd.Function):
    """``_SampleFn`` for every map of a ``PatchSampleF`` call at once: one gather launch forward, and in
    the backward one id prep, a normalise-backward launch per map and ONE dense launch for all maps
    (pnce_sample_multi_fwd / _bwd).  Inputs: raw flag, n, the n maps, the n id tensors."""

    @staticmethod
    def forward(ctx, raw, n, *args):
        lib = _lib.load()
        feats = [a.detach().contiguous() for a in args[:n]]
        ids = list(args[n:2 * n])
        dev = feats[0].device
        b = feats[0].shape[0]
        maps = (_lib.PnceSample * n)()
        rows, invs = [], []
        with _on_device(dev):
            for l, (f, i) in enumerate(zip(feats, ids)):
                _, c, h, w = f.shape
                p = i.numel()
                r = torch.empty(b * p, c, dtype=torch.float32, device=dev)
                v = None if raw else torch.empty(b * p, dtype=torch.float32, device=dev)
                rows.append(r)
                invs.append(v)
                maps[l].feat, maps[l].ids, maps[l].rows = f.data_ptr(), i.data_ptr(), r.data_ptr()
                maps[l].inv = None if raw else v.data_ptr()
                maps[l].C, maps[l].H, maps[l].W, maps[l].P = c, h, w, p
            _lib.check(lib.pnce_sample_multi_fwd(maps, n, b, _DTYPES[feats[0].dtype], _stream_ptr(dev)),
                       "pnce_sample_multi_fwd")
        ctx.meta = (raw, n, b, dev, feats[0].dtype, [tuple(f.shape) for f in feats])
        if raw:
            ctx.save_for_backward(*ids)
        else:
            ctx.save_for_backward(*ids, *rows, *invs)
        return tuple(rows)

    @staticmethod
    def backward(ctx, *drows):
        lib = _lib.load()
        raw, n, b, dev, dt, shapes = ctx.meta
        saved = ctx.saved_tensors
        ids = saved[:n]
        rows_s = None if raw else saved[n:2 * n]
        invs_s = None if raw else saved[2 * n:3 * n]
        maps = (_lib.PnceSample * n)()
        keep, dfeats = [], []
        with _on_device(dev):
            elem = 4 if dt is torch.float32 else 2
            with _grad_pool_ctx(sum(elem * sh[0] * sh[1] * sh[2] * sh[3] for sh in shapes), dev):
                dfeats = [torch.empty(sh, dtype=dt, device=dev) for sh in shapes]
            for l in range(n):
                _, c, h, w = shapes[l]
                p = ids[l].numel()
                g = drows[l]
                g = (torch.zeros(b * p, c, dtype=torch.float32, device=dev) if g is None
                     else g.detach().to(torch.float32).contiguous())
                d = dfeats[l]
                keep.append(g)
                maps[l].ids, maps[l].drows, maps[l].dfeat = ids[l].data_ptr(), g.data_ptr(), d.data_ptr()
                maps[l].rows = None if raw else rows_s[l].data_ptr()
                maps[l].inv = None if raw else invs_s[l].data_ptr()
                maps[l].C, maps[l].H, maps[l].W, maps[l].P = c, h, w, p
            nbytes = ctypes.c_size_t(0)
            _lib.check(lib.pnce_sample_multi_bwd_workspace_bytes(maps, n, b, ctypes.byref(nbytes)),
                       "pnce_sample_multi_bwd_workspace_bytes")
            ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
            _lib.check(lib.pnce_sample_multi_bwd(maps, n, b, _DTYPES[dt], ws.data_ptr(), nbytes.value,
                                                 _stream_ptr(dev)), "pnce_sample_multi_bwd")
        return (None, None, *dfeats, *([None] * n))


_NETF_STATUS = {}        # device index -> int32[1] the netF kernels raise on a protocol timeout (checked when polling)


def _netf_status(dev) -> torch.Tensor:
    t = _NETF_STATUS.get(dev.index)
    if t is None:
        t = _NETF_STATUS[dev.index] = torch.zeros(1, dtype=torch.int32, device=dev)
    return t


class _NetFFn(torch.autograd.Function):
    """``PatchSampleF(use_mlp=True).forward`` for every map at once, in libpnce: raw gather -> Linear(C_l, nc) -> ReLU ->
    Linear(nc, nc) -> L2 normalise on tcgen05 (``pnce_netf_fwd``: k_prep, k_wprep, k_gather_tc, 2 x k_gemm_tc_p), and its
    backward (``pnce_netf_bwd``: normalise backward + dY blob, dH, dX, k_wgrad_tc, k_wreduce, one dense launch).
    Inputs: nc, n, math, the n maps, the n id tensors, 4 n head parameters (w1, b1, w2, b2 per map)."""

    @staticmethod
    def forward(ctx, nc, n, math, *args):
        lib = _lib.load()
        nhwc = all(_is_nhwc(a) for a in args[:n])
        # grad mode is off in here: maps and parameters are used as they are (per-tensor detach / to / contiguous calls
        # were most of this function's host time)
        feats = [a if (nhwc or a.is_contiguous()) else a.contiguous() for a in args[:n]]
        ids = list(args[n:2 * n])
        params = [_f32c(a) for a in args[2 * n:]]
        dev = feats[0].device
        b = feats[0].shape[0]
        maps = (_lib.PnceSample * n)()
        heads = (_lib.PnceHead * n)()
        rows, invs = [], []
        key = [dev.index, b, nc, nhwc]
        with _on_device(dev):
            for l in range(n):
                f, i = feats[l], ids[l]
                _, c, h, w = f.shape
                p = i.numel()
                r = torch.empty(b * p, nc, dtype=torch.float32, device=dev)
                v = torch.empty(b * p, dtype=torch.float32, device=dev)
                rows.append(r)
                invs.append(v)
                m = maps[l]
                m.feat, m.ids, m.rows, m.inv = f.data_ptr(), i.data_ptr(), r.data_ptr(), v.data_ptr()
                m.C, m.H, m.W, m.P = c, h, w, p
                key += [c, h, w, p]
                hd = heads[l]
                hd.w1, hd.b1, hd.w2, hd.b2 = (params[4 * l].data_ptr(), params[4 * l + 1].data_ptr(),
                                              params[4 * l + 2].data_ptr(), params[4 * l + 3].data_ptr())
            key = tuple(key)
            ws_bytes = _NETF_WS_BYTES.get(key)
            if ws_bytes is None:
                nbytes = ctypes.c_size_t(0)
                _lib.check(lib.pnce_netf_workspace_bytes(maps, n, b, nc, ctypes.byref(nbytes)), "pnce_netf_workspace_bytes")
                if len(_NETF_WS_BYTES) > 256:
                    _NETF_WS_BYTES.clear()
                ws_bytes = _NETF_WS_BYTES[key] = nbytes.value
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            layout = _lib.LAYOUT_NHWC if nhwc else _lib.LAYOUT_NCHW
            _lib.check(lib.pnce_netf_fwd(maps, heads, n, b, _DTYPES[feats[0].dtype], layout, nc, _MATH[math], ws.data_ptr(),
                                         ws_bytes, _netf_status(dev).data_ptr(), _stream_ptr(dev)), "pnce_netf_fwd")
        ctx.meta = (nc, n, math, b, dev, layout, ws_bytes, [(tuple(f.shape), f.dtype) for f in feats],
                    [(a.shape, a.dtype) for a in args[2 * n:]])
        ctx.feat_like = feats                    # layout / dtype of the dense gradients (no data is read in the backward)
        ctx.save_for_backward(ws, *ids, *rows, *invs, *params)
        return tuple(rows)

    @staticmethod
    def backward(ctx, *drows):
        lib = _lib.load()
        nc, n, math, b, dev, layout, ws_bytes, fmeta, pmeta = ctx.meta
        saved = ctx.saved_tensors
        ws, ids, rows, invs, params = saved[0], saved[1:1 + n], saved[1 + n:1 + 2 * n], saved[1 + 2 * n:1 + 3 * n], saved[1 + 3 * n:]
        need_dense = any(ctx.needs_input_grad[3:3 + n])
        maps = (_lib.PnceSample * n)()
        heads = (_lib.PnceHead * n)()
        with _on_device(dev):
            keep = []
            dfeats = _empty_grads(ctx.feat_like, dev) if need_dense else [None] * n
            sizes = [p.numel() for p in params]
            flat = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
            ptr = flat.data_ptr()
            for l in range(n):
                (_, c, h, w), _dt = fmeta[l]
                p = ids[l].numel()
                g = drows[l]
                if g is None:
                    g = torch.zeros(b * p, nc, dtype=torch.float32, device=dev)
                elif g.dtype is not torch.float32 or not g.is_contiguous():
                    g = g.detach().to(torch.float32).contiguous()
                keep.append(g)
                d = dfeats[l]
                m = maps[l]
                m.ids, m.rows, m.inv, m.drows = ids[l].data_ptr(), rows[l].data_ptr(), invs[l].data_ptr(), g.data_ptr()
                m.dfeat = d.data_ptr() if d is not None else None
                m.C, m.H, m.W, m.P = c, h, w, p
                hd = heads[l]
                hd.w1, hd.b1, hd.w2, hd.b2 = (params[4 * l].data_ptr(), params[4 * l + 1].data_ptr(),
                                              params[4 * l + 2].data_ptr(), params[4 * l + 3].data_ptr())
                hd.dw1 = ptr; ptr += 4 * sizes[4 * l]
                hd.db1 = ptr; ptr += 4 * sizes[4 * l + 1]
                hd.dw2 = ptr; ptr += 4 * sizes[4 * l + 2]
                hd.db2 = ptr; ptr += 4 * sizes[4 * l + 3]
            _lib.check(lib.pnce_netf_bwd(maps, heads, n, b, _DTYPES[fmeta[0][1]], layout, nc, _MATH[math], ws.data_ptr(),
                                         ws_bytes, _netf_status(dev).data_ptr(), _stream_ptr(dev)), "pnce_netf_bwd")
        pgrads = [v.view(shape) if dt is torch.float32 else v.view(shape).to(dt)
                  for v, (shape, dt) in zip(torch.split_with_sizes(flat, sizes), pmeta)]
        return (None, None, None, *dfeats, *([None] * n), *pgrads)


_NETF_WS_BYTES = {}      # pnce_netf_workspace_bytes per (device, batch, nc, layout, map geometry, patch counts)


def netf_fused_supported(use_mlp, nc, feats, ids, math) -> bool:
    """The tcgen05 head kernels cover nc in {128, 256}, P <= 1024, C <= 256, maps of one batch size / dtype / device."""
    if not use_mlp or nc not in (128, 256) or math == "simt_f32" or not 0 < len(feats) <= _lib.MAX_LAYERS:
        return False
    f0 = feats[0]
    return all(f.dim() == 4 and f.shape[1] <= 256 and i.numel() <= 1024 and f.shape[0] == f0.shape[0] and f.dtype == f0.dtype
               and f.device == f0.device and f.dtype in _DTYPES for f, i in zip(feats, ids))


_ROWS_WS_BYTES = {}      # (batch, P, D) -> pnce_rows_loss_workspace_bytes, queried once per shape


class _RowsLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, batch, p, temperature, math):
        lib = _lib.load()
        qq = q.detach().to(torch.float32).contiguous()
        kk = k.detach().to(torch.float32).contiguous()
        d = qq.shape[1]
        dev = qq.device
        key = (batch, p, d)
        ws_bytes = _ROWS_WS_BYTES.get(key)
        if ws_bytes is None:
            nbytes = ctypes.c_size_t(0)
            _lib.check(lib.pnce_rows_loss_workspace_bytes(batch, p, d, ctypes.byref(nbytes)),
                       "pnce_rows_loss_workspace_bytes")
            ws_bytes = _ROWS_WS_BYTES[key] = nbytes.value
        nbytes = ctypes.c_size_t(ws_bytes)
        with _on_device(dev):
            ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
            out = torch.empty(2, dtype=torch.float32, device=dev)
            wq = _warn_queue(dev)
            slot, flag_ptr = wq.acquire()
            dq = torch.empty_like(qq)
            _lib.check(lib.pnce_rows_loss_fwd_bwd(qq.data_ptr(), kk.data_ptr(), batch, p, d, temperature,
                                                  _MATH[math], ws.data_ptr(), nbytes.value, out.data_ptr(),
                                                  flag_ptr or None, dq.data_ptr(), None, _stream_ptr(dev)),
                       "pnce_rows_loss_fwd_bwd")
        ctx.save_for_backward(dq)
        ctx.q_dtype = q.dtype
        return out.narrow(0, 0, 1).reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        (dq,) = ctx.saved_tensors
        return (dq * grad_out).to(ctx.q_dtype), None, None, None, None, None


class _RowsLossMultiFn(torch.autograd.Function):
    """``mean_l PatchNCELoss(feat_q[l], feat_k[l])`` for every layer of a ``PatchSampleF`` output in ONE call of the
    library (pnce_rows_loss_multi_fwd_bwd: one pack launch, one tcgen05 loss launch).  Inputs: batch, temperature, math,
    n, mb (minibatch negatives: pnce_rows_mb_fwd_bwd), the n query row tensors, the n (detached) key row tensors."""

    @staticmethod
    def forward(ctx, batch, temperature, math, n, mb, *args):
        lib = _lib.load()
        qs = [_f32c(a) for a in args[:n]]
        ks = [_f32c(a) for a in args[n:]]
        dev = qs[0].device
        rows = (_lib.PnceRows * n)()
        key = ["mb" if mb else "multi", batch]
        with _on_device(dev):
            dqs = [torch.empty_like(q) for q in qs]
            for l in range(n):
                r = rows[l]
                r.q, r.k, r.dq = qs[l].data_ptr(), ks[l].data_ptr(), dqs[l].data_ptr()
                r.P, r.D = qs[l].shape[0] // batch, qs[l].shape[1]
                key += [r.P, r.D]
            key = tuple(key)
            ws_bytes = _ROWS_WS_BYTES.get(key)
            if ws_bytes is None:
                nbytes = ctypes.c_size_t(0)
                wsq = lib.pnce_rows_mb_workspace_bytes if mb else lib.pnce_rows_loss_multi_workspace_bytes
                _lib.check(wsq(rows, n, batch, ctypes.byref(nbytes)), "rows workspace query")
                ws_bytes = _ROWS_WS_BYTES[key] = nbytes.value
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            out = torch.empty(1 + n, dtype=torch.float32, device=dev)
            slot, flag_ptr = _warn_queue(dev).acquire(mb)
            fn = lib.pnce_rows_mb_fwd_bwd if mb else lib.pnce_rows_loss_multi_fwd_bwd
            _lib.check(fn(rows, n, batch, temperature, _MATH[math], ws.data_ptr(), ws_bytes, out.data_ptr(),
                          flag_ptr or None, _stream_ptr(dev)), "pnce_rows_mb_fwd_bwd" if mb else "pnce_rows_loss_multi_fwd_bwd")
        ctx.save_for_backward(*dqs)
        ctx.q_dtypes = [a.dtype for a in args[:n]]
        ctx.layer_losses = out[1:]
        return out.narrow(0, 0, 1).reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        dqs = torch._foreach_mul(list(ctx.saved_tensors), grad_out)            # one launch for every layer
        dqs = [d if d.dtype is dt else d.to(dt) for d, dt in zip(dqs, ctx.q_dtypes)]
        return (None, None, None, None, None, *dqs, *([None] * len(dqs)))


def rows_patchnce_multi(feat_q, feat_k, temperature=0.07, num_patches=256, batch_size=None, math=None, mb=False):
    """``mean_l PatchNCELoss(feat_q[l], feat_k[l])`` over two LISTS of row tensors (one (B*P_l, D_l) pair per layer, as
    ``PatchSampleF`` returns them) -- upstream CUT's ``for f_q, f_k in zip(feat_q, feat_k): total += crit(f_q, f_k)``
    followed by ``/ n_layers``, as one call of the library when every layer fits the tensor-core kernel (P, D <= 256);
    other shapes take the per-layer calls.  ``mb``: minibatch negatives (``PatchNCELoss``), one library call
    (pnce_rows_mb_fwd_bwd) for every layer."""
    feat_q, feat_k = list(feat_q), list(feat_k)
    n = len(feat_q)
    if n == 0 or n != len(feat_k):
        raise RuntimeError("feat_q and feat_k must be two lists of the same, non-zero length")
    math = math or DEFAULT_MATH
    batches = []
    for q, k in zip(feat_q, feat_k):
        _require_cuda(q, "feat_q")
        _require_cuda(k, "feat_k")
        if q.shape != k.shape or q.dim() != 2:
            raise RuntimeError("feat_q and feat_k must both be (B*P, D)")
        rows = q.shape[0]
        if batch_size is None:
            p = min(int(num_patches), rows)
            if rows % p:
                raise RuntimeError(f"{rows} rows are not a multiple of num_patches={p}; pass batch_size")
            batches.append(rows // p)
        else:
            if rows % batch_size:
                raise RuntimeError(f"{rows} rows are not a multiple of batch_size={batch_size}")
            batches.append(int(batch_size))
    b0, dev = batches[0], feat_q[0].device
    if mb and b0 > 1:
        if any(b != b0 for b in batches) or any(q.device != dev for q in feat_q) or n > _lib.MAX_LAYERS:
            raise RuntimeError("nce_includes_all_negatives_from_minibatch on rows needs layers of one batch size and "
                               f"device, at most {_lib.MAX_LAYERS} of them")
        mb_check(b0, [q.shape[1] for q in feat_q], [q.shape[0] // b0 for q in feat_q], math, rows=True)
        ks = [k.detach() if k.requires_grad else k for k in feat_k]      # upstream CUT and the reference (:142) detach k
        return _RowsLossMultiFn.apply(b0, float(temperature), math, n, True, *feat_q, *ks)
    fused = (math != "simt_f32" and n <= _lib.MAX_LAYERS and all(b == b0 for b in batches)
             and all(q.device == dev and q.shape[0] // b0 <= 256 and q.shape[1] <= 256 for q in feat_q))
    if not fused:
        total = None
        for q, k, b in zip(feat_q, feat_k, batches):
            l = rows_patchnce(q, k, temperature, num_patches, b, math)
            total = l if total is None else total + l
        return total / n
    ks = [k.detach() if k.requires_grad else k for k in feat_k]          # upstream CUT and the reference (:142) detach k
    return _RowsLossMultiFn.apply(b0, float(temperature), math, n, False, *feat_q, *ks)


def rows_patchnce(feat_q, feat_k, temperature=0.07, num_patches=256, batch_size=None, math=None):
    """PatchNCELoss(feat_q, feat_k): rows (B*P, D), grouped per image, L2-normalised."""
    _require_cuda(feat_q, "feat_q")
    _require_cuda(feat_k, "feat_k")
    if feat_q.shape != feat_k.shape or feat_q.dim() != 2:
        raise RuntimeError("feat_q and feat_k must both be (B*P, D)")
    if feat_k.requires_grad:
        feat_k = feat_k.detach()          # upstream CUT and the reference (:142) detach k
    rows = feat_q.shape[0]
    if batch_size is None:
        p = min(int(num_patches), rows)
        if rows % p:
            raise RuntimeError(f"{rows} rows are not a multiple of num_patches={p}; pass batch_size")
        batch_size = rows // p
    p = rows // batch_size
    return _RowsLossFn.apply(feat_q, feat_k, batch_size, p, float(temperature), math or DEFAULT_MATH)


class PatchSampleF(nn.Module):
    """North-star ``PatchSampleF.forward(feats, num_patches, patch_ids)`` (SURVEY.md section 8 row
    a13): per-layer random-patch gather from NCHW maps + L2 normalisation, ids drawn like the
    reference (:60-63) when ``patch_ids`` is None.  Returns ``(list[(B*P_l, D_l)], list[(P_l,)])``.

    ``use_mlp=True`` adds the netF head Linear(C_l, nc) -> ReLU -> Linear(nc, nc) before the
    normalisation (created lazily per layer on first use, like upstream CUT's ``create_mlp``)."""

    def __init__(self, use_mlp: bool = False, nc: int = 256, init_gain: float = 0.02, math: Optional[str] = None):
        super().__init__()
        self.use_mlp = use_mlp
        self.nc = nc
        self.init_gain = init_gain
        self.mlp_init = False
        self.math = math                         # contraction engine of the fused head (None: DEFAULT_MATH)

    def create_mlp(self, feats):
        for mlp_id, feat in enumerate(feats):
            input_nc = feat.shape[1]
            mlp = nn.Sequential(nn.Linear(input_nc, self.nc), nn.ReLU(), nn.Linear(self.nc, self.nc))
            for m in mlp:
                if isinstance(m, nn.Linear):
                    nn.init.normal_(m.weight, 0.0, self.init_gain)
                    nn.init.zeros_(m.bias)
            setattr(self, f"mlp_{mlp_id}", mlp.to(feat.device))
        self.mlp_init = True

    def forward(self, feats, num_patches: int = 256, patch_ids=None):
        return_feats, return_ids = [], []
        if self.use_mlp and not self.mlp_init:
            self.create_mlp(feats)
        feats = list(feats)
        for feat in feats:
            _require_cuda(feat, "feat")
            if feat.dim() != 4:
                raise ValueError("feature maps must be (B, C, H, W)")
        if patch_ids is not None:
            return_ids = [patch_ids[k].to(device=f.device, dtype=torch.int64).contiguous() for k, f in enumerate(feats)]
        else:
            return_ids = draw_ids(feats, num_patches)
        math = self.math or DEFAULT_MATH
        if netf_fused_supported(self.use_mlp, self.nc, feats, return_ids, math):
            # the whole head in libpnce, on the tensor cores: gather -> Linear -> ReLU -> Linear -> normalise (and, through
            # autograd, d feat and the weight gradients); other shapes take the composition below (gather in libpnce,
            # the two Linear layers in ATen)
            params = _head_params(self, len(feats))
            return list(_NetFFn.apply(self.nc, len(feats), math, *feats, *return_ids, *params)), return_ids
        same = all(f.shape[0] == feats[0].shape[0] and f.dtype == feats[0].dtype and f.device == feats[0].device
                   for f in feats)
        if same and 0 < len(feats) <= _lib.MAX_LAYERS and feats[0].dtype in _DTYPES:
            # every map in one gather launch (and one dense launch in the backward)
            raw_rows = _SampleAllFn.apply(self.use_mlp, len(feats), *feats, *return_ids)
        else:
            raw_rows = [_SampleFn.apply(f, i, self.use_mlp) for f, i in zip(feats, return_ids)]
        for feat_id, rows in enumerate(raw_rows):
            if self.use_mlp:
                # gather (libpnce) -> Linear-ReLU-Linear -> x / max(||x||, 1e-6)
                mlp = getattr(self, f"mlp_{feat_id}")
                rows = torch.nn.functional.normalize(mlp(rows), dim=1, eps=NORM_EPS)
            return_feats.append(rows)
        return return_feats, return_ids


class _HeadCall:
    """What the two fused head calls need that is not a differentiable input."""
    __slots__ = ("src_feats", "ids_list", "temperature", "math", "dp_group", "mb", "group", "world")

    def __init__(self, src_feats, ids_list, temperature, math, dp_group=None, mb=False, group=None, world=1):
        self.src_feats, self.ids_list, self.temperature, self.math = src_feats, ids_list, float(temperature), math
        self.dp_group = dp_group      # process group whose ranks average the head gradients (None: single process)
        self.mb = mb                  # minibatch negatives (pnce_head_mb_fwd; the per-image call at B = 1)
        self.group = group            # global negatives: the process group of `world` ranks the keys are gathered over
        self.world = world            # > 1: pnce_head_mb_shard_*; 1: the rank's own batch


def _head_fwd(plan, nc, tgt, params):
    """pnce_head_fwd_ex (pnce_head_mb_fwd with minibatch negatives, pnce_head_mb_shard_* with global negatives) on one
    set of maps and head parameters -> (workspace, out, state for _head_bwd)."""
    lib = _lib.load()
    n = len(tgt)
    src, ids = plan.src_feats, plan.ids_list
    dev = tgt[0].device
    batch = tgt[0].shape[0]
    dtype = _DTYPES[tgt[0].dtype]
    layers = _layer_array(src, tgt, None, ids)
    heads = (_lib.PnceHead * n)()
    for l in range(n):
        h = heads[l]
        h.w1, h.b1, h.w2, h.b2 = (params[4 * l].data_ptr(), params[4 * l + 1].data_ptr(),
                                  params[4 * l + 2].data_ptr(), params[4 * l + 3].data_ptr())
    layout = _lib.LAYOUT_NHWC if _is_nhwc(tgt[0]) else _lib.LAYOUT_NCHW      # _prepare_maps made the layers uniform
    world = plan.world
    # B = 1 on one rank: minibatch negatives ARE the per-image loss -- the per-image call, bit for bit.  Under global
    # negatives the test is on the GLOBAL batch: a shard of one image still has world - 1 images of negatives elsewhere.
    mb = plan.mb and (batch > 1 or world > 1)
    key = (dev.index, dtype, layout, nc, mb, tuple(t.shape for t in tgt), tuple(layers[l].P for l in range(n)), world)
    ws_bytes = _HEAD_WS_BYTES.get(key)
    if ws_bytes is None:
        if len(_HEAD_WS_BYTES) > 256:       # a caller cycling through many shapes: do not grow without bound
            _HEAD_WS_BYTES.clear()
            _HEAD_SLOTS.clear()
        nbytes = ctypes.c_size_t(0)
        if world > 1:
            so, sb = ctypes.c_size_t(0), ctypes.c_size_t(0)
            _lib.check(lib.pnce_head_mb_shard_workspace_bytes(layers, n, batch, world, nc, ctypes.byref(nbytes),
                                                              ctypes.byref(so), ctypes.byref(sb)),
                       "pnce_head_mb_shard_workspace_bytes")
            _HEAD_SLOTS[key] = (so.value, sb.value)
        else:
            query = lib.pnce_head_mb_workspace_bytes if mb else lib.pnce_head_workspace_bytes
            _lib.check(query(layers, n, batch, nc, ctypes.byref(nbytes)), "pnce_head_workspace_bytes")
        ws_bytes = _HEAD_WS_BYTES[key] = nbytes.value
    with _on_device(dev):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty(1 + n, dtype=torch.float32, device=dev)
        wq = _warn_queue(dev)
        slot, flag_ptr = wq.acquire(plan.mb)
        if world > 1:
            _head_fwd_global(lib, plan, nc, key, layers, heads, batch, dtype, layout, ws, ws_bytes, out, flag_ptr or None,
                             _stream_ptr(dev))
        else:
            fwd = lib.pnce_head_mb_fwd if mb else lib.pnce_head_fwd_ex
            _lib.check(fwd(layers, heads, n, batch, dtype, layout, nc, plan.temperature, _MATH[plan.math],
                           ws.data_ptr(), ws_bytes, out.data_ptr(), flag_ptr or None, _stream_ptr(dev)), "pnce_head_fwd")
    return ws, out, (ws_bytes, layout, dev, batch, dtype, heads)


def _head_fwd_global(lib, plan, nc, key, layers, heads, batch, dtype, layout, ws, ws_bytes, out, flag_ptr, st):
    """Global negatives: this rank's head output up to its keys, which go into its slot of the workspace; the all-gather
    of the slots (the one collective of the mode; keys carry no gradient, so the backward is local); then the loss over
    every rank's keys."""
    from . import dp
    n, world, math = len(layers), plan.world, _MATH[plan.math]
    rank = dist.get_rank(plan.group)
    so, sb = _HEAD_SLOTS[key]
    _lib.check(lib.pnce_head_mb_shard_keys(layers, heads, n, batch, dtype, layout, nc, world, rank, math, ws.data_ptr(),
                                           ws_bytes, flag_ptr, st), "pnce_head_mb_shard_keys")
    dp.allgather_slots_(ws[so:so + world * sb], rank, plan.group)
    _lib.check(lib.pnce_head_mb_shard_loss(layers, heads, n, batch, dtype, layout, nc, world, rank, plan.temperature,
                                           math, ws.data_ptr(), ws_bytes, out.data_ptr(), flag_ptr, st),
               "pnce_head_mb_shard_loss")


def _head_bwd(plan, nc, tgt, params, ws, state, g, flat=None):
    """pnce_head_bwd_ex: dense d tgt_feat per layer + every head gradient in ONE flat fp32 buffer (so that the
    data-parallel all-reduce needs no packing) -> (grads, flat, sizes).  ``g``: fp32 scalar tensor on the device."""
    lib = _lib.load()
    ws_bytes, layout, dev, batch, dtype, heads = state
    n = len(tgt)
    group = plan.dp_group
    with _on_device(dev):
        grads = _empty_grads(tgt, dev)
        sizes = [p.numel() for p in params]
        if flat is None:
            flat = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
        layers = _layer_array(plan.src_feats, tgt, grads, plan.ids_list)
        ptr, k = flat.data_ptr(), 0
        for l in range(n):                                   # the weight pointers are those of the forward call
            h = heads[l]
            h.dw1 = ptr; ptr += 4 * sizes[k]
            h.db1 = ptr; ptr += 4 * sizes[k + 1]
            h.dw2 = ptr; ptr += 4 * sizes[k + 2]
            h.db2 = ptr; ptr += 4 * sizes[k + 3]
            k += 4
        tail = (nc, _MATH[plan.math], ws.data_ptr(), ws_bytes, g.data_ptr(), _stream_ptr(dev))
        head = (layers, heads, n, batch, dtype, layout)
        if group is None:
            _lib.check(lib.pnce_head_bwd_ex(*head, 3, *tail), "pnce_head_bwd")
        else:
            # data parallel: head gradients first, their all-reduce on a side stream UNDER the dense kernel
            from . import dp
            _lib.check(lib.pnce_head_bwd_ex(*head, 1, *tail), "pnce_head_bwd_params")
            main = torch.cuda.current_stream(dev)
            side = dp.comm_stream(dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                dp.allreduce_flat_(flat, group, average=True)
            flat.record_stream(side)
            _lib.check(lib.pnce_head_bwd_ex(*head, 2, *tail), "pnce_head_bwd_dense")
            main.wait_stream(side)
    return grads, flat, sizes


def _f32c(a):
    return a if (a.dtype is torch.float32 and a.is_contiguous()) else a.detach().to(torch.float32).contiguous()


class _FusedHeadPatchNCE(torch.autograd.Function):
    """All layers of the head path through the C ABI: pnce_head_fwd (prep, weight blobs, gather,
    2 GEMM launches, fused logits/CE/dY) and pnce_head_bwd (dH, dX, weight gradients, dense d tgt).
    Inputs: plan, L target maps, then 4 L head parameters (w1, b1, w2, b2 per layer)."""

    @staticmethod
    def forward(ctx, plan, nc, *args):
        n = len(plan.ids_list)
        # inside Function.forward grad mode is off: the arguments are used as they are (no detach / view per tensor --
        # with 4 parameters per layer those calls were a third of the step's host time at small batches, DESIGN.md 4.5)
        tgt = list(args[:n])
        params = [_f32c(a) for a in args[n:]]
        ws, out, state = _head_fwd(plan, nc, tgt, params)
        ctx.save_for_backward(ws)            # freed with the graph, right after backward() (see _FusedPatchNCE)
        ctx.plan, ctx.nc, ctx.state = plan, nc, state
        ctx.tgt_keep, ctx.params = tgt, params
        ctx.param_meta = [(a.shape, a.dtype) for a in args[n:]]
        ctx.layer_losses = out[1:]
        return out.narrow(0, 0, 1).reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        dev = ctx.state[2]
        g = grad_out
        if g.dtype is not torch.float32 or g.device != dev or not g.is_contiguous():
            g = g.detach().to(device=dev, dtype=torch.float32).contiguous()
        (ws,) = ctx.saved_tensors
        grads, flat, sizes = _head_bwd(ctx.plan, ctx.nc, ctx.tgt_keep, ctx.params, ws, ctx.state, g)
        pgrads = [v.view(shape) if dt is torch.float32 else v.view(shape).to(dt)
                  for v, (shape, dt) in zip(torch.split_with_sizes(flat, sizes), ctx.param_meta)]
        return (None, None, *grads, *pgrads)


_HEAD_WS_BYTES = {}      # pnce_head_workspace_bytes per (device, dtype, layout, nc, mb, map shapes, patch counts, world)
_HEAD_SLOTS = {}         # global negatives: (slot offset, slot bytes) per key of _HEAD_WS_BYTES


def _head_params(netF, n):
    """w1, b1, w2, b2 of mlp_0 .. mlp_{n-1}, read straight from the module dictionaries (nn.Sequential.__getitem__
    and Module.__getattr__ cost ~50 us per step for five layers: more than the GPU needs for a B = 1 step)."""
    params = []
    mods = netF._modules
    for l in range(n):
        seq = mods[f"mlp_{l}"]._modules
        p0, p2 = seq["0"]._parameters, seq["2"]._parameters
        params += [p0["weight"], p0["bias"], p2["weight"], p2["bias"]]
    return params


def fused_head_supported(netF: "PatchSampleF", feats, num_patches) -> bool:
    """The tcgen05 head kernels cover nc in {128, 256}, P <= 1024 and C <= 256 (every CUT layer up to 512^2, P = 1024)."""
    if not netF.use_mlp or netF.nc not in (128, 256):
        return False
    return all(f.shape[1] <= 256 and patch_count(num_patches, f.shape[2] * f.shape[3]) <= 1024 for f in feats)


def patchnce_with_head(netF: "PatchSampleF", src_feats, tgt_feats, temperature=0.07, num_patches=256,
                       patch_ids=None, math: Optional[str] = None, fused: Optional[bool] = None,
                       dp_group=None):
    """North-star composition (SURVEY.md section 8 row a13):
    ``feat_k, ids = netF(src_feats, num_patches, patch_ids)`` (no grad into k, as upstream CUT and the
    reference's ``detach`` :142), ``feat_q, _ = netF(tgt_feats, num_patches, ids)``, then
    ``mean_l PatchNCELoss(feat_q_l, feat_k_l)``.  Returns ``(loss, ids)``.

    ``fused`` (default: whenever the shapes allow) runs the whole thing -- gather, both Linear layers,
    normalisation, logits, CE and the complete backward including the head gradients -- in the
    tcgen05 kernels of libpnce; otherwise the module-split composition is used (libpnce gather /
    scatter / rows loss around ATen's Linear).

    ``dp_group`` (fused path; ``True`` = the default process group): data-parallel training with the batch
    sharded over the ranks -- the head gradients that come out of ``backward`` are already AVERAGED over
    the group: one flat all-reduce, started on a side stream as soon as the weight-gradient kernels are
    done, so it runs under the HBM-bound dense-gradient kernel (SURVEY.md section 8e).  Do not call
    ``allreduce_head_grads`` as well.

    Per-image negatives only.  For minibatch negatives (upstream CUT's ``nce_includes_all_negatives_from_minibatch``)
    call ``patchnce_with_head_minibatch``, the same fused chain with every image's keys as negatives."""
    if fused is None:
        fused = fused_head_supported(netF, tgt_feats, num_patches) and (math or DEFAULT_MATH) != "simt_f32"
    if not fused:
        with torch.no_grad():
            feat_k, ids = netF(src_feats, num_patches, patch_ids)
        feat_q, _ = netF(tgt_feats, num_patches, ids)
        batch = tgt_feats[0].shape[0]
        total = None
        for q, k in zip(feat_q, feat_k):
            l = rows_patchnce(q, k, temperature, num_patches, batch, math)
            total = l if total is None else total + l
        return total / len(feat_q), ids
    plan, tgt, params, ids = _head_begin(netF, src_feats, tgt_feats, temperature, num_patches, patch_ids, math, dp_group)
    loss = _FusedHeadPatchNCE.apply(plan, netF.nc, *tgt, *params)
    return loss, ids


def _head_begin(netF, src_feats, tgt_feats, temperature, num_patches, patch_ids, math, dp_group, mb=False,
                negatives_group=None):
    """Argument handling + id draw of one fused head call -> (plan, tgt maps, head parameters, ids).
    ``mb``: minibatch negatives -- the envelope (mb_check) is checked before anything touches the device.
    ``negatives_group`` (with ``mb``): global negatives -- the envelope applies to the global batch, and is checked
    before any collective as well."""
    if not fused_head_supported(netF, tgt_feats, num_patches):
        raise RuntimeError("fused head: nc must be 128 or 256, num_patches <= 1024 and C <= 256")
    group, world = _negatives_group(mb, negatives_group)
    if mb:
        p_list = ([int(i.numel()) for i in patch_ids] if patch_ids is not None else
                  [patch_count(num_patches, f.shape[2] * f.shape[3]) for f in tgt_feats])
        mb_check(tgt_feats[0].shape[0], [f.shape[1] for f in tgt_feats], p_list, math or DEFAULT_MATH, world=world)
    if not netF.mlp_init:
        netF.create_mlp(tgt_feats)
    src, tgt, _, uniform = _prepare_maps(src_feats, tgt_feats, math or DEFAULT_MATH, int(num_patches))
    if not uniform:
        raise RuntimeError("fused head: every layer must share batch size, dtype, device and layout (use fused=False)")
    if patch_ids is None:
        ids = draw_ids(tgt, num_patches)
    else:
        ids = [i.to(device=t.device, dtype=torch.int64).contiguous() for i, t in zip(patch_ids, tgt)]
    params = _head_params(netF, len(tgt))
    if dp_group is not None:
        from . import dp
        dp_group = dp.resolve_group(dp_group)          # None when not initialised or world size 1
    plan = _HeadCall(src, ids, temperature, math or DEFAULT_MATH, dp_group, mb, group, world)
    _warn_queue(tgt[0].device).poll()
    return plan, tgt, params, ids


def patchnce_with_head_minibatch(netF: "PatchSampleF", src_feats, tgt_feats, temperature=0.07, num_patches=256,
                                 patch_ids=None, math: Optional[str] = None, dp_group=None):
    """``patchnce_with_head`` (fused path) with minibatch negatives -- upstream CUT's
    ``nce_includes_all_negatives_from_minibatch`` on the head's output.  Returns ``(loss, ids)``.

    Per layer, with the ids shared by the batch and N = B * P rows in image-major order:
    ``q = normalize(netF(raw tgt patches))``, ``k = normalize(netF(raw src patches)).detach()``,
    ``Z = clamp(q k^T / tau, -50, 50)`` (N x N), loss_l = mean over the N rows of CE(Z_i, i); the total is the mean over
    the layers.  A non-finite layer contributes 0 and zero gradients (one warning per guarded layer); the head learns
    through q only.  The whole chain -- gather, both Linear layers, normalisation, the N x N logits (which never reach
    memory: k_loss_tc_mb), CE and the complete backward including the head gradients -- runs in the tcgen05 kernels of
    libpnce.  At B = 1 it is ``patchnce_with_head``, bit for bit.  Same ids from the same generator state as
    ``patchnce_with_head``.

    ``dp_group``: as in ``patchnce_with_head`` -- the head gradients are averaged over the group, and the negatives are
    the rank's own shard, as upstream CUT under DDP.  ``patchnce_with_head_global_negatives`` takes the negatives from
    every rank's shard instead.

    Envelope: nc = 128 or 256, tensor-core math (not simt_f32), C <= 256, P <= 1024 and B * round_up(P, 128) <= 65536
    per layer.  Outside it a RuntimeError is raised before any launch; there is no other implementation to fall back to.
    """
    plan, tgt, params, ids = _head_begin(netF, src_feats, tgt_feats, temperature, num_patches, patch_ids, math, dp_group,
                                         mb=True)
    loss = _FusedHeadPatchNCE.apply(plan, netF.nc, *tgt, *params)
    return loss, ids


def patchnce_with_head_global_negatives(netF: "PatchSampleF", src_feats, tgt_feats, temperature=0.07, num_patches=256,
                                        patch_ids=None, math: Optional[str] = None, negatives_group=True, dp_group=None):
    """``patchnce_with_head_minibatch`` with the negatives of the whole data-parallel batch (global negatives, the head's
    counterpart of ``PatchNCELoss(negatives_group=...)``).  Returns ``(loss, ids)``.

    ``negatives_group``: ``True`` (the default process group) or a ``ProcessGroup`` of W ranks.  Each rank holds an
    equal shard of B_l images, in rank order (``dp.shard_batch``), and every rank passes the same ids (one seed, or
    ``dp.broadcast_patch_ids``) and the same head parameters; neither is checked at run time.  Per layer, the rank's
    B_l * P query rows ``normalize(netF(raw tgt patches))`` are contrasted with the keys
    ``normalize(netF(raw src patches)).detach()`` of all W * B_l images, which are all-gathered without gradient in the
    forward; row i's positive is the key of the same global (image, patch).  Each rank returns the mean CE over its own
    rows, so the mean of the W losses is ``patchnce_with_head_minibatch`` on the global batch, and averaging the
    gradients over the ranks reproduces one GPU.  The guard is global: a layer is guarded on every rank (loss 0, zero
    gradients, one warning per forward) exactly when the one-GPU call on the global batch guards it.  ``None``, no
    process group, or a group of one rank: ``patchnce_with_head_minibatch`` itself, bit for bit.

    ``dp_group``: independent of ``negatives_group`` -- as in ``patchnce_with_head``, the head gradients are averaged
    over it (hidden under the dense-gradient kernel).  With ``negatives_group`` alone the head gradients are the rank's
    own: average netF's gradients yourself (``dp.GradReducer``, DDP).

    Envelope: ``patchnce_with_head_minibatch``'s applied to the global batch -- nc = 128 or 256, tensor-core math, C <= 256,
    P <= 1024 and W * B_l * round_up(P, 128) <= 65536 per layer.  Outside it a RuntimeError is raised before any launch
    or collective."""
    plan, tgt, params, ids = _head_begin(netF, src_feats, tgt_feats, temperature, num_patches, patch_ids, math, dp_group,
                                         mb=True, negatives_group=negatives_group)
    loss = _FusedHeadPatchNCE.apply(plan, netF.nc, *tgt, *params)
    return loss, ids


def head_loss_and_grads(netF: "PatchSampleF", src_feats, tgt_feats, temperature=0.07, num_patches=256,
                        patch_ids=None, math: Optional[str] = None, grad_output: Optional[torch.Tensor] = None,
                        dp_group=None):
    """``patchnce_with_head`` (fused path) and its complete backward in ONE call, without autograd -- the head-mode
    counterpart of ``PatchNCELoss.loss_and_grads``.  Returns ``(loss, [d (grad_output * loss) / d tgt_feats[l]], ids)``
    and ACCUMULATES the head gradients into ``p.grad`` of netF's parameters (assigned when ``p.grad is None``: views
    of one flat fp32 buffer, already averaged over ``dp_group``), exactly what ``loss.backward(grad_output)`` leaves
    there.  Same ids, kernels and values as the autograd route; no ``Function.apply``, no engine hand-off and no
    ``AccumulateGrad`` per parameter (20 of them for five layers): at the batches the reference trains with, that
    host work is longer than the GPU's (DESIGN.md 4.5).  For loops that drive the generator's backward themselves:
    ``torch.autograd.backward(tgt_feats, grads)``.  Per-image negatives only: ``head_minibatch_loss_and_grads`` is the
    counterpart with minibatch negatives."""
    if (math or DEFAULT_MATH) == "simt_f32":
        raise RuntimeError("head_loss_and_grads runs the tensor-core head only")
    plan, tgt, params, ids = _head_begin(netF, src_feats, tgt_feats, temperature, num_patches, patch_ids, math, dp_group)
    return _head_loss_and_grads(netF, plan, tgt, params, ids, grad_output)


def head_minibatch_loss_and_grads(netF: "PatchSampleF", src_feats, tgt_feats, temperature=0.07, num_patches=256,
                                  patch_ids=None, math: Optional[str] = None, grad_output: Optional[torch.Tensor] = None,
                                  dp_group=None):
    """``patchnce_with_head_minibatch`` and its complete backward in ONE call, without autograd: returns
    ``(loss, [d (grad_output * loss) / d tgt_feats[l]], ids)`` and ACCUMULATES the head gradients into ``p.grad`` of
    netF's parameters exactly as ``head_loss_and_grads`` does.  Same ids, kernels and values as
    ``patchnce_with_head_minibatch(...)`` followed by ``loss.backward(grad_output)``; same envelope and errors."""
    plan, tgt, params, ids = _head_begin(netF, src_feats, tgt_feats, temperature, num_patches, patch_ids, math, dp_group,
                                         mb=True)
    return _head_loss_and_grads(netF, plan, tgt, params, ids, grad_output)


def head_global_negatives_loss_and_grads(netF: "PatchSampleF", src_feats, tgt_feats, temperature=0.07,
                                         num_patches=256, patch_ids=None, math: Optional[str] = None,
                                         grad_output: Optional[torch.Tensor] = None, negatives_group=True,
                                         dp_group=None):
    """``patchnce_with_head_global_negatives`` and its complete backward in ONE call, without autograd: returns
    ``(loss, [d (grad_output * loss) / d tgt_feats[l]], ids)`` and ACCUMULATES the head gradients into ``p.grad`` of
    netF's parameters exactly as ``head_minibatch_loss_and_grads`` does.  Same ids, kernels, collectives and values as
    ``patchnce_with_head_global_negatives(...)`` followed by ``loss.backward(grad_output)``; same envelope and errors."""
    plan, tgt, params, ids = _head_begin(netF, src_feats, tgt_feats, temperature, num_patches, patch_ids, math, dp_group,
                                         mb=True, negatives_group=negatives_group)
    return _head_loss_and_grads(netF, plan, tgt, params, ids, grad_output)


def _head_loss_and_grads(netF, plan, tgt, params, ids, grad_output):
    """The body of the autograd-free head entries: forward, backward, accumulation into ``p.grad``."""
    dev = tgt[0].device
    with torch.no_grad():
        tgt = [t.detach() for t in tgt]
        w = [_f32c(p_) for p_ in params]
        ws, out, state = _head_fwd(plan, netF.nc, tgt, w)
        g = grad_output
        if g is None:
            g = _one(dev)
        elif g.dtype is not torch.float32 or g.device != dev or not g.is_contiguous():
            g = g.detach().to(device=dev, dtype=torch.float32).contiguous()
        grads, flat, sizes = _head_bwd(plan, netF.nc, tgt, w, ws, state, g)
        views = None
        for k, p_ in enumerate(params):
            if not p_.requires_grad:
                continue
            if views is None:
                views = torch.split_with_sizes(flat, sizes)
            v = views[k].view(p_.shape)
            if p_.dtype is not torch.float32:
                v = v.to(p_.dtype)
            if p_.grad is None:
                p_.grad = v
            else:
                p_.grad.add_(v)
    return out[0], grads, ids


_ONES = {}


def _one(dev) -> torch.Tensor:
    """A device-resident fp32 1.0 per device (the upstream gradient of a plain ``backward()``)."""
    t = _ONES.get(dev.index)
    if t is None:
        t = _ONES[dev.index] = torch.ones((), dtype=torch.float32, device=dev)
    return t


def install_reference_shim(optimiser_side: bool = False, d_side: bool = False,
                           nce_includes_all_negatives_from_minibatch: bool = False, negatives_group=None):
    """Make ``from GAN_Variant1.losses.patchnce_cut import compute_patchnce_loss`` resolve to this
    implementation, so the unchanged reference training loop (train_cutpp.py:28) uses the B200
    path.  Call before importing ``GAN_Variant1.training.train_cutpp``.

    ``optimiser_side=True`` also re-points the two optimiser-side seams of SURVEY.md section 8f row 3 (the
    reference package must be importable): ``GAN_Variant1.utils.io_ckpt.EMA`` (imported by name at
    train_cutpp.py:34) -> the one-launch ``EMA``, and ``AMPContext.step_optimizer`` (amp_utils.py:29) -> the
    three-launch ``amp_step_optimizer``.  ``d_side=True`` does the same for row 4: ``training.diffaugment.DiffAugment``
    (imported by name at train_cutpp.py:30) and ``losses.adv_hinge.discriminator_hinge_loss`` / ``generator_hinge_loss``.

    ``nce_includes_all_negatives_from_minibatch`` becomes the default of the shimmed ``compute_patchnce_loss`` and
    ``PatchNCELoss``: the reference loop passes only three keywords to ``compute_patchnce_loss`` (train_cutpp.py:285-292),
    so this is how ``patchnce.nce_includes_all_negatives_from_minibatch`` of the config reaches the loss.
    ``negatives_group`` (with that flag only, ValueError otherwise) becomes their default as well: global negatives
    over the ranks of a data-parallel run (``PatchNCELoss``)."""
    import functools
    import types
    if negatives_group is not None and not nce_includes_all_negatives_from_minibatch:
        raise ValueError("negatives_group needs nce_includes_all_negatives_from_minibatch=True")
    if d_side:
        import importlib
        from . import dside
        importlib.import_module("GAN_Variant1.training.diffaugment").DiffAugment = dside.DiffAugment
        ah = importlib.import_module("GAN_Variant1.losses.adv_hinge")
        ah.discriminator_hinge_loss, ah.generator_hinge_loss = dside.discriminator_hinge_loss, dside.generator_hinge_loss
    if optimiser_side:
        import importlib
        from .amp_step import amp_step_optimizer
        from .ema import EMA
        importlib.import_module("GAN_Variant1.utils.io_ckpt").EMA = EMA
        importlib.import_module("GAN_Variant1.utils.amp_utils").AMPContext.step_optimizer = amp_step_optimizer
    mod = types.ModuleType("GAN_Variant1.losses.patchnce_cut")
    if nce_includes_all_negatives_from_minibatch:
        kw = {"nce_includes_all_negatives_from_minibatch": True}
        if negatives_group is not None:
            kw["negatives_group"] = negatives_group
        mod.PatchNCELoss = functools.partial(PatchNCELoss, **kw)
        mod.compute_patchnce_loss = functools.partial(compute_patchnce_loss, **kw)
    else:
        mod.PatchNCELoss = PatchNCELoss
        mod.compute_patchnce_loss = compute_patchnce_loss
    mod.__doc__ = "B200-native PatchNCE (gan_variant_research_b200) behind the reference's module path."
    sys.modules["GAN_Variant1.losses.patchnce_cut"] = mod
    pkg = sys.modules.get("GAN_Variant1.losses")
    if pkg is not None:
        setattr(pkg, "patchnce_cut", mod)
    return mod
