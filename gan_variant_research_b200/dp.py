"""Data-parallel plumbing for the PatchNCE path (SURVEY.md section 8e): one process per GPU.

The path shards on the batch dimension and needs NO collective in the reference-exact mode:
negatives are per image (patchnce_cut.py:83-94), the dense ``d tgt_feat`` stays on the rank that
owns the image.  Two things have to agree across ranks:

* the ``patch_ids`` of every layer -- the reference shares ONE draw per layer across the whole batch
  (patchnce_cut.py:63): seed the id generator identically on all ranks, or ``broadcast_patch_ids``;
* the loss scale -- each rank averages over its own B/N images, so gradients are averaged over
  ranks (what DDP does); for the dense feature gradients this is a local ``1 / world_size`` factor.

Only the netF head (north-star extension, absent from the reference) owns parameters whose
gradients must be summed: ``allreduce_head_grads`` does it as ONE flat all-reduce (<= 2.1 MB, latency
bound on NVLink 5) on the current stream; torch.distributed (NCCL on GPUs, gloo in the CPU tests)
is plumbing here.

Global negatives (``PatchNCELoss(..., nce_includes_all_negatives_from_minibatch=True, negatives_group=...)``) add one
collective to the forward: the all-gather of every rank's detached keys (``allgather_slots_``).  The backward stays
local.
"""
from __future__ import annotations

from typing import Iterable, List, Optional

import torch
import torch.distributed as dist


def _world(group=None) -> int:
    return dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1


def shard_batch(tensors: Iterable[torch.Tensor], rank: Optional[int] = None, world: Optional[int] = None,
                group=None) -> List[torch.Tensor]:
    """This rank's contiguous slice of the batch dimension of every tensor (equal shards)."""
    world = _world(group) if world is None else world
    rank = (dist.get_rank(group) if world > 1 else 0) if rank is None else rank
    out = []
    for t in tensors:
        b = t.shape[0]
        if b % world:
            raise ValueError(f"batch {b} is not divisible by world size {world}")
        per = b // world
        out.append(t[rank * per:(rank + 1) * per])
    return out


def broadcast_patch_ids(ids: List[torch.Tensor], src: int = 0, group=None) -> List[torch.Tensor]:
    """Make every rank use rank ``src``'s ids (in place; one small broadcast per layer, <= 32 KB)."""
    if _world(group) > 1:
        for t in ids:
            dist.broadcast(t, src=src, group=group)
    return ids


_COMM_STREAMS = {}


def comm_stream(device) -> "torch.cuda.Stream":
    """Side stream the overlapped head-gradient all-reduce runs on (one per device)."""
    key = torch.device(device).index
    st = _COMM_STREAMS.get(key)
    if st is None:
        st = _COMM_STREAMS[key] = torch.cuda.Stream(device=device)
    return st


def resolve_group(group):
    """``True`` -> the default process group; returns None when there is nothing to reduce over."""
    if not (dist.is_available() and dist.is_initialized()):
        return None
    if group is True:
        group = dist.group.WORLD
    return group if dist.get_world_size(group) > 1 else None


def allgather_slots_(region: torch.Tensor, rank: int, group=None) -> torch.Tensor:
    """In-place all-gather of equal slots: ``region`` (a flat uint8 tensor of ``world`` slots) holds this rank's bytes
    in slot ``rank``; afterwards slot ``w`` holds rank ``w``'s.  The key exchange of global negatives
    (``PatchNCELoss(negatives_group=...)``): ordered after the work already queued on the current stream, and the
    current stream waits for it -- no host synchronisation under NCCL."""
    world = dist.get_world_size(group)
    if world == 1:
        return region
    slots = region.view(world, -1)
    if dist.get_backend(group) == "nccl":
        dist.all_gather_into_tensor(region, slots[rank], group=group)      # NCCL allgather in place
    else:
        # gloo takes CUDA tensors in the list form only; the input must not alias an output it writes
        dist.all_gather(list(slots.unbind(0)), slots[rank].clone(), group=group)
    return region


def allreduce_flat_(flat: torch.Tensor, group=None, average: bool = True) -> torch.Tensor:
    """In-place sum (or mean) of one flat buffer over the ranks, on the current stream."""
    world = _world(group)
    if world == 1:
        return flat
    if average and dist.get_backend(group) == "nccl":
        dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=group)
    else:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        if average:
            flat.div_(world)
    return flat


def allreduce_head_grads(module: torch.nn.Module, group=None, average: bool = True) -> int:
    """Sum (or average) the gradients of ``module``'s parameters over the ranks with one flat
    all-reduce.  Returns the number of elements reduced (0 when there is nothing to do)."""
    world = _world(group)
    grads = [p.grad for p in module.parameters() if p.grad is not None]
    if world == 1 or not grads:
        return 0
    flat = torch.cat([g.reshape(-1).to(torch.float32) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    if average:
        flat.div_(world)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n
    return off


class _MultiCopy:
    """Bucket <-> gradients in one launch each way: ``pnce_multi_axpby`` (mode 1, dst = src; include/pnce.h, the kernel
    behind ``EMA``) over device tables of the bucket's slot addresses and of the gradients' addresses.  A reducer over the
    reference generator's 48 parameter tensors otherwise issues 96 slice copies per backward and is bound by their host
    time, not by NCCL.  The gradient table is re-uploaded only when a gradient tensor has moved (``zero_grad`` drops the
    tensors, the caching allocator usually hands the same blocks back)."""

    def __init__(self, flat, slots):
        from . import _lib
        self._lib = _lib
        self.dev = flat.device
        self.params = [p for p, _, _ in slots]
        chunk = _lib.load().pnce_multi_chunk_elems()
        ct, cs = [], []
        for t, (_, _, n) in enumerate(slots):
            for e in range(0, n, chunk):
                ct.append(t)
                cs.append(e)
        self.n_chunks = len(ct)
        self.chunk_tensor = torch.tensor(ct, dtype=torch.int32, device=self.dev)
        self.chunk_start = torch.tensor(cs, dtype=torch.int64, device=self.dev)
        self.numel = torch.tensor([n for _, _, n in slots], dtype=torch.int64, device=self.dev)
        base, item = flat.data_ptr(), flat.element_size()
        self.slot_ptrs = torch.tensor([base + off * item for _, off, _ in slots], dtype=torch.int64, device=self.dev)
        self.grad_ptr_list, self.grad_ptrs = None, None

    def _grads(self):
        grads = [p.grad for p in self.params]
        for g in grads:
            if g is None or g.dtype != torch.float32 or not g.is_cuda or not g.is_contiguous() or g.is_sparse:
                return None
        ptrs = [g.data_ptr() for g in grads]
        if ptrs != self.grad_ptr_list:
            self.grad_ptr_list = ptrs
            self.grad_ptrs = torch.tensor(ptrs, dtype=torch.int64, device=self.dev)
        return grads

    def _launch(self, dst, src):
        import ctypes
        st = torch.cuda.current_stream(self.dev).cuda_stream
        with torch.cuda.device(self.dev):
            self._lib.check(self._lib.load().pnce_multi_axpby(dst.data_ptr(), src.data_ptr(), self.numel.data_ptr(),
                                                              self.chunk_tensor.data_ptr(), self.chunk_start.data_ptr(),
                                                              self.n_chunks, ctypes.c_float(0.0), ctypes.c_float(0.0), 1, st),
                            "pnce_multi_axpby")

    def pack(self) -> bool:
        if self._grads() is None:
            return False
        self._launch(self.slot_ptrs, self.grad_ptrs)
        return True

    def unpack(self) -> bool:
        grads = self._grads()
        if grads is None:
            return False
        self._launch(self.grad_ptrs, self.slot_ptrs)
        torch._C._increment_version(grads)           # written through raw pointers: tell autograd's version counters
        return True


class GradReducer:
    """Data-parallel gradient averaging around the UNCHANGED reference training step (SURVEY.md section 8f row 1,
    BASELINE config 5: "NCCL allreduce of netF/G/D grads"): attach it to the generator's and the
    discriminator's parameters once, and every ``backward()`` of ``train_step`` (training/train_cutpp.py:253,
    :261, :307 -- ``amp_ctx.scale_backward``) leaves ``.grad`` averaged over the ranks by the time it returns,
    i.e. before ``amp_ctx.step_optimizer`` unscales, clips and steps (utils/amp_utils.py:29-41).  Nothing
    in ``train_cutpp.py`` changes; ranks feed different shards of the batch (``shard_batch``).

    Mechanics (what DDP's reducer does, kept small): parameters are grouped into flat fp32 buckets of
    ``bucket_bytes`` in reverse registration order (gradients arrive roughly back to front); a
    post-accumulate-grad hook marks each gradient ready; a full bucket is packed (one multi-tensor launch of
    libpnce on GPUs, ``_MultiCopy``) and all-reduced (mean) on a side stream while the backward pass keeps
    running; an end-of-backward callback launches the buckets that only filled partially (a pass that touches
    a subset of the parameters, e.g. the D step), joins the side stream and copies the averaged values back
    into ``.grad`` (again one launch per complete bucket).  Scaled (GradScaler)
    gradients average like any others; an inf on one rank becomes an inf on all, so every rank skips the
    same steps."""

    def __init__(self, params, group=None, bucket_bytes: int = 32 << 20, average: bool = True):
        self.group = group
        self.average = average
        self.params = [p for p in params if p.requires_grad]
        self.world = _world(group)
        self.buckets = []            # each: dict(flat, slots=[(param, offset, numel)], ready=set(), launched=bool)
        self.where = {}              # id(param) -> (bucket index, slot index)
        cur, cur_elems = [], 0
        for p in reversed(self.params):
            if cur and (cur_elems + p.numel()) * 4 > bucket_bytes:
                self._close_bucket(cur)
                cur, cur_elems = [], 0
            cur.append(p)
            cur_elems += p.numel()
        if cur:
            self._close_bucket(cur)
        self._callback_queued = False
        self._handles = [p.register_post_accumulate_grad_hook(self._on_grad) for p in self.params]

    def _close_bucket(self, plist):
        dev = plist[0].device
        slots, off = [], 0
        for k, p in enumerate(plist):
            slots.append((p, off, p.numel()))
            self.where[id(p)] = (len(self.buckets), k)
            off += (p.numel() + 3) // 4 * 4          # every slot starts on a 16-byte boundary (128-bit copies)
        flat = torch.zeros(off, dtype=torch.float32, device=dev)
        self.buckets.append({"flat": flat, "slots": slots, "ready": set(), "launched": False,
                             "multi": _MultiCopy(flat, slots) if flat.is_cuda else None})

    def remove(self):
        for h in self._handles:
            h.remove()
        self._handles = []

    # ---- hooks -------------------------------------------------------------------------------
    def _on_grad(self, p):
        if self.world == 1:
            return
        bi, si = self.where[id(p)]
        b = self.buckets[bi]
        b["ready"].add(si)                               # the gradient is copied when its bucket is launched
        if not self._callback_queued:
            self._callback_queued = True
            torch.autograd.Variable._execution_engine.queue_callback(self._finalize)
        if len(b["ready"]) == len(b["slots"]):
            self._launch(b)

    def _launch(self, b):
        flat = b["flat"]
        b["launched"] = True
        # gradients -> bucket: ONE multi-tensor launch of libpnce when the whole bucket is ready and every gradient is a
        # contiguous fp32 CUDA tensor (the usual case), one copy per ready slot otherwise
        if not (len(b["ready"]) == len(b["slots"]) and b["multi"] is not None and b["multi"].pack()):
            for si in b["ready"]:
                p, off, n = b["slots"][si]
                flat[off:off + n].copy_(p.grad.detach().reshape(-1))
        if flat.is_cuda:
            main = torch.cuda.current_stream(flat.device)
            side = comm_stream(flat.device)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                allreduce_flat_(flat, self.group, self.average)
        else:
            allreduce_flat_(flat, self.group, self.average)

    def _finalize(self):
        self._callback_queued = False
        touched = [b for b in self.buckets if b["ready"]]
        for b in touched:                      # same set on every rank: same autograd graph everywhere
            if not b["launched"]:
                self._launch(b)
        for b in touched:
            flat = b["flat"]
            if flat.is_cuda:
                torch.cuda.current_stream(flat.device).wait_stream(comm_stream(flat.device))
            if not (len(b["ready"]) == len(b["slots"]) and b["multi"] is not None and b["multi"].unpack()):
                for si in b["ready"]:
                    p, off, n = b["slots"][si]
                    p.grad.copy_(flat[off:off + n].view_as(p.grad))
            b["ready"] = set()
            b["launched"] = False
