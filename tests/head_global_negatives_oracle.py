"""Oracle for the netF head with global negatives (``patchnce_with_head_global_negatives``).  TEST INFRASTRUCTURE ONLY.

Rank r of W holds images r * B_l ... r * B_l + B_l - 1 of a global batch of B = W * B_l images.  Per layer its B_l * P
query rows ``q = normalize(netF(raw tgt patches of its images))`` are contrasted with the keys
``k = normalize(netF(raw src patches)).detach()`` of all B * P rows of the global batch (image-major, as in
``head_minibatch_oracle``); row i's positive is the key of the same global (image, patch).  The rank's loss is the mean
row CE over its own rows, the mean over layers on top.  The guard is the global one: a layer contributes a constant 0
(no gradient at all) on every rank exactly when ``head_minibatch_oracle.layer_loss`` on the global batch guards it.

Built on ``head_minibatch_oracle``'s pieces; tests/test_head_global_negatives.py pins it to ``head_minibatch_loss``: at
W = 1 it is that function, and for W > 1 the mean of the W shard losses is the global loss, the shard gradients w.r.t.
tgt divided by W are the global gradient's slices and the head gradients summed over the ranks and divided by W are
the global head gradients.  Device-agnostic: run it in float64 on the GPU for the large batches."""
import torch
import torch.nn.functional as F

import head_minibatch_oracle as hmo
from oracle import patchnce_oracle as orc


def layer_loss_shard(src, tgt, ids, head, world, rank, temperature, warn=None):
    """One layer on rank ``rank`` of ``world``; ``src`` and ``tgt`` are the GLOBAL batch (B, C, H, W).  Differentiable
    w.r.t. the rank's slice of ``tgt`` and the head (through q only)."""
    b = tgt.shape[0]
    if b % world:
        raise ValueError(f"batch {b} is not divisible by world size {world}")
    bl = b // world
    with torch.no_grad():                                       # the guard of the global group
        seen = []
        hmo.layer_loss(src, tgt.detach(), ids, tuple(w.detach() for w in head), temperature, seen)
    if seen:
        if warn is not None:
            warn.append("layer")
        return torch.zeros((), dtype=tgt.dtype, device=tgt.device)
    k = orc.head_forward_torch(hmo.raw_rows(src, ids), *head).detach()                  # (B * P, nc), every rank's
    q = orc.head_forward_torch(hmo.raw_rows(tgt[rank * bl:(rank + 1) * bl], ids), *head)   # (B_l * P, nc), this rank's
    z = (q @ k.t() / temperature).clamp(-orc.LOGIT_CLAMP, orc.LOGIT_CLAMP)
    lo = rank * bl * ids.numel()
    return F.cross_entropy(z, torch.arange(lo, lo + z.shape[0], device=z.device))


def head_global_negatives_loss(src_feats, tgt_feats, ids_list, heads, world, rank, temperature=0.07, warn=None):
    """All layers on rank ``rank``: sum_l loss_l / L."""
    total = 0.0
    for s, t, i, h in zip(src_feats, tgt_feats, ids_list, heads):
        total = total + layer_loss_shard(s, t, i, h, world, rank, temperature, warn)
    return total / len(src_feats)
