"""Oracle for the netF head with minibatch negatives (``patchnce_with_head_minibatch``).  TEST INFRASTRUCTURE ONLY.

PARITY PINNED THROUGH THE B = 1 IDENTITY AND AN INDEPENDENT RESTATEMENT: the reference has no head and no code that
reads nce_includes_all_negatives_from_minibatch, so there is no reference run to freeze.  Per layer the function below
applies ``oracle.patchnce_oracle.head_forward_torch`` to the raw gathered rows of both sides (k detached, as in
``patchnce_head_loss_torch``), then the minibatch law of ``tests/minibatch_oracle.py`` to the B * P rows: one N x N
problem, the +-50 clamp, mean CE over the N rows, the non-finite guard on that group.  At B = 1 that is
``patchnce_head_loss_torch`` (tests/test_head_minibatch.py checks it, and an independent autograd expression).
Device-agnostic: run it in float64 on the GPU for the large batches."""
import torch
import torch.nn.functional as F

from oracle import patchnce_oracle as orc


def raw_rows(x, ids):
    """(B, C, H, W) + ids (P,) -> the raw sampled patches (B * P, C), image-major."""
    b, c = x.shape[:2]
    return x.reshape(b, c, -1)[:, :, ids].transpose(1, 2).reshape(-1, c)


def layer_loss(src, tgt, ids, head, temperature, warn=None):
    """One layer: ``head`` = (w1, b1, w2, b2).  Differentiable w.r.t. tgt and the head (through q only).  A non-finite
    group contributes a constant 0 (no gradient at all: the kernel's zero row gradient)."""
    k = orc.head_forward_torch(raw_rows(src, ids), *head).detach()
    q = orc.head_forward_torch(raw_rows(tgt, ids), *head)
    z = (q @ k.t() / temperature).clamp(-orc.LOGIT_CLAMP, orc.LOGIT_CLAMP)
    loss = F.cross_entropy(z, torch.arange(z.shape[0], device=z.device))
    if not torch.isfinite(loss):
        if warn is not None:
            warn.append("layer")
        return torch.zeros((), dtype=loss.dtype, device=loss.device)
    return loss


def head_minibatch_loss(src_feats, tgt_feats, ids_list, heads, temperature=0.07, warn=None):
    """All layers: sum_l loss_l / L."""
    total = 0.0
    for s, t, i, h in zip(src_feats, tgt_feats, ids_list, heads):
        total = total + layer_loss(s, t, i, h, temperature, warn)
    return total / len(src_feats)
