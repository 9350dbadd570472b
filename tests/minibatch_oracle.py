"""CPU oracle for minibatch negatives (upstream CUT's nce_includes_all_negatives_from_minibatch, batch_dim_for_bmm = 1).
TEST INFRASTRUCTURE ONLY.

PARITY PINNED THROUGH THE B = 1 IDENTITY AND AN INDEPENDENT RESTATEMENT: the reference declares the config key
(configs/train_gan_cutpp.yaml:80) but no reference code reads it, so there is no reference run to freeze.  Both functions
below ARE the per-image functions of ``oracle/patchnce_oracle.py``, applied to one "image" whose P' = B * P patches are
the sampled patches of every image (image-major): a (1, C, B * P, 1) map with ids arange(B * P).  At B = 1 that map holds
the same rows in the same order, so the golden fixtures that pin the per-image functions pin these as well
(tests/test_minibatch_negatives.py checks the identity, and an independent autograd expression)."""
import numpy as np
import torch

from oracle import patchnce_oracle as orc


def batch_as_one_image(x, ids):
    """(B, C, H, W) + ids (P,) -> the (1, C, B*P, 1) map of the sampled patches of every image, image-major."""
    b_sz, c_sz = x.shape[0], x.shape[1]
    cols = x.reshape(b_sz, c_sz, -1)[:, :, ids]                  # (B, C, P) gather  patchnce_cut.py:66-74
    if isinstance(cols, torch.Tensor):
        return cols.permute(1, 0, 2).reshape(1, c_sz, -1, 1)
    return np.ascontiguousarray(cols.transpose(1, 0, 2)).reshape(1, c_sz, -1, 1)


def layer_loss_torch_mb(src, tgt, ids, temperature, warn=None):
    """One layer with minibatch negatives: gather, normalize, logits of the (1, B*P, C) view, /tau, clamp, CE over the
    B*P rows with label = own row, the non-finite guard of patchnce_cut.py:97-99 on that single group.  Differentiable
    w.r.t. tgt."""
    p = ids.numel()
    one = torch.arange(src.shape[0] * p, device=src.device)
    return orc.layer_loss_torch(batch_as_one_image(src, ids), batch_as_one_image(tgt, ids), one, temperature, warn)


def layer_loss_and_grad_np_mb(src, tgt, ids, temperature, n_layers=1, upstream=1.0):
    """float64 forward + analytic backward with minibatch negatives: ``(layer_loss, dense_grad_tgt)``.  The factor of
    d loss / d tgt is upstream / (B * P * n_layers), as in per-image mode; a non-finite group contributes 0 and its
    sampled target patches holding a NaN/Inf come out NaN (the NaN law of ``orc.layer_loss_and_grad_np``)."""
    src = np.asarray(src, dtype=np.float64)
    tgt = np.asarray(tgt, dtype=np.float64)
    ids = np.asarray(ids, dtype=np.int64)
    b_sz, c_sz, h, w = tgt.shape
    p = ids.shape[0]
    loss, _, g1 = orc.layer_loss_and_grad_np(batch_as_one_image(src, ids), batch_as_one_image(tgt, ids),
                                             np.arange(b_sz * p), temperature, n_layers, upstream)
    g1 = g1.reshape(c_sz, b_sz, p)
    grad = np.zeros((b_sz, c_sz, h * w), dtype=np.float64)
    with np.errstate(all="ignore"):
        for b in range(b_sz):
            np.add.at(grad[b].T, ids, g1[:, b, :].T)                 # duplicate ids accumulate
    return loss, grad.reshape(b_sz, c_sz, h, w)
