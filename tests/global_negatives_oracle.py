"""CPU oracle for global negatives (minibatch negatives across data-parallel ranks, ``negatives_group``).
TEST INFRASTRUCTURE ONLY.

Rank r of W holds images r * B_l ... r * B_l + B_l - 1 of a global batch of B = W * B_l images.  Its loss is the mean row
CE of its own B_l * P query rows against the keys of all B * P rows of the global batch, rows image-major as in
``minibatch_oracle.batch_as_one_image``; its gradient is d loss_r / d tgt_r.  The guard is that of the global group
(patchnce_cut.py:97-99 on the N = B * P rows): a non-finite query row on any rank, or a non-finite key, gives every rank a
0 loss and a zero upstream gradient, so only the rank's sampled target patches holding a NaN/Inf come out NaN.

The same float64 steps as ``oracle.patchnce_oracle.layer_loss_and_grad_np``, restricted to a block of rows; the tests
pin it to ``minibatch_oracle.layer_loss_and_grad_np_mb``: the mean of the W shard losses is the full-batch loss and
the shard gradients divided by W are the full-batch gradient's slices."""
import numpy as np

from minibatch_oracle import batch_as_one_image
from oracle import patchnce_oracle as orc


def layer_loss_and_grad_np_shard(src, tgt, ids, temperature, world, rank, n_layers=1, upstream=1.0):
    """One layer on rank ``rank`` of ``world``; ``src`` and ``tgt`` are the GLOBAL batch.  Returns
    ``(shard_loss, dense_grad_of_the_shard)``, the gradient of upstream * shard_loss / n_layers w.r.t. tgt_rank."""
    src = np.asarray(src, dtype=np.float64)
    tgt = np.asarray(tgt, dtype=np.float64)
    ids = np.asarray(ids, dtype=np.int64)
    b_sz, c_sz, h, w = tgt.shape
    if b_sz % world:
        raise ValueError(f"batch {b_sz} is not divisible by world size {world}")
    bl, p = b_sz // world, ids.shape[0]
    k_raw = batch_as_one_image(src, ids).reshape(c_sz, -1).T                 # (B*P, C) keys of every rank
    q_all = batch_as_one_image(tgt, ids).reshape(c_sz, -1).T
    lo = rank * bl * p
    q_raw = q_all[lo:lo + bl * p]
    grad = np.zeros((bl, c_sz, h * w), dtype=np.float64)
    with np.errstate(all="ignore"):
        k_hat, _ = orc._normalize_np(k_raw)
        q_hat, q_n = orc._normalize_np(q_raw)
        z_raw = (q_hat @ k_hat.T) / temperature
        z = np.clip(z_raw, -orc.LOGIT_CLAMP, orc.LOGIT_CLAMP)
        m = z.max(axis=1, keepdims=True)
        e = np.exp(z - m)
        s = e.sum(axis=1, keepdims=True)
        rows = np.arange(bl * p)
        loss = ((np.log(s) + m)[:, 0] - z[rows, lo + rows]).mean()
        if not (np.isfinite(q_all).all() and np.isfinite(k_raw).all() and np.isfinite(loss)):
            bad = ~np.isfinite(q_raw).all(axis=1)
            for b in range(bl):
                grad[b][:, ids[bad[b * p:(b + 1) * p]]] = np.nan
            return 0.0, grad.reshape(bl, c_sz, h, w)
        mask = (z_raw >= -orc.LOGIT_CLAMP) & (z_raw <= orc.LOGIT_CLAMP)
        onehot = np.zeros_like(z)
        onehot[rows, lo + rows] = 1.0
        d_z = (e / s - onehot) * mask * (upstream / (p * bl * n_layers))
        d_qhat = (d_z @ k_hat) / temperature
        big = q_n >= orc.NORM_EPS
        proj = (q_hat * d_qhat).sum(-1, keepdims=True)
        d_x = np.where(big, (d_qhat - q_hat * proj) / np.maximum(q_n, orc.NORM_EPS), d_qhat / orc.NORM_EPS)
        for b in range(bl):
            np.add.at(grad[b].T, ids, d_x[b * p:(b + 1) * p])                 # duplicate ids accumulate
    return float(loss), grad.reshape(bl, c_sz, h, w)
