"""CPU oracle for global negatives on the row route (``rows_patchnce_global_negatives``).  TEST INFRASTRUCTURE ONLY.

Rows are used as given (already L2-normalised, as ``PatchSampleF`` returns them).  ``q`` and ``k`` are the GLOBAL
(W * B_l * P, D) rows of one layer, image-major; rank r of W holds rows [r * N_l, (r + 1) * N_l) with N_l = B_l * P.
Its loss is the mean row CE of its own query rows against all W * N_l keys, Z = clamp(q k^T / tau, +-50), row i's label
the key of the same global row; its gradient is d loss_r / d q_r.  The guard is that of the global group: a non-finite
query row on any rank, a non-finite key, or a non-finite loss gives every rank a 0 loss and a zero gradient (the row
route writes zero d q rows for a guarded layer).

The tests pin it to an autograd restatement at W = 1 and, for W in {2, 4}, to W = 1 itself: the mean of the shard losses
is the one-group loss and the shard gradients divided by W are its rows."""
import numpy as np

LOGIT_CLAMP = 50.0


def layer_loss_and_grad_rows_shard(q, k, temperature, world, rank, n_layers=1, upstream=1.0):
    """One layer on rank ``rank`` of ``world`` -> ``(shard_loss, d (upstream * shard_loss / n_layers) / d q_rank)``."""
    q = np.asarray(q, dtype=np.float64)
    k = np.asarray(k, dtype=np.float64)
    n = q.shape[0]
    if n % world:
        raise ValueError(f"{n} rows are not divisible by world size {world}")
    nl = n // world
    lo = rank * nl
    qr = q[lo:lo + nl]
    grad = np.zeros_like(qr)
    with np.errstate(all="ignore"):
        z_raw = (qr @ k.T) / temperature
        z = np.clip(z_raw, -LOGIT_CLAMP, LOGIT_CLAMP)
        m = z.max(axis=1, keepdims=True)
        e = np.exp(z - m)
        s = e.sum(axis=1, keepdims=True)
        rows = np.arange(nl)
        loss = ((np.log(s) + m)[:, 0] - z[rows, lo + rows]).mean()
        if not (np.isfinite(q).all() and np.isfinite(k).all() and np.isfinite(loss)):
            return 0.0, grad
        mask = (z_raw >= -LOGIT_CLAMP) & (z_raw <= LOGIT_CLAMP)
        onehot = np.zeros_like(z)
        onehot[rows, lo + rows] = 1.0
        d_z = (e / s - onehot) * mask * (upstream / (nl * n_layers))
        grad = (d_z @ k) / temperature
    return float(loss), grad
