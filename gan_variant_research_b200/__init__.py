"""B200-native PatchNCE contrastive path (CUT variant of Cameronr11/GAN-Variant-Research).

Public surface = the reference's seam (``GAN_Variant1/losses/patchnce_cut.py``) plus the
north-star module split; see ``patchnce.py``.  Importing this package never touches CUDA; the
first call into an op loads ``libpnce.so`` (built in-tree for sm_100a) and fails loudly if it,
or a CUDA device, is missing.
"""
from .patchnce import (  # noqa: F401
    DEFAULT_MATH,
    PatchNCELoss,
    PatchSampleF,
    compute_patchnce_loss,
    draw_patch_ids,
    draw_patch_ids_all,
    draw_ids,
    fused_head_supported,
    fused_patchnce,
    gradient_is_compressed,
    head_loss_and_grads,
    head_global_negatives_loss_and_grads,
    head_minibatch_loss_and_grads,
    install_reference_shim,
    patch_count,
    patchnce_with_head,
    patchnce_with_head_global_negatives,
    patchnce_with_head_minibatch,
    pinned_as_device,
    poll_nonfinite_warnings,
    rows_patchnce,
    rows_patchnce_multi,
    set_gradient_compression,
)
from .ema import EMA  # noqa: F401
from .dside import DiffAugment, discriminator_hinge_loss, generator_hinge_loss  # noqa: F401
from .amp_step import FusedAdamStep, amp_step_optimizer  # noqa: F401
from .feature_reuse import EncoderFeatureCache, enable_encoder_feature_reuse  # noqa: F401
from .dp import GradReducer, allreduce_head_grads, broadcast_patch_ids, shard_batch  # noqa: F401

__all__ = [
    "PatchNCELoss", "PatchSampleF", "compute_patchnce_loss", "fused_patchnce", "rows_patchnce", "rows_patchnce_multi",
    "draw_patch_ids", "draw_patch_ids_all", "draw_ids", "pinned_as_device", "patch_count", "install_reference_shim", "poll_nonfinite_warnings",
    "DEFAULT_MATH", "patchnce_with_head", "head_loss_and_grads", "patchnce_with_head_minibatch",
    "head_minibatch_loss_and_grads", "patchnce_with_head_global_negatives", "head_global_negatives_loss_and_grads",
    "set_gradient_compression", "gradient_is_compressed", "allreduce_head_grads", "broadcast_patch_ids", "shard_batch", "GradReducer", "EMA",
    "EncoderFeatureCache", "enable_encoder_feature_reuse", "FusedAdamStep", "amp_step_optimizer",
    "DiffAugment", "discriminator_hinge_loss", "generator_hinge_loss",
]
