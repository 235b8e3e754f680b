"""clipk: B200-native (sm_100a) fused contrastive loss behind open_clip's ClipLoss API."""
from .loss import ClipLoss, CoCaLoss, DistillClipLoss, SigLipLoss, create_loss, gather_features  # noqa: F401
from .ops import fused_clip_loss, fused_normalize_clip_loss, gpu_launches  # noqa: F401
from .siglip import siglip_loss  # noqa: F401
from .metrics import clip_val_loss, get_clip_metrics, logits_panels, target_ranks, zero_shot_accuracy  # noqa: F401
from .ict import ict_retrieval_loss  # noqa: F401

__all__ = ["ClipLoss", "CoCaLoss", "DistillClipLoss", "SigLipLoss", "create_loss", "gather_features", "fused_clip_loss",
           "fused_normalize_clip_loss", "siglip_loss", "gpu_launches", "clip_val_loss", "get_clip_metrics", "target_ranks",
           "zero_shot_accuracy", "logits_panels", "ict_retrieval_loss"]
