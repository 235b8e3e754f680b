"""Drop-in replacement for open_CLIP/src/open_clip/loss.py (ClipLoss and friends) on B200.

Same names, constructor arguments, method signatures and return conventions as the reference module:

    gather_features(image_features, text_features, local_loss, gather_with_grad, rank, world_size, use_horovod)
    ClipLoss(local_loss, gather_with_grad, cache_labels, rank, world_size, use_horovod)
        .get_ground_truth(device, num_logits)            reference loss.py:91-102
        .get_logits(image_features, text_features, s)    reference loss.py:104-121  (materialising)
        .forward(image_features, text_features, logit_scale, output_dict=False)     reference loss.py:123-140
    CoCaLoss, DistillClipLoss                            reference loss.py:143-221
    create_loss(args)                                    reference factory.py:250-278

`ClipLoss.forward` does not build logits: it calls clipk.ops.fused_clip_loss, which runs the fused step or the general
route of libclipk.so.  Deviations from the reference, all deliberate:
  * the loss is returned in fp32 even for pure-bf16 inputs (the reference returns bf16 there, which alone costs
    up to 2^-9 relative);
  * no per-step rank-0 prints (reference loss.py:79,110);
  * use_horovod=True raises NotImplementedError (horovod is not part of this build);
  * with world_size > 1 the backward always runs a reduce-scatter, also for gather_with_grad=False, because
    the column block of the text gradient is produced on the ranks that own the image rows.  Values match the
    reference in all four modes.
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

from . import distill
from .ops import fused_clip_loss, _all_gather_rows, _GatherRowsWithGrad
from .siglip import siglip_loss


def gather_features(image_features, text_features, local_loss=False, gather_with_grad=False, rank=0, world_size=1,
                    use_horovod=False, group=None):
    """Rank-major [world*b, d] copies of both feature matrices (reference loss.py:20-64).

    `group` (not in the reference, optional, last): the process group to gather over when it is not WORLD, e.g.
    Megatron's data-parallel group; `rank` / `world_size` are then the values inside that group.

    gather_with_grad=True : gradients flow back through the gather (reduce-scatter SUM).
    gather_with_grad=False: gathered rows carry no gradient, except that with local_loss=False this rank's own
                            rows are the live tensors, so they still receive theirs (loss.py:57-60).
    """
    if use_horovod:
        raise NotImplementedError("clipk: the horovod gather path of the reference is not part of this build")
    if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError("gather_features needs an initialised torch.distributed process group")
    if gather_with_grad:
        return (_GatherRowsWithGrad.apply(image_features, world_size, group),
                _GatherRowsWithGrad.apply(text_features, world_size, group))
    with torch.no_grad():
        all_i = _all_gather_rows(image_features, world_size, group)
        all_t = _all_gather_rows(text_features, world_size, group)
    if not local_loss:
        b = image_features.shape[0]
        lo, hi = rank * b, (rank + 1) * b
        all_i = torch.cat((all_i[:lo], image_features, all_i[hi:]), dim=0)
        all_t = torch.cat((all_t[:lo], text_features, all_t[hi:]), dim=0)
    return all_i, all_t


class ClipLoss(nn.Module):
    def __init__(self, local_loss=False, gather_with_grad=False, cache_labels=False, rank=0, world_size=1,
                 use_horovod=False):
        super().__init__()
        if use_horovod:
            raise NotImplementedError("clipk: use_horovod=True is not supported")
        self.local_loss = local_loss
        self.gather_with_grad = gather_with_grad
        self.cache_labels = cache_labels
        self.rank = rank
        self.world_size = world_size
        self.use_horovod = use_horovod
        # label cache, same observable state as the reference (loss.py:87-89)
        self.prev_num_logits = 0
        self.labels = {}
        # collectives run on WORLD like the reference's; set_process_group() narrows them (Megatron DP group)
        self.group = None

    def set_process_group(self, group, rank=None, world_size=None):
        """Run the gather / statistics exchange / reduce-scatter over `group` instead of WORLD.  rank and world_size
        default to this process's values inside the group.  Not in the reference (its ClipLoss always uses WORLD,
        loss.py:50-56); needed when the data-parallel group is a subset of the job (megatron/core/parallel_state.py)."""
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world_size = dist.get_world_size(group) if world_size is None else world_size
        self.labels, self.prev_num_logits = {}, 0
        return self

    def get_ground_truth(self, device, num_logits) -> torch.Tensor:
        """int64 arange labels, offset by num_logits*rank in local-loss mode; cached per device when enabled."""
        hit = self.prev_num_logits == num_logits and device in self.labels
        if hit:
            return self.labels[device]
        labels = torch.arange(num_logits, device=device, dtype=torch.long)
        if self.world_size > 1 and self.local_loss:
            labels = labels + num_logits * self.rank
        if self.cache_labels:
            self.labels[device] = labels
            self.prev_num_logits = num_logits
        return labels

    def get_logits(self, image_features, text_features, logit_scale):
        """Materialised (logits_per_image, logits_per_text); only DistillClipLoss needs them."""
        if self.world_size > 1:
            all_i, all_t = gather_features(image_features, text_features, self.local_loss, self.gather_with_grad,
                                           self.rank, self.world_size, self.use_horovod, self.group)
            if self.local_loss:
                per_image = logit_scale * image_features @ all_t.T
                per_text = logit_scale * text_features @ all_i.T
            else:
                per_image = logit_scale * all_i @ all_t.T
                per_text = per_image.T
        else:
            per_image = logit_scale * image_features @ text_features.T
            per_text = logit_scale * text_features @ image_features.T
        return per_image, per_text

    def forward(self, image_features, text_features, logit_scale, output_dict=False):
        if self.cache_labels:
            # the fused kernels index the positives themselves; the label cache is kept in the state the reference's
            # forward leaves it in (loss.py:131 calls get_ground_truth on every step)
            n = image_features.shape[0]
            self.get_ground_truth(image_features.device, n if (self.local_loss or self.world_size == 1) else n * self.world_size)
        loss = fused_clip_loss(image_features, text_features, logit_scale, self.local_loss, self.gather_with_grad,
                               self.rank, self.world_size, self.group)
        return {"contrastive_loss": loss} if output_dict else loss


class CoCaLoss(ClipLoss):
    def __init__(self, caption_loss_weight, clip_loss_weight, pad_id=0, local_loss=False, gather_with_grad=False,
                 cache_labels=False, rank=0, world_size=1, use_horovod=False):
        super().__init__(local_loss=local_loss, gather_with_grad=gather_with_grad, cache_labels=cache_labels,
                         rank=rank, world_size=world_size, use_horovod=use_horovod)
        self.clip_loss_weight = clip_loss_weight
        self.caption_loss_weight = caption_loss_weight
        self.caption_loss = nn.CrossEntropyLoss(ignore_index=pad_id)

    def forward(self, image_features, text_features, logits, labels, logit_scale, output_dict=False):
        clip_loss = self.clip_loss_weight * super().forward(image_features, text_features, logit_scale)
        caption_loss = self.caption_loss_weight * self.caption_loss(logits.permute(0, 2, 1), labels)
        if output_dict:
            return {"contrastive_loss": clip_loss, "caption_loss": caption_loss}
        return clip_loss, caption_loss


class DistillClipLoss(ClipLoss):
    """Contrastive loss of the student plus the cross-entropy of the student's softmax against a teacher's
    (reference loss.py:186-221).  Single-process calls with bf16 operands (bf16 features, or fp32 under bf16 autocast)
    take the fused contrastive loss and the panel-based distillation term of clipk/distill.py: no N x N matrix is ever
    held (tests/test_distill_gpu.py; CLIPK_FUSED_DISTILL=0 switches it off).  Everything else evaluates the reference's
    formula on materialised logits (get_logits), parity-pinned by tests/golden/shells."""

    def dist_loss(self, teacher_logits, student_logits):
        # -sum_j p_t(j) * log_softmax(student)(j) = lse(student) - sum_j p_t(j) * student(j), since sum_j p_t(j) = 1
        expected = (teacher_logits.softmax(dim=1) * student_logits).sum(dim=1)
        return (torch.logsumexp(student_logits, dim=1) - expected).mean()

    def forward(self, image_features, text_features, logit_scale, dist_image_features, dist_text_features,
                dist_logit_scale, output_dict=False):
        if os.environ.get("CLIPK_FUSED_DISTILL", "1") != "0" and distill.applicable(
                image_features, text_features, dist_image_features, dist_text_features, self.world_size):
            contrastive_loss = fused_clip_loss(image_features, text_features, logit_scale)
            distill_loss = distill.fused_distill_term(image_features, text_features, logit_scale,
                                                      dist_image_features, dist_text_features, dist_logit_scale)
        else:
            student = self.get_logits(image_features, text_features, logit_scale)
            teacher = self.get_logits(dist_image_features, dist_text_features, dist_logit_scale)
            labels = self.get_ground_truth(image_features.device, student[0].shape[0])
            contrastive_loss = sum(F.cross_entropy(lg, labels) for lg in student) / 2
            distill_loss = sum(self.dist_loss(t, lg) for t, lg in zip(teacher, student)) / 2
        if output_dict:
            return {"contrastive_loss": contrastive_loss, "distill_loss": distill_loss}
        return contrastive_loss, distill_loss


class SigLipLoss(nn.Module):
    """open_clip's SigLipLoss (open_clip >= 2.21; not in the 2.15 reference tree): the pairwise sigmoid loss of
    "Sigmoid Loss for Language Image Pre-Training" (Zhai et al., 2023).  forward calls clipk.siglip.siglip_loss: bf16
    operands run on the clipk_siglip kernels without the [b, N] logits, everything else on the materialising formula.
    The loss and the logit_scale / logit_bias gradients are per rank, as in open_clip; `bidir` only chooses open_clip's
    communication pattern, so it changes no value here (the text rows are all-gathered with NCCL either way)."""

    def __init__(self, cache_labels=False, rank=0, world_size=1, bidir=True, use_horovod=False):
        super().__init__()
        if use_horovod:
            raise NotImplementedError("clipk: use_horovod=True is not supported")
        self.cache_labels = cache_labels
        self.rank = rank
        self.world_size = world_size
        self.bidir = bidir
        self.use_horovod = use_horovod
        self.prev_num_logits = 0
        self.labels = {}
        self.group = None

    set_process_group = ClipLoss.set_process_group

    def get_ground_truth(self, device, dtype, num_logits, negative_only=False) -> torch.Tensor:
        """-1 everywhere, +1 on the diagonal unless negative_only (open_clip's labels of one block)."""
        labels = -torch.ones((num_logits, num_logits), device=device, dtype=dtype)
        if not negative_only:
            labels = 2 * torch.eye(num_logits, device=device, dtype=dtype) + labels
        return labels

    def get_logits(self, image_features, text_features, logit_scale, logit_bias=None):
        """Materialised logits of one block: logit_scale * I @ T^T (+ logit_bias)."""
        logits = logit_scale * image_features @ text_features.T
        if logit_bias is not None:
            logits = logits + logit_bias
        return logits

    def forward(self, image_features, text_features, logit_scale, logit_bias, output_dict=False):
        loss = siglip_loss(image_features, text_features, logit_scale, logit_bias, self.rank, self.world_size, self.group)
        return {"contrastive_loss": loss} if output_dict else loss


def create_loss(args):
    """Same flag plumbing as the reference factory (factory.py:250-278); cache_labels is always on there.  --siglip
    (open_clip >= 2.21) returns SigLipLoss, checked after the distill and coca branches as open_clip does."""
    common = dict(local_loss=args.local_loss, gather_with_grad=args.gather_with_grad, cache_labels=True,
                  rank=args.rank, world_size=args.world_size, use_horovod=args.horovod)
    if getattr(args, "distill", False):
        return DistillClipLoss(**common)
    if "coca" in args.model.lower():
        return CoCaLoss(caption_loss_weight=args.coca_caption_loss_weight,
                        clip_loss_weight=args.coca_contrastive_loss_weight, **common)
    if getattr(args, "siglip", False):
        return SigLipLoss(rank=args.rank, world_size=args.world_size)
    return ClipLoss(**common)
