"""SigLipLoss's pairwise sigmoid loss (open_clip >= 2.21, loss.py SigLipLoss) without the b x N logits.

On rank r of W (b local rows, N = W*b, off = r*b), with s = logit_scale (already exponentiated) and t = logit_bias:

    l_ij = s x_i.y_j + t,   z_ij = +1 if j == off + i else -1,   loss_r = (1/b) sum_ij softplus(-z_ij l_ij)

which is what open_clip's forward computes: its own block with labels 2*eye - 1 plus the W - 1 neighbour blocks with
negative-only labels, every block divided by b.  The loss and dlogit_scale / dlogit_bias are per rank (not reduced: DDP
averages them); the text gradient of rank r sums every rank's gradient on its rows, as neighbour_exchange_with_grad
sends them back.

Two routes, decided once in siglip_loss:
  kernels  bf16 operands on CUDA (bf16 features, or fp32 under bf16 autocast, cast once): clipk_siglip_forward /
           clipk_siglip_backward on the features padded to whole 64-column blocks (_kernel_features), the text rows of
           all ranks gathered with NCCL before the forward and the fp32 text gradient reduce-scattered after the backward.
  formula  everything else (fp32 outside autocast, fp16 features, fp32 under fp16 autocast): open_clip's formula in
           torch on MATERIALISED logits, a [b, N] matrix per call.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import ops
from .ops import (_FEATURE_DTYPES, _GatherRowsWithGrad, _all_gather_rows, _autocast_bf16, _backend, _caller_grad,
                  _kernel_features, _reduce_scatter_rows)


def _scalar(v, dev):
    return v.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()


class _SigLipKernels(torch.autograd.Function):
    """The kernel route: one clipk_siglip_forward and one clipk_siglip_backward per call."""

    @staticmethod
    def forward(ctx, image_features, text_features, logit_scale, logit_bias, rank, world_size, group):
        be = _backend()
        b, d_in = image_features.shape
        W = int(world_size)
        dev = image_features.device
        img, txt = image_features.detach(), text_features.detach()
        if img.dtype == torch.float32:          # bf16 autocast: the matmul runs on bf16 operands
            img, txt = img.to(torch.bfloat16), txt.to(torch.bfloat16)
        X, Yl = _kernel_features(img), _kernel_features(txt)
        Y = _all_gather_rows(Yl, W, group) if W > 1 else Yl
        scale = _scalar(logit_scale, dev)
        bias = None if logit_bias is None else _scalar(logit_bias, dev)
        off = rank * b if W > 1 else 0
        loss, state = be.siglip_forward(X, Y, scale, bias, off)
        # the inputs themselves are saved so that autograd notices an in-place change before the backward reads them
        ctx.save_for_backward(image_features, text_features)
        ctx.ops = (X, Y, scale, bias, state)
        ctx.cfg = (W, off, group, image_features.dtype, d_in, logit_scale.dtype, logit_scale.shape,
                   None if logit_bias is None else (logit_bias.dtype, logit_bias.shape))
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        _ = ctx.saved_tensors            # raises if the features were modified in place since the forward
        be = _backend()
        X, Y, scale, bias, state = ctx.ops
        W, off, group, in_dtype, d_in, s_dtype, s_shape, b_meta = ctx.cfg
        want_feat = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        want_s, want_t = ctx.needs_input_grad[2], bias is not None and ctx.needs_input_grad[3]
        go = grad_out.detach().to(torch.float32).reshape(1).contiguous()
        dX, dY, ds, dt = be.siglip_backward(X, Y, scale, bias, off, state, go, want_feat, want_feat, want_s, want_t)
        d_image = d_text = d_scale = d_bias = None
        if want_feat:
            dT = _reduce_scatter_rows(dY, W, group) if W > 1 else dY
            d_image, d_text = _caller_grad(be, dX, d_in, in_dtype), _caller_grad(be, dT, d_in, in_dtype)
        if want_s:
            d_scale = ds.reshape(s_shape).to(s_dtype)
        if want_t:
            d_bias = dt.reshape(b_meta[1]).to(b_meta[0])
        ctx.ops = None
        return d_image, d_text, d_scale, d_bias, None, None, None


def siglip_formula(image_features, text_features, logit_scale, logit_bias=None, rank=0, world_size=1, group=None):
    """open_clip's SigLipLoss forward as a torch expression on materialised [b, N] logits (the formula route).  The
    matmul runs in the features' dtype (or the autocast dtype); the log-sigmoid sum in fp32."""
    b = image_features.shape[0]
    W = int(world_size)
    text_all = _GatherRowsWithGrad.apply(text_features, W, group) if W > 1 else text_features
    logits = (logit_scale * image_features @ text_all.T).float()
    if logit_bias is not None:
        logits = logits + logit_bias
    labels = -torch.ones_like(logits)
    off = rank * b if W > 1 else 0
    idx = torch.arange(b, device=logits.device)
    labels[idx, idx + off] = 1.0
    return -F.logsigmoid(labels * logits).sum() / b


def siglip_loss(image_features, text_features, logit_scale, logit_bias=None, rank=0, world_size=1, group=None):
    """loss = SigLipLoss(rank, world_size).forward(I, T, s, t) of open_clip, on this rank.  Picks the route once, before
    anything is launched: the kernels for bf16 operands (bf16 features, or fp32 under bf16 autocast) on CUDA, the
    materialising formula for everything else.  logit_scale / logit_bias may be Python floats or 0-dim / [1] tensors;
    logit_bias=None means t = 0.  An empty batch returns NaN with empty gradients and launches nothing."""
    if image_features.dim() != 2 or image_features.shape != text_features.shape:
        raise ValueError("image_features and text_features must both be [batch, dim]")
    if image_features.dtype != text_features.dtype:
        raise TypeError("image_features and text_features must have the same dtype")
    dtype, dev = image_features.dtype, image_features.device
    if dtype not in _FEATURE_DTYPES:
        raise TypeError(f"clipk: unsupported feature dtype {dtype} (bf16, fp16 and fp32 only)")
    if not isinstance(logit_scale, torch.Tensor):
        logit_scale = torch.tensor(float(logit_scale), dtype=torch.float32, device=dev)
    if logit_bias is not None and not isinstance(logit_bias, torch.Tensor):
        logit_bias = torch.tensor(float(logit_bias), dtype=torch.float32, device=dev)
    if image_features.shape[0] == 0:
        nan = (image_features.sum() + text_features.sum()).float() * logit_scale.float().sum() * float("nan")
        return nan if logit_bias is None else nan * logit_bias.float().sum()
    bf16_operands = dtype == torch.bfloat16 or (dtype == torch.float32 and _autocast_bf16(dev))
    if bf16_operands and (dev.type == "cuda" or ops._TEST_BACKEND is not None):
        return _SigLipKernels.apply(image_features, text_features, logit_scale, logit_bias, rank, world_size, group)
    return siglip_formula(image_features, text_features, logit_scale, logit_bias, rank, world_size, group)
