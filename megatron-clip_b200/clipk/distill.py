"""Distillation term of DistillClipLoss (reference loss.py:187-216) without the four materialised logit matrices.

    dist_loss(teacher_logits, student_logits) = -(softmax(teacher) * log_softmax(student)).sum(1).mean(0)     loss.py:188-189
                                              = mean_i [ lse(S_i) - sum_j softmax(T_i)(j) * S_ij ]

taken in both directions (rows: image -> text, columns: text -> image) and halved (loss.py:212-215).  The log-sum-exps
of the student's and of the teacher's logits come from the fused forward sweep of each model (clipk_fwd_both); only the
cross term needs both logits of an element at once.  It is read from pairs of bounded fp32 panels made on the tensor
cores (clipk_gemm16, <= PANEL_BYTES each) - rows x N at a time instead of N x N x 4 matrices plus their softmax
temporaries.  The backward recomputes the panels, forms
    G = P_row(S) - P_row(T) + P_col(S) - P_col(T)          (fp16 x 2^14, clipk_distill_grad)
and multiplies it into the student's features with the same fp16 gradient GEMMs as the loss (dI = G T, dT = G^T I);
dlogit_scale needs no backward pass: d lse/ds = E/s and d cross/ds = cross/s, both known from the forward.

Scope: single process (world_size == 1), bf16 features (fp32 features under bf16 autocast are cast like the loss does).
Everything else stays on the reference's materialising formula in clipk/loss.py.
Verified against the oracle on a B200 (tests/test_distill_gpu.py) and on the CPU emulation of the kernel entries
(tests/test_distill_cpu.py); default for the shapes `applicable` accepts, CLIPK_FUSED_DISTILL=0 switches it off.
"""
from __future__ import annotations

import torch

from . import ops

PANEL_BYTES = 256 << 20


def _panel_rows(rows, cols4, panel_bytes):
    per = max(256, panel_bytes // (4 * cols4) // 256 * 256)
    return min(per, rows, 65535 // 256 * 256)


class _Model:
    """One model's side of the term: operands, log-sum-exps and the scalar that turns raw panel products into logits."""

    def __init__(self, be, image, text, scale, cols4):
        dev = image.device
        n = image.shape[0]
        self.scale = scale.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        self.image, self.text = ops._kernel_features(image), ops._kernel_features(text)
        X, Y = be.prepare(self.image), be.prepare(self.text)
        parts = torch.empty(1, 3, n, dtype=torch.float32, device=dev)
        row_stats, pos, _ = be.fwd_both(X, Y, self.scale, 0, col_out=parts[0])
        self.lse_row, self.lse_col, _ = be.finalize(row_stats, pos, parts, 0)
        # expected logit under the row / column softmax (dot / sum of the sweep's statistics)
        self.e_row = row_stats[2] / row_stats[1]
        self.e_col = parts[0, 2] / parts[0, 1]
        keys = self.text if cols4 == n else torch.nn.functional.pad(self.text, (0, 0, 0, cols4 - n))
        self.Q, self.K = be.dense_operand(self.image), be.dense_operand(keys)
        self.mul = self.scale              # bf16 operands carry no power-of-two scale: logits = raw product * logit_scale


class _DistillTerm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image, text, scale, t_image, t_text, t_scale, panel_bytes):
        be = ops._backend()
        n, width = image.shape
        dev = image.device
        cols4 = (n + 3) // 4 * 4
        stu = _Model(be, image.detach(), text.detach(), scale, cols4)
        tea = _Model(be, t_image.detach(), t_text.detach(), t_scale, cols4)
        per = _panel_rows(n, cols4, panel_bytes)
        S = torch.empty(per, cols4, dtype=torch.float32, device=dev)
        T = torch.empty(per, cols4, dtype=torch.float32, device=dev)
        npanels = (n + per - 1) // per
        row_cross = torch.empty(n, dtype=torch.float32, device=dev)
        col_parts = torch.empty(npanels, n, dtype=torch.float32, device=dev)
        for p in range(npanels):
            r0 = p * per
            m = min(per, n - r0)
            be.logits_panel(stu.Q, stu.K, r0, m, S)
            be.logits_panel(tea.Q, tea.K, r0, m, T)
            be.distill_cross(S, T, m, n, stu.mul, tea.mul, tea.lse_row, tea.lse_col, r0, row_cross, col_parts[p])
        col_cross = col_parts.sum(dim=0)
        loss = ((stu.lse_row - row_cross).mean() + (stu.lse_col - col_cross).mean()) / 2
        # s * dloss/ds: d lse/ds = E / s and d cross/ds = cross / s
        s_dloss = ((stu.e_row - row_cross).mean() + (stu.e_col - col_cross).mean()) / 2
        ctx.save_for_backward(stu.lse_row, stu.lse_col, tea.lse_row, tea.lse_col, stu.scale, s_dloss)
        ctx.models = (stu, tea)
        ctx.cfg = (n, width, cols4, per, image.dtype, tuple(scale.shape), scale.dtype)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        be = ops._backend()
        s_lr, s_lc, t_lr, t_lc, s_scale, s_dloss = ctx.saved_tensors
        stu, tea = ctx.models
        n, width, cols4, per, in_dtype, scale_shape, scale_dtype = ctx.cfg
        go = grad_out.detach().to(torch.float32).reshape(1)
        d_image = d_text = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            dev = s_lr.device
            image16, inv_i = be.grad_operand(stu.image)        # exact fp16 copies of the student's bf16 features
            text16, inv_t = be.grad_operand(stu.text)
            dpad = image16.shape[1]
            S = torch.empty(per, cols4, dtype=torch.float32, device=dev)
            T = torch.empty(per, cols4, dtype=torch.float32, device=dev)
            G = torch.empty(per, (n + 7) // 8 * 8, dtype=torch.float16, device=dev)
            dX = torch.empty(n, dpad, dtype=torch.float32, device=dev)
            dY = torch.empty(n, dpad, dtype=torch.float32, device=dev)
            for p in range((n + per - 1) // per):
                r0 = p * per
                m = min(per, n - r0)
                be.logits_panel(stu.Q, stu.K, r0, m, S)
                be.logits_panel(tea.Q, tea.K, r0, m, T)
                be.distill_grad(S, T, m, n, stu.mul, tea.mul, s_lr, t_lr, s_lc, t_lc, r0, G)
                Gp = G[:m, :n]
                be.gemm(Gp, text16, dX[r0:r0 + m], False, True, True, False)      # dX rows     = G   [m x n] . text
                be.gemm(Gp, image16[r0:r0 + m], dY, True, True, True, p > 0)      # dY (+)=       G^T [n x m] . image rows
            coef = go * s_scale / (2.0 * n * 16384.0)
            d_image = (dX[:, :width] * (coef * inv_t)).to(in_dtype)
            d_text = (dY[:, :width] * (coef * inv_i)).to(in_dtype)
        d_scale = None
        if ctx.needs_input_grad[2]:
            d_scale = (s_dloss * go[0] / s_scale[0]).reshape(scale_shape).to(scale_dtype)
        return d_image, d_text, d_scale, None, None, None, None


def applicable(image_features, text_features, dist_image_features, dist_text_features, world_size):
    """True when the panel path handles this call; otherwise DistillClipLoss keeps the materialising formula."""
    feats = (image_features, text_features, dist_image_features, dist_text_features)
    if world_size != 1 or any(f.dim() != 2 or f.shape[0] != image_features.shape[0] or f.shape[0] == 0 for f in feats):
        return False
    if image_features.shape != text_features.shape or dist_image_features.shape != dist_text_features.shape:
        return False
    autocast_bf16 = ops._autocast_bf16(image_features.device)
    return all(f.dtype == torch.bfloat16 or (autocast_bf16 and f.dtype == torch.float32) for f in feats)


def fused_distill_term(image_features, text_features, logit_scale, dist_image_features, dist_text_features,
                       dist_logit_scale, panel_bytes=PANEL_BYTES):
    """(dist_loss(teacher per-image, student per-image) + dist_loss(teacher per-text, student per-text)) / 2
    (loss.py:212-215), differentiable with respect to the student's features and logit_scale."""
    dev = image_features.device

    def as_scale(s):
        return s if isinstance(s, torch.Tensor) else torch.tensor(float(s), dtype=torch.float32, device=dev)

    def bf16(x):
        return x if x.dtype == torch.bfloat16 else x.to(torch.bfloat16)

    return _DistillTerm.apply(bf16(image_features), bf16(text_features), as_scale(logit_scale),
                              bf16(dist_image_features), bf16(dist_text_features), as_scale(dist_logit_scale),
                              panel_bytes)
