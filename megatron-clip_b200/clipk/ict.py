"""One-directional retrieval loss of the reference's ICT pre-training (pretrain_ict.py:73-114) on the fused kernels.

The reference all-gathers the query and the context embeddings over the data-parallel group (pretrain_ict.py:45-70: the
backward of that gather hands every rank only ITS OWN chunk of the gradient, no reduction), forms the full
N x N score matrix `all_query @ all_context.T` on EVERY rank, takes log_softmax over the rows, the NLL of the diagonal,
multiplies the loss by the data-parallel world size and reports the loss and top-k retrieval accuracies averaged over
the group.  Only one direction (query -> context) is normalised, so this is the row half of ClipLoss:

    loss_r  = W / N * sum_i (lse_i - S_ii)                      (identical on all ranks; i over ALL N queries)
    dq_loc  = 1/b * (P - Id)[R_r, :]  @ c_all                   P = softmax over rows, R_r = this rank's rows
    dc_loc  = 1/b * (P - Id)[:, R_r]^T @ q_all

Here every rank evaluates only its own b x N row block for the statistics and dq (clipk_fwd_stats, clipk_bwd with
alpha = 1, beta = 0) and its own N x b column block for dc - which, transposed, is the same kernel with the roles of the
operands swapped and the ROW log-sum-exps of all N queries in the place of the column ones (alpha = 0, beta = 1).  No
N x N matrix exists anywhere; the work per rank is 10 b N d FLOP instead of the reference's 6 N^2 d.
"""
from __future__ import annotations

import math

import torch
import torch.distributed as dist

from . import ops
from .ops import _all_gather_rows


class _IctLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, query, context, score_scale, rank, world, group):
        be = ops._backend()
        if query.dim() != 2 or query.shape != context.shape or query.dtype != context.dtype:
            raise ValueError("query and context embeddings must both be [batch, dim] of one dtype")
        b, d_in = query.shape
        N = world * b
        dev = query.device
        in_dtype = query.dtype
        q, c = ops._kernel_features(query.detach()), ops._kernel_features(context.detach())
        scale = torch.tensor([float(score_scale)], dtype=torch.float32, device=dev)
        q_all = _all_gather_rows(q, world, group) if world > 1 else q
        c_all = _all_gather_rows(c, world, group) if world > 1 else c
        Xq, Xc = be.prepare(q), be.prepare(c)
        Yq, Yc = (be.prepare(q_all), be.prepare(c_all)) if world > 1 else (Xq, Xc)
        off = rank * b if world > 1 else 0
        stats, pos = be.fwd_stats(Xq, Yc, scale, off, True)          # rows: this rank's queries against all contexts
        lse = stats[0] + stats[1].log()
        part = (lse - pos).sum().reshape(1)
        lse_all = _all_gather_rows(lse, world, group) if world > 1 else lse
        if world > 1:
            dist.all_reduce(part, group=group)
        # mean over all N rows, then "loss * data_parallel_world_size" (pretrain_ict.py:104)
        loss = part[0] / N * world
        ctx.save_for_backward(query, context, scale, lse, lse_all)
        ctx.operands = (Xq, Xc, Yq, Yc)
        ctx.cfg = (b, d_in, off, world, in_dtype)
        ctx.pos = pos
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        be = ops._backend()
        _, _, scale, lse, lse_all = ctx.saved_tensors
        Xq, Xc, Yq, Yc = ctx.operands
        b, d_in, off, world, in_dtype = ctx.cfg
        # d loss / d S_ij = W / N * (P - Id)_ij = (P - Id)_ij / b
        gscale = (grad_out.detach().to(torch.float32).reshape(1) / b).contiguous()
        Gq, Gc = be.prepare_grad(Xq), be.prepare_grad(Xc)
        GYq, GYc = (be.prepare_grad(Yq), be.prepare_grad(Yc)) if world > 1 else (Gq, Gc)
        dq = dc = None
        if ctx.needs_input_grad[0]:
            # block [b queries x N contexts], softmax over its rows: alpha = 1 (lse of this rank's queries), beta = 0
            dq, _ = be.bwd(Xq, Yc, Gq, GYc, scale, off, lse, lse_all, 1.0, 0.0, gscale, True, False)
        if ctx.needs_input_grad[1]:
            # block [b contexts x N queries] = the transposed column block: the softmax runs over ITS columns' index, so
            # the log-sum-exps of all N queries take the column slot: alpha = 0, beta = 1
            dc, _ = be.bwd(Xc, Yq, Gc, GYq, scale, off, lse, lse_all, 0.0, 1.0, gscale, True, False)
        dq, dc = (None if g is None else ops._caller_grad(be, g, d_in, in_dtype) for g in (dq, dc))
        return dq, dc, None, None, None, None


def ict_retrieval_loss(query_logits, context_logits, retriever_score_scaling=False, hidden_size=None, group=None,
                       report_topk_accuracies=()):
    """`loss_func` of pretrain_ict.py:73-114 for one rank's (query, context) embeddings: returns (loss, stats_dict) with
    loss already multiplied by the data-parallel world size and stats_dict = {"loss": averaged loss, "top{k}_acc": %}.

    group: the data-parallel group (pretrain_ict.py:36-42 uses mpu.get_data_parallel_group()); None = WORLD."""
    distributed = dist.is_available() and dist.is_initialized()
    world = dist.get_world_size(group) if distributed else 1
    rank = dist.get_rank(group) if distributed else 0
    score_scale = 1.0
    if retriever_score_scaling:
        if hidden_size is None:
            raise ValueError("retriever_score_scaling needs hidden_size (args.hidden_size of the reference)")
        score_scale = 1.0 / math.sqrt(hidden_size)
    loss = _IctLoss.apply(query_logits, context_logits, score_scale, rank, world, group)
    stats = [(loss.detach() / world).reshape(1)]
    if report_topk_accuracies:
        from . import metrics
        with torch.no_grad():
            c_all = _all_gather_rows(context_logits.detach().contiguous(), world, group) if world > 1 else context_logits.detach()
            ranks = metrics.target_ranks(query_logits.detach(), c_all, diag_offset=rank * query_logits.shape[0])
            for k in report_topk_accuracies:
                stats.append((ranks < int(k)).float().mean().reshape(1))
    averaged = torch.cat(stats)
    if distributed:
        dist.all_reduce(averaged, group=group)
        averaged = averaged / world
    out = {"loss": averaged[0]}
    for i, k in enumerate(report_topk_accuracies):
        out[f"top{k}_acc"] = averaged[1 + i] * 100
    return loss, out
