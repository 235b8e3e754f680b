"""CPU oracle for the ClipLoss / gather_features hot path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import this file.  The product (``megatron-clip_b200/clipk``) never does: it fails loudly when the CUDA
library is missing.

Parity status: PINNED.  The reference's own tests hold no golden value for this path
(open_CLIP/tests/test_training_simple.py only checks "does not crash"), so the oracle is pinned against
outputs of the reference itself: ``tests/golden/make_golden.py`` imports the unmodified
``/root/reference/open_CLIP/src/open_clip/loss.py`` (single process and gloo world sizes 2 and 4, all four
``(local_loss, gather_with_grad)`` modes) and stores its loss / gradients in ``tests/golden/*.npz``;
``tests/test_oracle_cpu.py`` checks every function below against those files.

Two restatements live here:

* ``clip_loss_world`` - numpy float64, written from the data flow of the reference (which tensor is matmul'ed
  with which, which gradient is routed where by the collectives), not from torch autograd.  This is the checker.
* ``TorchPort`` - the same forward written with torch CPU ops (matmul + cross_entropy + autograd), i.e. the
  arithmetic the reference executes on host cores.  ``bench.py`` times it as the CPU baseline ("port").

The numerics of the reference live in PyTorch (torch.matmul, F.cross_entropy, torch.distributed.nn.all_gather;
pinned by the reference at torch==2.0.1, requirements.txt:40; 2.11.0 here), called from
open_CLIP/src/open_clip/loss.py:50-51,55-56,112-119,135-138.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence

import numpy as np


# --------------------------------------------------------------------------------------------------------------
# labels  (reference: open_CLIP/src/open_clip/loss.py:91-102, ClipLoss.get_ground_truth)
# --------------------------------------------------------------------------------------------------------------
def ground_truth(num_logits: int, rank: int = 0, world_size: int = 1, local_loss: bool = False) -> np.ndarray:
    """int64 labels; offset by num_logits*rank only when world_size>1 and local_loss (loss.py:95-96)."""
    labels = np.arange(num_logits, dtype=np.int64)
    if world_size > 1 and local_loss:
        labels = labels + np.int64(num_logits) * np.int64(rank)
    return labels


# --------------------------------------------------------------------------------------------------------------
# gather  (reference: loss.py:20-64, gather_features) - values only; the gradient routing is in clip_loss_world
# --------------------------------------------------------------------------------------------------------------
def gather_features(per_rank: Sequence[np.ndarray]) -> np.ndarray:
    """Rank-major concatenation: rows r*b..(r+1)*b come from rank r (loss.py:50-51 / :61-62)."""
    return np.concatenate([np.asarray(x) for x in per_rank], axis=0)


def _logsumexp_rows(a: np.ndarray) -> np.ndarray:
    m = a.max(axis=1, keepdims=True)
    return (m + np.log(np.exp(a - m).sum(axis=1, keepdims=True)))[:, 0]


def _ce_mean_and_grad(logits: np.ndarray, labels: np.ndarray):
    """mean cross entropy over rows and d(mean CE)/d(logits)  (F.cross_entropy, loss.py:135-138)."""
    n = logits.shape[0]
    lse = _logsumexp_rows(logits)
    loss = float(np.mean(lse - logits[np.arange(n), labels]))
    p = np.exp(logits - lse[:, None])
    p[np.arange(n), labels] -= 1.0
    return loss, p / n


@dataclass
class RankResult:
    loss: float
    d_image: np.ndarray   # [b, d] gradient wrt this rank's image_features
    d_text: np.ndarray    # [b, d] gradient wrt this rank's text_features
    d_scale: float        # gradient wrt logit_scale on this rank (never all-reduced by the loss)
    labels: np.ndarray    # int64 labels used on this rank


def clip_loss_world(images: Sequence[np.ndarray], texts: Sequence[np.ndarray], logit_scale: float,
                    local_loss: bool = False, gather_with_grad: bool = False,
                    grad_output: float = 1.0) -> List[RankResult]:
    """float64 loss and gradients of ClipLoss.forward on every rank of a world.

    ``images[r]`` / ``texts[r]`` are rank r's local [b, d] features.  World size 1 follows loss.py:117-119;
    world size > 1 follows loss.py:105-116 for the logits and loss.py:48-62 for which gathered gradient
    reaches which rank:

    * gather_with_grad=True : torch.distributed.nn.all_gather, whose backward is a reduce-scatter SUM, so rank q
      receives the sum over all ranks r of rank r's gradient on chunk q of the gathered tensor (loss.py:50-51).
    * gather_with_grad=False, local_loss=False: the own chunk is replaced by the live tensor (loss.py:57-60), so
      rank q receives only its own gradient on chunk q.
    * gather_with_grad=False, local_loss=True : gathered tensors carry no gradient at all.
    """
    W = len(images)
    assert len(texts) == W
    I = [np.asarray(x, dtype=np.float64) for x in images]
    T = [np.asarray(x, dtype=np.float64) for x in texts]
    b, d = I[0].shape
    s = float(logit_scale)
    go = float(grad_output)

    if W == 1:
        A = s * I[0] @ T[0].T          # logits_per_image (loss.py:118)
        B = s * T[0] @ I[0].T          # logits_per_text  (loss.py:119)
        labels = ground_truth(b)
        la, dA = _ce_mean_and_grad(A, labels)
        lb, dB = _ce_mean_and_grad(B, labels)
        dA *= go / 2
        dB *= go / 2
        dI = s * (dA @ T[0] + dB.T @ T[0])
        dT = s * (dA.T @ I[0] + dB @ I[0])
        ds = float(np.sum(dA * (I[0] @ T[0].T)) + np.sum(dB * (T[0] @ I[0].T)))
        return [RankResult((la + lb) / 2, dI, dT, ds, labels)]

    I_all = gather_features(I)
    T_all = gather_features(T)
    N = W * b
    # per-rank gradients on (local I, local T, gathered I, gathered T) before the collectives' backward
    g_loc_I = [np.zeros((b, d)) for _ in range(W)]
    g_loc_T = [np.zeros((b, d)) for _ in range(W)]
    g_all_I = [np.zeros((N, d)) for _ in range(W)]
    g_all_T = [np.zeros((N, d)) for _ in range(W)]
    losses, dss, labs = [], [], []
    for r in range(W):
        if local_loss:
            A = s * I[r] @ T_all.T     # loss.py:112
            B = s * T[r] @ I_all.T     # loss.py:113
            labels = ground_truth(b, r, W, True)
            la, dA = _ce_mean_and_grad(A, labels)
            lb, dB = _ce_mean_and_grad(B, labels)
            dA *= go / 2
            dB *= go / 2
            g_loc_I[r] += s * dA @ T_all
            g_all_T[r] += s * dA.T @ I[r]
            g_loc_T[r] += s * dB @ I_all
            g_all_I[r] += s * dB.T @ T[r]
            ds = float(np.sum(dA * (I[r] @ T_all.T)) + np.sum(dB * (T[r] @ I_all.T)))
        else:
            A = s * I_all @ T_all.T    # loss.py:115
            labels = ground_truth(N, r, W, False)
            la, dA = _ce_mean_and_grad(A, labels)
            lb, dB = _ce_mean_and_grad(A.T, labels)   # logits_per_text = logits_per_image.T (loss.py:116)
            dA = (dA + dB.T) * (go / 2)
            g_all_I[r] += s * dA @ T_all
            g_all_T[r] += s * dA.T @ I_all
            ds = float(np.sum(dA * (I_all @ T_all.T)))
        losses.append((la + lb) / 2)
        dss.append(ds)
        labs.append(labels)

    out = []
    for q in range(W):
        sl = slice(q * b, (q + 1) * b)
        dI = g_loc_I[q].copy()
        dT = g_loc_T[q].copy()
        if gather_with_grad:
            for r in range(W):
                dI += g_all_I[r][sl]
                dT += g_all_T[r][sl]
        elif not local_loss:
            dI += g_all_I[q][sl]
            dT += g_all_T[q][sl]
        out.append(RankResult(losses[q], dI, dT, dss[q], labs[q]))
    return out


def clip_loss_single(image: np.ndarray, text: np.ndarray, logit_scale: float, grad_output: float = 1.0) -> RankResult:
    return clip_loss_world([image], [text], logit_scale, grad_output=grad_output)[0]


def round_to_bf16(x: np.ndarray) -> np.ndarray:
    """Round-to-nearest-even float32 -> bfloat16 -> float32, in numpy (used to build bf16 test inputs)."""
    u = np.asarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


# --------------------------------------------------------------------------------------------------------------
# torch CPU port: what the reference executes on host cores.  Timed by bench.py as the CPU baseline.
# --------------------------------------------------------------------------------------------------------------
class TorchPort:
    """Single-process (world_size == 1) forward of ClipLoss with torch CPU ops; backward by autograd.

    Mirrors the op sequence of loss.py:117-119 (two matmuls with the scale on the left operand) and
    loss.py:135-138 (two mean cross-entropies, halved), plus the arange label cache of loss.py:91-102.
    """

    def __init__(self):
        self._labels = None

    def labels(self, n: int, device=None):
        import torch
        if self._labels is None or self._labels.numel() != n or self._labels.device != torch.device(device or "cpu"):
            self._labels = torch.arange(n, dtype=torch.long, device=device)
        return self._labels

    def __call__(self, image_features, text_features, logit_scale):
        import torch.nn.functional as F
        a = logit_scale * image_features @ text_features.T
        b = logit_scale * text_features @ image_features.T
        y = self.labels(a.shape[0], a.device)
        return (F.cross_entropy(a, y) + F.cross_entropy(b, y)) / 2

    def fwd_bwd(self, image_features, text_features, logit_scale):
        """One 'step' of the metric: forward + backward; returns (loss, dI, dT, ds) as tensors."""
        import torch
        i = image_features.detach().requires_grad_(True)
        t = text_features.detach().requires_grad_(True)
        s = logit_scale.detach().requires_grad_(True)
        loss = self(i, t, s)
        loss.backward()
        return loss.detach(), i.grad, t.grad, s.grad


def synthetic_features(b: int, d: int, seed: int, rank: int = 0):
    """The synthetic workload of SURVEY.md section 8(d): positives at cos~0.3, negatives ~N(0, 1/d).

    numpy float32; identical on any box (numpy's PCG64 stream), so CPU and GPU arms see the same values.
    """
    rng = np.random.default_rng(seed + rank)
    x = rng.standard_normal((b, d), dtype=np.float32)
    z = rng.standard_normal((b, d), dtype=np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    z /= np.linalg.norm(z, axis=1, keepdims=True)
    t = 0.3 * x + 0.954 * z
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    return x.astype(np.float32), t.astype(np.float32)


def distill_loss_single(image, text, logit_scale, t_image, t_text, t_logit_scale, grad_output=1.0):
    """float64 distillation term of DistillClipLoss.forward, single process (reference loss.py:187-189, 200-216):
        dist_loss(t, s) = -(softmax(t, 1) * log_softmax(s, 1)).sum(1).mean(0),
        distill_loss = (dist_loss(teacher per-image, student per-image) + dist_loss(teacher per-text, student per-text)) / 2
    Returns (loss, d_image, d_text, d_scale) with respect to the STUDENT (the teacher carries no gradient)."""
    I, T = np.asarray(image, dtype=np.float64), np.asarray(text, dtype=np.float64)
    tI, tT = np.asarray(t_image, dtype=np.float64), np.asarray(t_text, dtype=np.float64)
    s, ts, go = float(logit_scale), float(t_logit_scale), float(grad_output)
    n = I.shape[0]
    C = I @ T.T
    S = s * C                                  # student logits_per_image (loss.py:118); per_text is its transpose
    Tl = ts * tI @ tT.T

    def softmax(x, axis):
        e = np.exp(x - x.max(axis=axis, keepdims=True))
        return e / e.sum(axis=axis, keepdims=True)

    def lse(x, axis):
        m = x.max(axis=axis)
        return m + np.log(np.exp(x - np.expand_dims(m, axis)).sum(axis=axis))

    loss = ((lse(S, 1) - (softmax(Tl, 1) * S).sum(1)).mean() + (lse(S, 0) - (softmax(Tl, 0) * S).sum(0)).mean()) / 2
    G = (softmax(S, 1) - softmax(Tl, 1) + softmax(S, 0) - softmax(Tl, 0)) * (go / (2 * n))     # dloss / dS
    return loss, s * G @ T, s * G.T @ I, float((G * C).sum())
