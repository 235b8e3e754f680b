"""float64 numpy oracle of open_clip's SigLipLoss (open_clip >= 2.21, loss.py), per data-parallel rank.

Rank r of W holds b rows of image features x_i and text features y_i; N = W*b, off = r*b, Y_all = all ranks' text rows in
rank-major order, s = logit_scale (already exponentiated), t = logit_bias, go = grad_output:

    l_ij   = s x_i.y_j + t                           i < b, j < N
    z_ij   = +1 if j == off + i else -1
    loss_r = (1/b) sum_ij softplus(-z_ij l_ij)          per rank, not reduced
    g_ij   = sigma(l_ij) - [j == off + i]
    dx_i   = go (s/b) sum_j g_ij y_j
    dY_r   = go (s/b) sum_i g_ij x_i                    [N, d]; d_text of rank r = sum over ranks of rows [off, off + b)
    ds     = go (1/b) sum_ij g_ij x_i.y_j,   dt = go (1/b) sum_ij g_ij        (per rank)
"""
from collections import namedtuple

import numpy as np
from scipy.special import expit

SigLipGrads = namedtuple("SigLipGrads", "loss d_image d_text d_scale d_bias")


def siglip_world(images, texts, logit_scale, logit_bias=0.0, grad_output=1.0):
    """images, texts: one [b, d] array per rank.  Returns one SigLipGrads per rank (float64)."""
    X_all = [np.asarray(x, dtype=np.float64) for x in images]
    Y = np.concatenate([np.asarray(t, dtype=np.float64) for t in texts])
    W, (b, d) = len(X_all), X_all[0].shape
    s, t, go = float(logit_scale), float(logit_bias), float(grad_output)
    idx = np.arange(b)
    per_rank, d_text = [], np.zeros((W * b, d))
    for r, X in enumerate(X_all):
        off = r * b
        dots = X @ Y.T
        L = s * dots + t
        z = -np.ones_like(L)
        z[idx, idx + off] = 1.0
        loss = np.logaddexp(0.0, -z * L).sum() / b
        G = expit(L)
        G[idx, idx + off] = -expit(-L[idx, idx + off])      # sigma(l) - 1 without the cancellation
        d_image = go * s / b * (G @ Y)
        d_text += go * s / b * (G.T @ X)
        per_rank.append((loss, d_image, go / b * (G * dots).sum(), go / b * G.sum()))
    return [SigLipGrads(loss, d_image, d_text[r * b:(r + 1) * b], ds, dt)
            for r, (loss, d_image, ds, dt) in enumerate(per_rank)]


def siglip_single(image, text, logit_scale, logit_bias=0.0, grad_output=1.0):
    return siglip_world([image], [text], logit_scale, logit_bias, grad_output)[0]


def siglip_block(image, text_all, logit_scale, logit_bias=0.0, grad_output=1.0, diag_offset=0):
    """One rank's block as clipk_siglip_forward / _backward see it: image [b, d], text_all [N, d] (every rank's text
    rows), the positive of row i at column diag_offset + i.  Returns SigLipGrads whose d_text is the block's UNREDUCED
    [N, d] partial go (s/b) G^T X; summing the blocks of all ranks and taking rows [r*b, (r+1)*b) gives siglip_world's
    d_text of rank r."""
    X, Y = np.asarray(image, dtype=np.float64), np.asarray(text_all, dtype=np.float64)
    b, N = X.shape[0], Y.shape[0]
    s, t, go = float(logit_scale), float(logit_bias), float(grad_output)
    i, j = np.arange(b), np.arange(b) + int(diag_offset)
    assert 0 <= diag_offset and diag_offset + b <= N
    dots = X @ Y.T
    L = s * dots + t
    z = -np.ones_like(L)
    z[i, j] = 1.0
    G = expit(L)
    G[i, j] = -expit(-L[i, j])
    return SigLipGrads(np.logaddexp(0.0, -z * L).sum() / b, go * s / b * (G @ Y), go * s / b * (G.T @ X),
                       go / b * (G * dots).sum(), go / b * G.sum())
