"""The loss's device-side choices at their bounds, against float64 on the exact operand values.

Both passes pick an algorithm on the device from a numeric bound:
  * forward (fwd_bound, csrc/gemm_core.cuh): ONE sweep with the global reference c = u - 90 (log2 units,
    u = |s| max|x_i| max|y_j| log2(e) 1.001) when (a) u <= 96, or (b) every positive logit is >= u - 175 (use_minpos:
    the fused step always, clipk_fwd_both for a square block with diagonal positives); the exact two-sweep form otherwise;
  * backward (grad_prep_kernel, csrc/clipk.cu): the FAST one-ex2 recompute when the spread of all row and column
    log-sum-exps is <= 100 log2 units; the exact form on every tile otherwise.
A bound that is too loose flushes whole rows to zero (forward) or overflows 2^(v - c) (backward); a mean loss within 2e-3
hides one wrong row of a thousand, so everything here is checked per row and per column, and every case asserts which
forward ran and that its inputs sit in the band it targets (at least 0.5 % from the threshold).
"""
import math

import numpy as np
import pytest
import torch

from oracle import cliploss_oracle as O
from tests.test_parity_gpu import TILE_EDGES

pytestmark = pytest.mark.gpu

LOG2E = 1.0 / math.log(2.0)
FWD_SAFE_U, FWD_REF_SHIFT, FWD_POS_MARGIN = 96.0, 90.0, 175.0      # gemm_core.cuh
FAST_SPREAD = 100.0                                                  # grad_prep_kernel, clipk.cu
GUARD = 0.005                                                        # inputs at least 0.5 % from the threshold they target
GRAD_TOL = {torch.bfloat16: 2e-3, torch.float32: 1e-5}


# ------------------------------------------------------------------------------------------------------------ inputs
def _unit(a):
    return a / np.linalg.norm(a, axis=-1, keepdims=True)


def collapsed(n, d, seed, anti=None):
    """Early-training / modality-gap geometry: every text row normalize(t0 + 0.1 z_j), image rows the same except the
    `anti` rows (default: both edges of the first 128-row block and the last row), which are normalize(-t0 + 0.1 z):
    every logit of those rows sits near -u, the worst case for rule (a)."""
    rng = np.random.default_rng(seed)
    t0 = _unit(rng.standard_normal(d))
    x = _unit(t0 + 0.1 * _unit(rng.standard_normal((n, d))))
    t = _unit(t0 + 0.1 * _unit(rng.standard_normal((n, d))))
    anti = [0, 127, 128, n - 1] if anti is None else anti
    x[anti] = _unit(-t0 + 0.1 * _unit(rng.standard_normal((len(anti), d))))
    return x.astype(np.float32), t.astype(np.float32)


BAD_ROWS = (127, 128)


def bad_positives(n, d, cos, seed=21):
    """O.synthetic_features with the positives of BAD_ROWS at cosine `cos`; every other text leans away from the bad
    image rows and every other image away from the bad texts, so that a bad pair's positive is the largest term of its
    row and of its column by far."""
    x, t = O.synthetic_features(n, d, seed=seed)
    rng = np.random.default_rng(seed + 1)
    q, _ = np.linalg.qr(rng.standard_normal((d, 2 * len(BAD_ROWS))))
    e, f = q[:, :len(BAD_ROWS)].T, q[:, len(BAD_ROWS):].T              # orthonormal directions
    k = len(BAD_ROWS)
    raw = cos * math.sqrt(k)                                            # t_i has norm sqrt(k) before normalising
    good = np.setdiff1d(np.arange(n), BAD_ROWS)
    t[good] = _unit(t[good] - 2.0 * e.sum(0))
    x[good] = _unit(x[good] - 2.0 * f.sum(0))
    for a, i in enumerate(BAD_ROWS):
        x[i] = e[a]
        others = e.sum(0) - e[a]
        t[i] = _unit(raw * e[a] + math.sqrt(1.0 - raw * raw) * f[a] - others)
    return x.astype(np.float32), t.astype(np.float32)


def graded(n, d, seed, top=4.5):
    """Rows with graded norms 0.1 .. 6 in the collapsed geometry (every other row anti-aligned, norms up to `top`):
    the row log-sum-exps spread over a couple of hundred log2 units at the initial logit scale."""
    rng = np.random.default_rng(seed)
    t0 = _unit(rng.standard_normal(d))
    t = _unit(t0 + 0.3 * _unit(rng.standard_normal((n, d))))
    sign = np.where(np.arange(n) % 2 == 0, 1.0, -1.0)
    norms = np.where(sign > 0, np.linspace(0.1, 6.0, n), np.linspace(0.1, top, n))
    x = norms[:, None] * _unit(sign[:, None] * t0 + 0.3 * _unit(rng.standard_normal((n, d))))
    return x.astype(np.float32), t.astype(np.float32)


# ------------------------------------------------------------------------------------------------------- the rules
def _expect_single(X, Y, s, use_minpos):
    """fwd_bound on the operand values (torch tensors of any dtype): (single sweep expected, u, relative distance of the
    inputs from rule (a)'s threshold u = 96, relative distance of min_i x_i . y_i from rule (b)'s threshold)."""
    Xd, Yd = X.double(), Y.double()
    u = abs(s) * Xd.pow(2).sum(1).max().sqrt().item() * Yd.pow(2).sum(1).max().sqrt().item() * LOG2E * 1.001
    by_norm = u <= FWD_SAFE_U
    margin_a = abs(u - FWD_SAFE_U) / FWD_SAFE_U
    by_pos, margin_b = False, float("nan")
    if use_minpos:
        minpos = (Xd * Yd[:X.shape[0]]).sum(1).min().item()
        thr = (u - FWD_POS_MARGIN) / (s * LOG2E)
        by_pos = s > 0 and minpos >= thr
        margin_b = abs(minpos - thr) / abs(thr)
    return by_norm or by_pos, u, margin_a, margin_b


def _spread(S):
    """LSE spread of all rows and columns (log2 units): what grad_prep_kernel compares with 100."""
    lse = torch.cat([torch.logsumexp(S, 1), torch.logsumexp(S, 0)])
    return (lse.max() - lse.min()).item() * LOG2E


def _rows_close(got, ref, tol, what):
    """||err_i|| <= tol (||ref_i|| + mean_k ||ref_k||) for every row i; a NaN or Inf anywhere fails (the reference is
    finite: a range failure of the backward shows up as inf * 0 = NaN, which no comparison with a bound would flag)."""
    bad = (~torch.isfinite(got)).any(dim=1).nonzero().flatten()
    assert bad.numel() == 0, (what, "non-finite rows", bad[:8].tolist(), bad.numel())
    err = (got.double() - ref.double()).norm(dim=1)
    rn = ref.double().norm(dim=1)
    bound = tol * (rn + rn.mean())
    ratio = err / bound
    bad = (~(ratio <= 1)).nonzero().flatten()
    assert bad.numel() == 0, (what, bad[:8].tolist(), float(ratio.max()))


# ---------------------------------------------------------------------------------------------- the entry helper
def _run_entry(X, Y, s, off=0, exact=False):
    """clipk_fwd_both -> clipk_finalize -> clipk_bwd, the calls of the general route (X, Y on the GPU)."""
    from clipk import ops
    be = ops._backend()
    Xo, Yo = be.prepare(X), be.prepare(Y)
    sc = torch.tensor([s], device="cuda")
    parts = torch.empty(1, 3, Y.shape[0], dtype=torch.float32, device="cuda")
    rs, pos, _ = be.fwd_both(Xo, Yo, sc, off, col_out=parts[0], exact=exact)
    lse_row, lse_col, _ = be.finalize(rs, pos, parts, off)
    gscale = torch.tensor([1.0 / (2 * X.shape[0])], device="cuda")
    dX, dY = be.bwd(Xo, Yo, be.prepare_grad(Xo), be.prepare_grad(Yo), sc, off, lse_row, lse_col, 1.0, 1.0, gscale,
                    True, True)
    torch.cuda.synchronize()
    return rs, pos, lse_row, lse_col, dX, dY


def check_entry(X, Y, s, off=0, exact=False):
    """Runs the entry calls on X [rows, d], Y [cols, d] (bf16 or fp32, on the GPU) and checks them against float64:
    LSEs and positives elementwise, dX / dY row by row, and which forward ran (the single sweep reports its global
    reference (u - 90) ln 2 in the max plane of every row).  Returns (lse_row, lse_col, single sweep expected, S)."""
    rows, cols = X.shape[0], Y.shape[0]
    rs, pos, lse_row, lse_col, dX, dY = _run_entry(X, Y, s, off, exact)
    S = s * (X.double() @ Y.double().T)
    # test_fwd_both_matches_direct_statistics's tolerance, scaled by the largest logit (= s for unit features): every
    # logit, and so every probability, carries an error relative to that magnitude
    big = max(1.0, s / 14.0, float(S.abs().max()) / 14.0)
    tol = 2e-5 * big
    lr, lc = torch.logsumexp(S, 1), torch.logsumexp(S, 0)
    assert torch.isfinite(lse_row).all() and torch.isfinite(lse_col).all()
    assert torch.allclose(lse_row.double(), lr, rtol=0, atol=tol), ("lse_row", float((lse_row.double() - lr).abs().max()))
    assert torch.allclose(lse_col.double(), lc, rtol=0, atol=tol), ("lse_col", float((lse_col.double() - lc).abs().max()))
    idx = torch.arange(rows, device="cuda")
    ok = (idx + off >= 0) & (idx + off < cols)
    assert torch.allclose(pos[ok].double(), S[idx[ok], idx[ok] + off], rtol=0, atol=tol)

    single = (X.dtype == torch.bfloat16 and not exact and
              _expect_single(X, Y, s, rows == cols and off == 0)[0])
    if single:
        u = _expect_single(X, Y, s, False)[1]
        assert bool((rs[0] == rs[0][0]).all()), "single sweep expected: one global reference in the max plane"
        assert abs(float(rs[0][0]) - (u - FWD_REF_SHIFT) / LOG2E) <= 1e-3 * max(1.0, u), (float(rs[0][0]), u)
    else:
        assert torch.allclose(rs[0].double(), S.max(1).values, rtol=0, atol=tol), "exact form expected: true row maxima"

    G = torch.exp(S - lr[:, None]) + torch.exp(S - lc[None, :])
    G[idx[ok], idx[ok] + off] -= 2.0
    g = s / (2 * rows)
    gtol = GRAD_TOL[X.dtype] * (big if X.dtype == torch.float32 else 1.0)     # bf16: fp16 G and bf16 values dominate
    _rows_close(dX, g * G @ Y.double(), gtol, "dX")
    _rows_close(dY, g * G.T @ X.double(), gtol, "dY")
    return lse_row, lse_col, single, S


# ---------------------------------------------------------------------------------------------- the fused step
def check_fused(x, t, s):
    """ClipLoss (the fused step) on bf16 features against O.clip_loss_single: loss, dlogit_scale, and dI / dT row by
    row.  Returns whether the forward took the single sweep."""
    from clipk import ClipLoss, ops
    I = torch.from_numpy(x).cuda().bfloat16().requires_grad_(True)
    T = torch.from_numpy(t).cuda().bfloat16().requires_grad_(True)
    S = torch.tensor(s, device="cuda", requires_grad=True)
    loss = ClipLoss(cache_labels=True)(I, T, S)
    loss.backward()
    torch.cuda.synchronize()
    single = ops.last_forward_was_single_sweep()
    ref = O.clip_loss_single(I.detach().float().cpu().numpy(), T.detach().float().cpu().numpy(), s)
    tol = 2e-3
    assert abs(loss.item() - ref.loss) <= tol * abs(ref.loss), (loss.item(), ref.loss)
    assert abs(S.grad.item() - ref.d_scale) <= tol * max(abs(ref.d_scale), 1.0 / s), (S.grad.item(), ref.d_scale)
    _rows_close(I.grad.float().cpu(), torch.from_numpy(ref.d_image), tol, "dI")
    _rows_close(T.grad.float().cpu(), torch.from_numpy(ref.d_text), tol, "dT")
    return single


def _bf16(a):
    return torch.from_numpy(a).cuda().bfloat16()


# ------------------------------------------------------------------------------------------------------- cases
# (name, s, expected single sweep, rule targeted, LSE spread band in log2 units)
COLLAPSED = [
    # rule (a) holds with ~1 % margin; anti-aligned rows put the spread above 150: exact backward
    ("rule_a_inside", 65.5, True, "a", (150.0, 1e9)),
    # rule (a) fails, rule (b) fails (anti-aligned positives): exact forward; a bound loosened to ~112 would flush the
    # anti-aligned rows completely
    ("rule_a_outside", 76.0, False, "a", (150.0, 1e9)),
    # spread just below the FAST backward's limit, single sweep
    ("fast_at_limit", 32.5, True, "a", (85.0, 97.0)),
    # spread ~140: exact backward; 2^(v - c) of the FAST form would already overflow here (v - c reaches ~130), so a
    # limit loosened anywhere past ~130 fails on these inputs
    ("exact_bwd_past_overflow", 49.0, True, "a", (135.0, 145.0)),
]


@pytest.mark.parametrize("name,s,want_single,rule,band", COLLAPSED, ids=[c[0] for c in COLLAPSED])
@pytest.mark.parametrize("n,d", [(1024, 256), (640, 512)])
def test_collapsed_embeddings(name, s, want_single, rule, band, n, d):
    x, t = collapsed(n, d, seed=n + d)
    X, Y = _bf16(x), _bf16(t)
    single, u, margin_a, _ = _expect_single(X, Y, s, True)
    assert single == want_single and margin_a >= GUARD, (u, margin_a)
    S = s * (X.double() @ Y.double().T)
    spread = _spread(S)
    assert band[0] <= spread <= band[1] and abs(spread - FAST_SPREAD) >= GUARD * FAST_SPREAD, spread
    assert check_fused(x, t, s) is want_single
    _, _, single_entry, _ = check_entry(X, Y, s)
    assert single_entry is want_single


@pytest.mark.parametrize("cos,want_single", [(-0.19, True), (-0.235, False)])
def test_positives_bound_edges_at_scale_100(cos, want_single):
    """Rule (b) at logit_scale = 100: bad positives at cosine -0.19 keep the single sweep, at -0.235 they do not (the
    threshold is near -0.21 for unit features); both must be accurate in every row and column."""
    s, n, d = 100.0, 1024, 256
    x, t = bad_positives(n, d, cos)
    X, Y = _bf16(x), _bf16(t)
    single, u, margin_a, margin_b = _expect_single(X, Y, s, True)
    assert single == want_single and margin_b >= GUARD and u > FWD_SAFE_U * (1 + GUARD), (u, margin_b)
    S = s * (X.double() @ Y.double().T)
    b = torch.tensor(BAD_ROWS, device="cuda")
    pos = S[b, b]
    assert (pos - s * cos).abs().max() < 0.02 * s
    # the bad pair's positive carries its row and its column: everything else at least 10 below it
    others_r = S[b].clone()
    others_r[torch.arange(len(BAD_ROWS)), b] = -float("inf")
    others_c = S[:, b].clone()
    others_c[b, torch.arange(len(BAD_ROWS))] = -float("inf")
    assert (others_r.max(1).values < pos - 10).all() and (others_c.max(0).values < pos - 10).all()
    assert check_fused(x, t, s) is want_single
    _, _, single_entry, _ = check_entry(X, Y, s)
    assert single_entry is want_single


def test_wide_spread_fp32_entry():
    """fp32 features (two fp16 planes per operand, two-plane G) with graded norms at the initial scale: the LSE spread
    is about 200 log2 units, so every tile of the backward takes the exact form."""
    s = 1 / 0.07
    x, t = graded(1000, 256, seed=3)
    X, Y = torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda()
    spread = _spread(s * (X.double() @ Y.double().T))
    assert 170.0 <= spread <= 240.0, spread
    check_entry(X, Y, s)


ADVERSARIAL = [("collapsed_65.5", 65.5), ("collapsed_76", 76.0), ("collapsed_32.5", 32.5), ("collapsed_49", 49.0),
               ("bad_pos_-0.19", 100.0), ("bad_pos_-0.235", 100.0)]


@pytest.mark.parametrize("name,s", ADVERSARIAL, ids=[a[0] for a in ADVERSARIAL])
def test_single_sweep_and_exact_form_agree(name, s):
    """The same adversarial inputs through clipk_fwd_both with and without `exact`: every row and column LSE agrees."""
    if name.startswith("collapsed"):
        x, t = collapsed(1024, 256, seed=1280)
    else:
        x, t = bad_positives(1024, 256, float(name.split("_")[-1]))
    X, Y = _bf16(x), _bf16(t)
    out = []
    for exact in (False, True):
        lr, lc, single, _ = check_entry(X, Y, s, exact=exact)
        out.append((lr, lc))
    assert (out[0][0] - out[1][0]).abs().max().item() <= 1e-5 * max(1.0, s / 14.0)
    assert (out[0][1] - out[1][1]).abs().max().item() <= 1e-5 * max(1.0, s / 14.0)


# ------------------------------------------------------------------------------------------- tile-count edges
@pytest.mark.parametrize("rows,cols", TILE_EDGES)
def test_tile_count_edges_backward(rows, cols):
    """The shapes whose tile count straddles the 74 clusters of the persistent sweeps (test_parity_gpu.TILE_EDGES)
    through the backward as well."""
    if torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the shapes are chosen for 74 clusters (148 SMs)")
    x, t = O.synthetic_features(max(rows, cols), 64, seed=5)
    check_entry(_bf16(x[:rows]), _bf16(t[:cols]), 1 / 0.07)


# ------------------------------------------------------------------------------------------------ non-finite inputs
@pytest.mark.parametrize("which", ["image", "text"])
@pytest.mark.parametrize("value", [float("nan"), float("inf")], ids=["nan", "inf"])
def test_non_finite_feature_propagates(which, value):
    """One NaN or +Inf in one feature row: the loss is non-finite, as torch fp32 computes it (what GradScaler and
    training loops test for), and a gradient the fp32 reference makes non-finite has a non-finite entry too.  The
    operand statistics turn a non-finite feature into an unbounded u, so the forward takes the exact form."""
    from clipk import ClipLoss, ops
    n, d, s = 512, 256, 1 / 0.07
    x, t = O.synthetic_features(n, d, seed=8)
    (x if which == "image" else t)[200, 17] = value
    I = torch.from_numpy(x).cuda().bfloat16().requires_grad_(True)
    T = torch.from_numpy(t).cuda().bfloat16().requires_grad_(True)
    loss = ClipLoss(cache_labels=True)(I, T, torch.tensor(s, device="cuda", requires_grad=True))
    loss.backward()
    torch.cuda.synchronize()
    assert ops.last_forward_was_single_sweep() is False
    I2 = I.detach().float().requires_grad_(True)
    T2 = T.detach().float().requires_grad_(True)
    labels = torch.arange(n, device="cuda")
    a = s * I2 @ T2.T
    ref = (torch.nn.functional.cross_entropy(a, labels) + torch.nn.functional.cross_entropy(a.T, labels)) / 2
    ref.backward()
    assert not math.isfinite(ref.item())
    assert not math.isfinite(loss.item()), loss.item()
    for got, want, what in ((I.grad, I2.grad, "dI"), (T.grad, T2.grad, "dT")):
        if not bool(torch.isfinite(want).all()):
            assert not bool(torch.isfinite(got).all()), what
