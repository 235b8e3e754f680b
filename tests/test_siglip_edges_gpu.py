"""SigLipLoss's kernels at the edges of their geometry and numerics, one B200, against float64 on the bf16 values upcast:
one rank's block of a larger batch (diagonals that start mid-tile or cross tile, half-tile and epilogue-chunk
boundaries), forced small backward panels, partial backwards, poisoned workspaces, the state words the forward hands to
the backward, the whole logit range, batch and width edges, and where NaN features leave NaN in the outputs.

clipk_siglip_forward / _backward are called directly (CudaBackend.siglip_forward / siglip_backward) wherever the
geometry is the point: they take Y of N rows and any diag_offset, as rank diag_offset / b of N / b would."""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from scipy.special import expit

from oracle import siglip_oracle as SO
from tests.test_siglip_gpu import REGIMES, _check, _pair, _run

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P2E_CAP = 2.0 ** 64


def _be():
    from clipk import ops
    return ops._backend()


def _dev(v):
    return None if v is None else torch.tensor([v], dtype=torch.float32, device="cuda")


def _host(v):
    return None if v is None else v.detach().cpu().clone()


def _call(X, Y, s, bias, off, go=1.0, want=(True, True, True, True)):
    """clipk_siglip_forward, then clipk_siglip_backward with the outputs in `want` (d_x, d_y, d_scale, d_bias).
    Returns the loss, the 8 state words and the fp32 outputs on the host (None where not wanted)."""
    be = _be()
    S, B, GO = _dev(s), _dev(bias), _dev(go)
    loss, state = be.siglip_forward(X, Y, S, B, off)
    dX, dY, ds, dt = be.siglip_backward(X, Y, S, B, off, state, GO, *want)
    torch.cuda.synchronize()
    return SimpleNamespace(loss=_host(loss), state=_host(state), dX=_host(dX), dY=_host(dY), ds=_host(ds), dt=_host(dt))


def _filled(n, byte, dtype=torch.float32):
    return torch.full((n * 4,), byte, dtype=torch.uint8, device="cuda").view(dtype)


def _raw_call(X, Y, s, bias, off, go, byte):
    """Both entries on the clipk_siglip struct CudaBackend._c_siglip builds, with the workspace, state, d_x, d_y,
    d_scale and d_bias all filled with `byte` first; the workspace is filled again between the two calls, since
    nothing in it may live from one call to the next."""
    from clipk import _lib
    be = _be()
    S, B, GO = _dev(s), _dev(bias), _dev(go)
    state = _filled(_lib.SIGLIP_STATE_WORDS, byte)
    c, _ = be._c_siglip(X, Y, S, B, off, state)
    ws = torch.full((c.workspace_bytes,), byte, dtype=torch.uint8, device="cuda")
    c.workspace = ws.data_ptr()
    _lib.check(be.lib.clipk_siglip_forward(ctypes.byref(c)), "clipk_siglip_forward")
    ws.fill_(byte)
    dX, dY = _filled(X.numel(), byte).view(X.shape), _filled(Y.numel(), byte).view(Y.shape)
    ds, dt = _filled(1, byte), _filled(1, byte)
    c.grad_out = GO.data_ptr()
    c.d_x, c.d_y, c.d_scale, c.d_bias = dX.data_ptr(), dY.data_ptr(), ds.data_ptr(), dt.data_ptr()
    _lib.check(be.lib.clipk_siglip_backward(ctypes.byref(c)), "clipk_siglip_backward")
    torch.cuda.synchronize()
    return SimpleNamespace(loss=_host(state[0]), state=_host(state[:6]), dX=_host(dX), dY=_host(dY), ds=_host(ds),
                           dt=_host(dt))


def _np(t):
    return t.detach().double().cpu().numpy()


def _reference(X, Y, s, bias, go, off):
    """siglip_block in float64 plus what the bars need: sums of |g| |x.y| and |g|, the extreme logits, max |g|."""
    Xn, Yn = (X if isinstance(X, np.ndarray) else _np(X)), (Y if isinstance(Y, np.ndarray) else _np(Y))
    t = 0.0 if bias is None else bias
    ref = SO.siglip_block(Xn, Yn, s, t, go, off)
    dots = Xn @ Yn.T
    L = s * dots + t
    i = np.arange(len(Xn))
    pos = L[i, i + off]
    G = expit(L)
    G[i, i + off] = expit(-pos)                     # |g|
    neg = L.copy()
    neg[i, i + off] = -np.inf
    mag = np.linalg.norm(Xn, axis=1).max() * np.linalg.norm(Yn, axis=1).max()
    return SimpleNamespace(loss=ref.loss, d_x=ref.d_image, d_y=ref.d_text, ds=ref.d_scale, dt=ref.d_bias,
                           ds_mag=(G * np.abs(dots)).sum(), dt_mag=G.sum(), gmax=G.max(), maxneg=neg.max(),
                           minpos=pos.min(), l_tol=1e-5 * (abs(s) * mag + abs(t)) + 1e-6, s=s, go=go, b=len(Xn))


def _rows_close(got, want, what, tol=1e-2):
    """each row's error <= tol * max(its float64 norm, 1e-3 * the largest row norm): a positive in the wrong column
    changes one row by O(1) and hides inside a whole-matrix norm; and <= 2e-3 normwise"""
    got = got if isinstance(got, np.ndarray) else _np(got)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err, nrm = np.linalg.norm(got - want, axis=1), np.linalg.norm(want, axis=1)
    bound = tol * np.maximum(nrm, 1e-3 * nrm.max())
    bad = np.nonzero(~(err <= bound))[0]
    assert bad.size == 0, f"{what}: {bad.size} rows off, first {bad[:8]}: err {err[bad[:8]]} bound {bound[bad[:8]]}"
    assert np.linalg.norm(got - want) <= 2e-3 * np.linalg.norm(want), what


def _check_scalars(loss, ds, dt, ref):
    """loss <= 1e-4 relative; d_scale, d_bias <= 1e-3 |go| / b of the sums of |g| |x.y| and |g|"""
    k = 1e-3 * abs(ref.go) / ref.b
    assert abs(float(loss) - ref.loss) <= 1e-4 * abs(ref.loss), (float(loss), ref.loss)
    assert abs(float(ds) - ref.ds) <= k * ref.ds_mag, (float(ds), ref.ds)
    assert abs(float(dt) - ref.dt) <= k * ref.dt_mag, (float(dt), ref.dt)


def _check_state(state, ref):
    """[2] largest negative logit and [3] smallest positive logit against float64 within fp32 rounding of the logits;
    [1] gmax = max(sigma([2]), sigma(-[3])) (the fp32 expression of siglip_reduce_kernel); [4] = 2^e puts gmax in
    [2^13, 2^14) unless the cap e = 64 holds it lower (gmax = 0 takes 2^14); [5] = go s / (b 2^e)."""
    st = state.double().numpy()
    if np.isinf(ref.maxneg):
        assert st[2] == -np.inf, st[2]
    else:
        assert abs(st[2] - ref.maxneg) <= ref.l_tol, (st[2], ref.maxneg)
    assert abs(st[3] - ref.minpos) <= ref.l_tol, (st[3], ref.minpos)
    f = np.float32
    sig = lambda x: f(1) / (f(1) + np.exp(-f(x)))           # noqa: E731
    gm = max(sig(st[2]) if st[2] > -np.inf else f(0), sig(-st[3]))
    assert abs(st[1] - gm) <= 1e-6 * gm, (st[1], gm)
    assert abs(st[1] - ref.gmax) <= (ref.l_tol + 1e-5) * ref.gmax, (st[1], ref.gmax)
    p2e = st[4]
    assert p2e == 2.0 ** round(np.log2(p2e)), p2e
    if st[1] == 0:
        assert p2e == 2.0 ** 14
    elif p2e == P2E_CAP:
        assert st[1] * p2e < 2.0 ** 14, (st[1], p2e)
    else:
        assert 2.0 ** 13 <= st[1] * p2e < 2.0 ** 14, (st[1], p2e)
    assert abs(st[5] - ref.go * ref.s / ref.b / p2e) <= 1e-6 * abs(ref.go * ref.s / ref.b / p2e), (st[5], p2e)


def _check_all(out, ref):
    _check_scalars(out.loss, out.ds, out.dt, ref)
    _rows_close(out.dX, ref.d_x, "d_x")
    _rows_close(out.dY, ref.d_y, "d_y partial")
    _check_state(out.state, ref)


# ---- 1. one rank's block on one GPU ------------------------------------------------------------------------------------
# (b, W, r, d): offsets 300 / 600 / 900 start mid-tile and mid-half; 1000 on W = 2 crosses column 1024; b = 129, 257
# put the diagonal across the 128-row and 256-row blocks; b = 1 is a block of one row; d = 576 is the first streaming
# (not A-resident) width, 768 another.
RANK_BLOCKS = [(300, 4, 0, 128), (300, 4, 1, 128), (300, 4, 2, 128), (300, 4, 3, 128), (1000, 2, 1, 512),
               (129, 3, 2, 64), (1, 8, 5, 64), (640, 2, 1, 576), (257, 2, 1, 768)]


def _rank_block(b, W, r, d, pos_cos, seed):
    feats = [_pair(b, d, seed=seed + 17 * k, pos_cos=pos_cos) for k in range(W)]
    return feats[r][0], torch.cat([f[1] for f in feats]), r * b


@pytest.mark.parametrize("regime", list(REGIMES))
@pytest.mark.parametrize("b,W,r,d", RANK_BLOCKS)
def test_rank_block_against_oracle(b, W, r, d, regime):
    """X = images[r], Y = every rank's text rows, positives at column r*b + i: the loss, d_scale, d_bias, d_x row by row,
    the [N, d] partial d_y row by row, and the state words.  The bias variant in every regime; no bias and
    grad_output = -2.5 in the init regime."""
    s, bias, pos_cos = REGIMES[regime]
    X, Y, off = _rank_block(b, W, r, d, pos_cos, seed=b * W + d)
    variants = [(bias, 1.0)] + ([(None, 1.0), (bias, -2.5)] if regime == "init" else [])
    for t, go in variants:
        _check_all(_call(X, Y, s, t, off, go), _reference(X, Y, s, t, go, off))


# ---- 2-4. forced small backward panels, partial backwards, poisoned buffers ----------------------------------------------
# choose_panel reads CLIPK_PANEL_RB / CLIPK_PANEL_CB once per shape and caches its choice, so each panel setting runs in
# a process of its own: "forced" with 256 x 256 panels, "default" with the library's choice.
PANEL_SHAPES = {"wide": (1000, 4000, 1000), "square": (1000, 1000, 0)}     # b, N, diag_offset
PANEL_D, PANEL_S, PANEL_T = 128, 10.0, -10.0
PANEL_COUNTS = {"wide": "4 x 16", "square": "4 x 4"}


def _panel_inputs(name):
    b, N, off = PANEL_SHAPES[name]
    feats = [_pair(b, PANEL_D, seed=900 + 7 * k + len(name)) for k in range(N // b)]
    return feats[off // b][0], torch.cat([f[1] for f in feats]), off


def _panel_worker(path):
    """Every panel-dependent call of the tests below, saved to `path` for the parent process to check."""
    from clipk import siglip_loss
    out = {}
    for name in PANEL_SHAPES:
        X, Y, off = _panel_inputs(name)
        args = (X, Y, PANEL_S, PANEL_T, off, 1.0)
        r = dict(full=_call(*args), again=_call(*args), dx=_call(*args, want=(True, False, False, False)),
                 dy=_call(*args, want=(False, True, False, False)), scalars=_call(*args, want=(False, False, True, True)),
                 poisoned=_raw_call(*args, 0xFF), zeroed=_raw_call(*args, 0))
        if off == 0 and X.shape == Y.shape:       # siglip_loss on features that do not require grad: scalars only
            S, B = (torch.tensor(v, device="cuda", requires_grad=True) for v in (PANEL_S, PANEL_T))
            siglip_loss(X, Y, S, B).backward()
            torch.cuda.synchronize()
            r["autograd"] = SimpleNamespace(ds=_host(S.grad), dt=_host(B.grad))
        out[name] = {k: vars(v) for k, v in r.items()}
    torch.save(out, path)


@pytest.fixture(scope="module")
def panel_runs(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("siglip_panels")
    code = ("import sys; sys.path[:0] = ['.', 'megatron-clip_b200']\n"
            "from tests.test_siglip_edges_gpu import _panel_worker; _panel_worker(sys.argv[1])\n")
    runs = {}
    for mode, forced in (("forced", {"CLIPK_PANEL_RB": "1", "CLIPK_PANEL_CB": "1"}), ("default", {})):
        env = {k: v for k, v in os.environ.items() if not k.startswith("CLIPK_PANEL")}
        env.update(forced, CLIPK_VERBOSE="1")
        path = str(tmp / f"{mode}.pt")
        p = subprocess.run([sys.executable, "-c", code, path], cwd=ROOT, env=env, capture_output=True, text=True,
                           timeout=600)
        assert p.returncode == 0, p.stderr[-3000:]
        out = torch.load(path, weights_only=False)
        runs[mode] = ({n: {k: SimpleNamespace(**v) for k, v in r.items()} for n, r in out.items()}, p.stderr)
    return runs


def _panel_line(stderr, name):
    b, N, _ = PANEL_SHAPES[name]
    lines = [ln for ln in stderr.splitlines() if f"for a {b} x {N} x {PANEL_D} block" in ln]
    assert len(lines) == 1, stderr[-2000:]
    return lines[0]


def test_panel_counts(panel_runs):
    """The forced process really ran 4 x 16 and 4 x 4 panels of 256 x 256; the library's own choice keeps the square
    shape in one panel (the single-panel case of the tests below)."""
    for name, count in PANEL_COUNTS.items():
        assert f"({count} panels" in _panel_line(panel_runs["forced"][1], name)
    assert "(1 x 1 panels" in _panel_line(panel_runs["default"][1], "square")


@pytest.mark.parametrize("name", list(PANEL_SHAPES))
def test_forced_panels_against_oracle(panel_runs, name):
    """Per-panel positive offsets (negative, or past the panel), the accumulate flags of the row sums and of both GEMMs,
    and the hand-off of the row-sum slots and of the G buffer from panel to panel: against float64 row by row, and
    against the default panels of the same call (the loss bit for bit: the forward does not depend on the panels)."""
    X, Y, off = _panel_inputs(name)
    ref = _reference(X, Y, PANEL_S, PANEL_T, 1.0, off)
    forced, default = panel_runs["forced"][0][name]["full"], panel_runs["default"][0][name]["full"]
    for out in (forced, default):
        _check_all(out, ref)
    assert torch.equal(forced.loss, default.loss) and torch.equal(forced.state[:4], default.state[:4])
    for k in ("dX", "dY"):
        u, v = getattr(forced, k), getattr(default, k)
        assert (u - v).norm() <= 2e-3 * v.norm(), k


@pytest.mark.parametrize("mode", ["forced", "default"])
@pytest.mark.parametrize("name", list(PANEL_SHAPES))
def test_two_calls_bit_identical(panel_runs, mode, name):
    a, b = panel_runs[mode][0][name]["full"], panel_runs[mode][0][name]["again"]
    for k in ("loss", "state", "dX", "dY", "ds", "dt"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k


@pytest.mark.parametrize("mode", ["forced", "default"])
@pytest.mark.parametrize("name", list(PANEL_SHAPES))
def test_partial_backwards_match_the_full_one(panel_runs, mode, name):
    """d_x only and d_y only (one GEMM per panel instead of the pair), and the scalars only (recompute and row sums, no
    GEMMs, no fp16 copies; from Python whenever the features do not require grad): each output bit for bit the full
    backward's."""
    r = panel_runs[mode][0][name]
    full = r["full"]
    assert r["dx"].dY is None and r["dx"].ds is None and torch.equal(r["dx"].dX, full.dX)
    assert r["dy"].dX is None and r["dy"].dt is None and torch.equal(r["dy"].dY, full.dY)
    assert r["scalars"].dX is None and r["scalars"].dY is None
    assert torch.equal(r["scalars"].ds, full.ds) and torch.equal(r["scalars"].dt, full.dt)
    for k in ("dx", "dy", "scalars"):
        assert torch.equal(r[k].state, full.state), k
    if "autograd" in r:
        assert torch.equal(r["autograd"].ds.reshape(1), full.ds) and torch.equal(r["autograd"].dt.reshape(1), full.dt)


@pytest.mark.parametrize("mode", ["forced", "default"])
@pytest.mark.parametrize("name", list(PANEL_SHAPES))
def test_poisoned_buffers(panel_runs, mode, name):
    """Workspace, state, d_x, d_y, d_scale and d_bias filled with 0xFF bytes (NaN in fp32 and fp16) give bit for bit
    what zero-filled ones give, and what the library's own buffers give: nothing is read before it is written."""
    r = panel_runs[mode][0][name]
    for k in ("loss", "state", "dX", "dY", "ds", "dt"):
        u, v, w = getattr(r["poisoned"], k), getattr(r["zeroed"], k), getattr(r["full"], k)
        assert torch.equal(u, v), k
        assert torch.equal(v, w[:6] if k == "state" else w), k


# ---- 5. state words and masking -----------------------------------------------------------------------------------------
def test_masked_columns_and_rows_stay_out_of_the_state():
    """b = 100 rows whose positives are columns 200..299 of N = 300: the diagonal crosses column 256, the last row's
    positive is the last real column, and the last tile holds 212 columns past N, which TMA reads as zeros (logit t),
    like the 28 rows past b of the 128-row block.  With t = 8 every real negative sits at l = -2 and the positives at
    38, except the last row's at 0.5: the block's largest |g|, sigma(-0.5).  A column or row past the block leaking into
    the maxima would read 8 and move gmax to sigma(8).  Then b = N = 1: no negative at all."""
    b, N, off, d, s, t = 100, 300, 200, 320, 40.0, 8.0
    X, Y = torch.zeros(b, d, dtype=torch.float64), torch.zeros(N, d, dtype=torch.float64)
    X[:, d - 1], Y[:, d - 1] = 0.5, -0.5
    X[torch.arange(b), torch.arange(b)] = 1.0
    X[b - 1, b - 1] = 0.0625
    Y[torch.arange(N), (torch.arange(N) - off) % N] = 1.0       # y_{off+i} pairs with x_i
    X, Y = X.to(torch.bfloat16).cuda(), Y.to(torch.bfloat16).cuda()
    ref = _reference(X, Y, s, t, 1.0, off)
    assert ref.maxneg == -2.0 and ref.minpos == 0.5 and ref.gmax == expit(-0.5)
    out = _call(X, Y, s, t, off)
    _check_all(out, ref)
    assert float(out.state[3]) == 0.5                              # fmaf(-0.1875, 40, 8), exact
    x1, y1 = _pair(1, 64, seed=3)
    ref1 = _reference(x1, y1, 10.0, -10.0, 1.0, 0)
    out1 = _call(x1, y1, 10.0, -10.0, 0)
    _check_all(out1, ref1)
    assert float(out1.state[2]) == -np.inf


# ---- 6. the logit range -------------------------------------------------------------------------------------------------
GRAD_FLOOR = 2.0 ** -78      # gmax below it: gmax * 2^64 (the capped 2^e) is below fp16's smallest normal


def _below_floor_grads(got, want, gmax):
    """A block whose every |g| is gmax < GRAD_FLOOR: with e capped at 64 the fp16 G panel holds subnormals or zeros, so
    each entry rounds by at most half a subnormal unit, 2^-25 / 2^64.  The gradients stay finite and no larger than
    float64's beyond that (and 1 % for the fp32 and bf16 roundings after it)."""
    rho = 2.0 ** -25 / (gmax * P2E_CAP)
    assert np.isfinite(got).all()
    assert np.linalg.norm(got) <= (1 + rho) * (1 + 1e-2) * np.linalg.norm(want), rho
    assert (np.abs(got) <= (1 + rho) * (1 + 1e-2) * np.abs(want) + 1e-30).all(), rho


@pytest.mark.parametrize("L", [-0.5, -2.0, -8.0, -16.0, -30.0, -45.0, -60.0, -80.0, 0.5, 2.0, 8.0, 16.0, 30.0, 45.0,
                               60.0, 80.0])
def test_logit_range(L):
    """x_i = e_i + 0.25 e_{d-1}, y_j = a e_j + 0.5 e_{d-1}, so x_i.y_j = a [i = j] + 0.125 exactly; s = 2|L| and
    t = L - 0.125 s put every negative at logit L and every positive at -L (a = 1, L < 0: a well-separated batch; a = -1,
    L > 0: every pair misclassified).  b = N = 300, d = 384: a partial tile and rows past b.

    The loss, d_scale and d_bias hold their bars in every band: a term dropped to 0 or rounded (1 + e -> 1) is an O(1)
    error.  The feature gradients hold 2e-3 normwise while gmax * 2^e stays in fp16's normal range, i.e. down to
    gmax = 2^-78 (L ~ -54): measured floor, L = -45 passes, L = -60 is below it.  Below the floor (e capped at 64) the
    fp16 G panel holds subnormals or zeros: the gradients stay finite and no larger than float64's beyond half an fp16
    subnormal unit per entry."""
    b, d = 300, 384
    a = 1.0 if L < 0 else -1.0
    s, t = 2 * abs(L), L - 0.125 * 2 * abs(L)
    X, Y = torch.zeros(b, d, dtype=torch.float64), torch.zeros(b, d, dtype=torch.float64)
    X[:, d - 1], Y[:, d - 1] = 0.25, 0.5
    X[torch.arange(b), torch.arange(b)] = 1.0
    Y[torch.arange(b), torch.arange(b)] = a
    X, Y = X.to(torch.bfloat16).cuda(), Y.to(torch.bfloat16).cuda()
    ref = _reference(X, Y, s, t, 1.0, 0)
    assert abs(ref.maxneg - L) <= 1e-12 * abs(L) and abs(ref.minpos + L) <= 1e-12 * abs(L)
    out = _call(X, Y, s, t, 0)
    _check_scalars(out.loss, out.ds, out.dt, ref)
    _check_state(out.state, ref)
    p2e = float(out.state[4])
    for got, want in ((_np(out.dX), ref.d_x), (_np(out.dY), ref.d_y)):
        assert np.isfinite(got).all()
        if ref.gmax >= GRAD_FLOOR:
            assert np.linalg.norm(got - want) <= 2e-3 * np.linalg.norm(want), (L, ref.gmax)
        else:
            assert p2e == P2E_CAP
            _below_floor_grads(got, want, ref.gmax)        # every |g| of this batch is gmax


# ---- 7. batch and width edges through siglip_loss ------------------------------------------------------------------------
def _loss_route_check(x, t, s, bias, out):
    """_check's bars, plus d_image and d_text row by row"""
    _check(x, t, s, bias, out)
    X, T = _np(x), _np(t)
    ref = SO.siglip_single(X, T, s, 0.0 if bias is None else bias)
    _rows_close(out[1], ref.d_image, "d_image")
    _rows_close(out[2], ref.d_text, "d_text")


def _below_floor_check(x, t, s, bias, out):
    """A one-pair block below the gradient floor: the loss, d_scale and d_bias at their bars (fp32 sums), the feature
    gradients by _below_floor_grads"""
    loss, dI, dT, dS, dB = out
    ref = _reference(x, t, s, bias, 1.0, 0)
    assert len(_np(x)) == 1 and ref.gmax < GRAD_FLOOR, ref.gmax
    _check_scalars(loss, dS, dB, ref)
    for got, want in ((dI, ref.d_x), (dT, ref.d_y)):
        _below_floor_grads(_np(got), want, ref.gmax)


@pytest.mark.parametrize("regime", ["init", "separated"])
@pytest.mark.parametrize("b,d", [(1, 64), (2, 64), (127, 64), (129, 64), (257, 64), (300, 8), (300, 72), (300, 520),
                                 (300, 576)])
def test_batch_and_width_edges(b, d, regime):
    """b = 1 (no negatives), 2, and around the 128- and 256-row blocks; widths that _kernel_features pads to 64, 128
    and 576, and 576 itself, the first streaming width.  b = 1 in the separated regime is one positive at
    l = 100 * 0.95 - 15 = 80, g = -sigma(-80) ~ 2^-116: the whole block lies below the gradient floor (DESIGN 4.8), so
    its feature gradients are held to the floor's promise, its loss and scalar gradients to the usual bars."""
    s, bias, pos_cos = REGIMES[regime]
    x, t = _pair(b, d, seed=3 * b + d, pos_cos=pos_cos)
    out = _run(x, t, s, bias)
    if b == 1 and regime == "separated":
        _below_floor_check(x, t, s, bias, out)
    else:
        _loss_route_check(x, t, s, bias, out)


def test_fp32_features_under_bf16_autocast_at_a_padded_width():
    x, t = _pair(300, 72, seed=77)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = _run(x, t, 10.0, -10.0, dtype=torch.float32)
    assert out[1].dtype == torch.float32 and out[2].dtype == torch.float32
    _loss_route_check(x, t, 10.0, -10.0, out)


# ---- 8. NaN placement ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("row", [127, 128, 255])
@pytest.mark.parametrize("side", ["image", "text"])
def test_nan_placement(side, row):
    """A NaN in image row k makes row k of d_image and all of d_text NaN (every text row gets a term of row k), and the
    text case the mirror; loss, d_scale and d_bias are NaN either way.  The NaN entries of every output are open_clip's
    formula's in float64, and the finite ones hold the bars: the forward's maxima drop the NaN (fmaxf), which must leave
    the finite part's 2^e right."""
    b, d, s, bias = 300, 128, 10.0, -10.0
    x, t = _pair(b, d, seed=400 + row)
    (x if side == "image" else t)[row, 5] = float("nan")
    loss, dI, dT, dS, dB = _run(x, t, s, bias)
    ref = SO.siglip_single(_np(x), _np(t), s, bias)
    for got, want in ((loss, ref.loss), (dS, ref.d_scale), (dB, ref.d_bias)):
        assert np.isnan(want) and torch.isnan(got).all()
    for got, want, what in ((_np(dI), ref.d_image, "d_image"), (_np(dT), ref.d_text, "d_text")):
        assert np.array_equal(np.isnan(got), np.isnan(want)), (what, np.argwhere(np.isnan(got) != np.isnan(want))[:4])
        fin = ~np.isnan(want).any(axis=1)
        assert fin.sum() == (0 if (what == "d_text") == (side == "image") else b - 1), what
        if fin.any():
            _rows_close(got[fin], want[fin], what)
