"""Parity of the CUDA path (through the C ABI, via the drop-in ClipLoss) with the oracle and the reference goldens.

Tolerances are the ones BASELINE.json states: 1e-5 relative for fp32 inputs, 2e-3 relative for bf16 inputs
(bf16 is compared with the oracle evaluated on the same bf16 values upcast - SURVEY.md App. B), labels bit-exact.
"""
import numpy as np
import pytest
import torch

from oracle import cliploss_oracle as O
from tests.util import golden_files, load_golden, make_inputs, rel

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 2e-3}


def run_clipk(x, t, s, dtype, grad_output=1.0, **kw):
    from clipk import ClipLoss
    I = torch.from_numpy(x).cuda().to(dtype).requires_grad_(True)
    T = torch.from_numpy(t).cuda().to(dtype).requires_grad_(True)
    S = torch.tensor(s, device="cuda", dtype=torch.float32, requires_grad=True)
    loss = ClipLoss(**kw)(I, T, S)
    (loss * grad_output).backward()
    torch.cuda.synchronize()
    return (loss.item(), I.grad.float().cpu().numpy(), T.grad.float().cpu().numpy(), S.grad.item(), I, T)


def check(x, t, s, dtype, grad_output=1.0, tol=None, ulp_floor=False):
    """ulp_floor: batches of 1..3 rows, where lse - pos and P - 1 cancel far below the size of the logits (b = 1: the
    loss and the gradients are exactly 0).  Their errors get an absolute floor of a few fp32 ulps of a logit of size s,
    eps = 2^-20 s, on the loss and on every softmax entry of G (times |features| and the gradient's scale)."""
    tol = tol or TOL[dtype]
    loss, dI, dT, ds, I, T = run_clipk(x, t, s, dtype, grad_output)
    # the oracle sees exactly the values the kernel saw
    xin = I.detach().float().cpu().numpy()
    tin = T.detach().float().cpu().numpy()
    ref = O.clip_loss_single(xin, tin, s, grad_output)
    assert I.grad.dtype == dtype and T.grad.dtype == dtype
    eps = 2.0 ** -20 * s if ulp_floor else 0.0
    gfloor = eps * 2 * abs(grad_output) * s / (2 * x.shape[0])       # per unit of feature norm, both softmaxes
    assert abs(loss - ref.loss) <= tol * abs(ref.loss) + eps, ("loss", loss, ref.loss)
    for got, want, other, what in ((dI, ref.d_image, tin, "dI"), (dT, ref.d_text, xin, "dT")):
        err = np.linalg.norm(got - want)
        assert err <= tol * np.linalg.norm(want) + gfloor * np.linalg.norm(other), (what, err, np.linalg.norm(want))
        assert np.abs(got - want).max() <= 2 * tol * np.abs(want).max() + gfloor * x.shape[0] * np.abs(other).max(), what
    # dlogit_scale is a sum of cancelling terms of size ~1/s each; tolerance relative to max(|ds|, 1/s)
    assert abs(ds - ref.d_scale) <= tol * max(abs(ref.d_scale), 1.0 / s), ("ds", ds, ref.d_scale)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("b,d", [(16, 1024), (100, 512), (257, 640), (256, 512), (1000, 128), (2048, 256), (520, 768),
                                 (768, 1024), (300, 1280)] +
                         # degenerate batches (b = 1: loss and gradients exactly 0) and both sides of the 128-row block
                         [(b, d) for d in (64, 128) for b in (1, 2, 3, 127, 129, 255)])
def test_single_gpu_unit_inputs(b, d, dtype):
    x, t = make_inputs(b, d, seed=b + d)
    check(x, t, 1 / 0.07, dtype, ulp_floor=b <= 3)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_scale_100_and_grad_output(dtype):
    x, t = make_inputs(300, 256, seed=9)
    # at s=100 the fp32 reference itself is ~1e-4 from exact (SURVEY App. B); allow 5e-5 for the fp32 kernel
    check(x, t, 100.0, dtype, grad_output=3.0, tol=5e-5 if dtype == torch.float32 else 4e-3)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_unnormalised_inputs(dtype):
    x, t = make_inputs(200, 192, seed=4, kind="raw")
    check(x, t, 1 / 0.07, dtype)


def test_scale_one_bf16():
    x, t = make_inputs(128, 256, seed=5)
    check(x, t, 1.0, torch.bfloat16)


@pytest.mark.parametrize("b,d,dtype,tol", [(300, 100, torch.bfloat16, 2e-3), (257, 36, torch.float32, 1e-5),
                                           (200, 72, torch.float16, 1e-3), (384, 512, torch.float16, 1e-3)])
def test_odd_widths_and_fp16_features(b, d, dtype, tol):
    """Embedding widths that are not a multiple of the 64-element K block (zero-padded on the host) and fp16 features
    (open_clip --precision fp16; carried exactly by the fp32 split-precision path, gradients rounded back to fp16:
    2^-11 relative per element, hence 1e-3)."""
    x, t = make_inputs(b, d, seed=b + d)
    check(x, t, 1 / 0.07, dtype, tol=tol)


def test_multi_panel_rows_and_cols():
    """Several G panels in both directions (8 MB budget, set before the library reads it: a fresh process): dX accumulates
    over the column panels, dY over the row panels (TMA reduce-adds after the first panel's stores)."""
    import json, os, subprocess, sys
    code = (
        "import sys, json, torch, numpy as np\n"
        "sys.path.insert(0, 'megatron-clip_b200'); sys.path.insert(0, '.')\n"
        "from clipk import ClipLoss\n"
        "from oracle import cliploss_oracle as O\n"
        "x, t = O.synthetic_features(4300, 128, seed=12)\n"
        "I = torch.from_numpy(x).cuda().bfloat16().requires_grad_(True)\n"
        "T = torch.from_numpy(t).cuda().bfloat16().requires_grad_(True)\n"
        "S = torch.tensor(1 / 0.07, device='cuda', requires_grad=True)\n"
        "loss = ClipLoss()(I, T, S); loss.backward(); torch.cuda.synchronize()\n"
        "ref = O.clip_loss_single(I.detach().float().cpu().numpy(), T.detach().float().cpu().numpy(), 1 / 0.07)\n"
        "r = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))\n"
        "print(json.dumps([abs(loss.item() - ref.loss) / ref.loss, r(I.grad.float().cpu().numpy(), ref.d_image), "
        "r(T.grad.float().cpu().numpy(), ref.d_text), abs(S.grad.item() - ref.d_scale) / max(abs(ref.d_scale), 0.07)]))\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CLIPK_PANEL_MB="8", CLIPK_VERBOSE="1")
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "panels" in out.stderr and "(1 x 1 panels" not in out.stderr, out.stderr[-500:]      # really several panels
    errs = json.loads(out.stdout.strip().splitlines()[-1])
    assert all(e <= 2e-3 for e in errs), errs


@pytest.mark.parametrize("path", golden_files(world=1), ids=lambda p: p.split("/")[-1][:-4])
def test_reference_goldens_world1(path):
    z, W, ranks = load_golden(path)
    g = ranks[0]
    x = g["image"].astype(np.float32)
    t = g["text"].astype(np.float32)
    s, go = float(z["scale"]), float(z["grad_output"])
    loss, dI, dT, ds, _, _ = run_clipk(x, t, s, torch.float32, go)
    tol = 1e-5 if s < 50 else 2e-4
    assert abs(loss - float(g["loss"])) <= tol * abs(float(g["loss"]))
    assert rel(dI, g["d_image"]) <= tol and rel(dT, g["d_text"]) <= tol
    assert abs(ds - float(g["d_scale"])) <= tol * max(abs(float(g["d_scale"])), go / s)


def test_api_variants():
    from clipk import ClipLoss
    x, t = make_inputs(64, 128, seed=1)
    I = torch.from_numpy(x).cuda().bfloat16().requires_grad_(True)
    T = torch.from_numpy(t).cuda().bfloat16().requires_grad_(True)
    mod = ClipLoss(cache_labels=True)
    out = mod(I, T, 14.285, output_dict=True)            # python float scale, dict output
    assert set(out) == {"contrastive_loss"}
    out["contrastive_loss"].backward()
    ref = O.clip_loss_single(I.detach().float().cpu().numpy(), T.detach().float().cpu().numpy(), 14.285)
    assert abs(out["contrastive_loss"].item() - ref.loss) < 2e-3 * ref.loss
    # non-contiguous views are accepted
    big = torch.from_numpy(np.concatenate([x, x], axis=1)).cuda().bfloat16()
    l2 = mod(big[:, :128], T.detach(), torch.tensor(14.285, device="cuda"))
    assert abs(l2.item() - ref.loss) < 2e-3 * ref.loss
    # labels: bit exact, cached
    lab = mod.get_ground_truth(I.device, 64)
    assert lab.dtype == torch.long and torch.equal(lab.cpu(), torch.arange(64))
    assert mod.get_ground_truth(I.device, 64) is lab


def test_autocast_fp32_inputs_take_bf16_path():
    from clipk import ClipLoss
    x, t = make_inputs(128, 256, seed=2)
    I = torch.from_numpy(x).cuda().requires_grad_(True)
    T = torch.from_numpy(t).cuda().requires_grad_(True)
    s = torch.tensor(1 / 0.07, device="cuda", requires_grad=True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss = ClipLoss()(I, T, s)
    loss.backward()
    assert I.grad.dtype == torch.float32
    ref = O.clip_loss_single(O.round_to_bf16(x), O.round_to_bf16(t), 1 / 0.07)
    assert abs(loss.item() - ref.loss) < 2e-3 * ref.loss
    assert rel(I.grad.cpu().numpy(), ref.d_image) < 2e-3


def test_large_properties_c2_shape():
    """BASELINE config size on one GPU (N = 32768, d = 512, bf16): properties that need no O(N^2) oracle.

    (1) dlogit_scale = <I, dI> / s, which holds exactly for the analytic gradient;  (2) every row of the softmax
    gradient sums to zero, so sum_i dT_i-weighted identity: sum over rows of dI equals G-weighted sum of T - checked
    through <1, dI> = <colsum(G), T> being finite and the loss being within the analytic bounds [0, log N + 2s].
    """
    from clipk import ClipLoss
    N, d, s = 32768, 512, 1 / 0.07
    x, t = make_inputs(N, d, seed=1234)
    I = torch.from_numpy(x).cuda().bfloat16().requires_grad_(True)
    T = torch.from_numpy(t).cuda().bfloat16().requires_grad_(True)
    S = torch.tensor(s, device="cuda", requires_grad=True)
    loss = ClipLoss()(I, T, S)
    loss.backward()
    torch.cuda.synchronize()
    assert 0.0 < loss.item() < np.log(N) + 2 * s
    ds_from_dI = (I.detach().float() * I.grad.float()).sum().item() / s
    ds_from_dT = (T.detach().float() * T.grad.float()).sum().item() / s
    assert abs(ds_from_dI - S.grad.item()) <= 5e-3 * abs(S.grad.item())
    assert abs(ds_from_dT - S.grad.item()) <= 5e-3 * abs(S.grad.item())
    # sub-block check against the oracle: the loss restricted to a 512-sample world is a different problem, but the
    # statistics of the first rows can be checked against a direct fp32 computation of those rows
    rows = I.detach()[:256].float() @ T.detach().float().T * s
    lse = torch.logsumexp(rows, dim=1)
    pos = rows[torch.arange(256), torch.arange(256)]
    # image->text CE of the first 256 rows, computed by the kernel path via a local-rows call
    from clipk import ops
    be = ops._backend()
    X = be.prepare(I.detach()[:256])
    Y = be.prepare(T.detach())
    sc = torch.tensor([s], device="cuda")
    stats, p = be.fwd_stats(X, Y, sc, 0, True)
    torch.cuda.synchronize()
    assert torch.allclose(stats[0] + stats[1].log(), lse, rtol=0, atol=2e-3)
    expect = (torch.softmax(rows, dim=1) * rows).sum(dim=1)
    assert torch.allclose(stats[2] / stats[1], expect, rtol=0, atol=2e-3)
    assert torch.allclose(p, pos, rtol=0, atol=2e-3)


# tile counts (256 x 256 tiles) around the cluster count of the persistent sweeps, min(74, tiles) clusters = 148 SMs / 2
# on a B200: 73, 74, 75, 147 and 150 tiles (the last with a ragged last column tile)
TILE_EDGES = [(256, 73 * 256), (256, 74 * 256), (256, 74 * 256 + 1), (513, 49 * 256), (768, 50 * 256 - 3)]


@pytest.mark.parametrize("rows,cols,d,s,off", [
    (256, 256, 512, 1 / 0.07, 0),          # one tile
    (1000, 3000, 256, 1 / 0.07, 500),      # ragged rows and columns, positives off the main diagonal
    (384, 4100, 64, 20.0, 128),            # one K block, columns just past a tile boundary
    (1536, 1800, 512, 60.0, 0),            # logit_scale 60: still one sweep (reference u - 90 uses both ends of the fp32 range)
    (2048, 2048, 512, 100.0, 0),           # logit_scale 100: the norm bound fails -> exact two-sweep mode on device
    (520, 520, 768, 1 / 0.07, 0),          # d > 512: the resident-rows kernel does not apply -> streaming sweeps
] + [(rows, cols, 64, 1 / 0.07, 0) for rows, cols in TILE_EDGES])
def test_fwd_both_matches_direct_statistics(rows, cols, d, s, off):
    """clipk_fwd_both (one sweep feeding row AND column statistics when the logits are bounded; exact fallback
    otherwise) against fp64 statistics of the same bf16 values."""
    from clipk import ops
    if (rows, cols) in TILE_EDGES and torch.cuda.get_device_properties(0).multi_processor_count != 148:
        pytest.skip("the tile-count shapes are chosen for 74 clusters (148 SMs)")
    from oracle import cliploss_oracle as O
    n = max(rows, cols)
    x, t = O.synthetic_features(n, d, seed=5)
    I = torch.from_numpy(x[:rows]).cuda().bfloat16().contiguous()
    T = torch.from_numpy(t[:cols]).cuda().bfloat16().contiguous()
    be = ops._backend()
    X, Y = be.prepare(I), be.prepare(T)
    sc = torch.tensor([s], device="cuda")
    rs, pos, cs = be.fwd_both(X, Y, sc, off)
    torch.cuda.synchronize()
    S = (I.double() @ T.double().T) * float(sc[0])
    tol = 2e-5 * max(1.0, s / 14.0)
    lse_r, lse_c = rs[0] + rs[1].log(), cs[0] + cs[1].log()
    assert torch.allclose(lse_r.double(), torch.logsumexp(S, 1), rtol=0, atol=tol)
    assert torch.allclose(lse_c.double(), torch.logsumexp(S, 0), rtol=0, atol=tol)
    assert torch.allclose((rs[2] / rs[1]).double(), (torch.softmax(S, 1) * S).sum(1), rtol=0, atol=5 * tol)
    assert torch.allclose((cs[2] / cs[1]).double(), (torch.softmax(S, 0) * S).sum(0), rtol=0, atol=5 * tol)
    idx = torch.arange(rows, device="cuda")
    ok = idx + off < cols
    assert torch.allclose(pos[ok].double(), S[idx[ok], idx[ok] + off], rtol=0, atol=tol)
    if X.amax is not None:
        assert float(X.amax) == float(I.abs().max()) and float(Y.amax) == float(T.abs().max())


def test_single_sweep_and_exact_mode_agree():
    """Same inputs through the single sweep and through the exact two-sweep form (clipk_fwd_both's `exact` argument): the
    log-sum-exps of every row and column agree to fp32 rounding."""
    from clipk import ops
    x, t = O.synthetic_features(1500, 512, seed=9)
    I, T = torch.from_numpy(x).cuda().bfloat16(), torch.from_numpy(t).cuda().bfloat16()
    be = ops._backend()
    X, Y = be.prepare(I), be.prepare(T)
    sc = torch.tensor([1 / 0.07], device="cuda")
    outs = []
    for exact in (False, True):
        rs, pos, cs = be.fwd_both(X, Y, sc, 0, exact=exact)
        torch.cuda.synchronize()
        outs.append(((rs[0] + rs[1].log()).cpu().numpy(), (cs[0] + cs[1].log()).cpu().numpy(), pos.cpu().numpy()))
    for a, b in zip(outs[0], outs[1]):
        assert np.abs(a - b).max() <= 1e-5


def test_tmem_fragment_layout_hook():
    """tcgen05.ld.16x256b puts (lane, column) where the single-sweep epilogue expects it."""
    from clipk import _lib
    lib = _lib.load()
    out = torch.zeros(8 * 32 * 16, dtype=torch.int32, device="cuda")
    _lib.check(lib.clipk_debug_tmem_layout(out.data_ptr(), torch.cuda.current_stream().cuda_stream), "layout")
    torch.cuda.synchronize()
    o = out.cpu().view(4, 2, 32, 16)
    for w in range(4):
        for h in range(2):
            for t in range(32):
                for k in range(16):
                    g, c = t // 4, 2 * (t % 4)
                    lane = w * 32 + h * 16 + g + (8 if (k % 4) >= 2 else 0)
                    col = 8 * (k // 4) + c + (k % 2)
                    assert int(o[w, h, t, k]) == lane * 1000 + col


def test_megatron_loss_func_adapter_on_gpu():
    """The pretrain_CLIP.py loss_func replacement on the real kernels: loss, gradients and the top-1 accuracy (from the
    exact column maxima) against the reference's inlined formula (pretrain_CLIP.py:115-136)."""
    import torch.nn.functional as F
    from clipk.megatron_adapter import make_loss_func
    g = torch.Generator().manual_seed(11)
    text = torch.nn.functional.normalize(torch.randn(700, 256, generator=g), dim=-1)
    image = torch.nn.functional.normalize(0.25 * text + torch.nn.functional.normalize(torch.randn(700, 256, generator=g), dim=-1), dim=-1)
    text, image = (10 * text).cuda().requires_grad_(True), image.cuda().requires_grad_(True)   # un-normalised on one side
    loss, out = make_loss_func()(text, image)
    loss.backward()
    t2, i2 = text.detach().clone().requires_grad_(True), image.detach().clone().requires_grad_(True)
    labels = torch.arange(700, device="cuda")
    tl, il = t2.double() @ i2.double().T, i2.double() @ t2.double().T
    ref = (F.cross_entropy(tl, labels) + F.cross_entropy(il, labels)) / 2
    ref.backward()
    acc = (tl.argmax(-1) == labels).float().mean()
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))
    assert abs(float(out["accuracy"]) - float(acc)) <= 2.0 / 700
    assert rel(text.grad.cpu().numpy(), t2.grad.float().cpu().numpy()) <= 1e-5
    assert rel(image.grad.cpu().numpy(), i2.grad.float().cpu().numpy()) <= 1e-5


def test_full_size_step_against_torch_fp32_on_gpu():
    """BASELINE.json's benchmark shape (N = 32768, d = 512, bf16): loss, dI, dT and dlogit_scale of the fused path
    against the reference's op sequence (loss.py:112-119,135-138) evaluated in fp32 on the same GPU from the same bf16
    values (TF32 off).  The fp32 logits of that evaluation take 4.3 GB; the fused path never forms them."""
    from clipk import ClipLoss
    free, _ = torch.cuda.mem_get_info()
    if free < 40 << 30:
        pytest.skip("needs ~40 GB of free device memory for the fp32 reference")
    N, d, s = 32768, 512, 1 / 0.07
    x, t = O.synthetic_features(N, d, seed=1234)
    I = torch.from_numpy(x).cuda().bfloat16().requires_grad_(True)
    T = torch.from_numpy(t).cuda().bfloat16().requires_grad_(True)
    S = torch.tensor(s, device="cuda", requires_grad=True)
    loss = ClipLoss(local_loss=True, gather_with_grad=True, cache_labels=True)(I, T, S)
    loss.backward()
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        I2 = I.detach().float().requires_grad_(True)
        T2 = T.detach().float().requires_grad_(True)
        S2 = torch.tensor(s, device="cuda", requires_grad=True)
        labels = torch.arange(N, device="cuda")
        per_image = S2 * I2 @ T2.T
        ref = (torch.nn.functional.cross_entropy(per_image, labels) + torch.nn.functional.cross_entropy(per_image.T, labels)) / 2
        ref.backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    r = lambda a, b: float((a.float() - b).norm() / b.norm())
    assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item())
    assert r(I.grad, I2.grad) <= 2e-3 and r(T.grad, T2.grad) <= 2e-3
    assert abs(S.grad.item() - S2.grad.item()) <= 1e-4 * abs(S2.grad.item())
    # size-independent properties of the gradient: the softmax gradient has zero row and column sums, so
    # sum_i dI_i = (1^T G) T = 0 up to the positives' part ... checked through the identity sum(dI * I) == sum(dT * T)
    # (both equal s * sum(G * C), C = I T^T), which holds for any inputs
    lhs, rhs = (I.grad.float() * I.detach().float()).sum().item(), (T.grad.float() * T.detach().float()).sum().item()
    assert abs(lhs - rhs) <= 2e-3 * max(abs(lhs), abs(rhs), 1e-6)
    del per_image
    torch.cuda.empty_cache()


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 4e-3)])
def test_fused_normalize_clip_loss(dtype, tol):
    """Opt-in entry (SURVEY 8 f-1): raw embeddings in, F.normalize (model.py:216,231) + ClipLoss (loss.py:123-140) out,
    gradients with respect to the RAW embeddings (normalisation Jacobian included), against torch in fp64.  In bf16 the
    normalised features are rounded to bf16 before the loss, like the reference's autocast tower outputs, so the
    yardstick rounds them too and the tolerance covers two bf16 roundings (features in, gradients out)."""
    from clipk import fused_normalize_clip_loss
    g = torch.Generator().manual_seed(17)
    b, d, s = 900, 256, 1 / 0.07
    raw_t = torch.randn(b, d, generator=g) * 3.0
    raw_i = 0.4 * raw_t + torch.randn(b, d, generator=g) * 2.0
    I = raw_i.cuda().to(dtype).requires_grad_(True)
    T = raw_t.cuda().to(dtype).requires_grad_(True)
    S = torch.tensor(s, device="cuda", requires_grad=True)
    loss = fused_normalize_clip_loss(I, T, S)
    loss.backward()
    I2 = I.detach().double().requires_grad_(True)
    T2 = T.detach().double().requires_grad_(True)
    S2 = torch.tensor(s, device="cuda", dtype=torch.float64, requires_grad=True)
    ni, nt = torch.nn.functional.normalize(I2, dim=-1), torch.nn.functional.normalize(T2, dim=-1)
    if dtype == torch.bfloat16:     # straight-through rounding of the normalised features, as the kernels see them
        ni = ni + (ni.detach().bfloat16().double() - ni.detach())
        nt = nt + (nt.detach().bfloat16().double() - nt.detach())
    labels = torch.arange(b, device="cuda")
    logits = S2 * ni @ nt.T
    ref = (torch.nn.functional.cross_entropy(logits, labels) + torch.nn.functional.cross_entropy(logits.T, labels)) / 2
    ref.backward()
    r = lambda a, c: float((a.double() - c).norm() / c.norm())
    assert abs(loss.item() - ref.item()) <= max(tol, 1e-5) * abs(ref.item())
    assert r(I.grad, I2.grad) <= tol and r(T.grad, T2.grad) <= tol
    assert abs(S.grad.item() - S2.grad.item()) <= max(tol, 1e-4) * abs(S2.grad.item())


@pytest.mark.parametrize("name,b,N,d,rank", [
    ("C2 shard, 8 ranks", 4096, 32768, 512, 7),
    ("C3 shard, 8 ranks", 8192, 65536, 768, 3),
    ("C3 one rank", 65536, 65536, 768, 0),
    ("C4 shard, 8 ranks", 20480, 163840, 1024, 5),
])
def test_rank_block_at_baseline_sizes(name, b, N, d, rank):
    """One rank's b x N block at the sizes of BASELINE.json configs[1..3] (SURVEY 8: C2, C3, C4), through the same
    backend calls the autograd function makes (forward statistics, finalize, backward), bf16.  No O(b*N) oracle:
    sampled rows and columns are recomputed directly in fp32 on the GPU from the same bf16 values, and the
    size-independent identity <X, dX> = <Y, dY> (both equal s * sum(G * X Y^T)) covers the whole block."""
    from clipk import ops
    need = (N * d * 10 + b * d * 10 + 2 * (b // 128 + 1) * N * 4 + (1 << 30))
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need >> 20} MiB of free device memory")
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    off, s = rank * b, 1 / 0.07
    Yf = torch.nn.functional.normalize(torch.randn(N, d, device="cuda", generator=g), dim=-1)
    Z = torch.nn.functional.normalize(torch.randn(b, d, device="cuda", generator=g), dim=-1)
    X = torch.nn.functional.normalize(0.3 * Yf[off:off + b] + 0.954 * Z, dim=-1).bfloat16()   # positives: cos ~ 0.3
    Y = Yf.bfloat16()
    del Yf, Z
    be = ops._backend()
    sc = torch.tensor([s], device="cuda")
    Xo, Yo = be.prepare(X), be.prepare(Y)
    parts = torch.empty(1, 3, N, dtype=torch.float32, device="cuda")
    row_stats, pos, _ = be.fwd_both(Xo, Yo, sc, off, col_out=parts[0])
    lse_row, lse_col, sums = be.finalize(row_stats, pos, parts, off)
    gscale = torch.tensor([1.0 / (2 * b)], device="cuda")
    dX, dY = be.bwd(Xo, Yo, be.prepare_grad(Xo), be.prepare_grad(Yo), sc, off, lse_row, lse_col, 1.0, 1.0, gscale,
                    True, True)
    torch.cuda.synchronize()
    assert dX.shape == (b, d) and dY.shape == (N, d)
    assert bool(torch.isfinite(dX).all()) and bool(torch.isfinite(dY).all()) and bool(torch.isfinite(sums).all())

    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        Xf, Yf = X.float(), Y.float()
        ri = torch.randperm(b, device="cuda", generator=g)[:96].sort().values
        ri[0], ri[-1] = 0, b - 1                                   # first and last row of the block
        cj = torch.randperm(N, device="cuda", generator=g)[:96].sort().values
        cj[0], cj[1], cj[-1] = 0, off, N - 1                        # first, a positive's and the last column
        S_r = s * Xf[ri] @ Yf.T                                     # [96, N]
        S_c = s * Xf @ Yf[cj].T                                     # [b, 96]
        assert torch.allclose(lse_row[ri], torch.logsumexp(S_r, 1), rtol=0, atol=2e-4)
        assert torch.allclose(lse_col[cj], torch.logsumexp(S_c, 0), rtol=0, atol=2e-4)
        assert torch.allclose(pos[ri], S_r[torch.arange(96, device="cuda"), ri + off], rtol=0, atol=2e-4)
        # cross-entropy sums of the block against the kernel's own statistics
        assert abs(sums[0].item() - (lse_row - pos).double().sum().item()) <= 1e-4 * abs(sums[0].item())
        # sampled gradient rows / columns; the other direction's LSEs come from the kernel (checked just above)
        gs = s * gscale.item()
        G_r = torch.exp(S_r - lse_row[ri, None]) + torch.exp(S_r - lse_col[None, :])
        G_r[torch.arange(96, device="cuda"), ri + off] -= 2.0
        ref_dX = gs * G_r @ Yf
        G_c = torch.exp(S_c - lse_row[:, None]) + torch.exp(S_c - lse_col[None, cj])
        inside = (cj >= off) & (cj < off + b)
        G_c[(cj - off)[inside], torch.arange(96, device="cuda")[inside]] -= 2.0
        ref_dY = gs * G_c.T @ Xf
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    r = lambda a, c: float((a.double() - c.double()).norm() / c.double().norm())
    assert r(dX[ri], ref_dX) <= 2e-3, ("dX", r(dX[ri], ref_dX))
    assert r(dY[cj], ref_dY) <= 2e-3, ("dY", r(dY[cj], ref_dY))
    lhs, rhs = (Xf * dX).double().sum().item(), (Yf * dY).double().sum().item()
    assert abs(lhs - rhs) <= 2e-3 * max(abs(lhs), abs(rhs)), (lhs, rhs)


@pytest.mark.parametrize("rows,cols,d,off", [(1024, 4096, 256, 1024), (700, 2100, 512, 0), (512, 1536, 768, 512)])
def test_split_row_col_backward_equals_two_passes(rows, cols, d, off):
    """clipk_bwd's split_row_col (local_loss without gather_with_grad, loss.py:53-56): dX from the row softmax and dY from
    the column softmax out of ONE recompute with two planes, against the two single-softmax passes it replaces."""
    from clipk import ops
    be = ops._backend()
    x, _ = O.synthetic_features(rows, d, seed=11)
    _, t = O.synthetic_features(cols, d, seed=12)
    X = be.prepare(torch.from_numpy(x).cuda().bfloat16())
    Y = be.prepare(torch.from_numpy(t).cuda().bfloat16())
    sc = torch.tensor([1 / 0.07], device="cuda")
    parts = torch.empty(1, 3, cols, dtype=torch.float32, device="cuda")
    rs, pos, _ = be.fwd_both(X, Y, sc, off, col_out=parts[0])
    lse_row, lse_col, _ = be.finalize(rs, pos, parts, off)
    Xg, Yg = be.prepare_grad(X), be.prepare_grad(Y)
    gs = torch.tensor([1.0 / (2 * rows)], device="cuda")
    dX1, _ = be.bwd(X, Y, Xg, Yg, sc, off, lse_row, lse_col, 1.0, 0.0, gs, True, False)
    _, dY1 = be.bwd(X, Y, Xg, Yg, sc, off, lse_row, lse_col, 0.0, 1.0, gs, False, True)
    dX2, dY2 = be.bwd(X, Y, Xg, Yg, sc, off, lse_row, lse_col, 1.0, 1.0, gs, True, True, split=True)
    torch.cuda.synchronize()
    # same fp16 G entries, same fp16 operands: only the summation order inside the tensor core may differ
    assert rel(dX2.cpu().numpy(), dX1.cpu().numpy()) <= 2e-6 and rel(dY2.cpu().numpy(), dY1.cpu().numpy()) <= 2e-6
    assert float(dX1.abs().sum()) > 0 and float(dY1.abs().sum()) > 0
