"""SigLipLoss on the clipk_siglip kernels (B200): parity against the float64 oracle on the bf16 values upcast, numerics in
the regimes that stress the epilogues, determinism, memory, the kernel list of a step, and NCCL data parallelism."""
import os
import tempfile

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import siglip_oracle as SO

pytestmark = pytest.mark.gpu


def _pair(b, d, seed, pos_cos=None):
    """unit-norm bf16 features; pos_cos: text row i = pos_cos * x_i + sqrt(1 - pos_cos^2) * noise (the positive pair's
    cosine), else independent rows (a hard batch: positive cosine ~ 0)"""
    g = torch.Generator().manual_seed(seed)
    x = F.normalize(torch.randn(b, d, generator=g, dtype=torch.float64), dim=-1)
    n = F.normalize(torch.randn(b, d, generator=g, dtype=torch.float64), dim=-1)
    if pos_cos is None:
        t = n
    else:
        n = F.normalize(n - (n * x).sum(-1, keepdim=True) * x, dim=-1)
        t = pos_cos * x + (1 - pos_cos ** 2) ** 0.5 * n
    return x.to(torch.bfloat16).cuda(), t.to(torch.bfloat16).cuda()


def _run(x, t, s, bias, go=1.0, dtype=None):
    from clipk import SigLipLoss
    I = (x if dtype is None else x.to(dtype)).clone().requires_grad_(True)
    T = (t if dtype is None else t.to(dtype)).clone().requires_grad_(True)
    S = torch.tensor(s, device="cuda", requires_grad=True)
    B = None if bias is None else torch.tensor(bias, device="cuda", requires_grad=True)
    loss = SigLipLoss()(I, T, S, B)
    (loss * go).backward()
    torch.cuda.synchronize()
    return loss, I.grad, T.grad, S.grad, None if B is None else B.grad


def _check(x, t, s, bias, out, go=1.0):
    """loss <= 1e-4 rel; ds, dt <= 1e-3 of the sums of magnitudes; feature gradients <= 2e-3 normwise and
    max |err| <= 4e-3 max |ref| (ClipLoss's bf16 bar)"""
    loss, dI, dT, dS, dB = out
    X, Tn = x.double().cpu().numpy(), t.double().cpu().numpy()
    ref = SO.siglip_single(X, Tn, s, 0.0 if bias is None else bias, go)
    assert abs(float(loss) - ref.loss) <= 1e-4 * abs(ref.loss), (float(loss), ref.loss)
    L = s * X @ Tn.T + (0.0 if bias is None else bias)
    from scipy.special import expit
    G = np.abs(expit(L))
    np.fill_diagonal(G, expit(-np.diag(L)))
    k = 1e-3 * abs(go) / len(X)
    assert abs(float(dS) - ref.d_scale) <= k * (G * np.abs(X @ Tn.T)).sum(), (float(dS), ref.d_scale)
    if dB is not None:
        assert abs(float(dB) - ref.d_bias) <= k * G.sum(), (float(dB), ref.d_bias)
    for got, want in ((dI, ref.d_image), (dT, ref.d_text)):
        got = got.double().cpu().numpy()
        assert np.linalg.norm(got - want) <= 2e-3 * np.linalg.norm(want)
        assert np.abs(got - want).max() <= 4e-3 * np.abs(want).max()


REGIMES = {"init": (10.0, -10.0, None), "s100": (100.0, -15.0, None), "separated": (100.0, -15.0, 0.95),
           "hard": (100.0, -15.0, 0.0)}


@pytest.mark.parametrize("regime", list(REGIMES))
@pytest.mark.parametrize("b,d", [(128, 64), (300, 100), (300, 512), (4096, 512), (1000, 768), (300, 1024)])
def test_parity_against_oracle(b, d, regime):
    """b = 300, 1000: N not a multiple of 256; d = 100: padded to 128; d = 768, 1024: the streaming (not A-resident)
    sweeps."""
    s, bias, pos_cos = REGIMES[regime]
    x, t = _pair(b, d, seed=b + d, pos_cos=pos_cos)
    _check(x, t, s, bias, _run(x, t, s, bias))


def test_separated_batch_keeps_tiny_gradients():
    """Orthonormal image rows, text row i = 0.99 x_i + 0.14 n_i with n orthogonal to every x: at s = 40, t = -20 the
    positives sit at l = +19.6 and every negative at l = -20, so every |g| is ~2e-9.  The loss is a sum of such terms and
    the gradients are made of them: the G panel's power of two must lift them out of fp16's subnormals."""
    b, d = 128, 256
    q, _ = torch.linalg.qr(torch.randn(d, d, generator=torch.Generator().manual_seed(5), dtype=torch.float64))
    x, n = q[:, :b].T, q[:, b:2 * b].T
    t = 0.99 * x + (1 - 0.99 ** 2) ** 0.5 * n
    x, t = x.to(torch.bfloat16).cuda(), t.to(torch.bfloat16).cuda()
    out = _run(x, t, 40.0, -20.0)
    _check(x, t, 40.0, -20.0, out)
    assert 0 < float(out[0]) < 1e-5


def test_no_bias_grad_output_and_autocast():
    x, t = _pair(384, 256, seed=9)
    _check(x, t, 10.0, None, _run(x, t, 10.0, None, go=-2.5), go=-2.5)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = _run(x, t, 10.0, -10.0, dtype=torch.float32)       # fp32 features, cast to bf16 once
    assert out[1].dtype == torch.float32 and out[0].dtype == torch.float32
    _check(x, t, 10.0, -10.0, out)


def test_row_strided_views():
    from clipk import siglip_loss
    x, t = _pair(256, 128, seed=11)
    big_x = torch.zeros(256, 192, dtype=torch.bfloat16, device="cuda")
    big_t = torch.zeros(256, 192, dtype=torch.bfloat16, device="cuda")
    big_x[:, :128], big_t[:, :128] = x, t
    big_x.requires_grad_(True)
    big_t.requires_grad_(True)
    loss = siglip_loss(big_x[:, :128], big_t[:, :128], 10.0, -10.0)
    loss.backward()
    ref = _run(x, t, 10.0, -10.0)
    assert torch.equal(loss.detach(), ref[0].detach())
    assert torch.equal(big_x.grad[:, :128], ref[1]) and torch.equal(big_t.grad[:, :128], ref[2])


def test_in_place_change_raises():
    from clipk import siglip_loss
    x, t = _pair(256, 128, seed=13)
    I, T = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
    loss = siglip_loss(I * 1, T, 10.0, -10.0)
    with torch.no_grad():
        T.mul_(2.0)
    with pytest.raises(RuntimeError):
        loss.backward()


def test_two_calls_are_bit_identical():
    x, t = _pair(2048, 512, seed=17)
    a, b = _run(x, t, 10.0, -10.0), _run(x, t, 10.0, -10.0)
    for u, v in zip(a, b):
        assert torch.equal(u, v)


def test_nan_feature_gives_nan_loss():
    x, t = _pair(256, 128, seed=19)
    x[3, 5] = float("nan")
    loss, dI, _, _, _ = _run(x, t, 10.0, -10.0)
    assert torch.isnan(loss) and torch.isnan(dI).any()


def test_peak_memory_far_below_the_logits():
    """b = N = 16384, d = 512: the bf16 logits alone would be b * N * 2 = 512 MiB; the fused step's extra memory (G panel,
    fp16 operand copies, fp32 gradient accumulators, bf16 gradients) stays below 40 % of that."""
    b, d = 16384, 512
    x, t = _pair(b, d, seed=23)
    from clipk import siglip_loss
    I, T = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
    siglip_loss(I, T, 10.0, -10.0).backward()           # warm-up: caches, workspace shapes
    I.grad = T.grad = None
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    siglip_loss(I, T, 10.0, -10.0).backward()
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert extra <= 0.4 * b * b * 2, extra


def test_profiler_kernel_list_has_no_materialising_ops():
    from torch.profiler import ProfilerActivity, profile
    from clipk import siglip_loss
    x, t = _pair(1024, 256, seed=29)
    I, T = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
    siglip_loss(I, T, 10.0, -10.0).backward()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        siglip_loss(I, T, 10.0, -10.0).backward()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    assert any("siglip_fwd_kernel" in n for n in names) and any("siglip_grad_kernel" in n for n in names), names
    assert not any(n in ("aten::mm", "aten::matmul", "aten::addmm") or "logsigmoid" in n or "log_sigmoid" in n
                   for n in names), names


def test_full_size_step_against_torch_fp32_on_gpu():
    """N = 32768, d = 512 against the formula evaluated in fp32 on the GPU, 2048 rows at a time (fp64 on the CPU would
    take minutes at this size)."""
    b, d, s, bias = 32768, 512, 10.0, -10.0
    x, t = _pair(b, d, seed=31)
    loss, dI, dT, dS, dB = _run(x, t, s, bias)
    X, Tf = x.float(), t.float()
    ref_loss, dX, dY = 0.0, torch.zeros(b, d, device="cuda"), torch.zeros(b, d, device="cuda")
    ds = dt = ds_mag = dt_mag = 0.0
    for r0 in range(0, b, 2048):
        dots = X[r0:r0 + 2048] @ Tf.T
        L = s * dots + bias
        idx = torch.arange(L.shape[0], device="cuda")
        z = -torch.ones_like(L)
        z[idx, idx + r0] = 1.0
        ref_loss += float(F.softplus(-z * L).double().sum())
        G = torch.sigmoid(L)
        G[idx, idx + r0] = -torch.sigmoid(-L[idx, idx + r0])
        dX[r0:r0 + 2048] = s / b * G @ Tf
        dY += s / b * G.T @ X[r0:r0 + 2048]
        ds += float((G * dots).double().sum()) / b
        dt += float(G.double().sum()) / b
        ds_mag += float((G.abs() * dots.abs()).double().sum()) / b
        dt_mag += float(G.abs().double().sum()) / b
    ref_loss /= b
    assert abs(float(loss) - ref_loss) <= 1e-4 * ref_loss
    assert abs(float(dB) - dt) <= 1e-3 * dt_mag and abs(float(dS) - ds) <= 1e-3 * ds_mag
    for got, want in ((dI, dX), (dT, dY)):
        assert (got.float() - want).norm() <= 2e-3 * want.norm()


def _dist_worker(rank, world, tmp):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "megatron-clip_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    from clipk import SigLipLoss
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"file://{tmp}/store", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    x, t = _pair(640, 256, seed=40 + rank)
    I, T = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
    S = torch.tensor(10.0, device="cuda", requires_grad=True)
    B = torch.tensor(-10.0, device="cuda", requires_grad=True)
    loss = SigLipLoss(rank=rank, world_size=world)(I, T, S, B)
    loss.backward()
    torch.cuda.synchronize()
    np.savez(f"{tmp}/sig{rank}.npz", loss=loss.item(), image=x.float().cpu().numpy(), text=t.float().cpu().numpy(),
             d_image=I.grad.float().cpu().numpy(), d_text=T.grad.float().cpu().numpy(), d_scale=S.grad.item(),
             d_bias=B.grad.item())
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_nccl_ranks_against_oracle(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_dist_worker, args=(world, tmp), nprocs=world, join=True)
        outs = [dict(np.load(f"{tmp}/sig{r}.npz")) for r in range(world)]
    ref = SO.siglip_world([o["image"] for o in outs], [o["text"] for o in outs], 10.0, -10.0)
    for o, g in zip(outs, ref):
        assert abs(float(o["loss"]) - g.loss) <= 1e-4 * abs(g.loss)
        for k in ("d_image", "d_text"):
            assert np.linalg.norm(o[k] - getattr(g, k)) <= 2e-3 * np.linalg.norm(getattr(g, k))
        assert abs(float(o["d_scale"]) - g.d_scale) <= 1e-3 * max(abs(g.d_scale), abs(g.d_bias))
        assert abs(float(o["d_bias"]) - g.d_bias) <= 1e-3 * abs(g.d_bias)
