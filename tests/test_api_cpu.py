"""Host-side checks that need no GPU: the C-ABI library loads and exports every symbol include/clipk.h declares, the
drop-in module mirrors the reference's names and label semantics bit-exactly, and the product refuses to run without
a GPU instead of falling back."""
import ctypes
import os
import re
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from clipk import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "clipk.h")).read()
    declared = set(re.findall(r"\b(clipk_[a-z0-9_]+)\s*\(", header))
    assert {"clipk_fwd_stats", "clipk_fwd_both", "clipk_finalize", "clipk_bwd", "clipk_to_f16", "clipk_cast", "clipk_gemm16"} <= declared
    for name in declared:
        assert hasattr(lib, name), name                 # dlsym resolves it
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    assert lib.clipk_version() == 2


def test_abi_reports_errors_without_a_gpu():
    from clipk import _lib
    lib = _lib.load()
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    rc = lib.clipk_check_device()
    assert rc != 0
    assert len(lib.clipk_last_error()) > 0
    # argument validation comes before any CUDA call
    assert lib.clipk_cast(None, None, 4, 0, None) == -1
    assert lib.clipk_fwd_workspace_bytes(128, 128, 64, 0) > 0
    assert lib.clipk_bwd_workspace_bytes(128, 128, 64, 3) > 0


def test_no_cpu_fallback():
    from clipk import ClipLoss
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    I = torch.randn(8, 16, requires_grad=True)
    T = torch.randn(8, 16, requires_grad=True)
    with pytest.raises(Exception):
        ClipLoss()(I, T, torch.tensor(10.0))


def test_module_surface_matches_reference():
    import clipk
    from clipk import loss as L
    for name in ("ClipLoss", "CoCaLoss", "DistillClipLoss", "create_loss", "gather_features"):
        assert hasattr(clipk, name)
    import inspect
    sig = inspect.signature(L.ClipLoss.__init__)
    assert list(sig.parameters)[1:] == ["local_loss", "gather_with_grad", "cache_labels", "rank", "world_size", "use_horovod"]
    assert [p.default for p in list(sig.parameters.values())[1:]] == [False, False, False, 0, 1, False]
    assert list(inspect.signature(L.ClipLoss.forward).parameters)[1:] == ["image_features", "text_features", "logit_scale", "output_dict"]
    # the reference's parameters in the reference's order; `group` is an optional extension after them
    assert list(inspect.signature(L.gather_features).parameters) == ["image_features", "text_features", "local_loss", "gather_with_grad", "rank", "world_size", "use_horovod", "group"]
    assert inspect.signature(L.gather_features).parameters["group"].default is None
    with pytest.raises(NotImplementedError):
        L.ClipLoss(use_horovod=True)


def test_labels_bit_exact_and_cache_semantics():
    from clipk import ClipLoss
    from oracle import cliploss_oracle as O
    dev = torch.device("cpu")
    for (ll, W, r, n) in [(False, 1, 0, 16), (True, 4, 2, 8), (False, 4, 3, 32), (True, 2, 1, 100)]:
        m = ClipLoss(local_loss=ll, cache_labels=True, rank=r, world_size=W)
        lab = m.get_ground_truth(dev, n)
        assert lab.dtype == torch.long
        assert np.array_equal(lab.numpy(), O.ground_truth(n, r, W, ll))
        assert m.get_ground_truth(dev, n) is lab                  # cached
        lab2 = m.get_ground_truth(dev, n + 4)                      # accum-freq changes num_logits: cache invalidated
        assert lab2.numel() == n + 4 and m.prev_num_logits == n + 4
    m = ClipLoss(cache_labels=False)
    assert m.get_ground_truth(dev, 4) is not m.get_ground_truth(dev, 4) and m.labels == {}


def test_create_loss_plumbing():
    from clipk import create_loss, ClipLoss, CoCaLoss, DistillClipLoss
    a = types.SimpleNamespace(distill=False, model="ViT-B-32", local_loss=True, gather_with_grad=True, rank=3,
                              world_size=8, horovod=False)
    m = create_loss(a)
    assert type(m) is ClipLoss and m.local_loss and m.gather_with_grad and m.cache_labels and m.rank == 3 and m.world_size == 8
    a.model = "coca_ViT-B-32"
    a.coca_caption_loss_weight, a.coca_contrastive_loss_weight = 2.0, 1.0
    assert type(create_loss(a)) is CoCaLoss
    a.distill = True
    assert type(create_loss(a)) is DistillClipLoss


def test_single_process_host_logic_with_emulated_kernels():
    """W = 1 autograd plumbing (output_dict, float scale, grad_output) with the kernel calls emulated on CPU."""
    from clipk import ClipLoss, ops
    from oracle import cliploss_oracle as O
    from tests.emu_backend import EmuBackend
    ops.set_backend_for_testing(EmuBackend())
    try:
        x, t = O.synthetic_features(24, 32, seed=3)
        I = torch.from_numpy(x).requires_grad_(True)
        T = torch.from_numpy(t).requires_grad_(True)
        s = torch.tensor(12.5, requires_grad=True)
        out = ClipLoss()(I, T, s, output_dict=True)
        (out["contrastive_loss"] * 2.0).backward()
        ref = O.clip_loss_single(x, t, 12.5, grad_output=2.0)
        assert abs(out["contrastive_loss"].item() - ref.loss) < 1e-5 * ref.loss
        assert np.linalg.norm(I.grad.numpy() - ref.d_image) < 1e-5 * np.linalg.norm(ref.d_image)
        assert np.linalg.norm(T.grad.numpy() - ref.d_text) < 1e-5 * np.linalg.norm(ref.d_text)
        assert abs(s.grad.item() - ref.d_scale) < 1e-5 * abs(ref.d_scale)
        l2 = ClipLoss()(I.detach(), T.detach(), 12.5)              # python-float scale, no grads
        assert abs(l2.item() - ref.loss) < 1e-5 * ref.loss
    finally:
        ops.set_backend_for_testing(None)


@pytest.mark.parametrize("d,dtype,tol", [(100, torch.float32, 1e-5), (36, torch.float32, 1e-5), (72, torch.float16, 2e-3),
                                         (64, torch.float16, 2e-3), (200, torch.bfloat16, 8e-3)])
def test_odd_widths_and_fp16_features_host_logic(d, dtype, tol):
    """Widths that are not a multiple of the 64-element K block are zero-padded on the host and the padding's gradient
    columns dropped; fp16 features go through the fp32 path and come back as fp16.  Kernel calls emulated on CPU."""
    from clipk import ClipLoss, ops
    from oracle import cliploss_oracle as O
    from tests.emu_backend import EmuBackend
    seen = []

    class Spy(EmuBackend):
        def prepare(self, x):
            seen.append((tuple(x.shape), x.dtype))
            return super().prepare(x)

    ops.set_backend_for_testing(Spy())
    try:
        x, t = O.synthetic_features(20, d, seed=d)
        I = torch.from_numpy(x).to(dtype).requires_grad_(True)
        T = torch.from_numpy(t).to(dtype).requires_grad_(True)
        s = torch.tensor(9.0, requires_grad=True)
        loss = ClipLoss()(I, T, s)
        loss.backward()
        assert all(shape[1] % 64 == 0 for shape, _ in seen), seen           # the kernels only ever see whole K blocks
        assert all(dt == (torch.bfloat16 if dtype == torch.bfloat16 else torch.float32) for _, dt in seen), seen
        assert I.grad.shape == I.shape and I.grad.dtype == dtype and T.grad.dtype == dtype and loss.dtype == torch.float32
        ref = O.clip_loss_single(I.detach().float().numpy(), T.detach().float().numpy(), 9.0)
        assert abs(loss.item() - ref.loss) <= 1e-5 * ref.loss
        assert np.linalg.norm(I.grad.float().numpy() - ref.d_image) <= tol * np.linalg.norm(ref.d_image)
        assert np.linalg.norm(T.grad.float().numpy() - ref.d_text) <= tol * np.linalg.norm(ref.d_text)
        assert abs(s.grad.item() - ref.d_scale) <= 1e-5 * max(abs(ref.d_scale), 1 / 9.0)
        with pytest.raises(TypeError):
            ClipLoss()(I.detach().double(), T.detach().double(), s)
    finally:
        ops.set_backend_for_testing(None)


def test_empty_batch_is_nan_like_the_reference():
    """Zero rows: the reference's F.cross_entropy means over nothing -> NaN loss, empty gradients (loss.py:135-138).
    Handled on the host, before any kernel: works without a GPU."""
    from clipk import ClipLoss
    I = torch.zeros(0, 64, requires_grad=True)
    T = torch.zeros(0, 64, requires_grad=True)
    s = torch.tensor(10.0, requires_grad=True)
    loss = ClipLoss()(I, T, s)
    assert loss.dim() == 0 and torch.isnan(loss)
    loss.backward()
    assert I.grad.shape == (0, 64) and T.grad.shape == (0, 64)
    ref = (torch.nn.functional.cross_entropy(s * I.detach() @ T.detach().T, torch.arange(0)) +
           torch.nn.functional.cross_entropy(s * T.detach() @ I.detach().T, torch.arange(0))) / 2
    assert torch.isnan(ref)


def test_megatron_loss_func_adapter_matches_reference_formula():
    """clipk.megatron_adapter.make_loss_func keeps the signature and return convention of pretrain_CLIP.py:115-136;
    on the CPU emulation backend (host logic only) its values equal the reference's inlined formula."""
    import torch.nn.functional as F
    from clipk import ops
    from clipk.megatron_adapter import make_loss_func
    from tests.emu_backend import EmuBackend
    ops.set_backend_for_testing(EmuBackend())
    try:
        g = torch.Generator().manual_seed(3)
        text = torch.randn(48, 32, generator=g, requires_grad=True)
        image = (text.detach() * 0.7 + 0.5 * torch.randn(48, 32, generator=g)).requires_grad_(True)
        loss, out = make_loss_func()(text, image)
        loss.backward()
        t2, i2 = text.detach().clone().requires_grad_(True), image.detach().clone().requires_grad_(True)
        labels = torch.arange(48)
        tl, il = t2.float() @ i2.float().T, i2.float() @ t2.float().T
        ref = (F.cross_entropy(tl, labels) + F.cross_entropy(il, labels)) / 2
        ref.backward()
        acc = (tl.argmax(-1) == labels).float().mean()
        assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))
        assert float(out["loss"]) == pytest.approx(float(ref), rel=1e-5)
        assert float(out["accuracy"]) == pytest.approx(float(acc), abs=1e-6)
        assert torch.allclose(text.grad, t2.grad, rtol=1e-4, atol=1e-6)
        assert torch.allclose(image.grad, i2.grad, rtol=1e-4, atol=1e-6)
    finally:
        ops.set_backend_for_testing(None)


def test_fused_normalize_entry_host_logic():
    """fused_normalize_clip_loss on the CPU emulation backend: normalise + loss + Jacobian against torch autograd."""
    import torch.nn.functional as F
    from clipk import ops, fused_normalize_clip_loss
    from tests.emu_backend import EmuBackend
    ops.set_backend_for_testing(EmuBackend())
    try:
        g = torch.Generator().manual_seed(5)
        I = (torch.randn(40, 24, generator=g) * 2).requires_grad_(True)
        T = (torch.randn(40, 24, generator=g) * 3).requires_grad_(True)
        s = torch.tensor(8.0, requires_grad=True)
        loss = fused_normalize_clip_loss(I, T, s)
        loss.backward()
        I2, T2, s2 = I.detach().clone().requires_grad_(True), T.detach().clone().requires_grad_(True), torch.tensor(8.0, requires_grad=True)
        logits = s2 * F.normalize(I2, dim=-1) @ F.normalize(T2, dim=-1).T
        labels = torch.arange(40)
        ref = (F.cross_entropy(logits, labels) + F.cross_entropy(logits.T, labels)) / 2
        ref.backward()
        assert float(loss) == pytest.approx(float(ref), rel=1e-5)
        assert torch.allclose(I.grad, I2.grad, rtol=1e-4, atol=1e-6) and torch.allclose(T.grad, T2.grad, rtol=1e-4, atol=1e-6)
        assert float(s.grad) == pytest.approx(float(s2.grad), rel=1e-4)
    finally:
        ops.set_backend_for_testing(None)


@pytest.mark.parametrize("normalize", [False, True])
def test_fused_step_route_host_logic(normalize):
    """bf16 features of a width that is a multiple of 64 take the fused step (clipk_step_forward / _backward): buffers,
    coefficients, saved state and the label cache, with the two entries emulated on the CPU."""
    from clipk import ClipLoss, ops, fused_normalize_clip_loss
    from oracle import cliploss_oracle as O
    from tests.emu_backend import EmuBackend
    be = EmuBackend()
    calls = []
    fwd, bwd = be.step_forward, be.step_backward
    be.step_forward = lambda st: (calls.append("f"), fwd(st))[1]
    be.step_backward = lambda st: (calls.append("b"), bwd(st))[1]
    ops.set_backend_for_testing(be)
    try:
        g = torch.Generator().manual_seed(11)
        raw_i, raw_t = torch.randn(48, 128, generator=g) * 1.7, torch.randn(48, 128, generator=g) * 0.6
        if not normalize:
            raw_i, raw_t = torch.nn.functional.normalize(raw_i, dim=-1), torch.nn.functional.normalize(raw_t, dim=-1)
        I = raw_i.bfloat16().requires_grad_(True)
        T = raw_t.bfloat16().requires_grad_(True)
        s = torch.tensor(9.0, requires_grad=True)
        mod = ClipLoss(cache_labels=True)
        loss = fused_normalize_clip_loss(I, T, s) if normalize else mod(I, T, s)
        (loss * 1.5).backward()
        assert calls == ["f", "b"]
        assert loss.dtype == torch.float32 and I.grad.dtype == torch.bfloat16 and s.grad.shape == s.shape
        if not normalize:
            assert mod.prev_num_logits == 48 and torch.equal(mod.labels[I.device], torch.arange(48))
        # reference: the oracle on the operand values (normalised in fp64, rounded to bf16), chained through the Jacobian
        x64, t64 = I.detach().double(), T.detach().double()
        if normalize:
            xn, tn = x64 / x64.norm(dim=-1, keepdim=True), t64 / t64.norm(dim=-1, keepdim=True)
        else:
            xn, tn = x64, t64
        xo, to = xn.bfloat16().double().numpy(), tn.bfloat16().double().numpy()
        ref = O.clip_loss_single(xo, to, 9.0, grad_output=1.5)
        dI, dT = torch.from_numpy(ref.d_image), torch.from_numpy(ref.d_text)
        if normalize:
            for gr, y, x in ((dI, torch.from_numpy(xo), x64), (dT, torch.from_numpy(to), t64)):
                gr.copy_((gr - y * (gr * y).sum(-1, keepdim=True)) / x.norm(dim=-1, keepdim=True))
        assert abs(loss.item() - ref.loss) <= 1e-5 * ref.loss
        assert (I.grad.double() - dI).norm() <= 8e-3 * dI.norm() and (T.grad.double() - dT).norm() <= 8e-3 * dT.norm()
        assert abs(s.grad.item() - ref.d_scale) <= 1e-5 * abs(ref.d_scale)
    finally:
        ops.set_backend_for_testing(None)


def test_in_place_change_of_the_features_is_detected():
    """The features are read again by the backward (in place, no copy): autograd must notice a modification in between."""
    from clipk import ClipLoss, ops
    from tests.emu_backend import EmuBackend
    ops.set_backend_for_testing(EmuBackend())
    try:
        base = torch.nn.functional.normalize(torch.randn(16, 64), dim=-1).bfloat16().requires_grad_(True)
        I = base * 1.0                      # non-leaf, so that it may be modified in place
        T = torch.nn.functional.normalize(torch.randn(16, 64), dim=-1).bfloat16().requires_grad_(True)
        loss = ClipLoss()(I, T, torch.tensor(5.0))
        I.mul_(2.0)
        with pytest.raises(RuntimeError, match="modified by an inplace operation"):
            loss.backward()
    finally:
        ops.set_backend_for_testing(None)


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the GPU arm): exactly one JSON line on stdout
    with the contract's keys; here with a tiny sample so that it takes seconds."""
    import json, subprocess, sys
    env = dict(os.environ, OMP_NUM_THREADS="2")
    code = ("import sys; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0'];"
            "import runpy, bench; bench.CPU_SAMPLE_BATCH = 512; bench.CPU_ARM_BUDGET_S = 0.0; bench.main()")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "samples/s" and j["higher_is_better"] is True
    # the reference module itself when baseline/_ref holds it (the build container, the GPU box), else the oracle's port
    assert j["cpu_baseline"]["kind"] in ("reference", "port") and j["cpu_baseline"]["cores"] >= 1
    assert j["cpu_baseline"]["sample_batch"] == 512 and j["cpu_baseline"]["extrapolated"] is True
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0 and j["value"] > 0


def test_bench_dump_outputs_writes_float32_with_a_seeded_row_sample(tmp_path):
    """`bench.py --dump-outputs`: float32 .npy per output; a matrix above the budget becomes the same sorted row sample
    on every call, so that dumps of two builds line up row for row."""
    import bench
    g = torch.Generator().manual_seed(0)
    rows = bench.DUMP_MATRIX_BYTES // (4 * 64)
    big = torch.randn(3 * rows, 64, generator=g).bfloat16()
    small = torch.randn(rows, 64, generator=g).bfloat16()
    for out in ("a", "b"):
        bench.dump_outputs(str(tmp_path / out), {"loss": torch.tensor(1.5), "big": big, "small": small})
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("loss", "big", "small")}
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["loss"].shape == () and float(a["loss"]) == 1.5
    assert np.array_equal(a["small"], small.float().numpy())
    assert a["big"].shape == (rows, 64) and a["big"].nbytes <= bench.DUMP_MATRIX_BYTES
    assert np.array_equal(a["big"], np.load(tmp_path / "b" / "big.npy"))
    full = big.float().numpy()
    idx = [int(np.flatnonzero((full == r).all(axis=1))[0]) for r in a["big"][:50]]
    assert idx == sorted(set(idx))                  # distinct rows of the input, in order


@pytest.mark.parametrize("n,d,s", [(96, 48, 1 / 0.07), (130, 32, 100.0)])
def test_bench_parity_checker_matches_the_oracle(n, d, s):
    """bench.py's parity phase checks the benchmark's own shapes against `torch_fp32_reference` (chunked fp32 torch, no
    N x N matrix held).  That checker is itself pinned here: single process, against the fp64 oracle."""
    import bench
    from oracle import cliploss_oracle as O
    x, t = O.synthetic_features(n, d, seed=2)
    I, T = torch.from_numpy(x), torch.from_numpy(t)
    loss, dI, dT, ds = bench.torch_fp32_reference(I, T, s, 0, 1, True, True, chunk=50)
    ref = O.clip_loss_single(x, t, s)
    tol = 2e-5 if s < 50 else 3e-4
    assert abs(loss - ref.loss) <= tol * abs(ref.loss)
    assert np.linalg.norm(dI.numpy() - ref.d_image) <= tol * np.linalg.norm(ref.d_image)
    assert np.linalg.norm(dT.numpy() - ref.d_text) <= tol * np.linalg.norm(ref.d_text)
    assert abs(ds - ref.d_scale) <= tol * max(abs(ref.d_scale), 1 / s)
