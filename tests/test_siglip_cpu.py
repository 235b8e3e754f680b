"""SigLipLoss on the CPU: the float64 oracle against a transcription of open_clip's code, and the host orchestration of
clipk.siglip (routes, padding, gather / reduce-scatter over gloo, gradient shapes and dtypes) on emulated kernel entries."""
import os
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from oracle import siglip_oracle as SO
from tests.emu_backend import EmuBackend


class SigEmu(EmuBackend):
    """clipk_siglip_forward / _backward in float64 with CudaBackend's signatures and return conventions."""

    def __init__(self):
        self.calls = []

    @staticmethod
    def _G(X, Y, scale, bias, off):
        assert X.dtype == torch.bfloat16 and Y.dtype == torch.bfloat16 and X.shape[1] % 64 == 0 and X.is_contiguous()
        x, y = X.double(), Y.double()
        dots = x @ y.T
        L = float(scale[0]) * dots + (0.0 if bias is None else float(bias[0]))
        i = torch.arange(x.shape[0])
        return x, y, dots, L, i, i + off

    def siglip_forward(self, X, Y, scale, bias, diag_offset):
        self.calls.append("siglip_forward")
        x, _, _, L, i, j = self._G(X, Y, scale, bias, diag_offset)
        z = -torch.ones_like(L)
        z[i, j] = 1.0
        state = torch.zeros(8, dtype=torch.float32)
        state[0] = float(F.softplus(-z * L).sum() / x.shape[0])
        return state[0], state

    def siglip_backward(self, X, Y, scale, bias, diag_offset, state, grad_out, want_dx, want_dy, want_ds, want_dt):
        self.calls.append("siglip_backward")
        x, y, dots, L, i, j = self._G(X, Y, scale, bias, diag_offset)
        G = torch.sigmoid(L)
        G[i, j] = -torch.sigmoid(-L[i, j])
        k = float(grad_out[0]) / x.shape[0]
        s = float(scale[0])
        return ((k * s * G @ y).float() if want_dx else None, (k * s * G.T @ x).float() if want_dy else None,
                torch.tensor([k * float((G * dots).sum())]) if want_ds else None,
                torch.tensor([k * float(G.sum())]) if want_dt else None)


@pytest.fixture
def install():
    from clipk import ops
    yield ops.set_backend_for_testing
    ops.set_backend_for_testing(None)


def _features(b, d, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (F.normalize(torch.randn(b, d, generator=g, dtype=torch.float64), dim=-1) * scale,
            F.normalize(torch.randn(b, d, generator=g, dtype=torch.float64), dim=-1) * scale)


@pytest.mark.parametrize("world", [1, 2, 4])
def test_oracle_matches_open_clip_transcription(world):
    """open_clip's SigLipLoss.forward written out with this module's get_ground_truth / get_logits: _loss on the own block
    with 2*eye - 1 labels plus the neighbour blocks with negative_only labels, each / b; autograd gives the gradients."""
    from clipk import SigLipLoss
    mod = SigLipLoss()
    b, d, s0, t0, go = 6, 16, 7.5, -3.0, 1.7
    feats = [_features(b, d, 100 + r) for r in range(world)]
    xs = [f[0].clone().requires_grad_(True) for f in feats]
    ts = [f[1].clone().requires_grad_(True) for f in feats]

    def _loss(img, txt, s, t, negative_only=False):
        logits = mod.get_logits(img, txt, s, t)
        labels = mod.get_ground_truth(img.device, img.dtype, img.shape[0], negative_only=negative_only)
        return -F.logsigmoid(labels * logits).sum() / img.shape[0]

    ref = SO.siglip_world([x.detach().numpy() for x in xs], [t.detach().numpy() for t in ts], s0, t0, go)
    d_text = [torch.zeros(b, d, dtype=torch.float64) for _ in range(world)]
    for r in range(world):
        s = torch.tensor(s0, dtype=torch.float64, requires_grad=True)
        t = torch.tensor(t0, dtype=torch.float64, requires_grad=True)
        loss = _loss(xs[r], ts[r], s, t) + sum(_loss(xs[r], ts[k], s, t, True) for k in range(world) if k != r)
        grads = torch.autograd.grad(loss * go, [xs[r], s, t] + ts)
        assert abs(float(loss.detach()) - ref[r].loss) <= 1e-12 * abs(ref[r].loss)
        assert np.abs(grads[0].numpy() - ref[r].d_image).max() <= 1e-12 * np.abs(ref[r].d_image).max()
        assert abs(float(grads[1]) - ref[r].d_scale) <= 1e-12 * max(abs(ref[r].d_scale), 1.0)
        assert abs(float(grads[2]) - ref[r].d_bias) <= 1e-12 * max(abs(ref[r].d_bias), 1.0)
        for k in range(world):
            d_text[k] += grads[3 + k]
    for r in range(world):
        assert np.abs(d_text[r].numpy() - ref[r].d_text).max() <= 1e-12 * np.abs(ref[r].d_text).max()


@pytest.mark.parametrize("world", [1, 3])
def test_oracle_blocks_sum_to_world(world):
    """siglip_block on rank r's geometry (X = images[r], all text rows, positives at r*b + i): the loss, d_image,
    d_scale and d_bias of siglip_world's rank r, and the [N, d] text partials summed over the ranks its d_text."""
    b, d, s, t, go = 5, 12, 9.0, -4.0, -1.3
    feats = [_features(b, d, 200 + r, scale=1.2) for r in range(world)]
    images, texts = [f[0].numpy() for f in feats], [f[1].numpy() for f in feats]
    ref = SO.siglip_world(images, texts, s, t, go)
    text_all = np.concatenate(texts)
    blocks = [SO.siglip_block(images[r], text_all, s, t, go, diag_offset=r * b) for r in range(world)]
    d_text = sum(blk.d_text for blk in blocks)
    assert d_text.shape == (world * b, d)
    for r, (blk, g) in enumerate(zip(blocks, ref)):
        assert abs(blk.loss - g.loss) <= 1e-13 * abs(g.loss)
        for got, want in ((blk.d_image, g.d_image), (d_text[r * b:(r + 1) * b], g.d_text)):
            assert np.abs(got - want).max() <= 1e-13 * np.abs(want).max()
        assert abs(blk.d_scale - g.d_scale) <= 1e-13 * max(abs(g.d_scale), 1.0)
        assert abs(blk.d_bias - g.d_bias) <= 1e-13 * max(abs(g.d_bias), 1.0)


def _sig_struct(rows=300, cols=600, d=128, diag_offset=300):
    """A clipk_siglip that passes every argument check: non-null fake device pointers, 16-byte aligned rows, a 256-byte
    aligned workspace of exactly clipk_siglip_workspace_bytes().  Only ever handed to the library without a GPU, where
    the first CUDA call fails before anything is dereferenced."""
    import ctypes
    from clipk import _lib
    c = _lib.Siglip()
    c.rows, c.cols, c.d = rows, cols, d
    c.x, c.ldx, c.y, c.ldy = 0x100000, d, 0x200000, d
    c.logit_scale, c.logit_bias, c.state, c.diag_offset = 0x300000, 0x300100, 0x300200, diag_offset
    c.workspace = 0x1000000
    c.workspace_bytes = _lib.load().clipk_siglip_workspace_bytes(ctypes.byref(c))
    return c


def test_siglip_abi_validates_arguments_without_a_gpu():
    """clipk_siglip_forward / _backward check their arguments before any CUDA call: each bad field gives its own return
    code, and a struct that passes every check gets as far as the device query (which fails without a GPU)."""
    import ctypes
    from clipk import _lib
    lib = _lib.load()
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    EINVAL, EUNSUPPORTED, EWORKSPACE = -1, -2, -4

    def rc(**fields):
        c = _sig_struct()
        for k, v in fields.items():
            setattr(c, k, v)
        return lib.clipk_siglip_forward(ctypes.byref(c)), lib.clipk_siglip_backward(ctypes.byref(c))

    ok = _sig_struct()
    assert ok.workspace_bytes > 0
    assert lib.clipk_siglip_forward(ctypes.byref(ok)) not in (0, EINVAL, EUNSUPPORTED, EWORKSPACE)
    ok.grad_out = 0x300300
    ok.d_bias = 0x300400
    assert lib.clipk_siglip_backward(ctypes.byref(ok)) not in (0, EINVAL, EUNSUPPORTED, EWORKSPACE)
    ok.grad_out = None
    assert lib.clipk_siglip_backward(ctypes.byref(ok)) == EINVAL                 # grad_out is required
    assert rc(d=100) == (EUNSUPPORTED, EUNSUPPORTED)
    assert rc(diag_offset=301) == (EINVAL, EINVAL)                               # diag_offset + rows > cols
    assert rc(diag_offset=-1) == (EINVAL, EINVAL)
    assert rc(cols=299, diag_offset=0) == (EINVAL, EINVAL)
    assert rc(ldx=64) == (EINVAL, EINVAL)                                        # ldx < d
    assert rc(ldy=127) == (EINVAL, EINVAL)
    assert rc(x=0x100008) == (EINVAL, EINVAL)                                    # x off 16-byte alignment
    assert rc(workspace=0x1000080) == (EINVAL, EINVAL)                           # workspace off 256-byte alignment
    assert rc(workspace_bytes=ok.workspace_bytes - 1) == (EWORKSPACE, EWORKSPACE)
    assert rc(state=None) == (EINVAL, EINVAL)
    assert rc(rows=0) == (EINVAL, EINVAL)
    c = _sig_struct()
    c.rows = 0
    assert lib.clipk_siglip_workspace_bytes(ctypes.byref(c)) == 0
    assert lib.clipk_siglip_workspace_bytes(None) == 0


def _case(name, rank, world):
    """(features, s, t, grad_output, dtype) of a named case on `rank`"""
    d = 72 if name == "odd_width" else 64
    x, t = _features(8, d, 10 * rank + len(name), scale=1.3)
    dtype = {"fp32_formula": torch.float32}.get(name, torch.bfloat16)
    s, bias = (10.0, -4.0) if name == "python_floats" else (torch.tensor(10.0, requires_grad=True),
                                                            torch.tensor(-4.0, requires_grad=True))
    if name == "no_bias":
        bias = None
    go = 2.5 if name == "grad_output" else 1.0
    return x.to(dtype), t.to(dtype), s, bias, go


CASES = ["base", "no_bias", "python_floats", "grad_output", "odd_width", "fp32_formula"]


def _worker(rank, world, tmp):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "megatron-clip_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    from clipk import SigLipLoss, ops
    torch.set_num_threads(1)
    dist.init_process_group("gloo", init_method=f"file://{tmp}/store", rank=rank, world_size=world)
    out = {}
    for name in CASES:
        be = SigEmu()
        ops.set_backend_for_testing(be)
        x, t, s, bias, go = _case(name, rank, world)
        I, T = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
        loss = SigLipLoss(rank=rank, world_size=world)(I, T, s, bias)
        (loss * go).backward()
        out[name] = dict(loss=float(loss), d_image=I.grad.float().numpy(), d_text=T.grad.float().numpy(),
                         calls=list(be.calls), grad_dtype=str(I.grad.dtype), loss_dtype=str(loss.dtype),
                         d_scale=float(s.grad) if isinstance(s, torch.Tensor) else None,
                         d_bias=float(bias.grad) if isinstance(bias, torch.Tensor) else None)
    torch.save(out, f"{tmp}/sig{rank}.pt")
    ops.set_backend_for_testing(None)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_orchestration_against_oracle_over_gloo(world):
    """Per-rank loss, d_image, d_text (after the reduce-scatter), d_scale and d_bias of the kernel route on emulated
    entries, and of the fp32 formula route, against the oracle on the values the route computes with."""
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(world, tmp), nprocs=world, join=True)
        outs = [torch.load(f"{tmp}/sig{r}.pt", weights_only=False) for r in range(world)]
    for name in CASES:
        cases = [_case(name, r, world) for r in range(world)]
        s = float(cases[0][2])
        bias = cases[0][3]
        ref = SO.siglip_world([c[0].double().numpy() for c in cases], [c[1].double().numpy() for c in cases], s,
                              0.0 if bias is None else float(bias), cases[0][4])
        kernels = name != "fp32_formula"
        # bf16 gradients are rounded once from fp32: bf16 tolerances; the formula runs in fp32
        tol = 8e-3 if kernels else 1e-5
        for r in range(world):
            o, g = outs[r][name], ref[r]
            assert o["calls"] == (["siglip_forward", "siglip_backward"] if kernels else []), (name, o["calls"])
            assert o["loss_dtype"] == "torch.float32"
            assert o["grad_dtype"] == ("torch.bfloat16" if kernels else "torch.float32"), name
            assert o["d_image"].shape == cases[r][0].shape
            assert abs(o["loss"] - g.loss) <= 1e-5 * abs(g.loss), (name, r)
            for k in ("d_image", "d_text"):
                want = getattr(g, k)
                assert np.linalg.norm(o[k] - want) <= tol * np.linalg.norm(want), (name, r, k)
            if o["d_scale"] is not None:
                assert abs(o["d_scale"] - g.d_scale) <= 1e-5 * max(abs(g.d_scale), 1e-3), (name, r)
            if o["d_bias"] is not None:
                assert abs(o["d_bias"] - g.d_bias) <= 1e-5 * max(abs(g.d_bias), 1e-3), (name, r)
            assert (o["d_bias"] is None) == (bias is None or name == "python_floats")


@pytest.mark.parametrize("dtype,route", [(torch.bfloat16, "kernels"), (torch.float32, "formula"),
                                         (torch.float16, "formula")])
def test_route_by_dtype(install, dtype, route):
    """bf16 takes the kernel entries; fp32 outside autocast and fp16 evaluate the formula (fp32 under bf16 autocast
    needs CUDA autocast: tests/test_siglip_gpu.py)."""
    from clipk import siglip_loss
    be = SigEmu()
    install(be)
    x, t = _features(16, 64, 3)
    I, T = x.to(dtype).requires_grad_(True), t.to(dtype).requires_grad_(True)
    s, bias = torch.tensor(10.0, requires_grad=True), torch.tensor(-10.0, requires_grad=True)
    loss = siglip_loss(I, T, s, bias)
    loss.backward()
    assert be.calls == (["siglip_forward", "siglip_backward"] if route == "kernels" else [])
    ref = SO.siglip_single(x.to(dtype).double().numpy(), t.to(dtype).double().numpy(), 10.0, -10.0)
    assert loss.dtype == torch.float32 and abs(float(loss) - ref.loss) <= 2e-3 * ref.loss
    assert I.grad.dtype == dtype and T.grad.dtype == dtype and s.grad.shape == () and bias.grad.dtype == torch.float32


class _Refuse:
    def __getattr__(self, name):
        raise AssertionError(f"the backend was called ({name}) for an empty batch")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_empty_batch(install, dtype):
    from clipk import SigLipLoss
    install(_Refuse())
    I = torch.zeros(0, 64, dtype=dtype, requires_grad=True)
    T = torch.zeros(0, 64, dtype=dtype, requires_grad=True)
    s, t = torch.tensor(10.0, requires_grad=True), torch.tensor(-10.0, requires_grad=True)
    loss = SigLipLoss()(I, T, s, t)
    assert loss.dim() == 0 and torch.isnan(loss)
    loss.backward()
    assert I.grad.shape == (0, 64) and T.grad.shape == (0, 64) and I.grad.dtype == dtype


def test_module_surface():
    from clipk import SigLipLoss, create_loss
    args = SimpleNamespace(local_loss=False, gather_with_grad=False, rank=1, world_size=4, horovod=False,
                           model="ViT-B-16-SigLIP", siglip=True)
    m = create_loss(args)
    assert type(m) is SigLipLoss and m.rank == 1 and m.world_size == 4
    mod = SigLipLoss()
    gt = mod.get_ground_truth(torch.device("cpu"), torch.float32, 3)
    assert torch.equal(gt, 2 * torch.eye(3) - 1)
    assert torch.equal(mod.get_ground_truth(torch.device("cpu"), torch.float64, 3, negative_only=True),
                       -torch.ones(3, 3, dtype=torch.float64))
    x, t = _features(4, 8, 1)
    assert torch.allclose(mod.get_logits(x, t, 3.0, -1.0), 3.0 * x @ t.T - 1.0)
    assert torch.allclose(mod.get_logits(x, t, 3.0), 3.0 * x @ t.T)
    out = mod(x.float(), t.float(), 10.0, -10.0, output_dict=True)
    ref = SO.siglip_single(x.float().double().numpy(), t.float().double().numpy(), 10.0, -10.0)
    assert set(out) == {"contrastive_loss"} and abs(float(out["contrastive_loss"]) - ref.loss) <= 1e-5 * ref.loss
    with pytest.raises(NotImplementedError):
        SigLipLoss(use_horovod=True)
