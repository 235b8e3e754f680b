"""Which route a loss call takes, decided once in clipk.ops.fused_clip_loss before anything is launched: the fused step
or the general route, the empty batch without any backend call, and fused_normalize_clip_loss on the general route
when several ranks get no peer context.  Kernel entries emulated on the CPU (tests/emu_backend.py); gloo for W = 2."""
import os
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F


def _spy(peer=True):
    """EmuBackend that records which entry each forward started with; without `peer` it has no peer context to give
    (symmetric memory unavailable, or no room for another shape)."""
    from tests.emu_backend import EmuBackend

    class Spy(EmuBackend):
        def __init__(self):
            self.calls = []

        def peer_context(self, *args):
            return super().peer_context(*args) if peer else None

        def step_forward(self, st):
            self.calls.append("step_forward")
            return super().step_forward(st)

        def step_backward(self, st):
            self.calls.append("step_backward")
            return super().step_backward(st)

        def fwd_both(self, *args, **kwargs):
            self.calls.append("fwd_both")
            return super().fwd_both(*args, **kwargs)

    return Spy()


@pytest.fixture
def install():
    from clipk import ops
    yield ops.set_backend_for_testing
    ops.set_backend_for_testing(None)


@pytest.mark.parametrize("dtype,d,route", [(torch.bfloat16, 64, "step_forward"), (torch.bfloat16, 72, "fwd_both"),
                                           (torch.float32, 64, "fwd_both"), (torch.float16, 64, "fwd_both")])
def test_route_on_one_rank(install, dtype, d, route):
    """bf16 operands with d % 64 == 0 take the fused step; other widths, fp32 outside autocast and fp16 the general
    route.  (fp32 under bf16 autocast needs CUDA autocast: tests/test_parity_gpu.py.)"""
    from clipk import fused_clip_loss
    be = _spy()
    install(be)
    g = torch.Generator().manual_seed(d)
    I = F.normalize(torch.randn(16, d, generator=g), dim=-1).to(dtype).requires_grad_(True)
    T = F.normalize(torch.randn(16, d, generator=g), dim=-1).to(dtype).requires_grad_(True)
    loss = fused_clip_loss(I, T, torch.tensor(10.0))
    loss.backward()
    assert be.calls[0] == route and ("step_forward" in be.calls) == (route == "step_forward")
    assert torch.isfinite(loss) and I.grad.dtype == dtype and I.grad.shape == (16, d)


class _Refuse:
    def __getattr__(self, name):
        raise AssertionError(f"the backend was called ({name}) for an empty batch")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_empty_batch_of_the_normalising_entry(install, dtype):
    """Zero rows through fused_normalize_clip_loss: NaN loss and empty gradients, like fused_clip_loss, and no backend
    call."""
    from clipk import fused_normalize_clip_loss
    install(_Refuse())
    I = torch.zeros(0, 64, dtype=dtype, requires_grad=True)
    T = torch.zeros(0, 64, dtype=dtype, requires_grad=True)
    s = torch.tensor(10.0, requires_grad=True)
    loss = fused_normalize_clip_loss(I, T, s)
    assert loss.dim() == 0 and torch.isnan(loss)
    loss.backward()
    assert I.grad.shape == (0, 64) and T.grad.shape == (0, 64) and I.grad.dtype == dtype


def _worker(rank, world, tmp):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "megatron-clip_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    from clipk import fused_clip_loss, fused_normalize_clip_loss, ops
    torch.set_num_threads(1)
    dist.init_process_group("gloo", init_method=f"file://{tmp}/store", rank=rank, world_size=world)
    out = {}
    # W = 2 with and without a peer context: the fused step, or the general route
    for peer in (True, False):
        be = _spy(peer)
        ops.set_backend_for_testing(be)
        g = torch.Generator().manual_seed(rank)
        I = F.normalize(torch.randn(8, 64, generator=g), dim=-1).bfloat16().requires_grad_(True)
        T = F.normalize(torch.randn(8, 64, generator=g), dim=-1).bfloat16().requires_grad_(True)
        fused_clip_loss(I, T, torch.tensor(10.0), rank=rank, world_size=world).backward()
        out[f"calls_peer{int(peer)}"] = np.array(be.calls)
    # the raw features of a call the fused step would take, had the backend a peer context for it
    be = _spy(peer=False)
    ops.set_backend_for_testing(be)
    g = torch.Generator().manual_seed(10 + rank)
    I = (torch.randn(128, 64, generator=g) * 1.7).bfloat16().requires_grad_(True)
    T = (torch.randn(128, 64, generator=g) * 0.6).bfloat16().requires_grad_(True)
    s = torch.tensor(10.0, requires_grad=True)
    loss = fused_normalize_clip_loss(I, T, s, local_loss=True, gather_with_grad=True, rank=rank, world_size=world)
    loss.backward()
    np.savez(f"{tmp}/route{rank}.npz", loss=loss.detach().numpy(), image=I.detach().float().numpy(),
             text=T.detach().float().numpy(), d_image=I.grad.float().numpy(), d_text=T.grad.float().numpy(),
             d_scale=s.grad.numpy(), calls_normalize=np.array(be.calls), **out)
    ops.set_backend_for_testing(None)
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_without_a_peer_context():
    """On two ranks the fused step needs the backend's peer context; without one, fused_clip_loss takes the general
    route, and fused_normalize_clip_loss normalises first and then takes it too.  The normalised loss and its gradients
    with respect to the raw bf16 features are checked against the float64 oracle chained through F.normalize's
    autograd; the general route rounds the normalised features to bf16, hence bf16-sized tolerances."""
    from oracle import cliploss_oracle as O
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(2, tmp), nprocs=2, join=True)
        outs = [dict(np.load(f"{tmp}/route{r}.npz")) for r in range(2)]
    for o in outs:
        assert list(o["calls_peer1"]) == ["step_forward", "step_backward"]
        assert list(o["calls_peer0"]) == ["fwd_both"]
        assert list(o["calls_normalize"]) == ["fwd_both"]
    xs = [torch.from_numpy(o["image"]).double().requires_grad_(True) for o in outs]
    ts = [torch.from_numpy(o["text"]).double().requires_grad_(True) for o in outs]
    yi, yt = [F.normalize(x, dim=-1) for x in xs], [F.normalize(t, dim=-1) for t in ts]
    ref = O.clip_loss_world([y.detach().numpy() for y in yi], [y.detach().numpy() for y in yt], 10.0, True, True)
    for r, (o, g) in enumerate(zip(outs, ref)):
        torch.autograd.backward([yi[r], yt[r]], [torch.from_numpy(g.d_image), torch.from_numpy(g.d_text)])
        assert abs(float(o["loss"]) - g.loss) <= 1e-3 * abs(g.loss), r
        for k, want in (("d_image", xs[r].grad), ("d_text", ts[r].grad)):
            assert (torch.from_numpy(o[k]).double() - want).norm() <= 8e-3 * want.norm(), (r, k)
        assert abs(float(o["d_scale"]) - g.d_scale) <= 1e-3 * max(abs(g.d_scale), 1 / 10.0), r
