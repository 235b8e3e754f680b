"""Pin the oracle (oracle/cliploss_oracle.py) against golden outputs of the unmodified reference loss.py."""
import glob
import os

import numpy as np
import pytest

from oracle import cliploss_oracle as O

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


def _load(path):
    z = dict(np.load(path))
    W = int(z["world"])
    ranks = [{k[len(f"r{r}_"):]: v for k, v in z.items() if k.startswith(f"r{r}_")} for r in range(W)]
    return z, W, ranks


def test_golden_present():
    assert len(GOLD) >= 21


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[:-4] for p in GOLD])
def test_oracle_matches_reference(path):
    z, W, ranks = _load(path)
    res = O.clip_loss_world([r["image"] for r in ranks], [r["text"] for r in ranks], float(z["scale"]),
                            bool(z["local_loss"]), bool(z["gather_with_grad"]), float(z["grad_output"]))
    # the reference ran in float64 or float32; the oracle always in float64 on the same stored inputs
    tol = 1e-12 if str(z["dtype"]) == "float64" else 2e-5
    if str(z["dtype"]) == "float32" and float(z["scale"]) > 50:
        tol = 2e-4   # fp32 reference at s=100 on raw inputs is itself ~1e-4 from exact (SURVEY App. B)
    for r in range(W):
        g, o = ranks[r], res[r]
        assert g["labels"].dtype == np.int64
        assert np.array_equal(g["labels"], o.labels)          # labels bit-exact
        assert abs(float(g["loss"]) - o.loss) <= tol * max(1.0, abs(o.loss))
        for name, ov in (("d_image", o.d_image), ("d_text", o.d_text)):
            gv = g[name].astype(np.float64)
            assert np.linalg.norm(gv - ov) <= tol * max(np.linalg.norm(ov), 1e-30), name
        assert abs(float(g["d_scale"]) - o.d_scale) <= tol * max(abs(o.d_scale), 1e-6)


def test_labels_modes():
    assert np.array_equal(O.ground_truth(4), np.arange(4))
    assert np.array_equal(O.ground_truth(4, rank=2, world_size=4, local_loss=True), np.arange(8, 12))
    assert np.array_equal(O.ground_truth(8, rank=2, world_size=4, local_loss=False), np.arange(8))
    assert O.ground_truth(3).dtype == np.int64


def test_torch_port_matches_oracle():
    import torch
    x, t = O.synthetic_features(64, 48, seed=3)
    loss, dI, dT, ds = O.TorchPort().fwd_bwd(torch.from_numpy(x), torch.from_numpy(t), torch.tensor(1 / 0.07))
    ref = O.clip_loss_single(x, t, 1 / 0.07)
    assert abs(float(loss) - ref.loss) < 1e-5 * abs(ref.loss)
    assert np.linalg.norm(dI.numpy() - ref.d_image) < 1e-5 * np.linalg.norm(ref.d_image)
    assert np.linalg.norm(dT.numpy() - ref.d_text) < 1e-5 * np.linalg.norm(ref.d_text)
    assert abs(float(ds) - ref.d_scale) < 1e-4 * abs(ref.d_scale)


@pytest.mark.gpu
def test_torch_port_on_cuda_tensors():
    """bench.py times the port on the GPU as the eager baseline: its labels must follow the logits to the device."""
    import torch
    x, t = O.synthetic_features(64, 48, seed=3)
    port = O.TorchPort()
    port.fwd_bwd(torch.from_numpy(x), torch.from_numpy(t), torch.tensor(1 / 0.07))      # a CPU call first: labels cached there
    loss, dI, dT, ds = port.fwd_bwd(torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda(), torch.tensor(1 / 0.07).cuda())
    ref = O.clip_loss_single(x, t, 1 / 0.07)
    assert loss.is_cuda and abs(float(loss) - ref.loss) < 1e-4 * abs(ref.loss)
    assert np.linalg.norm(dI.cpu().numpy() - ref.d_image) < 1e-4 * np.linalg.norm(ref.d_image)
    assert np.linalg.norm(dT.cpu().numpy() - ref.d_text) < 1e-4 * np.linalg.norm(ref.d_text)


def test_bf16_rounding_helper():
    import torch
    x = np.random.default_rng(0).standard_normal(1000).astype(np.float32)
    assert np.array_equal(O.round_to_bf16(x), torch.from_numpy(x).bfloat16().float().numpy())
