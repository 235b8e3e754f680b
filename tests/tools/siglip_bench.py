"""Manual measurement (not collected by pytest): SigLipLoss forward + backward on one GPU, the fused kernels
(clipk.siglip_loss on bf16) against the torch-eager formula on the same bf16 inputs (clipk.siglip.siglip_formula, which
materialises the [b, N] logits).  Per step: CUDA events around forward + backward, a 256 MiB L2 flush between steps,
every shape warmed up first; the median over the steps is reported.  Also the per-kernel times of one fused step
(clipk_profile_begin / _end), the peak memory of one step above the inputs, and the card and its power limit.

    python tests/tools/siglip_bench.py --out DIR [--steps 20] [--warmup 3]

Writes DIR/siglip_bench.json."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "..", "megatron-clip_b200"))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from clipk import _lib, siglip_loss  # noqa: E402
from clipk.siglip import siglip_formula  # noqa: E402

SHAPES = [(32768, 512), (65536, 768)]
SCALES = [(10.0, -10.0), (100.0, -10.0)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else None
    except Exception as e:          # the numbers are still worth having without the card line
        return f"nvidia-smi failed: {e!r}"


def inputs(n, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = F.normalize(torch.randn(n, d, device="cuda", generator=g), dim=-1)
    t = F.normalize(0.3 * x + F.normalize(torch.randn(n, d, device="cuda", generator=g), dim=-1), dim=-1)
    return x.bfloat16().requires_grad_(True), t.bfloat16().requires_grad_(True)


def step_fn(fn, x, t, s, b):
    S = torch.tensor(s, device="cuda", requires_grad=True)
    B = torch.tensor(b, device="cuda", requires_grad=True)

    def run():
        x.grad = t.grad = S.grad = B.grad = None
        fn(x, t, S, B).backward()
    return run


def measure(run, steps, warmup, flush):
    for _ in range(warmup):
        run()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    times.sort()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    run()
    torch.cuda.synchronize()
    return {"median_ms": times[len(times) // 2], "min_ms": times[0], "max_ms": times[-1], "steps": steps,
            "peak_extra_bytes": torch.cuda.max_memory_allocated() - base}


def kernel_times(run):
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.clipk_profile_begin(stream), "clipk_profile_begin")
    run()
    buf = ctypes.create_string_buffer(8192)
    _lib.check(lib.clipk_profile_end(buf, len(buf)), "clipk_profile_end")
    out = {}
    for item in buf.value.decode().split(";"):
        if item:
            name, n, ms = item.split(":")
            out[name] = {"launches": int(n), "ms": float(ms)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("siglip_bench.py measures on the GPU; no CUDA device here")
    os.makedirs(a.out, exist_ok=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = {"card": card(), "torch": torch.__version__, "cases": []}
    for n, d in SHAPES:
        x, t = inputs(n, d, seed=n + d)
        for s, b in SCALES:
            case = {"N": n, "d": d, "logit_scale": s, "logit_bias": b,
                    "mma_flops": 8 * n * n * d}           # sweep, recompute and the two gradient GEMMs
            fused = step_fn(siglip_loss, x, t, s, b)
            case["fused"] = measure(fused, a.steps, a.warmup, flush)
            case["fused"]["kernels"] = kernel_times(fused)
            try:
                case["eager"] = measure(step_fn(siglip_formula, x, t, s, b), a.steps, a.warmup, flush)
            except torch.OutOfMemoryError as e:
                case["eager"] = {"error": f"out of memory: {str(e).splitlines()[0]}"}
            torch.cuda.empty_cache()
            if "median_ms" in case["eager"]:
                case["speedup"] = case["eager"]["median_ms"] / case["fused"]["median_ms"]
            print(json.dumps(case), flush=True)
            result["cases"].append(case)
        del x, t
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "siglip_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
