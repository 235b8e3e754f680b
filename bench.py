#!/usr/bin/env python
"""bench.py - ClipLoss fwd+bwd samples/s (BASELINE.json: global batch 32768, d=512, bf16, at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl clipk|reference]
                    [--config c2|c3|c4] [--mode local|global] [--gwg 0|1] [--logit-scale S] [--skip-extras]
                    [--dump-outputs DIR]

One process per GPU (under torchrun for N > 1; RANK / LOCAL_RANK / WORLD_SIZE from the environment).  The global batch
is fixed, so the N-GPU runs are a strong-scaling series: each rank owns global_batch / N rows.

Default workload (c2): ClipLoss(local_loss=True, gather_with_grad=True) forward + backward on synthetic unit-norm
embeddings (positives at cos ~0.3, SURVEY.md 8d), N = 32768, d = 512, bf16, logit_scale = 1/0.07.
  c3: N = 65536, d = 768, local_loss=False (global mode)            (BASELINE.json configs[2])
  c4: N = 163840, d = 1024, local_loss=True, gather_with_grad=True   (BASELINE.json configs[3])

What one run does, in order (rank 0 prints ONE JSON line at the end):
  1. parity (untimed): all four (local_loss, gather_with_grad) modes at a small size against the fp64 oracle, then the
     benchmark's own shapes through the very ClipLoss call that is timed, against a chunked fp32 torch evaluation of the
     reference formula on the same GPU(s).  A failure is reported in the line and the process exits non-zero.
  2. `value`: K steps with the inputs resident in HBM, every step inside its own CUDA event pair, a 256 MiB L2 flush
     between steps (outside the pairs), max over ranks.  With --dump-outputs DIR, rank 0 then writes what the last of
     these steps returned as float32 DIR/<name>.npy: loss, d_logit_scale, and d_image / d_text, each cut to a seeded
     sample of 16 MB of rows when larger.  The inputs are seeded, so two builds can be compared file by file.
  3. `e2e`: the same call fed from pinned host buffers (H2D of both feature matrices and D2H of the loss inside the timed
     region); `serial_*` is the conservative single-stream figure, the headline prefetches the next step's inputs.
  4. per-kernel times of one rank's step from the library's own event profile -> roofline of the dominant kernel.
  5. the reference's op sequence on the same GPU(s) (`gpu_eager_baseline`), other operating points (`extras`:
     logit_scale = 100, c3 / c4 when they fit), and - one GPU only - the reference on the host cores (`cpu_baseline`).

--impl reference runs the reference's own ClipLoss (open_CLIP/src/open_clip/loss.py, installed unmodified under
baseline/_ref by __graft_entry__.build()) on the host cores at the REAL workload size when K + W such steps fit in a
few minutes, else on a bounded sample which the line names.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "megatron-clip_b200"))

CONFIGS = {
    "c2": dict(N=32768, d=512, local=True, gwg=True, what="ViT-B/32 embeddings, BASELINE.json configs[1]"),
    "c3": dict(N=65536, d=768, local=False, gwg=True, what="ViT-L/14 embeddings, global mode, BASELINE.json configs[2]"),
    "c4": dict(N=163840, d=1024, local=True, gwg=True, what="ViT-H/14 embeddings, BASELINE.json configs[3]"),
}
INIT_SCALE = 1.0 / 0.07
METRIC = "ClipLoss fwd+bwd samples/s @ global batch 32K, d=512"
CPU_SAMPLE_BATCH = 8192           # calibration size of the CPU arms (cost grows with batch^2)
CPU_ARM_BUDGET_S = 240.0          # whole `--impl reference` run
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
DUMP_MATRIX_BYTES = 16 << 20      # per gradient matrix written by --dump-outputs (as float32)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return {"tflops_sustained": j.get("bf16_tflops_sustained", 1401.9), "tflops_burst": j.get("bf16_tflops", 1661.2),
                "hbm_gbs": j.get("hbm_gbs", 6542.7), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi polling the clocks of one GPU during the timed region.  The samples go to a file that is read after
    the run: a reader thread in this process would fight the launching thread for the interpreter lock."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path, self.fh = index, None, None, None

    def start(self):
        import tempfile
        try:
            self.fh = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.path = self.fh.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("CLIPK_BENCH_SMI_MS", "50")],
                                         stdout=self.fh, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.3)         # let the first samples land before the timed region starts
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.fh.close()
        with open(self.path) as f:
            rows = [[c.strip() for c in line.split(",")] for line in f if line.strip()]
        os.unlink(self.path)
        sm, mx, power, reasons = [], None, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                power.append(float(r[3]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                pass
        # clocks under load = the samples taken while the GPU drew the most power (busier half)
        order = sorted(range(len(sm)), key=lambda i: power[i])
        load = sorted(sm[i] for i in order[len(order) // 2:])
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power) if power else None}


# ------------------------------------------------------------------------------------------------ the reference module
def load_reference_loss():
    """The reference's loss.py, unmodified, from baseline/_ref (copied there by __graft_entry__.build() in the build
    container; /root/reference does not exist on the GPU box).  It is imported in isolation - `import open_clip` needs
    ftfy, timm, ... - as a stub package whose __path__ is the directory.  None when the copy is not there."""
    d = os.path.join(REF_DIR, "open_clip")
    if not (os.path.exists(os.path.join(d, "loss.py")) and os.path.exists(os.path.join(d, "tprofiler.py"))):
        return None
    if "open_clip.loss" in sys.modules:
        return sys.modules["open_clip.loss"]
    pkg = types.ModuleType("open_clip")
    pkg.__path__ = [d]
    sys.modules["open_clip"] = pkg
    for n in ("tprofiler", "loss"):
        spec = importlib.util.spec_from_file_location("open_clip." + n, os.path.join(d, n + ".py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules["open_clip." + n] = m
        spec.loader.exec_module(m)
    return sys.modules["open_clip.loss"]


class _Quiet:
    """The reference prints a line per constructed loss and per get_logits call: keep stdout to the one JSON line."""

    def __enter__(self):
        self._out = sys.stdout
        sys.stdout = sys.stderr

    def __exit__(self, *a):
        sys.stdout = self._out


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_inputs(batch, d):
    import torch
    from oracle import cliploss_oracle as O
    x, t = O.synthetic_features(batch, d, seed=1234)
    return torch.from_numpy(x), torch.from_numpy(t)


def cpu_step_fn(kind_out):
    """fwd+bwd of the reference ClipLoss on CPU tensors (the reference module itself when baseline/_ref holds it, else
    the oracle's torch port of the same op sequence)."""
    import torch
    L = load_reference_loss()
    if L is not None:
        with _Quiet():
            mod = L.ClipLoss(cache_labels=True)
        kind_out.append("reference")

        def step(I, T, s):
            i, t, sc = I.detach().requires_grad_(True), T.detach().requires_grad_(True), s.detach().requires_grad_(True)
            loss = mod(i, t, sc)
            loss.backward()
            return loss
        return step
    from oracle import cliploss_oracle as O
    port = O.TorchPort()
    kind_out.append("port")
    return lambda I, T, s: port.fwd_bwd(I, T, s)[0]


def cpu_c1(step, threads):
    """BASELINE.md 2.1: B = 256, d = 512, fp32, 5 warm-ups, median of 200."""
    import torch
    torch.set_num_threads(threads)
    I, T = cpu_inputs(256, 512)
    s = torch.tensor(INIT_SCALE)
    for _ in range(5):
        step(I, T, s)
    ts = []
    for _ in range(200):
        t0 = time.perf_counter()
        step(I, T, s)
        ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return {"threads": threads, "median_ms": med * 1e3, "samples_per_s": 256 / med}


def cpu_timed(step, batch, d, steps, warmup):
    import torch
    I, T = cpu_inputs(batch, d)
    s = torch.tensor(INIT_SCALE)
    for _ in range(warmup):
        step(I, T, s)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step(I, T, s)
        ts.append(time.perf_counter() - t0)
    return sum(ts) / len(ts)


def cpu_pick_batch(step, N, d, nsteps, budget_s):
    """Largest of N, N/2, N/4, ... whose nsteps steps fit the budget, from one calibration step at CPU_SAMPLE_BATCH."""
    import torch
    cal = min(CPU_SAMPLE_BATCH, N)
    I, T = cpu_inputs(cal, d)
    s = torch.tensor(INIT_SCALE)
    step(I, T, s)
    t0 = time.perf_counter()
    step(I, T, s)
    t_cal = time.perf_counter() - t0
    b = N
    while b > cal and t_cal * (b / cal) ** 2 * nsteps > budget_s:
        b //= 2
    return b, t_cal


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cfg = CONFIGS[args.config]
    N, d = cfg["N"], cfg["d"]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kind = []
    step = cpu_step_fn(kind)
    nsteps = args.steps + args.warmup
    batch, t_cal = cpu_pick_batch(step, N, d, nsteps, CPU_ARM_BUDGET_S)
    sec = cpu_timed(step, batch, d, args.steps, args.warmup)
    full = sec * (N / batch) ** 2              # == sec when the real size ran
    sample = (f"{'reference open_clip ClipLoss' if kind[0] == 'reference' else 'torch port of the reference ops'}, CPU fp32, "
              f"fwd+bwd at batch {batch}, d={d}, {cores} threads, {sec * 1e3:.0f} ms/step")
    sample += " - the real workload size" if batch == N else f", scaled by ({N}/{batch})^2 to the global-batch-{N} step"
    value = N / full
    cb = {"value": value, "unit": "samples/s", "cores": cores, "kind": kind[0], "sample": sample, "sample_batch": batch,
          "extrapolated": batch != N}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"ClipLoss fwd+bwd, global batch {N}, d={d} ({cfg['what']}), the reference on host cores",
                   "global_batch": N, "d": d, "step_batch": batch},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ GPU arm helpers
def torch_fp32_reference(I, T, s, rank, world, local, gwg, chunk=2048):
    """loss, dI, dT, ds of ClipLoss on this rank from the reference's formula (loss.py:104-140, closed forms of SURVEY
    App. A) in plain fp32 torch ops on the GPU, row chunk by row chunk so that no N x N matrix is held.  Independent of
    every clipk kernel and collective path (NCCL all_reduce / reduce_scatter only)."""
    import torch
    import torch.distributed as dist
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        X, Yl = I.detach().float(), T.detach().float()
        b, d = X.shape
        N = world * b
        if world > 1:
            Y = torch.empty(N, d, dtype=torch.float32, device=X.device)
            dist.all_gather_into_tensor(Y, Yl)
        else:
            Y = Yl
        off = rank * b if world > 1 else 0
        sv = float(s)
        lse_row = torch.empty(b, device=X.device)
        pos = torch.empty(b, device=X.device)
        cmax = torch.full((N,), -float("inf"), device=X.device)
        csum = torch.zeros(N, device=X.device)
        for r0 in range(0, b, chunk):
            S = sv * X[r0:r0 + chunk] @ Y.T
            lse_row[r0:r0 + chunk] = torch.logsumexp(S, dim=1)
            idx = torch.arange(r0, min(r0 + chunk, b), device=X.device)
            pos[r0:r0 + chunk] = S[idx - r0, idx + off]
            m = torch.maximum(cmax, S.max(dim=0).values)
            csum = csum * torch.exp(cmax - m) + torch.exp(S - m[None, :]).sum(dim=0)
            cmax = m
        if world > 1:
            gm = cmax.clone()
            dist.all_reduce(gm, op=dist.ReduceOp.MAX)
            csum = csum * torch.exp(cmax - gm)
            dist.all_reduce(csum)
            cmax = gm
        lse_col = cmax + csum.log()
        part = torch.stack(((lse_row - pos).sum(), (lse_col[off:off + b] - pos).sum()))
        if world > 1 and not local:
            dist.all_reduce(part)
            loss = part.sum() / (2.0 * N)
        else:
            loss = part.sum() / (2.0 * b)
        c = 1.0 / (2.0 * b) if (world == 1 or local or gwg) else 1.0 / (2.0 * N)
        a_row, a_col = 1.0, 1.0
        dI = torch.empty_like(X)
        dY = torch.zeros(N, d, device=X.device)
        ds_acc = torch.zeros((), device=X.device, dtype=torch.float64)
        for r0 in range(0, b, chunk):
            Xc = X[r0:r0 + chunk]
            S = sv * Xc @ Y.T
            G = a_row * torch.exp(S - lse_row[r0:r0 + chunk, None]) + a_col * torch.exp(S - lse_col[None, :])
            idx = torch.arange(r0, min(r0 + chunk, b), device=X.device)
            G[idx - r0, idx + off] -= 2.0
            ds_acc += (G * S).sum().double()
            dI[r0:r0 + chunk] = (sv * c) * (G @ Y)
            dY += (sv * c) * (G.T @ Xc)
        if world > 1:
            dT = torch.empty(b, d, device=X.device)
            dist.reduce_scatter_tensor(dT, dY)
        else:
            dT = dY
        # dlogit_scale: per rank, never all-reduced in local mode; the global loss is all-reduced (App. A)
        ds = ds_acc / sv * (1.0 / (2.0 * b) if (world == 1 or local) else 1.0 / (2.0 * N))
        if world > 1 and not local:
            dsv = ds.clone()
            dist.all_reduce(dsv)
            ds = dsv
        return float(loss), dI, dT, float(ds)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300))


def parse_profile(text):
    out = {}
    for item in text.split(";"):
        if item:
            name, n, ms = item.rsplit(":", 2)
            out[name] = {"launches": int(n), "ms": float(ms)}
    return out


def dump_outputs(out_dir, tensors):
    """--dump-outputs: each tensor as float32 <out_dir>/<name>.npy.  A matrix larger than DUMP_MATRIX_BYTES is cut to
    a seeded sample of its rows (sorted; the same rows for the same shape), which keeps the dump under 64 MB."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tensors.items():
        t = t.detach()
        if t.dim() == 2 and t.numel() * 4 > DUMP_MATRIX_BYTES:
            rows = DUMP_MATRIX_BYTES // (4 * t.shape[1])
            idx = np.sort(np.random.default_rng(0).choice(t.shape[0], rows, replace=False))
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_clipk(args):
    import torch
    import torch.distributed as dist
    from clipk import ClipLoss, ops, _lib
    from oracle import cliploss_oracle as O   # synthetic input generator, parity checker and cpu_baseline leg only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = dict(CONFIGS[args.config])
    if args.mode:
        cfg["local"] = args.mode == "local"
    if args.gwg is not None:
        cfg["gwg"] = bool(args.gwg)
    N, DIM = cfg["N"], cfg["d"]
    assert N % world == 0
    b = N // world
    scale_value = args.logit_scale
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def bar():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_ok(flag):
        t = torch.tensor([1 if flag else 0], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def make(bb, dd, seed, dtype=torch.bfloat16):
        x, t = O.synthetic_features(bb, dd, seed=seed, rank=rank)
        return torch.from_numpy(x).to(dtype), torch.from_numpy(t).to(dtype)

    # ------------------------------------------------------------------ 1. parity (untimed)
    def parity_small():
        """all four modes, b = 640 per rank, d = 256, bf16, against oracle.clip_loss_world (fp64, rank 0)"""
        res = {}
        ok = True
        modes = [(True, True), (True, False), (False, True), (False, False)] if world > 1 else [(False, False)]
        for ll, gwg in modes:
            xi, ti = make(640, 256, 77)
            I, T = xi.to(dev).requires_grad_(True), ti.to(dev).requires_grad_(True)
            S = torch.tensor(INIT_SCALE, device=dev, requires_grad=True)
            loss = ClipLoss(local_loss=ll, gather_with_grad=gwg, cache_labels=True, rank=rank, world_size=world)(I, T, S)
            loss.backward()
            mine = torch.cat((I.grad.float().flatten(), T.grad.float().flatten(), loss.detach().reshape(1), S.grad.reshape(1)))
            feats = torch.cat((I.detach().float().flatten(), T.detach().float().flatten()))
            if world > 1:
                allm = [torch.empty_like(mine) for _ in range(world)]
                allf = [torch.empty_like(feats) for _ in range(world)]
                dist.all_gather(allm, mine)
                dist.all_gather(allf, feats)
            else:
                allm, allf = [mine], [feats]
            err = 0.0
            if rank == 0:
                n = 640 * 256
                imgs = [f[:n].reshape(640, 256).cpu().numpy() for f in allf]
                txts = [f[n:].reshape(640, 256).cpu().numpy() for f in allf]
                ref = O.clip_loss_world(imgs, txts, INIT_SCALE, ll, gwg)
                for r in range(world):
                    m = allm[r].cpu()
                    g = ref[r]
                    e = [rel_l2(m[:n], torch.from_numpy(g.d_image).flatten()), rel_l2(m[n:2 * n], torch.from_numpy(g.d_text).flatten()),
                         abs(float(m[2 * n]) - g.loss) / abs(g.loss), abs(float(m[2 * n + 1]) - g.d_scale) / max(abs(g.d_scale), 0.07)]
                    err = max(err, max(e))
            res[f"ll{int(ll)}_gwg{int(gwg)}"] = err
            ok = ok and (err <= 2e-3)
        return all_ok(ok), res

    def parity_shard():
        """the benchmark's shapes through the timed ClipLoss call, against the chunked fp32 torch reference"""
        xi, ti = make(b, DIM, 1234)
        I, T = xi.to(dev).requires_grad_(True), ti.to(dev).requires_grad_(True)
        S = torch.tensor(scale_value, device=dev, requires_grad=True)
        mod = ClipLoss(local_loss=cfg["local"], gather_with_grad=cfg["gwg"], cache_labels=True, rank=rank, world_size=world)
        loss = mod(I, T, S)
        loss.backward()
        single = ops.last_forward_was_single_sweep()
        rl, rI, rT, rs = torch_fp32_reference(I, T, scale_value, rank, world, cfg["local"], cfg["gwg"])
        e = {"loss": abs(loss.item() - rl) / abs(rl), "d_image": rel_l2(I.grad, rI), "d_text": rel_l2(T.grad, rT),
             "d_scale": abs(S.grad.item() - rs) / max(abs(rs), 1.0 / scale_value)}
        worst = torch.tensor([max(e.values())], device=dev)
        if world > 1:
            dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        e["max_over_ranks"] = float(worst.item())
        return all_ok(worst.item() <= 2e-3), e, single

    def run_parity():
        ok_s, small = parity_small()
        ok_b, shard, single = parity_shard()
        return {"ok": bool(ok_s and ok_b), "tolerance": 2e-3, "small_all_modes_vs_fp64_oracle": small,
                "bench_shapes_vs_fp32_torch": shard, "single_sweep_forward": single,
                "peer_path": bool(world > 1 and len(ops._PEER_CONTEXTS) > 0)}

    parity = run_parity()
    if not parity["ok"] and world > 1 and parity["peer_path"]:
        # the peer-memory collectives gave wrong numbers on this box: report it, and measure the NCCL route instead
        first = parity
        os.environ["CLIPK_PEER"] = "0"
        parity = run_parity()
        parity["peer_path_failed_first"] = first
    bar()

    # ------------------------------------------------------------------ 2. / 3. timed legs
    xi, ti = make(b, DIM, 1234)
    I_host, T_host = xi.pin_memory(), ti.pin_memory()
    I = I_host.to(dev).requires_grad_(True)
    T = T_host.to(dev).requires_grad_(True)
    S = torch.tensor(scale_value, device=dev, requires_grad=True)
    loss_mod = ClipLoss(local_loss=cfg["local"], gather_with_grad=cfg["gwg"], cache_labels=True, rank=rank, world_size=world)
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def make_step(mod, Ii, Ti, Si):
        def step():
            Ii.grad = Ti.grad = Si.grad = None
            loss = mod(Ii, Ti, Si)
            loss.backward()
            return loss
        return step

    step_resident = make_step(loss_mod, I, T, S)

    def step_e2e():
        i = I_host.to(dev, non_blocking=True).requires_grad_(True)
        tt = T_host.to(dev, non_blocking=True).requires_grad_(True)
        S.grad = None
        loss = loss_mod(i, tt, S)
        loss.backward()
        loss_host.copy_(loss.detach(), non_blocking=True)
        return loss

    last_out = {}       # what the last timed step returned (--dump-outputs)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        bar()
        # every step has its own event pair; the L2 flush between steps is enqueued outside the pairs and the host
        # does not synchronise inside the timed region
        launches = 0
        pairs = []
        t_host = time.perf_counter()
        for _ in range(steps):
            flush.fill_(1)                          # L2 flush, outside the event pair
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            la = ops.gpu_launches()
            e0.record()
            last_out["loss"] = fn()
            e1.record()
            launches += ops.gpu_launches() - la
            pairs.append((e0, e1))
        host_ms = (time.perf_counter() - t_host) * 1e3 / steps      # time the host needs to ENQUEUE one step
        torch.cuda.synchronize()
        total_ms = sum(e0.elapsed_time(e1) for e0, e1 in pairs)
        bar()
        tt = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)   # max over ranks
        return tt.item() / steps, launches, host_ms

    def timed_pipelined(steps, warmup):
        """e2e with the input copies double-buffered, the way a host-fed training loop prefetches: the H2D copy of
        step k+1's features runs on a copy stream while step k's kernels run (it may not start before step k's timed
        region has begun), and step k+1 waits for it inside its own event pair."""
        main = torch.cuda.current_stream(dev)
        copy_stream = torch.cuda.Stream(device=dev)
        bufs = [(torch.empty(I_host.shape, dtype=I_host.dtype, device=dev), torch.empty(T_host.shape, dtype=T_host.dtype, device=dev))
                for _ in range(2)]
        ready = [torch.cuda.Event(), torch.cuda.Event()]

        def prefetch(k, after):
            copy_stream.wait_event(after)
            with torch.cuda.stream(copy_stream):
                bufs[k % 2][0].copy_(I_host, non_blocking=True)
                bufs[k % 2][1].copy_(T_host, non_blocking=True)
                ready[k % 2].record(copy_stream)

        bar()
        total = warmup + steps
        begin = torch.cuda.Event()
        begin.record(main)
        prefetch(0, begin)
        pairs = []
        for k in range(total):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(main)
            if k + 1 < total:
                prefetch(k + 1, e0)      # buffer (k+1)%2 was last read by step k-1, which precedes e0 on `main`
            main.wait_event(ready[k % 2])
            i = bufs[k % 2][0].detach().requires_grad_(True)
            tt = bufs[k % 2][1].detach().requires_grad_(True)
            S.grad = None
            loss = loss_mod(i, tt, S)
            loss.backward()
            loss_host.copy_(loss.detach(), non_blocking=True)
            e1.record(main)
            if k >= warmup:
                pairs.append((e0, e1))
        torch.cuda.synchronize()
        total_ms = sum(e0.elapsed_time(e1) for e0, e1 in pairs)
        bar()
        tt = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return tt.item() / steps, float(loss_host)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches, host_ms = timed(step_resident, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": last_out["loss"].detach(), "d_image": I.grad, "d_text": T.grad,
                                         "d_logit_scale": S.grad})
    loss_resident = float(step_resident().detach())
    single_sweep = ops.last_forward_was_single_sweep()
    e2e_steps = max(3, args.steps // 2)
    ms_e2e_serial, _, _ = timed(step_e2e, e2e_steps, 3)
    ms_e2e, e2e_mode = ms_e2e_serial, "serial: H2D, step and D2H on one stream"
    if os.environ.get("CLIPK_BENCH_E2E", "pipelined") == "pipelined":
        ms_pipe, loss_pipe = timed_pipelined(e2e_steps, 3)
        if all_ok(abs(loss_pipe - loss_resident) <= 1e-5 * abs(loss_resident)):
            ms_e2e = ms_pipe
            e2e_mode = ("double-buffered: the H2D copy of step k+1 runs on a copy stream during step k (not before "
                        "step k's timed region begins); step k+1 waits for it inside its own event pair")
        else:
            e2e_mode += f"; pipelined run rejected (loss {loss_pipe} != {loss_resident})"

    # ------------------------------------------------------------------ 4. per-kernel times of this rank's step
    lib = _lib.load()
    prof_steps = 5
    for _ in range(2):
        step_resident()
    bar()
    _lib.check(lib.clipk_profile_begin(torch.cuda.current_stream(dev).cuda_stream), "clipk_profile_begin")
    for _ in range(prof_steps):
        step_resident()
    import ctypes
    buf = ctypes.create_string_buffer(8192)
    _lib.check(lib.clipk_profile_end(buf, len(buf)), "clipk_profile_end")
    kern = parse_profile(buf.value.decode())
    for k in kern.values():
        k["launches_per_step"] = k["launches"] / prof_steps
        k["ms_per_launch"] = k["ms"] / k["launches"]
        k["ms_per_step"] = k["ms"] / prof_steps
        del k["launches"], k["ms"]
    prof_total = sum(k["ms_per_step"] for k in kern.values())
    for k in kern.values():
        k["share_of_profiled_step"] = k["ms_per_step"] / prof_total if prof_total > 0 else None
    bar()

    # ------------------------------------------------------------------ 5a. the reference's ops on the same GPU(s)
    def eager_baseline():
        L = load_reference_loss()
        if L is not None:
            with _Quiet():
                mod = L.ClipLoss(local_loss=cfg["local"], gather_with_grad=cfg["gwg"], cache_labels=True, rank=rank,
                                 world_size=world)
            what = "reference open_clip ClipLoss (baseline/_ref) on CUDA, bf16, NCCL"
        else:
            port = O.TorchPort()
            mod = port
            what = "torch port of the reference ops on CUDA, bf16"
            if world > 1:
                return {"unavailable": "baseline/_ref missing and the port is single-process"}
        try:
            torch.cuda.reset_peak_memory_stats(dev)

            def fn():
                I.grad = T.grad = S.grad = None
                with _Quiet():
                    loss = mod(I, T, S)
                loss.backward()
                return loss
            t, _, _ = timed(fn, 5, 3)
            return {"ms_per_step": t, "value": N / (t * 1e-3), "unit": "samples/s", "what": what,
                    "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9, "loss": float(fn().detach())}
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            return {"oom": True, "what": what}

    eager = None if args.skip_extras else eager_baseline()
    I.grad = T.grad = S.grad = None
    bar()

    # ------------------------------------------------------------------ 5b. other operating points
    def quick(cfg_name, s_val, steps=5, warmup=3, gwg=None, eager=False):
        c = CONFIGS[cfg_name]
        if c["N"] % world:
            return {"skipped": "global batch not divisible"}
        bb = c["N"] // world
        gwg = c["gwg"] if gwg is None else gwg
        try:
            xq, tq = make(bb, c["d"], 4321)
            Iq, Tq = xq.to(dev).requires_grad_(True), tq.to(dev).requires_grad_(True)
            Sq = torch.tensor(s_val, device=dev, requires_grad=True)
            mod = ClipLoss(local_loss=c["local"], gather_with_grad=gwg, cache_labels=True, rank=rank, world_size=world)
            t, _, _ = timed(make_step(mod, Iq, Tq, Sq), steps, warmup)
            f_alg = 6.0 * bb * c["N"] * c["d"]
            pk = peaks()
            out = {"ms_per_step": t, "value": c["N"] / (t * 1e-3), "unit": "samples/s", "global_batch": c["N"], "d": c["d"],
                   "local_batch": bb, "mode": "local" if c["local"] else "global", "gather_with_grad": gwg,
                   "logit_scale": s_val, "single_sweep_forward": ops.last_forward_was_single_sweep(),
                   "frac_of_burst_peak": f_alg / (t * 1e-3) / 1e12 / pk["tflops_burst"]}
        except torch.OutOfMemoryError:
            torch.cuda.empty_cache()
            return {"oom": True}
        if eager:
            out["reference_eager"] = quick_eager(c, gwg, Iq, Tq, Sq)
        return out

    def quick_eager(c, gwg, Iq, Tq, Sq):
        """The reference module itself on the same inputs and GPUs (an out-of-memory error is a result: SURVEY 8d)."""
        L = load_reference_loss()
        if L is None:
            return {"unavailable": "baseline/_ref missing"}
        with _Quiet():
            ref = L.ClipLoss(local_loss=c["local"], gather_with_grad=gwg, cache_labels=True, rank=rank, world_size=world)

        def fn():
            Iq.grad = Tq.grad = Sq.grad = None
            with _Quiet():
                loss = ref(Iq, Tq, Sq)
            loss.backward()
            return loss
        res = None
        try:
            torch.cuda.reset_peak_memory_stats(dev)
            t, _, _ = timed(fn, 3, 2)
            res = {"ms_per_step": t, "value": c["N"] / (t * 1e-3), "unit": "samples/s",
                   "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9}
        except torch.OutOfMemoryError:
            pass
        Iq.grad = Tq.grad = Sq.grad = None
        torch.cuda.empty_cache()
        return res if res is not None else {"oom": True}

    extras = {}
    if not args.skip_extras and args.config == "c2" and abs(scale_value - INIT_SCALE) < 1e-6:
        extras["c2_logit_scale_100"] = quick("c2", 100.0)
        extras["c3_global"] = quick("c3", INIT_SCALE, steps=3, warmup=2, eager=True)
        extras["c3_global_no_gather_grad"] = quick("c3", INIT_SCALE, steps=3, warmup=2, gwg=False)
        if world == 8:
            extras["c4"] = quick("c4", INIT_SCALE, steps=3, warmup=2, eager=True)

    # nvidia-smi cannot sample faster than every ~50 ms and the timed region lasts ~0.1 s, so the sampler stays on from
    # before the timed region until the end of a short untimed continuation of the same step; `clocks` is the busier
    # half of those samples.
    probe_s = float(os.environ.get("CLIPK_BENCH_CLOCK_PROBE_S", "0.8"))
    probe_steps = 0
    try:
        n_probe = int(min(400, probe_s / max(ms * 1e-3, 1e-4)))
        for _ in range(n_probe):
            step_resident()
            probe_steps += 1
        torch.cuda.synchronize()
    except Exception as e:      # the probe must never cost the run its result line
        print(f"clock probe stopped: {e!r}", file=sys.stderr)
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["window"] = (f"timed region, e2e legs, profile and extras, then {probe_steps} more untimed steps "
                            f"(~{probe_s} s) of the same workload")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        sys.exit(0 if parity["ok"] else 3)

    # ------------------------------------------------------------------ roofline
    pk = peaks()
    f_alg = 6.0 * b * N * DIM                                  # SURVEY 8(d): three dense passes over the b x N block
    f_exec = 8.0 * b * N * DIM                                 # issued: 1 fwd sweep (rows + columns) + recompute + 2 gradient GEMMs
    step_tflops = f_alg / (ms * 1e-3) / 1e12
    rp, cp = ctypes.c_longlong(0), ctypes.c_longlong(0)
    lib.clipk_bwd_panel(b, N, DIM, ctypes.byref(rp), ctypes.byref(cp))
    dom = "gemm_pair_kernel"
    roofline = {"bound": "tensor", "unit": "TFLOP/s", "peak": pk["tflops_burst"],
                "peak_note": "burst cuBLAS bf16 figure of MEASURED_PEAKS.json: the timed region is a fraction of a second "
                             "(BASELINE.md's target column uses the same denominator); sustained: "
                             f"{pk['tflops_sustained']}", "peak_source": pk["source"]}
    if dom in kern:
        k = kern[dom]
        # algorithmic work of one launch: both gradient GEMMs of one panel = 4 * rows * cols * d, averaged over the
        # launches of a step (edge panels are smaller)
        flops_per_launch = 4.0 * b * N * DIM / k["launches_per_step"]
        ach = flops_per_launch / (k["ms_per_launch"] * 1e-3) / 1e12
        roofline.update({"kernel": f"clipk::{dom} (dX = G Y and dY = G^T X tiles of one {rp.value} x {cp.value} panel, tcgen05 "
                                   "cta_group::2 256x256x64)", "achieved": ach, "frac": ach / pk["tflops_burst"],
                         "frac_of_sustained_peak": ach / pk["tflops_sustained"],
                         "algorithmic_flops_per_launch": flops_per_launch, "ms_per_launch": k["ms_per_launch"],
                         "share_of_step": k["share_of_profiled_step"]})
    else:
        roofline.update({"kernel": "whole step", "achieved": step_tflops, "frac": step_tflops / pk["tflops_burst"]})
    # DRAM traffic of the dominant kernel comes from an ncu --set full capture, not from this run: read from the
    # committed summary when there is one for this shape
    roofline["traffic"] = None
    tfile = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if os.path.exists(tfile) and world == 1 and args.config == "c2":
        try:
            with open(tfile) as f:
                tj = json.load(f)
            roofline["traffic"] = tj.get(dom, {}).get("dram_bytes_per_launch")
            roofline["traffic_source"] = tj.get("source")
        except (OSError, ValueError):
            pass
    roofline["whole_step"] = {"algorithmic_flops_per_gpu": f_alg, "executed_mma_flops_per_gpu": f_exec,
                              "achieved_tflops": step_tflops, "frac_of_burst_peak": step_tflops / pk["tflops_burst"],
                              "frac_of_sustained_peak": step_tflops / pk["tflops_sustained"],
                              "definition": "SURVEY 8d: F_alg = 6 b N d over t_step, per GPU"}
    # a power-capped part: a 0.07 s timed region runs ~15 % faster than a 0.4 s one (profiles/README.md)
    roofline["timed_region_s"] = ms * args.steps * 1e-3
    roofline["kernels"] = kern
    roofline["kernels_note"] = (f"library event profile over {prof_steps} steps of this run (an event after every launch; the "
                                "time between consecutive events goes to the kernel launched in between)")
    if world > 1:
        gather_in = (world - 1) * b * DIM * 2
        stats_in = (world - 1) * 3 * N * 4
        rs_out = (world - 1) * b * DIM * 4
        t_link = max(gather_in + stats_in, rs_out) / 900e9 * 1e3
        nv = {"gather_bytes_in": gather_in, "colstats_bytes_in": stats_in, "grad_bytes_out": rs_out,
              "ms_at_900GBs_per_direction": t_link,
              "roofline_ms_per_step": max(f_alg / (pk["tflops_burst"] * 1e12) * 1e3, t_link)}
        if "peer_allgather_kernel" in kern:
            g = kern["peer_allgather_kernel"]
            nv["allgather_kernels_ms_per_step"] = g["ms_per_step"]
            nv["allgather_GBs"] = (gather_in + stats_in) / (g["ms_per_step"] * 1e-3) / 1e9
        roofline["nvlink"] = nv

    cb = None
    if world == 1 and not os.environ.get("CLIPK_BENCH_QUICK"):     # development runs may skip the CPU leg
        cores = os.cpu_count() or 1
        kind = []
        cstep = cpu_step_fn(kind)
        c1 = [cpu_c1(cstep, cores), cpu_c1(cstep, 1)]
        torch.set_num_threads(cores)
        batch, _ = cpu_pick_batch(cstep, N, DIM, 3, 30.0)
        sec = cpu_timed(cstep, batch, DIM, 2, 1)
        full = sec * (N / batch) ** 2
        cb = {"value": N / full, "unit": "samples/s", "cores": cores, "kind": kind[0],
              "sample": (f"fwd+bwd of the {'reference module' if kind[0] == 'reference' else 'torch port'} on CPU fp32 at batch "
                         f"{batch}, d={DIM}: {sec * 1e3:.0f} ms/step (1 warm-up + 2 timed)"
                         + ("" if batch == N else f", scaled by ({N}/{batch})^2")),
              "extrapolated": batch != N, "c1_batch256_d512_fp32_median_of_200": c1}

    out = {
        "metric": METRIC, "value": N / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"ClipLoss local_loss={cfg['local']} gather_with_grad={cfg['gwg']} fwd+bwd, {cfg['what']}",
                   "name": args.config, "global_batch": N, "local_batch": b, "d": DIM,
                   "logit_scale": scale_value, "parallelism": f"dp{world}",
                   "l2": "256 MiB buffer overwritten between timed steps (L2 flush), outside the per-step event pairs"},
        "clocks": clocks,
        "e2e": {"value": N / (ms_e2e * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": 2 * b * DIM * 2, "d2h_bytes_per_step": 4, "mode": e2e_mode,
                "serial_ms_per_step": ms_e2e_serial, "serial_value": N / (ms_e2e_serial * 1e-3)},
        "gpu_launches": launches, "host_enqueue_ms_per_step": host_ms, "single_sweep_forward": single_sweep,
        "parity": parity,
        "roofline": roofline,
        "gpu_eager_baseline": eager,
        "extras": extras,
        "cpu_baseline": cb,
    }
    print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()
    if not parity["ok"]:
        sys.exit(3)


def main():
    # exactly ONE JSON line may reach stdout: libraries (NCCL's version banner) write there too, so everything but the
    # final line is sent to stderr at the file-descriptor level
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="clipk", choices=["clipk", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--mode", default=None, choices=["local", "global"])
    ap.add_argument("--gwg", type=int, default=None, choices=[0, 1])
    ap.add_argument("--logit-scale", type=float, default=INIT_SCALE)
    ap.add_argument("--skip-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and gradients of the last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "clipk":
        ap.error("--dump-outputs applies to --impl clipk")
    args.warmup = max(args.warmup, 3) if args.impl == "clipk" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_clipk(args)


if __name__ == "__main__":
    main()
