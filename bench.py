#!/usr/bin/env python
"""Benchmark of the hot path: denoising steps/s of the MDM sampling loop at B=64, L=196, D=263 (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's engine (CUDA kernels through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU implementation of the same path
                                                             # (the pinned CPU restatement, oracle/; /root/reference does
                                                             #  not exist on the GPU box)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's samples to DIR/sample.npy,
                                                             # to compare two builds output for output

One "step" is one iteration of `p_sample_loop` over one batch of 64 motions: one denoiser pass (8-layer MDM
transformer over 64 x 197 tokens) + the posterior/noise update -- everything the reference does in one loop
iteration (SURVEY.md 8(d)).  Workload = BASELINE.json configs[1]: unconditional DDPM, T=1000, random-init weights,
synthetic inputs.  Multi-GPU is weak scaling: every rank samples its own 64 motions (no per-step traffic) and one
NCCL all-gather of the finished samples closes the timed region; `value` counts the steps of all ranks.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's banner / debug lines do not belong on stdout

# Rank 0 prints exactly ONE JSON line on stdout.  Libraries (NCCL's version banner, torch warnings) write to fd 1
# whenever they like, so fd 1 is pointed at stderr for the life of the process and the JSON line goes to the saved fd.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B, D, L, S, T = 64, 263, 196, 197, 1000
D_MODEL, FF, LAYERS, HEADS = 512, 1024, 8, 4
DUMP_LIMIT_BYTES = 64 << 20
METRIC = "denoising steps/sec (B=64, L=196, D=263, 1000 steps)"
WORKLOAD = "configs[1]: unconditional DDPM p_sample_loop, T=1000, B=64 per GPU, L=196, D=263, MDM 8L/512d/ff1024/4h"
MIN_WARMUP = 3
UNIT = "denoising steps/s (one step = one MDM pass + posterior update over a batch of 64)"


def flops_per_pass(batch: int) -> float:
    """SURVEY.md 8(d): algorithmic FLOPs of one MDM.forward (GEMM + attention contractions only)."""
    tok = S * batch
    per_tok_layer = 2 * D_MODEL * 3 * D_MODEL + 2 * D_MODEL * D_MODEL + 2 * 2 * D_MODEL * FF + 2 * 2 * S * D_MODEL
    return LAYERS * tok * per_tok_layer + 2 * 2 * D * D_MODEL * L * batch + 2 * 2 * D_MODEL * D_MODEL * batch


KERNEL_FLOPS = {  # algorithmic FLOPs per launch at `batch` sequences of S tokens
    "qkv": lambda b: 2.0 * S * b * D_MODEL * 3 * D_MODEL,
    "out_proj": lambda b: 2.0 * S * b * D_MODEL * D_MODEL,
    "out_proj_ln1": lambda b: 2.0 * S * b * D_MODEL * D_MODEL,
    "ffn1": lambda b: 2.0 * S * b * D_MODEL * FF,
    "ffn2": lambda b: 2.0 * S * b * D_MODEL * FF,
    "ffn2_ln2": lambda b: 2.0 * S * b * D_MODEL * FF,
    "attention": lambda b: 2.0 * 2 * S * S * D_MODEL * b,
    "frame_embed": lambda b: 2.0 * L * b * D * D_MODEL,
    "out_head": lambda b: 2.0 * L * b * D * D_MODEL,
    # one chained launch = out-proj + FFN1 + FFN2 + the next layer's QKV projection (the last one: + the output head)
    "chain": lambda b: 2.0 * S * b * D_MODEL * (D_MODEL + 2 * FF + 3 * D_MODEL),
    "chain_last": lambda b: 2.0 * S * b * D_MODEL * (D_MODEL + 2 * FF) + 2.0 * L * b * D * D_MODEL,
}


def measured_peaks(timed_region_s: float):
    """Roofline denominators: MEASURED_PEAKS.json (driver-written).  Its burst figure is the denominator for a kernel
    timed alone or inside a short region; the sustained one only for a kernel timed inside a seconds-long step."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    burst = timed_region_s < 1.0
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        key = "bf16_tflops" if burst or "bf16_tflops_sustained" not in p else "bf16_tflops_sustained"
        return {"bf16_tflops": p[key], "hbm_gbs": p.get("hbm_gbs"),
                "source": f"MEASURED_PEAKS.json {key} (cuBLAS bf16; timed region {timed_region_s:.2f} s -> {'burst' if key == 'bf16_tflops' else 'sustained'})"}
    return {"bf16_tflops": 1650.0 if burst else 1400.0, "hbm_gbs": 6650.0,
            "source": f"fallback of B200_PROFILING.md ({'burst' if burst else 'sustained'})"}


class NvmlSampler:
    """SM clock and throttle reasons sampled IN-PROCESS through NVML every ~5 ms (nvidia-smi's 100 ms period cannot
    resolve a 40 ms timed region).  Same summary format as ClockSampler; falls back to it when NVML is unavailable."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index: int, period_s: float = 0.005):
        self.index, self.period, self.rows, self.windows = index, period_s, [], []
        self.ok, self._stop, self.thread = False, threading.Event(), None
        self.fallback = None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.index
            if visible:
                try:
                    phys = int(visible.split(",")[self.index])
                except (ValueError, IndexError):
                    phys = self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001  (no NVML in this environment)
            self.fallback = ClockSampler(self.index)
            self.fallback.__enter__()
        return self

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:  # noqa: BLE001
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((time.time(), mhz, mask))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def __exit__(self, *a):
        if self.fallback:
            self.fallback.__exit__()
            return
        self._stop.set()
        if self.thread:
            self.thread.join(timeout=1)

    def window(self, name, t0, t1):
        if self.fallback:
            self.fallback.window(name, t0, t1)
        self.windows.append((name, t0, t1))

    def summary(self):
        if self.fallback:
            out = self.fallback.summary()
            out["sampler"] = "nvidia-smi -lms 100"
            return out
        name, t0, t1 = self.windows[0]
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        sm = sorted(r[1] for r in rows)
        mask = 0
        for r in rows:
            mask |= r[2]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": [n for bit, n in self.REASONS if mask & bit], "samples": len(sm), "window": name,
                "sampler": f"NVML in-process, {self.period * 1e3:.0f} ms period"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.windows = []  # (name, t0, t1) host-clock windows that bracket device work (barrier + synchronize on both sides)

    def __enter__(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:  # noqa: BLE001
                self.proc.kill()

    def window(self, name, t0, t1):
        self.windows.append((name, t0, t1))

    def summary(self):
        """Samples inside the timed region; when it is shorter than nvidia-smi's 100 ms period can resolve, the samples
        of the end-to-end region (the same workload, also under load) are added and `window` says so."""
        used, rows = [], []
        for name, t0, t1 in self.windows:
            rows += [r for (ts, r) in self.rows if t0 <= ts <= t1]
            used.append(name)
            if len(rows) >= 3:
                break
        out = self._summarise(rows)
        out["window"] = "+".join(used)
        return out

    def _summarise(self, rows):
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def usable_cpus() -> int:
    """Host threads this process may actually use: affinity mask and cgroup CPU quota, not just os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, int(float(parts[0]) / float(parts[1]) + 0.5)))
            else:
                quota = int(parts[0])
                if quota > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                        n = min(n, max(1, int(quota / int(f.read()) + 0.5)))
        except (OSError, ValueError, IndexError):
            continue
    return n


def cpu_reference_steps(max_steps: int, budget_s: float, warmup: int = 1):
    """The reference's CPU implementation of one loop iteration at B=64 (pinned restatement, all usable host threads)."""
    from oracle import condmdi_oracle as O
    threads = usable_cpus()
    torch.set_num_threads(threads)
    sd = O.random_state_dict(seed=0)
    tab = O.make_tables("")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, D, 1, L, generator=g)
    noise = torch.randn(B, D, 1, L, generator=g)
    c = O.Conditioning()
    t_idx = T - 1
    with torch.no_grad():
        for _ in range(warmup):
            x = O.p_sample(sd, tab, x, torch.full((B,), t_idx), c, noise)["sample"]
            t_idx = (t_idx - 1) % T  # past t = 0 the walk starts over at t = T - 1
        done, t0 = 0, time.perf_counter()
        while done < max_steps:
            x = O.p_sample(sd, tab, x, torch.full((B,), t_idx), c, noise)["sample"]
            t_idx = (t_idx - 1) % T
            done += 1
            if time.perf_counter() - t0 > budget_s:
                break
        dt = time.perf_counter() - t0
    return done, dt, threads, x


def dump_outputs(path: str, arrays: dict):
    """Write each array as <path>/<name>.npy in float32.  An output larger than DUMP_LIMIT_BYTES keeps a fixed, seeded
    choice of its motions (rows of dim 0), in their original order."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().to("cpu", torch.float32)
        rows = DUMP_LIMIT_BYTES // (a[0].numel() * 4)
        if a.shape[0] > rows:
            a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values]
        np.save(os.path.join(path, f"{name}.npy"), a.numpy())


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return  # the CPU arm runs on rank 0 only
    warm = max(args.warmup, MIN_WARMUP)
    done, dt, threads, x = cpu_reference_steps(args.steps, budget_s=float("inf"), warmup=warm)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sample": x})
    value = done / dt
    sample = f"{done} consecutive DDPM steps (t={T - 1 - warm}..) of the B=64 unconditional loop on the host CPU, fp32, {threads} threads"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
            "warmup": warm, "ms_per_step": 1e3 * dt / done, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32", "data": "synthetic (random-init weights, N(0,1) inputs)",
            "config": {"workload": WORKLOAD, "global_batch": args.gpus * B},
            "note": "reference = the reference's PyTorch CPU p_sample (pinned restatement in oracle/; /root/reference is absent on "
                    "the GPU box).  ONE host CPU whatever --gpus says: a batch of 64 per step, all usable threads; it does not "
                    "scale with N, so only the N=1 ratio compares like with like",
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def eager_library_baseline(dev, steps: int = 20):
    """The same DDPM step with STOCK torch.nn.TransformerEncoder kernels (cuBLAS / ATen) on this GPU: fp32 as the
    reference computes it, and with TF32 matmuls allowed (outside the fp32 parity gate) -- "the library to beat"."""
    import math

    import torch.nn as nn

    class EagerMDM(nn.Module):
        def __init__(self):
            super().__init__()
            self.pose = nn.Linear(D, D_MODEL)
            layer = nn.TransformerEncoderLayer(d_model=D_MODEL, nhead=HEADS, dim_feedforward=FF, dropout=0.1, activation="gelu")
            self.enc = nn.TransformerEncoder(layer, num_layers=LAYERS, enable_nested_tensor=False)
            self.time = nn.Sequential(nn.Linear(D_MODEL, D_MODEL), nn.SiLU(), nn.Linear(D_MODEL, D_MODEL))
            self.final = nn.Linear(D_MODEL, D)
            pe = torch.zeros(5000, D_MODEL)
            pos = torch.arange(0, 5000, dtype=torch.float).unsqueeze(1)
            div = torch.exp(torch.arange(0, D_MODEL, 2).float() * (-math.log(10000.0) / D_MODEL))
            pe[:, 0::2], pe[:, 1::2] = torch.sin(pos * div), torch.cos(pos * div)
            self.register_buffer("pe", pe.unsqueeze(1))

        def forward(self, x, t):
            emb = self.time(self.pe[t])
            h = self.pose(x.permute(3, 0, 1, 2).reshape(L, -1, D))
            seq = torch.cat((emb.permute(1, 0, 2), h), 0)
            seq = seq + self.pe[: seq.shape[0]]
            return self.final(self.enc(seq)[1:]).reshape(L, -1, D, 1).permute(1, 2, 3, 0)

    torch.manual_seed(0)
    model = EagerMDM().to(dev).eval()
    c1, c2, lv = (torch.rand(T, device=dev) for _ in range(3))

    def step(x, t):
        x0 = model(x, t)
        mean = c1[t].view(-1, 1, 1, 1) * x0 + c2[t].view(-1, 1, 1, 1) * x
        return mean + (t != 0).float().view(-1, 1, 1, 1) * torch.exp(0.5 * lv[t].view(-1, 1, 1, 1)) * torch.randn_like(x)

    out = {"what": "stock torch.nn.TransformerEncoder (eager, eval), same step (one pass + posterior update), B=64, this GPU, same run"}
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for name, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            x = torch.randn(B, D, 1, L, device=dev)
            with torch.no_grad():
                for i in range(3):
                    x = step(x, torch.full((B,), T - 1 - i, device=dev))
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(steps):
                    x = step(x, torch.full((B,), T - 4 - i, device=dev))
                e1.record()
                torch.cuda.synchronize()
            out[f"{name}_steps_per_s"] = round(steps / (e0.elapsed_time(e1) * 1e-3), 2)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    del model
    torch.cuda.empty_cache()
    return out


def other_configs(C, dev, world: int):
    """BASELINE.json configs[2], [3], [4] at B=64 on this rank's GPU, through the public reference-facing API
    (ClassifierFreeSampleModel, p_sample_loop / ddim_sample_loop), bounded to <= 100 steps each (device-timed)."""
    text = C.MDM(njoints=D, nfeats=1, latent_dim=D_MODEL, ff_size=FF, num_layers=LAYERS, num_heads=HEADS, cond_mode="text",
                 cond_mask_prob=0.1).to(dev)
    plain = C.MDM(njoints=D, nfeats=1, latent_dim=D_MODEL, ff_size=FF, num_layers=LAYERS, num_heads=HEADS, cond_mode="no_cond").to(dev)
    g = torch.Generator().manual_seed(1)
    cond = torch.randn(B, 512, generator=g).to(dev)
    text.encode_text = lambda t: cond
    cfg = C.ClassifierFreeSampleModel(text)
    x_obs = torch.randn(B, D, 1, L, generator=g).to(dev)
    kf = C.get_keyframes_mask(x_obs, torch.full((B,), L), "benchmark_sparse", trans_length=5)
    y_mask = torch.ones(B, 1, 1, L, dtype=torch.bool, device=dev)
    scale = torch.full((B,), 2.5, device=dev)
    d1000 = C.create_gaussian_diffusion()
    d100 = C.create_gaussian_diffusion(use_ddim=True)
    d1000.rng = d100.rng = "engine"

    def timed(diff, model, y, sampler, total, n):
        def run(k):
            getattr(diff, sampler)(model, (B, D, 1, L), model_kwargs={"y": y}, skip_timesteps=total - k)
        run(MIN_WARMUP)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(n)
        e1.record()
        torch.cuda.synchronize()
        return {"steps_per_s": round(n / (e0.elapsed_time(e1) * 1e-3), 2), "steps": n}

    y3 = {"text": [""] * B, "text_scale": scale, "mask": y_mask, "imputate": 1, "stop_imputation_at": 1,
          "replacement_distribution": "conditional", "inpainted_motion": x_obs, "inpainting_mask": kf}
    y4 = dict(y3, reconstruction_guidance=True, reconstruction_weight=20.0, gradient_schedule=None, diffusion_steps=1000,
              stop_recguidance_at=0)
    out = {"note": f"per GPU (B=64 on each of {world} rank(s); rank 0's numbers), device-timed, bounded step counts; one step = "
                   "everything the reference does in one loop iteration"}
    out["configs[2] CFG 2.5 + benchmark_sparse keyframe imputation, DDPM (2 passes/step)"] = timed(d1000, cfg, y3, "p_sample_loop", T, 100)
    out["configs[3] CFG + imputation + reconstruction guidance w=20, T_trans=5, DDPM (2 passes + input-VJP per step)"] = \
        timed(d1000, cfg, y4, "p_sample_loop", T, 30)
    out["configs[4] DDIM-100 (ddim_sample_loop, eta=0), unconditional, per GPU"] = timed(d100, plain, {}, "ddim_sample_loop", 100, 100)
    for m in (text, plain):
        for eng in getattr(m, "_condmdi_engines", {}).values():
            eng.close()
    torch.cuda.empty_cache()
    return out


def run_engine(args):
    import torch.distributed as dist

    import condmdi_b200 as C

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    precision = C.capi.PRECISION_BF16 if args.precision == "bf16" else C.capi.PRECISION_BF16X3

    torch.manual_seed(0)
    model = C.MDM(njoints=D, nfeats=1, latent_dim=D_MODEL, ff_size=FF, num_layers=LAYERS, num_heads=HEADS, cond_mode="no_cond")
    model = model.to(dev)
    diffusion = C.create_gaussian_diffusion()
    eng = model.engine_for(dev, max_batch=B, precision=precision)
    eng.set_schedule(diffusion.betas, diffusion.timestep_map)
    gathered = torch.empty((world * B, D, 1, L), device=dev) if world > 1 else None

    def loop(nsteps, skip=0, seed=1):
        """nsteps iterations of the 1000-step loop for this rank's 64 motions (+ the all-gather when sharded)."""
        out = None
        left = nsteps
        while left > 0:
            n = min(left, T - skip)
            out = eng.sample(B, skip_timesteps=skip, num_steps=n, seed=seed, sample_offset=rank * B)["sample"]
            left -= n
            skip = 0
        if world > 1:
            dist.all_gather_into_tensor(gathered, out)
        return out

    # ---- warm-up (graph capture, clocks) ----
    clocks = NvmlSampler(local)
    clocks.__enter__()
    warm = max(args.warmup, MIN_WARMUP)
    loop(warm)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- timed: K steps, inputs resident on the device ----
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = eng.launch_count
    barrier()
    w0 = time.time()
    e0.record()
    out = loop(args.steps)
    e1.record()
    barrier()
    clocks.window("timed", w0, time.time())
    if args.dump_outputs and rank == 0:
        # what the timed loop hands its caller: this rank's samples, or every rank's after the all-gather
        dump_outputs(args.dump_outputs, {"sample": gathered if world > 1 else out})
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count - launches0
    tms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms.item())
    value = world * args.steps / (ms * 1e-3)

    # ---- end to end through the C ABI with HOST buffers: x_T from pinned memory in, samples out ----
    x_host = torch.randn(B, D, 1, L).pin_memory()
    out_host = torch.empty(B, D, 1, L).pin_memory()
    eng.sample(B, x_T=x_host, num_steps=3, seed=1, host_buffers=True, out=out_host)
    barrier()
    t0, w0 = time.perf_counter(), time.time()
    left = args.steps
    while left > 0:
        n = min(left, T)
        eng.sample(B, x_T=x_host, num_steps=n, seed=1, sample_offset=rank * B, host_buffers=True, out=out_host)
        left -= n
    if world > 1:
        dist.all_gather_into_tensor(gathered, out_host.to(dev, non_blocking=True))
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks.window("e2e", w0, time.time())
    clocks.__exit__()
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    calls = -(-args.steps // T)
    e2e = {"value": world * args.steps / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": calls * x_host.numel() * 4 / args.steps, "d2h_bytes_per_step": calls * out_host.numel() * 4 / args.steps,
           "note": "cmdi_sample with host_buffers=1: pinned x_T copied in, finished samples copied out, inside the timed region"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel, measured live (CUDA events between the launches of one pass) ----
    peaks = measured_peaks(ms * 1e-3)
    prof = eng.profile_pass(B)
    prof = eng.profile_pass(B)  # second pass: warm
    by_kind = {}
    for name, t_ms in prof:
        k = by_kind.setdefault(name, [0.0, 0])
        k[0] += t_ms
        k[1] += 1
    step_ms = sum(v[0] for v in by_kind.values())
    dom = max((k for k in by_kind if k in KERNEL_FLOPS), key=lambda k: by_kind[k][0])
    dom_ms = by_kind[dom][0] / by_kind[dom][1]
    achieved = KERNEL_FLOPS[dom](B) / (dom_ms * 1e-3) / 1e12
    split = 3 if precision == C.capi.PRECISION_BF16X3 else 1
    traffic, traffic_src = None, None
    try:  # DRAM bytes of the dominant kernel from the committed `ncu --set full` capture (per launch, like `achieved`)
        with open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("kernel") == dom:
            traffic, traffic_src = tr["dram_bytes_read"] + tr["dram_bytes_write"], tr["source"]
    except (OSError, ValueError, KeyError):
        pass
    kname = "linear_chain_kernel (out-proj + FFN1 + FFN2 + next QKV of one encoder layer)" if dom.startswith("chain") else f"linear2_kernel ({dom})"
    roofline = {"bound": "tensor", "kernel": f"{kname}, {by_kind[dom][1]} launches/step", "achieved": achieved,
                "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"], "traffic": traffic,
                "traffic_unit": "bytes of DRAM read + written per launch", "traffic_source": traffic_src,
                "peak_source": peaks["source"], "launch_ms": dom_ms, "share_of_step": by_kind[dom][0] / step_ms,
                "mma_terms_per_product": split, "tensor_pipe_frac_incl_split": split * achieved / peaks["bf16_tflops"],
                "frac_ceiling": 1.0 / split,  # fp32-parity mode spends `split` MMAs per algorithmic product
                "whole_step_algorithmic_tflops": flops_per_pass(B) * args.steps / (ms * 1e-3) / 1e12,
                "per_kernel_ms_per_step": {k: round(v[0], 4) for k, v in by_kind.items()},
                "between_kernels_ms_per_step": round(ms / args.steps - step_ms, 4),
                "note": "achieved = algorithmic FLOPs (2MNK, fp32-equivalent product) / event-timed launch; the bf16x3 split "
                        "issues 3 MMAs per product, so the tensor pipe does `mma_terms_per_product` x that work; "
                        "between_kernels = graph-replayed step time minus the sum of the per-kernel times (the step kernel, "
                        "kernel tails / ramps at the kernel boundaries, graph launch)"}

    # ---- CPU baseline on this box's host cores: a bounded sample of the same workload ----
    cpu = None  # timed at N=1 only (the other ranks' processes would compete for the same host cores)
    if world == 1:
        done, dt, threads, _ = cpu_reference_steps(max_steps=12, budget_s=25.0)
        cpu = {"value": done / dt, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{done} consecutive DDPM steps of the same B=64 loop on the host CPU (fp32 PyTorch restatement of the reference)"}

    # ---- the other BASELINE configs and the library (eager PyTorch) baseline, same run, same GPU ----
    configs = other_configs(C, dev, world) if not args.skip_configs else None
    library = eager_library_baseline(dev) if (world == 1 and not args.skip_configs) else None

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16x3 (bf16 hi/lo operand split, fp32 accumulate: fp32-parity mode)" if split == 3 else "bf16 (fp32 accumulate; fast mode, outside the fp32 parity gate)",
            "data": "synthetic (random-init weights, engine Philox noise)",
            "config": {"workload": WORKLOAD,
                       "global_batch": world * B, "parallelism": f"batch-sharded x{world}, one NCCL all-gather of finished samples",
                       "l2": "per-step working set (weights 70 MB as bf16 hi+lo, activations ~0.4 GB) exceeds the 126 MB L2; no explicit flush",
                       "cuda_graph": f"one captured {len(prof) + 1}-kernel step graph, replayed per step, step index on the device"},
            "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "configs": configs, "library_baseline": library}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16"])
    ap.add_argument("--skip-configs", action="store_true", help="only configs[1]: skip the configs block and the eager-PyTorch baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the samples of the last timed step as DIR/sample.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
