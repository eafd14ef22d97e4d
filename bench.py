"""Benchmark of the DDPM hot path (BASELINE.json metric: denoising steps/sec on (B,32,512)-derived latents).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
  python bench.py --impl reference --steps K --warmup W    # CPU restatement of the reference path (oracle)
  python bench.py --steps K --warmup W --dump-outputs bench_outputs   # + the last timed step's outputs as .npy

Headline workload (config.workload) = BASELINE.json configs[1]: ddpm-mel-32seq-512.cfg (TransformerDDPM L6/H8/K2/M2048,
C=42 after slice-mel-512), batch 128 per GPU, one optimizer step = device threefry draws + q_sample + forward +
backward + NCCL all-reduce + clip + Adam.  A "step" is one pass of that hot path over one batch; value =
samples x steps / s over all GPUs (weak scaling).  The same invocation also measures the other BASELINE configs and
puts them into the line's `extra` block (each with ms/step and its fraction of the sustained bf16 peak):
  cfg3  sample_ncsn reverse step, 1000 samples per GPU (weak) and 1000/N per GPU (strong)
  cfg4  ddpm-mel-32seq-512-large training, 128 per GPU (batch 1024 over 8 GPUs)
  cfg5  ddpm-multi-32seq-512 (C=146) reverse step, 1000 per GPU and 1000/N per GPU
  c512  the C=512 "no slice" variant of the headline model (the metric string says Bx32x512), training 128 per GPU
With N > 1 the line also carries the data-parallel proof: `dp_rank_divergence` (max - min over ranks of a bitwise
parameter checksum after the timed steps; must be 0) and `dp_vs_single_rel_l2` (all-reduced gradient of one step vs
the same global batch on one GPU).

The reference arm and the cpu_baseline leg run the CPU oracle (oracle/, torch fp32) and never import the product
package, so no product shared library is mapped into a reference process.

--dump-outputs DIR writes what the last of the K timed steps handed back to its caller as DIR/<name>.npy (rank 0):
  train   loss.npy, grad_norm.npy (the step's global mean loss and clipped gradient norm) and params.npy (the updated
          parameters, flattened in layout order)
  sample  samples.npy (the (N, 32, C) state after the reverse step)
Inputs are seeded, so two builds run with the same arguments can be compared array for array.  An array of more than
DUMP_MAX_VALUES values is stored as its values at DUMP_MAX_VALUES fixed, seeded positions (params.npy of the base model
is such a sample), which keeps a dump well under 64 MB.  The backward pass accumulates some gradients with float
atomics, so train dumps agree to a tolerance, not bit for bit: two runs of one build with --steps 20 --warmup 5 (B200,
1000 W power limit) differed by 8e-5 relative in loss and 1.6e-4 in the rel-L2 of params.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "denoising steps/sec (Bx32x512 latents)"
UNIT = "sample-steps/s"

BASE = dict(arch="TransformerDDPM", num_layers=6, num_heads=8, num_mlp_layers=2, mlp_dims=2048, seq_len=32)
LARGE = dict(arch="TransformerDDPM", num_layers=8, num_heads=16, num_mlp_layers=3, mlp_dims=2048, seq_len=32)
MODELS = {
    "base_c42": dict(channels=42, **BASE),       # ddpm-mel-32seq-512.cfg
    "large_c42": dict(channels=42, **LARGE),     # ddpm-mel-32seq-512-large.cfg
    "base_c146": dict(channels=146, **BASE),     # ddpm-multi-32seq-512.cfg (TransformerDDPM4 == TransformerDDPM)
    "base_c512": dict(channels=512, **BASE),     # --slice_ckpt='' variant
}
HEADLINE_WL = "train ddpm-mel-32seq-512.cfg (TransformerDDPM L6 H8 K2 M2048 C42), batch 128/GPU"
DUMP_MAX_VALUES = 1 << 22       # per dumped array: 16 MiB of float32


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy in float32 (float64 stays float64).  An array with more than
    DUMP_MAX_VALUES values is replaced by its flattened values at DUMP_MAX_VALUES positions drawn without replacement by
    np.random.default_rng(0) and sorted, so the same positions are kept in every run."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        a = a if a.dtype == np.float64 else a.astype(np.float32)
        if a.size > DUMP_MAX_VALUES:
            pos = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_VALUES, replace=False))
            a = a.reshape(-1)[pos]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    print(f"bench: wrote {', '.join(f'{n}.npy' for n in arrays)} to {out_dir}", file=sys.stderr, flush=True)


def flat_params(named: dict) -> np.ndarray:
    """Parameter tensors (name -> array, in layout order) as one flat float32 vector."""
    return np.concatenate([np.asarray(v, np.float32).reshape(-1) for v in named.values()])


def synthetic_batch(batch: int, seed: int, channels: int = 42):
    """(B,32,512) N(0,1) 'MusicVAE' latents -> slice `channels` dims -> min/max normalise to [-1,1]
    (input_pipeline.py:36-48)."""
    rng = np.random.default_rng(seed)
    raw = rng.standard_normal((batch, 32, 512)).astype(np.float32)
    if channels < 512:
        idx = np.sort(np.random.default_rng(1234).choice(512, channels, replace=False))
        raw = raw[..., idx]
    x = np.ascontiguousarray(raw)
    lo, hi = x.min(), x.max()
    return np.ascontiguousarray((2.0 * (x - lo) / (hi - lo) - 1.0).astype(np.float32))


class ClockSampler(threading.Thread):
    def __init__(self, device_index: int):
        super().__init__(daemon=True)
        self.idx = device_index
        self.stop_flag = threading.Event()
        self.rows = []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.idx)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return p.get("bf16_tflops", 1590.0), p.get("bf16_tflops_sustained", 1400.0), p.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


# ----------------------------------------------------------------------------------------------- CPU arm (oracle)
def host_threads() -> int:
    """Threads the CPU arm may use: the scheduler affinity mask clipped by a cgroup CPU quota (if any) and by 64."""
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(np.ceil(int(quota) / int(period)))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 64))


def _oracle_kw(m):
    return dict(num_layers=m["num_layers"], num_heads=m["num_heads"], num_mlp_layers=m["num_mlp_layers"],
                mlp_dims=m["mlp_dims"])


class CpuTrainStep:
    """Oracle (torch CPU fp32 restatement of train_ncsn.py:260-288): draws are supplied tensors, one call = forward +
    autograd backward + global-norm clip + Adam.  Pure oracle/ code: nothing of the product package is imported."""

    def __init__(self, batch: int, threads: int, model="base_c42"):
        from oracle import ddpm_oracle as O
        from oracle import layout as LY
        self.O = O
        torch.set_num_threads(threads)
        self.m = MODELS[model]
        self.p = {k: torch.from_numpy(v) for k, v in LY.init_params(seed=1, **self.m).items()}
        self.mom = {k: torch.zeros_like(v) for k, v in self.p.items()}
        self.var = {k: torch.zeros_like(t) for k, t in self.p.items()}
        self.n = 0
        self.set_batch(batch)

    def set_batch(self, batch: int):
        O = self.O
        self.batch = batch
        self.x0 = torch.from_numpy(synthetic_batch(batch, 0, self.m["channels"]))
        rng = np.random.default_rng(2)
        self.eps = torch.from_numpy(rng.standard_normal(tuple(self.x0.shape)).astype(np.float32))
        ap = O.alphas_prod_with_one(O.create_noise_schedule(1e-6, 0.01, 1000, "linear"))
        self.used = torch.from_numpy(ap[rng.integers(1, 1001, batch) - 1])

    def step(self) -> float:
        t0 = time.perf_counter()
        (self.p, self.mom, self.var), self.loss, self.grad_norm, _ = self.O.train_step(
            self.m["arch"], self.p, self.mom, self.var, self.n, self.x0, self.used, self.eps, 1e-3,
            model_kw=_oracle_kw(self.m))
        self.n += 1
        return time.perf_counter() - t0


def cpu_train_step_rate(batch: int, min_seconds: float, max_steps: int, threads: int):
    """(sample-steps/s, steps, seconds, batch) of the CPU restatement at the workload's own batch: one untimed warm-up
    step, then steps until `min_seconds` have passed (at most `max_steps`).  The batch only shrinks if a single step
    would blow the budget."""
    job = CpuTrainStep(batch, threads)
    w = job.step()
    while w > max(6.0, min_seconds) and job.batch > 1:
        job.set_batch(max(1, job.batch // 2))
        w = job.step()
    t0 = time.perf_counter()
    n = 0
    while n < max_steps and (n == 0 or time.perf_counter() - t0 < min_seconds):
        job.step()
        n += 1
    dt = time.perf_counter() - t0
    return job.batch * n / dt, n, dt, job.batch


def run_reference(args):
    """bench.py --impl reference: the CPU oracle on the headline config (same workload string, same per-step batch
    128 x N unless one step would not fit the time budget), all host threads, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, int(os.environ.get("WORLD_SIZE", str(args.gpus))))
    threads = host_threads()
    budget = 170.0                      # seconds for the W + K steps
    want = (args.batch or 128) * world
    job = CpuTrainStep(want, threads)
    w = job.step()                      # sizing probe (also pays the first-call costs); not reported
    per_step = budget / max(1, args.warmup + args.steps)
    while w > per_step and job.batch > 1:
        job.set_batch(max(1, job.batch // 2))
        w = job.step()
    for _ in range(args.warmup):
        job.step()
    times = [job.step() for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"loss": np.atleast_1d(np.asarray(job.loss, np.float32)),
                                         "grad_norm": np.atleast_1d(np.asarray(job.grad_norm, np.float32)),
                                         "params": flat_params({k: v.detach().numpy() for k, v in job.p.items()})})
    sb = job.batch
    ms = 1e3 * float(np.mean(times))
    value = sb / (ms / 1e3)
    # this arm must not map any product code: only oracle/ (torch CPU) may have been imported
    maps = open("/proc/self/maps").read() if os.path.exists("/proc/self/maps") else ""
    product_loaded = sorted({ln.split("/")[-1] for ln in maps.splitlines() if "libsmd" in ln})
    assert "smd_b200" not in sys.modules and not product_loaded, "the reference arm imported product code"
    note = ("CPU restatement of the reference path (oracle/, torch fp32; JAX 0.2.8 / flax 0.3.0 are not installable); "
            + (f"each step is the full batch-{sb} optimizer step" if sb == want else
               f"each step is a batch-{sb} sample of the batch-{want} step (a full step exceeded the time budget)"))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": HEADLINE_WL, "global_batch": want, "parallelism": f"dp{world}",
                       "sample_batch": sb, "note": note},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{args.steps} optimizer steps at batch {sb} (fwd + autograd bwd + clip + Adam), "
                                       f"torch CPU fp32, {threads} threads"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- GPU arm
def time_dominant_gemm(eng, M_tokens: int, cta_group: int, iters: int = 20):
    """Average duration of the dominant kernel (2048x2048 res-block GEMM over M tokens) alone, L2 flushed."""
    from smd_b200 import lib as L
    lib = eng.lib
    A = torch.randn(M_tokens, 2048, device="cuda").to(torch.bfloat16)
    B = torch.randn(2048, 2048, device="cuda").to(torch.bfloat16)
    out = torch.empty(M_tokens, 2048, device="cuda")
    bias = torch.zeros(2048, device="cuda")
    stats = torch.zeros(M_tokens, 2, device="cuda")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    total = 0.0
    for i in range(iters + 3):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(lib.smd_gemm_bf16(A.data_ptr(), B.data_ptr(), M_tokens, 2048, 2048, 0, 0, 256, cta_group,
                                  bias.data_ptr(), None, 0, out.data_ptr(), None, stats.data_ptr(), None, None, st))
        e1.record()
        torch.cuda.synchronize()
        if i >= 3:
            total += e0.elapsed_time(e1)
    return total / iters  # ms


class Ctx:
    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dev = torch.device(f"cuda:{self.local}")
        self.betas = np.linspace(1e-6, 0.01, 1000, dtype=np.float32)
        self.tpeak, self.tsust, self.hbm, self.peak_src = peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, eng):
        for i in range(warmup):
            fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = eng.launch_count()
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t)
        return ms / steps, eng.launch_count() - launches0


def make_train(ctx: Ctx, model: str, B: int):
    from smd_b200 import Engine, ModelConfig
    m = MODELS[model]
    cfg = ModelConfig(**m)
    eng = Engine(cfg, max_batch=B, cta_group=ctx.args.cta_group, training=True)
    eng.set_params(eng.init_params(seed=1))
    eng.init_train_state(ema=False)
    eng.objective_setup(ctx.betas)
    x_host = torch.from_numpy(synthetic_batch(B, 100 + ctx.rank, m["channels"])).pin_memory()
    x_dev = x_host.to(ctx.dev, non_blocking=True)
    loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_done = [None, None]
    world, rank = ctx.world, ctx.rank

    def draws(i):
        # rows [rank*B, (rank+1)*B) of the global batch's threefry streams (utils/losses.py:270-294)
        return eng.draws((i, 17), B, global_batch=B * world, first_row=rank * B)

    def step_resident(i):
        u, e = draws(i)
        eng.train_step(x_dev, u, e, lr=1e-3, world_size=world)

    def step_e2e(i):
        xb = x_host.to(ctx.dev, non_blocking=True)                   # H2D of this step's batch (pinned)
        u, e = draws(i)
        loss, _ = eng.train_step(xb, u, e, lr=1e-3, world_size=world)
        # D2H of the step's loss into pinned memory, every step; the host consumes it one step late (like a logger
        # would), so it never stalls the launch of the next step -- the timed region still ends with a full sync
        j = i & 1
        if loss_done[j] is not None:
            loss_done[j].synchronize()
            _ = float(loss_host[j][0])
        loss_host[j].copy_(loss, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        loss_done[j] = ev

    def outputs():
        # what train_step hands its caller (global mean loss, clipped gradient norm) and the parameters it updated
        return {"loss": eng.loss_mean, "grad_norm": eng.grad_norm, "params": flat_params(eng.flat_to_dict(eng.params))}

    return dict(eng=eng, cfg=cfg, units=B, flops=3.0 * cfg.flops_fwd_per_sample() * B, resident=step_resident,
                e2e=step_e2e, h2d=x_host.numel() * 4, d2h=4, tokens=B * 32, x_host=x_host, outputs=outputs)


def make_sample(ctx: Ctx, model: str, N: int):
    from smd_b200 import Engine, ModelConfig
    m = MODELS[model]
    cfg = ModelConfig(**m)
    eng = Engine(cfg, max_batch=N, cta_group=ctx.args.cta_group, training=False)
    eng.set_params(eng.init_params(seed=1))
    eng.sampler_setup(ctx.betas, key=(0, 5))
    eng.set_sampler_shard(ctx.rank * N, N * ctx.world)
    C = m["channels"]
    x_host = torch.from_numpy(np.random.default_rng(ctx.rank).standard_normal((N, 32, C)).astype(np.float32)).pin_memory()
    x_dev = x_host.to(ctx.dev)
    out_host = torch.empty((N, 32, C), dtype=torch.float32).pin_memory()

    def step_resident(i):
        eng.sample(x_dev, steps=1, use_graph=True)

    def step_e2e(i):
        xb = x_host.to(ctx.dev, non_blocking=True)
        eng.sample(xb, steps=1, use_graph=False)
        out_host.copy_(xb, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    return dict(eng=eng, cfg=cfg, units=N, flops=cfg.flops_fwd_per_sample() * N, resident=step_resident, e2e=step_e2e,
                h2d=x_host.numel() * 4, d2h=x_host.numel() * 4, tokens=N * 32, outputs=lambda: {"samples": x_dev})


def extra_entry(ctx: Ctx, name: str, what: str, job, steps: int, warmup: int):
    ms, _ = ctx.timed(job["resident"], steps, warmup, job["eng"])
    tf = job["flops"] / (ms / 1e3) / 1e12
    return {"name": name, "workload": what, "per_gpu": job["units"], "global": job["units"] * ctx.world,
            "ms_per_step": ms, "value": job["units"] * ctx.world / (ms / 1e3), "unit": UNIT,
            "step_tflops_per_gpu": tf, "step_frac_of_sustained_peak": tf / ctx.tsust}


def dp_proof(ctx: Ctx, eng, B: int):
    """(dp_rank_divergence, dp_vs_single_rel_l2, dp_vs_single_dloss): replicas bit-identical after the timed steps;
    the all-reduced data-parallel gradient of one step equals the single-GPU gradient of the same global batch."""
    from smd_b200 import Engine
    dist = ctx.dist
    chk = eng.params.view(torch.int32).to(torch.int64).sum().reshape(1)
    lo, hi = chk.clone(), chk.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    divergence = float((hi - lo).item())
    x = torch.from_numpy(synthetic_batch(B, 100 + ctx.rank)).to(ctx.dev)
    u, e = eng.draws((12345, 17), B, global_batch=B * ctx.world, first_row=ctx.rank * B)
    eng.compute_grads(x, u, e, global_batch=B * ctx.world)
    eng.reduce_grads(ctx.world)
    torch.cuda.synchronize()
    rel = dl = None
    if ctx.rank == 0:
        G = B * ctx.world
        one = Engine(eng.cfg, max_batch=G, cta_group=ctx.args.cta_group, training=True)
        one.set_params(eng.params.clone())
        one.init_train_state()
        one.objective_setup(ctx.betas)
        xa = torch.cat([torch.from_numpy(synthetic_batch(B, 100 + r)) for r in range(ctx.world)]).to(ctx.dev)
        ua, ea = one.draws((12345, 17), G)
        one.compute_grads(xa, ua, ea, global_batch=G)
        torch.cuda.synchronize()
        rel = float((eng.grads.double() - one.grads.double()).norm() / one.grads.double().norm())
        dl = abs(float(eng.loss_mean) - float(one.loss_mean)) / abs(float(one.loss_mean))
        del one
    dist.barrier()
    return divergence, rel, dl


def run_gpu(args):
    ctx = Ctx(args)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(ctx.local)
    if ctx.world > 1:
        ctx.dist.init_process_group("nccl", device_id=ctx.dev)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    world, rank = ctx.world, ctx.rank

    if args.workload == "train":
        B = args.batch or 128
        job = make_train(ctx, "base_c42", B)
        wl = HEADLINE_WL if B == 128 else f"train ddpm-mel-32seq-512.cfg (TransformerDDPM L6 H8 K2 M2048 C42), batch {B}/GPU"
    else:
        B = args.batch or 1000
        job = make_sample(ctx, "base_c42", B)
        wl = f"sample ddpm-mel-32seq-512.cfg (TransformerDDPM L6 H8 K2 M2048 C42), {B} samples/GPU, 1 reverse step"
    eng = job["eng"]

    # multi-rank runs: NCCL finishes setting up its channels / buffer registrations during the first few dozen
    # collectives (measured at 2 and 8 GPUs: the first ~25 steps run 5-20 % slower, profiles/r02_dp_warmup_ab.txt), so
    # a fixed number of extra untimed steps runs before the W warm-up steps; K timed steps stay exactly K
    settle = 30 if world > 1 else 0
    for i in range(settle):
        job["resident"](100000 + i)
    clocks = ClockSampler(ctx.local)
    clocks.start()
    ms_step, launches = ctx.timed(job["resident"], args.steps, args.warmup, eng)
    clocks.stop_flag.set()
    clocks.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, job["outputs"]())     # before the e2e leg runs further steps
    ms_e2e, _ = ctx.timed(job["e2e"], args.steps, max(3, args.warmup // 2), eng)

    units, flops_step = job["units"], job["flops"]
    value = units * world / (ms_step / 1e3)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": wl, "global_batch": units * world, "parallelism": f"dp{world}",
                       "cta_group": args.cta_group, "steps_per_s": 1e3 / ms_step,
                       "step_tflops": flops_step * world / (ms_step / 1e3) / 1e12,
                       "step_frac_of_sustained_peak": flops_step / (ms_step / 1e3) / 1e12 / ctx.tsust,
                       "l2": ("per-step working set (params+grads+Adam ~400 MB, activations ~1 GB) >> 126 MB L2; no flush"
                              if args.workload == "train" else
                              "per-step working set (bf16 weights 51 MB + activations ~1 GB at 32000 tokens) >> 126 MB L2; "
                              "no flush"),
                       "precision": "bf16 tensor-core operands, fp32 accumulate / master weights / LN / softmax / Adam",
                       "rng": "device threefry draws (labels, alpha-bar, eps) are inside the timed step",
                       "untimed_settle_steps": settle},
            "clocks": clocks.summary(),
            "e2e": {"value": units * world / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": job["h2d"], "d2h_bytes_per_step": job["d2h"]},
            "gpu_launches": int(launches)}

    if world > 1 and args.workload == "train":
        div, rel, dl = dp_proof(ctx, eng, units)
        line["dp_rank_divergence"] = div
        line["dp_vs_single_rel_l2"] = rel
        line["dp_vs_single_dloss_rel"] = dl

    m_tokens = job["tokens"]
    g_ms = time_dominant_gemm(eng, m_tokens, args.cta_group) if rank == 0 else None
    del job, eng
    torch.cuda.empty_cache()

    if not args.no_extra:
        xs, xw = max(5, args.steps // 2), 3
        extra = []
        per = max(1, 1000 // world)
        jobs = [("cfg3_sample_n1000_per_gpu", "sample ddpm-mel-32seq-512.cfg, 1000 samples/GPU, 1 reverse step (weak)",
                 lambda: make_sample(ctx, "base_c42", 1000))]
        if world > 1:
            jobs.append(("cfg3_sample_n1000_total", f"sample ddpm-mel-32seq-512.cfg, 1000 samples total = {per}/GPU (strong)",
                         lambda: make_sample(ctx, "base_c42", per)))
        jobs.append(("cfg4_large_train_b128_per_gpu", f"train ddpm-mel-32seq-512-large.cfg (L8 H16 K3), batch 128/GPU = {128 * world} global",
                     lambda: make_train(ctx, "large_c42", 128)))
        jobs.append(("cfg5_multi_sample_n1000_per_gpu", "sample ddpm-multi-32seq-512.cfg (C=146), 1000 samples/GPU (weak)",
                     lambda: make_sample(ctx, "base_c146", 1000)))
        if world > 1:
            jobs.append(("cfg5_multi_sample_n1000_total", f"sample ddpm-multi-32seq-512.cfg (C=146), 1000 samples total = {per}/GPU (strong)",
                         lambda: make_sample(ctx, "base_c146", per)))
        jobs.append(("c512_noslice_train_b128_per_gpu", "train base model on unsliced C=512 latents, batch 128/GPU",
                     lambda: make_train(ctx, "base_c512", 128)))
        for name, what, mk in jobs:
            j = mk()
            extra.append(extra_entry(ctx, name, what, j, xs, xw))
            del j
            torch.cuda.empty_cache()
        line["extra"] = extra

    if rank == 0:
        gflop = 2.0 * m_tokens * 2048 * 2048
        ach = gflop / (g_ms / 1e3) / 1e12
        line["roofline"] = {"bound": "tensor", "achieved": ach, "peak": ctx.tpeak, "unit": "TFLOP/s",
                            "frac": ach / ctx.tpeak,
                            "traffic": None,     # DRAM bytes need an ncu capture; see profiles/ (not measurable in-run)
                            "algorithmic_bytes": m_tokens * 2048 * 6 + 2048 * 2048 * 2 + m_tokens * 8 + 8192,
                            "peak_source": f"MEASURED_PEAKS.json bf16_tflops ({ctx.peak_src}, burst: kernel timed alone)",
                            "kernel": f"gemm_bf16_tcgen05_kernel<{args.cta_group}> [{m_tokens}x2048x2048] res-block GEMM "
                                      "+ bias + row-stat epilogue", "ms_per_launch": g_ms}
        if not args.no_cpu:
            threads = host_threads()
            rate, n, dt, sb = cpu_train_step_rate(128, 12.0, 10, threads)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"{n} optimizer steps at batch {sb} in {dt:.1f}s, torch CPU fp32 restatement "
                                              f"of the reference path (oracle/; JAX unavailable), {threads} threads"}
        print(json.dumps(line), flush=True)
    if world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "sample"])
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--cta-group", dest="cta_group", type=int, default=2)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra BASELINE configs")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
