"""bench.py -- headline benchmark: sampled trajectories / second for a full ``sample()`` call.

Workload (BASELINE.json configs[1], SURVEY 8d "cfg2"): JannerUNet1d(in 14, model_dim 32, dim_mult [1,2,2,2], k=5),
H=32, d=14, DiscreteDiffusionSDE(predict_noise=False, 100 diffusion steps, cosine), DDPM solver with 100 sampling
steps, temperature 0.5, fix_mask on the first observation, batch 4096 candidate trajectories PER GPU (weak scaling),
synthetic weights (seed 0) / inputs (seed 1) / noise (seed 2 + rank).  The workload definitions live in
``cleandiffuser_b200/workloads.py`` and are the ones the full-size parity tests run (tests/test_baseline_configs_gpu.py).

Math mode: ``tf32`` (the library default): tcgen05 kind::tf32 over fp32 activations and weights, fp32 accumulate -- the
arithmetic of the reference's own GPU path (cuDNN TF32 convs); ``--math bf16`` / ``--math fp32`` select the other programs.

One "step" = one complete ``sample()`` call (initial noise, 100 reverse iterations, final all-gather when N > 1).

  python bench.py --gpus 1 --steps 5 --warmup 3              # this framework (CUDA engine through the C ABI)
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs OUT   # + the last timed step's samples as OUT/x0.npy
  python bench.py --impl reference --steps 2 --warmup 1      # CPU arm: the reference's algorithm (oracle port) on host cores
  torchrun ... bench.py --gpus N ...                         # one rank per GPU, NCCL

Prints ONE JSON line (rank 0).  See the task contract for the keys; additionally:
  roofline            live per-kernel measurement of the dominant kernel family (fused conv GEMM) via cds_plan_profile
  cpu_baseline        the oracle port timed on the host cores on a bounded sample of the same workload
  gpu_eager_baseline  the SAME sample() on the SAME GPU through this package's PyTorch loop (CDS_BACKEND=torch: ATen / cuDNN /
                      cuBLAS kernels launched op by op from Python, TF32 convs as torch defaults) -- what the reference's own
                      code path costs on this B200 (SURVEY 8d's "beat this" number); N = 1 only
  other_configs       short measurements of BASELINE configs 3 / 4 / 5 at their per-GPU batch on the same ranks (value is the
                      whole-job aggregate like the headline), with their tensor-roofline fraction
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

H, D, T_DIFF, S_STEPS, BATCH = 32, 14, 100, 100, 4096
OBS = 11
WORKLOAD = "cfg2: JannerUNet1d H=32 d=14, DiscreteDiffusionSDE DDPM 100 steps, batch 4096/GPU"
# SURVEY 8(d): canonical algorithmic HBM bytes per trajectory for a full 100-step sample() (per-fused-conv
# activation traffic + x_t/noise + amortised weights)
ALG_BYTES_PER_TRAJ = 33.82e6


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def build_agent(device, seed=0):
    """cfg2's diffusion object (cleandiffuser_b200/workloads.py::cfg2) -> (agent, denoiser, fix_mask)"""
    from cleandiffuser_b200 import workloads
    wl = workloads.cfg2(device, batch=1, steps=T_DIFF, seed=seed)
    return wl.agent, wl.agent.model["diffusion"], wl.agent.fix_mask[0].cpu()


def make_prior(batch, seed=1):
    g = torch.Generator().manual_seed(seed)
    prior = torch.zeros(batch, H, D)
    prior[:, 0, :OBS] = torch.randn(batch, OBS, generator=g)
    return prior


def tensor_peaks():
    """(tf32 dense TFLOP/s, bf16 dense TFLOP/s, source): bf16 measured (MEASURED_PEAKS.json, sustained), tf32 = half of it (the
    tensor pipe runs kind::tf32 at half the bf16 rate; no measured tf32 figure exists in MEASURED_PEAKS.json)"""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            bf16 = json.load(f)["bf16_tflops_sustained"]
        return bf16 / 2, bf16, "MEASURED_PEAKS.json bf16_tflops_sustained (tf32 = half)"
    return 1125.0, 2250.0, "fallback (B200_PROFILING.md nominal dense)"


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def wait_first(self, timeout=5.0):
        """nvidia-smi needs ~0.5 s before its first line: block until it is sampling (so that the timed region is covered)."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)
        return len(self.rows)

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, first=0, last=None):
        """Rows [first, last) = the samples taken while the measured workload was running."""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[first:last]:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arm
def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def cpu_reference_arm(steps, warmup, sample_batch=256):
    """The reference's algorithm on the host cores: oracle port of JannerUNet1d + DiscreteDiffusionSDE.sample
    (PyTorch CPU primitives, exactly what the reference executes on CPU), on a bounded sample of the workload.
    Thread count: the fastest of {64, 32, 16} (capped by the core count) on a 2-forward probe (small convs stop scaling, and
    get much slower, long before 128 threads); the count used is reported as ``cores``."""
    import oracle.nets as onets
    import oracle.sampler as osamp
    _, net, mask = build_agent("cpu")
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    fn = lambda x, t, c=None: onets.janner_unet(sd, x, t, c, emb_dim=32, kernel_size=5, n_stages=4)  # noqa: E731
    prior = make_prior(sample_batch)
    g = torch.Generator().manual_seed(2)
    ncpu = os.cpu_count() or 1
    best = (None, 1)
    for nt in sorted({min(ncpu, 64), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
        torch.set_num_threads(nt)
        xp, tp = torch.randn(sample_batch, H, D), torch.full((sample_batch,), 7)
        with torch.no_grad():
            fn(xp, tp)
            t0 = time.perf_counter()
            for _ in range(2):
                fn(xp, tp)
            dt = time.perf_counter() - t0
        log(f"cpu probe: {nt} threads -> {dt / 2 * 1e3:.1f} ms / forward (B={sample_batch})")
        if best[0] is None or dt < best[0]:
            best = (dt, nt)
    torch.set_num_threads(best[1])

    def one():
        tape = lambda like: torch.randn(like.shape, generator=g)  # noqa: E731
        with torch.no_grad():
            return osamp.sample_discrete(fn, prior, tape, T=T_DIFF, steps=S_STEPS, solver="ddpm", temperature=0.5,
                                         fix_mask=mask[None], predict_noise=False)
    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return sample_batch * steps / dt, dt / steps, sample_batch


def device_timed(fn, n, dist, world, device):
    """n calls of fn bracketed by barrier + synchronize, CUDA events on the current stream, MAX over ranks (ms)."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def measure_other_configs(device, world, dist, math, reps=2):
    """BASELINE configs 3 / 4 / 5 at their per-GPU batch: every rank runs its own share (weak scaling, like the headline), one
    warm-up call (plan build, graph capture) + ``reps`` timed calls, device time, max over ranks.  Roofline: algorithmic FLOPs
    per trajectory (SURVEY 8d) against the tensor peak of the math mode."""
    from cleandiffuser_b200 import workloads
    from cleandiffuser_b200.engine import runtime
    tf32_peak, bf16_peak, src = tensor_peaks()
    peak = {"tf32": tf32_peak, "bf16": bf16_peak}.get(math)
    out = {}
    for name in ("cfg3", "cfg4", "cfg5"):
        try:
            wl = workloads.BUILDERS[name](device)
            prior, cond = wl.prior.to(device), None if wl.cond is None else wl.cond.to(device)
            B = prior.shape[0]
            before = runtime.STATS["engine_calls"]

            def call():
                return wl.sample(device, prior=prior, cond=cond)
            with torch.no_grad():
                call()
                torch.cuda.synchronize()
                ms = device_timed(call, reps, dist, world, device) / reps
            v = world * B / (ms * 1e-3)
            tfl = v * wl.gflop / 1e3 / world
            out[name] = {"workload": wl.describe, "value": v, "unit": "trajectories/s", "ms_per_call": ms, "batch_per_gpu": B,
                         "n_gpus": world, "dtype": math, "gflop_per_traj": wl.gflop, "tflops_per_gpu": tfl,
                         "roofline": {"bound": "tensor", "achieved": tfl, "peak": peak, "unit": "TFLOP/s",
                                      "frac": (tfl / peak) if peak else None, "peak_source": src},
                         "engine_calls": runtime.STATS["engine_calls"] - before}
            if wl.hbm_mb:                                # the config is HBM-bound: activations far larger than L2 between every pair of operators
                gbs = v * wl.hbm_mb / 1e3 / world
                out[name]["roofline_hbm"] = {"bound": "hbm", "alg_mb_per_traj": wl.hbm_mb, "achieved": gbs, "peak": peaks()[0],
                                             "unit": "GB/s", "frac": gbs / peaks()[0]}
            log(f"{name}: {ms:.1f} ms / call, {v:,.0f} traj/s, {tfl:.0f} TFLOP/s per GPU")
            del wl, prior, cond
            torch.cuda.empty_cache()
        except Exception as e:            # a secondary measurement must never take the headline line down
            out[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            log(f"{name}: FAILED {out[name]['error']}")
    return out


def gpu_eager_baseline(agent, prior_dev, kw, B):
    """cfg2's sample() on this GPU through the PyTorch loop of this package (the reference's algorithm step for step, ATen kernels
    launched from Python, cuDNN convs in TF32 as torch defaults): 1 warm-up + 1 timed call."""
    old = os.environ.get("CDS_BACKEND")
    os.environ["CDS_BACKEND"] = "torch"
    try:
        with torch.no_grad():
            agent.sample(prior_dev, **kw)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            agent.sample(prior_dev, **kw)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        return {"value": B / (ms * 1e-3), "unit": "trajectories/s", "ms_per_step": ms, "batch": B,
                "what": "this package's PyTorch path (CDS_BACKEND=torch): the reference's loop and modules as ATen/cuDNN/cuBLAS "
                        "launches from Python, torch default precision (cudnn.allow_tf32=True, matmul fp32)",
                "cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32),
                "matmul_allow_tf32": bool(torch.backends.cuda.matmul.allow_tf32)}
    finally:
        if old is None:
            os.environ.pop("CDS_BACKEND", None)
        else:
            os.environ["CDS_BACKEND"] = old


def dump_outputs(out_dir, arrays, budget=64_000_000, seed=0):
    """Each array -> out_dir/<name>.npy in float32.  An array larger than its share of the byte budget keeps a fixed sample
    of its rows (trajectories): the same seeded choice, in ascending order, on every run with the same arguments."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = budget // len(arrays) - 4096                              # room for the .npy header
    for name, a in arrays.items():
        a = a.float()
        n, rows = a.shape[0], max(1, share // (a[0].numel() * 4))
        if n > rows:
            keep = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:rows].sort().values
            a = a[keep]
            log(f"dump: {name} sampled to {rows} of {n} rows (seed {seed})")
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())
        log(f"dump: {os.path.join(out_dir, name + '.npy')} {tuple(a.shape)} float32")


# ------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="trajectories per GPU (default: the BASELINE config)")
    ap.add_argument("--math", default=os.environ.get("CDS_MATH", "tf32"), choices=["tf32", "bf16", "fp32"],
                    help="tf32 (default = the library default): tcgen05 kind::tf32 over fp32 activations; bf16: tcgen05 with bf16 "
                         "operands and activations; fp32: CUDA-core FMA")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--cpu-sample-batch", type=int, default=256, help="trajectories per step of the CPU arm (bounded sample)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32; trajectories beyond a 64 MB budget "
                         "are replaced by a fixed seeded sample of them), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path's samples; it does not apply to --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": WORKLOAD, "backbone": "JannerUNet1d(14,32,[1,2,2,2],k5)", "horizon": H, "dim": D,
              "solver": "ddpm", "sample_steps": S_STEPS, "batch_per_gpu": args.batch,
              "global_batch": args.batch * world, "parallelism": f"dp{world}",
              "l2": "working set (fp32 activations + 99-slot noise tape, ~1.5 GB) exceeds the 126 MB L2; no explicit flush"}

    if args.impl == "reference":
        if rank != 0:
            return
        # K timed steps after W warm-up steps as asked; a step = one full 100-step sample() on a BOUNDED sample of the batch
        # (cpu_sample_batch trajectories; the full 4096 would take ~35 s per step on these cores).  The sample size is shrunk
        # if K + W steps would not end within a few minutes.
        sb = args.cpu_sample_batch
        while sb > 32 and (args.steps + args.warmup) * (sb / 100.0) > 240:      # ~100 traj/s on 16 threads -> seconds per step
            sb //= 2
        value, sec, sb = cpu_reference_arm(args.steps, max(args.warmup, 0), sample_batch=sb)
        cores = torch.get_num_threads()
        config = dict(config, cpu_sample_batch=sb,
                      note=f"CPU arm: every step runs the full 100-step sample() on {sb} of the {args.batch} trajectories "
                           "(bounded sample; throughput in trajectories/s is batch-size independent to first order)")
        line = {"impl": "reference", "metric": "sampled trajectories/sec (H=32, 100 DDPM steps)", "value": value,
                "unit": "trajectories/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 0),
                "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": "trajectories/s", "cores": cores, "kind": "port",
                                 "sample": f"full 100-step sample() on {sb} trajectories per step (oracle port of the reference "
                                           f"algorithm, torch CPU fp32, {cores} threads)"},
                "e2e": {"value": value, "unit": "trajectories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a CUDA device"
    os.environ["CDS_BACKEND"] = "cuda"          # a silent PyTorch fallback would invalidate the number
    os.environ["CDS_MATH"] = args.math
    torch.cuda.set_device(local_rank)
    device = f"cuda:{local_rank}"
    dist = None
    saved_stdout = None
    if world > 1:
        import torch.distributed as dist
        # keep stdout to the ONE JSON line: NCCL prints its version banner to stdout when NCCL_DEBUG is set in the environment
        # (communicators are created lazily, at the first collective) -> everything written to fd 1 until the result line
        # goes to stderr instead
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        import datetime
        # a collective that has not completed within 3 minutes is a bug (the longest rank-0-only stretch is a few seconds)
        dist.init_process_group("nccl", device_id=torch.device(device), timeout=datetime.timedelta(seconds=180))

    from cleandiffuser_b200.engine import runtime
    agent, net, mask = build_agent(device)
    B = args.batch
    prior_host = make_prior(B, seed=1 + rank).pin_memory()
    prior_dev = prior_host.to(device)
    gathered = torch.empty(world * B, H, D, device=device) if world > 1 else None
    kw = dict(solver="ddpm", n_samples=B, sample_steps=S_STEPS, temperature=0.5)
    torch.manual_seed(2 + rank)
    last = {}

    def step_resident():
        x0, _ = agent.sample(prior_dev, **kw)
        if world > 1:
            dist.all_gather_into_tensor(gathered, x0)      # the one collective of the path: finished samples
        if args.dump_outputs:
            last["x0"] = x0                                # a fresh tensor per call: later calls do not overwrite it
        return x0

    def step_e2e():
        x0, _ = agent.sample(prior_host.to(device, non_blocking=True), **kw)
        if world > 1:
            dist.all_gather_into_tensor(gathered, x0)
            return gathered[rank * B:(rank + 1) * B].cpu()
        return x0.cpu()

    def timed(fn, n):
        return device_timed(fn, n, dist, world, device)

    with torch.no_grad():
        log("warm-up")
        for i in range(max(args.warmup, 3)):
            step_resident()
            torch.cuda.synchronize()
            log(f"warm-up step {i} done")
        runtime.STATS["time_loop"] = True
        runtime.STATS["loop_events"] = []
        with ClockSampler(local_rank) as clk:
            clk.wait_first()
            step_resident()                       # the sampler's first rows already see the GPU under this load
            torch.cuda.synchronize()
            row0 = len(clk.rows)
            runtime.STATS["loop_events"] = []
            ms = timed(step_resident, args.steps)
            if args.dump_outputs and rank == 0:       # copied now: the e2e steps below reuse the gather buffer
                outputs = {"x0": (gathered if world > 1 else last["x0"]).cpu()}
            row1 = len(clk.rows)
            extended = 0
            t_ext = time.time()
            while len(clk.rows) - row0 < 5 and time.time() - t_ext < 3.0:    # short timed regions: keep the same load running
                agent.sample(prior_dev, **kw)                                 # (un-timed) until a few samples exist.  NO collective
                                                                              # here: the number of extra steps differs per rank
                torch.cuda.synchronize()
                extended += 1
            clocks = clk.summary(row0, None)
            clocks["samples_inside_timed_region"] = row1 - row0
            clocks["untimed_steps_of_the_same_load_sampled_after"] = extended
        runtime.STATS["time_loop"] = False
        loop_ms = [a.elapsed_time(b) for a, b in runtime.STATS["loop_events"][:args.steps]]      # one event pair per sample() call
        loop_ms_mean = sum(loop_ms) / max(len(loop_ms), 1)
        log(f"timed: {ms / args.steps:.1f} ms/step; reverse loop alone {loop_ms_mean:.2f} ms "
            f"({loop_ms_mean * 1e3 / S_STEPS:.1f} us / iteration)")
        launches = runtime.STATS["launches"] * args.steps
        step_e2e()
        ms_e2e = timed(step_e2e, args.steps)
        log(f"e2e: {ms_e2e / args.steps:.1f} ms/step")

    value = world * B * args.steps / (ms / 1e3)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    hbm_peak, peak_src = peaks()

    # ---- live per-kernel roofline of the dominant kernel family (fused conv GEMMs: 40 of the 41 launches of an iteration) --
    roofline = None
    if rank == 0:
        plan = next(iter(agent._engine_plans.values()))
        ops = plan.program.ops
        plan.x.copy_(torch.randn_like(plan.x) * 0.5)
        stream = torch.cuda.current_stream().cuda_stream
        plan.handle.profile(50, stream, len(ops))                     # warm
        per_op = [0.0] * len(ops)
        reps = 5
        for _ in range(reps):
            for i, v in enumerate(plan.handle.profile(50, stream, len(ops))):
                per_op[i] += v / reps
        in_iter = [not (op.flags & 1) for op in ops]                  # CDS_OPF_ONCE operators are not part of the iteration
        conv_ms, conv_bytes, conv_flops, n_conv = 0.0, 0.0, 0.0, 0
        for op, t_ms, live in zip(ops, per_op, in_iter):
            if op.kind != 0 or not live:
                continue
            c = op.u.conv
            n_conv += 1
            conv_ms += t_ms
            # SURVEY 8(d) canonical accounting: every fused conv reads its input(s) and writes its output once, fp32
            conv_bytes += 4.0 * c.batch * (c.L_in * c.C_in + c.L_out * c.C_out * c.phases
                                           + (c.L_out * c.res_C if c.res_w else 0) + (c.L_out * c.C_out if c.res else 0))
            conv_flops += 2.0 * c.batch * c.L_out * c.C_out * c.phases * (c.taps * c.C_in + (c.res_C if c.res_w else 0))
        iter_ms = sum(t for t, live in zip(per_op, in_iter) if live)
        for i, (op, t_ms) in enumerate(zip(ops, per_op)):
            if op.kind == 0:
                c = op.u.conv
                log(f"op {i:2d} conv {('f32', 'bf16', 'tf32')[c.math]:4s} L {c.L_in:3d}->{c.L_out * c.phases:3d} C {c.C_in:4d}->{c.C_out:4d} "
                    f"k{c.taps} s{c.stride} gn{c.groups} res{'W' if c.res_w else ('I' if c.res else '-')}: {t_ms * 1e3:8.1f} us")
            else:
                log(f"op {i:2d} kind {op.kind}{' (once per call)' if op.flags & 1 else ''}: {t_ms * 1e3:8.1f} us")
        log(f"iteration total {iter_ms * 1e3:.1f} us (direct launches, event-bracketed)")
        share = conv_ms / iter_ms
        # the timed region replays CUDA graphs (no per-launch events possible inside): the conv kernels' time per iteration is
        # the event-timed loop time x their share of the iteration (share from the event-bracketed direct launches above;
        # the ncu launch list under profiles/ gives the same share)
        loop_iter_ms = loop_ms_mean / S_STEPS
        conv_ms_graph = loop_iter_ms * share
        achieved = conv_bytes / (conv_ms_graph * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            ent = tj.get(args.math) if isinstance(tj.get(args.math), dict) else None
            if ent:
                traffic, traffic_src = ent.get("conv_dram_bytes_per_launch"), ent.get("source")
        tf32_peak, bf16_peak, tsrc = tensor_peaks()
        tpeak = {"tf32": tf32_peak, "bf16": bf16_peak}.get(args.math)
        tfl = conv_flops / (conv_ms_graph * 1e-3) / 1e12
        roofline = {"bound": "hbm", "kernel": "conv_tc_kernel / conv_ps_kernel (fused Conv1d+GroupNorm+Mish+FiLM+residual), all "
                                              f"{n_conv} conv launches of one reverse iteration",
                    "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                    "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                    "how": "algorithmic bytes (SURVEY 8d: fp32 in+out of every fused conv) of one iteration / (event-timed graph-replay "
                           "loop time per iteration x conv share of the iteration)",
                    "launches_per_iter": n_conv, "avg_launch_us": conv_ms_graph / max(n_conv, 1) * 1e3,
                    "alg_bytes_per_launch": conv_bytes / max(n_conv, 1), "alg_bytes_per_iter": conv_bytes,
                    "conv_share_of_iter": share, "tflops_effective": tfl,
                    "tensor": {"achieved": tfl, "peak": tpeak, "unit": "TFLOP/s", "frac": (tfl / tpeak) if tpeak else None,
                               "peak_source": tsrc, "note": "nominal conv FLOPs incl. zero-padding taps"},
                    "direct_launch": {"avg_launch_us": conv_ms / max(n_conv, 1) * 1e3,
                                      "achieved": conv_bytes / (conv_ms * 1e-3) / 1e9},
                    "sample_level": {"alg_bytes_per_traj": ALG_BYTES_PER_TRAJ,
                                     "achieved_GBs": ALG_BYTES_PER_TRAJ * value / world / 1e9,
                                     "frac": ALG_BYTES_PER_TRAJ * value / world / 1e9 / hbm_peak}}

    eager = None
    if rank == 0 and world == 1 and not args.no_eager_baseline:
        try:
            eager = gpu_eager_baseline(agent, prior_dev, kw, B)
            log(f"gpu eager baseline: {eager['ms_per_step']:.0f} ms / step, {eager['value']:,.0f} traj/s")
        except Exception as e:
            eager = {"error": f"{type(e).__name__}: {e}"[:300]}

    # free cfg2's plan before the other configs build theirs
    others = None
    if not args.no_other_configs and args.math in ("tf32", "bf16"):
        for pl in list(agent._engine_plans.values()):
            pl.close()
        agent._engine_plans.clear()
        torch.cuda.empty_cache()
        others = measure_other_configs(device, world, dist, args.math)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, sec, sb = cpu_reference_arm(1, 1, sample_batch=args.cpu_sample_batch)
        cpu_baseline = {"value": v, "unit": "trajectories/s", "cores": torch.get_num_threads(), "kind": "port",
                        "sample": f"one full 100-step sample() on {sb} trajectories ({sec:.1f} s), oracle port of the "
                                  f"reference algorithm on torch CPU fp32"}

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)

    if saved_stdout is not None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if rank == 0:
        line = {"metric": "sampled trajectories/sec (H=32, 100 DDPM steps)", "value": value, "unit": "trajectories/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"fp32": "f32", "tf32": "tf32 (fp32 activations and weights in HBM, tcgen05 kind::tf32, f32 accumulate)",
                          "bf16": "bf16 operands and activations / f32 accumulate"}[args.math], "data": "synthetic",
                "config": config, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "trajectories/s", "h2d_bytes_per_step": prior_host.numel() * 4,
                        "d2h_bytes_per_step": B * H * D * 4, "ms_per_step": ms_e2e / args.steps},
                "loop_ms_per_step": loop_ms_mean, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_baseline,
                "gpu_eager_baseline": eager, "other_configs": others,
                "engine": {"calls": runtime.STATS["engine_calls"], "fallbacks": runtime.STATS["fallbacks"]}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
