#!/usr/bin/env python3
"""bench.py -- headline benchmark of the batched TinyMPC ADMM hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Workload (BASELINE.json metric "MPC QP solves/sec (batched quadrotor, N=10) ...", configs[2]):
quadrotor hover nx=12 nu=4 N=10, 2^20 independent problems PER GPU with per-problem x0 and
per-problem full Xref/Uref arrays, box constraints, tol 1e-3, max_iter 100 (SURVEY.md section 8d C3).
One "step" = one pass of the hot path over the whole batch.  Multi-GPU = the batch sharded by
problem index, one process per GPU, no collective on the data path ("weak" scaling: 2^20 per GPU).

Printed JSON line (rank 0):
  value      solves/s, whole job, inputs/outputs resident in HBM, CUDA-event timed, max over ranks
  e2e        the same through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside)
  roofline   FP32 CUDA-core roofline of the solve kernel (the bounding one, SURVEY 8d) + HBM fraction
  cpu_baseline  the reference C++ solver (oracle/_ref) looped over a bounded prefix of the same batch
--impl reference times that CPU reference as the main line instead.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# algorithmic work per ADMM iteration / bytes per solve, SURVEY.md section 8d (box constraints)
def flops_per_iter(n, m, N, spec=None):
    """SURVEY 8d: box-only count, plus -- when `spec` enables them -- the per-family terms of the same table: 6 flop per trajectory
    element of every enabled cone / linear family, ~20 per (step, cone), 4 dim + 2 per (step, linear row), and the structured
    adaptive-rho evaluation every 5th iteration."""
    F = (N - 1) * (4 * n * n + 8 * n * m + 2 * m * m + 5 * n + 3 * m) + 15 * (n * N + m * (N - 1)) + (2 * n * n + 3 * n)
    if spec is not None:
        if spec.en_state_soc and len(spec.qcx):
            F += 6 * n * N + 20 * N * len(spec.qcx)
        if spec.en_input_soc and len(spec.qcu):
            F += 6 * m * (N - 1) + 20 * (N - 1) * len(spec.qcu)
        if spec.en_state_linear:
            F += 6 * n * N + (4 * n + 2) * N * len(spec.blin_x)
        if spec.en_input_linear:
            F += 6 * m * (N - 1) + (4 * m + 2) * (N - 1) * len(spec.blin_u)
        if spec.adaptive_rho:
            F += ((N - 1) * (4 * n * n + 4 * n * m) + 2 * n * n + 12 * (n * N + m * (N - 1))) // 5
    return F


def bytes_per_solve(n, m, N):
    return 4 * (n + n * N + m * (N - 1)) + 4 * (n * N + m * (N - 1)) + 8


DUMP_PROBLEMS = 1 << 16      # --dump-outputs sample: 2^16 problems of the largest shape (quadrotor) are 41 MB of float32
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, outputs, B):
    """Writes the per-problem outputs of a step (dict name -> device tensor with the problem index first) as
    out_dir/<name>.npy in float32, restricted to a fixed sample of the batch: every problem up to DUMP_PROBLEMS, otherwise
    DUMP_PROBLEMS indices drawn with seed 0, in increasing order.  Iteration counts and status codes are exact in float32."""
    import torch
    if B <= DUMP_PROBLEMS:
        idx = np.arange(B)
    else:
        idx = np.sort(np.random.default_rng(0).choice(B, DUMP_PROBLEMS, replace=False))
    arrays = {}
    for name, t in outputs.items():
        arrays[name] = t[torch.from_numpy(idx).to(t.device)].to(torch.float32).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}"
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


def fp32_peak_tflops():
    """FP32 CUDA-core peak: measured by profiles/microbench/ffma_bench.cu on this pool (see
    profiles/microbench/RESULTS.md); MEASURED_PEAKS.json carries no FP32 figure."""
    f = ROOT / "profiles" / "microbench" / "fp32_peak.json"
    if f.exists():
        d = json.loads(f.read_text())
        return float(d["fp32_tflops"]), d.get("how", "measured FFMA micro-benchmark")
    return 148 * 128 * 2 * 1.965e9 / 1e12, "nominal 148 SM x 128 lanes x 2 x 1.965 GHz (no measurement file)"


def hbm_peak_gbs():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.t = index, [], threading.Event(), None

    def _nvml_handle(self):
        """NVML handle of the CUDA device `index` (by UUID, so that CUDA_VISIBLE_DEVICES remapping does not matter); None -> fall
        back to spawning nvidia-smi (100 ms per sample instead of 0.1 ms)."""
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(self.index).uuid))
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            return pynvml, h
        except Exception:
            return None

    def _run_nvml(self, pynvml, h):
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        bits = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
        while not self.stop_flag.is_set():
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append([str(sm), str(mx)] + ["Active" if (r & b) else "Not Active" for _, b in bits])
            except Exception:
                pass
            self.stop_flag.wait(0.005)

    def _run(self):
        if self.nv is not None:
            return self._run_nvml(*self.nv)
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([t.strip() for t in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def __enter__(self):
        self.nv = self._nvml_handle()       # NVML initialisation (~0.1 s) happens here, before the timed region
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop_flag.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no_samples"]}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = []
        for k, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(s[2 + k].lower().startswith("active") for s in self.samples):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons, "samples": len(sm)}


def bind_to_gpu_cpus(local):
    """Pin this rank (and the pinned host buffers it is about to allocate: first touch) to the CPUs next to its GPU, so that the
    end-to-end path of every rank crosses its own PCIe root instead of the socket interconnect.  Returns the previous affinity
    (restored before the CPU baseline, which uses all host threads) and a note for the report."""
    prev = os.sched_getaffinity(0)
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(local).uuid))
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        now = os.sched_getaffinity(0)
        return prev, f"gpu-local ({len(now)} of {len(prev)} cpus)"
    except Exception as ex:
        return prev, f"unchanged ({type(ex).__name__})"


def reference_arm(args, P, spec, batch_np, build="ref"):
    """The reference's own CPU implementation (oracle/_ref = unmodified reference C++ built by
    oracle/Makefile; falls back to the C port) on all host threads, bounded sample per step.  build: "ref" (-O3 -DNDEBUG, the
    reference's Release flags) or "ref_O2" (-O2, asserts on: the second row BASELINE.md section 3 asks for)."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import oracle as O
    kind = "reference" if O.available(build) else "port"
    impl = build if kind == "reference" else "port"
    if kind == "port" and not O.available("port"):
        subprocess.check_call(["make", "-C", str(ROOT / "oracle"), "liboracle_port.so"])
    cores = os.cpu_count() or 1
    # probe to size the sample at ~ args.cpu_seconds per step
    probe = batch_np.slice(0, min(batch_np.size, 64 * cores))
    t0 = time.perf_counter(); O.solve_batch(spec, probe, impl, cores); dt = time.perf_counter() - t0
    rate = probe.size / max(dt, 1e-6)
    n = int(min(batch_np.size, max(probe.size, rate * args.cpu_seconds)))
    sample = batch_np.slice(0, n)
    for _ in range(min(args.warmup, 1)):
        O.solve_batch(spec, sample, impl, cores)
    t0 = time.perf_counter()
    iters = 0
    for _ in range(args.steps_cpu):
        r = O.solve_batch(spec, sample, impl, cores)
        iters += int(r["iter"].sum())
    dt = time.perf_counter() - t0
    sps = n * args.steps_cpu / dt
    return dict(value=sps, unit="solves/s", cores=cores, kind=kind,
                sample=f"first {n} problems of the same batch x {args.steps_cpu} passes, {cores} threads, cold start per problem",
                ns_per_admm_iter=dt * 1e9 / max(iters, 1), ms_per_step=dt * 1e3 / args.steps_cpu, mean_iters=iters / (n * args.steps_cpu))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20, help="problems per GPU")
    ap.add_argument("--scale", type=float, default=1.0, help="difficulty of the synthetic batch (SURVEY 8d: 0.3 easy, 1.0 hard)")
    ap.add_argument("--config", default="quadrotor", choices=["quadrotor", "cartpole", "rocket", "quadrotor_adaptive"])
    ap.add_argument("--precision", type=int, default=0, help="32 / 64; 0 = the family's parity-exact default (fp32 exact-count mode; fp64 under adaptive rho)")
    ap.add_argument("--mixed", type=float, default=-1.0,
                    help="relative band of the exact-count mode (fp32 pass + fp64 re-solve of the problems whose termination decision is "
                         "within the band of a tolerance); -1 = the family's measured band (default: the mode that reproduces the "
                         "reference's iteration counts), 0 = plain fp32")
    ap.add_argument("--fixer-sms", dest="fixer_sms", type=int, default=-2,
                    help="exact-count mode: SMs left to the concurrent fp64 consumer (0 = 13 %% of the device, -1 = always the sequential two-pass "
                         "form, -2 = library default: two-pass form on the device, concurrent pair inside the streamed host pipeline)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch problems per GPU; strong: --batch problems in total, split by problem index over the GPUs "
                         "(BASELINE config 3 as worded: 1M problems sharded across 8 B200)")
    ap.add_argument("--parity-n", dest="parity_n", type=int, default=10000, help="problems of the parity gate (prefix of rank 0's shard)")
    ap.add_argument("--variant", type=int, default=0, help="kernel variant (0 = default; A/B baselines 1, 2, 5)")
    ap.add_argument("--cpu-seconds", dest="cpu_seconds", type=float, default=8.0)
    ap.add_argument("--steps-cpu", dest="steps_cpu", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--order", type=int, default=-1, help="option order of the library (claim the hardest problems first); -1 = library default (1), 0 = index order")
    ap.add_argument("--e2e-mode", dest="e2e_mode", default="compact", choices=["compact", "full"],
                    help="I/O mode of the headline end-to-end number (the other one is reported as e2e_other)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write x, u, iter and status of the last one as DIR/<name>.npy (float32) for a fixed sample "
                         f"of at most {DUMP_PROBLEMS} problems of rank 0's shard, so that two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3   # timing rule: at least 3 warm-up steps

    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
        # rank 0 prints exactly one JSON line: NCCL writes its version banner to stdout at every level from VERSION up (WARN included),
        # so unless somebody asked for INFO / TRACE output, its log goes to the null device
        os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", os.devnull)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    P = importlib.import_module("tinympc-matlab_b200.problems")
    spec = dict(quadrotor=P.quadrotor, cartpole=P.cartpole, rocket=P.rocket,
                quadrotor_adaptive=lambda: P.quadrotor(adaptive=True))[args.config]()
    n, m, N = spec.nx, spec.nu, spec.N
    if args.precision == 0:
        args.precision = P.exact_precision(spec) if args.mixed < 0 else 32
    world_cfg = max(world, args.gpus)      # the reference arm runs on rank 0 alone but describes the same job
    if args.scaling == "strong":
        assert args.batch % world_cfg == 0, "--scaling strong needs --batch divisible by the number of GPUs"
        per_gpu = args.batch // world_cfg
    else:
        per_gpu = args.batch
    workload = f"{args.config} nx={n} nu={m} N={N}, {per_gpu} problems/GPU, per-problem x0+Xref+Uref, box constraints, " \
               f"tol {spec.abs_pri_tol:g}, max_iter {spec.max_iter}, difficulty scale {args.scale}"
    # identical in both arms (the driver compares the dicts); run-specific facts go to the top-level "run" key
    config = {"workload": workload, "batch_per_gpu": per_gpu, "scale": args.scale,
              "l2_policy": "inputs+outputs per step (%.0f MB) exceed the 126 MB L2" % (bytes_per_solve(n, m, N) * per_gpu / 1e6),
              "parallelism": f"problem-index shards x{world_cfg}, no collective",
              "e2e_io": ("compact: x0 + one reference state per problem in (the config's Xref is that state replicated over the horizon; "
                         "none for a reference-free config), u0 + iter + status out; the full-trajectory mode is reported as e2e_other; "
                         "a config whose references vary over the horizon has only the full mode") if args.e2e_mode == "compact" else
                        "full: x0 + Xref + Uref in, x + u + iter + status out"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        batch_np = P.make_batch(spec, min(per_gpu, 1 << 18), args.scale, seed=1234 + 3)
        args.steps_cpu = max(1, args.steps)
        cb = reference_arm(args, P, spec, batch_np)
        line = {"impl": "reference", "metric": "solves_per_sec", "value": cb["value"], "unit": "solves/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "ns_per_admm_iter": cb["ns_per_admm_iter"], "mean_iters": cb["mean_iters"],
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    run = {}
    prev_affinity, run["cpu_affinity"] = bind_to_gpu_cpus(local) if (world > 1 and not os.environ.get("BENCH_NO_AFFINITY")) else (os.sched_getaffinity(0), "unchanged (single rank)")
    tm = importlib.import_module("tinympc-matlab_b200")
    S = importlib.import_module("tinympc-matlab_b200.sharding")
    B = per_gpu
    # the job is world*B problems (weak: B = --batch; strong: B = --batch / world), rank r owns the contiguous index range [lo, hi)
    lo, hi = S.shard_range(world * B, rank, world)
    assert hi - lo == B
    batch_np = P.make_batch(spec, B, args.scale, seed=1234 + 3 + 1000 * rank)   # each rank generates its own shard
    solver = tm.TinyMPC()
    solver.setup_from_spec(spec, devices=[local])
    solver.cuda.set_option("precision", args.precision)
    solver.cuda.set_option("variant", args.variant)
    band = P.exact_band(spec) if args.mixed < 0 else args.mixed
    if args.precision == 64:
        band = 0.0
    solver.cuda.set_option("mixed", band)
    solver.cuda.set_option("fixer_sms", args.fixer_sms)
    if args.order >= 0:
        solver.cuda.set_option("order", args.order)
    run["order"] = "library default (hardest first)" if args.order < 0 else ("hardest first" if args.order else "index order")
    run["fixer_sms"] = args.fixer_sms
    run["mixed_band"] = band
    run["e2e_mode"] = args.e2e_mode
    run["mode"] = "fp64" if args.precision == 64 else (f"exact-count: fp32 pass + fp64 re-solve of the problems within {band:g} of a tolerance" if band > 0 else "plain fp32")

    tdev = lambda a: None if a is None else torch.from_numpy(a).to(dev)
    x0, Xref, Uref = tdev(batch_np.x0), tdev(batch_np.Xref), tdev(batch_np.Uref)
    x = torch.empty((B, N, n), device=dev); u = torch.empty((B, N - 1, m), device=dev)
    it = torch.empty(B, dtype=torch.int32, device=dev); st = torch.empty(B, dtype=torch.int32, device=dev)
    ptr = lambda a: None if a is None else a.data_ptr()
    stream = torch.cuda.current_stream()

    def step():
        solver.cuda.solve_batch_device(B, ptr(x0), ptr(Xref), ptr(Uref), ptr(x), ptr(u), ptr(it), ptr(st), stream=stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    solver.cuda.set_option("pass_timing", 1)     # CUDA events around the two passes of the exact-count mode, on the launching stream
    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = solver.cuda.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record(stream)
        for _ in range(args.steps):
            step()
        e1.record(stream)
        barrier()
    ms = e0.elapsed_time(e1)
    kernel_of_step = solver.cuda.last_kernel         # the e2e runs below go through other pipelines
    pass_ms = solver.cuda.last_pass_ms() if (band > 0 and args.precision == 32) else None   # (fp32 pass, fp64 pass) of the last timed step
    launches = solver.cuda.launch_count - launches0
    marked = solver.cuda.last_marked if band > 0 else 0
    iters_one = int(it.sum().item())                 # identical every step (same inputs)
    unsolved = float((st == 11).float().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"x": x, "u": u, "iter": it, "status": st}, B)
    ms_all, (iters_all, launches_all) = S.reduce_report(ms, [iters_one, launches], dist, dev)   # max of times, sum of work
    launches_all = int(launches_all)
    value = world * B * args.steps / (ms_all * 1e-3)
    ns_iter = ms_all * 1e6 / (iters_all * args.steps)

    # ---- the same resident step with compact I/O (device pointers: one reference state per problem in, first control out): what
    # the kernels cost when they neither read a replicated reference nor write trajectories -- the floor of the compact e2e mode
    resident_compact = None
    const_ref = batch_np.Xref is None or bool((batch_np.Xref == batch_np.Xref[:, :1]).all())
    if const_ref and (batch_np.Uref is None or not batch_np.Uref.any()):
        xc_dev = None if Xref is None else Xref[:, 0, :].contiguous()
        u0_dev = torch.empty((B, m), device=dev)
        it_c = torch.empty_like(it); st_c = torch.empty_like(st)

        def step_c():
            solver.cuda.solve_batch_device(B, ptr(x0), None, None, None, None, ptr(it_c), ptr(st_c), xref_const=ptr(xc_dev), u0=ptr(u0_dev),
                                           stream=stream.cuda_stream)
        for _ in range(2):
            step_c()
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kc = max(1, args.steps // 2)
        c0.record(stream)
        for _ in range(kc):
            step_c()
        c1.record(stream)
        barrier()
        ms_c = S.reduce_report(c0.elapsed_time(c1), [0], dist, dev)[0]
        assert torch.equal(it_c, it) and torch.equal(u0_dev, u[:, 0, :]), "compact device path and full device path disagree"
        resident_compact = {"value": world * B * kc / (ms_c * 1e-3), "unit": "solves/s", "ms_per_step": ms_c / kc, "kernel": solver.cuda.last_kernel,
                            "io": "device-resident, x0" + ("" if xc_dev is None else " + one reference state per problem") + " in, u0 + iter + status out"}

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, copies inside the timed region), two I/O modes:
    #   full    : what the reference-shaped interface moves -- x0, full Xref (nx x N), full Uref in; full x, u, iter, status out
    #   compact : x0 + ONE reference state per problem (xref_const: config 3 replicates its set point over the horizon) in;
    #             first control u0 + iter + status out (tinympc_cuda_batch_in::xref_const, tinympc_cuda_batch_out::u0)
    # `e2e` (the headline) is the mode --e2e-mode names; the other one is reported next to it.
    e2e = None
    e2e_other = None
    if not args.no_e2e:
        pin = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        npv = lambda t: None if t is None else t.numpy()
        kk = max(1, args.steps // 2)
        ipin = lambda: torch.empty(B, dtype=torch.int32).pin_memory().numpy()

        def timed(call):
            call()                                                  # warm-up (allocations)
            barrier()
            t0 = time.perf_counter()
            for _ in range(kk):
                call()
            barrier()
            tt = torch.tensor([time.perf_counter() - t0], device=dev)
            if dist is not None:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        def run_full():
            hx0, hXr, hUr = pin(batch_np.x0), pin(batch_np.Xref), pin(batch_np.Uref)
            hout = dict(x=torch.empty((B, N, n)).pin_memory().numpy(), u=torch.empty((B, N - 1, m)).pin_memory().numpy(), iter=ipin(), status=ipin())
            dt = timed(lambda: solver.cuda.solve_batch(npv(hx0), npv(hXr), npv(hUr), out=hout))
            assert np.array_equal(hout["iter"], it.cpu().numpy()), "host-buffer path and device path disagree"
            h2d = 4 * (B * n + (B * N * n if hXr is not None else 0) + (B * (N - 1) * m if hUr is not None else 0))
            d2h = 4 * (B * N * n + B * (N - 1) * m) + 8 * B
            return {"value": world * B * kk / dt, "unit": "solves/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": dt * 1e3 / kk,
                    "io": "full: x0 + Xref[nx x N] + Uref[nu x (N-1)] in, x + u + iter + status out", "pipeline": solver.cuda.last_timing()}

        def run_compact():
            const_ref = batch_np.Xref is None or bool((batch_np.Xref == batch_np.Xref[:, :1]).all())
            zero_uref = batch_np.Uref is None or not batch_np.Uref.any()
            if not (const_ref and zero_uref):
                return None            # the config's references vary over the horizon: no compact form
            hx0, hxc = pin(batch_np.x0), (None if batch_np.Xref is None else pin(batch_np.Xref[:, 0, :]))
            hout = dict(u0=torch.empty((B, m)).pin_memory().numpy(), iter=ipin(), status=ipin())
            dt = timed(lambda: solver.cuda.solve_batch(npv(hx0), xref_const=npv(hxc), out=hout, compact_out=True))
            assert np.array_equal(hout["iter"], it.cpu().numpy()), "compact host path and device path disagree"
            assert np.array_equal(hout["u0"], u[:, 0, :].cpu().numpy()), "compact host path returns a different first control"
            return {"value": world * B * kk / dt, "unit": "solves/s", "h2d_bytes_per_step": 4 * B * n * (1 if hxc is None else 2), "d2h_bytes_per_step": 4 * B * m + 8 * B,
                    "ms_per_step": dt * 1e3 / kk,
                    "io": "compact: x0" + ("" if hxc is None else " + one reference state per problem") + " in, u0 + iter + status out",
                    "pipeline": solver.cuda.last_timing()}

        full, compact = run_full(), run_compact()
        if args.e2e_mode == "compact" and compact is not None:
            e2e, e2e_other = compact, full
        else:
            e2e, e2e_other = full, compact

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- parity gate (SURVEY 8d): the first parity_n problems of this very run against the reference C++ on the same inputs
    parity = None
    if args.parity_n > 0:
        try:
            sys.path.insert(0, str(ROOT / "oracle"))
            import oracle as O
            pimpl = "ref" if O.available("ref") else "port"
            npar = min(B, args.parity_n)
            g = O.solve_batch(spec, batch_np.slice(0, npar), pimpl, os.cpu_count() or 1)
            rx, ru = x[:npar].cpu().numpy(), u[:npar].cpu().numpy()
            ri, rs = it[:npar].cpu().numpy(), st[:npar].cpu().numpy()
            same = (ri == g["iter"]) & (rs == g["status"])
            parity = {"n": npar, "oracle": "reference C++ (oracle/_ref)" if pimpl == "ref" else "C port (oracle/tinympc_oracle.c)",
                      "count_mismatch": int((ri != g["iter"]).sum()), "status_mismatch": int((rs != g["status"]).sum()),
                      "max_abs_dx": float(np.abs(rx - g["x"]).max()), "max_abs_du": float(np.abs(ru - g["u"]).max()),
                      # a problem that never converges (status 11 at max_iter) keeps making large steps, so rounding differences
                      # are not damped the way they are on a converging one: report the two groups separately
                      "max_abs_dxu_converged": float(max(np.abs(rx - g["x"])[g["status"] == 1].max(initial=0), np.abs(ru - g["u"])[g["status"] == 1].max(initial=0))),
                      "max_abs_dxu_at_max_iter": float(max(np.abs(rx - g["x"])[g["status"] != 1].max(initial=0), np.abs(ru - g["u"])[g["status"] != 1].max(initial=0))),
                      "max_abs_dx_matched": float(np.abs(rx[same] - g["x"][same]).max()) if same.any() else None,
                      "max_abs_du_matched": float(np.abs(ru[same] - g["u"][same]).max()) if same.any() else None,
                      "tolerance": "identical iter/status; |dx|, |du| <= 1e-4 absolute (north_star)", "mode": run["mode"]}
            parity["pass"] = bool(parity["count_mismatch"] == 0 and parity["status_mismatch"] == 0 and
                                  parity["max_abs_dx"] <= 1e-4 and parity["max_abs_du"] <= 1e-4)
        except Exception as ex:
            parity = {"n": 0, "error": repr(ex)}

    F = flops_per_iter(n, m, N, spec)
    peak_tf, peak_how = fp32_peak_tflops()
    hbm_pk, hbm_how = hbm_peak_gbs()
    # The dominant kernel: the only one of a plain step; in the exact-count mode the fp32 pass (its duration measured live with CUDA
    # events on the launching stream, tinympc_cuda_last_pass_ms), which executes the iterations of every problem -- a marked problem
    # is iterated up to the check that marks it -- i.e. the algorithmic flops of the whole batch.  The fp64 pass is reported beside it.
    t_step = ms / args.steps * 1e-3
    t_launch = pass_ms[0] * 1e-3 if pass_ms else t_step
    ach_tf = F * iters_one / t_launch / 1e12
    ach_gbs = bytes_per_solve(n, m, N) * B / t_launch / 1e9
    roof = {"bound": "fp32_cuda_core", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
            "traffic": None, "peak_source": peak_how, "flops_per_admm_iter": F, "kernel": kernel_of_step.split("+")[0].split("|")[0],
            "kernel_ms": t_launch * 1e3, "step_ms": t_step * 1e3, "step_kernels": kernel_of_step,
            "frac_of_whole_step": F * iters_one / t_step / 1e12 / peak_tf,
            "fp64_pass_ms": pass_ms[1] if pass_ms else None,
            "hbm": {"achieved": ach_gbs, "peak": hbm_pk, "unit": "GB/s", "frac": ach_gbs / hbm_pk, "peak_source": hbm_how,
                    "bytes_per_solve": bytes_per_solve(n, m, N)}}
    # DRAM traffic of the same kernel on the same workload from the committed `ncu --set full` capture
    # (profiles/r01/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum per launch)
    for prof in (ROOT / "profiles" / "r02" / "traffic.json", ROOT / "profiles" / "r01" / "traffic.json"):
        if not prof.exists() or roof["traffic"] is not None:
            continue
        for key, t in json.loads(prof.read_text()).items():
            if key.startswith(f"{args.config}_b{B}_s{args.scale:g}") and t.get("kernel") == roof["kernel"]:
                roof["traffic"] = t["dram_bytes_per_launch"]
                roof["traffic_algorithmic"] = bytes_per_solve(n, m, N) * B

    line = {"metric": "solves_per_sec", "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_all / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32" if args.precision == 32 else "f64", "data": "synthetic", "config": config,
            "ns_per_admm_iter": ns_iter, "mean_iters": iters_all / (world * B), "unsolved_frac": unsolved,
            "clocks": clk.summary(), "e2e": e2e, "fp64_resolved": int(marked), "gpu_launches": launches_all, "roofline": roof,
            "e2e_other": e2e_other, "resident_compact": resident_compact, "parity": parity, "run": run}
    if not args.no_cpu_baseline:
        os.sched_setaffinity(0, prev_affinity)
        try:
            cb = reference_arm(args, P, spec, batch_np.slice(0, min(B, 1 << 18)))
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "ns_per_admm_iter")}
            line["cpu_baseline"]["flags"] = "-O3 -DNDEBUG (the reference's Release build)"
            import oracle as O
            if O.available("ref_O2"):      # BASELINE.md section 3: the same sources at -O2
                half = argparse.Namespace(**{**vars(args), "cpu_seconds": args.cpu_seconds / 2, "steps_cpu": 1, "warmup": 0})
                cb2 = reference_arm(half, P, spec, batch_np.slice(0, min(B, 1 << 17)), build="ref_O2")
                line["cpu_baseline_O2"] = {**{k: cb2[k] for k in ("value", "unit", "cores", "kind", "sample", "ns_per_admm_iter")}, "flags": "-O2"}
        except Exception as ex:  # the checker is optional for the GPU number, never the other way round
            line["cpu_baseline"] = {"value": None, "unit": "solves/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(ex)}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
