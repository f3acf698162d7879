#!/usr/bin/env python3
"""A/B of the sparse-A fp32 instances (Tpp3Cfg::SA, tmpc_tpp3.cuh) against their dense twins (option dense_a = 1), in one process.

The batch is bench.py's: make_batch(spec, B, 1.0, seed=1234 + 3), device-resident, solved with the library defaults of the benchmark
(precision 32, exact-count mode with the family's band, hardest-first order).  The two arms alternate for ROUNDS rounds, the arm that
goes first alternating too.  Each arm of a round: WARMUP steps, then STEPS steps timed as one window with CUDA events (the step time),
then STEPS steps each followed by tinympc_cuda_last_pass_ms (the fp32 pass of each step, events on the launching stream; the median is
reported).  The iterates of the two arms must be identical: iter, status, x and u compared with == (+0 equals -0).
The card's name, power limit and SM clocks are read in the same run.  Prints one JSON line per arm and round and a summary line;
writes them to OUT as well when it is given.
Usage: python profiles/tools/sparse_a_ab.py [--config quadrotor|cartpole] [--batch B] [--rounds R] [--steps S] [--out FILE]"""
import argparse
import importlib
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
tm = importlib.import_module("tinympc-matlab_b200")
P = importlib.import_module("tinympc-matlab_b200.problems")

ap = argparse.ArgumentParser()
ap.add_argument("--config", default="quadrotor", choices=["quadrotor", "cartpole"])
ap.add_argument("--batch", type=int, default=1 << 20)
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--steps", type=int, default=30)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--out", default=None)
a = ap.parse_args()
assert a.rounds >= 5 and a.steps >= 20

assert torch.cuda.is_available(), "this A/B needs a CUDA device"
dev = torch.device("cuda:0")
rows = []


def emit(row):
    rows.append(row)
    print(json.dumps(row), flush=True)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()


spec = getattr(P, a.config)()
B = a.batch
b = P.make_batch(spec, B, 1.0, seed=1234 + 3)
s = tm.TinyMPC()
s.setup_from_spec(spec, devices=[0])
cs = s.cuda
cs.set_option("precision", 32)
cs.set_option("mixed", P.exact_band(spec))
cs.set_option("pass_timing", 1)
emit(dict(what="card", card=card(), config=a.config, batch=B, rounds=a.rounds, steps=a.steps, band=P.exact_band(spec)))

t = lambda v: None if v is None else torch.from_numpy(v).to(dev)
x0, Xr, Ur = t(b.x0), t(b.Xref), t(b.Uref)
ptr = lambda v: None if v is None else v.data_ptr()
stream = torch.cuda.current_stream()
outs = {}
for arm in (0, 1):
    outs[arm] = dict(x=torch.empty((B, spec.N, spec.nx), device=dev), u=torch.empty((B, spec.N - 1, spec.nu), device=dev),
                     iter=torch.empty(B, dtype=torch.int32, device=dev), status=torch.empty(B, dtype=torch.int32, device=dev))


def step(arm):
    o = outs[arm]
    cs.solve_batch_device(B, ptr(x0), ptr(Xr), ptr(Ur), ptr(o["x"]), ptr(o["u"]), ptr(o["iter"]), ptr(o["status"]), stream=stream.cuda_stream)


res = {0: dict(step=[], fp32=[]), 1: dict(step=[], fp32=[])}
kernels = {}
for r in range(a.rounds):
    for arm in ((0, 1) if r % 2 == 0 else (1, 0)):
        cs.set_option("dense_a", arm)
        for _ in range(a.warmup):
            step(arm)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(a.steps):
            step(arm)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_step = e0.elapsed_time(e1) / a.steps
        fp32 = []
        for _ in range(a.steps):
            step(arm)
            fp32.append(cs.last_pass_ms()[0])
        ms_fp32 = statistics.median(fp32)
        kernels.setdefault(arm, cs.last_kernel)
        assert cs.last_kernel == kernels[arm], (cs.last_kernel, kernels[arm])
        res[arm]["step"].append(ms_step)
        res[arm]["fp32"].append(ms_fp32)
        emit(dict(what="round", round=r, dense_a=arm, kernel=cs.last_kernel, step_ms=round(ms_step, 4), fp32_pass_ms=round(ms_fp32, 4),
                  marked=cs.last_marked, msolves_s=round(B / ms_step / 1e3, 2)))

same = {k: bool(torch.equal(outs[0][k], outs[1][k])) for k in ("iter", "status", "x", "u")}
assert all(same.values()), f"the two arms differ: {same}"


def stats(v):
    return dict(median=round(statistics.median(v), 4), min=round(min(v), 4), max=round(max(v), 4))


sm, dn = res[0], res[1]
summary = dict(what="summary", config=a.config, kernel_sparse=kernels[0], kernel_dense=kernels[1], identical=same,
               step_ms_sparse=stats(sm["step"]), step_ms_dense=stats(dn["step"]),
               fp32_ms_sparse=stats(sm["fp32"]), fp32_ms_dense=stats(dn["fp32"]),
               step_gain_pct=round(100 * (statistics.median(dn["step"]) / statistics.median(sm["step"]) - 1), 2),
               fp32_gain_pct=round(100 * (statistics.median(dn["fp32"]) / statistics.median(sm["fp32"]) - 1), 2),
               step_ranges_overlap=max(sm["step"]) >= min(dn["step"]), fp32_ranges_overlap=max(sm["fp32"]) >= min(dn["fp32"]),
               card_after=card())
emit(summary)
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text("".join(json.dumps(r) + "\n" for r in rows))
