#!/usr/bin/env python3
"""Model batches (tinympc_cuda_solve_batch_models) against family batches on one GPU: 2^20 quadrotor problems, every one with its
own model (B scaled as by a +-30 % mass / inertia change, Q, R diagonals and rho scaled by factors in [0.5, 2]; caches from the
batched precompute), device-resident inputs, CUDA events around each call, two warm-up calls per path, the two paths of a pair
alternated REPS times on the same x0 / Xref / Uref.  The model arrays are 4 712 bytes per problem, 4.9 GB in all: far more than the
126 MB of L2, so every problem's model comes from HBM.  Pairs:
  fp64: the model form of the lane-group kernel against the family's lane-group kernel (the cost of per-problem coefficients)
  fp32: the model form of the warp-per-problem kernel against the family's (option force_wpp)
The host entry end to end is NOT measured: it is computed from sizes (the model upload at a stated PCIe rate).
Writes one JSON line per pair (and a header line with the card) to stdout, and to the file OUT when it is given.
Usage: python profiles/tools/model_batch_bench.py [B] [OUT]"""
import importlib
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
tm = importlib.import_module("tinympc-matlab_b200")
P = importlib.import_module("tinympc-matlab_b200.problems")
capi = tm.capi

B = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
OUT = Path(sys.argv[2]) if len(sys.argv) > 2 else None
REPS = 5
CHUNK = 1 << 16
PCIE_GBPS = 50.0     # sustained H2D of a PCIe Gen5 x16 link with pinned buffers, for the computed host-entry figure

assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
spec = P.quadrotor()
nx, nu, N = spec.nx, spec.nu, spec.N
rows = [dict(what="card", card=card, batch=B)]
print(json.dumps(rows[0]), flush=True)

# ---- per-problem models, built chunk by chunk straight into device arrays (column-major per problem, capi.pack_models' layout)
rng = np.random.default_rng(0)
A0, B0 = np.asarray(spec.A, np.float64), np.asarray(spec.B, np.float64).reshape(nx, nu)
dm = {}
t_pre = 0.0
for c0 in range(0, B, CHUNK):
    n = min(CHUNK, B - c0)
    mass, inertia = rng.uniform(0.7, 1.3, n), rng.uniform(0.7, 1.3, n)
    Bm = np.repeat(B0[None], n, 0)
    Bm[:, [0, 1, 2, 6, 7, 8]] /= mass[:, None, None]
    Bm[:, [3, 4, 5, 9, 10, 11]] /= inertia[:, None, None]
    Qd = spec.Qdiag * rng.uniform(0.5, 2.0, (n, nx))
    Rd = spec.Rdiag * rng.uniform(0.5, 2.0, (n, nu))
    rho = spec.rho * rng.uniform(0.5, 2.0, n)
    A = np.repeat(A0[None], n, 0)
    f = np.repeat(np.asarray(spec.f, np.float64)[None], n, 0)
    t0 = time.perf_counter()
    pc = capi.precompute_batch(A, Bm, Qd + rho[:, None], Rd + rho[:, None], rho, f)    # tiny_setup's Q + rho (SURVEY quirk Q1)
    t_pre += time.perf_counter() - t0
    m = dict(A=A, B=Bm, f=f, Q=Qd + rho[:, None], R=Rd + rho[:, None], rho=rho, Kinf=pc["Kinf"], Pinf=pc["Pinf"], Quu_inv=pc["Quu_inv"],
             AmBKt=pc["AmBKt"], APf=pc["APf"], BPf=pc["BPf"])
    for field, a in capi.pack_models(m, n, nx, nu).items():
        if field not in dm:
            dm[field] = torch.empty((B,) + a.shape[1:], dtype=torch.float64, device=dev)
        dm[field][c0:c0 + n].copy_(torch.from_numpy(a))
model_bytes = sum(v[0].numel() * 8 for v in dm.values())
ptrs = {k: v.data_ptr() for k, v in dm.items()}

b = P.make_batch(spec, B, 1.0, seed=7)
t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
x0, Xr, Ur = t(b.x0), t(b.Xref), t(b.Uref)
x = torch.empty((B, N, nx), device=dev); u = torch.empty((B, N - 1, nu), device=dev)
it = torch.empty(B, dtype=torch.int32, device=dev); st = torch.empty(B, dtype=torch.int32, device=dev)
stream = torch.cuda.current_stream().cuda_stream


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


for prec, force in ((64, 0), (32, 1)):
    s = tm.TinyMPC()
    s.setup_from_spec(spec, devices=[0])
    cu = s.cuda
    cu.set_option("precision", prec)
    cu.set_option("force_wpp", force)
    fam = lambda: cu.solve_batch_device(B, x0.data_ptr(), Xr.data_ptr(), Ur.data_ptr(), x.data_ptr(), u.data_ptr(), it.data_ptr(),
                                        st.data_ptr(), stream=stream)
    mdl = lambda: cu.solve_batch_models_device(ptrs, B, x0.data_ptr(), Xr.data_ptr(), Ur.data_ptr(), x.data_ptr(), u.data_ptr(),
                                               it.data_ptr(), st.data_ptr(), stream=stream)
    res = {}
    for name, fn in (("family", fam), ("models", mdl)):
        for _ in range(2):
            timed(fn)
        res[name] = dict(kernel=cu.last_kernel, mean_iter=float(it.double().mean().item()), ms=[])
    for _ in range(REPS):
        for name, fn in (("family", fam), ("models", mdl)):
            res[name]["ms"].append(round(timed(fn), 3))
    row = dict(what=f"fp{prec}", card=card, batch=B)
    for name, r in res.items():
        med = float(np.median(r["ms"]))
        row[name] = dict(kernel=r["kernel"], ms=r["ms"], median_ms=med, mean_iter=round(r["mean_iter"], 3),
                         solves_per_s=round(B / med * 1e3), ns_per_problem_iteration=round(med * 1e6 / (B * r["mean_iter"]), 4))
    row["model_over_family_per_iteration"] = round(row["models"]["ns_per_problem_iteration"] / row["family"]["ns_per_problem_iteration"], 4)
    rows.append(row)
    print(json.dumps(row), flush=True)
    del s

rows.append(dict(what="host_entry", card=card, batch=B, measured=False, model_bytes_per_problem=model_bytes,
                 model_upload_gb=round(model_bytes * B / 1e9, 3), computed_upload_ms_at_pcie=round(model_bytes * B / (PCIE_GBPS * 1e9) * 1e3, 1),
                 pcie_gbps_assumed=PCIE_GBPS, precompute_s_measured=round(t_pre, 2)))
print(json.dumps(rows[-1]), flush=True)
if OUT is not None:
    OUT.parent.mkdir(parents=True, exist_ok=True)
    OUT.write_text("".join(json.dumps(r) + "\n" for r in rows))
