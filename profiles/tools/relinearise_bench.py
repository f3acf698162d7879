#!/usr/bin/env python3
"""A relinearised closed loop of fp64 quadrotor model sessions, fed through the host entries and through the device entries.

Every step: torch forms A_k, B_k of every solver on the GPU from its current state (row i of the nominal A and B scaled with
1 + 0.05 tanh(x_i)), the cache is computed, the session gets the new models, solves and steps.
  host path:   x0 read to the host, A_k / B_k copied to the host, tinympc_cuda_precompute_batch (host arrays), session_set_models
               (host arrays);
  device path: read_device, tinympc_cuda_precompute_batch_device writing straight into the model arrays, session_set_models_device.
Phases are timed with a host clock around work that ends in torch.cuda.synchronize(); the precompute kernel alone with CUDA events
around tinympc_cuda_precompute_batch_device on the default stream.  The two paths alternate round by round in one process, each
with its own session, after one untimed warm-up step.  Prints the card's name and power limit, then one JSON line per (batch, path,
round); a file named as the last argument gets the same lines.

    relinearise_bench.py [rounds] [out.jsonl]
"""
import ctypes as C
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
sys.path.insert(0, str(ROOT / "oracle"))
sys.path.insert(0, str(ROOT / "tests"))
P = importlib.import_module("tinympc-matlab_b200.problems")
capi = importlib.import_module("tinympc-matlab_b200.capi")
import cases  # noqa: E402
import oracle as O  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
out_path = sys.argv[2] if len(sys.argv) > 2 else None
STEPS = 3

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
lines = [json.dumps(dict(card=card))]
print(lines[0], flush=True)

base = P.quadrotor()
nx, nu = base.nx, base.nu
CACHE = ("Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf")
f64 = dict(dtype=torch.float64, device="cuda")


class Loop:
    """one session and its model arrays (column-major per solver); `path` selects the entries that feed it"""

    def __init__(self, B, path, b, Qm, Rm, rho):
        self.B, self.path = B, path
        self.s = capi.CudaSolver()
        self.s.set_option("precision", 64)
        self.s.set_family(cases.family_from_spec(base, O.get_cache(base, "port")))
        self.A0 = torch.tensor(base.A, **f64)
        self.B0 = torch.tensor(np.asarray(base.B).reshape(nx, nu), **f64)
        self.T = dict(Adyn=torch.empty((B, nx, nx), **f64), Bdyn=torch.empty((B, nu, nx), **f64), Q=Qm.clone(), R=Rm.clone(),
                      rho=rho.clone(), Kinf=torch.empty((B, nx, nu), **f64), Pinf=torch.empty((B, nx, nx), **f64),
                      Quu_inv=torch.empty((B, nu, nu), **f64), AmBKt=torch.empty((B, nx, nx), **f64), APf=torch.empty((B, nx), **f64),
                      BPf=torch.empty((B, nu), **f64))
        self.dp = {k: v.data_ptr() for k, v in self.T.items()}
        if path == "host":   # pinned host copies of the model arrays
            self.H = {k: torch.empty(v.shape, dtype=torch.float64, pin_memory=True) for k, v in self.T.items()}
            for k in ("Q", "R", "rho"):
                self.H[k].copy_(self.T[k])
            self.hp = {k: v.data_ptr() for k, v in self.H.items()}
        self.x = torch.tensor(b.x0.astype(np.float64), **f64)
        self.form()
        self.cache(timed=False)
        self.ses = self.s.session(B, models_device=self.dp)
        self.ses.set_x_ref(b.Xref.astype(np.float64))
        self.ses.write_device("x0", self.x.data_ptr())
        torch.cuda.synchronize()

    def form(self):
        g = 1.0 + 0.05 * torch.tanh(self.x)[:, :, None]
        self.T["Adyn"].copy_((self.A0 * g).transpose(1, 2))
        self.T["Bdyn"].copy_((self.B0 * g).transpose(1, 2))

    def cache(self, timed=True):
        if self.path == "device":
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            capi.precompute_batch_device(self.B, nx, nu, self.dp["Adyn"], self.dp["Bdyn"], self.dp["Q"], self.dp["R"], self.dp["rho"],
                                         {k: self.dp[k] for k in CACHE})
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)
        self.H["Adyn"].copy_(self.T["Adyn"]); self.H["Bdyn"].copy_(self.T["Bdyn"])
        dp = lambda k: C.cast(C.c_void_p(self.hp[k]), capi.c_dp)
        cin = capi.CPrecomputeIn(self.B, nx, nu, dp("Adyn"), dp("Bdyn"), None, dp("Q"), dp("R"), dp("rho"))
        co = capi.CPrecomputeOut(*[dp(k) for k in CACHE], None, None, None, None, None)
        assert capi.load().tinympc_cuda_precompute_batch(C.byref(cin), C.byref(co)) == 0
        if not timed:    # set-up: the device arrays get the same cache
            for k in CACHE:
                self.T[k].copy_(self.H[k])
        return None

    def set_models(self):
        if self.path == "device":
            self.ses.set_models_device(self.dp)
        else:
            self.s._check(self.s.L.tinympc_cuda_session_set_models(self.ses.h, C.byref(capi.models_struct(self.hp))))

    def read_x(self):
        if self.path == "device":
            self.ses.read_device("x0", self.x.data_ptr())
        else:
            self.x.copy_(torch.from_numpy(self.ses.read("x0")))

    def step(self):
        t, kern = {}, None

        def phase(name, fn):
            nonlocal kern
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            t[name] = (time.perf_counter() - t0) * 1e3
            if name == "precompute":
                kern = r

        phase("read_x", self.read_x)
        phase("form", self.form)
        phase("precompute", self.cache)
        phase("set_models", self.set_models)
        phase("solve", self.ses.solve)
        phase("step", self.ses.step)
        return t, kern


for B in (1 << 16, 1 << 20):
    rng = np.random.default_rng(5)
    b = P.make_batch(base, B, 0.3, seed=11)
    rho = base.rho * rng.uniform(0.5, 2.0, B)
    Qm = torch.tensor(base.Qdiag * rng.uniform(0.5, 2.0, (B, nx)) + rho[:, None], **f64)
    Rm = torch.tensor(base.Rdiag * rng.uniform(0.5, 2.0, (B, nu)) + rho[:, None], **f64)
    loops = {path: Loop(B, path, b, Qm, Rm, torch.tensor(rho, **f64)) for path in ("host", "device")}
    for lp in loops.values():
        lp.step()                                   # warm-up
    for r in range(rounds):
        for path, lp in loops.items():
            acc, kms = [], []
            for _ in range(STEPS):
                t, k = lp.step()
                acc.append(t)
                if k is not None:
                    kms.append(k)
            ms = {k: round(float(np.mean([a[k] for a in acc])), 3) for k in acc[0]}
            line = dict(batch=B, path=path, round=r, steps=STEPS, kernel=lp.s.last_kernel, ms_per_step=ms,
                        total_ms_per_step=round(sum(ms.values()), 3), last_step_mean_iters=round(float(lp.ses.read("iter").mean()), 2))
            if kms:
                line["precompute_kernel_ms"] = round(float(np.mean(kms)), 3)
            lines.append(json.dumps(line))
            print(lines[-1], flush=True)
    for lp in loops.values():
        lp.ses.close(); lp.s.close()
    del loops
    torch.cuda.synchronize()

if out_path:
    Path(out_path).write_text("\n".join(lines) + "\n")
