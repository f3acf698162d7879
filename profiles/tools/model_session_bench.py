#!/usr/bin/env python3
"""Warm closed loops (solve + step) of quadrotor sessions: a model session whose solvers carry distinct models against the family
session, on the lane-group fp64 kernel (precision 64) and on the warp-per-problem fp32 kernel (precision 32).

One process; the arms alternate round by round; CUDA events around each timed window of `steps` closed-loop steps, after
`warm` untimed steps that bring the sessions to the warm regime.  The session calls synchronise, so the events bracket them
completely.  Prints the card's name and power limit, then one JSON line per (batch, precision, arm, round); a file named as the
last argument gets the same lines.

    model_session_bench.py [rounds] [out.jsonl]
"""
import importlib
import json
import subprocess
import sys
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
from test_gpu_model_batches import model_of, quadrotor_models  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 3
out_path = sys.argv[2] if len(sys.argv) > 2 else None
K, WARM, STEPS = 32, 3, 10

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
lines = [json.dumps(dict(card=card))]
print(lines[0], flush=True)

specs = quadrotor_models(P, k=K, seed=0)
caches = [O.get_cache(p, "port") for p in specs]
base = P.quadrotor()
bcache = O.get_cache(base, "port")
one = [model_of(p, c) for p, c in zip(specs, caches)]


def models_for(B):
    which = np.arange(B) % K                       # neighbours carry different models
    return {k: np.stack([np.asarray(one[j][k], np.float64) for j in range(K)])[which] for k in one[0]}


def make(B, prec, arm, b, models):
    s = capi.CudaSolver()
    s.set_option("precision", prec)
    s.set_family(cases.family_from_spec(base, bcache))
    ses = s.session(B, models=models if arm == "models" else None)
    ses.set_x_ref(b.Xref.astype(np.float64))
    ses.set_x0(b.x0.astype(np.float64))
    return s, ses


for B in (1 << 16, 1 << 20):
    b = P.make_batch(base, B, 0.3, seed=11)
    models = models_for(B)
    for prec in (64, 32):
        arms = {arm: make(B, prec, arm, b, models) for arm in ("family", "models")}
        for arm, (s, ses) in arms.items():
            for _ in range(WARM):
                ses.solve(); ses.step()
        for r in range(rounds):
            for arm, (s, ses) in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                iters = 0.0
                e0.record()
                for _ in range(STEPS):
                    ses.solve(); ses.step()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                iters = float(ses.read("iter").mean())       # the last step's mean count (reading is outside the window)
                line = json.dumps(dict(batch=B, precision=prec, arm=arm, round=r, kernel=s.last_kernel, steps=STEPS,
                                       ms_per_step=round(ms / STEPS, 3), solves_per_sec=round(B * STEPS / (ms / 1e3)),
                                       last_step_mean_iters=round(iters, 2)))
                lines.append(line)
                print(line, flush=True)
        for s, ses in arms.values():
            ses.close(); s.close()
        torch.cuda.synchronize()

if out_path:
    Path(out_path).write_text("\n".join(lines) + "\n")
