#!/usr/bin/env python3
"""Outputs of the host entry tinympc_cuda_precompute_batch on seeded inputs, for comparing two builds bit for bit.

    precompute_dump.py dump <repo root> <out.npz>     run the library of that tree, write every output array
    precompute_dump.py compare <a.npz> <b.npz>        print one line per array: bit-identical or the largest difference

Inputs: 4096 perturbed models of each of cartpole, quadrotor and rocket (dynamics by 1 %, costs by 0.5 .. 2, rho by 0.5 .. 2, as
tests/test_gpu_precompute.py perturbs them) and of a random shape with nu > nx (2 states, 3 inputs), with the sensitivities.
"""
import importlib
import sys
from pathlib import Path

import numpy as np


def inputs(P, family, n=4096):
    rng = np.random.default_rng(1234)
    if family == "wide":
        nx, nu = 2, 3
        A = np.eye(nx)[None] + 0.1 * rng.standard_normal((n, nx, nx))
        return A, rng.standard_normal((n, nx, nu)), rng.uniform(1, 2, (n, nx)), rng.uniform(1, 2, (n, nu)), rng.uniform(0.5, 2, n), \
            0.1 * rng.standard_normal((n, nx))
    p = getattr(P, family)()
    A = p.A[None] * (1.0 + 0.01 * rng.standard_normal((n,) + p.A.shape))
    B = np.asarray(p.B).reshape(p.nx, p.nu)[None] * (1.0 + 0.01 * rng.standard_normal((n, p.nx, p.nu)))
    rho = p.rho * rng.uniform(0.5, 2.0, n)
    Q = p.Qdiag[None] * rng.uniform(0.5, 2.0, (n, p.nx)) + rho[:, None]
    R = p.Rdiag[None] * rng.uniform(0.5, 2.0, (n, p.nu)) + rho[:, None]
    return A, B, Q, R, rho, np.broadcast_to(np.asarray(p.f, np.float64).ravel(), (n, p.nx)).copy()


def dump(root, out):
    sys.path.insert(0, str(Path(root).resolve()))
    P = importlib.import_module("tinympc-matlab_b200.problems")
    capi = importlib.import_module("tinympc-matlab_b200.capi")
    res = {}
    for fam in ("cartpole", "quadrotor", "rocket", "wide"):
        A, B, Q, R, rho, f = inputs(P, fam)
        for k, v in capi.precompute_batch(A, B, Q, R, rho, f, sensitivities=True).items():
            res[f"{fam}/{k}"] = v
    np.savez(out, **res)


def compare(a, b):
    x, y = np.load(a), np.load(b)
    same = 0
    for k in sorted(set(x.files) | set(y.files)):
        if k not in x.files or k not in y.files:
            print(f"{k}: only in one file")
        elif x[k].tobytes() == y[k].tobytes():
            same += 1
            print(f"{k}: bit-identical {x[k].shape}")
        else:
            print(f"{k}: DIFFERS, max |a - b| = {np.abs(x[k].astype(np.float64) - y[k]).max():.3e}")
    print(f"{same} of {len(set(x.files) | set(y.files))} arrays bit-identical")
    return 0 if same == len(set(x.files) | set(y.files)) else 1


if __name__ == "__main__":
    if sys.argv[1] == "dump":
        dump(sys.argv[2], sys.argv[3])
    else:
        sys.exit(compare(sys.argv[2], sys.argv[3]))
