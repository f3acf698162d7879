"""The C ABI of model batches (tinympc_cuda_models, tinympc_cuda_solve_batch_models[_device]) without a GPU: the Python mirror of the
struct has the C layout, the entry points are exported, and without a device every call fails instead of falling back."""
import ctypes
import importlib
import subprocess
from pathlib import Path

import numpy as np
import pytest

import cases

ROOT = Path(__file__).resolve().parents[1]
FIELDS = ["Adyn", "Bdyn", "fdyn", "Q", "R", "rho", "Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf", "dKinf_drho", "dPinf_drho"]


@pytest.fixture(scope="module")
def tm():
    return importlib.import_module("tinympc-matlab_b200")


def test_models_struct_layout_matches_the_header(tm, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "tinympc_b200.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(tinympc_cuda_models));\n'
                   + "".join(f'    printf("%zu\\n", offsetof(tinympc_cuda_models, {f}));\n' for f in FIELDS) + "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-I", str(ROOT / "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    C = tm.capi.CModels
    assert got == [ctypes.sizeof(C)] + [getattr(C, f).offset for f in FIELDS]
    assert [f for f, _ in C._fields_] == FIELDS


def test_model_entry_points_are_exported(tm):
    out = subprocess.check_output(["nm", "-D", "--defined-only", str(tm.capi.LIB_PATH)], text=True)
    syms = {line.split()[-1] for line in out.splitlines() if line.strip()}
    for name in ("tinympc_cuda_solve_batch_models", "tinympc_cuda_solve_batch_models_device", "tiny_solve_batch_models",
                 "tinympc_host_solve_batch_models"):
        assert name in syms, name


def test_pack_models_writes_column_major_chunks(tm):
    rng = np.random.default_rng(0)
    B, nx, nu = 3, 4, 2
    m = dict(A=rng.standard_normal((B, nx, nx)), B=rng.standard_normal((B, nx, nu)), Q=rng.random((B, nx)), R=rng.random((B, nu)),
             rho=rng.random(B), Kinf=rng.standard_normal((B, nu, nx)))
    a = tm.capi.pack_models(m, B, nx, nu)
    assert set(a) == {"Adyn", "Bdyn", "Q", "R", "rho", "Kinf"}
    for b in range(B):
        assert np.array_equal(a["Bdyn"][b].ravel(), m["B"][b].ravel(order="F"))
        assert np.array_equal(a["Kinf"][b].ravel(), m["Kinf"][b].ravel(order="F"))
    with pytest.raises(ValueError):
        tm.capi.pack_models(dict(A=np.zeros((B, nx, nu))), B, nx, nu)


def test_no_cpu_fallback_for_model_batches_without_gpu(tm):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = tm.capi.load()
    assert L.tinympc_cuda_device_count() == 0
    with pytest.raises(tm.TinympcCudaError) as e:
        tm.CudaSolver()
    assert e.value.code == 2          # ENODEVICE
    p = cases.P.cartpole()
    s = tm.TinyMPC()
    s.setup_from_spec(p)
    B = 4
    models = dict(A=np.repeat(p.A[None], B, 0), B=np.repeat(np.asarray(p.B).reshape(p.nx, p.nu)[None], B, 0),
                  Q=np.repeat((p.Qdiag + p.rho)[None], B, 0), R=np.repeat((p.Rdiag + p.rho)[None], B, 0), rho=np.full(B, p.rho),
                  Kinf=np.zeros((B, p.nu, p.nx)), Pinf=np.zeros((B, p.nx, p.nx)), Quu_inv=np.zeros((B, p.nu, p.nu)),
                  AmBKt=np.zeros((B, p.nx, p.nx)))
    with pytest.raises(tm.TinympcCudaError) as e:
        s.solve_batch(np.zeros((p.nx, B)), models=models)
    assert e.value.code == 2
