"""The gateway's 'solve_batch_models' command (tinympc-matlab_b200/matlab/bindings.cpp) built against the stub mex.h, driven by
tests/stub_mex/mex_models_driver.cpp with two cartpole models: argument errors on the CPU, and on the GPU the problems that carry
the G2 model of examples/cartpole_example_one_solve.m reproduce its 51 iterations."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import cases

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "tinympc-matlab_b200"


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    lib = PKG / "libtinympc_b200.so"
    if not lib.exists():
        import __graft_entry__
        __graft_entry__.build()
    exe = tmp_path_factory.mktemp("mex") / "mex_models_driver"
    srcs = [ROOT / "tests" / "stub_mex" / "mex_models_driver.cpp", PKG / "matlab" / "bindings.cpp"]
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", str(ROOT / "tests" / "stub_mex"), "-I", str(PKG / "csrc" / "host"),
                           "-I", str(ROOT / "include"), *map(str, srcs), "-o", str(exe), f"-L{PKG}", "-ltinympc_b200", f"-Wl,-rpath,{PKG}"])
    return exe


def run(exe, mode):
    out = subprocess.run([str(exe), mode], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout.splitlines()


def test_solve_batch_models_argument_errors_on_host(driver):
    lines = run(driver, "host")
    assert "setup_status 0" in lines
    assert lines.count("error_id TinyMPC:InvalidInput") == 2      # wrong argument count, a model array of the wrong size
    assert lines[-1] == "host_only_done"


@pytest.mark.gpu
def test_solve_batch_models_reproduces_the_g2_example_on_gpu(driver):
    lines = run(driver, "gpu")
    assert "error_id TinyMPC:SolveBatchFailed" in lines           # Kinf missing: the library's EINVAL
    it = [int(v) for v in next(l for l in lines if l.startswith("models_iter")).split()[1:]]
    st = [int(v) for v in next(l for l in lines if l.startswith("models_status")).split()[1:]]
    u0 = [float(v) for v in next(l for l in lines if l.startswith("models_u0")).split()[1:]]
    _, _, g = cases.load("G2_cartpole_ubound")
    assert it[0] == it[2] == 51 and st[0] == st[2] == 1
    assert abs(u0[0] - g["u"][0, 0, 0]) < 1e-6 and u0[0] == u0[2]
    assert it[1] == it[3] and u0[1] == u0[3] and (it[1], u0[1]) != (it[0], u0[0]), "the second model must change the solve"
    assert lines[-1] == "models_done"
