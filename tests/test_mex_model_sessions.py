"""The gateway's 'session_create_models' and 'session_set_models' commands (tinympc-matlab_b200/matlab/bindings.cpp) built against
the stub mex.h, driven by tests/stub_mex/mex_model_sessions_driver.cpp with two cartpole models: argument errors on the CPU, and on
the GPU the copies that carry the G2 model of examples/cartpole_example_one_solve.m take the counts of a family session of the G2
solver at every step of a closed loop, 51 at the first."""
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "tinympc-matlab_b200"


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    lib = PKG / "libtinympc_b200.so"
    if not lib.exists():
        import __graft_entry__
        __graft_entry__.build()
    exe = tmp_path_factory.mktemp("mex") / "mex_model_sessions_driver"
    srcs = [ROOT / "tests" / "stub_mex" / "mex_model_sessions_driver.cpp", PKG / "matlab" / "bindings.cpp"]
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", str(ROOT / "tests" / "stub_mex"), "-I", str(PKG / "csrc" / "host"),
                           "-I", str(ROOT / "include"), *map(str, srcs), "-o", str(exe), f"-L{PKG}", "-ltinympc_b200", f"-Wl,-rpath,{PKG}"])
    return exe


def run(exe, mode):
    out = subprocess.run([str(exe), mode], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    return out.stdout.splitlines()


def test_model_session_argument_errors_on_host(driver):
    lines = run(driver, "host")
    assert "setup_status 0" in lines
    assert lines.count("error_id TinyMPC:InvalidInput") == 2      # wrong argument count, a model array of the wrong size
    assert lines.count("error_id TinyMPC:NotInitialized") == 1    # set_models without a session
    assert lines[-1] == "host_only_done"


@pytest.mark.gpu
def test_model_session_reproduces_the_g2_closed_loop_on_gpu(driver):
    lines = run(driver, "gpu")
    counts = lambda arm, t: [int(v) for v in next(l for l in lines if l.startswith(f"{arm}_iter{t} ")).split()[1:]]
    assert counts("family", 0) == [51] * 4 and counts("models", 0)[0] == counts("models", 0)[2] == 51
    assert counts("models", 0)[1] != 51, "the second model must change the solve"
    for t in (0, 1):   # before the swap: the G2 copies of the model session follow the family session exactly
        f, m = counts("family", t), counts("models", t)
        assert m[0] == m[2] == f[0] and m[1] == m[3], (t, f, m)
    for t in (2, 3):   # after it: copies 0 and 2 carry the second model, 1 and 3 the G2 model, pairwise equal
        m = counts("models", t)
        assert m[0] == m[2] and m[1] == m[3], (t, m)
    assert lines[-1] == "sessions_done"
