"""Helpers of the model-session tests (tests/test_gpu_model_sessions.py): the closed loop driven on a device session and on one
reference session per solver, and a reference session whose model can be replaced between two solves.

The model arrays are built by tests/test_gpu_model_batches.py (model_of, stack, quadrotor_models); this module only adds what
sessions need on top of them."""
import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import oracle as O

ROOT = Path(__file__).resolve().parent.parent
_HOOK = None


def hook_lib():
    """The C port with port_session_set_model (tests/oracle_hooks/port_session_set_model.c), built once per process into a
    temporary directory"""
    global _HOOK
    if _HOOK is None:
        out = Path(tempfile.mkdtemp(prefix="tmpc_hook_")) / "liboracle_port_hook.so"
        subprocess.check_call(["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-I", str(ROOT / "oracle"), "-o", str(out),
                               str(ROOT / "tests" / "oracle_hooks" / "port_session_set_model.c"), "-lm", "-lpthread"])
        _HOOK = C.CDLL(str(out))
    return _HOOK


class SwapSession(O.Session):
    """oracle.Session on the C port, plus set_model: the model and cache of a live reference solver replaced between two solves"""

    def __init__(self, p):
        self.L, self.p, self.pre = hook_lib(), p, "port"
        self._keep = O._Keep()
        self._cp = O.c_problem(p, self._keep)
        fn = self.L.port_session_create
        fn.restype = C.c_void_p
        self.h = C.c_void_p(fn(C.byref(self._cp)))
        if not self.h:
            raise RuntimeError("session_create failed")

    def set_model(self, p):
        keep = O._Keep()
        cp = O.c_problem(p, keep)
        fn = self.L.port_session_set_model
        fn.restype = C.c_int
        if fn(self.h, C.byref(cp)):
            raise RuntimeError("port_session_set_model failed")
        self.p = p

    def rho(self) -> float:
        fn = self.L.port_session_rho
        fn.restype = C.c_double
        return fn(self.h)


def reference_loop(sessions, specs_at, x0, steps):
    """Closed loop {set_x0; solve; x0 = A x0 + B u0 + f} on one reference session per solver.  specs_at(t) is the list of every
    solver's spec at step t (its model for the propagation).  Returns per step: iter, status, sol_x, work_u0, the next x0 and (port
    sessions with the hook) cache->rho at exit."""
    xr = np.array(x0, np.float64)
    out = []
    for t in range(steps):
        specs = specs_at(t)
        it, st, rho = np.zeros(len(sessions), int), np.zeros(len(sessions), int), np.full(len(sessions), np.nan)
        sx = np.zeros((len(sessions),) + (specs[0].N, specs[0].nx))
        wu = np.zeros((len(sessions), specs[0].nu))
        for k, r in enumerate(sessions):
            r.set_x0(xr[k])
            g = r.solve()
            it[k], st[k], sx[k], wu[k] = g["iter"], g["status"], g["x"], g["work_u0"]
            if isinstance(r, SwapSession):
                rho[k] = r.rho()
        nxt = np.stack([p.A @ xr[k] + np.asarray(p.B).reshape(p.nx, p.nu) @ wu[k] + p.f for k, p in enumerate(specs)])
        out.append(dict(iter=it, status=st, sol_x=sx, work_u0=wu, x0=nxt, rho=rho))
        xr = nxt
    return out


SESSION_FIELDS = ("iter", "status", "sol_x", "sol_u", "x", "u", "rho", "residuals", "x0")


def read_all(ses):
    return {f: ses.read(f) for f in SESSION_FIELDS}
