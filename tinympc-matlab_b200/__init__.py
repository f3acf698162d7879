"""tinympc-matlab_b200 -- B200-native batched TinyMPC ADMM solver behind the reference's own surface.

This package holds only what the hot path needs:
  csrc/           CUDA kernels (sm_100a), the C ABI (include/tinympc_b200.h) and the host C++ mirror of the
                  reference API (tiny_setup / tiny_solve / ... + tiny_solve_batch)
  matlab/         TinyMPC.m and the MEX gateway with the new solve_batch command
  capi.py         ctypes binding of the C ABI
  problems.py     the BASELINE.json problem families and synthetic batch generators
and, below, ``TinyMPC``: a Python mirror of the MATLAB class (reference src/TinyMPC.m:1-436) with the same
method names, argument meaning and defaults, used by the tests and bench.py the way a MATLAB user uses the
original.  Every solve runs on the GPU through the C ABI; there is no CPU fallback.

Import with ``importlib.import_module("tinympc-matlab_b200")`` (the directory name is not an identifier).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .capi import CudaSolver, TinympcCudaError  # noqa: F401

__all__ = ["TinyMPC", "CudaSolver", "TinympcCudaError", "capi"]


def _dp(a):
    return a.ctypes.data_as(capi.c_dp)


def _cm(a, rows, cols):
    """math-shaped (rows, cols) array -> contiguous column-major buffer"""
    a = np.asarray(a, np.float64).reshape(rows, cols)
    return np.ascontiguousarray(a.T).ravel()


class TinyMPC:
    """Python mirror of the MATLAB ``TinyMPC`` handle class (src/TinyMPC.m).

    Differences from the original, all additive: ``solve_batch`` (the new batched entry point),
    ``set_sensitivity_matrices`` really stores the matrices (the reference MEX command is a no-op,
    src/bindings.cpp:319-361), and ``solve`` returns the true solver status next to the MATLAB-compatible 0.
    Trajectories follow MATLAB's shapes: states nx x N, controls nu x (N-1).
    """

    def __init__(self):
        # defaults of src/TinyMPC.m:24-40
        self.nx = self.nu = self.N = 0
        self.A = self.B = self.Q = self.R = None
        self.rho = 1.0
        self.is_setup = False
        self.settings = dict(abs_pri_tol=1e-4, abs_dua_tol=1e-4, max_iter=100, check_termination=1,
                             en_state_bound=False, en_input_bound=False, en_state_soc=False, en_input_soc=False,
                             en_state_linear=False, en_input_linear=False, adaptive_rho=False,
                             adaptive_rho_min=0.1, adaptive_rho_max=10.0, adaptive_rho_enable_clipping=True)
        self.x_min = self.x_max = self.u_min = self.u_max = None
        self.dK = self.dP = self.dC1 = self.dC2 = None
        self._L = None
        self._h = None
        self._cuda = None
        self._devices = None
        self.last_status = None     # true tiny_solve return value of the last solve (0 converged / 1 max_iter)

    # ------------------------------------------------------------------ setup (src/TinyMPC.m:42-104)
    def setup(self, A, B, Q, R, N, **opts):
        A, B, Q, R = (np.atleast_2d(np.asarray(m, np.float64)) for m in (A, B, Q, R))
        assert A.shape[0] == A.shape[1], "A must be square"
        assert A.shape[0] == B.shape[0], "A and B row dimensions must match"
        assert Q.shape[0] == A.shape[0], "Q must match A dimensions"
        assert R.shape[0] == B.shape[1], "R must match B column dimension"
        assert N >= 2, "N must be >= 2"
        self.nx, self.nu, self.N = A.shape[0], B.shape[1], int(N)
        self.A, self.B, self.Q, self.R = A, B, Q, R
        o = dict(rho=1.0, fdyn=None, verbose=False, abs_pri_tol=1e-4, abs_dua_tol=1e-4, max_iter=100, check_termination=1,
                 en_state_bound=False, en_input_bound=False, adaptive_rho=False, adaptive_rho_min=0.1, adaptive_rho_max=10.0,
                 adaptive_rho_enable_clipping=True)
        for k, v in opts.items():       # parse_options ignores unknown names (src/TinyMPC.m:368-376)
            if k in o:
                o[k] = v
        self.rho = float(o["rho"])
        for k in ("abs_pri_tol", "abs_dua_tol", "max_iter", "check_termination", "adaptive_rho", "adaptive_rho_min",
                  "adaptive_rho_max", "adaptive_rho_enable_clipping"):
            self.settings[k] = o[k]
        self.settings["en_state_bound"] = self.settings["en_input_bound"] = False     # only via set_bound_constraints
        fdyn = np.zeros(self.nx) if o["fdyn"] is None else np.asarray(o["fdyn"], np.float64).ravel()
        self._L = capi.load()
        if self._h:
            self._L.tinympc_host_free(self._h)
            self._h, self._cuda = None, None
        status = C.c_int(0)
        a, b, f = _cm(A, self.nx, self.nx), _cm(B, self.nx, self.nu), np.ascontiguousarray(fdyn)
        q, r = _cm(Q, self.nx, self.nx), _cm(R, self.nu, self.nu)
        h = self._L.tinympc_host_setup(_dp(a), _dp(b), _dp(f), _dp(q), _dp(r), self.rho, self.nx, self.nu, self.N,
                                       int(bool(o["verbose"])), C.byref(status))
        if status.value != 0 or not h:
            raise RuntimeError(f"TinyMPC:SetupFailed: Setup failed with status {status.value}")
        self._h = C.c_void_p(h)
        self.is_setup = True
        if self._devices:
            self._set_devices(self._devices)
        self._push_settings()

    def setup_from_spec(self, p, devices=None):
        """Convenience for tests / bench: a problems.ProblemSpec -> setup + constraints + settings, going through the
        same host C++ calls a C++ user of the reference API would make (C++ defaults, no MEX argument swap)."""
        self._devices = list(devices) if devices else None
        self.setup(p.A, np.asarray(p.B).reshape(p.nx, p.nu), np.diag(p.Qdiag), np.diag(p.Rdiag), p.N, rho=p.rho, fdyn=p.f)
        if p.x_min is not None:
            self._check(self._L.tinympc_host_set_bound_constraints(
                self._h, *(_dp(np.ascontiguousarray(b, np.float64).ravel()) for b in (p.x_min, p.x_max, p.u_min, p.u_max))))
        if len(p.Acx) or len(p.Acu):
            self._cones_raw(p.Acx, p.qcx, p.cx, p.Acu, p.qcu, p.cu)
        nsl = int(np.asarray(p.Alin_x).shape[0]) if np.asarray(p.Alin_x).size else 0
        nil = int(np.asarray(p.Alin_u).shape[0]) if np.asarray(p.Alin_u).size else 0
        if nsl or nil:
            self._linear_raw(p.Alin_x, p.blin_x, p.Alin_u, p.blin_u)
        for k in self.settings:
            self.settings[k] = getattr(p, k)
        if p.sens_mode == 1:
            self._L.tinympc_host_init_sensitivity(self._h)
        elif p.sens_mode == 2:
            self.set_sensitivity_matrices(p.dKinf, p.dPinf, p.dC1, p.dC2)
        self._push_settings()
        return self

    # ------------------------------------------------------------------ setters (src/TinyMPC.m:106-139)
    def set_x0(self, x0):
        self._check_setup()
        a = np.ascontiguousarray(np.asarray(x0, np.float64).ravel())
        self._check(self._L.tinympc_host_set_x0(self._h, _dp(a)))

    def set_x_ref(self, x_ref):
        self._check_setup()
        a = _cm(self._expand_matrix(x_ref, self.nx, self.N), self.nx, self.N)
        self._check(self._L.tinympc_host_set_x_ref(self._h, _dp(a)))

    def set_u_ref(self, u_ref):
        self._check_setup()
        a = _cm(self._expand_matrix(u_ref, self.nu, self.N - 1), self.nu, self.N - 1)
        self._check(self._L.tinympc_host_set_u_ref(self._h, _dp(a)))

    def update_settings(self, **kw):
        self._check_setup()
        for k, v in kw.items():
            if k in self.settings:
                self.settings[k] = v
        self._push_settings()

    # ------------------------------------------------------------------ solve (src/TinyMPC.m:141-157)
    def solve(self):
        """Returns 0 like the MATLAB class (src/TinyMPC.m:145-146); the real status is in ``last_status``."""
        self._check_setup()
        rc = self._L.tinympc_host_solve(self._h)
        if rc < 0:
            raise TinympcCudaError(-rc, self._L.tinympc_host_last_error(self._h).decode())
        self.last_status = rc
        return 0

    def get_solution(self):
        self._check_setup()
        x = np.zeros(self.nx * self.N)
        u = np.zeros(self.nu * (self.N - 1))
        self._L.tinympc_host_get_solution(self._h, _dp(x), _dp(u))
        return dict(states=x.reshape(self.N, self.nx).T.copy(), controls=u.reshape(self.N - 1, self.nu).T.copy())

    def get_stats(self):
        """[iter, status, primal_residual_state, primal_residual_input] of the MEX get_stats (+ duals, rho)."""
        it, st = C.c_int(0), C.c_int(0)
        res = np.zeros(5)
        self._L.tinympc_host_get_stats(self._h, C.byref(it), C.byref(st), _dp(res))
        return dict(iter=it.value, status=st.value, primal_residual_state=res[0], primal_residual_input=res[1],
                    dual_residual_state=res[2], dual_residual_input=res[3], rho=res[4])

    def work_u0(self):
        """work->u.col(0): the control the reference's closed-loop examples apply (quadrotor_hovering.cpp:91)."""
        u0 = np.zeros(self.nu)
        self._L.tinympc_host_get_work_u0(self._h, _dp(u0))
        return u0

    # ------------------------------------------------------------------ NEW: batched entry point
    def solve_batch(self, X0, Xref=None, Uref=None, x_min=None, x_max=None, u_min=None, u_max=None, models=None):
        """Solve B independent problems of this family that differ in x0 / references / bounds (cold start each).

        MATLAB shapes: X0 nx x B; Xref nx x N x B (or nx x N / nx x 1: shared, expanded like set_x_ref); Uref likewise;
        optional per-problem bounds nx x N x B / nu x (N-1) x B.  Returns dict(states nx x N x B, controls nu x (N-1) x B,
        iter B, status B, residuals 4 x B, rho B).
        models: every problem's own dynamics, costs and cache (the dict of capi.pack_models, e.g. capi.precompute_batch's
        output merged with A, B, f, Q, R, rho), as a loop of setup + solve over solvers with different models would use them;
        this object then supplies the horizon, settings and constraints only.
        """
        self._check_setup()
        X0 = np.asarray(X0, np.float64)
        if X0.ndim == 1:
            X0 = X0[:, None]
        B = X0.shape[1]
        nx, nu, N = self.nx, self.nu, self.N

        def traj(a, dim, steps):
            if a is None:
                return None
            a = np.asarray(a, np.float64)
            if a.ndim < 3:
                a = np.repeat(self._expand_matrix(a, dim, steps)[:, :, None], B, axis=2)
            assert a.shape == (dim, steps, B), f"expected {(dim, steps, B)}, got {a.shape}"
            return np.ascontiguousarray(np.transpose(a, (2, 1, 0)), np.float32)      # (B, steps, dim)

        x0 = np.ascontiguousarray(X0.T, np.float32)
        arrs = [traj(Xref, nx, N), traj(Uref, nu, N - 1), traj(x_min, nx, N), traj(x_max, nx, N), traj(u_min, nu, N - 1), traj(u_max, nu, N - 1)]
        ptr = lambda a: None if a is None else a.ctypes.data
        cin = capi.CBatchIn(B, x0.ctypes.data, *[ptr(a) for a in arrs])
        out = dict(x=np.empty((B, N, nx), np.float32), u=np.empty((B, N - 1, nu), np.float32), iter=np.empty(B, np.int32),
                   status=np.empty(B, np.int32), residuals=np.empty((B, 4), np.float32), rho=np.empty(B, np.float32))
        co = capi.CBatchOut(*[out[k].ctypes.data for k in ("x", "u", "iter", "status", "residuals", "rho")])
        if models is None:
            rc = self._L.tinympc_host_solve_batch(self._h, C.byref(cin), C.byref(co))
        else:
            arrays = capi.pack_models(models, B, nx, nu)
            rc = self._L.tinympc_host_solve_batch_models(self._h, C.byref(capi.models_struct(arrays)), C.byref(cin), C.byref(co))
        if rc:
            raise TinympcCudaError(rc, self._L.tinympc_host_last_error(self._h).decode())
        return dict(states=np.transpose(out["x"], (2, 1, 0)).astype(np.float64), controls=np.transpose(out["u"], (2, 1, 0)).astype(np.float64),
                    iter=out["iter"], status=out["status"], residuals=out["residuals"].T, rho=out["rho"])

    @property
    def cuda(self) -> CudaSolver:
        """The underlying C-ABI solver (family uploaded) for device-resident batches; owned by this object."""
        self._check_setup()
        h = self._L.tinympc_host_cuda_handle(self._h)
        if not h:
            raise TinympcCudaError(2, self._L.tinympc_host_last_error(self._h).decode() or "no CUDA device")
        if self._cuda is None or self._cuda.h.value != h:
            self._cuda = CudaSolver(borrowed_handle=h)
        self._cuda.dims = (self.nx, self.nu, self.N)
        return self._cuda

    def set_option(self, name, value):
        """precision (32 fast / 64 exact parity), chunks, ctas_per_sm, variant, force_wpp"""
        self._check_setup()
        rc = self._L.tinympc_host_set_option(self._h, name.encode(), float(value))
        if rc:
            raise TinympcCudaError(rc, self._L.tinympc_host_last_error(self._h).decode())

    # ------------------------------------------------------------------ codegen (src/TinyMPC.m:159-182)
    def codegen(self, output_dir):
        """Generate the standalone project data (tiny_data.cpp / tiny_data.hpp / tiny_main.cpp, as the reference's tiny_codegen
        writes them) plus tinympc/tiny_b200_family.h, the same solver as a constant family table of the batched C ABI."""
        self._check_setup()
        self._push_settings()
        status = self._L.tinympc_host_codegen(self._h, str(output_dir).encode(), None, None, None, None, 0)
        if status != 0:
            raise RuntimeError(f"TinyMPC:CodegenFailed: Code generation failed with status: {status}")

    def codegen_with_sensitivity(self, output_dir, dK, dP, dC1, dC2):
        self._check_setup()
        self.set_sensitivity_matrices(dK, dP, dC1, dC2)
        self._push_settings()
        arrs = [_cm(dK, self.nu, self.nx), _cm(dP, self.nx, self.nx), _cm(dC1, self.nu, self.nu), _cm(dC2, self.nx, self.nx)]
        status = self._L.tinympc_host_codegen(self._h, str(output_dir).encode(), *[_dp(a) for a in arrs], 0)
        if status != 0:
            raise RuntimeError(f"TinyMPC:CodegenWithSensitivityFailed: Code generation with sensitivity failed with status: {status}")

    # ------------------------------------------------------------------ sensitivities / cache helpers (src/TinyMPC.m:184-241)
    def set_sensitivity_matrices(self, dK, dP, dC1, dC2):
        self._check_setup()
        self._validate_sensitivity(dK, dP, dC1, dC2)
        self.dK, self.dP, self.dC1, self.dC2 = (np.asarray(m, np.float64) for m in (dK, dP, dC1, dC2))
        nx, nu = self.nx, self.nu
        self._L.tinympc_host_set_sensitivity(self._h, _dp(_cm(dK, nu, nx)), _dp(_cm(dP, nx, nx)), _dp(_cm(dC1, nu, nu)), _dp(_cm(dC2, nx, nx)))

    def compute_cache_terms(self):
        """MATLAB-side Riccati of src/TinyMPC.m:194-221 (single +rho, Pinf seeded with Q, 1e-8 regularisation)."""
        self._check_setup()
        K, P, C1, C2 = self._solve_lqr(self.rho, seed_q=True, reg=True)
        return K, P, C1, C2

    def compute_sensitivity_autograd(self):
        """Finite differences d/drho of (K, P, C1, C2), src/TinyMPC.m:223-241 (h = 1e-6)."""
        self._check_setup()
        h = 1e-6
        K0, P0, C10, C20 = self._solve_lqr(self.rho)
        K1, P1, C11, C21 = self._solve_lqr(self.rho + h)
        return (K1 - K0) / h, (P1 - P0) / h, (C11 - C10) / h, (C21 - C20) / h

    def get_cache(self):
        nx, nu = self.nx, self.nu
        bufs = dict(Kinf=np.zeros(nu * nx), Pinf=np.zeros(nx * nx), Quu_inv=np.zeros(nu * nu), AmBKt=np.zeros(nx * nx), APf=np.zeros(nx), BPf=np.zeros(nu))
        self._L.tinympc_host_get_cache(self._h, *(_dp(bufs[k]) for k in ("Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf")))
        shp = dict(Kinf=(nu, nx), Pinf=(nx, nx), Quu_inv=(nu, nu), AmBKt=(nx, nx), APf=(nx,), BPf=(nu,))
        return {k: bufs[k].reshape(shp[k], order="F") for k in bufs}

    # ------------------------------------------------------------------ constraints (src/TinyMPC.m:243-317)
    def set_linear_constraints(self, Alin_x, blin_x, Alin_u, blin_u):
        self._check_setup()
        self._linear_raw(Alin_x, blin_x, Alin_u, blin_u)
        self.settings["en_state_linear"] = np.size(Alin_x) > 0 and np.size(blin_x) > 0
        self.settings["en_input_linear"] = np.size(Alin_u) > 0 and np.size(blin_u) > 0
        self._push_settings()

    def set_bound_constraints(self, x_min, x_max, u_min, u_max):
        self._check_setup()
        self.x_min = self._expand_bounds(x_min, self.nx, self.N, -1e17)
        self.x_max = self._expand_bounds(x_max, self.nx, self.N, +1e17)
        self.u_min = self._expand_bounds(u_min, self.nu, self.N - 1, -1e17)
        self.u_max = self._expand_bounds(u_max, self.nu, self.N - 1, +1e17)
        bufs = [_cm(self.x_min, self.nx, self.N), _cm(self.x_max, self.nx, self.N), _cm(self.u_min, self.nu, self.N - 1), _cm(self.u_max, self.nu, self.N - 1)]
        self._check(self._L.tinympc_host_set_bound_constraints(self._h, *(_dp(b) for b in bufs)))
        self.settings["en_state_bound"] = self.settings["en_input_bound"] = True
        self._push_settings()

    def set_cone_constraints(self, Acx, qcx, cx, Acu, qcu, cu):
        """MATLAB order: states first, then inputs (src/TinyMPC.m:280).  The reference MEX layer forwards them to the
        core as (Acu,qcu,cu, Acx,qcx,cx) while the core's definition is state-first (SURVEY.md quirk Q3), so the INPUT
        spec lands in the workspace's state slots and vice versa; this mirror reproduces that hand-over exactly."""
        self._check_setup()
        self._cones_raw(Acu, qcu, cu, Acx, qcx, cx)      # what src/bindings.cpp:465-466 does
        self.settings["en_state_soc"] = np.size(Acx) > 0 and np.size(qcx) > 0 and np.size(cx) > 0
        self.settings["en_input_soc"] = np.size(Acu) > 0 and np.size(qcu) > 0 and np.size(cu) > 0
        self._push_settings()

    def set_equality_constraints(self, Aeq_x, beq_x, Aeq_u, beq_u):
        """Aeq x == beq as two inequalities per row (src/TinyMPC.m:296-317)."""
        Ax = bx = Au = bu = np.zeros((0, 0))
        if np.size(Aeq_x):
            Aeq_x, beq_x = np.atleast_2d(Aeq_x), np.asarray(beq_x, np.float64).ravel()
            Ax, bx = np.vstack([Aeq_x, -Aeq_x]), np.concatenate([beq_x, -beq_x])
        if np.size(Aeq_u):
            Aeq_u, beq_u = np.atleast_2d(Aeq_u), np.asarray(beq_u, np.float64).ravel()
            Au, bu = np.vstack([Aeq_u, -Aeq_u]), np.concatenate([beq_u, -beq_u])
        self.set_linear_constraints(Ax, bx, Au, bu)

    def reset(self):
        if self.is_setup:
            self._L.tinympc_host_free(self._h)
            self._h, self._cuda, self.is_setup = None, None, False

    def reset_workspace(self):
        """Back to the state tiny_setup leaves (cold start)."""
        self._check_setup()
        self._L.tinympc_host_reset_workspace(self._h)

    def __del__(self):
        try:
            self.reset()
        except Exception:
            pass

    # ------------------------------------------------------------------ private helpers
    def _check_setup(self):
        if not self.is_setup:
            raise RuntimeError("TinyMPC:NotSetup: Solver not setup. Call setup() first.")

    def _check(self, rc):
        if rc:
            raise RuntimeError(f"TinyMPC: host call failed with status {rc}")

    def _set_devices(self, devices):
        arr = (C.c_int * len(devices))(*devices)
        self._L.tinympc_host_set_devices(self._h, arr, len(devices))

    def _push_settings(self):
        s = self.settings
        self._check(self._L.tinympc_host_update_settings(
            self._h, float(s["abs_pri_tol"]), float(s["abs_dua_tol"]), int(s["max_iter"]), int(s["check_termination"]),
            int(bool(s["en_state_bound"])), int(bool(s["en_input_bound"])), int(bool(s["en_state_soc"])), int(bool(s["en_input_soc"])),
            int(bool(s["en_state_linear"])), int(bool(s["en_input_linear"])), int(bool(s["adaptive_rho"])),
            float(s["adaptive_rho_min"]), float(s["adaptive_rho_max"]), int(bool(s["adaptive_rho_enable_clipping"]))))

    def _cones_raw(self, A1, q1, c1, A2, q2, c2):
        i = lambda a: np.ascontiguousarray(np.round(np.asarray(a, np.float64)).astype(np.int32).ravel())
        d = lambda a: np.ascontiguousarray(np.asarray(a, np.float64).ravel())
        A1, q1, c1, A2, q2, c2 = i(A1), i(q1), d(c1), i(A2), i(q2), d(c2)
        ip = lambda a: a.ctypes.data_as(capi.c_ip)
        self._check(self._L.tinympc_host_set_cone_constraints(self._h, len(A1), ip(A1), ip(q1), _dp(c1), len(A2), ip(A2), ip(q2), _dp(c2)))

    def _linear_raw(self, Alin_x, blin_x, Alin_u, blin_u):
        Ax = np.atleast_2d(np.asarray(Alin_x, np.float64)) if np.size(Alin_x) else np.zeros((0, self.nx))
        Au = np.atleast_2d(np.asarray(Alin_u, np.float64)) if np.size(Alin_u) else np.zeros((0, self.nu))
        bx, bu = np.asarray(blin_x, np.float64).ravel(), np.asarray(blin_u, np.float64).ravel()
        a1 = _cm(Ax, Ax.shape[0], self.nx) if Ax.shape[0] else np.zeros(1)
        a2 = _cm(Au, Au.shape[0], self.nu) if Au.shape[0] else np.zeros(1)
        b1 = np.ascontiguousarray(bx) if bx.size else np.zeros(1)
        b2 = np.ascontiguousarray(bu) if bu.size else np.zeros(1)
        self._check(self._L.tinympc_host_set_linear_constraints(self._h, Ax.shape[0], _dp(a1), _dp(b1), Au.shape[0], _dp(a2), _dp(b2)))

    def _solve_lqr(self, rho, seed_q=False, reg=True):
        """Iterative DARE of src/TinyMPC.m:336-366 (the idare fallback branch) / :194-221."""
        Qr, Rr = self.Q + rho * np.eye(self.nx), self.R + rho * np.eye(self.nu)
        P = self.Q.copy() if seed_q else Qr.copy()
        K = np.zeros((self.nu, self.nx))
        for it in range(5000):
            Kp = K
            K = np.linalg.solve(Rr + self.B.T @ P @ self.B + (1e-8 * np.eye(self.nu) if reg else 0), self.B.T @ P @ self.A)
            P = Qr + self.A.T @ P @ (self.A - self.B @ K)
            if it > 0 and np.linalg.norm(K - Kp, 2) < 1e-10:
                break
        return K, P, np.linalg.inv(Rr + self.B.T @ P @ self.B), (self.A - self.B @ K).T

    @staticmethod
    def _expand_bounds(inp, dim, horizon, default):
        """src/TinyMPC.m:378-391"""
        if inp is None or np.size(inp) == 0:
            return default * np.ones((dim, horizon))
        a = np.asarray(inp, np.float64)
        if a.size == 1:
            return float(a) * np.ones((dim, horizon))
        if a.shape == (dim, 1) or a.shape == (dim,):
            return np.repeat(a.reshape(dim, 1), horizon, axis=1)
        if a.shape == (1, dim):
            return np.repeat(a.reshape(dim, 1), horizon, axis=1)
        return a

    @staticmethod
    def _expand_matrix(ref, dim, horizon):
        """src/TinyMPC.m:393-405"""
        a = np.asarray(ref, np.float64)
        if a.size == 1:
            return float(a) * np.ones((dim, horizon))
        if a.shape == (dim, 1) or a.shape == (dim,) or a.shape == (1, dim):
            return np.repeat(a.reshape(dim, 1), horizon, axis=1)
        return a

    def _validate_sensitivity(self, dK, dP, dC1, dC2):
        assert np.shape(dK) == (self.nu, self.nx), "dK must be nu x nx"
        assert np.shape(dP) == (self.nx, self.nx), "dP must be nx x nx"
        assert np.shape(dC1) == (self.nu, self.nu), "dC1 must be nu x nu"
        assert np.shape(dC2) == (self.nx, self.nx), "dC2 must be nx x nx"
