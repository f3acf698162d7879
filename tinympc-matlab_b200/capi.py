"""ctypes binding of the C ABI in include/tinympc_b200.h (libtinympc_b200.so, built in-tree).

This is plumbing only: it marshals numpy / torch buffers into the plain-pointer structs of the C ABI.
All solver arithmetic happens in the CUDA library; if the library is missing or no CUDA device is
usable the calls raise -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB_PATH = HERE / "libtinympc_b200.so"

c_dp = C.POINTER(C.c_double)
c_fp = C.POINTER(C.c_float)
c_ip = C.POINTER(C.c_int)

ERRORS = {1: "EINVAL", 2: "ENODEVICE", 3: "ECUDA", 4: "EUNSUPPORTED", 5: "ENOTREADY"}

HOST_EXPORTS = [
    "tinympc_host_setup", "tinympc_host_free", "tinympc_host_set_bound_constraints", "tinympc_host_set_cone_constraints",
    "tinympc_host_set_linear_constraints", "tinympc_host_update_settings", "tinympc_host_set_x0", "tinympc_host_set_x_ref",
    "tinympc_host_set_u_ref", "tinympc_host_solve", "tinympc_host_get_solution", "tinympc_host_get_stats", "tinympc_host_get_cache",
    "tinympc_host_set_cache_terms", "tinympc_host_init_sensitivity", "tinympc_host_set_sensitivity", "tinympc_host_reset_workspace",
    "tinympc_host_solve_batch", "tinympc_host_solve_batch_models", "tinympc_host_set_devices", "tinympc_host_set_option", "tinympc_host_cuda_handle", "tinympc_host_codegen",
    "tiny_codegen", "tiny_codegen_with_sensitivity",
    # the C++ API mirror itself (extern "C" names of the reference, tiny_api.hpp:10-50)
    "tiny_setup", "tiny_set_bound_constraints", "tiny_set_cone_constraints", "tiny_set_linear_constraints",
    "tiny_precompute_and_set_cache", "tiny_solve", "tiny_update_settings", "tiny_set_default_settings", "tiny_set_x0",
    "tiny_set_x_ref", "tiny_set_u_ref", "tiny_initialize_sensitivity_matrices", "tiny_solve_batch",
]

EXPORTS = [
    "tinympc_cuda_create", "tinympc_cuda_destroy", "tinympc_cuda_set_family", "tinympc_cuda_solve_batch",
    "tinympc_cuda_solve_batch_device", "tinympc_cuda_solve_workspace", "tinympc_cuda_set_option", "tinympc_cuda_device_count", "tinympc_cuda_num_devices",
    "tinympc_cuda_last_kernel", "tinympc_cuda_launch_count", "tinympc_cuda_last_timing", "tinympc_cuda_last_pass_ms", "tinympc_cuda_last_marked", "tinympc_cuda_plan_compact_chunks", "tinympc_cuda_last_error",
    "tinympc_cuda_version", "tinympc_cuda_host_alloc", "tinympc_cuda_host_free",
    "tinympc_cuda_session_create", "tinympc_cuda_session_destroy", "tinympc_cuda_session_set_x0", "tinympc_cuda_session_set_x_ref",
    "tinympc_cuda_session_set_u_ref", "tinympc_cuda_session_solve", "tinympc_cuda_session_step", "tinympc_cuda_session_read",
    "tinympc_cuda_precompute_batch", "tinympc_cuda_solve_batch_models", "tinympc_cuda_solve_batch_models_device",
]


class TinympcCudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"tinympc_cuda error {ERRORS.get(code, code)}: {msg}")
        self.code = code


class CFamily(C.Structure):
    _fields_ = [
        ("nx", C.c_int), ("nu", C.c_int), ("N", C.c_int),
        ("Adyn", c_dp), ("Bdyn", c_dp), ("fdyn", c_dp), ("Q", c_dp), ("R", c_dp),
        ("rho", C.c_double),
        ("Kinf", c_dp), ("Pinf", c_dp), ("Quu_inv", c_dp), ("AmBKt", c_dp), ("APf", c_dp), ("BPf", c_dp),
        ("dKinf_drho", c_dp), ("dPinf_drho", c_dp),
        ("abs_pri_tol", C.c_double), ("abs_dua_tol", C.c_double),
        ("max_iter", C.c_int), ("check_termination", C.c_int),
        ("en_state_bound", C.c_int), ("en_input_bound", C.c_int), ("en_state_soc", C.c_int), ("en_input_soc", C.c_int),
        ("en_state_linear", C.c_int), ("en_input_linear", C.c_int),
        ("adaptive_rho", C.c_int), ("adaptive_rho_min", C.c_double), ("adaptive_rho_max", C.c_double),
        ("adaptive_rho_enable_clipping", C.c_int),
        ("x_min", c_dp), ("x_max", c_dp), ("u_min", c_dp), ("u_max", c_dp),
        ("numStateCones", C.c_int), ("numInputCones", C.c_int),
        ("Acx", c_ip), ("qcx", c_ip), ("cx", c_dp), ("Acu", c_ip), ("qcu", c_ip), ("cu", c_dp),
        ("numStateLinear", C.c_int), ("numInputLinear", C.c_int),
        ("Alin_x", c_dp), ("blin_x", c_dp), ("Alin_u", c_dp), ("blin_u", c_dp),
    ]


class CBatchIn(C.Structure):
    _fields_ = [("batch", C.c_int), ("x0", C.c_void_p), ("Xref", C.c_void_p), ("Uref", C.c_void_p),
                ("x_min", C.c_void_p), ("x_max", C.c_void_p), ("u_min", C.c_void_p), ("u_max", C.c_void_p), ("xref_const", C.c_void_p)]


class CBatchOut(C.Structure):
    _fields_ = [("x", C.c_void_p), ("u", C.c_void_p), ("iter", C.c_void_p), ("status", C.c_void_p),
                ("residuals", C.c_void_p), ("rho", C.c_void_p), ("u0", C.c_void_p)]


class CModels(C.Structure):
    """tinympc_cuda_models: per-problem model arrays, double, one column-major chunk per problem"""
    _fields_ = [("Adyn", C.c_void_p), ("Bdyn", C.c_void_p), ("fdyn", C.c_void_p), ("Q", C.c_void_p), ("R", C.c_void_p), ("rho", C.c_void_p),
                ("Kinf", C.c_void_p), ("Pinf", C.c_void_p), ("Quu_inv", C.c_void_p), ("AmBKt", C.c_void_p), ("APf", C.c_void_p), ("BPf", C.c_void_p),
                ("dKinf_drho", C.c_void_p), ("dPinf_drho", C.c_void_p)]


# models dict key -> (CModels field, math shape per problem given (nx, nu)); matrices are stored column-major per problem
MODEL_FIELDS = (("A", "Adyn", lambda nx, nu: (nx, nx)), ("B", "Bdyn", lambda nx, nu: (nx, nu)), ("f", "fdyn", lambda nx, nu: (nx,)),
                ("Q", "Q", lambda nx, nu: (nx,)), ("R", "R", lambda nx, nu: (nu,)), ("rho", "rho", lambda nx, nu: ()),
                ("Kinf", "Kinf", lambda nx, nu: (nu, nx)), ("Pinf", "Pinf", lambda nx, nu: (nx, nx)), ("Quu_inv", "Quu_inv", lambda nx, nu: (nu, nu)),
                ("AmBKt", "AmBKt", lambda nx, nu: (nx, nx)), ("APf", "APf", lambda nx, nu: (nx,)), ("BPf", "BPf", lambda nx, nu: (nu,)),
                ("dKinf", "dKinf_drho", lambda nx, nu: (nu, nx)), ("dPinf", "dPinf_drho", lambda nx, nu: (nx, nx)))


def pack_models(models: dict, batch: int, nx: int, nu: int) -> dict:
    """Math-shaped per-problem models -> the column-major float64 arrays of tinympc_cuda_models.

    models: A (B, nx, nx), B (B, nx, nu), f (B, nx), Q (B, nx), R (B, nu) (work->Q / work->R: diagonal + rho), rho (B,), Kinf (B, nu, nx),
    Pinf (B, nx, nx), Quu_inv (B, nu, nu), AmBKt (B, nx, nx), APf (B, nx), BPf (B, nu), dKinf, dPinf (adaptive rho) -- the shapes
    precompute_batch returns, so its output merges in directly.  Keys that are absent or None stay NULL.  Returns {CModels field: array}."""
    out = {}
    for key, field, shape in MODEL_FIELDS:
        a = models.get(key)
        if a is None:
            continue
        a = np.asarray(a, np.float64)
        want = (batch,) + shape(nx, nu)
        if a.shape != want:
            raise ValueError(f"models[{key!r}]: expected shape {want}, got {a.shape}")
        out[field] = np.ascontiguousarray(np.swapaxes(a, 1, 2) if a.ndim == 3 else a)
    return out


def models_struct(arrays: dict) -> CModels:
    """CModels over host numpy arrays (pack_models) or device pointers (ints)"""
    m = CModels()
    for field, a in arrays.items():
        setattr(m, field, a if isinstance(a, int) else a.ctypes.data)
    return m


class CPrecomputeIn(C.Structure):
    _fields_ = [("batch", C.c_int), ("nx", C.c_int), ("nu", C.c_int), ("Adyn", c_dp), ("Bdyn", c_dp), ("fdyn", c_dp), ("Q", c_dp), ("R", c_dp), ("rho", c_dp)]


class CPrecomputeOut(C.Structure):
    _fields_ = [("Kinf", c_dp), ("Pinf", c_dp), ("Quu_inv", c_dp), ("AmBKt", c_dp), ("APf", c_dp), ("BPf", c_dp),
                ("dKinf_drho", c_dp), ("dPinf_drho", c_dp), ("dC1_drho", c_dp), ("dC2_drho", c_dp), ("iters", c_ip)]


_lib = None


def precompute_batch(A, B, Q, R, rho, f=None, sensitivities=False) -> dict:
    """Batched tiny_precompute_and_set_cache on the GPU (tinympc_cuda_precompute_batch): A (n, nx, nx), B (n, nx, nu), Q (n, nx),
    R (n, nu) diagonals, rho (n,), optional f (n, nx).  Returns math-shaped arrays Kinf (n, nu, nx), Pinf (n, nx, nx), Quu_inv,
    AmBKt, APf, BPf, iters (+ dKinf, dPinf, dC1, dC2 with sensitivities=True)."""
    L = load()
    A = np.asarray(A, np.float64); Bm = np.asarray(B, np.float64)
    n, nx, nu = A.shape[0], A.shape[1], Bm.shape[2]
    cm = lambda a: np.ascontiguousarray(np.swapaxes(a, 1, 2))          # per-problem column-major
    a_, b_ = cm(A), cm(Bm)
    q_, r_ = np.ascontiguousarray(Q, np.float64), np.ascontiguousarray(R, np.float64)
    rho_ = np.ascontiguousarray(np.broadcast_to(np.asarray(rho, np.float64), (n,)))
    f_ = None if f is None else np.ascontiguousarray(f, np.float64)
    dp = lambda a: None if a is None else a.ctypes.data_as(c_dp)
    cin = CPrecomputeIn(n, nx, nu, dp(a_), dp(b_), dp(f_), dp(q_), dp(r_), dp(rho_))
    o = dict(Kinf=np.empty((n, nx, nu)), Pinf=np.empty((n, nx, nx)), Quu_inv=np.empty((n, nu, nu)), AmBKt=np.empty((n, nx, nx)),
             APf=np.empty((n, nx)), BPf=np.empty((n, nu)), iters=np.empty(n, np.int32))
    if sensitivities:
        o.update(dKinf=np.empty((n, nx, nu)), dPinf=np.empty((n, nx, nx)), dC1=np.empty((n, nu, nu)), dC2=np.empty((n, nx, nx)))
    co = CPrecomputeOut(dp(o["Kinf"]), dp(o["Pinf"]), dp(o["Quu_inv"]), dp(o["AmBKt"]), dp(o["APf"]), dp(o["BPf"]),
                        dp(o.get("dKinf")), dp(o.get("dPinf")), dp(o.get("dC1")), dp(o.get("dC2")), o["iters"].ctypes.data_as(c_ip))
    rc = L.tinympc_cuda_precompute_batch(C.byref(cin), C.byref(co))
    if rc:
        raise TinympcCudaError(rc, "tinympc_cuda_precompute_batch failed")
    # the C ABI returns column-major (rows x cols) chunks: as (cols, rows) C arrays -> transpose to math shape
    for k in ("Kinf", "Pinf", "Quu_inv", "AmBKt", "dKinf", "dPinf", "dC1", "dC2"):
        if k in o:
            o[k] = np.ascontiguousarray(np.swapaxes(o[k], 1, 2))
    return o


def load():
    """Load the in-tree CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise FileNotFoundError(f"{LIB_PATH} not built: run `python tinympc-matlab_b200/build.py` (or __graft_entry__.build())")
        L = C.CDLL(str(LIB_PATH))
        L.tinympc_cuda_create.argtypes = [C.POINTER(C.c_void_p), c_ip, C.c_int]
        L.tinympc_cuda_destroy.argtypes = [C.c_void_p]
        L.tinympc_cuda_set_family.argtypes = [C.c_void_p, C.POINTER(CFamily)]
        L.tinympc_cuda_solve_batch.argtypes = [C.c_void_p, C.POINTER(CBatchIn), C.POINTER(CBatchOut)]
        L.tinympc_cuda_solve_batch_device.argtypes = [C.c_void_p, C.c_int, C.POINTER(CBatchIn), C.POINTER(CBatchOut), C.c_void_p]
        L.tinympc_cuda_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_double]
        L.tinympc_cuda_num_devices.argtypes = [C.c_void_p]
        L.tinympc_cuda_last_kernel.argtypes = [C.c_void_p]
        L.tinympc_cuda_last_kernel.restype = C.c_char_p
        L.tinympc_cuda_launch_count.argtypes = [C.c_void_p]
        L.tinympc_cuda_launch_count.restype = C.c_longlong
        L.tinympc_cuda_last_timing.argtypes = [C.c_void_p, c_dp]
        L.tinympc_cuda_last_pass_ms.argtypes = [C.c_void_p, c_dp]
        L.tinympc_cuda_last_pass_ms.restype = C.c_int
        L.tinympc_cuda_last_marked.argtypes = [C.c_void_p]
        L.tinympc_cuda_last_marked.restype = C.c_longlong
        L.tinympc_cuda_plan_compact_chunks.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]
        L.tinympc_cuda_plan_compact_chunks.restype = C.c_int
        L.tinympc_cuda_last_error.argtypes = [C.c_void_p]
        L.tinympc_cuda_last_error.restype = C.c_char_p
        L.tinympc_cuda_version.restype = C.c_char_p
        L.tinympc_cuda_host_alloc.argtypes = [C.c_size_t]
        L.tinympc_cuda_host_alloc.restype = C.c_void_p
        L.tinympc_cuda_host_free.argtypes = [C.c_void_p]
        L.tinympc_cuda_session_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.tinympc_cuda_session_destroy.argtypes = [C.c_void_p]
        L.tinympc_cuda_session_set_x0.argtypes = [C.c_void_p, c_dp]
        L.tinympc_cuda_session_set_x_ref.argtypes = [C.c_void_p, c_dp, C.c_int]
        L.tinympc_cuda_session_set_u_ref.argtypes = [C.c_void_p, c_dp, C.c_int]
        L.tinympc_cuda_session_solve.argtypes = [C.c_void_p]
        L.tinympc_cuda_session_step.argtypes = [C.c_void_p, C.c_int]
        L.tinympc_cuda_session_read.argtypes = [C.c_void_p, C.c_char_p, c_dp]
        L.tinympc_cuda_precompute_batch.argtypes = [C.POINTER(CPrecomputeIn), C.POINTER(CPrecomputeOut)]
        L.tinympc_cuda_solve_batch_models.argtypes = [C.c_void_p, C.POINTER(CModels), C.POINTER(CBatchIn), C.POINTER(CBatchOut)]
        L.tinympc_cuda_solve_batch_models_device.argtypes = [C.c_void_p, C.c_int, C.POINTER(CModels), C.POINTER(CBatchIn), C.POINTER(CBatchOut),
                                                             C.c_void_p]
        # plain-C shim over the host C++ API mirror (csrc/host/tiny_capi_shim.cpp)
        dp, ip, vp = c_dp, c_ip, C.c_void_p
        L.tinympc_host_setup.argtypes = [dp, dp, dp, dp, dp, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, ip]
        L.tinympc_host_setup.restype = vp
        L.tinympc_host_free.argtypes = [vp]
        L.tinympc_host_codegen.argtypes = [vp, C.c_char_p, dp, dp, dp, dp, C.c_int]
        L.tinympc_host_set_bound_constraints.argtypes = [vp, dp, dp, dp, dp]
        L.tinympc_host_set_cone_constraints.argtypes = [vp, C.c_int, ip, ip, dp, C.c_int, ip, ip, dp]
        L.tinympc_host_set_linear_constraints.argtypes = [vp, C.c_int, dp, dp, C.c_int, dp, dp]
        L.tinympc_host_update_settings.argtypes = [vp, C.c_double, C.c_double] + [C.c_int] * 9 + [C.c_double, C.c_double, C.c_int]
        L.tinympc_host_set_x0.argtypes = [vp, dp]
        L.tinympc_host_set_x_ref.argtypes = [vp, dp]
        L.tinympc_host_set_u_ref.argtypes = [vp, dp]
        L.tinympc_host_solve.argtypes = [vp]
        L.tinympc_host_get_solution.argtypes = [vp, dp, dp]
        L.tinympc_host_get_stats.argtypes = [vp, ip, ip, dp]
        L.tinympc_host_get_work_u0.argtypes = [vp, dp]
        L.tinympc_host_get_cache.argtypes = [vp, dp, dp, dp, dp, dp, dp]
        L.tinympc_host_set_cache_terms.argtypes = [vp, dp, dp, dp, dp]
        L.tinympc_host_init_sensitivity.argtypes = [vp]
        L.tinympc_host_set_sensitivity.argtypes = [vp, dp, dp, dp, dp]
        L.tinympc_host_reset_workspace.argtypes = [vp]
        L.tinympc_host_solve_batch.argtypes = [vp, C.POINTER(CBatchIn), C.POINTER(CBatchOut)]
        L.tinympc_host_solve_batch_models.argtypes = [vp, C.POINTER(CModels), C.POINTER(CBatchIn), C.POINTER(CBatchOut)]
        L.tinympc_host_set_devices.argtypes = [vp, ip, C.c_int]
        L.tinympc_host_set_option.argtypes = [vp, C.c_char_p, C.c_double]
        L.tinympc_host_last_error.argtypes = [vp]
        L.tinympc_host_last_error.restype = C.c_char_p
        L.tinympc_host_cuda_handle.argtypes = [vp]
        L.tinympc_host_cuda_handle.restype = vp
        _lib = L
    return _lib


def _colmajor(a):
    return np.ascontiguousarray(np.asarray(a, np.float64).T).ravel()


class _Hold:
    def __init__(self):
        self.refs = []

    def d(self, a, matrix=False):
        if a is None:
            return None
        a = _colmajor(a) if matrix else np.ascontiguousarray(np.asarray(a, np.float64)).ravel()
        self.refs.append(a)
        return a.ctypes.data_as(c_dp)

    def i(self, a):
        a = np.ascontiguousarray(np.asarray(a, np.int32)).ravel()
        self.refs.append(a)
        return a.ctypes.data_as(c_ip)


def family_struct(fam: dict, hold: _Hold) -> CFamily:
    """fam: dict with the TinySolver contents (math-shaped numpy arrays; trajectories (steps, dim))."""
    f = CFamily()
    nx, nu, N = int(fam["nx"]), int(fam["nu"]), int(fam["N"])
    f.nx, f.nu, f.N = nx, nu, N
    f.Adyn, f.Bdyn = hold.d(fam["Adyn"], True), hold.d(np.asarray(fam["Bdyn"]).reshape(nx, nu), True)
    f.fdyn, f.Q, f.R = hold.d(fam.get("fdyn", np.zeros(nx))), hold.d(fam["Q"]), hold.d(fam["R"])
    f.rho = float(fam["rho"])
    f.Kinf, f.Pinf = hold.d(np.asarray(fam["Kinf"]).reshape(nu, nx), True), hold.d(fam["Pinf"], True)
    f.Quu_inv, f.AmBKt = hold.d(np.asarray(fam["Quu_inv"]).reshape(nu, nu), True), hold.d(fam["AmBKt"], True)
    f.APf, f.BPf = hold.d(fam.get("APf", np.zeros(nx))), hold.d(fam.get("BPf", np.zeros(nu)))
    if fam.get("dKinf_drho") is not None:
        f.dKinf_drho = hold.d(np.asarray(fam["dKinf_drho"]).reshape(nu, nx), True)
        f.dPinf_drho = hold.d(fam["dPinf_drho"], True)
    for k, default in (("abs_pri_tol", 1e-3), ("abs_dua_tol", 1e-3), ("max_iter", 1000), ("check_termination", 1),
                       ("en_state_bound", 0), ("en_input_bound", 0), ("en_state_soc", 0), ("en_input_soc", 0),
                       ("en_state_linear", 0), ("en_input_linear", 0), ("adaptive_rho", 0), ("adaptive_rho_min", 1.0),
                       ("adaptive_rho_max", 100.0), ("adaptive_rho_enable_clipping", 1)):
        setattr(f, k, type(default)(fam.get(k, default)))
    f.x_min, f.x_max = hold.d(fam.get("x_min")), hold.d(fam.get("x_max"))
    f.u_min, f.u_max = hold.d(fam.get("u_min")), hold.d(fam.get("u_max"))
    Acx, Acu = np.asarray(fam.get("Acx", []), np.int32), np.asarray(fam.get("Acu", []), np.int32)
    f.numStateCones, f.numInputCones = len(Acx), len(Acu)
    if len(Acx):
        f.Acx, f.qcx, f.cx = hold.i(Acx), hold.i(fam["qcx"]), hold.d(fam["cx"])
    if len(Acu):
        f.Acu, f.qcu, f.cu = hold.i(Acu), hold.i(fam["qcu"]), hold.d(fam["cu"])
    Alx, Alu = np.asarray(fam.get("Alin_x", np.zeros((0, nx)))), np.asarray(fam.get("Alin_u", np.zeros((0, nu))))
    f.numStateLinear = int(Alx.shape[0]) if Alx.size else 0
    f.numInputLinear = int(Alu.shape[0]) if Alu.size else 0
    if f.numStateLinear:
        f.Alin_x, f.blin_x = hold.d(Alx, True), hold.d(fam["blin_x"])
    if f.numInputLinear:
        f.Alin_u, f.blin_u = hold.d(Alu, True), hold.d(fam["blin_u"])
    return f


class CudaSolver:
    """Thin object wrapper over the opaque tinympc_cuda_solver handle."""

    def __init__(self, devices=None, borrowed_handle=None):
        self.L = load()
        self.h = C.c_void_p()
        self.owned = borrowed_handle is None
        self.dims = None
        if borrowed_handle is not None:       # handle owned by a host-side TinySolver (tiny_b200_cuda_handle)
            self.h = C.c_void_p(borrowed_handle)
            return
        if devices:
            arr = (C.c_int * len(devices))(*devices)
            rc = self.L.tinympc_cuda_create(C.byref(self.h), arr, len(devices))
        else:
            rc = self.L.tinympc_cuda_create(C.byref(self.h), None, 0)
        if rc:
            raise TinympcCudaError(rc, "tinympc_cuda_create failed (no CUDA device?)")
        self.dims = None

    def _check(self, rc):
        if rc:
            raise TinympcCudaError(rc, self.L.tinympc_cuda_last_error(self.h).decode())

    def close(self):
        if self.h and self.owned:
            self.L.tinympc_cuda_destroy(self.h)
        self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name: str, value: float):
        self._check(self.L.tinympc_cuda_set_option(self.h, name.encode(), float(value)))

    def set_family(self, fam: dict):
        hold = _Hold()
        cf = family_struct(fam, hold)
        self._check(self.L.tinympc_cuda_set_family(self.h, C.byref(cf)))
        self.dims = (cf.nx, cf.nu, cf.N)

    @property
    def last_kernel(self) -> str:
        return self.L.tinympc_cuda_last_kernel(self.h).decode()

    @property
    def launch_count(self) -> int:
        return int(self.L.tinympc_cuda_launch_count(self.h))

    @property
    def last_marked(self) -> int:
        """problems the last "mixed" solve handed to the fp64 pass"""
        return int(self.L.tinympc_cuda_last_marked(self.h))

    def last_timing(self):
        ms = (C.c_double * 3)()
        self.L.tinympc_cuda_last_timing(self.h, ms)
        return dict(total_ms=ms[0], kernel_ms=ms[1], chunks=int(ms[2]))

    def last_pass_ms(self):
        """(fp32 pass, compaction + fp64 pass) of the last device-resident exact-count solve; None unless option pass_timing = 1"""
        ms = (C.c_double * 2)()
        return None if self.L.tinympc_cuda_last_pass_ms(self.h, ms) else (ms[0], ms[1])

    # ---- host buffers (numpy) ---------------------------------------------------------------
    def solve_batch(self, x0, Xref=None, Uref=None, x_min=None, x_max=None, u_min=None, u_max=None,
                    want_residuals=True, want_rho=True, out=None, xref_const=None, compact_out=False, models=None) -> dict:
        """xref_const (B, nx): one reference state per problem held over the horizon (instead of Xref);
        compact_out: return only u0 (B, nu), iter, status -- the trajectories stay on the device.
        models: every problem's own model (see pack_models), tinympc_cuda_solve_batch_models; None: the family's."""
        nx, nu, N = self.dims
        keep = []

        def fptr(a, shape):
            if a is None:
                return None
            a = np.ascontiguousarray(a, np.float32)
            if a.shape != shape:
                raise ValueError(f"expected shape {shape}, got {a.shape}")
            keep.append(a)
            return a.ctypes.data

        x0 = np.ascontiguousarray(x0, np.float32)
        B = x0.shape[0]
        cin = CBatchIn(B, fptr(x0, (B, nx)), fptr(Xref, (B, N, nx)), fptr(Uref, (B, N - 1, nu)),
                       fptr(x_min, (B, N, nx)), fptr(x_max, (B, N, nx)), fptr(u_min, (B, N - 1, nu)), fptr(u_max, (B, N - 1, nu)),
                       fptr(xref_const, (B, nx)))
        if out is None:
            if compact_out:
                out = dict(u0=np.empty((B, nu), np.float32), iter=np.empty(B, np.int32), status=np.empty(B, np.int32))
            else:
                out = dict(x=np.empty((B, N, nx), np.float32), u=np.empty((B, N - 1, nu), np.float32),
                           iter=np.empty(B, np.int32), status=np.empty(B, np.int32))
                if want_residuals:
                    out["residuals"] = np.empty((B, 4), np.float32)
                if want_rho:
                    out["rho"] = np.empty(B, np.float32)
        opt = lambda k: out[k].ctypes.data if k in out else None
        co = CBatchOut(opt("x"), opt("u"), out["iter"].ctypes.data, out["status"].ctypes.data, opt("residuals"), opt("rho"), opt("u0"))
        if models is None:
            self._check(self.L.tinympc_cuda_solve_batch(self.h, C.byref(cin), C.byref(co)))
        else:
            arrays = pack_models(models, B, nx, nu)
            self._check(self.L.tinympc_cuda_solve_batch_models(self.h, C.byref(models_struct(arrays)), C.byref(cin), C.byref(co)))
        return out

    def solve_batch_models(self, models: dict, x0, **kw) -> dict:
        """Problems that each bring their own model (tinympc_cuda_solve_batch_models); `models` as for pack_models, the rest as for
        solve_batch."""
        return self.solve_batch(x0, models=models, **kw)

    def session(self, batch: int, dev_index: int = 0) -> "CudaSession":
        """`batch` warm-started solvers of the family, resident on the device (tinympc_cuda_session_*)."""
        return CudaSession(self, batch, dev_index)

    # ---- device buffers (raw pointers, e.g. torch.Tensor.data_ptr()) ---------------------------
    def solve_batch_device(self, batch: int, x0, Xref, Uref, x, u, iters, status, residuals=None, rho=None,
                           x_min=None, x_max=None, u_min=None, u_max=None, stream=None, dev_index=0, xref_const=None, u0=None):
        cin = CBatchIn(batch, x0, Xref, Uref, x_min, x_max, u_min, u_max, xref_const)
        co = CBatchOut(x, u, iters, status, residuals, rho, u0)
        self._check(self.L.tinympc_cuda_solve_batch_device(self.h, dev_index, C.byref(cin), C.byref(co), stream))

    def solve_batch_models_device(self, models: dict, batch: int, x0, Xref, Uref, x, u, iters, status, residuals=None, rho=None,
                                  x_min=None, x_max=None, u_min=None, u_max=None, stream=None, dev_index=0, xref_const=None, u0=None):
        """tinympc_cuda_solve_batch_models_device: models maps CModels field names (Adyn, Bdyn, fdyn, Q, R, rho, Kinf, Pinf, Quu_inv,
        AmBKt, APf, BPf, dKinf_drho, dPinf_drho) to device pointers of the column-major float64 arrays (pack_models' layout)."""
        cin = CBatchIn(batch, x0, Xref, Uref, x_min, x_max, u_min, u_max, xref_const)
        co = CBatchOut(x, u, iters, status, residuals, rho, u0)
        self._check(self.L.tinympc_cuda_solve_batch_models_device(self.h, dev_index, C.byref(models_struct(models)), C.byref(cin), C.byref(co),
                                                                  stream))


class CudaSession:
    """A batch of warm-started solvers on the device: the closed-loop pattern of the reference
    (tinympc/TinyMPC/examples/quadrotor_hovering.cpp:73-93) for `batch` independent systems at once."""

    def __init__(self, solver: CudaSolver, batch: int, dev_index: int = 0):
        self.solver, self.L, self.batch = solver, solver.L, int(batch)
        self.nx, self.nu, self.N = solver.dims
        self.h = C.c_void_p()
        solver._check(self.L.tinympc_cuda_session_create(solver.h, dev_index, self.batch, C.byref(self.h)))

    def close(self):
        if self.h:
            self.L.tinympc_cuda_session_destroy(self.h)
        self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _arr(self, a, shape_batch, shape_one):
        """(pointer, broadcast flag, keep-alive array) for a per-solver array or one array shared by all solvers"""
        if a is None:
            return None, 0, None
        a = np.ascontiguousarray(a, np.float64)
        if a.shape == shape_one:
            return a.ctypes.data_as(c_dp), 1, a
        if a.shape != shape_batch:
            raise ValueError(f"expected shape {shape_batch} or {shape_one}, got {a.shape}")
        return a.ctypes.data_as(c_dp), 0, a

    def set_x0(self, x0):
        x0 = np.ascontiguousarray(x0, np.float64)
        if x0.shape != (self.batch, self.nx):
            raise ValueError(f"expected shape {(self.batch, self.nx)}, got {x0.shape}")
        self.solver._check(self.L.tinympc_cuda_session_set_x0(self.h, x0.ctypes.data_as(c_dp)))

    def set_x_ref(self, Xref):
        p, bc, keep = self._arr(Xref, (self.batch, self.N, self.nx), (self.N, self.nx))
        self.solver._check(self.L.tinympc_cuda_session_set_x_ref(self.h, p, bc))

    def set_u_ref(self, Uref):
        p, bc, keep = self._arr(Uref, (self.batch, self.N - 1, self.nu), (self.N - 1, self.nu))
        self.solver._check(self.L.tinympc_cuda_session_set_u_ref(self.h, p, bc))

    def solve(self):
        self.solver._check(self.L.tinympc_cuda_session_solve(self.h))

    def step(self, use_solution: bool = False):
        """x0 <- A x0 + B u0 + f on the device; u0 = work->u[:, 0] (default) or solution->u[:, 0]"""
        self.solver._check(self.L.tinympc_cuda_session_step(self.h, 1 if use_solution else 0))

    def read(self, field: str) -> np.ndarray:
        nx, nu, N, B = self.nx, self.nu, self.N, self.batch
        shape = {"x0": (B, nx), "x": (B, N, nx), "sol_x": (B, N, nx), "u": (B, N - 1, nu), "sol_u": (B, N - 1, nu),
                 "iter": (B,), "status": (B,), "rho": (B,), "residuals": (B, 4)}[field]
        out = np.empty(shape, np.float64)
        self.solver._check(self.L.tinympc_cuda_session_read(self.h, field.encode(), out.ctypes.data_as(c_dp)))
        return out.astype(np.int32) if field in ("iter", "status") else out
