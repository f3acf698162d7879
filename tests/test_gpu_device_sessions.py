"""GPU tests of the device-resident model-session entries and the device-resident cache precompute
(tinympc_cuda_precompute_batch_device, tinympc_cuda_session_create_models_device / _set_models_device / _write_device / _read_device).

What is checked:
  * the device precompute gives the host precompute's outputs bit for bit (cartpole, quadrotor, rocket, with and without the
    sensitivities, and a shape with nu > nx);
  * a session driven through the device entries stays bit-identical to one driven through the host entries, after every call,
    on the lane-group kernel's model sessions and on the warp-per-problem kernel in fp64, fp32 and with adaptive rho; read_device
    equals session_read;
  * a closed loop relinearised on the GPU (torch forms A_k, B_k from the state read with read_device, precompute_batch_device
    writes the caches into the model arrays, set_models_device) takes the iteration counts of one reference session per solver
    fed the same models and caches;
  * the stream contract, in both directions, and that the entries return without waiting;
  * every EINVAL case, each leaving the session as it was.
"""
import ctypes as C
import importlib
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

import oracle as O
from model_sessions_ref import SESSION_FIELDS, read_all
from test_gpu_model_sessions import refs_of, solver
from test_gpu_precompute import perturbed

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
EINVAL = 1
SLEEP_CYCLES = 200_000_000           # torch.cuda._sleep: ~0.1 s of a busy stream


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def capi(torch):
    return importlib.import_module("tinympc-matlab_b200.capi")


def cm(a):
    """math-shaped (n, rows, cols) -> column-major chunks per problem"""
    return np.ascontiguousarray(np.swapaxes(a, 1, 2))


class Dev:
    """host arrays -> float64 tensors on cuda:0, kept alive with their pointers"""

    def __init__(self, torch, arrays: dict):
        self.t = {k: torch.from_numpy(np.ascontiguousarray(v, np.float64)).cuda() for k, v in arrays.items()}
        self.p = {k: v.data_ptr() for k, v in self.t.items()}


def bits(a):
    return np.ascontiguousarray(a, np.float64).tobytes()


# ---- 1. precompute: device entry against host entry ---------------------------------------------------------------------------
def precompute_inputs(family, problems):
    if family == "wide":                                        # nu > nx
        rng = np.random.default_rng(3)
        n, nx, nu = 24, 2, 3
        A = np.eye(nx)[None] + 0.1 * rng.standard_normal((n, nx, nx))
        B = rng.standard_normal((n, nx, nu))
        return A, B, rng.uniform(1, 2, (n, nx)), rng.uniform(1, 2, (n, nu)), rng.uniform(0.5, 2, n), 0.1 * rng.standard_normal((n, nx))
    p = dict(cartpole=problems.cartpole, quadrotor=problems.quadrotor, rocket=problems.rocket)[family]()
    return perturbed(p, 24, seed=5)


PRE_SHAPES = lambda nx, nu: dict(Kinf=(nu, nx), Pinf=(nx, nx), Quu_inv=(nu, nu), AmBKt=(nx, nx), APf=(nx,), BPf=(nu,))
SENS_SHAPES = lambda nx, nu: dict(dKinf_drho=(nu, nx), dPinf_drho=(nx, nx), dC1_drho=(nu, nu), dC2_drho=(nx, nx))
HOST_KEY = dict(dKinf_drho="dKinf", dPinf_drho="dPinf", dC1_drho="dC1", dC2_drho="dC2")


def precompute_device(torch, capi, A, B, Q, R, rho, f, sens, stream=None, ins=None):
    n, nx, nu = A.shape[0], A.shape[1], B.shape[2]
    ins = ins or Dev(torch, dict(A=cm(A), B=cm(B), Q=Q, R=R, rho=rho, f=f))
    shapes = dict(PRE_SHAPES(nx, nu), **(SENS_SHAPES(nx, nu) if sens else {}))
    # (cols, rows) in C order is the column-major (rows x cols) chunk
    out = {k: torch.full((n,) + s[::-1], float("nan"), dtype=torch.float64, device="cuda") for k, s in shapes.items()}
    out["iters"] = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    capi.precompute_batch_device(n, nx, nu, ins.p["A"], ins.p["B"], ins.p["Q"], ins.p["R"], ins.p["rho"],
                                 {k: v.data_ptr() for k, v in out.items()}, f=ins.p["f"], stream=stream)
    return ins, out


def assert_precompute_equal(out, h):
    for k, t in out.items():
        d = t.cpu().numpy()
        d = np.swapaxes(d, 1, 2) if d.ndim == 3 else d
        assert np.ascontiguousarray(d).tobytes() == np.ascontiguousarray(h[HOST_KEY.get(k, k)]).tobytes(), k


@pytest.mark.parametrize("sens", [False, True], ids=["cache", "sensitivities"])
@pytest.mark.parametrize("family", ["cartpole", "quadrotor", "rocket", "wide"])
def test_precompute_device_entry_is_bit_identical_to_the_host_entry(family, sens, torch, capi, problems):
    A, B, Q, R, rho, f = precompute_inputs(family, problems)
    Q, R = Q + rho[:, None], R + rho[:, None]                    # the model's work->Q, work->R (quirk Q1)
    h = capi.precompute_batch(A, B, Q, R, rho, f, sensitivities=sens)
    _, out = precompute_device(torch, capi, A, B, Q, R, rho, f, sens)
    torch.cuda.synchronize()
    assert_precompute_equal(out, h)
    assert (h["iters"] > 1).all()


# ---- model sets -----------------------------------------------------------------------------------------------------------------
def model_set(capi, p, k, seed, adaptive=False):
    """k models perturbed from p (test_gpu_precompute.perturbed) with their caches from the host precompute, math-shaped"""
    A, B, Q, R, rho, f = perturbed(p, k, seed)
    o = capi.precompute_batch(A, B, Q + rho[:, None], R + rho[:, None], rho, f, sensitivities=adaptive)
    m = dict(A=A, B=B, f=f, Q=Q + rho[:, None], R=R + rho[:, None], rho=rho,
             **{x: o[x] for x in ("Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf")})
    if adaptive:
        m["dKinf"], m["dPinf"] = o["dKinf"], o["dPinf"]
    return m


def tile(m, batch):
    which = np.arange(batch) % len(m["rho"])
    return {k: v[which] for k, v in m.items()}


def case_problem(problems, name):
    return dict(quadrotor=problems.quadrotor, cartpole20=lambda: problems.cartpole(N=20),
                adaptive=lambda: problems.quadrotor(adaptive=True))[name]()


# ---- 2. host entries against device entries, bit for bit ------------------------------------------------------------------------
@pytest.mark.parametrize("name, precision, force_wpp, kernel", [
    ("quadrotor", 64, 0, "gpp_f64_12x4x10_box_g16_v0_mdl_session"),
    ("cartpole20", 64, 0, "gpp_f64_4x1x20_box_g8_v0_mdl_session"),
    ("quadrotor", 64, 1, "wpp_f64_mdl_session"),
    ("quadrotor", 32, 0, "wpp_f32_mdl_session"),
    ("adaptive", 64, 0, "wpp_f64_mdl_session"),
], ids=["quadrotor_gpp", "cartpole20_gpp", "quadrotor_wpp64", "quadrotor_wpp32", "adaptive_wpp"])
def test_device_entries_are_bit_identical_to_the_host_entries(name, precision, force_wpp, kernel, torch, capi, problems, oracle_mod):
    p = case_problem(problems, name)
    adaptive = bool(p.adaptive_rho)
    cache = oracle_mod.get_cache(p, "port")
    B, steps = 40, 8
    nx, nu = p.nx, p.nu
    m1, m2 = tile(model_set(capi, p, 8, 1, adaptive), B), tile(model_set(capi, p, 8, 2, adaptive), B)
    d1, d2 = Dev(torch, capi.pack_models(m1, B, nx, nu)), Dev(torch, capi.pack_models(m2, B, nx, nu))
    b = problems.make_batch(p, B, 0.6, seed=13)
    Xref, Uref = refs_of(b, p, B)
    s = solver(capi, p, cache, precision, force_wpp)
    hs = s.session(B, models=m1)
    ds = s.session(B, models_device=d1.p)
    keep = []

    def dev(a):
        keep.append(torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda())
        return keep[-1].data_ptr()

    def check(what):
        for f in SESSION_FIELDS:
            h, d = hs.read(f), ds.read(f)
            assert bits(h) == bits(d), f"{name}: {what}: {f} differs"
            buf = torch.full(d.shape, float("nan"), dtype=torch.float64, device="cuda")
            ds.read_device(f, buf.data_ptr())
            assert bits(buf.cpu().numpy()) == bits(d), f"{name}: {what}: read_device({f}) differs from read"

    check("create")
    hs.set_x_ref(Xref[0]); ds.write_device("Xref", dev(Xref[0]), broadcast=True); check("Xref broadcast")
    hs.set_u_ref(Uref); ds.write_device("Uref", dev(Uref), broadcast=False); check("Uref")
    hs.set_x0(b.x0.astype(np.float64)); ds.write_device("x0", dev(b.x0.astype(np.float64))); check("x0")
    for t in range(steps):
        if t == 3:
            hs.set_models(m2); ds.set_models_device(d2.p); check(f"set_models at {t}")
        if t == 5:
            hs.set_x_ref(Xref[::-1]); ds.write_device("Xref", dev(Xref[::-1])); check(f"Xref at {t}")
            hs.set_u_ref(Uref[1]); ds.write_device("Uref", dev(Uref[1]), broadcast=True); check(f"Uref broadcast at {t}")
        if t == 6:
            x = hs.read("x0") + 0.05
            hs.set_x0(x); ds.write_device("x0", dev(x)); check(f"x0 at {t}")
        hs.solve(); ds.solve()
        assert s.last_kernel == kernel, s.last_kernel
        check(f"solve {t}")
        hs.step(); ds.step(); check(f"step {t}")
    hs.close(); ds.close(); s.close()


# ---- 3. relinearised closed loop against the reference --------------------------------------------------------------------------
_HOOK = None


def cache_hook():
    """the C port with port_session_set_cache (tests/oracle_hooks/port_session_set_cache.c), built once into a temporary directory"""
    global _HOOK
    if _HOOK is None:
        out = Path(tempfile.mkdtemp(prefix="tmpc_cache_hook_")) / "liboracle_port_cache_hook.so"
        subprocess.check_call(["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-I", str(ROOT / "oracle"), "-o", str(out),
                               str(ROOT / "tests" / "oracle_hooks" / "port_session_set_cache.c"), "-lm", "-lpthread"])
        _HOOK = C.CDLL(str(out))
    return _HOOK


class CacheSession(O.Session):
    """oracle.Session on the C port whose model AND cache are replaced between two solves by given arrays"""

    def __init__(self, p):
        self.L, self.p, self.pre = cache_hook(), p, "port"
        self._keep = O._Keep()
        self._cp = O.c_problem(p, self._keep)
        fn = self.L.port_session_create
        fn.restype = C.c_void_p
        self.h = C.c_void_p(fn(C.byref(self._cp)))
        assert self.h

    def set_model_and_cache(self, p, Kinf, Pinf, Quu_inv, AmBKt, APf, BPf):
        keep = O._Keep()
        cp = O.c_problem(p, keep)
        d = lambda a: keep.d(np.asarray(a, np.float64).ravel())     # column-major chunks already
        fn = self.L.port_session_set_cache
        fn.restype = C.c_int
        assert fn(self.h, C.byref(cp), d(Kinf), d(Pinf), d(Quu_inv), d(AmBKt), d(APf), d(BPf)) == 0
        self.p = p


def test_relinearised_closed_loop_matches_the_reference(torch, capi, problems, oracle_mod):
    p = problems.quadrotor()
    nx, nu, B, steps = p.nx, p.nu, 32, 12
    s = solver(capi, p, oracle_mod.get_cache(p, "port"), 64)
    rng = np.random.default_rng(17)
    Qd, Rd = p.Qdiag * rng.uniform(0.5, 2.0, (B, nx)), p.Rdiag * rng.uniform(0.5, 2.0, (B, nu))
    rho = p.rho * rng.uniform(0.5, 2.0, B)
    cuda = dict(dtype=torch.float64, device="cuda")
    A0, B0 = torch.tensor(p.A, **cuda), torch.tensor(np.asarray(p.B).reshape(nx, nu), **cuda)
    # the session's model arrays, column-major per solver; the precompute writes the cache fields in place
    T = dict(Adyn=torch.empty((B, nx, nx), **cuda), Bdyn=torch.empty((B, nu, nx), **cuda), Q=torch.tensor(Qd + rho[:, None], **cuda),
             R=torch.tensor(Rd + rho[:, None], **cuda), rho=torch.tensor(rho, **cuda), Kinf=torch.empty((B, nx, nu), **cuda),
             Pinf=torch.empty((B, nx, nx), **cuda), Quu_inv=torch.empty((B, nu, nu), **cuda), AmBKt=torch.empty((B, nx, nx), **cuda),
             APf=torch.empty((B, nx), **cuda), BPf=torch.empty((B, nu), **cuda))
    ptrs = {k: v.data_ptr() for k, v in T.items()}

    def relinearise(x):
        g = 1.0 + 0.05 * torch.tanh(x)[:, :, None]               # row i of A and B scaled with state i
        T["Adyn"].copy_((A0 * g).transpose(1, 2))
        T["Bdyn"].copy_((B0 * g).transpose(1, 2))
        capi.precompute_batch_device(B, nx, nu, ptrs["Adyn"], ptrs["Bdyn"], ptrs["Q"], ptrs["R"], ptrs["rho"],
                                     {k: ptrs[k] for k in ("Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf")})

    b = problems.make_batch(p, B, 0.6, seed=19)
    Xref, Uref = refs_of(b, p, B)
    x = torch.tensor(b.x0.astype(np.float64), **cuda)
    relinearise(x)
    ses = s.session(B, models_device=ptrs)
    ses.set_x_ref(Xref)
    ses.set_u_ref(Uref)
    ses.write_device("x0", x.data_ptr())
    refs = []
    for k in range(B):
        refs.append(CacheSession(p.with_(Qdiag=Qd[k], Rdiag=Rd[k], rho=float(rho[k]))))
        refs[-1].set_x_ref(Xref[k]); refs[-1].set_u_ref(Uref[k])
    xr = b.x0.astype(np.float64)
    for t in range(steps):
        if t:
            ses.read_device("x0", x.data_ptr())
            relinearise(x)
            ses.set_models_device(ptrs)
        h = {k: v.cpu().numpy() for k, v in T.items()}           # for the reference only
        Ak, Bk = np.swapaxes(h["Adyn"], 1, 2), np.swapaxes(h["Bdyn"], 1, 2)
        ses.solve()
        it, st = ses.read("iter"), ses.read("status")
        ses.step()
        git, gst, nxt = np.zeros(B, int), np.zeros(B, int), np.zeros((B, nx))
        for k, r in enumerate(refs):
            r.set_model_and_cache(p.with_(A=Ak[k], B=Bk[k], Qdiag=Qd[k], Rdiag=Rd[k], rho=float(rho[k])),
                                  h["Kinf"][k], h["Pinf"][k], h["Quu_inv"][k], h["AmBKt"][k], h["APf"][k], h["BPf"][k])
            r.set_x0(xr[k])
            g = r.solve()
            git[k], gst[k] = g["iter"], g["status"]
            nxt[k] = Ak[k] @ xr[k] + Bk[k] @ g["work_u0"] + p.f
        assert np.array_equal(it, git) and np.array_equal(st, gst), (t, np.flatnonzero(it != git), it, git)
        x0 = ses.read("x0")
        assert np.abs(x0 - nxt).max() <= 1e-8 * max(1.0, np.abs(nxt).max()), t
        xr = nxt
    assert len({tuple(r) for r in np.round(xr, 3)}) > 1
    ses.close(); s.close()


# ---- 4. the stream contract -----------------------------------------------------------------------------------------------------
def test_stream_contract(torch, capi, problems, oracle_mod):
    p = problems.quadrotor()
    B = 64
    s = solver(capi, p, oracle_mod.get_cache(p, "port"), 64)
    m1, m2 = tile(model_set(capi, p, 8, 1), B), tile(model_set(capi, p, 8, 2), B)
    d1 = Dev(torch, capi.pack_models(m1, B, p.nx, p.nu))
    d2 = Dev(torch, capi.pack_models(m2, B, p.nx, p.nu))
    ses = s.session(B, models_device=d1.p)
    b = problems.make_batch(p, B, 0.6, seed=3)
    Xref, Uref = refs_of(b, p, B)
    ses.set_x_ref(Xref); ses.set_u_ref(Uref); ses.set_x0(b.x0.astype(np.float64))
    ses.solve()
    side, other = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()

    def produce(stream, pairs):
        """on `stream`: a long sleep, then dst <- src for every pair.  Until then every dst holds valid inputs, so a missing wait
        gives wrong numbers, never a fault"""
        torch.cuda.synchronize()                 # the tensors the test just made are complete
        with torch.cuda.stream(stream):
            torch.cuda._sleep(SLEEP_CYCLES)
            for dst, src in pairs:
                dst.copy_(src)

    # write_device runs after the producer
    x_old = ses.read("x0")
    buf, new = torch.tensor(x_old, device="cuda"), torch.tensor(x_old + 0.25, device="cuda")
    produce(side, [(buf, new)])
    ses.write_device("x0", buf.data_ptr(), stream=side.cuda_stream)
    assert not side.query(), "write_device waited for the stream"
    side.synchronize()
    assert bits(ses.read("x0")) == bits(x_old + 0.25)

    # set_models_device runs after the producer (rho tells the model sets apart)
    staged = Dev(torch, capi.pack_models(m1, B, p.nx, p.nu))
    produce(side, [(staged.t[k], d2.t[k]) for k in staged.t])
    ses.set_models_device(staged.p, stream=side.cuda_stream)
    assert not side.query(), "set_models_device waited for the stream"
    side.synchronize()
    assert bits(ses.read("rho")) == bits(m2["rho"])

    # precompute_batch_device runs after the producer
    A, Bm, Q, R, rho, f = perturbed(p, 16, seed=5)
    A2 = A * 1.001
    Q, R = Q + rho[:, None], R + rho[:, None]
    ins = Dev(torch, dict(A=cm(A), B=cm(Bm), Q=Q, R=R, rho=rho, f=f))
    a2 = torch.from_numpy(cm(A2)).cuda()        # held until the side stream has read it
    produce(side, [(ins.t["A"], a2)])
    _, out = precompute_device(torch, capi, A, Bm, Q, R, rho, f, False, stream=side.cuda_stream, ins=ins)
    assert not side.query(), "precompute_batch_device waited for the stream"
    side.synchronize()
    assert_precompute_equal(out, capi.precompute_batch(A2, Bm, Q, R, rho, f))

    # the other direction: work the caller queues after read_device sees its result.  A write_device behind a sleep on `other`
    # holds the session's stream, so the read (and with it the caller's copy, if it did not wait) would come too early.
    x_late = torch.tensor(x_old - 0.5, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(other):
        torch.cuda._sleep(SLEEP_CYCLES)
    ses.write_device("x0", x_late.data_ptr(), stream=other.cuda_stream)
    dst = torch.full((B, p.nx), float("nan"), dtype=torch.float64, device="cuda")
    ses.read_device("x0", dst.data_ptr(), stream=side.cuda_stream)
    assert not side.query(), "read_device waited for the session's stream"
    with torch.cuda.stream(side):
        seen = dst.clone()
    side.synchronize()
    assert bits(seen.cpu().numpy()) == bits(x_old - 0.5)
    ses.close(); s.close()


# ---- 5. errors --------------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_session_as_it_was(torch, capi, problems, oracle_mod):
    p = problems.quadrotor()
    B, nx, nu = 24, p.nx, p.nu
    s = solver(capi, p, oracle_mod.get_cache(p, "port"), 64)
    L, h = s.L, C.c_void_p()
    m = tile(model_set(capi, p, 8, 1), B)
    host = capi.pack_models(m, B, nx, nu)
    d = Dev(torch, host)
    ses = s.session(B, models_device=d.p)
    b = problems.make_batch(p, B, 0.6, seed=7)
    Xref, Uref = refs_of(b, p, B)
    ses.set_x_ref(Xref); ses.set_u_ref(Uref); ses.set_x0(b.x0.astype(np.float64))
    ses.solve(); ses.step()
    before = read_all(ses)

    def unchanged(what):
        after = read_all(ses)
        for f in SESSION_FIELDS:
            assert bits(after[f]) == bits(before[f]), (what, f)

    raw = torch.zeros(B * nx * p.N + 2, dtype=torch.float64, device="cuda")
    misaligned = raw.data_ptr() + 8
    x0_host = np.zeros((B, nx))
    other = None
    if torch.cuda.device_count() > 1:
        other = torch.zeros(B * nx * nx, dtype=torch.float64, device="cuda:1")

    def set_models(arrays):
        return L.tinympc_cuda_session_set_models_device(ses.h, C.byref(capi.models_struct(arrays)), None)

    def create(arrays, solver_=s):
        rc = solver_.L.tinympc_cuda_session_create_models_device(solver_.h, 0, B, C.byref(capi.models_struct(arrays)), None, C.byref(h))
        assert not h, "a failed create returned a session"
        return rc

    bad_models = [(f"missing {k}", {x: v for x, v in d.p.items() if x != k})
                  for k in ("Adyn", "Bdyn", "Q", "R", "rho", "Kinf", "Pinf", "Quu_inv", "AmBKt")]
    bad_models += [("misaligned Adyn", dict(d.p, Adyn=misaligned)), ("host Kinf", dict(d.p, Kinf=host["Kinf"].ctypes.data))]
    if other is not None:
        bad_models.append(("Pinf on another device", dict(d.p, Pinf=other.data_ptr())))
    for what, arrays in bad_models:
        assert set_models(arrays) == EINVAL, what
        unchanged(what)
        assert create(arrays) == EINVAL, what
        unchanged(what)
    assert L.tinympc_cuda_session_set_models_device(ses.h, None, None) == EINVAL
    assert L.tinympc_cuda_session_create_models_device(s.h, 0, B, None, None, C.byref(h)) == EINVAL and not h
    # adaptive rho without the two sensitivities
    pa = problems.quadrotor(adaptive=True)
    sa = solver(capi, pa, oracle_mod.get_cache(pa, "port"), 64)
    da = Dev(torch, capi.pack_models(tile(model_set(capi, pa, 4, 1, adaptive=True), B), B, nx, nu))
    for drop in ("dKinf_drho", "dPinf_drho"):
        assert create({k: v for k, v in da.p.items() if k != drop}, sa) == EINVAL
        assert "adaptive_rho" in sa.L.tinympc_cuda_last_error(sa.h).decode()
    sa.close()
    # set_models_device on a family session
    fam = s.session(B)
    with pytest.raises(capi.TinympcCudaError) as e:
        fam.set_models_device(d.p)
    assert e.value.code == EINVAL
    fam.close()
    # session I/O
    good = torch.zeros((B, nx * p.N), dtype=torch.float64, device="cuda")
    io = [("write", "x", good.data_ptr()), ("write", "Kinf", good.data_ptr()), ("write", "x0", None), ("write", "x0", misaligned),
          ("write", "x0", x0_host.ctypes.data), ("read", "Xref", good.data_ptr()), ("read", "bogus", good.data_ptr()),
          ("read", "x", None), ("read", "x", misaligned), ("read", "x0", x0_host.ctypes.data)]
    if other is not None:
        io += [("write", "x0", other.data_ptr()), ("read", "x0", other.data_ptr())]
    for op, field, ptr in io:
        rc = (L.tinympc_cuda_session_write_device(ses.h, field.encode(), ptr, 0, None) if op == "write"
              else L.tinympc_cuda_session_read_device(ses.h, field.encode(), ptr, None))
        assert rc == EINVAL, (op, field, ptr)
        unchanged((op, field))
    # the precompute
    n = 4
    A, Bm, Q, R, rho, f = perturbed(p, n, seed=1)
    ins = Dev(torch, dict(A=cm(A), B=cm(Bm), Q=Q, R=R, rho=rho))
    outs = Dev(torch, {k: np.zeros((n,) + s_) for k, s_ in PRE_SHAPES(nx, nu).items()})
    args = dict(ins.p)
    for what, a, o in [("NULL A", dict(args, A=None), outs.p), ("misaligned B", dict(args, B=misaligned), outs.p),
                       ("host Q", dict(args, Q=Q.ctypes.data), outs.p), ("NULL Kinf", args, dict(outs.p, Kinf=None)),
                       ("host Pinf", args, dict(outs.p, Pinf=np.zeros((n, nx, nx)).ctypes.data))]:
        with pytest.raises(capi.TinympcCudaError) as e:
            capi.precompute_batch_device(n, nx, nu, a["A"], a["B"], a["Q"], a["R"], a["rho"], o)
        assert e.value.code == EINVAL, what
    unchanged("end")
    ses.close(); s.close()

