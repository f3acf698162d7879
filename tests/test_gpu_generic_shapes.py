"""GPU tests of the shapes and feature mixes that have no compiled kernel: random families (tests/generic_families.py) run on
the run-time-shaped instance of the warp-per-problem kernel (tmpc_wpp.cu, wpp_kernel<T, 0, 0>) through every entry that
reaches it -- batches in fp64, fp32 and the exact-count mode, the chunked host pipeline and compact I/O, tiny_solve through the
MATLAB-class mirror, device sessions -- and the batched cache precompute (tmpc_precompute.cu) at shapes other than the shipped
ones.  The reference is the oracle's C restatement of the reference solver (or the reference library itself when it is built).

None of the (nx, nu) pairs below is (12, 4), (4, 1) or (6, 3), the pairs with compiled instances.  What each shape exercises:
  1 x 1 x 2    smallest shape, a single backward step
  2 x 3 x 8    more inputs than states
  5 x 2 x 40   N > 32: each lane projects several time steps onto the cones and half-spaces
  10 x 3 x 75  fp32 workspaces of a CTA just inside the 200 KiB shared-memory limit (iterated in shared memory)
  10 x 3 x 76  just outside it (iterated in global memory)
  36 x 5 x 6   nx > 32: lanes stride over the rows of every mat-vec
  7 x 7 x 12   nu = nx with every feature on (4 cones per side, 3 linear rows per side, adaptive rho)
"""
import importlib

import numpy as np
import pytest

import cases
import generic_families as G
from test_gpu_parity import compare, solve_gpu

pytestmark = pytest.mark.gpu

# name -> (nx, nu, N, seed, batch size, family options)
CASES = {
    "1x1x2": (1, 1, 2, 1, 3000, dict(affine=True, state_bound=True)),
    "2x3x8_all": (2, 3, 8, 1, 1500, dict(affine=True, state_bound=True, cones=(2, 2), linear=(1, 2), adaptive=True, check=2, max_iter=200)),
    "5x2x40_cones": (5, 2, 40, 2, 1000, dict(affine=True, cones=(3, 0), linear=(3, 2), max_iter=200)),
    "5x2x40_max15": (5, 2, 40, 1, 1500, dict(affine=True, max_iter=15, check=3)),
    "10x3x75": (10, 3, 75, 1, 1000, dict(affine=True, state_bound=True, check=3)),
    "10x3x76": (10, 3, 76, 2, 1000, dict(affine=True, state_bound=True)),
    "36x5x6": (36, 5, 6, 1, 600, dict(affine=True, linear=(2, 1), adaptive=True)),
    "7x7x12_all": (7, 7, 12, 2, 600, dict(affine=True, state_bound=True, cones=(4, 4), linear=(3, 3), adaptive=True, check=2, max_iter=200)),
}

# fp32 iteration-count flips (one check interval early / late where a residual lands within fp32 rounding of a tolerance),
# measured on a B200 (1000 W): 10x3x75 0/1000, 10x3x76 3/1000, 2x3x8_all 0/1500, 36x5x6 0/600
FLIP_BOUND = {"10x3x75": 0.002, "10x3x76": 0.006, "36x5x6": 0.004, "2x3x8_all": 0.002}


def make(name, B=None):
    nx, nu, N, seed, B0, kw = CASES[name]
    return G.family(nx, nu, N, seed, B or B0, **kw)


def reference(oracle_mod, p, b):
    return oracle_mod.solve_batch(p, b, "ref" if oracle_mod.available("ref") else "port")


def wpp_workspace_floats(nx, nu, N):
    """WppLayout::make (tmpc_wpp.cu): 13 trajectories of states, 13 of inputs, nu scratch, 8 scalars, Kinf, Pinf, rounded to 4"""
    return (13 * nx * N + 13 * nu * (N - 1) + nu + 8 + nu * nx + nx * nx + 3) & ~3


@pytest.fixture(scope="module")
def capi():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return importlib.import_module("tinympc-matlab_b200.capi")


@pytest.fixture(scope="module")
def tm():
    return importlib.import_module("tinympc-matlab_b200")


@pytest.mark.parametrize("name", sorted(CASES))
def test_fp64_batch_matches_the_reference(name, capi, oracle_mod):
    """the run-time-shaped kernel in fp64: the reference's iteration count and status on every problem, x / u to float32
    output rounding, and under adaptive rho the final rho of every problem"""
    p, b = make(name)
    g = reference(oracle_mod, p, b)
    G.assert_nontrivial(p, g, name)
    r = solve_gpu(capi, oracle_mod, p, b, 64)
    assert r["kernel"] == "wpp_f64_generic", r["kernel"]
    flips, dx, du = compare(r, g, 64, name)
    if p.adaptive_rho:
        assert len(np.unique(np.round(g["rho"], 3))) > 5, "the batch does not adapt rho"
        assert np.abs(r["rho"] - g["rho"]).max() <= 1e-5 * max(1.0, float(np.abs(g["rho"]).max())), name
    print(f"\n[generic] {name} fp64: kernel={r['kernel']} median iter {np.median(g['iter'])}, {int((g['status'] == 1).sum())}/{b.size} "
          f"converged, max|dx|={dx:.2e} max|du|={du:.2e}")


def test_fp32_workspace_placement_boundary():
    """10 x 3 x 75 keeps the four workspaces of a CTA in shared memory (<= 200 KiB, tmpc_wpp.cu wpp_launch), 10 x 3 x 76 does
    not: a layout change that moves the boundary shows up here, and the fp32 cases below then no longer cover both sides"""
    lim = 200 * 1024
    assert 4 * wpp_workspace_floats(10, 3, 75) * 4 <= lim < 4 * wpp_workspace_floats(10, 3, 76) * 4


@pytest.mark.parametrize("name", sorted(FLIP_BOUND))
def test_fp32_batch_matches_the_reference(name, capi, oracle_mod):
    """fp32: count flips bounded; on the problems that converged with the reference's count, x / u within 1e-4 absolute scaled
    by max(1, |x|max)"""
    p, b = make(name)
    g = reference(oracle_mod, p, b)
    G.assert_nontrivial(p, g, name)
    r = solve_gpu(capi, oracle_mod, p, b, 32)
    assert r["kernel"] == "wpp_f32_generic", r["kernel"]
    B = b.size
    same = (r["iter"] == g["iter"]) & (r["status"] == g["status"])
    flips = int((~same).sum())
    print(f"\n[generic] {name} fp32: kernel={r['kernel']} {flips}/{B} count flips ({flips / B:.4f})")
    assert flips <= FLIP_BOUND[name] * B, f"{name}: {flips}/{B} iteration/status mismatches"
    conv = same & (g["status"] == 1)
    assert conv.sum() >= 10, f"{name}: {int(conv.sum())} converged problems to compare"
    scale = max(1.0, float(np.abs(g["x"]).max()))
    err = np.maximum(np.abs(r["x"] - g["x"]).reshape(B, -1).max(1), np.abs(r["u"] - g["u"]).reshape(B, -1).max(1))
    assert err[conv].max() <= 1e-4 * scale, f"{name}: {err[conv].max():.3e} on a converged problem"


@pytest.mark.parametrize("name", ["5x2x40_cones", "36x5x6"])
def test_exact_count_option_runs_the_shape_in_fp64(name, capi, oracle_mod, problems):
    """option "mixed" on a shape without a compiled fp32 / fp64 kernel pair: the whole batch runs in fp64, exactly"""
    p, b = make(name)
    g = reference(oracle_mod, p, b)
    r = solve_gpu(capi, oracle_mod, p, b, 32, mixed=problems.exact_band(p))
    assert r["kernel"] == "wpp_f64_generic" and r["marked"] == 0, (r["kernel"], r["marked"])
    compare(r, g, 64, f"{name} exact-count option")


def test_cold_start_reuse_and_batch_position(capi, oracle_mod):
    """more problems than resident warps (16 per SM): a warp cold-starts its next problem in the same scratch workspace
    (zeroed up to zero_end, Kinf / Pinf / rho reloaded).  Under adaptive rho, with cones and linear rows, a permuted batch
    returns the permuted results bit for bit, and a strided sample matches the reference."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 16 * sms * 2 + 101
    nx, nu, N, seed, _, kw = CASES["2x3x8_all"]
    p, b = G.family(nx, nu, N, seed, B, **kw)
    perm = np.random.default_rng(3).permutation(B)
    bp = cases.P.Batch(*(np.ascontiguousarray(a[perm]) for a in (b.x0, b.Xref, b.Uref)))
    r = solve_gpu(capi, oracle_mod, p, b, 64)
    rp = solve_gpu(capi, oracle_mod, p, bp, 64)
    assert r["kernel"] == rp["kernel"] == "wpp_f64_generic"
    for k in ("iter", "status", "x", "u", "rho", "residuals"):
        assert np.array_equal(r[k][perm], rp[k]), f"field {k} depends on the position of the problem in the batch"
    sample = cases.P.Batch(b.x0[::3], b.Xref[::3], b.Uref[::3])
    g = reference(oracle_mod, p, sample)
    G.assert_nontrivial(p, g, "cold-start sample")
    # a few problems of this family that run into max_iter under adaptive rho amplify rounding: a relative change of 1e-15 in A
    # moves their solution by up to ~4e-6.  Those are held to the reference's counts only.
    g2 = reference(oracle_mod, p.with_(A=p.A * (1 + 1e-15)), sample)
    stable = np.abs(g["x"] - g2["x"]).reshape(len(g["x"]), -1).max(1) < 1e-9
    assert stable.mean() > 0.99
    rs = {k: r[k][::3] for k in ("iter", "status", "x", "u", "rho")}
    assert np.array_equal(rs["iter"], g["iter"]) and np.array_equal(rs["status"], g["status"])
    rs = {k: v[stable] for k, v in rs.items()}
    rs["kernel"] = r["kernel"]
    compare(rs, {k: g[k][stable] for k in ("iter", "status", "x", "u")}, 64, "cold-start sample")
    assert np.abs(rs["rho"] - g["rho"][stable]).max() <= 1e-5 * max(1.0, float(np.abs(g["rho"]).max()))


def test_chunked_host_pipeline_and_compact_io(capi, oracle_mod):
    """~70 000 problems of an uncompiled shape through the chunked host pipeline: 5 chunks over the three per-stream scratch
    slots return what one chunk does, in every field; compact I/O (one reference state per problem in, the first control out,
    expanded on the device for this kernel) returns the full-trajectory call's counts and first controls bit for bit"""
    p, b = G.family(3, 2, 10, 5, 70001, affine=True, state_bound=True)
    s = capi.CudaSolver()
    s.set_family(cases.family_from_spec(p, oracle_mod.get_cache(p, "port")))
    s.set_option("chunks", 1)
    r1 = s.solve_batch(b.x0, b.Xref, b.Uref)
    assert s.last_kernel == "wpp_f32_generic" and s.last_timing()["chunks"] == 1, (s.last_kernel, s.last_timing())
    s.set_option("chunks", 5)
    r5 = s.solve_batch(b.x0, b.Xref, b.Uref)
    assert s.last_timing()["chunks"] == 5, s.last_timing()
    for k in ("iter", "status", "x", "u", "residuals", "rho"):
        assert np.array_equal(r1[k], r5[k]), f"chunked pipeline differs in {k}"
    assert (r1["status"] == 1).any() and (r1["status"] != 1).any() and np.median(r1["iter"]) > 4
    full = s.solve_batch(b.x0, b.Xref, None)
    xc = np.ascontiguousarray(b.Xref[:, 0, :])
    for chunks in (1, 5):
        s.set_option("chunks", chunks)
        c = s.solve_batch(b.x0, xref_const=xc, compact_out=True)
        assert s.last_kernel == "wpp_f32_generic", s.last_kernel
        assert np.array_equal(c["iter"], full["iter"]) and np.array_equal(c["status"], full["status"]), chunks
        assert np.array_equal(c["u0"], full["u"][:, 0, :]), chunks
    s.close()


@pytest.mark.parametrize("name", ["36x5x6", "2x3x8_all"])
def test_tiny_solve_warm_start_closed_loop(name, tm, oracle_mod):
    """tiny_solve through the MATLAB-class mirror (explicit_workspace 1, the host mirror's own cache) in a 10-step closed loop
    against a reference solver driven the same way: the same iteration count and status at every step, states and work->u[:, 0]
    within 1e-9"""
    p, b = make(name, B=1)
    s = tm.TinyMPC().setup_from_spec(p)
    ref = oracle_mod.Session(p, "ref" if oracle_mod.available("ref") else "port")
    Xref, Uref = b.Xref[0].astype(np.float64), b.Uref[0].astype(np.float64)
    s.set_x_ref(Xref.T); s.set_u_ref(Uref.T)
    ref.set_x_ref(Xref); ref.set_u_ref(Uref)
    x = b.x0[0].astype(np.float64)
    Bm = np.asarray(p.B).reshape(p.nx, p.nu)
    iters = []
    for k in range(10):
        s.set_x0(x); ref.set_x0(x)
        s.solve()
        g = ref.solve()
        st = s.get_stats()
        assert st["iter"] == g["iter"] and st["status"] == g["status"], (k, st["iter"], g["iter"])
        sc = max(1.0, float(np.abs(g["x"]).max()))
        assert np.abs(s.get_solution()["states"].T - g["x"]).max() < 1e-9 * sc, k
        assert np.abs(s.work_u0() - g["work_u0"]).max() < 1e-9 * sc, k
        iters.append(g["iter"])
        x = p.A @ x + Bm @ g["work_u0"] + p.f
    ref.close()
    assert max(iters) > 4, iters


def test_session_closed_loop_at_an_uncompiled_shape(tm, oracle_mod):
    """{solve; step} for 12 steps on 24 fp64 solvers of an uncompiled shape (nu > nx, linear rows), the step on the
    device: every solver takes the
    iterations, and produces the trajectory, of a reference solver driven the same way"""
    O = oracle_mod
    # well conditioned (a relative change of 1e-15 in A moves the reference's closed loop by < 1e-13; with input cones the loop
    # runs almost every solve into max_iter and amplifies rounding to 1e-1), 59 % of the solves stopped at max_iter
    p, b = G.family(3, 5, 10, 5, 24, affine=True, linear=(1, 1))
    impl = "ref" if O.available("ref") else "port"
    s = tm.TinyMPC().setup_from_spec(p, devices=[0])
    s.cuda.set_option("precision", 64)
    ses = s.cuda.session(24)
    Xref, Uref = b.Xref.astype(np.float64), b.Uref.astype(np.float64)
    ses.set_x_ref(Xref); ses.set_u_ref(Uref)
    xr = b.x0.astype(np.float64)
    ses.set_x0(xr)
    refs = [O.Session(p, impl) for _ in range(24)]
    for k in range(24):
        refs[k].set_x_ref(Xref[k]); refs[k].set_u_ref(Uref[k])
    Bm = np.asarray(p.B).reshape(p.nx, p.nu)
    for t in range(12):
        ses.solve()
        assert s.cuda.last_kernel == "wpp_f64_session", s.cuda.last_kernel
        it, st, sx, wu = ses.read("iter"), ses.read("status"), ses.read("sol_x"), ses.read("u")
        for k in range(24):
            refs[k].set_x0(xr[k])
            r = refs[k].solve()
            assert it[k] == r["iter"] and st[k] == r["status"], (t, k, it[k], r["iter"])
            assert np.abs(sx[k] - r["x"]).max() < 1e-8 * max(1.0, np.abs(r["x"]).max())
            assert np.abs(wu[k, 0] - r["work_u0"]).max() < 1e-8 * max(1.0, np.abs(r["work_u0"]).max())
            xr[k] = p.A @ xr[k] + Bm @ r["work_u0"] + p.f
        ses.step()
        assert np.abs(ses.read("x0") - xr).max() < 1e-8 * max(1.0, np.abs(xr).max())
    for r in refs:
        r.close()
    ses.close()


def test_session_step_rejects_more_than_32_states(tm, capi, oracle_mod):
    """the device step gives each state one lane: with nx = 36 it returns TINYMPC_CUDA_EUNSUPPORTED with a message naming the
    limit, leaves x0 and the caller's current device as they were, and the session still solves like the reference"""
    import torch
    p, b = make("36x5x6", B=8)
    s = tm.TinyMPC().setup_from_spec(p, devices=[0])
    s.cuda.set_option("precision", 64)
    ses = s.cuda.session(8)
    ses.set_x_ref(b.Xref.astype(np.float64)); ses.set_u_ref(b.Uref.astype(np.float64))
    ses.set_x0(b.x0.astype(np.float64))
    x0 = ses.read("x0")
    dev = torch.cuda.device_count() - 1          # a current device other than the session's where there is one
    torch.cuda.set_device(dev)
    try:
        assert ses.L.tinympc_cuda_session_step(ses.h, 0) == 4
        assert torch.cuda.current_device() == dev
    finally:
        torch.cuda.set_device(0)
    msg = ses.L.tinympc_cuda_last_error(s.cuda.h).decode()
    assert "nx <= 32" in msg, msg
    with pytest.raises(capi.TinympcCudaError):
        ses.step()
    assert np.array_equal(ses.read("x0"), x0)
    ses.solve()
    g = reference(oracle_mod, p, b)
    assert np.array_equal(ses.read("iter").astype(np.int32), g["iter"]) and np.array_equal(ses.read("status").astype(np.int32), g["status"])
    assert np.abs(ses.read("sol_x") - g["x"]).max() < 1e-8 * max(1.0, float(np.abs(g["x"]).max()))
    ses.close()


# ---- batched cache precompute (tinympc_cuda_precompute_batch) --------------------------------------------------------------------
def precompute_inputs(nx, nu, n, seed):
    rng = np.random.default_rng(seed)
    A = np.array([G.dynamics(nx, nu, rng)[0] for _ in range(n)])
    A *= rng.uniform(0.5, 0.9, (n, 1, 1)) / np.abs(np.linalg.eigvals(A)).max(1)[:, None, None]
    # stable dynamics and inputs of magnitude 0.05-0.15: a marginally controllable pair (a single input into 16 states, a near-zero
    # B) leaves the recursion thousands of iterations from its fixed point, where the 1e-10 stop of the sensitivity recursion is
    # no longer small against the forward-difference step of 1e-6
    B = 0.1 * rng.uniform(0.5, 1.5, (n, nx, nu)) * rng.choice([-1.0, 1.0], (n, nx, nu))
    Q, R, rho = rng.uniform(1.0, 10.0, (n, nx)), rng.uniform(0.1, 1.0, (n, nu)), rng.uniform(0.5, 5.0, n)
    return A, B, Q, R, rho, 0.05 * rng.standard_normal((n, nx))


def check_cache(o, A, B, Q, R, rho, f, idx, oracle_mod, name):
    """tiny_setup hands Q + rho to the precompute, which adds rho again (SURVEY quirk Q1): o was computed from Q + rho"""
    nx, nu = A.shape[1], B.shape[2]
    for b in idx:
        p = cases.P.ProblemSpec("pre", nx, nu, 2, A[b], B[b], f[b], Q[b], R[b], float(rho[b]))
        g = oracle_mod.get_cache(p, "port")
        for k in ("Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf"):
            ref = np.asarray(g[k]).reshape(o[k][b].shape)
            err = np.abs(o[k][b] - ref).max() / max(1.0, np.abs(ref).max())
            assert err < 1e-9, f"{name} problem {b}: {k} differs by {err:.2e} (relative)"


@pytest.mark.parametrize("nx,nu", [(1, 1), (2, 3), (3, 8), (16, 1), (16, 8)])
def test_precompute_batch_at_generic_shapes(nx, nu, capi, oracle_mod):
    """per-problem (A, B, f, Q, R, rho) at shapes up to the nx <= 16, nu <= 8 limit (16 x 8: 70 KB of shared memory per CTA),
    nu > nx among them: the cache against the reference's recursion, the rho-sensitivities against a forward difference of
    scipy's DARE solution"""
    n = 16
    A, B, Q, R, rho, f = precompute_inputs(nx, nu, n, seed=nx * 100 + nu)
    Qr, Rr = Q + rho[:, None], R + rho[:, None]
    o = capi.precompute_batch(A, B, Qr, Rr, rho, f)
    check_cache(o, A, B, Q, R, rho, f, range(n), oracle_mod, f"{nx}x{nu}")
    os_ = capi.precompute_batch(A, B, Qr, Rr, rho, f, sensitivities=True)
    for k in ("Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf"):
        assert np.array_equal(o[k], os_[k]), k
    h = 1e-6
    for b in range(n):
        lo = G.lqr(A[b], B[b], Qr[b] + rho[b], Rr[b] + rho[b])
        hi = G.lqr(A[b], B[b], Qr[b] + rho[b] + h, Rr[b] + rho[b] + h)
        for k, i in (("dKinf", 0), ("dPinf", 1), ("dC1", 2), ("dC2", 3)):
            ref = (hi[i] - lo[i]) / h
            err = np.abs(os_[k][b] - ref).max() / max(1e-12, np.abs(ref).max())
            assert err < 5e-3, f"{nx}x{nu} problem {b}: {k} differs by {err:.2e} (relative to its largest entry)"
    assert (o["iters"] > 1).all() and (o["iters"] <= 1000).all()


def test_precompute_large_batch_and_limits(capi, oracle_mod):
    """~5 000 problems: every warp runs the recursion for several problems in its shared-memory slot; a strided subset against
    the reference.  Shapes beyond nx <= 16, nu <= 8 are rejected with EINVAL."""
    nx, nu, n = 16, 8, 5003
    A, B, Q, R, rho, f = precompute_inputs(nx, nu, n, seed=7)
    o = capi.precompute_batch(A, B, Q + rho[:, None], R + rho[:, None], rho, f)
    check_cache(o, A, B, Q, R, rho, f, range(0, n, 97), oracle_mod, "large batch")
    for nx, nu in ((17, 1), (2, 9)):
        A, B, Q, R, rho, f = precompute_inputs(nx, nu, 2, seed=1)
        with pytest.raises(capi.TinympcCudaError) as e:
            capi.precompute_batch(A, B, Q, R, rho, f)
        assert e.value.code == 1, e.value
