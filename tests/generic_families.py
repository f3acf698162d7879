"""Seeded random problem families of any shape (nx, nu, N) and feature mix, for the tests of the shapes that have no
compiled thread-per-problem kernel (the run-time-shaped warp-per-problem kernel) and of the batched cache precompute.

The same ProblemSpec and the same float32 batch go to the CPU oracle and to the GPU; the cache the GPU gets is the
oracle port's (oracle_mod.get_cache(p, "port")), as in the other parity tests."""
import numpy as np
from scipy.linalg import solve_discrete_are

import cases

P = cases.P

# (nx, nu) pairs with compiled kernel instances (tmpc_wpp.cu wpp_launch, the thread-per-problem tables): never used here
COMPILED_SHAPES = {(12, 4), (4, 1), (6, 3)}


def dynamics(nx, nu, rng, dt=0.1):
    """A = I + dt M scaled to a spectral radius in [1.0, 1.05] (marginally unstable open loop), B = dt * randn"""
    A0 = np.eye(nx) + dt * rng.standard_normal((nx, nx)) / np.sqrt(nx)
    A = A0 * (rng.uniform(1.0, 1.05) / np.abs(np.linalg.eigvals(A0)).max())
    return A, dt * rng.standard_normal((nx, nu))


def lqr(A, B, Qd, Rd):
    """converged infinite-horizon LQR of (A, B, diag Qd, diag Rd): Kinf, Pinf, Quu_inv, AmBKt"""
    P_ = solve_discrete_are(A, B, np.diag(Qd), np.diag(Rd))
    S = np.diag(Rd) + B.T @ P_ @ B
    K = np.linalg.solve(S, B.T @ P_ @ A)
    return K, P_, np.linalg.inv(S), (A - B @ K).T


def sensitivities(A, B, Qd, Rd, rho, h=1e-6):
    """d/drho of (Kinf, Pinf, Quu_inv, AmBKt) of the cache the solver holds (Q + 2 rho, R + 2 rho, SURVEY quirk Q1), by a
    forward difference of scipy's DARE solution (what TinyMPC.m:223-241 does with idare)"""
    lo, hi = lqr(A, B, Qd + 2 * rho, Rd + 2 * rho), lqr(A, B, Qd + 2 * (rho + h), Rd + 2 * (rho + h))
    return [(b - a) / h for a, b in zip(lo, hi)]


def cone_list(n, k, rng):
    """k cones (offset, dim) inside [0, n): the first ends at the last component (at a non-zero offset when n > 1), the
    second has dimension 1, the others start and end anywhere; apertures mu in [1, 3]"""
    A, q = [], []
    for j in range(k):
        if j == 0:
            d = int(rng.integers(1, n)) if n > 1 else 1
            a = n - d
        elif j == 1:
            d, a = 1, int(rng.integers(0, n))
        else:
            a = int(rng.integers(0, n))
            d = int(rng.integers(1, n - a + 1))
        A.append(a)
        q.append(d)
    return np.array(A, np.int32), np.array(q, np.int32), rng.uniform(1.0, 3.0, k)


def family(nx, nu, N, seed, B, *, affine=False, input_bound=True, state_bound=False, cones=(0, 0), linear=(0, 0),
           adaptive=False, check=1, max_iter=100, refs=True, xscale=1.0):
    """(ProblemSpec, Batch) of B problems of a random family.

    Costs: Qdiag in [1, 10], Rdiag in [0.1, 1], rho in [0.5, 5].  affine: a non-zero f (so APf, BPf are non-zero).
    input_bound: |u| <= the median over the batch of max_a |Kinf x0|_a, so that about half of the problems start on it.
    state_bound: |x_c| <= the 0.95 quantile of |x0_c| over the batch, so that some problems start outside the box.
    cones = (state, input) cone counts (0-4), linear = (state, input) half-space row counts (a x <= 2 |a| xscale,
    a u <= |a| * the input bound), adaptive: adaptive rho with
    explicit sensitivities (sens_mode 2).  refs: a random reference state held over the horizon and a random Uref."""
    assert (nx, nu) not in COMPILED_SHAPES
    rng = np.random.default_rng(seed)
    A, Bm = dynamics(nx, nu, rng)
    f = 0.05 * rng.standard_normal(nx) if affine else np.zeros(nx)
    Qd, Rd, rho = rng.uniform(1.0, 10.0, nx), rng.uniform(0.1, 1.0, nu), float(rng.uniform(0.5, 5.0))
    p = P.ProblemSpec(f"random_{nx}x{nu}x{N}", nx, nu, N, A, Bm, f, Qd, Rd, rho, max_iter=max_iter, check_termination=check)
    x0 = xscale * rng.standard_normal((B, nx))
    if cones[0]:
        # x0 is not free: a problem whose x0 lies outside a state cone never converges, so the axis of every state cone is
        # made non-negative in x0 (the problems whose x0 still lies outside the cone are the non-converging part of the batch)
        p.Acx, p.qcx, p.cx = cone_list(nx, cones[0], rng)
        p.en_state_soc = 1
        x0[:, p.Acx + p.qcx - 1] = np.abs(x0[:, p.Acx + p.qcx - 1])
    Xref = Uref = None
    if refs:
        Xref = np.repeat((0.2 * xscale * rng.standard_normal((B, 1, nx))), N, axis=1)
        Uref = 0.05 * rng.standard_normal((B, N - 1, nu))
    K = lqr(A, Bm, Qd + 2 * rho, Rd + 2 * rho)[0]
    ub = float(np.median(np.abs(x0 @ K.T).max(1)))
    if input_bound or state_bound:
        xb = np.quantile(np.abs(x0), 0.95, axis=0) if state_bound else np.full(nx, 1e17)
        p.x_min, p.x_max = np.tile(-xb, (N, 1)), np.tile(xb, (N, 1))
        u = ub if input_bound else 1e17
        p.u_min, p.u_max = np.full((N - 1, nu), -u), np.full((N - 1, nu), u)
        p.en_state_bound, p.en_input_bound = int(state_bound), int(input_bound)
    if cones[1]:
        p.Acu, p.qcu, p.cu = cone_list(nu, cones[1], rng)
        p.en_input_soc = 1
    if linear[0]:
        p.Alin_x = rng.standard_normal((linear[0], nx))
        p.blin_x = 2 * xscale * np.linalg.norm(p.Alin_x, axis=1)
        p.en_state_linear = 1
    if linear[1]:
        p.Alin_u = rng.standard_normal((linear[1], nu))
        p.blin_u = ub * np.linalg.norm(p.Alin_u, axis=1)
        p.en_input_linear = 1
    if adaptive:
        p.adaptive_rho, p.sens_mode = 1, 2
        p.dKinf, p.dPinf, p.dC1, p.dC2 = sensitivities(A, Bm, Qd, Rd, rho)
    f32 = lambda a: None if a is None else np.ascontiguousarray(a, np.float32)
    return p, P.Batch(f32(x0), f32(Xref), f32(Uref))


def assert_nontrivial(p, g, name, min_median_iter=4):
    """a batch a test may pass on: some problems converge and some do not, the median iteration count is above a few, and
    where the input bound is on, some u of the solution sits on it"""
    conv = g["status"] == 1
    assert conv.any() and not conv.all(), f"{name}: {int(conv.sum())}/{len(conv)} problems converge"
    assert np.median(g["iter"]) > min_median_iter, f"{name}: median iteration count {np.median(g['iter'])}"
    if p.en_input_bound:
        assert (np.abs(g["u"]) == p.u_max[0, 0]).any(), f"{name}: no control on its bound"
