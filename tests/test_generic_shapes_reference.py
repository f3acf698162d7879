"""CPU tests of the checker at shapes other than the shipped ones: before the oracle's C restatement (oracle/tinympc_oracle.c,
"port") serves as the reference of tests/test_gpu_generic_shapes.py, its cache and its solve are checked against independent
dense computations at those shapes -- and first at the three shipped shapes, where the port is known to match the reference.

Unconstrained solve.  With nothing to project, update_slack gives vnew = x + g and update_dual g <- g + x - vnew = 0, so from
the first iteration on g = y = 0 and at the fixed point v = x, z = u.  update_linear_cost (admm.cpp:214-247) then builds, with
work->Q = Qdiag + rho and work->R = Rdiag + rho (tiny_api.cpp:107-108),
    q_i = -Q xr_i - rho x_i,   r_i = -R ur_i - rho u_i,   p_{N-1} = -Pinf' xr_{N-1} - rho x_{N-1},
and backward_pass_grad / forward_pass (admm.cpp:13-32) close the loop:
    d_i = Quu_inv (B' p_{i+1} + r_i + BPf),   p_i = q_i + AmBKt p_{i+1} - Kinf' r_i + APf,   (i = N-2 .. 0)
    u_i = -Kinf x_i - d_i,                    x_{i+1} = A x_i + B u_i + f,                   x_0 = x0.
These are 2 N nx + 2 (N-1) nu linear equations in (x, u, d, p): `fixed_point` solves them densely.
When the cache is the exact infinite-horizon solution of (A, B, Q + rho, R + rho) -- Pinf the DARE solution, Quu_inv =
(R + rho + B' Pinf B)^-1, Kinf = Quu_inv B' Pinf A, AmBKt = (A - B Kinf)', APf = AmBKt Pinf f, BPf = B' Pinf f -- the pass
above is the dynamic programme (Riccati form) of the equality-constrained QP whose stage Hessians are Q + rho, R + rho and whose
cost-to-go at step N-1 is Pinf, with the linear terms q_i, r_i, p_{N-1}.  Its stationarity conditions with q, r, p substituted are
    (Q + rho) x_i - Q xr_i - rho x_i = Q (x_i - xr_i)              for 1 <= i <= N-2,
    (R + rho) u_i - R ur_i - rho u_i = R (u_i - ur_i)              for 0 <= i <= N-2,
    Pinf x_{N-1} - Pinf' xr_{N-1} - rho x_{N-1},
plus the multiplier terms, i.e. the ADMM fixed point minimises
    sum_{i=1}^{N-2} 1/2 (x_i - xr_i)' Q (x_i - xr_i) + sum_{i=0}^{N-2} 1/2 (u_i - ur_i)' R (u_i - ur_i)
        + 1/2 x_{N-1}' (Pinf - rho I) x_{N-1} - (Pinf' xr_{N-1})' x_{N-1}
subject to x_0 = x0, x_{i+1} = A x_i + B u_i + f: `dense_qp` solves its KKT system with numpy.linalg.solve.
The cache the solver actually holds stops the Riccati recursion at max|Kinf - Kinf_prev| < 1e-5 (tiny_api.cpp:277), which
leaves it up to ~1e-4 (relative) away from the DARE solution at these shapes; the port is therefore held to the fixed point of
its own cache at 1e-6, and the identity fixed point == QP minimiser is checked with an exact DARE cache at 1e-9.
"""
import numpy as np
import pytest

import cases
import generic_families as G

P = cases.P

# the shapes of tests/test_gpu_generic_shapes.py
SHAPES = [(1, 1, 2), (2, 3, 8), (5, 2, 40), (10, 3, 75), (10, 3, 76), (36, 5, 6), (7, 7, 12)]


def shipped(name):
    return dict(cartpole=P.cartpole, quadrotor=P.quadrotor, rocket=P.rocket)[name]()


def spec_and_batch(case, B=6):
    if isinstance(case, str):
        p = shipped(case)
        b = P.make_batch(p, B, 1.0, seed=3)
    else:
        p, b = G.family(*case, seed=sum(case), B=B, affine=True)
    return p, b


def unconstrained(p):
    return p.with_(en_state_bound=0, en_input_bound=0, en_state_soc=0, en_input_soc=0, en_state_linear=0, en_input_linear=0,
                   adaptive_rho=0, sens_mode=0, abs_pri_tol=1e-9, abs_dua_tol=1e-9, max_iter=20000, check_termination=1)


def refs(p, b, k):
    Xr = b.Xref[k].astype(np.float64) if b.Xref is not None else np.zeros((p.N, p.nx))
    Ur = b.Uref[k].astype(np.float64) if b.Uref is not None else np.zeros((p.N - 1, p.nu))
    return b.x0[k].astype(np.float64), Xr, Ur


def exact_cache(p):
    Bm = np.asarray(p.B).reshape(p.nx, p.nu)
    K, Pinf, S, AK = G.lqr(p.A, Bm, p.Qdiag + 2 * p.rho, p.Rdiag + 2 * p.rho)
    return dict(Kinf=K, Pinf=Pinf, Quu_inv=S, AmBKt=AK, APf=AK @ Pinf @ p.f, BPf=Bm.T @ Pinf @ p.f)


def fixed_point(p, c, x0, Xr, Ur):
    """the ADMM fixed point of an unconstrained solve: the update equations of the module docstring, solved densely"""
    nx, nu, N, rho = p.nx, p.nu, p.N, p.rho
    Bm, A = np.asarray(p.B).reshape(nx, nu), p.A
    Qw, Rw = np.diag(p.Qdiag + rho), np.diag(p.Rdiag + rho)
    K, S, AK, Pinf = c["Kinf"], c["Quu_inv"], c["AmBKt"], c["Pinf"]
    nX, nU = nx * N, nu * (N - 1)
    X = lambda i: slice(i * nx, (i + 1) * nx)
    U = lambda i: slice(nX + i * nu, nX + (i + 1) * nu)
    D = lambda i: slice(nX + nU + i * nu, nX + nU + (i + 1) * nu)
    Pp = lambda i: slice(nX + 2 * nU + i * nx, nX + 2 * nU + (i + 1) * nx)
    n = 2 * nX + 2 * nU
    M, rhs, row = np.zeros((n, n)), np.zeros(n), [0]

    def eq(terms, b):
        r = slice(row[0], row[0] + len(b))
        for cols, m in terms:
            M[r, cols] += m
        rhs[r] = b
        row[0] += len(b)

    I, Iu = np.eye(nx), np.eye(nu)
    eq([(X(0), I)], x0)
    for i in range(N - 1):
        eq([(X(i + 1), I), (X(i), -A), (U(i), -Bm)], p.f)                                       # forward_pass, x
        eq([(U(i), Iu), (X(i), K), (D(i), Iu)], np.zeros(nu))                                  # forward_pass, u
        eq([(D(i), Iu), (Pp(i + 1), -S @ Bm.T), (U(i), rho * S)], S @ (c["BPf"] - Rw @ Ur[i]))  # d with r substituted
        eq([(Pp(i), I), (X(i), rho * I), (Pp(i + 1), -AK), (U(i), -rho * K.T)], c["APf"] - Qw @ Xr[i] + K.T @ Rw @ Ur[i])
    eq([(Pp(N - 1), I), (X(N - 1), rho * I)], -Pinf.T @ Xr[N - 1])                            # terminal linear cost
    z = np.linalg.solve(M, rhs)
    return z[:nX].reshape(N, nx), z[nX:nX + nU].reshape(N - 1, nu)


def dense_qp(p, Pinf, x0, Xr, Ur):
    """minimiser of the QP of the module docstring: its KKT system, solved densely"""
    nx, nu, N, rho = p.nx, p.nu, p.N, p.rho
    Bm = np.asarray(p.B).reshape(nx, nu)
    Qw, Rw = np.diag(p.Qdiag + rho), np.diag(p.Rdiag + rho)
    nX, nz = nx * N, nx * N + nu * (N - 1)
    X = lambda i: slice(i * nx, (i + 1) * nx)
    U = lambda i: slice(nX + i * nu, nX + (i + 1) * nu)
    H, h = np.zeros((nz, nz)), np.zeros(nz)
    for i in range(N - 1):
        H[X(i), X(i)], h[X(i)] = Qw, -Qw @ Xr[i]      # (the x_0 block is fixed by its constraint)
        H[U(i), U(i)], h[U(i)] = Rw, -Rw @ Ur[i]
    H[X(N - 1), X(N - 1)], h[X(N - 1)] = Pinf - rho * np.eye(nx), -Pinf.T @ Xr[N - 1]
    C, d = np.zeros((nX, nz)), np.zeros(nX)
    C[X(0), X(0)], d[X(0)] = np.eye(nx), x0
    for i in range(N - 1):
        C[X(i + 1), X(i + 1)], C[X(i + 1), X(i)], C[X(i + 1), U(i)], d[X(i + 1)] = np.eye(nx), -p.A, -Bm, p.f
    z = np.linalg.solve(np.block([[H, C.T], [C, np.zeros((nX, nX))]]), np.concatenate([-h, d]))
    return z[:nX].reshape(N, nx), z[nX:nz].reshape(N - 1, nu)


CASES = ["cartpole", "quadrotor", "rocket"] + SHAPES
IDS = lambda c: c if isinstance(c, str) else "x".join(map(str, c))


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_port_cache_matches_the_dare_solution(case, oracle_mod):
    """get_cache(p, "port") against scipy's DARE on (Qdiag + 2 rho, Rdiag + 2 rho).  The recursion stops when Kinf moves by
    less than 1e-5 in one step, which leaves it up to ~1.4e-4 (relative to the largest entry) short of the fixed point here."""
    p, _ = spec_and_batch(case)
    c, e = oracle_mod.get_cache(p, "port"), exact_cache(p)
    for k in ("Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf"):
        err = np.abs(np.asarray(c[k]).reshape(e[k].shape) - e[k]).max() / max(1.0, np.abs(e[k]).max())
        assert err < 5e-4, f"{IDS(case)}: {k} differs from the DARE solution by {err:.2e} (relative)"


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_fixed_point_is_the_qp_minimiser(case):
    """with an exact DARE cache the fixed-point equations of the ADMM updates and the KKT system of the QP have one solution"""
    p, b = spec_and_batch(case, B=2)
    c = exact_cache(p)
    for k in range(b.size):
        x0, Xr, Ur = refs(p, b, k)
        xf, uf = fixed_point(p, c, x0, Xr, Ur)
        xq, uq = dense_qp(p, c["Pinf"], x0, Xr, Ur)
        sc = max(1.0, np.abs(xq).max(), np.abs(uq).max())
        assert max(np.abs(xf - xq).max(), np.abs(uf - uq).max()) < 1e-9 * sc


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_port_unconstrained_solve_reaches_the_dense_solution(case, oracle_mod):
    """the port at abs_pri_tol = abs_dua_tol = 1e-9 converges to the dense fixed point of its own cache within 1e-6 and to the QP
    minimiser of the exact cache within the cache's own distance from it"""
    p, b = spec_and_batch(case)
    q = unconstrained(p)
    c = oracle_mod.get_cache(q, "port")
    g = oracle_mod.solve_batch(q, b, "port")
    assert (g["status"] == 1).all() and (g["iter"] > 5).all(), g["iter"]
    pq = exact_cache(q)["Pinf"]
    for k in range(b.size):
        x0, Xr, Ur = refs(q, b, k)
        xf, uf = fixed_point(q, c, x0, Xr, Ur)
        sc = max(1.0, np.abs(xf).max(), np.abs(uf).max())
        err = max(np.abs(g["x"][k] - xf).max(), np.abs(g["u"][k] - uf).max()) / sc
        assert err < 1e-6, f"{IDS(case)} problem {k}: {err:.2e} from the fixed point of the port's cache"
        xq, uq = dense_qp(q, pq, x0, Xr, Ur)
        err = max(np.abs(g["x"][k] - xq).max(), np.abs(g["u"][k] - uq).max()) / sc
        assert err < 1e-3, f"{IDS(case)} problem {k}: {err:.2e} from the QP minimiser"
