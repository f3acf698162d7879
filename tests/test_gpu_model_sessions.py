"""GPU tests of model sessions (tinympc_cuda_session_create_models / _set_models): closed-loop sessions of warm-started solvers in
which every solver carries its own dynamics, costs and cache.

The reference of a model session is one reference session per solver, built from that solver's spec and driven through the same
closed loop {set_x0; solve; x0 = A_b x0 + B_b u0 + f_b}.  What is checked:
  * identity: a session whose every solver carries the family's model and cache reproduces the family session bit for bit, after
    every solve and every step, on the session form of the lane-group model kernel and on the warp-per-problem kernel;
  * parity with the reference on distinct quadrotor models (fp64: exact iteration counts), with adaptive rho, on a random shape
    with cones, rows and an affine term, and in fp32 within the fp32 tolerance; that the parity test can fail;
  * set_models mid-loop against reference sessions whose model is replaced the same way; set_models with the models a session
    already has changes nothing; on an adaptive-rho session it resets the rho adaptive rho has moved;
  * the EINVAL cases.
"""
import importlib

import numpy as np
import pytest

import cases
import generic_families as G
from model_sessions_ref import SESSION_FIELDS, SwapSession, read_all, reference_loop
from test_gpu_model_batches import model_of, quadrotor_models, stack

pytestmark = pytest.mark.gpu

STEPS = 12


@pytest.fixture(scope="module")
def capi():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return importlib.import_module("tinympc-matlab_b200.capi")


@pytest.fixture(scope="module")
def problems():
    return importlib.import_module("tinympc-matlab_b200.problems")


def impl_of(oracle_mod):
    return "ref" if oracle_mod.available("ref") else "port"


def solver(capi, p, cache, precision, force_wpp=0):
    s = capi.CudaSolver()
    s.set_option("precision", precision)
    s.set_option("force_wpp", force_wpp)
    s.set_family(cases.family_from_spec(p, cache))
    return s


def refs_of(b, p, B):
    Xref = b.Xref[:B].astype(np.float64) if b.Xref is not None else np.zeros((B, p.N, p.nx))
    Uref = b.Uref[:B].astype(np.float64) if b.Uref is not None else np.zeros((B, p.N - 1, p.nu))
    return Xref, Uref


def start(ses, x0, Xref, Uref):
    ses.set_x_ref(Xref)
    ses.set_u_ref(Uref)
    ses.set_x0(x0)


def gpu_loop(s, ses, steps, before_solve=None):
    """the closed loop on the device: per step, every session field after the solve and x0 after the step, and the kernel"""
    out = []
    for t in range(steps):
        if before_solve:
            before_solve(t)
        ses.solve()
        r = read_all(ses)
        r["kernel"] = s.last_kernel
        ses.step()
        r["x0_next"] = ses.read("x0")
        out.append(r)
    return out


def reference_sessions(oracle_mod, specs, Xref, Uref, impl=None):
    impl = impl or impl_of(oracle_mod)
    out = []
    for k, p in enumerate(specs):
        r = oracle_mod.Session(p, impl) if impl != "swap" else SwapSession(p)
        r.set_x_ref(Xref[k])
        r.set_u_ref(Uref[k])
        out.append(r)
    return out


def assert_tracks_reference(gl, rl, specs, exact=True, tol=1e-8, what=""):
    for t, (r, g) in enumerate(zip(gl, rl)):
        if exact:
            assert np.array_equal(r["iter"], g["iter"]) and np.array_equal(r["status"], g["status"]), \
                (what, t, np.flatnonzero(r["iter"] != g["iter"]), r["iter"], g["iter"])
            scale = max(1.0, float(np.abs(g["sol_x"]).max()))
            assert np.abs(r["sol_x"] - g["sol_x"]).max() <= tol * scale, (what, t)
            assert np.abs(r["u"][:, 0] - g["work_u0"]).max() <= tol * max(1.0, float(np.abs(g["work_u0"]).max())), (what, t)
            # the device step with each solver's own model, from the device's own u0
            own = np.stack([p.A @ r["x0"][k] + np.asarray(p.B).reshape(p.nx, p.nu) @ r["u"][k, 0] + p.f for k, p in enumerate(specs(t))])
            assert np.abs(r["x0_next"] - own).max() <= tol * max(1.0, float(np.abs(own).max())), (what, t)
        else:
            assert np.abs(r["sol_x"] - g["sol_x"]).max() < tol, (what, t)
            assert np.abs(r["x0_next"] - g["x0"]).max() < tol, (what, t)


# ---- 1. identity with family sessions -------------------------------------------------------------------------------------------
def _case(problems, name):
    if name == "quadrotor":
        p = problems.quadrotor()
    elif name == "cartpole10":
        p = problems.cartpole(N=10)
    elif name == "cartpole20":
        p = problems.cartpole(N=20)
    elif name == "rocket":
        p = problems.rocket()
    elif name == "quadrotor_adaptive":
        p = problems.quadrotor(adaptive=True)
    else:
        return G.family(*name, seed=3, B=48, affine=True, state_bound=True, cones=(2, 1), linear=(1, 1), adaptive=True, check=2)
    return p, problems.make_batch(p, 48, 0.6, seed=11)


@pytest.mark.parametrize("name, precision, force_wpp, kernel", [
    ("quadrotor", 64, 0, "gpp_f64_12x4x10_box_g16_v0"),
    ("cartpole10", 64, 0, "gpp_f64_4x1x10_box_g8_v0"),
    ("cartpole20", 64, 0, "gpp_f64_4x1x20_box_g8_v0"),
    ("rocket", 64, 0, "wpp_f64"),
    ("quadrotor_adaptive", 64, 0, "wpp_f64"),
    ("quadrotor", 32, 0, "wpp_f32"),
    ((5, 2, 12), 32, 0, "wpp_f32"),
    ((5, 2, 12), 64, 0, "wpp_f64"),
    ("quadrotor", 64, 1, "wpp_f64"),
], ids=["quadrotor_gpp", "cartpole10_gpp", "cartpole20_gpp", "rocket_wpp", "adaptive_wpp", "quadrotor_wpp32", "generic_wpp32",
        "generic_wpp64", "quadrotor_force_wpp"])
def test_family_model_everywhere_is_bit_identical_to_the_family_session(name, precision, force_wpp, kernel, capi, oracle_mod, problems):
    p, b = _case(problems, name)
    cache = oracle_mod.get_cache(p, "port")
    B = 40
    Xref, Uref = refs_of(b, p, B)
    x0 = b.x0[:B].astype(np.float64)
    s = solver(capi, p, cache, precision, force_wpp)
    fam = s.session(B)
    start(fam, x0, Xref, Uref)
    gf = gpu_loop(s, fam, STEPS)
    mdl = s.session(B, models=stack([model_of(p, cache)], np.zeros(B, int)))
    start(mdl, x0, Xref, Uref)
    gm = gpu_loop(s, mdl, STEPS)
    for t, (a, c) in enumerate(zip(gm, gf)):
        for k in SESSION_FIELDS + ("x0_next",):
            assert np.array_equal(a[k], c[k]), f"{name}: step {t}: {k} differs ({a['kernel']} against {c['kernel']})"
    assert gf[0]["kernel"] == kernel + "_session" and gm[0]["kernel"] == kernel + "_mdl_session", (gf[0]["kernel"], gm[0]["kernel"])
    if force_wpp:   # the warp-per-problem kernel takes the lane-group kernel's counts
        s2 = solver(capi, p, cache, precision, 0)
        m2 = s2.session(B, models=stack([model_of(p, cache)], np.zeros(B, int)))
        start(m2, x0, Xref, Uref)
        g2 = gpu_loop(s2, m2, STEPS)
        assert g2[0]["kernel"] == "gpp_f64_12x4x10_box_g16_v0_mdl_session"
        for a, c in zip(g2, gm):
            assert np.array_equal(a["iter"], c["iter"]) and np.array_equal(a["status"], c["status"])
        m2.close(); s2.close()
    fam.close(); mdl.close(); s.close()


# ---- 2. distinct models against the reference -----------------------------------------------------------------------------------
B_DISTINCT, K_DISTINCT = 48, 16


def _distinct(problems, oracle_mod, adaptive=False, k=K_DISTINCT, seed=0):
    specs = quadrotor_models(problems, k=k, seed=seed)
    if adaptive:
        for p in specs:
            p.adaptive_rho, p.sens_mode = 1, 1
    caches = [oracle_mod.get_cache(p, "port") for p in specs]
    return specs, caches


def _model_session(capi, specs, caches, which, precision, x0, Xref, Uref, force_wpp=0):
    s = solver(capi, specs[0], caches[0], precision, force_wpp)
    ses = s.session(len(which), models=stack([model_of(p, c) for p, c in zip(specs, caches)], which))
    start(ses, x0, Xref, Uref)
    return s, ses


@pytest.fixture(scope="module")
def distinct_case(problems, oracle_mod):
    specs, caches = _distinct(problems, oracle_mod)
    which = np.arange(B_DISTINCT) % K_DISTINCT                # neighbours carry different models
    b = problems.make_batch(specs[0], B_DISTINCT, 0.6, seed=21)
    Xref, Uref = refs_of(b, specs[0], B_DISTINCT)
    x0 = b.x0.astype(np.float64)
    per = [specs[j] for j in which]
    rl = reference_loop(reference_sessions(oracle_mod, per, Xref, Uref), lambda t: per, x0, STEPS)
    return specs, caches, which, x0, Xref, Uref, rl


@pytest.mark.parametrize("force_wpp", [0, 1], ids=["gpp", "wpp"])
def test_distinct_models_match_the_reference(force_wpp, distinct_case, capi):
    specs, caches, which, x0, Xref, Uref, rl = distinct_case
    s, ses = _model_session(capi, specs, caches, which, 64, x0, Xref, Uref, force_wpp)
    gl = gpu_loop(s, ses, STEPS)
    assert gl[0]["kernel"] == ("wpp_f64_mdl_session" if force_wpp else "gpp_f64_12x4x10_box_g16_v0_mdl_session")
    per = [specs[j] for j in which]
    assert_tracks_reference(gl, rl, lambda t: per, what="distinct")
    assert np.array_equal(gl[-1]["rho"], np.array([p.rho for p in per]))
    ses.close(); s.close()


def test_the_distinct_model_test_can_fail(distinct_case, oracle_mod):
    """reference sessions that all carry model 0 take other iteration counts on a sizeable share of the steps"""
    specs, caches, which, x0, Xref, Uref, rl = distinct_case
    per0 = [specs[0]] * len(which)
    r0 = reference_loop(reference_sessions(oracle_mod, per0, Xref, Uref), lambda t: per0, x0, STEPS)
    differ = np.mean([np.mean(a["iter"] != c["iter"]) for a, c in zip(r0, rl)])
    assert differ > 0.1, differ


# ---- 3. adaptive rho with distinct models -----------------------------------------------------------------------------------------
def test_adaptive_rho_with_distinct_models(problems, oracle_mod, capi):
    specs, caches = _distinct(problems, oracle_mod, adaptive=True, k=8, seed=4)
    B = 24
    which = np.arange(B) % len(specs)
    b = problems.make_batch(specs[0], B, 0.6, seed=23)
    Xref, Uref = refs_of(b, specs[0], B)
    x0 = b.x0.astype(np.float64)
    per = [specs[j] for j in which]
    rl = reference_loop(reference_sessions(oracle_mod, per, Xref, Uref, impl="swap"), lambda t: per, x0, STEPS)
    s, ses = _model_session(capi, specs, caches, which, 64, x0, Xref, Uref)
    gl = gpu_loop(s, ses, STEPS)
    assert gl[0]["kernel"] == "wpp_f64_mdl_session"
    assert_tracks_reference(gl, rl, lambda t: per, what="adaptive")
    for t, (r, g) in enumerate(zip(gl, rl)):   # cache->rho at exit of every solve
        assert np.abs(r["rho"] - g["rho"]).max() <= 1e-6 * np.abs(g["rho"]).max(), t
    assert any((g["rho"] != np.array([p.rho for p in per])).any() for g in rl), "adaptive rho never moved"
    ses.close(); s.close()


# ---- 4. set_models mid-loop -------------------------------------------------------------------------------------------------------
SWAP_AT = 6


@pytest.mark.parametrize("precision, force_wpp, adaptive", [(64, 0, False), (64, 1, False), (64, 0, True)],
                         ids=["gpp", "wpp", "adaptive_wpp"])
def test_set_models_mid_loop_matches_the_reference(precision, force_wpp, adaptive, problems, oracle_mod, capi):
    specs, caches = _distinct(problems, oracle_mod, adaptive=adaptive, k=12, seed=7)
    B = 24
    which = np.arange(B) % 8                                       # models 0-7 first
    which2 = (which + 3) % 8                                       # a permutation of them ...
    which2[::4] = 8 + np.arange(B // 4) % 4                        # ... and the fresh models 8-11
    assert (which2 != which).all()
    b = problems.make_batch(specs[0], B, 0.6, seed=29)
    Xref, Uref = refs_of(b, specs[0], B)
    x0 = b.x0.astype(np.float64)
    per, per2 = [specs[j] for j in which], [specs[j] for j in which2]
    at = lambda t: per if t < SWAP_AT else per2
    refs = reference_sessions(oracle_mod, per, Xref, Uref, impl="swap")
    rl = reference_loop(refs, at, x0, SWAP_AT)
    for r, p in zip(refs, per2):
        r.set_model(p)
    rl += reference_loop(refs, lambda t: per2, rl[-1]["x0"], STEPS - SWAP_AT)
    s, ses = _model_session(capi, specs, caches, which, precision, x0, Xref, Uref, force_wpp)
    new_models = stack([model_of(p, c) for p, c in zip(specs, caches)], which2)

    def swap(t):
        if t == SWAP_AT:
            ses.set_models(new_models)
            assert np.array_equal(ses.read("rho"), np.array([p.rho for p in per2]))   # adaptive rho's moves are undone
    gl = gpu_loop(s, ses, STEPS, swap)
    assert_tracks_reference(gl, rl, at, what="set_models")
    if adaptive:
        for t, (r, g) in enumerate(zip(gl, rl)):
            assert np.abs(r["rho"] - g["rho"]).max() <= 1e-6 * np.abs(g["rho"]).max(), t
    ses.close(); s.close()


@pytest.mark.parametrize("precision, force_wpp, adaptive", [(64, 0, False), (64, 1, True), (32, 0, False)],
                         ids=["gpp", "adaptive_wpp", "wpp32"])
def test_set_models_with_the_same_models_changes_nothing(precision, force_wpp, adaptive, problems, oracle_mod, capi):
    specs, caches = _distinct(problems, oracle_mod, adaptive=adaptive, k=8, seed=9)
    B = 32
    which = np.arange(B) % len(specs)
    b = problems.make_batch(specs[0], B, 0.6, seed=31)
    Xref, Uref = refs_of(b, specs[0], B)
    x0 = b.x0.astype(np.float64)
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    s, a = _model_session(capi, specs, caches, which, precision, x0, Xref, Uref, force_wpp)
    _, c = _model_session(capi, specs, caches, which, precision, x0, Xref, Uref, force_wpp)
    ga = gpu_loop(s, a, STEPS)

    def again(t):
        if t == SWAP_AT:
            c.set_models(models)
    gc = gpu_loop(s, c, STEPS, again)
    # under adaptive rho the call resets a rho, Kinf and Pinf that the solves have moved (checked against the reference in
    # test_set_models_mid_loop_matches_the_reference), so the two sessions part there
    last = SWAP_AT if adaptive else STEPS
    for t, (u, v) in enumerate(zip(ga[:last], gc[:last])):
        for k in SESSION_FIELDS + ("x0_next",):
            assert np.array_equal(u[k], v[k]), (t, k)
    if adaptive:
        assert (ga[SWAP_AT - 1]["rho"] != np.array([specs[j].rho for j in which])).any(), "adaptive rho never moved"
    a.close(); c.close(); s.close()


# ---- 5. fp32 ---------------------------------------------------------------------------------------------------------------------
def test_fp32_model_session_tracks_the_reference(distinct_case, capi):
    specs, caches, which, x0, Xref, Uref, rl = distinct_case
    s, ses = _model_session(capi, specs, caches, which, 32, x0, Xref, Uref)
    gl = gpu_loop(s, ses, STEPS)
    assert gl[0]["kernel"] == "wpp_f32_mdl_session"
    assert_tracks_reference(gl, rl, None, exact=False, tol=2e-3, what="fp32")
    ses.close(); s.close()


# ---- 6. a generic shape with cones, rows, an affine term and adaptive rho --------------------------------------------------------
@pytest.mark.parametrize("precision", [64, 32])
def test_generic_shape_with_distinct_models(precision, capi, oracle_mod):
    nx, nu, N = 5, 2, 12
    specs = []
    for j in range(6):
        p, _ = G.family(nx, nu, N, seed=40 + j, B=64, affine=True, state_bound=True, cones=(2, 1), linear=(1, 1), adaptive=True,
                        check=2, max_iter=150)
        specs.append(p)
    p0, b = G.family(nx, nu, N, seed=40, B=24, affine=True, state_bound=True, cones=(2, 1), linear=(1, 1), adaptive=True,
                     check=2, max_iter=150)
    for p in specs:   # the constraints and settings of model 0's family for every solver; dynamics, costs, rho, sensitivities per model
        for k in ("x_min", "x_max", "u_min", "u_max", "Acx", "qcx", "cx", "Acu", "qcu", "cu", "Alin_x", "blin_x", "Alin_u", "blin_u",
                  "en_state_bound", "en_input_bound", "en_state_soc", "en_input_soc", "en_state_linear", "en_input_linear",
                  "adaptive_rho_min", "adaptive_rho_max", "adaptive_rho_enable_clipping"):
            setattr(p, k, getattr(p0, k))
    caches = [oracle_mod.get_cache(p, "port") for p in specs]
    B = b.size
    which = (np.arange(B) * 5) % len(specs)
    Xref, Uref = refs_of(b, p0, B)
    x0 = b.x0.astype(np.float64)
    per = [specs[j] for j in which]
    rl = reference_loop(reference_sessions(oracle_mod, per, Xref, Uref, impl="swap"), lambda t: per, x0, 8)
    s, ses = _model_session(capi, specs, caches, which, precision, x0, Xref, Uref)
    gl = gpu_loop(s, ses, 8)
    assert gl[0]["kernel"] == f"wpp_f{precision}_mdl_session"
    if precision == 64:
        for t, (r, g) in enumerate(zip(gl, rl)):
            assert np.array_equal(r["iter"], g["iter"]) and np.array_equal(r["status"], g["status"]), (t, r["iter"], g["iter"])
    else:
        flips = np.mean([np.mean(r["iter"] != g["iter"]) for r, g in zip(gl, rl)])
        assert flips <= 0.25, flips
    ses.close(); s.close()


# ---- 7. errors --------------------------------------------------------------------------------------------------------------------
def test_errors(distinct_case, capi, problems, oracle_mod):
    specs, caches, which, x0, Xref, Uref, _ = distinct_case
    C = capi.C
    EINVAL = 1
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    B = len(which)
    s = solver(capi, specs[0], caches[0], 64)
    L, h = s.L, C.c_void_p()

    def create(arrays, batch=B, dev=0):
        return L.tinympc_cuda_session_create_models(s.h, dev, batch, C.byref(capi.models_struct(arrays)), C.byref(h))

    full = capi.pack_models(models, B, 12, 4)
    for missing in ("Adyn", "Bdyn", "Q", "R", "rho", "Kinf", "Pinf", "Quu_inv", "AmBKt"):
        assert create({k: v for k, v in full.items() if k != missing}) == EINVAL, missing
        assert missing in L.tinympc_cuda_last_error(s.h).decode()
    assert create(full, batch=0) == EINVAL
    assert create(full, dev=7) == EINVAL and "dev_index" in L.tinympc_cuda_last_error(s.h).decode()
    assert L.tinympc_cuda_session_create_models(s.h, 0, B, None, C.byref(h)) == EINVAL
    # adaptive rho without the two sensitivities
    pa, ca = _distinct(problems, oracle_mod, adaptive=True, k=2, seed=1)
    sa = solver(capi, pa[0], ca[0], 64)
    ma = capi.pack_models(stack([model_of(p, c) for p, c in zip(pa, ca)], np.arange(4) % 2), 4, 12, 4)
    for drop in ("dKinf_drho", "dPinf_drho"):
        arr = {k: v for k, v in ma.items() if k != drop}
        assert sa.L.tinympc_cuda_session_create_models(sa.h, 0, 4, C.byref(capi.models_struct(arr)), C.byref(h)) == EINVAL
        assert "adaptive_rho" in sa.L.tinympc_cuda_last_error(sa.h).decode()
    sa.close()
    # set_models on a family session
    fam = s.session(B)
    with pytest.raises(capi.TinympcCudaError) as e:
        fam.set_models(models)
    assert e.value.code == EINVAL
    fam.close()
    # a failed set_models leaves the session as it was
    ses = s.session(B, models=models)
    start(ses, x0, Xref, Uref)
    ref = s.session(B, models=models)
    start(ref, x0, Xref, Uref)
    bad = {k: v for k, v in full.items() if k != "Kinf"}
    assert L.tinympc_cuda_session_set_models(ses.h, C.byref(capi.models_struct(bad))) == EINVAL
    assert L.tinympc_cuda_session_set_models(ses.h, None) == EINVAL
    ga, gb = gpu_loop(s, ses, 3), gpu_loop(s, ref, 3)
    for u, v in zip(ga, gb):
        for k in SESSION_FIELDS:
            assert np.array_equal(u[k], v[k]), k
    ses.close(); ref.close(); s.close()
