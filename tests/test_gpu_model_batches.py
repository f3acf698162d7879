"""GPU tests of model batches (tinympc_cuda_solve_batch_models): every problem of a batch brings its own dynamics, costs and cache.

The reference of a model batch is the reference solver run per model on the problems that carry it -- a loop of
{ tiny_setup(A_b, B_b, Q_b, R_b, rho_b); tiny_set_x0; tiny_solve } over solvers.  What is checked:
  * identity: a batch whose every problem carries the family's own model reproduces solve_batch on that family bit for bit, on the
    model form of the lane-group fp64 kernel (gpp, against the family's gpp) and of the warp-per-problem kernel (wpp, against the
    family's wpp): this pins the per-problem loads and the device-side coefficient products to the host's arithmetic;
  * parity with the reference on batches of 32 distinct quadrotor models interleaved over the problems (neighbouring problems of a
    warp and of a lane group carry different models), in fp64 (exact iteration counts) and fp32 (bounded flips), and on a random
    shape with cones, linear rows and adaptive rho with per-problem sensitivities (the final rho of every problem too);
  * that this parity test can fail: the reference with every problem given model 0 differs in its iteration counts;
  * the batched precompute feeding the solve; permutations, pipeline depths, the device entry, ragged sizes, two devices;
  * compact I/O, per-problem bounds, and the EINVAL / EUNSUPPORTED cases.
"""
import importlib

import numpy as np
import pytest

import cases
import generic_families as G
from test_gpu_parity import compare

pytestmark = pytest.mark.gpu

K_MODELS = 32
B_PARITY = 4096
WPP32_FLIP_BOUND = 0.04


@pytest.fixture(scope="module")
def capi():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return importlib.import_module("tinympc-matlab_b200.capi")


@pytest.fixture(scope="module")
def problems():
    return importlib.import_module("tinympc-matlab_b200.problems")


def reference(oracle_mod, p, b):
    return oracle_mod.solve_batch(p, b, "ref" if oracle_mod.available("ref") else "port")


def model_of(p, cache):
    """one problem's model in the math shapes of capi.pack_models (work->Q / work->R = diagonal + rho)"""
    m = dict(A=p.A, B=np.asarray(p.B).reshape(p.nx, p.nu), f=p.f, Q=p.Qdiag + p.rho, R=p.Rdiag + p.rho, rho=p.rho,
             Kinf=cache["Kinf"], Pinf=cache["Pinf"], Quu_inv=cache["Quu_inv"], AmBKt=cache["AmBKt"], APf=cache["APf"], BPf=cache["BPf"])
    if p.adaptive_rho:
        m["dKinf"], m["dPinf"] = cache["dKinf"], cache["dPinf"]
    return m


def stack(models, which):
    """per-problem model arrays: problem i carries models[which[i]]"""
    return {k: np.stack([np.asarray(models[j][k], np.float64) for j in which]) for k in models[0]}


def solver(capi, p, cache, precision, force_wpp=0, **opts):
    s = capi.CudaSolver()
    s.set_option("precision", precision)
    s.set_option("force_wpp", force_wpp)
    for k, v in opts.items():
        s.set_option(k, v)
    s.set_family(cases.family_from_spec(p, cache))
    return s


def solve_models(capi, p, cache, b, models, precision, force_wpp=0, **opts):
    s = solver(capi, p, cache, precision, force_wpp, **opts)
    r = s.solve_batch_models(models, b.x0, Xref=b.Xref, Uref=b.Uref, x_min=b.x_min, x_max=b.x_max, u_min=b.u_min, u_max=b.u_max)
    r["kernel"] = s.last_kernel
    s.close()
    return r


def assert_identical(r, q, what):
    for k in ("x", "u", "iter", "status", "residuals", "rho"):
        assert np.array_equal(r[k], q[k]), f"{what}: {k} differs ({r['kernel']} against {q['kernel']})"


# ---- 1. identity with the family path -------------------------------------------------------------------------------------------
def _family_case(problems, name):
    if name == "quadrotor":
        p = problems.quadrotor()
    elif name == "cartpole":
        p = problems.cartpole()
    elif name == "rocket":
        p = problems.rocket()
    elif name == "quadrotor_adaptive":
        p = problems.quadrotor(adaptive=True)
    else:
        return G.family(*name, seed=3, B=1200, affine=True, state_bound=True, cones=(2, 1), linear=(1, 1), adaptive=True, check=2)
    return p, problems.make_batch(p, 3000, 1.0, seed=5)


@pytest.mark.parametrize("name, precision, kernel", [
    ("quadrotor", 64, "gpp_f64_12x4x10_box_g16_v0"),
    ("cartpole", 64, "gpp_f64_4x1x20_box_g8_v0"),
    ("rocket", 64, "wpp_f64"),
    ((5, 2, 12), 64, "wpp_f64"),
    ("quadrotor_adaptive", 64, "wpp_f64"),
    ("quadrotor", 32, "wpp_f32"),
    ((5, 2, 12), 32, "wpp_f32"),
], ids=["quadrotor_gpp", "cartpole_gpp", "rocket_wpp", "generic_wpp", "adaptive_wpp", "quadrotor_wpp32", "generic_wpp32"])
def test_family_model_everywhere_is_bit_identical_to_the_family_path(name, precision, kernel, capi, oracle_mod, problems):
    p, b = _family_case(problems, name)
    cache = oracle_mod.get_cache(p, "port")
    wpp = kernel.startswith("wpp")
    s = solver(capi, p, cache, precision, force_wpp=int(wpp))
    fam = s.solve_batch(b.x0, b.Xref, b.Uref)
    fam["kernel"] = s.last_kernel
    s.close()
    models = stack([model_of(p, cache)], np.zeros(b.size, int))
    r = solve_models(capi, p, cache, b, models, precision, force_wpp=int(wpp))
    if wpp:
        assert fam["kernel"] == f"{kernel}_generic" and r["kernel"] == f"{kernel}_mdl_generic", (fam["kernel"], r["kernel"])
    else:   # the model form of the lane-group kernel runs without being forced
        assert fam["kernel"] == kernel and r["kernel"] == kernel + "_mdl", (fam["kernel"], r["kernel"])
        r2 = solve_models(capi, p, cache, b, models, precision, force_wpp=1)
        assert r2["kernel"] == "wpp_f64_mdl_generic"
        assert np.array_equal(r2["iter"], r["iter"]) and np.array_equal(r2["status"], r["status"])
    assert_identical(r, fam, str(name))


# ---- 2. / 3. / 4. parity with the reference on distinct models ------------------------------------------------------------------
def quadrotor_models(problems, k=K_MODELS, seed=0):
    """k quadrotor models: translational rows of B scaled as by a +-30 % mass change, rotational rows as by a +-30 % inertia change,
    Q and R diagonals scaled by factors in [0.5, 2], rho in [0.5, 2] x the nominal"""
    rng = np.random.default_rng(seed)
    base = problems.quadrotor()
    out = []
    for j in range(k):
        p = problems.quadrotor()
        Bm = np.asarray(base.B, np.float64).reshape(12, 4).copy()
        m, jn = rng.uniform(0.7, 1.3), rng.uniform(0.7, 1.3)
        Bm[[0, 1, 2, 6, 7, 8]] /= m
        Bm[[3, 4, 5, 9, 10, 11]] /= jn
        p.B = Bm
        p.Qdiag = base.Qdiag * rng.uniform(0.5, 2.0, 12)
        p.Rdiag = base.Rdiag * rng.uniform(0.5, 2.0, 4)
        p.rho = float(base.rho * rng.uniform(0.5, 2.0))
        p.name = f"quadrotor_model{j}"
        out.append(p)
    return out


def reference_per_model(oracle_mod, specs, which, b):
    """the reference solved per model on the problems that carry it, reassembled in batch order"""
    g = None
    for j, p in enumerate(specs):
        idx = np.flatnonzero(which == j)
        if not len(idx):
            continue
        gj = reference(oracle_mod, p, _take(b, idx))
        if g is None:
            g = {k: np.zeros((len(which),) + v.shape[1:], v.dtype) for k, v in gj.items()}
        for k in g:
            g[k][idx] = gj[k]
    return g


def _take(b, idx):
    t = lambda a: None if a is None else np.ascontiguousarray(a[idx])
    return type(b)(t(b.x0), t(b.Xref), t(b.Uref), t(b.x_min), t(b.x_max), t(b.u_min), t(b.u_max))


@pytest.fixture(scope="module")
def quad_case(problems, oracle_mod):
    specs = quadrotor_models(problems)
    caches = [oracle_mod.get_cache(p, "port") for p in specs]
    which = np.arange(B_PARITY) % K_MODELS                 # neighbours carry different models
    b = problems.make_batch(specs[0], B_PARITY, 1.0, seed=21)
    g = reference_per_model(oracle_mod, specs, which, b)
    return specs, caches, which, b, g


@pytest.mark.parametrize("precision", [64, 32])
def test_distinct_models_match_the_reference(precision, quad_case, capi, oracle_mod):
    specs, caches, which, b, g = quad_case
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    r = solve_models(capi, specs[0], caches[0], b, models, precision)
    assert r["kernel"] == ("gpp_f64_12x4x10_box_g16_v0_mdl" if precision == 64 else "wpp_f32_mdl_generic")
    if precision == 64:
        compare(r, g, 64, "quadrotor models fp64")
    else:
        # the warp-per-problem kernel (bit-identical to the family's, test above) is a direct-form fp32 kernel: on the quadrotor it flips
        # more termination decisions than the incremental-form fp32 kernels and lands up to ~1e-4 from the reference (measured on a B200
        # at 1000 W: 115 / 4096 flips, 1.0e-4 on a converged problem, 7.8e-5 at max_iter)
        same = (r["iter"] == g["iter"]) & (r["status"] == g["status"])
        assert (~same).mean() <= WPP32_FLIP_BOUND, f"{int((~same).sum())} / {len(same)} iteration/status mismatches"
        assert np.abs(r["x"][same] - g["x"][same]).max() <= 2e-4 and np.abs(r["u"][same] - g["u"][same]).max() <= 2e-4
    # per-problem rho: every problem reports its own model's rho
    assert np.array_equal(r["rho"], np.array([specs[j].rho for j in which], np.float32))


def test_the_distinct_model_test_can_fail(quad_case, oracle_mod):
    """a kernel that ignored the per-problem model (solved every problem with model 0) would disagree with the reference in its
    iteration counts on a large part of the batch"""
    specs, caches, which, b, g = quad_case
    g0 = reference(oracle_mod, specs[0], b)
    differ = float((g0["iter"] != g["iter"]).mean())
    assert differ > 0.5, f"only {differ:.1%} of the problems change their iteration count with their model"


def test_precompute_feeds_the_solve(quad_case, capi, oracle_mod):
    """caches from the batched precompute (tinympc_cuda_precompute_batch) go straight into the model batch; the reference is given
    the same caches (its own Riccati iteration stops at a slightly different point)"""
    specs, caches, which, b, _ = quad_case
    A = np.stack([p.A for p in specs]); Bm = np.stack([np.asarray(p.B).reshape(12, 4) for p in specs])
    rho = np.array([p.rho for p in specs])
    # tiny_setup stores Q + rho and its precompute adds rho once more (SURVEY quirk Q1): the cache is that of Q + 2 rho
    pc = capi.precompute_batch(A, Bm, np.stack([p.Qdiag + p.rho for p in specs]), np.stack([p.Rdiag + p.rho for p in specs]), rho)
    pre = [dict(Kinf=pc["Kinf"][j], Pinf=pc["Pinf"][j], Quu_inv=pc["Quu_inv"][j], AmBKt=pc["AmBKt"][j], APf=pc["APf"][j], BPf=pc["BPf"][j])
           for j in range(K_MODELS)]
    assert max(np.abs(pre[j]["Kinf"] - caches[j]["Kinf"]).max() for j in range(K_MODELS)) < 1e-3
    models = stack([model_of(p, c) for p, c in zip(specs, pre)], which)
    r = solve_models(capi, specs[0], caches[0], b, models, 64)
    # the reference with the same caches: the oracle's family path, one precomputed cache per model
    g = {k: None for k in ("x", "u", "iter", "status")}
    for j, p in enumerate(specs):
        idx = np.flatnonzero(which == j)
        rj = solve_gpu_with_cache(capi, p, pre[j], _take(b, idx))
        for k in g:
            if g[k] is None:
                g[k] = np.zeros((len(which),) + rj[k].shape[1:], rj[k].dtype)
            g[k][idx] = rj[k]
    compare(r, g, 64, "precomputed caches")


def solve_gpu_with_cache(capi, p, cache, b):
    """the family path (solve_batch) of one model with the given cache: the per-model loop the model batch replaces"""
    s = solver(capi, p, cache, 64)
    r = s.solve_batch(b.x0, b.Xref, b.Uref)
    s.close()
    return r


@pytest.mark.parametrize("precision", [64, 32])
def test_generic_shape_with_cones_rows_and_adaptive_rho(precision, capi, oracle_mod):
    nx, nu, N = 5, 2, 12
    specs, bs = [], []
    for j in range(8):
        p, b = G.family(nx, nu, N, seed=40 + j, B=256, affine=True, state_bound=True, cones=(2, 1), linear=(1, 1), adaptive=True,
                        check=2, max_iter=150)
        specs.append(p)
    # the constraints, settings and x0 of model 0's family for every problem; dynamics, costs, rho and sensitivities per model
    p0, b = G.family(nx, nu, N, seed=40, B=2048, affine=True, state_bound=True, cones=(2, 1), linear=(1, 1), adaptive=True,
                     check=2, max_iter=150)
    for p in specs:
        for k in ("x_min", "x_max", "u_min", "u_max", "Acx", "qcx", "cx", "Acu", "qcu", "cu", "Alin_x", "blin_x", "Alin_u", "blin_u",
                  "en_state_bound", "en_input_bound", "en_state_soc", "en_input_soc", "en_state_linear", "en_input_linear",
                  "adaptive_rho_min", "adaptive_rho_max", "adaptive_rho_enable_clipping"):
            setattr(p, k, getattr(p0, k))
    caches = [oracle_mod.get_cache(p, "port") for p in specs]
    which = (np.arange(b.size) * 5) % len(specs)
    g = reference_per_model(oracle_mod, specs, which, b)
    G.assert_nontrivial(p0, g, "generic models")
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    r = solve_models(capi, p0, caches[0], b, models, precision)
    assert r["kernel"] == f"wpp_f{precision}_mdl_generic"
    if precision == 64:
        same = (r["iter"] == g["iter"]) & (r["status"] == g["status"])
        assert same.all(), f"{int((~same).sum())} iteration/status mismatches"
        assert np.abs(r["rho"] - g["rho"]).max() <= 1e-6 * np.abs(g["rho"]).max()
        conv = g["status"] == 1        # problems stopped at max_iter amplify rounding (tests/test_gpu_generic_shapes.py)
        scale = max(1.0, float(np.abs(g["x"]).max()))
        assert np.abs(r["x"][conv] - g["x"][conv]).max() <= 1e-6 * scale
    else:
        assert ((r["iter"] != g["iter"]) | (r["status"] != g["status"])).mean() <= 0.01


# ---- 5. indexing ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", [64, 32])
def test_permuting_problems_with_their_models_permutes_the_results(precision, quad_case, capi):
    specs, caches, which, b, _ = quad_case
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    r = solve_models(capi, specs[0], caches[0], b, models, precision)
    perm = np.random.default_rng(3).permutation(b.size)
    rp = solve_models(capi, specs[0], caches[0], _take(b, perm), {k: v[perm] for k, v in models.items()}, precision)
    for k in ("x", "u", "iter", "status", "residuals", "rho"):
        assert np.array_equal(rp[k], r[k][perm]), k


def test_pipeline_depth_and_device_entry_agree(quad_case, capi):
    import torch
    specs, caches, which, b, _ = quad_case
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    r1 = solve_models(capi, specs[0], caches[0], b, models, 64, chunks=1)
    r4 = solve_models(capi, specs[0], caches[0], b, models, 64, chunks=4)
    for k in ("x", "u", "iter", "status", "residuals", "rho"):
        assert np.array_equal(r1[k], r4[k]), k
    s = solver(capi, specs[0], caches[0], 64)
    dev = torch.device("cuda", 0)
    packed = capi.pack_models(models, b.size, 12, 4)
    dm = {f: torch.from_numpy(a).to(dev) for f, a in packed.items()}
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    B, N = b.size, specs[0].N
    x = torch.empty((B, N, 12), device=dev); u = torch.empty((B, N - 1, 4), device=dev)
    it = torch.empty(B, dtype=torch.int32, device=dev); st = torch.empty(B, dtype=torch.int32, device=dev)
    rho = torch.empty(B, device=dev)
    x0, Xr, Ur = t(b.x0), t(b.Xref), t(b.Uref)
    s.solve_batch_models_device({f: v.data_ptr() for f, v in dm.items()}, B, x0.data_ptr(), Xr.data_ptr(), Ur.data_ptr(), x.data_ptr(),
                                u.data_ptr(), it.data_ptr(), st.data_ptr(), rho=rho.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert s.last_kernel == "gpp_f64_12x4x10_box_g16_v0_mdl"
    assert np.array_equal(x.cpu().numpy(), r1["x"]) and np.array_equal(u.cpu().numpy(), r1["u"])
    assert np.array_equal(it.cpu().numpy(), r1["iter"]) and np.array_equal(st.cpu().numpy(), r1["status"])
    assert np.array_equal(rho.cpu().numpy(), r1["rho"])
    s.close()


def test_two_device_split_matches_one_device(quad_case, capi):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device: the two-device split needs a second")
    specs, caches, which, b, _ = quad_case
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    for precision in (64, 32):
        r1 = solve_models(capi, specs[0], caches[0], b, models, precision)
        s = capi.CudaSolver(devices=[0, 1])
        s.set_option("precision", precision)
        s.set_family(cases.family_from_spec(specs[0], caches[0]))
        r2 = s.solve_batch_models(models, b.x0, Xref=b.Xref, Uref=b.Uref)
        s.close()
        for k in ("x", "u", "iter", "status", "residuals", "rho"):
            assert np.array_equal(r1[k], r2[k]), (precision, k)


@pytest.mark.parametrize("B", [1, 31, 33, 4097])
def test_ragged_batch_sizes(B, quad_case, capi, problems):
    specs, caches, _, _, _ = quad_case
    which = (np.arange(B) * 7) % K_MODELS
    b = problems.make_batch(specs[0], B, 1.0, seed=B)
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    r = solve_models(capi, specs[0], caches[0], b, models, 64)
    for j in np.unique(which)[:4]:      # each model's problems against that model's own family solve
        idx = np.flatnonzero(which == j)
        q = solve_gpu_with_cache(capi, specs[j], caches[j], _take(b, idx))
        for k in ("x", "u", "iter", "status"):
            assert np.array_equal(r[k][idx], q[k]), (B, j, k)
    r32 = solve_models(capi, specs[0], caches[0], b, models, 32)
    compare(r32, r, 32, f"ragged {B} fp32", max_flip_frac=max(WPP32_FLIP_BOUND, 1.0 / B), hard_tol=1e-3)


# ---- 6. compact I/O and per-problem bounds -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", [64, 32])
def test_compact_io(precision, quad_case, capi):
    specs, caches, which, b, _ = quad_case
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    s = solver(capi, specs[0], caches[0], precision)
    xc = np.ascontiguousarray(b.Xref[:, 0, :])
    Xfull = np.ascontiguousarray(np.repeat(xc[:, None, :], specs[0].N, axis=1))
    full = s.solve_batch_models(models, b.x0, Xref=Xfull)
    c = s.solve_batch_models(models, b.x0, xref_const=xc, compact_out=True)
    s.close()
    assert np.array_equal(c["iter"], full["iter"]) and np.array_equal(c["status"], full["status"])
    assert np.array_equal(c["u0"], full["u"][:, 0, :])


def test_per_problem_bounds_with_models(quad_case, capi, oracle_mod, problems):
    specs, caches, which, b, _ = quad_case
    rng = np.random.default_rng(9)
    B, N = b.size, specs[0].N
    ub = rng.uniform(0.2, 0.6, (B, 1, 4)).astype(np.float32)
    xb = rng.uniform(3.0, 6.0, (B, 1, 12)).astype(np.float32)
    bb = problems.Batch(b.x0, b.Xref, b.Uref, np.repeat(-xb, N, 1), np.repeat(xb, N, 1), np.repeat(-ub, N - 1, 1), np.repeat(ub, N - 1, 1))
    g = reference_per_model(oracle_mod, specs, which, bb)
    models = stack([model_of(p, c) for p, c in zip(specs, caches)], which)
    r = solve_models(capi, specs[0], caches[0], bb, models, 64)
    assert r["kernel"] == "wpp_f64_mdl_generic"      # the lane-group kernel takes shared bounds only
    compare(r, g, 64, "per-problem bounds with models")


# ---- 7. errors ---------------------------------------------------------------------------------------------------------------------
def test_errors(quad_case, capi, problems, oracle_mod):
    import torch
    specs, caches, which, b, _ = quad_case
    models = stack([model_of(p, c) for p, c in zip(specs[:1], caches[:1])], np.zeros(8, int))
    x0 = np.ascontiguousarray(b.x0[:8])

    def expect(code, fn, text):
        before = torch.cuda.current_device()
        with pytest.raises(capi.TinympcCudaError) as e:
            fn()
        assert e.value.code == code and text in str(e.value), str(e.value)
        assert torch.cuda.current_device() == before

    s = solver(capi, specs[0], caches[0], 64)
    assert s.solve_batch_models({k: v[:0] for k, v in models.items()}, x0[:0])["iter"].shape == (0,)        # batch 0: OK
    for missing in ("A", "B", "Q", "R", "rho", "Kinf", "Pinf", "Quu_inv", "AmBKt"):
        expect(1, lambda: s.solve_batch_models({k: v for k, v in models.items() if k != missing}, x0), "is required")
    # adaptive rho without the two sensitivities
    pa = problems.quadrotor(adaptive=True)
    ca = oracle_mod.get_cache(pa, "port")
    sa = solver(capi, pa, ca, 64)
    expect(1, lambda: sa.solve_batch_models(models, x0), "dKinf_drho")
    sa.close()
    # the exact-count mode has no model form
    s32 = solver(capi, specs[0], caches[0], 32, mixed=problems.exact_band(specs[0]))
    expect(4, lambda: s32.solve_batch_models(models, x0), "\"precision\" 64")
    s32.close()
    # a misaligned device pointer
    dev = torch.device("cuda", 0)
    packed = capi.pack_models(models, 8, 12, 4)
    dm = {f: torch.from_numpy(a).to(dev) for f, a in packed.items()}
    ptrs = {f: v.data_ptr() for f, v in dm.items()}
    ptrs["Kinf"] += 8
    x0d = torch.from_numpy(x0).to(dev)
    x = torch.empty((8, 10, 12), device=dev); u = torch.empty((8, 9, 4), device=dev)
    it = torch.empty(8, dtype=torch.int32, device=dev); st = torch.empty(8, dtype=torch.int32, device=dev)
    expect(1, lambda: s.solve_batch_models_device(ptrs, 8, x0d.data_ptr(), None, None, x.data_ptr(), u.data_ptr(), it.data_ptr(),
                                                  st.data_ptr()), "Kinf must be 16-byte aligned")
    s.close()
