"""Sparse-A fp32 instances on the GPU (run with -m gpu): the instance whose forward rollout skips the zero coefficient pairs of A
(Tpp3Cfg::SA, tmpc_tpp3.cuh) gives what its dense twin (option dense_a = 1) gives, compared with == on every output, in every
mode and pipeline that reaches it; and the dispatcher runs it exactly for the families whose float32 A fits its pattern."""
import importlib

import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu

B_BIG = 1 << 16
B_ORDERED = 1 << 18      # the device entry claims hardest-first from two waves of the persistent grid on (tmpc_capi.cu, build_order)


@pytest.fixture(scope="module")
def capi():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return importlib.import_module("tinympc-matlab_b200.capi")


@pytest.fixture(scope="module")
def fams(oracle_mod, problems):
    out = {}
    for name in ("quadrotor", "cartpole"):
        p = getattr(problems, name)()
        out[name] = (p, cases.family_from_spec(p, oracle_mod.get_cache(p, "port")), problems.make_batch(p, B_BIG, 1.0, seed=11))
    return out


def solver(capi, fam, dense_a, mixed=0.0, **opts):
    s = capi.CudaSolver()
    s.set_option("precision", 32)
    s.set_option("mixed", mixed)
    s.set_option("dense_a", dense_a)
    for k, v in opts.items():
        s.set_option(k, v)
    s.set_family(fam)
    return s


def host_solve(capi, fam, b, dense_a, mixed=0.0, n=None, compact=False, **opts):
    s = solver(capi, fam, dense_a, mixed, **opts)
    n = len(b.x0) if n is None else n
    if compact:
        r = s.solve_batch(b.x0[:n], xref_const=b.Xref[:n, 0], Uref=None if b.Uref is None else b.Uref[:n], compact_out=True)
    else:
        r = s.solve_batch(b.x0[:n], None if b.Xref is None else b.Xref[:n], None if b.Uref is None else b.Uref[:n])
    r["kernel"], r["marked"] = s.last_kernel, s.last_marked
    s.close()
    return r


def device_solve(capi, fam, p, b, dense_a, mixed, order):
    import torch
    dev = torch.device("cuda:0")
    s = solver(capi, fam, dense_a, mixed, order=order)
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    x0, Xr, Ur = t(b.x0), t(b.Xref), t(b.Uref)
    B = len(b.x0)
    o = dict(x=torch.empty((B, p.N, p.nx), device=dev), u=torch.empty((B, p.N - 1, p.nu), device=dev),
             iter=torch.empty(B, dtype=torch.int32, device=dev), status=torch.empty(B, dtype=torch.int32, device=dev),
             residuals=torch.empty((B, 4), device=dev))
    ptr = lambda a: None if a is None else a.data_ptr()
    s.solve_batch_device(B, ptr(x0), ptr(Xr), ptr(Ur), ptr(o["x"]), ptr(o["u"]), ptr(o["iter"]), ptr(o["status"]), residuals=ptr(o["residuals"]))
    torch.cuda.synchronize()
    r = {k: v.cpu().numpy() for k, v in o.items()}
    r["kernel"], r["marked"] = s.last_kernel, s.last_marked
    s.close()
    return r


def assert_same(rs, rd, what, variant="v0"):
    """sparse arm rs against dense arm rd: the sparse instance ran, and every output array is equal under == (+0 == -0)"""
    assert f"_sa_{variant}" in rs["kernel"] and "_sa_" not in rd["kernel"], (what, rs["kernel"], rd["kernel"])
    assert rs["kernel"].replace("_sa_", "_") == rd["kernel"], (what, rs["kernel"], rd["kernel"])
    arrays = [k for k in rs if isinstance(rs[k], np.ndarray)]
    assert {"iter", "status"} <= set(arrays), arrays
    for k in arrays:
        assert np.all(np.isfinite(rs[k])), (what, k)
        assert np.array_equal(rs[k], rd[k]), f"{what}: {k} differs between the sparse-A and the dense instance"
    assert rs["marked"] == rd["marked"], (what, rs["marked"], rd["marked"])


@pytest.mark.parametrize("name", ["quadrotor", "cartpole"])
@pytest.mark.parametrize("mode", ["fp32", "exact"])
def test_host_pipeline_matches_dense_twin(capi, fams, problems, name, mode):
    p, fam, b = fams[name]
    mixed = problems.exact_band(p) if mode == "exact" else 0.0
    rs, rd = (host_solve(capi, fam, b, d, mixed) for d in (0, 1))
    assert_same(rs, rd, f"{name} {mode} host")
    assert "x" in rs and "residuals" in rs
    if mode == "exact" and name == "quadrotor":
        assert rs["marked"] > 0, "the exact-count mode re-solved nothing: the comparison of its marked sets is empty"


@pytest.mark.parametrize("streamed", [1, 0])
def test_compact_io_matches_dense_twin(capi, fams, problems, streamed):
    p, fam, b = fams["quadrotor"]
    rs, rd = (host_solve(capi, fam, b, d, problems.exact_band(p), compact=True, streamed=streamed, compact_streamed=streamed) for d in (0, 1))
    assert "u0" in rs
    assert_same(rs, rd, f"compact streamed={streamed}")


@pytest.mark.parametrize("name", ["quadrotor", "cartpole"])
def test_device_entry_in_both_claim_orders_matches_dense_twin(capi, fams, problems, name):
    p, fam, _ = fams[name]
    b = problems.make_batch(p, B_ORDERED, 1.0, seed=12)
    res = {}
    for order in (0, 1):
        for d in (0, 1):
            res[order, d] = device_solve(capi, fam, p, b, d, problems.exact_band(p), order)
        assert_same(res[order, 0], res[order, 1], f"{name} device order={order}")
    for k in ("x", "u", "iter", "status", "residuals"):   # and the claim order changes nothing either
        assert np.array_equal(res[0, 0][k], res[1, 0][k]), (name, k)


@pytest.mark.parametrize("name", ["quadrotor", "cartpole"])
def test_small_batch_takes_the_sparse_plain_layout_twin(capi, fams, name):
    p, fam, b = fams[name]
    rs, rd = (host_solve(capi, fam, b, d, n=1024) for d in (0, 1))
    assert_same(rs, rd, f"{name} small batch", variant="v9")


def kernel_for(capi, oracle_mod, p):
    fam = cases.family_from_spec(p, oracle_mod.get_cache(p, "port"))
    s = solver(capi, fam, 0)
    rng = np.random.default_rng(3)
    s.solve_batch((0.1 * rng.standard_normal((64, p.nx))).astype(np.float32))
    k = s.last_kernel
    s.close()
    return k


def test_dispatch_follows_the_float32_pattern(capi, oracle_mod, problems):
    q, c = problems.quadrotor(), problems.cartpole()
    assert kernel_for(capi, oracle_mod, q).startswith("tpp3_f32_12x4x10_") and "_sa_" in kernel_for(capi, oracle_mod, q)
    assert "_sa_" in kernel_for(capi, oracle_mod, c)
    A = np.array(q.A, dtype=np.float64)
    assert A[2, 0] == 0.0
    for v in (1e-3, 1e-30):                         # outside the compiled pattern (1e-30 is a nonzero float32)
        Ah = A.copy()
        Ah[2, 0] = v
        k = kernel_for(capi, oracle_mod, q.with_(A=Ah))
        assert k.startswith("tpp3_f32_12x4x10_") and "_sa_" not in k, (v, k)
    As = A.copy()
    r, col = np.argwhere(A != 0)[-1]
    As[r, col] = 0.0                                # sparser than the pattern: still the sparse instance
    assert "_sa_" in kernel_for(capi, oracle_mod, q.with_(A=As))
