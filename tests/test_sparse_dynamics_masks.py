"""Sparse-A fp32 instances without a GPU: the nonzero patterns build.py compiles into them, their dense twins in the dispatch table,
and the pattern rules of the dispatcher (tmpc_sparse_a.h: the family's pattern, and which compiled pattern may serve it)."""
import importlib.util
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
PKG = ROOT / "tinympc-matlab_b200"


@pytest.fixture(scope="module")
def b():
    spec = importlib.util.spec_from_file_location("tmpc_build", PKG / "build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def pairs_of(A):
    """row-pair pattern of float32(A), one set of pair indices per column (pair nx // 2 = the odd tail row)"""
    A32 = np.asarray(A, dtype=np.float32)
    return [{r // 2 for r in range(A32.shape[0]) if A32[r, c] != 0} for c in range(A32.shape[1])]


def masks(pairs):
    return tuple(sum(1 << j for j in s) for s in pairs)


def test_patterns_are_the_nonzero_pairs_of_the_bundled_families(b, problems):
    pats = b.sparse_a_patterns()
    assert set(pats) == {(12, 4, 10), (4, 1, 20)}
    q, c = problems.quadrotor(), problems.cartpole()
    assert pats[(12, 4, 10)] == masks(pairs_of(q.A))
    assert pats[(4, 1, 20)] == masks(pairs_of(c.A))
    # the counts the forward rollout's product drops to: 26 of 72 pairs (quadrotor), 5 of 8 (cartpole)
    assert sum(len(s) for s in pairs_of(q.A)) == 26 and sum(len(s) for s in pairs_of(c.A)) == 5
    for inst in b.default_instances():
        if inst.get("sa"):
            assert inst["sa"] == pats[(inst["nx"], inst["nu"], inst["N"])]


def test_every_sparse_instance_has_a_dense_twin_after_it(b):
    inst = b.default_instances()
    names = [b.name_of(i) for i in inst]
    sparse = [k for k, i in enumerate(inst) if i.get("sa")]
    # variant 0 (refs / noref x fb / not, ppb) and the variant-9 plain-layout twins, for both shapes
    assert len(sparse) == 2 * 2 * 5
    for k in sparse:
        assert "_sa_" in names[k], names[k]
        twin = {**inst[k], "sa": None}
        at = [j for j, i in enumerate(inst) if i == twin]
        assert len(at) == 1 and at[0] > k, names[k]
        assert names[at[0]] == names[k].replace("_sa_", "_"), (names[k], names[at[0]])
    assert {(inst[k]["nx"], inst[k]["variant"]) for k in sparse} == {(12, 0), (12, 9), (4, 0), (4, 9)}


def test_generated_source_carries_the_pattern(b):
    inst = next(i for i in b.default_instances() if i.get("sa") and i["nx"] == 12)
    b.gen_sources(b.default_instances())          # idempotent: writes csrc/gen/*.cu only where the text changed
    src = (PKG / "csrc" / "gen" / f"{b.name_of(inst)}.cu").read_text()
    assert "SparsePairs<" + ", ".join(f"{m}u" for m in inst["sa"]) + ">>;" in src
    dense = (PKG / "csrc" / "gen" / f"{b.name_of({**inst, 'sa': None})}.cu").read_text()
    assert "SparsePairs" not in dense


DRIVER = r"""
#include <cstdio>
#include <cstdlib>
#include "tmpc_sparse_a.h"
// stdin: nx, the row-major A; then cases of (ncol, compiled masks...); prints the family's masks, then 1 / 0 per case
int main() {
    int nx; if (scanf("%d", &nx) != 1) return 2;
    double A[64 * 64]; unsigned fam[64];
    for (int e = 0; e < nx * nx; ++e) if (scanf("%lf", &A[e]) != 1) return 2;
    tmpc::a_pairs_of(A, nx, fam);
    for (int c = 0; c < nx; ++c) printf("%u ", fam[c]);
    printf("\n");
    int nc; unsigned inst[64];
    while (scanf("%d", &nc) == 1) {
        for (int c = 0; c < nc; ++c) if (scanf("%u", &inst[c]) != 1) return 2;
        printf("%d ", tmpc::a_pattern_covers(inst, nc, fam, nx) ? 1 : 0);
    }
    printf("\n");
    return 0;
}
"""


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    d = tmp_path_factory.mktemp("sparse_a")
    (d / "drv.cpp").write_text(DRIVER)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", str(PKG / "csrc"), str(d / "drv.cpp"), "-o", str(d / "drv")])

    def run(A, cases):
        A = np.asarray(A, dtype=np.float64)
        txt = f"{A.shape[0]} " + " ".join(repr(float(v)) for v in A.ravel()) + "\n"
        txt += "".join(f"{len(m)} " + " ".join(str(v) for v in m) + "\n" for m in cases)
        out = subprocess.run([str(d / "drv")], input=txt, capture_output=True, text=True, check=True).stdout.split("\n")
        return tuple(int(v) for v in out[0].split()), [bool(int(v)) for v in out[1].split()]
    return run


def test_family_pattern_is_taken_from_the_float32_matrix(driver, problems):
    for A in (problems.quadrotor().A, problems.cartpole().A):
        fam, _ = driver(A, [])
        assert fam == masks(pairs_of(A))
    A = np.eye(5)
    A[4, 1] = 1e-30                  # nonzero in float32: row 4 is the tail row of an odd nx -> bit 2
    A[0, 3] = 1e-50                  # zero in float32
    fam, _ = driver(A, [])
    assert fam == (1, 1 | 4, 2, 2, 4)


def test_a_compiled_pattern_serves_exactly_the_families_inside_it(driver, problems):
    q = np.asarray(problems.quadrotor().A, np.float64)
    pat = masks(pairs_of(q))
    dense = ()
    wider = tuple(m | 0b100000 for m in pat)
    _, ok = driver(q, [pat, dense, wider, pat[:11]])
    assert ok == [True, True, True, False]            # itself, dense, a superset; a pattern of another shape never
    hot = q.copy()
    hot[2, 0] = 1e-3                                   # pair 1 of column 0: outside the pattern
    tiny = q.copy()
    tiny[2, 0] = 1e-30
    sparser = q.copy()
    r, c = np.argwhere(q != 0)[0]
    sparser[r, c] = 0.0
    assert driver(hot, [pat, dense])[1] == [False, True]
    assert driver(tiny, [pat, dense])[1] == [False, True]
    assert driver(sparser, [pat, dense])[1] == [True, True]
    # hand-made 4x4 masks: bit j = pair j of the column
    A4 = np.zeros((4, 4))
    A4[0, 0] = A4[3, 2] = 1.0                          # pairs: column 0 -> pair 0, column 2 -> pair 1
    assert driver(A4, [(1, 0, 2, 0), (3, 3, 3, 3), (1, 0, 1, 0), (0, 0, 2, 0), (1, 0, 2)])[1] == [True, True, False, False, False]
