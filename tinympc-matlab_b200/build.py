#!/usr/bin/env python3
"""Build libtinympc_b200.so (sm_100a) in-tree.

Every kernel instance of INSTANCES becomes its own generated translation unit under csrc/gen/ so
that nvcc compiles them in parallel; csrc/gen/tmpc_table.cu lists them for the C-ABI dispatcher.
Usage: python tinympc-matlab_b200/build.py [-j N] [--force]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
GEN = CSRC / "gen"
OBJ = HERE / "build"
LIB = HERE / "libtinympc_b200.so"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr"]

BOX, CON, ADP = 0, 1, 2
FEAT_NAME = {BOX: "box", CON: "con", ADP: "adp"}
FEAT_ENUM = {BOX: "FEAT_BOX", CON: "FEAT_CONSTR", ADP: "FEAT_ADAPT"}

REFS_NONE, REFS_SMEM, REFS_L2 = 0, 1, 2


def inst(bits, nx, nu, N, feat, refs=REFS_SMEM, ppb=False, variant=0, block=None, minb=None, budget_kb=226, fb=False, gen=2, aff=None, tm=False, opq=None, max_warps=None, tib=None):
    max_warps = (24 if nx * N <= 80 else 16) if max_warps is None else max_warps   # small shapes: 6 warps per tensor-memory lane quarter
    tib = (not (nx == 12 and feat == BOX)) if tib is None else tib
    tm = tm and bits == 32 and gen == 2
    b, m = plan_block(nx, nu, N, feat, bits, refs, budget_kb, tm, max_warps)
    ntm = m if tm else 0      # tensor-memory instances: plan_block returns (block, arrays in tensor memory); always 1 CTA/SM
    if tm:
        m = 1
    aff = ((nx, nu) == (6, 3)) if aff is None else aff   # affine-term instances only where a shipped config needs them (rocket: gravity)
    # opaque (loop-variant) constant offsets pay off only where few warps hide the LDCU latency: measured +27 % on the
    # fp64 instances (8 warps/SM), -14 % on the fp32 tensor-memory instances (16 warps/SM, LDCU issue-rate bound)
    opq = (bits == 64) if opq is None else opq
    return dict(aff=aff, tm=tm, ntm=ntm, opq=opq, tib=tib, bits=bits, nx=nx, nu=nu, N=N, feat=feat, refs=refs, ppb=ppb, variant=variant, block=block or b, minb=minb or m, fb=fb, gen=gen)


def plan_hybrid(nx, nu, N, max_warps=24):
    """(warps, ttm) of the hybrid layout of tmpc_tpp3.cuh maximising the resident warps: x_1 .. x_{N-2} and t_0 .. t_{ttm-1} in the
    warp's share of the 512 tensor-memory columns, t_ttm .. t_{N-2} + u, u + y, -dd in shared memory, column N-1 in registers"""
    su = nu * (N - 1)
    for warps in range(max_warps, 3, -4):
        cols = 512 // (warps // 4)
        ttm = min(N - 1, cols // nx - (N - 2))
        if ttm < 0:
            continue
        smem_cols = 3 * su + (N - 1 - ttm) * nx
        if smem_cols * warps * 32 * 4 + 1024 + pack_elems(nx, nu, N) * 4 > 226 * 1024:
            continue
        if 65536 // (warps * 32) < 64 + 8 * nx:      # registers: ~126 + 2 nx (column N-1) on the quadrotor shape, ~90 with nx = 4
            continue
        return warps, ttm
    return None


def inst3(nx, nu, N, refs=True, ppb=False, fb=False, variant=0, max_warps=24, opq=False, tib=None, aff=None, feat=BOX, cones=(0, 0, 0, 0, 0, 0), hyb=False, conv=-1):
    """incremental-form kernel (tmpc_tpp3.cuh): x and t in tensor memory (2 nx N columns per thread), u, u + y, -dd in shared memory;
    with cones / linear rows (feat=CON) two more arrays of each kind (the pre-projection slacks of the two families)"""
    sx, su = nx * N, nu * (N - 1)
    ntm, nsm = (4, 5) if feat == CON else (2, 3)
    warps = min(max_warps, 4 * (512 // (ntm * sx)), ((226 * 1024 - 1024 - pack_elems(nx, nu, N) * 4) // (nsm * su * 4 * 32) // 4) * 4)
    ttm = -1
    if hyb:
        assert feat == BOX
        warps, ttm = plan_hybrid(nx, nu, N, max_warps)
    assert warps >= 4, "shape does not fit the incremental-form kernel"
    aff = ((nx, nu) == (6, 3)) if aff is None else aff
    # fast-box bounds read from time row 0 with immediate addresses: with the incremental-form kernel this is a gain on every shape
    # (quadrotor +3.3 %), unlike the direct form, where the hoisted bounds starved the coefficient stream of the quadrotor instance
    tib = True if tib is None else tib
    return dict(gen=3, bits=32, nx=nx, nu=nu, N=N, feat=feat, refs=3 if refs else 0, ppb=ppb, fb=fb, variant=variant, block=warps * 32, aff=aff,
                opq=opq, tib=tib, tm=True, minb=1, ntm=ntm, cones=cones, ttm=ttm, conv=conv)


def inst4(nx, nu, N, refs=True, fb=False, variant=0, aff=None, cones=(0, 0, 0, 0, 0, 0)):
    """mixed-precision kernel of the rocket family (tmpc_tpp4.cuh): fp64 iterates and cone duals, fp32 Riccati increments.
    Tensor memory per thread: (N-1) [dx | x | cone dual | multiplier] + input multipliers; shared memory: u, input cone dual
    (double), box duals, -dd."""
    scs, scd, ucs, ucd, nsl, nil = cones
    cw = 3 * nx + 2 * scd + 2 * nsl
    tm = (N - 1) * cw + 2 * nil * (N - 1)
    sm = 2 * (nu + ucd) * (N - 1) + nx * N + 2 * nu * (N - 1)
    warps = min(16, 4 * (512 // tm), ((226 * 1024 - 1024 - pack_elems(nx, nu, N) * 4) // (sm * 4 * 32) // 4) * 4)
    assert warps >= 4, "shape does not fit the mixed-precision kernel"
    aff = ((nx, nu) == (6, 3)) if aff is None else aff
    return dict(gen=4, bits=32, nx=nx, nu=nu, N=N, feat=CON, refs=3 if refs else 0, ppb=False, fb=fb, variant=variant, block=warps * 32, aff=aff,
                opq=False, tib=False, tm=True, minb=1, ntm=0, cones=cones, ttm=-1)


def instg(nx, nu, N, variant=0, adapt=False, cones=None, rolled=False, models=False):
    """lane-group-per-problem fp64 kernel (tmpc_gpp.cuh): one lane per state row and per input row, groups of 8 / 16 / 32 lanes;
    models: its model-batch form (gen 6, box only: gpp_kernel MODE 3), whose rows come from each problem's own model"""
    gs = 8 if nx + nu <= 8 else (16 if nx + nu <= 16 else 32)
    assert nx + nu <= 32
    assert not (models and (adapt or cones))
    return dict(gen=6 if models else 5, bits=64, nx=nx, nu=nu, N=N, feat=CON if cones else (ADP if adapt else BOX), refs=2, ppb=False, fb=False,
                variant=variant, block=128, aff=True, gs=gs, cones=cones, rolled=rolled)


def cols_per_thread(nx, nu, N, feat, refs, ntm=0):
    """shared-memory scalar columns per thread; ntm = number of state-sized arrays (TV, GC, GL, SXT) in tensor memory"""
    sx, su = nx * N, nu * (N - 1)
    nstate = 4 if feat == CON else 1
    cols = (nstate - min(ntm, nstate)) * sx + 2 * su + ((sx + su) if refs == REFS_SMEM else 0)
    if feat == CON:
        cols += 3 * su + max(nx, nu)
    return cols


def pack_elems(nx, nu, N):
    sx, su = nx * N, nu * (N - 1)
    n = 2 * nx * nx + su                                  # cold tail: Pinf, dPinf, d0
    return n + 4 * (nx + 2) + 4 * (nu + 2) + 40           # + room for a few linear rows and padding


def plan_block(nx, nu, N, feat, bits, refs, budget_kb=226, tm=False, max_warps=16):
    """(threads per CTA, CTAs per SM) maximising resident problems per SM for the all-in-shared-memory state columns"""
    if tm:
        # one CTA per SM owns the 512 tensor-memory columns; warps w, w+4, ... share a lane quarter.  Pick the number
        # of state arrays to keep there (1 for box kernels, 1..4 with cones / linear rows) that maximises the residency.
        best = (0, 0)
        for ntm in range(1, (4 if feat == CON else 1) + 1):
            per_thread = cols_per_thread(nx, nu, N, feat, refs, ntm) * 4
            avail = budget_kb * 1024 - (1024 + pack_elems(nx, nu, N) * 4)
            warps = min(max_warps, avail // per_thread // 32, 4 * (512 // (ntm * nx * N)))
            warps = (warps // 4) * 4
            if warps > best[0]:
                best = (warps, ntm)
        return max(4, best[0]) * 32, max(1, best[1])
    per_thread = cols_per_thread(nx, nu, N, feat, refs) * bits // 8
    best = (32, 1, 0)
    for ctas in range(1, 9):
        avail = budget_kb * 1024 - ctas * (1024 + pack_elems(nx, nu, N) * bits // 8)
        block = min(256, (avail // ctas // per_thread // 32) * 32)
        while block >= 32 and (ctas * block // 32) % 4 != 0 and ctas * block > 128:
            block -= 32          # whole multiples of 4 warps per SM: the register file is split over 4 sub-partitions
        if block < 32:
            continue
        if ctas * block > best[2]:
            best = (block, ctas, ctas * block)
    return best[0], best[1]


def default_instances():
    out = []
    shapes = [(12, 4, 10), (4, 1, 20), (4, 1, 10), (6, 3, 10)]
    # fp32 box-constrained batches: the incremental ("delta") form, tmpc_tpp3.cuh -- the default (variant 0)
    for (nx, nu, N) in shapes:
        # hybrid state layout where it buys resident warps: the quadrotor shape goes from 8 to 12 warps per SM (+6.7 %)
        hyb = plan_hybrid(nx, nu, N) is not None and plan_hybrid(nx, nu, N)[0] > inst3(nx, nu, N)["block"] // 32
        for fb in (True, False):      # fb: bounds constant over the horizon and containing 0 (the common case)
            out.append(inst3(nx, nu, N, refs=True, fb=fb, hyb=hyb))
            out.append(inst3(nx, nu, N, refs=False, fb=fb, hyb=hyb))
        out.append(inst3(nx, nu, N, refs=True, ppb=True, hyb=hyb))
    # box + second-order cones + linear inequalities (rocket landing, rocket_landing_constraints.m:40-55: one cone on the
    # first three states, one on the three inputs): the same form with two more slack families, cone blocks compiled in
    # (+ one linear row on each side, SURVEY G4; the last two numbers are the row counts)
    # default (variant 0): the mixed-precision kernel, tmpc_tpp4.cuh (fp64 iterates, fp32 increments); the all-fp32 incremental
    # form of round 1 stays as the A/B baseline, option variant=3
    for fb in (True, False):
        out.append(inst4(6, 3, 10, refs=True, fb=fb, cones=(0, 3, 0, 3, 1, 1)))
        out.append(inst4(6, 3, 10, refs=True, fb=fb, cones=(0, 3, 0, 3, 0, 0)))
        out.append(inst3(6, 3, 10, refs=True, fb=fb, feat=CON, cones=(0, 3, 0, 3, 1, 1), variant=3))
        out.append(inst3(6, 3, 10, refs=True, fb=fb, feat=CON, cones=(0, 3, 0, 3, 0, 0), variant=3))
    # fp64 box families with shared bounds: the lane-group-per-problem kernel (tmpc_gpp.cuh) -- 20x shorter iteration, which is what
    # the second pass of the exact-count mode and small fp64 batches need, and a higher fp64 throughput as well
    for (nx, nu, N) in shapes:
        out.append(instg(nx, nu, N))
    out.append(instg(12, 4, 10, adapt=True))     # adaptive rho: the fp64 path of BASELINE config 5
    # model batches (tinympc_cuda_solve_batch_models) of fp64 box families with shared bounds: every problem its own model
    for (nx, nu, N) in shapes:
        out.append(instg(nx, nu, N, models=True))
    # rocket family (one cone per side, with and without the two linear rows): fp64 batches and the second pass of its exact-count mode
    out.append(instg(6, 3, 10, cones=(0, 3, 0, 3, 1, 1)))
    out.append(instg(6, 3, 10, cones=(0, 3, 0, 3, 0, 0)))
    for bits in (32, 64):
        for (nx, nu, N) in shapes:
            if bits == 64:            # fp64 thread-per-problem direct form (admm.cpp order), tmpc_tpp2.cuh: per-problem bounds; A/B (variant 6) otherwise
                for fb in (True, False):
                    out.append(inst(bits, nx, nu, N, BOX, refs=REFS_L2, fb=fb, tm=True, variant=6))
                    out.append(inst(bits, nx, nu, N, BOX, refs=REFS_NONE, fb=fb, tm=True, variant=6))
                out.append(inst(bits, nx, nu, N, BOX, refs=REFS_L2, ppb=True, tm=True))
            # fp32: the direct-form cone kernels stay as the A/B baseline (variant 5)
            out.append(inst(bits, nx, nu, N, CON, refs=REFS_L2, fb=True, tm=True, variant=0 if bits == 64 else 5))
            out.append(inst(bits, nx, nu, N, CON, refs=REFS_L2, tm=True, variant=0 if bits == 64 else 5))
            if (nx, nu) == (12, 4):   # adaptive rho, thread per problem: the fp32 kernels; fp64 is A/B (variant 6) next to tmpc_gpp.cuh
                out.append(inst(bits, nx, nu, N, ADP, refs=REFS_L2, fb=True, tm=True, variant=0 if bits == 32 else 6))
                out.append(inst(bits, nx, nu, N, ADP, refs=REFS_L2, tm=True, variant=0 if bits == 32 else 6))
    # The plain state layout (x and t entirely in tensor memory, 8 warps per SM) of the shapes whose default is the hybrid one: fewer
    # instructions per iteration and a 25 % shorter iteration of a lone warp.  The dispatcher picks it for batches that fit one
    # wave of it (tmpc_capi.cu, kLatencyVariant); option variant=9 forces it.
    for (nx, nu, N) in shapes:
        if plan_hybrid(nx, nu, N) is not None and plan_hybrid(nx, nu, N)[0] > inst3(nx, nu, N)["block"] // 32:
            for fb in (True, False):
                out.append(inst3(nx, nu, N, refs=True, fb=fb, variant=9))
                out.append(inst3(nx, nu, N, refs=False, fb=fb, variant=9))
            out.append(inst3(nx, nu, N, refs=True, ppb=True, variant=9))
    # A/B: the costate recursion instead of the impulse-response form of the backward pass (tmpc_tpp3.cuh, Tpp3Cfg::CONV), option variant=7
    out.append(inst3(12, 4, 10, refs=True, fb=True, hyb=True, variant=7, conv=0))
    # A/B: the direct-form fp32 box kernels (16 / 24 warps per SM, tensor-memory TV) on the headline shapes, option variant=5
    out.append(inst(32, 12, 4, 10, BOX, refs=REFS_L2, variant=5, fb=True, tm=True))
    out.append(inst(32, 12, 4, 10, BOX, refs=REFS_L2, variant=5, tm=True))
    out.append(inst(32, 12, 4, 10, BOX, refs=REFS_L2, variant=5, ppb=True, tm=True))
    out.append(inst(32, 4, 1, 20, BOX, refs=REFS_NONE, variant=5, fb=True, tm=True))
    out.append(inst(32, 4, 1, 20, BOX, refs=REFS_L2, variant=5, fb=True, tm=True))
    return out


def name_of(i):
    t = "f32" if i["bits"] == 32 else "f64"
    if i["gen"] in (5, 6):
        cn = ("_c" + "".join(str(c) for c in i["cones"])) if i.get("cones") else ""
        return f"gpp_f64_{i['nx']}x{i['nu']}x{i['N']}_{FEAT_NAME[i['feat']]}{cn}_g{i['gs']}_v{i['variant']}{'_mdl' if i['gen'] == 6 else ''}"
    if i["gen"] == 4:
        cn = "_c" + "".join(str(c) for c in i["cones"])
        return f"tpp4_mix_{i['nx']}x{i['nu']}x{i['N']}_con{cn}{'' if i['refs'] else '_noref'}{'_fb' if i['fb'] else ''}{'_aff' if i['aff'] else ''}_v{i['variant']}"
    if i["gen"] == 3:
        cn = ("_c" + "".join(str(c) for c in i["cones"])) if i["feat"] == CON else ""
        return (f"tpp3_f32_{i['nx']}x{i['nu']}x{i['N']}_{FEAT_NAME[i['feat']]}{cn}{'' if i['refs'] else '_noref'}{'_ppb' if i['ppb'] else ''}{'_fb' if i['fb'] else ''}"
                f"{'_aff' if i['aff'] else ''}_v{i['variant']}")
    return (f"tpp{'' if i['gen'] == 1 else '2'}_{t}_{i['nx']}x{i['nu']}x{i['N']}_{FEAT_NAME[i['feat']]}{['_noref', '_refsm', ''][i['refs']]}"
            f"{'_ppb' if i['ppb'] else ''}{'_fb' if i['fb'] else ''}{'_aff' if (i['aff'] and i['gen'] == 2) else ''}{'_tm' if i['tm'] else ''}_v{i['variant']}")


def gen_sources(instances):
    GEN.mkdir(parents=True, exist_ok=True)
    names = []
    wanted = set()
    for i in instances:
        n = name_of(i)
        names.append(n)
        T = "float" if i["bits"] == 32 else "double"
        g = "" if i["gen"] == 1 else "2"
        b = lambda v: "true" if v else "false"
        if i["gen"] == 5:
            src = (
                "// generated by tinympc-matlab_b200/build.py -- do not edit\n"
                '#include "../tmpc_gpp.cuh"\n#include "../tmpc_registry.h"\nusing namespace tmpc;\n'
                f"using Cfg_{n} = GppCfg<{i['nx']}, {i['nu']}, {i['N']}, {i['gs']}, {i['block']}, {b(i['feat'] == ADP)}"
                + (f", {', '.join(str(c) for c in i['cones'])}, true" if i.get("cones") else (", 0, 0, 0, 0, 0, 0, false, true" if i.get("rolled") else "")) + ">;\n"
                f"TMPC_DEFINE_GPP_ENTRY({n}, Cfg_{n}, {i['variant']})\n"
            )
        elif i["gen"] == 6:
            # gpp_kernel<Cfg, 3> next to the family instance's gpp_kernel<Cfg, 0>: the same configuration type, a different kernel
            # symbol.  The configuration is spelled with every template argument.
            src = (
                "// generated by tinympc-matlab_b200/build.py -- do not edit\n"
                '#include "../tmpc_gpp.cuh"\n#include "../tmpc_registry.h"\nusing namespace tmpc;\n'
                f"using Cfg_{n} = GppCfg<{i['nx']}, {i['nu']}, {i['N']}, {i['gs']}, {i['block']}, false, 0, 0, 0, 0, 0, 0, false, false>;\n"
                f"TMPC_DEFINE_GPP_MDL_ENTRY({n}, Cfg_{n}, {i['variant']})\n"
            )
        elif i["gen"] == 4:
            src = (
                "// generated by tinympc-matlab_b200/build.py -- do not edit\n"
                '#include "../tmpc_tpp4.cuh"\n#include "../tmpc_registry.h"\nusing namespace tmpc;\n'
                f"using Cfg_{n} = Tpp4Cfg<{i['nx']}, {i['nu']}, {i['N']}, {i['block']}, {b(i['refs'])}, {b(i['fb'])}, {b(i['aff'])}, "
                f"{', '.join(str(c) for c in i['cones'])}>;\n"
                f"TMPC_DEFINE_TPP4_ENTRY({n}, Cfg_{n}, {i['feat']}, 32, {i['variant']})\n"
            )
        elif i["gen"] == 3:
            src = (
                "// generated by tinympc-matlab_b200/build.py -- do not edit\n"
                '#include "../tmpc_tpp3.cuh"\n#include "../tmpc_registry.h"\nusing namespace tmpc;\n'
                f"using Cfg_{n} = Tpp3Cfg<{i['nx']}, {i['nu']}, {i['N']}, {i['block']}, {b(i['refs'])}, {b(i['ppb'])}, {b(i['fb'])}, {b(i['aff'])}, "
                f"{b(i['opq'])}, {b(i['tib'])}, {FEAT_ENUM[i['feat']]}, {', '.join(str(c) for c in i['cones'])}, {i['ttm']}, {i['conv']}>;\n"
                f"TMPC_DEFINE_TPP3_ENTRY({n}, Cfg_{n}, {i['feat']}, 32, {i['variant']})\n"
            )
        else:
          src = (
            "// generated by tinympc-matlab_b200/build.py -- do not edit\n"
            f'#include "../tmpc_tpp{g}.cuh"\n#include "../tmpc_registry.h"\nusing namespace tmpc;\n'
            f"using Cfg_{n} = Tpp{g}Cfg<{T}, {i['nx']}, {i['nu']}, {i['N']}, {FEAT_ENUM[i['feat']]}, {i['block']}, "
            f"{i['refs']}, {'true' if i['ppb'] else 'false'}, {i['minb']}, {'true' if i['fb'] else 'false'}"
            f"{((', true' if i['aff'] else ', false') + (', %d' % i['ntm']) + (', true' if i['opq'] else ', false') + (', true' if i['tib'] else ', false')) if g else ''}>;\n"
            f"TMPC_DEFINE_TPP{g}_ENTRY({n}, Cfg_{n}, {i['feat']}, {i['bits']}, {i['variant']})\n"
        )
        path = GEN / f"{n}.cu"
        wanted.add(path.name)
        if not path.exists() or path.read_text() != src:
            path.write_text(src)
    table = ["// generated by tinympc-matlab_b200/build.py -- do not edit", '#include "../tmpc_registry.h"', "namespace tmpc {"]
    table += [f"extern const KernelEntry {n};" for n in names]
    table.append("static const KernelEntry* const kTable[] = {" + ", ".join("&" + n for n in names) + "};")
    table.append("const KernelEntry* const* kernel_table(int* count) { *count = (int)(sizeof(kTable) / sizeof(kTable[0])); return kTable; }")
    table.append("}  // namespace tmpc\n")
    tpath = GEN / "tmpc_table.cu"
    wanted.add(tpath.name)
    txt = "\n".join(table)
    if not tpath.exists() or tpath.read_text() != txt:
        tpath.write_text(txt)
    for stale in GEN.glob("*.cu"):
        if stale.name not in wanted:
            stale.unlink()
            for ext in (".o", ".d"):
                (OBJ / (stale.stem + ext)).unlink(missing_ok=True)
    return [GEN / f"{n}.cu" for n in names] + [tpath]


def up_to_date(obj: Path, dep: Path, src: Path) -> bool:
    """obj is newer than its source and every header the compiler reported for it (nvcc -MD dependency file)"""
    if not (obj.exists() and dep.exists()):
        return False
    t = obj.stat().st_mtime
    if src.stat().st_mtime > t:
        return False
    toks = dep.read_text().replace("\\\n", " ").split()
    for f in toks[1:]:
        if f == ":" or f.startswith(("/usr/", "/opt/")):   # separator, toolchain headers
            continue
        try:
            if os.stat(f).st_mtime > t:
                return False
        except OSError:
            return False
    return True


def compile_one(src: Path, force: bool, log_dir: Path):
    obj = OBJ / (src.stem + ".o")
    dep = OBJ / (src.stem + ".d")
    if not force and up_to_date(obj, dep, src):
        return obj, None
    cmd = [NVCC, *ARCH, *FLAGS, "-MD", "-MF", str(dep), "-I", str(CSRC), "-I", str(HERE.parent / "include"), "-c", str(src), "-o", str(obj)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    (log_dir / (src.stem + ".log")).write_text(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src.name}:\n{r.stdout}\n{r.stderr}")
    return obj, r.stderr


def build(jobs: int | None = None, force: bool = False, verbose: bool = True) -> Path:
    OBJ.mkdir(exist_ok=True)
    log_dir = OBJ / "logs"
    log_dir.mkdir(exist_ok=True)
    srcs = gen_sources(default_instances()) + [CSRC / "tmpc_capi.cu"]
    srcs += sorted(CSRC.glob("tmpc_wpp*.cu")) + [CSRC / "tmpc_precompute.cu"] + sorted((CSRC / "host").glob("*.cpp"))
    jobs = jobs or os.cpu_count() or 4
    with ThreadPoolExecutor(max_workers=jobs) as ex:
        results = list(ex.map(lambda s: compile_one(s, force, log_dir), srcs))
    objs = [str(o) for o, _ in results]
    rebuilt = sum(1 for _, log in results if log is not None)
    if rebuilt or not LIB.exists():
        cmd = [NVCC, *ARCH, "-shared", "-o", str(LIB), *objs, "-cudart", "static"]
        subprocess.check_call(cmd)
    if verbose:
        print(f"[build] {len(srcs)} translation units ({rebuilt} recompiled) -> {LIB}")
        for _, log in results:
            if log:
                for line in log.splitlines():
                    if "spill" in line and "0 bytes spill stores" not in line:
                        print("[build] ptxas:", line.strip())
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("-j", type=int, default=None)
    ap.add_argument("--force", action="store_true")
    a = ap.parse_args()
    build(a.j, a.force)
