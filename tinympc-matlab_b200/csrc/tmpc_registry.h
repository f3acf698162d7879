// tmpc_registry.h -- table of compiled kernel instances the C-ABI layer dispatches over.
// Each instance lives in its own generated translation unit (csrc/gen/*.cu, written by
// tinympc-matlab_b200/build.py from its instance list) so that nvcc can compile them in parallel.
#pragma once
#include <cuda_runtime.h>

#include "tmpc_common.h"
#include "tmpc_wpp.h"

namespace tmpc {

enum KernelFamily : int { KF_TPP = 0, KF_WPP = 1 };

struct KernelEntry {
    const char* name;
    int family;          // KF_TPP: thread per problem (throughput);  KF_WPP: warp per problem (latency / generic shapes)
    int nx, nu, N;       // 0 = any (runtime-sized kernel)
    int feat;            // FEAT_BOX / FEAT_CONSTR / FEAT_ADAPT
    int dtype_bits;      // 32 or 64
    int refs;            // 0: reference-free variant (Xref = Uref = NULL); 1: reference terms in shared memory; 2: in an L2-resident scratch
    int ppb;             // per-problem bounds variant
    int fastbox;         // 1: requires shared bounds that are constant over the horizon and contain 0
    int affine;          // 1: handles a non-zero affine term (fdyn, APf, BPf); 0: requires f = 0
    int block;           // threads per CTA
    int variant;         // tuning variant (0 = default); selected with the "variant" option
    int streaming;       // 1: honours SolveParams::avail_ptr / done_counters (the single-launch streamed host pipeline)
    size_t (*smem_bytes)(int pack_elems);
    cudaError_t (*prepare)(size_t smem);                                   // cudaFuncSetAttribute(max dynamic smem)
    cudaError_t (*occupancy)(int* ctas_per_sm, size_t smem);
    // master_pack: the family's double-precision pack (PackLayout L) on the host; the launcher
    // converts the hot tables into the kernel-parameter constant pack
    cudaError_t (*launch)(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* master_pack, const PackLayout& L);
    // 1: the second-order cones are compiled into the instance -- it serves only families whose cone list is exactly one
    // state cone on [scs, scs + scd) and one input cone on [ucs, ucs + ucd) (dim 0 = that side has no cone)
    // ... and so are the numbers of linear-inequality rows (state, input)
    int cone_fixed;
    int scs, scd, ucs, ucd, nsl, nil;
    int lanes_per_problem;   // 0 / 1: thread per problem; GS: a problem is spread over GS lanes (tmpc_gpp.cuh), a CTA holds block / GS problems
    // sessions (tinympc_cuda_session_solve): iterate p.batch persistent double-precision workspaces of layout W in place; NULL = the
    // instance has no session form (the warp-per-problem kernel serves the session)
    cudaError_t (*session_launch)(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* master_pack, const PackLayout& L,
                                  double* ws, const WppLayout& W, int full);
    // 1: honours SolveParams::xref_const (Xref = one state per problem, read in place of every column of the horizon) and
    // SolveParams::u0 (first control as the only solution output); 0: the library expands a compact reference on the device
    // before the launch and gathers u0 from the full trajectories after it
    int compact_ok;
    // 1: honours SolveParams::order_from (a streamed batch whose later part is claimed through a list built meanwhile)
    int order_from_ok;
    // 1: a model-batch instance (tinympc_cuda_solve_batch_models): launched through models_launch only, never for a family batch
    int models;
    cudaError_t (*models_launch)(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* master_pack, const PackLayout& L,
                                 const tinympc_cuda_models& m);
    // sparse-A instances (Tpp3Cfg::SA): the compiled nonzero pattern of A, a_cols (= nx) column masks of row pairs (bit j: rows 2j,
    // 2j+1; bit nx / 2: the odd tail row).  They serve only families whose float32 A is zero outside it.  a_cols = 0: dense.
    int a_cols;
    const unsigned* a_pairs;
    // model sessions (tinympc_cuda_session_create_models): session_launch on workspaces whose solvers each carry their own model, m
    // (device pointers, every solver's model resident); NULL = the warp-per-problem kernel serves them
    cudaError_t (*models_session_launch)(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* master_pack,
                                         const PackLayout& L, double* ws, const WppLayout& W, const tinympc_cuda_models& m);
};

const KernelEntry* const* kernel_table(int* count);   // defined in gen/tmpc_table.cu

}  // namespace tmpc

// one of these per generated translation unit
// packed-pair kernel (tmpc_tpp2.cuh)
#define TMPC_DEFINE_TPP2_ENTRY(SYM, CFG, FEATV, BITS, VAR)                                                          \
    namespace tmpc {                                                                                                \
    static size_t SYM##_smem(int pe) { return tpp2_smem_bytes<CFG>(pe); }                                           \
    static cudaError_t SYM##_prepare(size_t smem) {                                                                 \
        return cudaFuncSetAttribute(tpp2_kernel<CFG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);      \
    }                                                                                                               \
    static cudaError_t SYM##_occ(int* n, size_t smem) {                                                             \
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, tpp2_kernel<CFG>, CFG::BLOCK, smem);                \
    }                                                                                                               \
    static cudaError_t SYM##_launch(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* mp, \
                                    const PackLayout& L) {                                                          \
        typename CFG::CPack cpk;                                                                                    \
        fill_const_pack2(cpk, mp, L);                                                                               \
        tpp2_kernel<CFG><<<grid, CFG::BLOCK, smem, st>>>(p, cpk);                                                   \
        return cudaGetLastError();                                                                                  \
    }                                                                                                               \
    extern const KernelEntry SYM = {#SYM, KF_TPP, CFG::NX, CFG::NU, CFG::NH, FEATV, BITS, CFG::REFMODE,             \
                                    CFG::PPB ? 1 : 0, CFG::FB ? 1 : 0, CFG::AFF ? 1 : 0, CFG::BLOCK, VAR, 1, SYM##_smem, SYM##_prepare, \
                                    SYM##_occ, SYM##_launch};                                 \
    }

// incremental-form kernel (tmpc_tpp3.cuh)
#define TMPC_DEFINE_TPP3_ENTRY(SYM, CFG, FEATV, BITS, VAR)                                                          \
    namespace tmpc {                                                                                                \
    static size_t SYM##_smem(int pe) { return tpp3_smem_bytes<CFG>(pe); }                                           \
    static cudaError_t SYM##_prepare(size_t smem) {                                                                 \
        return cudaFuncSetAttribute(tpp3_kernel<CFG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);      \
    }                                                                                                               \
    static cudaError_t SYM##_occ(int* n, size_t smem) {                                                             \
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, tpp3_kernel<CFG>, CFG::BLOCK, smem);                \
    }                                                                                                               \
    static cudaError_t SYM##_launch(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* mp, \
                                    const PackLayout& L) {                                                          \
        typename CFG::CPack cpk;                                                                                    \
        fill_const_pack3(cpk, mp, L);                                                                               \
        tpp3_kernel<CFG><<<grid, CFG::BLOCK, smem, st>>>(p, cpk);                                                   \
        return cudaGetLastError();                                                                                  \
    }                                                                                                               \
    extern const KernelEntry SYM = {#SYM, KF_TPP, CFG::NX, CFG::NU, CFG::NH, FEATV, BITS, CFG::REFMODE,             \
                                    CFG::PPB ? 1 : 0, CFG::FB ? 1 : 0, CFG::AFF ? 1 : 0, CFG::BLOCK, VAR, 1, SYM##_smem, SYM##_prepare, \
                                    SYM##_occ, SYM##_launch, CFG::CONSTR ? 1 : 0, CFG::SCS, CFG::SCD, CFG::UCS, CFG::UCD, CFG::NSL, CFG::NIL, \
                                    0, nullptr, 1, 1, 0, nullptr, CFG::SA::NCOL, CFG::SA::kCols};                  \
    }

// mixed-precision rocket-family kernel (tmpc_tpp4.cuh)
#define TMPC_DEFINE_TPP4_ENTRY(SYM, CFG, FEATV, BITS, VAR)                                                          \
    namespace tmpc {                                                                                                \
    static size_t SYM##_smem(int pe) { return tpp4_smem_bytes<CFG>(pe); }                                           \
    static cudaError_t SYM##_prepare(size_t smem) {                                                                 \
        return cudaFuncSetAttribute(tpp4_kernel<CFG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);      \
    }                                                                                                               \
    static cudaError_t SYM##_occ(int* n, size_t smem) {                                                             \
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, tpp4_kernel<CFG>, CFG::BLOCK, smem);                \
    }                                                                                                               \
    static cudaError_t SYM##_launch(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* mp, \
                                    const PackLayout& L) {                                                          \
        typename CFG::CPack cpk;                                                                                    \
        fill_const_pack3(cpk, mp, L);                                                                               \
        tpp4_kernel<CFG><<<grid, CFG::BLOCK, smem, st>>>(p, cpk);                                                   \
        return cudaGetLastError();                                                                                  \
    }                                                                                                               \
    extern const KernelEntry SYM = {#SYM, KF_TPP, CFG::NX, CFG::NU, CFG::NH, FEATV, BITS, CFG::REFMODE,             \
                                    0, CFG::FB ? 1 : 0, CFG::AFF ? 1 : 0, CFG::BLOCK, VAR, 1, SYM##_smem, SYM##_prepare, \
                                    SYM##_occ, SYM##_launch, 1, CFG::SCS, CFG::SCD, CFG::UCS, CFG::UCD, CFG::NSL, CFG::NIL};                                 \
    }

// lane-group-per-problem fp64 kernel (tmpc_gpp.cuh)
#define TMPC_DEFINE_GPP_ENTRY(SYM, CFG, VAR)                                                                        \
    namespace tmpc {                                                                                                \
    static size_t SYM##_smem(int pe) { return gpp_smem_bytes<CFG>(pe); }                                            \
    static cudaError_t SYM##_prepare(size_t smem) {                                                                 \
        return cudaFuncSetAttribute(gpp_kernel<CFG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
    }                                                                                                               \
    static cudaError_t SYM##_occ(int* n, size_t smem) {                                                             \
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, gpp_kernel<CFG>, CFG::BLOCK, smem);                 \
    }                                                                                                               \
    static cudaError_t SYM##_launch(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* mp, \
                                    const PackLayout& L) {                                                          \
        GppTab<CFG::NX, CFG::NU, CFG::NH, CFG::GS, CFG::ADAPT> tab;                                                           \
        fill_gpp_tab(tab, mp, L, p);                                                                                \
        gpp_kernel<CFG><<<grid, CFG::BLOCK, smem, st>>>(p, tab, GppSession{});                                      \
        return cudaGetLastError();                                                                                  \
    }                                                                                                               \
    static cudaError_t SYM##_session(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* mp,\
                                     const PackLayout& L, double* ws, const WppLayout& W, int full) {               \
        if constexpr (CFG::ADAPT || CFG::CONSTR) { return cudaErrorNotSupported; } else {                                          \
        GppTab<CFG::NX, CFG::NU, CFG::NH, CFG::GS, CFG::ADAPT> tab;                                                 \
        fill_gpp_tab(tab, mp, L, p);                                                                                \
        auto go = [&](auto kernel) -> cudaError_t {                                                                 \
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
            if (e != cudaSuccess) return e;                                                                         \
            kernel<<<grid, CFG::BLOCK, smem, st>>>(p, tab, GppSession{ws, W, full});                                \
            return cudaGetLastError();                                                                              \
        };                                                                                                          \
        return full ? go(gpp_kernel<CFG, 2>) : go(gpp_kernel<CFG, 1>); }                                            \
    }                                                                                                               \
    extern const KernelEntry SYM = {#SYM, KF_TPP, CFG::NX, CFG::NU, CFG::NH, CFG::CONSTR ? 1 : (CFG::ADAPT ? 2 : 0) /* FEAT_CONSTR : FEAT_ADAPT : FEAT_BOX */, 64, 1 /* serves batches with and without references */, \
                                    0, 0, 1, CFG::BLOCK, VAR, 1, SYM##_smem, SYM##_prepare,                        \
                                    SYM##_occ, SYM##_launch, CFG::CONSTR ? 1 : 0, CFG::SCS, CFG::SCD, CFG::UCS, CFG::UCD, CFG::NSL, CFG::NIL, CFG::GS,     \
                                    (CFG::ADAPT || CFG::CONSTR) ? nullptr : SYM##_session, 1};                      \
    }

// model-batch form of the lane-group-per-problem fp64 kernel (gpp_kernel MODE 3): the shared bounds come from the family's table,
// every other row from the claimed problem's model; and its session form (MODE 4, reported as SYM_session)
#define TMPC_DEFINE_GPP_MDL_ENTRY(SYM, CFG, VAR)                                                                    \
    namespace tmpc {                                                                                                \
    static_assert(!CFG::ADAPT && !CFG::CONSTR, "model batches: box families only");                                 \
    static size_t SYM##_smem(int pe) { return gpp_smem_bytes<CFG>(pe); }                                            \
    static cudaError_t SYM##_prepare(size_t smem) {                                                                 \
        return cudaFuncSetAttribute(gpp_kernel<CFG, kGppModels>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);    \
    }                                                                                                               \
    static cudaError_t SYM##_occ(int* n, size_t smem) {                                                             \
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, gpp_kernel<CFG, kGppModels>, CFG::BLOCK, smem);              \
    }                                                                                                               \
    static cudaError_t SYM##_launch(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* mp, \
                                    const PackLayout& L, const tinympc_cuda_models& m) {                            \
        GppTab<CFG::NX, CFG::NU, CFG::NH, CFG::GS, false> tab;                                                      \
        fill_gpp_tab(tab, mp, L, p);                                                                                \
        GppSession ses{};                                                                                           \
        ses.models = m;                                                                                             \
        gpp_kernel<CFG, kGppModels><<<grid, CFG::BLOCK, smem, st>>>(p, tab, ses);                                            \
        return cudaGetLastError();                                                                                  \
    }                                                                                                               \
    static cudaError_t SYM##_session(const SolveParams& p, int grid, size_t smem, cudaStream_t st, const double* mp,\
                                     const PackLayout& L, double* ws, const WppLayout& W, const tinympc_cuda_models& m) { \
        GppTab<CFG::NX, CFG::NU, CFG::NH, CFG::GS, false> tab;                                                      \
        fill_gpp_tab(tab, mp, L, p);                                                                                \
        cudaError_t e = cudaFuncSetAttribute(gpp_kernel<CFG, kGppModelSession>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return e;                                                                             \
        GppSession ses{ws, W, 0};                                                                                   \
        ses.models = m;                                                                                             \
        gpp_kernel<CFG, kGppModelSession><<<grid, CFG::BLOCK, smem, st>>>(p, tab, ses);                             \
        return cudaGetLastError();                                                                                  \
    }                                                                                                               \
    extern const KernelEntry SYM = {#SYM, KF_TPP, CFG::NX, CFG::NU, CFG::NH, 0 /* FEAT_BOX */, 64, 1, 0, 0, 1, CFG::BLOCK, VAR, 0, \
                                    SYM##_smem, SYM##_prepare, SYM##_occ, nullptr, 0, 0, 0, 0, 0, 0, 0, CFG::GS, nullptr, 1, 0, \
                                    1, SYM##_launch, 0, nullptr, SYM##_session};                                    \
    }
