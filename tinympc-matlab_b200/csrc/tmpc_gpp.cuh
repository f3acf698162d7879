// tmpc_gpp.cuh -- "lane group per problem" ADMM kernel for sm_100a, fp64: the low-latency form of the hot path.
//
// Path (reference: tinympc/TinyMPC/src/tinympc/admm.cpp): solve :274-389 with backward_pass_grad :13-20, forward_pass :25-32,
// update_slack (box) :81-98, update_dual :181-187, update_linear_cost :214-247, termination_condition :253-271 -- direct form,
// reference order (backward, forward, slack, dual, linear cost, check), double precision.
//
// Why a second mapping.  The thread-per-problem kernels (tmpc_tpp2/3.cuh) run a problem's ~9 000 instructions per ADMM iteration
// on ONE thread: unbeatable for throughput when a million problems are waiting, but an fp64 iteration then takes ~37 us of
// dependent issue, and the exact-count mode (fp32 pass + fp64 re-solve of the few problems whose termination decision is too
// close to call) ends with a tail of up to max_iter x 37 us = 3.7 ms during which the GPU is nearly idle.  Here a problem is
// spread over a group of GS = 8 / 16 lanes of a warp -- the north-star mapping (problem per warp, shuffle reductions):
//   * lane l < NX owns ROW l of the state trajectory, lane NX + a owns row a of the input trajectory; each keeps its row of
//     the slack, the dual and the reference term for ALL time steps in registers (the time loops are fully unrolled, so the
//     arrays are statically indexed);
//   * every lane holds its rows of the matrices in registers (2 x (NX + NU) doubles).  Substituting u = -Kinf x - d into the
//     rollout, both sweeps become ONE fused product per time step in which state and input lanes run the same instruction
//     stream on different coefficients:
//        forward :  state lane r: x_{i+1,r} = (A - B Kinf)_r . x_i - B_r . d_i + f_r      input lane a: u_{i,a} = -Kinf_a . x_i - d_{i,a}
//        backward:  state lane r: p_{i,r} = q_{i,r} + AmBKt_r . p_{i+1} - Kinf'_r . r_i + APf_r
//                   input lane a: d_{i,a} = (Quu_inv B')_a . p_{i+1} + Quu_inv_a . r_i + (Quu_inv BPf)_a
//     (NX + NU = 16 DFMA per lane and step, four independent chains; the products Quu_inv B' and A - B Kinf are formed once on
//     the host in double -- 1e-16 relative to the reference's order of operations);
//   * the vector a step produces (x_{i+1}, or p_i and r_{i-1}) is handed to the group through a double-buffered shared-memory
//     slot: one 8-byte store per lane, __syncwarp, NX/2 + NU/2 broadcast 16-byte loads;
//   * slack, dual, linear-cost and residual terms are element-wise on the owning lane; the four infinity norms are shuffle
//     max-reductions over the group (admm.cpp:257-260).
// One ADMM iteration of the quadrotor shape is 18 such steps of ~45 instructions: 2.0 us on a lone warp, 18x shorter than the
// thread-per-problem fp64 iteration, and -- because the FP64 pipe sees four chains per lane and two problems per warp -- twice the
// fp64 throughput as well (23 against 11 M quadrotor solves/s).  Modes and variants of the one kernel:
//   batch (MODE 0)      fp64 batches (precision = 64), the second pass of the exact-count mode (index list or device queue, same
//                       SolveParams protocol as tmpc_tpp2.cuh), small batches of the compiled shapes
//   ADAPT               adaptive rho in the closed block form of rho_benchmark.cpp:146-212 (a rolled pass over parked columns)
//   CONSTR / ROLLED     the rocket family: one second-order cone per side and 0/1 linear rows; per-slot state in shared memory and
//                       rolled time loops, because the unrolled form no longer fits the 32 KB instruction cache
//   session (MODE 1)    persistent TinyWorkspace images iterated in place with the reference's warm-start semantics
//   workspace (MODE 2)  the same for ONE live workspace, every member written back: tiny_solve
//   models (MODE 3)     model batches (tinympc_cuda_solve_batch_models): a group that claims a problem loads its lanes' rows from that
//                       problem's own model and forms the products on the device in the host's order (fill_gpp_tab); box only
//   model session (MODE 4)  MODE 1 on the workspaces of a model session (tinympc_cuda_session_create_models): the workspace as in
//                       MODE 1, the lanes' rows from the solver's resident model as in MODE 3
#pragma once
#include "tmpc_tpp2.cuh"
#include "tmpc_wpp.h"

namespace tmpc {

template <int NX_, int NU_, int NH_, int GS_, int BLOCK_ = 128, bool ADAPT_ = false,
          int SCS_ = 0, int SCD_ = 0, int UCS_ = 0, int UCD_ = 0, int NSL_ = 0, int NIL_ = 0, bool CONSTR_ = false, bool ROLLED_ = CONSTR_>
struct GppCfg {
    using T = double;
    static constexpr int NX = NX_, NU = NU_, NH = NH_, GS = GS_, BLOCK = BLOCK_;
    static constexpr bool ADAPT = ADAPT_;   // adaptive rho (rho_benchmark.cpp:44-250 in closed block form, SURVEY.md section 8 a-8)
    // cone / half-space families (admm.cpp:100-175): at most one second-order cone per side on the elements [SCS, SCS + SCD) /
    // [UCS, UCS + UCD) (dim 0 = none) and at most one linear row per side, compiled into the instance like in tmpc_tpp3/4.cuh
    static constexpr bool CONSTR = CONSTR_;
    static constexpr int SCS = SCS_, SCD = SCD_, UCS = UCS_, UCD = UCD_, NSL = NSL_, NIL = NIL_;
    static_assert(CONSTR_ || (SCD_ == 0 && UCD_ == 0 && NSL_ == 0 && NIL_ == 0), "cones / rows need CONSTR");
    static_assert(!(CONSTR_ && ADAPT_), "adaptive rho with cones / rows stays on the warp-per-problem kernel");
    static_assert(NSL_ <= 1 && NIL_ <= 1 && SCS_ + SCD_ <= NX_ && UCS_ + UCD_ <= NU_, "one row per side; cone block inside the vector");
    static_assert(GS_ == 8 || GS_ == 16 || GS_ == 32, "group size: 8, 16 or 32 lanes");
    static_assert(NX_ + NU_ <= GS_, "one lane per state row and input row");
    static_assert(NX_ % 2 == 0 || true, "");
    // ROLLED: the per-slot state of the lane (dual, slack, reference, family duals) lives in shared memory instead of registers and
    // the two time loops stay rolled.  The cone / half-space families add ~150 instructions per step: unrolled, the loop of the rocket
    // instance was 47 KB -- past the 32 KB instruction cache -- and ran at a third of the box kernel's rate.
    static constexpr bool ROLLED = ROLLED_;
    static constexpr int TUNROLL = ROLLED ? 1 : 64;
    static constexpr int NSTATE = ROLLED ? (CONSTR_ ? 6 : 3) : 0;   // shared-memory state arrays per lane: G, V, RF (+ GC, GL, EC)
    // Register budget: the full 255 (two CTAs of 128 threads per SM).  Aiming at three CTAs (168 registers) made ptxas spill a few words
    // and re-read launch parameters inside the dependent chain of every step: 37 % slower in bulk (16.7 against 23.0 M fp64 quadrotor
    // solves/s) in spite of the 50 % more resident warps -- the kernel is bound by the latency of one group's step, not by issue.
    static constexpr int MINB = 2;        // CTAs per SM the register allocation aims at (the per-lane state grows with N)
    static constexpr int GPW = 32 / GS_;                 // problems per warp
    static constexpr int GPB = BLOCK_ / GS_;             // problems per CTA
    static constexpr int NV = NX_ + NU_;
    static constexpr int NXP = (NX_ + 1) & ~1, NUP = (NU_ + 1) & ~1;   // exchange slots padded to 16 bytes
    // shared memory per group (doubles): forward slot x (2 buffers), backward slot [p | r] (2 buffers), table of d (N-1 steps)
    static constexpr int oXB = 0, oPB = 2 * NXP, oDT = oPB + 2 * (NXP + NUP), oTC = oDT + (NH_ - 1) * NUP;   // oTC: [2 buffers][2][GS] pre-projection slacks (CONSTR)
    static constexpr int GWORDS = oTC + (CONSTR_ ? 4 * GS_ : 0);
    static constexpr int SX = NX_ * NH_, SU = NU_ * (NH_ - 1);
};

// Per-lane tables, built on the host in double from the family's master pack and passed in the kernel-parameter space.
template <int NX, int NU, int NH, int GS, bool ADAPT = false>
struct alignas(16) GppTab {
    double CF1[GS][NX], CF2[GS][NU], cf0[GS];     // forward : acc = cf0 + CF1 . x_i + CF2 . d_i
    double CB1[GS][NX], CB2[GS][NU], cb0[GS];     // backward: acc = cb0 + CB1 . p_{i+1} + CB2 . r_i (+ q_i on state lanes)
    double wref[GS];                               // Qd_r / Rd_a: weight of the lane's reference term (work->Q, work->R)
    double lo[NH][GS], hi[NH][GS];                 // box of the element the lane handles in forward slot s (state: column s + 1; input: step s); row NH-1: column 0
    double Pinf[NX][NX];                           // row-major: terminal term -(xref_N' Pinf)'
    // cone / half-space families: the one linear row of each side (coefficients, offset, ||a||^2)
    double ax[NX], au[NU], bx, bu, nrx, nru;     // nrx, nru = 1 / ||a||^2
    // adaptive rho: d/drho of the rows that contain Kinf (Kinf, Pinf move with rho; Quu_inv and AmBKt do not: the reference updates
    // its copies C1, C2, which the sweeps never read), the rows of A' / B' for the dual residual, dPinf/drho
    double dCF1[ADAPT ? GS : 1][NX], dCB2[ADAPT ? GS : 1][NU], AT[ADAPT ? GS : 1][NX], dPinf[ADAPT ? NX : 1][NX];
};

template <int NX, int NU, int NH, int GS, bool ADAPT>
inline void fill_gpp_tab(GppTab<NX, NU, NH, GS, ADAPT>& t, const double* pk, const PackLayout& L, const SolveParams& prm) {
    std::memset(&t, 0, sizeof(t));
    const double* A = pk + L.A; const double* B = pk + L.B; const double* K = pk + L.Kinf; const double* AK = pk + L.AmBKt;
    const double* Qi = pk + L.Quu_inv;
    const double inf = 1.0 / 0.0;
    for (int l = 0; l < GS; ++l) for (int s = 0; s < NH; ++s) { t.lo[s][l] = -inf; t.hi[s][l] = inf; }
    for (int r = 0; r < NX; ++r) {   // state lanes
        for (int c = 0; c < NX; ++c) {
            double acc = A[r * NX + c];
            for (int a = 0; a < NU; ++a) acc -= B[r * NU + a] * K[a * NX + c];     // (A - B Kinf)[r][c]
            t.CF1[r][c] = acc;
            t.CB1[r][c] = AK[r * NX + c];
        }
        for (int a = 0; a < NU; ++a) { t.CF2[r][a] = -B[r * NU + a]; t.CB2[r][a] = -K[a * NX + r]; }
        t.cf0[r] = pk[L.f + r];
        t.cb0[r] = pk[L.APf + r];
        t.wref[r] = pk[L.Qd + r];
        if (prm.en_state_bound)
            for (int s = 0; s < NH; ++s) {
                const int col = s == NH - 1 ? 0 : s + 1;
                t.lo[s][r] = pk[L.xmin + col * NX + r]; t.hi[s][r] = pk[L.xmax + col * NX + r];
            }
    }
    for (int a = 0; a < NU; ++a) {   // input lanes
        const int l = NX + a;
        for (int c = 0; c < NX; ++c) {
            t.CF1[l][c] = -K[a * NX + c];
            double acc = 0.0;
            for (int b = 0; b < NU; ++b) acc += Qi[a * NU + b] * B[c * NU + b];   // (Quu_inv B')[a][c]
            t.CB1[l][c] = acc;
        }
        for (int b = 0; b < NU; ++b) { t.CF2[l][b] = (a == b) ? -1.0 : 0.0; t.CB2[l][b] = Qi[a * NU + b]; }
        double acc = 0.0;
        for (int b = 0; b < NU; ++b) acc += Qi[a * NU + b] * pk[L.BPf + b];
        t.cb0[l] = acc;
        t.wref[l] = pk[L.Rd + a];
        if (prm.en_input_bound)
            for (int s = 0; s < NH - 1; ++s) { t.lo[s][l] = pk[L.umin + s * NU + a]; t.hi[s][l] = pk[L.umax + s * NU + a]; }
    }
    for (int r = 0; r < NX; ++r) for (int c = 0; c < NX; ++c) t.Pinf[r][c] = pk[L.Pinf + r * NX + c];
    t.nrx = t.nru = 1.0;
    if (L.nsl > 0) { for (int e = 0; e < NX; ++e) t.ax[e] = pk[L.Alin_x + e]; t.bx = pk[L.blin_x]; t.nrx = 1.0 / pk[L.nrm_x]; }
    if (L.nil > 0) { for (int e = 0; e < NU; ++e) t.au[e] = pk[L.Alin_u + e]; t.bu = pk[L.blin_u]; t.nru = 1.0 / pk[L.nrm_u]; }
    if constexpr (ADAPT) {
        const double* dK = pk + L.dKinf;
        for (int r = 0; r < NX; ++r) {
            for (int c = 0; c < NX; ++c) {
                double acc = 0.0;
                for (int a = 0; a < NU; ++a) acc -= B[r * NU + a] * dK[a * NX + c];      // d/drho (A - B Kinf)[r][c]
                t.dCF1[r][c] = acc;
                t.AT[r][c] = A[c * NX + r];                                               // (A' g)_r = sum_c A[c][r] g_c
                t.dPinf[r][c] = pk[L.dPinf + r * NX + c];
            }
            for (int a = 0; a < NU; ++a) t.dCB2[r][a] = -dK[a * NX + r];
        }
        for (int a = 0; a < NU; ++a) {
            const int l = NX + a;
            for (int c = 0; c < NX; ++c) { t.dCF1[l][c] = -dK[a * NX + c]; t.AT[l][c] = B[c * NU + a]; }   // (B' g)_a = sum_c B[c][a] g_c
        }
    }
}

// Session mode (tinympc_cuda_session_*, SURVEY.md 8 f-1): `batch` persistent solver workspaces in the layout of the warp-per-problem
// kernel (WppLayout, the members of TinyWorkspace in double) are iterated IN PLACE with the reference's warm-start semantics
// (admm.cpp:291-292, 379-380): the first backward pass runs on the q, r, p_N the previous solve left behind, the first dual residual
// compares against the stored work->v / work->z, and on exit x, u, vnew, znew, v, z, g, y, q, r, p_N, iter, status and the residuals go
// back (d and the inner columns of p are recomputed by every solve before they are read and are not written).
struct GppSession {
    double* ws;        // batch * W.size doubles, or NULL (batch mode)
    WppLayout W;
    int full;          // informational: the launcher instantiates MODE 2 (also write d, every column of p and the unused columns 0 and N-1
                       // of q: tiny_solve on ONE live workspace, whose owner may look at any member of TinyWorkspace afterwards) or MODE 1
    tinympc_cuda_models models;   // MODE 3 (model batches): the per-problem model arrays, device pointers; the tables of `tab` other
                                  // than the bounds are not read
};

// per-slot state of a lane: registers (statically indexed, unrolled time loops) or a shared-memory column [slot][thread]
template <typename E, int N> struct RegArr {
    E a[N];
    __device__ __forceinline__ E& operator[](int i) { return a[i]; }
    __device__ __forceinline__ const E& operator[](int i) const { return a[i]; }
};
template <typename E, int STRIDE> struct SmemArr {
    E* p;
    __device__ __forceinline__ E& operator[](int i) const { return p[i * STRIDE]; }
};

// max / min / clamp of finite-or-infinite doubles as one compare + select: the library fmax / fmin carry NaN handling that costs
// ~8 instructions per call in fp64, and this kernel takes ~6 of them per element and step (no NaN can arise: bounds may be infinite,
// iterates are finite).
__device__ __forceinline__ double gmax(double a, double b) { return a > b ? a : b; }
__device__ __forceinline__ double gmin(double a, double b) { return a < b ? a : b; }
// max(r, |a|) for r >= 0 without touching the FP64 pipe for the absolute value (the sign bit is cleared on the selected word)
__device__ __forceinline__ double gabsmax(double r, double a) {
    const bool keep = r > fabs(a);
    return __hiloint2double(keep ? __double2hiint(r) : (__double2hiint(a) & 0x7fffffff), keep ? __double2loint(r) : __double2loint(a));
}
__device__ __forceinline__ double gclamp(double t, double lo, double hi) { return gmin(hi, gmax(lo, t)); }   // admm.cpp:91-98 order

constexpr int kGppModels = 3;      // gpp_kernel MODE of model batches
constexpr int kGppModelSession = 4;   // gpp_kernel MODE of model sessions

template <class C, int MODE = 0>   // 0: batch; 1: sessions (what the next warm start reads is written back); 2: tiny_solve on one live workspace (every member);
                                   // 3: model batch (every problem brings its own matrices and cache, ses.models); 4: model session (1 with the rows of 3)
__global__ void __launch_bounds__(C::BLOCK, C::MINB)
gpp_kernel(const __grid_constant__ SolveParams prm, const __grid_constant__ GppTab<C::NX, C::NU, C::NH, C::GS, C::ADAPT> tab,
           const __grid_constant__ GppSession ses) {
    // (model mode is tested as MODE == kGppModels: one more constexpr local here changes the machine code of the other modes)
    constexpr bool SESSION = MODE == 1 || MODE == 2 || MODE == kGppModelSession, FULLWS = MODE == 2;
    static_assert(!(SESSION && C::ADAPT), "adaptive-rho sessions keep a cache per problem: they stay on the warp-per-problem kernel");
    static_assert(!((MODE == kGppModels || MODE == kGppModelSession) && (C::ADAPT || C::CONSTR)), "model batches with adaptive rho, cones or rows stay on the warp-per-problem kernel");
    using T = double;
    constexpr int NX = C::NX, NU = C::NU, NH = C::NH, GS = C::GS, NXP = C::NXP, NUP = C::NUP, SXL = C::SX, SUL = C::SU;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char gpp_smem[];
    T* const gbase = reinterpret_cast<T*>(gpp_smem) + (size_t)(threadIdx.x / GS) * C::GWORDS;
    T* const lo_t = reinterpret_cast<T*>(gpp_smem) + (size_t)C::GPB * C::GWORDS;   // [NH][GS] per CTA (identical for every group)
    T* const hi_t = lo_t + NH * GS;

    const int lane = threadIdx.x & 31;
    const int l = lane % GS;                       // role within the group
    const int gl0 = lane - l;                      // first lane of this group
    const bool is_x = l < NX, is_u = l >= NX && l < NX + NU;
    const int row = is_x ? l : (is_u ? l - NX : 0);
    const int lc = (is_x || is_u) ? l : 0;         // idle lanes compute lane 0's (discarded) values

    // adaptive rho: the rows read with a lane-dependent index at every adaptation live in shared memory (a divergent read of the
    // kernel-parameter bank is serialised address by address)
    T* const at_t = hi_t + NH * GS;                  // [GS][NX]  rows of A' / B'
    T* const dcf1_t = at_t + GS * NX;                // [GS][NX]
    T* const dcb2_t = dcf1_t + GS * NX;              // [GS][NU]
    T* const pinf_t = dcb2_t + GS * NU;              // [NX][NX]
    T* const dpinf_t = pinf_t + NX * NX;             // [NX][NX]
    // parking area: this lane's iterate and (adaptive rho) updated dual / (sessions) previous slack of every slot,
    // [group][array][slot][lane of the group]
    T* const sval = (C::ADAPT ? dpinf_t + NX * NX : hi_t + NH * GS + (size_t)C::NSTATE * NH * C::BLOCK) + (size_t)(threadIdx.x / GS) * 2 * NH * GS + l;
    T* const sdual = sval + NH * GS;
    T* const sold = sdual;      // sessions: work->v / work->z as the last iteration found it (adaptive rho and sessions never combine)
    for (int e = threadIdx.x; e < NH * GS; e += C::BLOCK) { lo_t[e] = tab.lo[e / GS][e % GS]; hi_t[e] = tab.hi[e / GS][e % GS]; }
    if constexpr (C::ADAPT) {
        for (int e = threadIdx.x; e < GS * NX; e += C::BLOCK) { at_t[(e % NX) * GS + e / NX] = tab.AT[e / NX][e % NX]; dcf1_t[(e % NX) * GS + e / NX] = tab.dCF1[e / NX][e % NX]; }   // [c][lane]: conflict free
        for (int e = threadIdx.x; e < GS * NU; e += C::BLOCK) dcb2_t[(e % NU) * GS + e / NU] = tab.dCB2[e / NU][e % NU];
        for (int e = threadIdx.x; e < NX * NX; e += C::BLOCK) { pinf_t[(e % NX) * NX + e / NX] = tab.Pinf[e / NX][e % NX]; dpinf_t[(e % NX) * NX + e / NX] = tab.dPinf[e / NX][e % NX]; }   // [c][row]
    }
    __syncthreads();

    // ---- this lane's rows of the matrices
    T cf1[NX], cf2[NU], cb1[NX], cb2[NU];
#pragma unroll
    for (int c = 0; c < NX; ++c) { cf1[c] = tab.CF1[lc][c]; cb1[c] = tab.CB1[lc][c]; }
#pragma unroll
    for (int a = 0; a < NU; ++a) { cf2[a] = tab.CF2[lc][a]; cb2[a] = tab.CB2[lc][a]; }
    T cf0 = tab.cf0[lc], cb0 = tab.cb0[lc], wref = tab.wref[lc];
    const T rho0 = prm.rho, tol_pri = prm.abs_pri_tol, tol_dua = prm.abs_dua_tol;
    const bool adaptive = C::ADAPT && prm.adaptive_rho != 0;
    const int max_iter = prm.max_iter, check_every = prm.check_termination;
    const int n_items = prm.batch_ptr ? min(*prm.batch_ptr, prm.batch) : prm.batch;
    const bool consumer = prm.q_tail != nullptr && prm.q_consume != 0;

    // ---- per-problem state of this lane: slot s = state column s + 1 / input step s; slot N-1 (state lanes) = column 0
    // dual (g / y) and slack (v / z) of the lane's row; cone / half-space duals and (vc - gc) + (vl - gl); reference term before
    // weighting: Xref / Uref of the row (slot N-2 of a state lane is replaced by PT below)
    T* const sst = reinterpret_cast<T*>(gpp_smem) + (size_t)C::GPB * C::GWORDS + 2 * NH * GS + threadIdx.x;   // ROLLED: [array][slot][thread]
    using ArrT = std::conditional_t<C::ROLLED, SmemArr<T, C::BLOCK>, RegArr<T, NH>>;
    using ArrC = std::conditional_t<C::ROLLED, SmemArr<T, C::BLOCK>, RegArr<T, 1>>;
    using ArrF = std::conditional_t<C::ROLLED, SmemArr<T, C::BLOCK>, RegArr<float, NH>>;
    ArrT G, V;
    ArrC GC, GL, EC;
    ArrF RF;
    if constexpr (C::ROLLED) {
        G.p = sst; V.p = sst + NH * C::BLOCK; RF.p = sst + 2 * NH * C::BLOCK;
        GC.p = sst + 3 * NH * C::BLOCK; GL.p = sst + 4 * NH * C::BLOCK; EC.p = sst + 5 * NH * C::BLOCK;     // CONSTR only
    }
    T PT = 0;                // state lanes: -(xref_N' Pinf)'_r
    T PT1 = 0;               // adaptive rho: its derivative, -(xref_N' dPinf)'_r
    // cache->rho and the accumulated rho' - rho0 of this problem; *_lc: the values update_linear_cost saw (it runs BEFORE the
    // adaptation inside an iteration, admm.cpp:326-357)
    T rho = rho0, rho_lc = rho0, dlt = 0, dlt_lc = 0;
    T x0r = 0;               // state lanes: x0_r
#pragma unroll
    for (int s = 0; s < NH; ++s) { G[s] = 0; V[s] = 0; RF[s] = 0.f; }

    int prob = 0, k = 0, next_check = check_every, claim = 0, seen = 0, unpub = -1;
    bool active = false, exhausted = false, pending = false;
    T m0 = 0;                // 0 on a problem's first iteration (q = r = p = 0 on the cold workspace, tiny_api.cpp:68-105), then 1
    T res_px = 0, res_dx = 0, res_pu = 0, res_du = 0;

    T* const tcb0 = gbase + C::oTC;  // [2 buffers][2][GS]: x + gc and x + gl of every lane of the group
    const bool lin_on = C::CONSTR && (is_x ? prm.en_state_linear != 0 : prm.en_input_linear != 0);   // with zero rows the family still adds x to the cost
    const bool soc_on = C::CONSTR && (is_x ? C::SCD > 0 : C::UCD > 0);
    const T arow = !C::CONSTR ? T(0) : (is_x ? (C::NSL > 0 ? tab.ax[row] : T(0)) : (C::NIL > 0 && is_u ? tab.au[row] : T(0)));
    T* wsp = ses.ws;                 // sessions: this problem's workspace
    T* const xb = gbase + C::oXB;    // [2][NXP]
    T* const pb = gbase + C::oPB;    // [2][NXP + NUP]
    T* const dt = gbase + C::oDT;    // [NH-1][NUP]

    for (;;) {
        // ------------------------------------------------------------------ refill idle groups (decisions are group-uniform)
        {
            if (l == 0) publish_done(prm, unpub);
            const bool want = !active && !exhausted && !pending;
            const unsigned mw = __ballot_sync(FULL, want && l == 0);
            if (mw) {
                const int leader = __ffs(mw) - 1;
                int base = 0;
                if (lane == leader) base = atomicAdd(prm.work_counter, __popc(mw));
                base = __shfl_sync(FULL, base, leader);
                if (want) {
                    claim = base + __popc(mw & ((1u << gl0) - 1u));
                    if (consumer) {
                        pending = true;
                    } else if (claim >= n_items) {
                        exhausted = true;
                    } else {
                        if (prm.index_list) claim = __ldg(prm.index_list + claim);
                        pending = true;
                    }
                }
            }
            // group leader resolves the claim (queue ticket / arrival watermark), the group follows
            int ok = 0, qp = claim;
            if (l == 0 && pending) {
                if (consumer) {
                    bool none = false;
                    int e = 0;
                    if (queue_take(prm, claim, e, none)) { ok = 1; qp = e; }
                    else if (none) ok = 2;
                } else {
                    ok = problem_ready(prm, claim, seen) ? 1 : 0;
                }
            }
            ok = __shfl_sync(FULL, ok, gl0);
            qp = __shfl_sync(FULL, qp, gl0);
            if (pending && ok == 2) { pending = false; exhausted = true; }
            const bool mine = pending && ok == 1;
            if (mine) {
                prob = qp;
                pending = false; active = true;
                k = 0; next_check = check_every; m0 = 0;
                res_px = res_dx = res_pu = res_du = 0;
                if constexpr (C::ADAPT) {   // pristine cache for every problem
                    if (dlt != T(0)) {
#pragma unroll
                        for (int c = 0; c < NX; ++c) cf1[c] = tab.CF1[lc][c];
#pragma unroll
                        for (int a = 0; a < NU; ++a) cb2[a] = tab.CB2[lc][a];
                    }
                    rho = rho_lc = rho0; dlt = dlt_lc = 0;
                }
#pragma unroll
                for (int s = 0; s < NH; ++s) { G[s] = 0; V[s] = 0; RF[s] = 0.f; }
                if constexpr (MODE == kGppModels || MODE == kGppModelSession) {
                    // this lane's rows of the problem's own model (column-major: M(i, j) = M[j * rows + i]), formed exactly as fill_gpp_tab
                    // forms them on the host: the same order, every product and sum rounded on its own (no contraction into an fma)
                    const tinympc_cuda_models& M = ses.models;
                    const size_t b = prob;
                    const double* A = M.Adyn + b * NX * NX; const double* B = M.Bdyn + b * NX * NU; const double* K = M.Kinf + b * NU * NX;
                    const double* Qi = M.Quu_inv + b * NU * NU;
                    if (is_u) {   // input lane a = row
#pragma unroll
                        for (int c = 0; c < NX; ++c) {
                            cf1[c] = -K[c * NU + row];
                            T acc = 0.0;
#pragma unroll
                            for (int e = 0; e < NU; ++e) acc = __dadd_rn(acc, __dmul_rn(Qi[e * NU + row], B[e * NX + c]));   // (Quu_inv B')[a][c]
                            cb1[c] = acc;
                        }
                        T acc = 0.0;
#pragma unroll
                        for (int e = 0; e < NU; ++e) {
                            cf2[e] = (e == row) ? -1.0 : 0.0;
                            cb2[e] = Qi[e * NU + row];
                            acc = __dadd_rn(acc, __dmul_rn(Qi[e * NU + row], M.BPf ? M.BPf[b * NU + e] : 0.0));
                        }
                        cf0 = 0.0;
                        cb0 = acc;
                        wref = M.R[b * NU + row];
                    } else {      // state lane r = row (idle lanes compute row 0's values, which nobody reads)
#pragma unroll
                        for (int c = 0; c < NX; ++c) {
                            T acc = A[c * NX + row];
#pragma unroll
                            for (int e = 0; e < NU; ++e) acc = __dsub_rn(acc, __dmul_rn(B[e * NX + row], K[c * NU + e]));   // (A - B Kinf)[r][c]
                            cf1[c] = acc;
                            cb1[c] = M.AmBKt[b * NX * NX + c * NX + row];
                        }
#pragma unroll
                        for (int e = 0; e < NU; ++e) { cf2[e] = -B[e * NX + row]; cb2[e] = -K[row * NU + e]; }
                        cf0 = M.fdyn ? M.fdyn[b * NX + row] : 0.0;
                        cb0 = M.APf ? M.APf[b * NX + row] : 0.0;
                        wref = M.Q[b * NX + row];
                    }
                    rho = rho_lc = M.rho[b];
                }
                if constexpr (C::CONSTR) {
#pragma unroll
                    for (int s = 0; s < NH; ++s) { GC[s] = 0; GL[s] = 0; EC[s] = 0; }
                }
                PT = 0; PT1 = 0;
                if constexpr (SESSION) {
                    wsp = ses.ws + (size_t)prob * ses.W.size;
                    m0 = 1;                                   // the stored q, r, p_N open the first backward pass (zeros on a cold workspace)
                    const int og = is_x ? ses.W.g + NX : ses.W.y, ov = is_x ? ses.W.v + NX : ses.W.z, st_ = is_x ? NX : NU;
                    if (is_x || is_u) {
#pragma unroll
                        for (int s = 0; s < NH - 1; ++s) { G[s] = wsp[og + s * st_ + row]; V[s] = wsp[ov + s * st_ + row]; }
                    }
                    if (is_x) { x0r = wsp[ses.W.x + row]; G[NH - 1] = wsp[ses.W.g + row]; V[NH - 1] = wsp[ses.W.v + row]; }
                } else
                if (is_x) {
                    x0r = static_cast<T>(__ldg(prm.x0 + (size_t)prob * NX + row));
                    if (prm.Xref) {
                        if (prm.xref_const) {   // compact reference input: one state per problem for every column of the horizon
                            const float v = __ldg(prm.Xref + (size_t)prob * NX + row);
#pragma unroll
                            for (int s = 0; s < NH - 1; ++s) RF[s] = v;
                        } else {
                            const float* src = prm.Xref + (size_t)prob * SXL + row;
#pragma unroll
                            for (int s = 0; s < NH - 1; ++s) RF[s] = __ldg(src + (s + 1) * NX);
                        }
                    }
                } else if (is_u) {
                    if (prm.Uref) {
                        const float* src = prm.Uref + (size_t)prob * SUL + row;
#pragma unroll
                        for (int s = 0; s < NH - 1; ++s) RF[s] = __ldg(src + s * NU);
                    }
                }
            }
            if (__any_sync(FULL, mine)) {
                // terminal term: PT_r = -(xref_N' Pinf)_r = -sum_c xref_N[c] Pinf[c][r]   (admm.cpp:238-240)
                if (mine && is_x) xb[row] = SESSION ? wsp[ses.W.Xref + (NH - 1) * NX + row] : static_cast<T>(RF[NH - 2]);
                __syncwarp();
                if (mine && is_x) {
                    T acc = 0, acc1 = 0;
#pragma unroll
                    for (int c = 0; c < NX; ++c) {
                        if constexpr (MODE == kGppModels || MODE == kGppModelSession) acc = fma(xb[c], ses.models.Pinf[(size_t)prob * NX * NX + row * NX + c], acc);   // Pinf(c, row)
                        else acc = fma(xb[c], tab.Pinf[c][row], acc);
                        if constexpr (C::ADAPT) acc1 = fma(xb[c], tab.dPinf[c][row], acc1);
                    }
                    PT = -acc; PT1 = -acc1;
                }
                __syncwarp();
            }
            if (!__any_sync(FULL, active)) {
                if (l == 0) publish_done(prm, unpub);
                if (!__any_sync(FULL, pending)) break;
                __nanosleep(256);
                continue;
            }
        }

        // weighted reference term of slot s: -(Xref .* Q) / -(Uref .* R); the terminal slot of a state lane holds PT instead
        auto refterm = [&](int s) -> T {
            if (s == NH - 2 && is_x) return C::ADAPT ? fma(dlt_lc, PT1, PT) : PT;
            if constexpr (SESSION) return -(wsp[(is_x ? ses.W.Xref + (s + 1) * NX : ses.W.Uref + s * NU) + row] * wref);
            else return -(static_cast<T>(RF[s]) * wref);
        };
        // w_s = q / r of slot s as update_linear_cost left it (admm.cpp:218-246): ref - rho (v - g); 0 on the cold workspace.
        // Sessions: the first backward pass of a solve reads what the PREVIOUS solve stored (its references may have changed since).
        auto lincost_now = [&](int s) -> T {
            if constexpr (C::CONSTR) return m0 * fma(-rho_lc, (V[s] - G[s]) + EC[s], refterm(s));   // + (vc - gc) + (vl - gl), admm.cpp:219-246
            else return m0 * fma(-rho_lc, V[s] - G[s], refterm(s));
        };
        auto lincost = [&](int s) -> T {
            if constexpr (SESSION) {
                if (s == NH - 1) return k == 0 ? wsp[ses.W.q + row] : fma(-rho_lc, V[NH - 1] - G[NH - 1], -(wsp[ses.W.Xref + row] * wref));   // q_0, full mode only
                if (k == 0) return wsp[(is_x ? (s == NH - 2 ? ses.W.p + (NH - 1) * NX : ses.W.q + (s + 1) * NX) : ses.W.r + s * NU) + row];
            }
            return lincost_now(s);
        };

        // ------------------------------------------------------------------ backward_pass_grad (admm.cpp:13-20)
        {
            // p_{N-1} (state lanes) and r_{N-2} (input lanes) open the sweep
            const T w = lincost(NH - 2);
            T* buf = pb + ((NH - 1) & 1) * (NXP + NUP);
            if (is_x) buf[row] = w; else if (is_u) buf[NXP + row] = w;
            __syncwarp();
#pragma unroll C::TUNROLL
            for (int i = NH - 2; i >= 0; --i) {
                const T* src = pb + ((i + 1) & 1) * (NXP + NUP);
                T pv[NXP], rv[NUP];
#pragma unroll
                for (int c = 0; c < NXP / 2; ++c) { const double2 t2 = *reinterpret_cast<const double2*>(src + 2 * c); pv[2 * c] = t2.x; pv[2 * c + 1] = t2.y; }
#pragma unroll
                for (int a = 0; a < NUP / 2; ++a) { const double2 t2 = *reinterpret_cast<const double2*>(src + NXP + 2 * a); rv[2 * a] = t2.x; rv[2 * a + 1] = t2.y; }
                // four chains: three over p, one over r
                T a0 = cb0, a1 = 0, a2 = 0, a3 = 0;
                constexpr int T3 = (NX + 2) / 3;
#pragma unroll
                for (int c = 0; c < NX; ++c) {
                    if (c < T3) a0 = fma(cb1[c], pv[c], a0);
                    else if (c < 2 * T3) a1 = fma(cb1[c], pv[c], a1);
                    else a2 = fma(cb1[c], pv[c], a2);
                }
#pragma unroll
                for (int a = 0; a < NU; ++a) a3 = fma(cb2[a], rv[a], a3);
                T acc = (a0 + a1) + (a2 + a3);
                if (i > 0) {
                    const T w1 = lincost(i - 1);          // state lane: q_i (column i = slot i-1); input lane: r_{i-1}
                    T* dst = pb + (i & 1) * (NXP + NUP);
                    if (is_x) dst[row] = acc + w1; else if (is_u) dst[NXP + row] = w1;
                    if constexpr (FULLWS) { if (is_x) wsp[ses.W.p + i * NX + row] = acc + w1; }
                } else {
                    if constexpr (FULLWS) { if (is_x) wsp[ses.W.p + row] = acc + lincost(NH - 1); }   // p_0 = q_0 + ... (never read)
                }
                if (is_u) dt[i * NUP + row] = acc;         // d_i
                __syncwarp();
            }
        }

        // ------------------------------------------------------------------ forward_pass + update_slack + update_dual + residuals
        T rp = 0, rd = 0;
        // adaptive rho: is the adaptation due at the end of this iteration (loop index i = k > 0, i % 5 == 0, admm.cpp:339)?  The
        // groups of a warp may be at different phases; the extra hand-offs are executed by the whole warp when any group is due.
        const bool due = adaptive && k > 0 && k % 5 == 0;
        const bool anydue = C::ADAPT && __any_sync(FULL, due);
        T a_pri = 0, a_prin = 0, a_dua = 0, a_duan = 0;
        auto element = [&](int s, T val) {   // the lane's element of slot s: vnew = clamp(x + g), g += x - vnew (admm.cpp:85-98, 184-187)
            const T lo = lo_t[s * GS + lc], hi = hi_t[s * GS + lc];
            const T t = val + G[s];
            const T vn = gclamp(t, lo, hi);
            if constexpr (SESSION) { sold[s * GS] = V[s]; sval[s * GS] = val; }
            G[s] = t - vn;
            rp = gabsmax(rp, val - vn);
            rd = gabsmax(rd, V[s] - vn);
            V[s] = vn;
        };
        {
            if (is_x) { xb[row] = x0r; element(NH - 1, x0r); }   // column 0: x_0 = x0 (never rewritten, admm.cpp:25-32)
            __syncwarp();
#pragma unroll C::TUNROLL
            for (int s = 0; s < NH - 1; ++s) {
                const T* src = xb + (s & 1) * NXP;
                T xv[NXP], dv[NUP];
#pragma unroll
                for (int c = 0; c < NXP / 2; ++c) { const double2 t2 = *reinterpret_cast<const double2*>(src + 2 * c); xv[2 * c] = t2.x; xv[2 * c + 1] = t2.y; }
#pragma unroll
                for (int a = 0; a < NUP / 2; ++a) { const double2 t2 = *reinterpret_cast<const double2*>(dt + s * NUP + 2 * a); dv[2 * a] = t2.x; dv[2 * a + 1] = t2.y; }
                T a0 = cf0, a1 = 0, a2 = 0, a3 = 0;
                constexpr int T3 = (NX + 2) / 3;
#pragma unroll
                for (int c = 0; c < NX; ++c) {
                    if (c < T3) a0 = fma(cf1[c], xv[c], a0);
                    else if (c < 2 * T3) a1 = fma(cf1[c], xv[c], a1);
                    else a2 = fma(cf1[c], xv[c], a2);
                }
#pragma unroll
                for (int a = 0; a < NU; ++a) a3 = fma(cf2[a], dv[a], a3);
                const T val = (a0 + a1) + (a2 + a3);      // x_{s+1,r} or u_{s,a}
                if (is_x && s < NH - 2) xb[((s + 1) & 1) * NXP + row] = val;
                if constexpr (!C::CONSTR) element(s, val);
                if constexpr (C::CONSTR) {
                    // cone and half-space families of the column (admm.cpp:100-175, 189-207): the pre-projection slacks x + gc, x + gl of
                    // the whole group go round together with x_{s+1} -- ONE hand-off per step -- and the projections (recomputed by every
                    // lane that owns a component) and the box work sit BEHIND the barrier, in one basic block with the loads and the
                    // product of the next step, which do not depend on them
                    const T tc = val + GC[s], tl = val + GL[s];
                    T* const tcb = tcb0 + (s & 1) * 2 * GS;
                    tcb[l] = tc;
                    tcb[GS + l] = tl;
                    __syncwarp();
                    element(s, val);
                    T vc = tc, vl = tl;
                    auto cone = [&](int base, auto dim, float mu, int me) {   // admm.cpp:39-60 with its float norm and float a / mu
                        constexpr int D = decltype(dim)::value;
                        if constexpr (D > 0) {
                            T w[D], ss = 0;
#pragma unroll
                            for (int e = 0; e < D; ++e) w[e] = tcb[base + e];
#pragma unroll
                            for (int e = 0; e < D - 1; ++e) ss = fma(w[e], w[e], ss);
                            const T u0 = w[D - 1] * static_cast<T>(mu);
                            // float(sqrt(ss)) and 1 / a without the library's fp64 sqrt / division (~70 instructions each, on every lane and
                            // step): float estimates + one Newton step in double, 1e-14 relative (the form tmpc_tpp4.cuh uses)
                            float y0f, r0f;
                            asm("sqrt.approx.f32 %0, %1;" : "=f"(y0f) : "f"(static_cast<float>(ss)));
                            asm("rcp.approx.f32 %0, %1;" : "=f"(r0f) : "f"(y0f));
                            const T y0 = static_cast<T>(y0f);
                            const T y1 = ss > 1e-30 ? fma(fma(-y0, y0, ss), static_cast<T>(0.5f * r0f), y0) : T(0);
                            const float a = static_cast<float>(y1);
                            const T ad = static_cast<T>(a), r0 = static_cast<T>(r0f);
                            const T ra = r0 * fma(-ad, r0, T(2));
                            const T fct = T(0.5) * fma(u0, ra, T(1));
                            const bool zero = ad <= -u0, inside = ad <= u0, mine = me >= 0 && me < D;
                            const T outv = me == D - 1 ? fct * static_cast<T>(a / mu) : fct * tc;   // the lane's own component is tc itself
                            vc = !mine ? tc : (zero ? T(0) : (inside ? tc : outv));
                        }
                    };
                    if (is_x) cone(C::SCS, std::integral_constant<int, C::SCD>{}, prm.cx[0], row - C::SCS);
                    else if (is_u) cone(NX + C::UCS, std::integral_constant<int, C::UCD>{}, prm.cu[0], row - C::UCS);
                    if constexpr (C::NSL > 0) {
                        if (is_x) {   // admm.cpp:70-73, 148-159: v <- v - (a.v - b) / ||a||^2 a  where a.v > b
                            T dv2 = 0;
#pragma unroll
                            for (int e = 0; e < NX; ++e) dv2 = fma(tab.ax[e], tcb[GS + e], dv2);
                            vl = dv2 > tab.bx ? tl - ((dv2 - tab.bx) * tab.nrx) * arow : tl;
                        }
                    }
                    if constexpr (C::NIL > 0) {
                        if (is_u) {
                            T dv2 = 0;
#pragma unroll
                            for (int e = 0; e < NU; ++e) dv2 = fma(tab.au[e], tcb[GS + NX + e], dv2);
                            vl = dv2 > tab.bu ? tl - ((dv2 - tab.bu) * tab.nru) * arow : tl;
                        }
                    }
                    GC[s] = tc - vc;
                    GL[s] = tl - vl;
                    EC[s] = (soc_on ? vc - GC[s] : T(0)) + (lin_on ? vl - GL[s] : T(0));
                }
                if constexpr (C::ADAPT) {
                    // Park this step's iterate and updated dual for the block pass of an adaptation, and take the primal rows -- inputs:
                    // u - znew (= rp); states: (A x + B u - x_next) - vnew_next = -f - vnew_next.  Unconditional: a branch on "due" here
                    // makes the compiler keep two copies of the unrolled sweep, which no longer fit the instruction cache.
                    sval[s * GS] = val;
                    sdual[s * GS] = G[s];
                    const T pa = is_x ? cf0 + V[s] : T(0), pb2 = is_x ? cf0 : val;
                    a_pri = gabsmax(a_pri, pa);
                    a_prin = gabsmax(gabsmax(a_prin, V[s]), pb2);
                }
                if constexpr (!C::CONSTR) { if (s < NH - 2) __syncwarp(); }
            }
            if constexpr (C::ADAPT) {
                if (anydue) {
                    // Closed block form of the dual residual of rho_benchmark.cpp:146-173 (SURVEY.md 8 a-8), one ROLLED pass over the parked
                    // columns (the unrolled sweeps above already fill most of the 32 KB instruction cache).  Column s: x-block
                    // A' g_{s+1} - g_s [s >= 1], u-block y_s + B' g_{s+1}, with Px = qv = Q .* x_s (R .* u_s).
                    __syncwarp();
                    const T* gsv = sdual - l;          // the group's row of slot s starts at gsv + s * GS (state lanes 0 .. NX-1)
                    const T* xsv = sval - l;
#pragma unroll 1
                    for (int s = 0; s < NH - 1; ++s) {
                        T at0 = 0, at1 = 0;
#pragma unroll
                        for (int c = 0; c < NX; ++c) { if (c & 1) at1 = fma(at_t[c * GS + lc], gsv[s * GS + c], at1); else at0 = fma(at_t[c * GS + lc], gsv[s * GS + c], at0); }
                        const T at = at0 + at1;
                        const T own = is_x ? (s >= 1 ? sval[(s - 1) * GS] : x0r) : sval[s * GS];           // x_s / u_s
                        const T aty = is_x ? (s >= 1 ? at - sdual[(s - 1) * GS] : at) : at + sdual[s * GS];   // - g_s / + y_s
                        const T qx = wref * own;
                        a_dua = gabsmax(a_dua, qx + qx + aty);
                        a_duan = gabsmax(gabsmax(a_duan, qx), aty);
                    }
                    {   // last state block: Px = Pinf x_N (the cache's current Pinf), qv = Q .* x_N, A'y = -g_N
                        T px0 = 0, px1 = 0;
#pragma unroll
                        for (int c = 0; c < NX; ++c) {
                            const T pc = fma(dlt, dpinf_t[c * NX + row], pinf_t[c * NX + row]);
                            if (c & 1) px1 = fma(pc, xsv[(NH - 2) * GS + c], px1); else px0 = fma(pc, xsv[(NH - 2) * GS + c], px0);
                        }
                        if (is_x) {
                            const T px = px0 + px1, qx = wref * sval[(NH - 2) * GS], aty = -G[NH - 2];
                            a_dua = gabsmax(a_dua, px + qx + aty);
                            a_duan = gabsmax(gabsmax(gabsmax(a_duan, px), qx), aty);
                        }
                    }
                    if (is_u) a_pri = gmax(a_pri, rp);      // input rows: u - znew
                    if (!(is_x || is_u)) { a_pri = a_prin = a_dua = a_duan = 0; }
#pragma unroll
                    for (int o = GS / 2; o > 0; o >>= 1) {
                        a_pri = gmax(a_pri, __shfl_xor_sync(FULL, a_pri, o));
                        a_prin = gmax(a_prin, __shfl_xor_sync(FULL, a_prin, o));
                        a_dua = gmax(a_dua, __shfl_xor_sync(FULL, a_dua, o));
                        a_duan = gmax(a_duan, __shfl_xor_sync(FULL, a_duan, o));
                    }
                    __syncwarp();
                }
            }
        }
        rho_lc = rho; dlt_lc = dlt;   // update_linear_cost of this iteration ran with the pre-adaptation cache
        if constexpr (C::ADAPT) {
            if (due) {   // predict_rho + update_matrices_with_derivatives (rho_benchmark.cpp:175-212)
                const T eps = 1e-10;
                const T npri = a_pri / (a_prin + eps), ndua = a_dua / (a_duan + eps);
                T nr = rho * sqrt(npri / (ndua + eps));
                if (prm.rho_clip) nr = gmin(gmax(nr, prm.rho_min), prm.rho_max);
                const T step = nr - rho;
#pragma unroll
                for (int c = 0; c < NX; ++c) cf1[c] = fma(step, dcf1_t[c * GS + lc], cf1[c]);
#pragma unroll
                for (int a = 0; a < NU; ++a) cb2[a] = fma(step, dcb2_t[a * GS + lc], cb2[a]);
                dlt += step;
                rho = nr;
            }
        }
        m0 = 1;
        k += 1;   // work->iter += 1 (admm.cpp:328)

        // ------------------------------------------------------------------ termination_condition (admm.cpp:253-271)
        bool finish = false;
        int st = 11;
        const bool chk = (k == next_check);              // group-uniform; the groups of a warp may differ
        if (__any_sync(FULL, chk)) {                     // the shuffles are executed by the whole warp
            T px = is_x ? rp : T(0), dx = is_x ? rd : T(0), pu = is_u ? rp : T(0), du = is_u ? rd : T(0);
#pragma unroll
            for (int o = GS / 2; o > 0; o >>= 1) {
                px = gmax(px, __shfl_xor_sync(FULL, px, o));
                dx = gmax(dx, __shfl_xor_sync(FULL, dx, o));
                pu = gmax(pu, __shfl_xor_sync(FULL, pu, o));
                du = gmax(du, __shfl_xor_sync(FULL, du, o));
            }
            if (chk) {
                next_check += check_every;
                res_px = px; res_dx = dx * rho; res_pu = pu; res_du = du * rho;
                if (res_px < tol_pri && res_pu < tol_pri && res_dx < tol_dua && res_du < tol_dua) { finish = true; st = 1; }
            }
        }
        if (k >= max_iter) finish = true;
        if (active && finish) {
            // solution = (vnew, znew) (admm.cpp:364-376, 384-388)
            if (!SESSION && prm.u0 != nullptr) {   // compact output: the first control is all the caller reads
                if (is_u) prm.u0[(size_t)prob * NU + row] = static_cast<float>(V[0]);
            } else if (!SESSION || prm.x != nullptr) {
            if (is_x) {
                float* dst = prm.x + (size_t)prob * SXL + row;
                dst[0] = static_cast<float>(V[NH - 1]);
#pragma unroll
                for (int s = 0; s < NH - 1; ++s) dst[(s + 1) * NX] = static_cast<float>(V[s]);
            } else if (is_u) {
                float* dst = prm.u + (size_t)prob * SUL + row;
#pragma unroll
                for (int s = 0; s < NH - 1; ++s) dst[s * NU] = static_cast<float>(V[s]);
            }
            }
            if constexpr (SESSION) {
                const bool conv = st == 1;     // converged: the reference returns BEFORE v <- vnew (admm.cpp:364-380)
                if (is_x || is_u) {
                    const int st_ = is_x ? NX : NU;
                    T* wx = wsp + (is_x ? ses.W.x + NX : ses.W.u) + row;
                    T* wvn = wsp + (is_x ? ses.W.vnew + NX : ses.W.znew) + row;
                    T* wv = wsp + (is_x ? ses.W.v + NX : ses.W.z) + row;
                    T* wg = wsp + (is_x ? ses.W.g + NX : ses.W.y) + row;
                    T* wq = wsp + (is_x ? ses.W.q + NX : ses.W.r) + row;
#pragma unroll
                    for (int s = 0; s < NH - 1; ++s) {
                        wx[s * st_] = sval[s * GS];
                        wvn[s * st_] = V[s];
                        wv[s * st_] = conv ? sold[s * GS] : V[s];
                        wg[s * st_] = G[s];
                        if (is_x && s == NH - 2) wsp[ses.W.p + (NH - 1) * NX + row] = lincost_now(s);
                        else wq[s * st_] = lincost_now(s);
                    }
                    if constexpr (FULLWS) {
                        if (is_u) {
#pragma unroll
                            for (int s = 0; s < NH - 1; ++s) wsp[ses.W.d + s * NU + row] = dt[s * NUP + row];
                        } else {   // q of the columns the backward pass never reads (admm.cpp:218-225 computes them all the same)
                            wsp[ses.W.q + row] = fma(-rho_lc, V[NH - 1] - G[NH - 1], -(wsp[ses.W.Xref + row] * wref));
                            wsp[ses.W.q + (NH - 1) * NX + row] = fma(-rho_lc, V[NH - 2] - G[NH - 2], -(wsp[ses.W.Xref + (NH - 1) * NX + row] * wref));
                        }
                    }
                    if (is_x) {
                        wsp[ses.W.vnew + row] = V[NH - 1];
                        wsp[ses.W.v + row] = conv ? sold[(NH - 1) * GS] : V[NH - 1];
                        wsp[ses.W.g + row] = G[NH - 1];
                    }
                }
                if (l == 0) {
                    T* sc = wsp + ses.W.scalars;
                    sc[0] = rho; sc[1] = static_cast<T>(k); sc[2] = static_cast<T>(st); sc[3] = res_px; sc[4] = res_dx; sc[5] = res_pu; sc[6] = res_du;
                    sc[7] = conv ? T(1) : T(0);
                }
            }
            if (l == 0) {
                prm.iter[prob] = k;
                prm.status[prob] = st;
                if (prm.residuals) *reinterpret_cast<float4*>(prm.residuals + 4 * (size_t)prob) =
                    make_float4(static_cast<float>(res_px), static_cast<float>(res_dx), static_cast<float>(res_pu), static_cast<float>(res_du));
                if (prm.rho_out) prm.rho_out[prob] = static_cast<float>(rho);
                if (prm.done_counters) unpub = prob;
            }
            active = false;
        }
    }
}

template <class C>
inline size_t gpp_smem_bytes(int) {
    return ((size_t)C::GPB * C::GWORDS + 2 * (size_t)C::NH * C::GS +
            (C::ADAPT ? 2 * (size_t)C::GS * C::NX + (size_t)C::GS * C::NU + 2 * (size_t)C::NX * C::NX : 0) +
            (size_t)C::NSTATE * C::NH * C::BLOCK + (C::CONSTR ? 0 : 2 * (size_t)C::NH * C::BLOCK)) * sizeof(double);
}

}  // namespace tmpc
