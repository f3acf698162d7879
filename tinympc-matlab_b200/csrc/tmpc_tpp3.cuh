// tmpc_tpp3.cuh -- batched ADMM throughput kernel for sm_100a, INCREMENTAL ("delta") form, fp32: box constraints, and box +
// one second-order cone per side + linear inequalities (the rocket family).
//
// Same path and mapping as tmpc_tpp2.cuh (one thread = one problem, packed f32x2 arithmetic, family matrices in the
// kernel-parameter constant bank, state in tensor memory + shared memory, lane refill); reference: admm.cpp:274-389.
// What changes is the ALGEBRA of the Riccati sweeps, to take the fp32 rounding noise out of the termination test.
//
// Why.  backward_pass_grad / forward_pass (admm.cpp:13-32) are one fixed affine map  x = L(q, r, p_N) + x_free.
// Evaluated from scratch every iteration (what the reference does, in double), the costates p ~ Pinf x reach 1e3..1e4
// for the quadrotor; in fp32 their rounding (~5e-4) lands in u and x as FRESH noise of 1e-5..1e-4 at every iteration,
// i.e. 1..10 % of a 1e-3 tolerance, and flips the threshold test of 1-2 % of the problems by one check interval
// (profiles/tools/noise_model.py reproduces that on the CPU).  L is linear, so
//     x(k+1) = x(k) + L_h( q(k) - q(k-1), r(k) - r(k-1), p_N(k) - p_N(k-1) ),      q(k) - q(k-1) = -rho (w(k) - w(k-1)),
// with L_h the homogeneous part (no f, APf, BPf, no reference terms).  The sweeps then run on increments whose size shrinks
// with the residuals, the fresh noise becomes proportional to the residual itself, and what was rounded earlier is a
// constant offset of ~1e-5 in x -- a slightly perturbed problem, not noise on the test.  Same flop count.
//
// One iteration here (reference order: backward, forward, slack, dual, linear cost, check):
//   forward : dx_0 = 0, du_i = -Kinf dx_i - dd_i, dx_{i+1} = A dx_i + B du_i;  X += dx, U += du          (admm.cpp:25-32)
//             (sparse-A instances, Tpp3Cfg::SA: A dx over the compiled nonzero pairs of A only)
//   sweep   : columns N-1 .. 0, fused: slack + dual + residuals of the column (admm.cpp:81-208, 253-260), the increment
//             dw of (slack - dual), then the Riccati step on (-rho dw) giving dd for the next forward    (admm.cpp:13-20, 214-247)
//   check   : admm.cpp:262-265, solution = (vnew, znew)
// The first iteration of a problem is the full affine map: forward with d0 (first backward pass on the zero workspace,
// host-precomputed), x0, f; its sweep adds the reference terms -(Xref .* Q), -(Uref .* R), -(xref_N' Pinf)' ONCE (q(0) = 0).
// Those terms are parked in the T / TZ state columns at refill time (the cold slack t(0) is 0 by definition, so the
// columns are free until the first sweep overwrites them): no scratch buffer, no reference traffic per iteration.
//
// State per problem: X (x), T (t = x + g_prev, pre-clamp slack: v = clamp(t), g = t - v) in tensor memory (2 nx N columns
// per thread), U, TZ, DD (u, u + y_prev, -dd) in shared memory; cone / half-space families add their pre-projection slacks
// (TC, TL in tensor memory, TZC, TZL in shared memory).  The HYBRID layout (Tpp3Cfg::HYB) spreads X and T over registers,
// tensor memory and shared memory to fit a third warp per scheduler on the quadrotor shape; see the comment there.
// Throughput devices shared with tmpc_tpp2.cuh: persistent grid, batched lane refill (adaptive threshold), streamed host
// pipeline hooks (arrival watermark, per-chunk completion counters).
#pragma once
#include <type_traits>

#include "tmpc_tpp2.cuh"

#ifndef TMPC_TUNROLL_SMALL
#define TMPC_TUNROLL_SMALL 10
#endif

namespace tmpc {

enum : int { REFS_STATE = 3 };   // registry "refs" code: reference terms parked in the state columns

// constant-bank pack of the incremental-form instances: the matrices of ConstPack2 + the linear-inequality rows
// (coefficients row-major, offsets b, 1 / ||a||^2 for project_hyperplane, admm.cpp:70-73)
// CONV: + the impulse-response tables of the backward pass (Tpp3Cfg::CONV): NG[k] = -Quu_inv B' AmBKt^k (k = 0 .. N-2, each NU x NX,
// column-major like every other table) and NQ = -Quu_inv.
// SA (sparse-A instances, Tpp3Cfg::SA): AS = the coefficients of A on SA's nonzero pairs, packed (SparsePairs::pack) for the
// forward rollout's masked product.
template <int NX, int NU, int NH, int NSL, int NIL, bool CONV = false, class SA = SparsePairs<>>
struct alignas(16) ConstPack3 : ConstPack2<float, NX, NU, NH, false> {
    float Alx[NSL > 0 ? NSL * NX : 1], blx[NSL > 0 ? NSL : 1], inx[NSL > 0 ? NSL : 1];
    float Alu[NIL > 0 ? NIL * NU : 1], blu[NIL > 0 ? NIL : 1], inu[NIL > 0 ? NIL : 1];
    float NG[CONV ? (NH - 1) * NX * pad2(NU) : 2], NQ[CONV ? NU * pad2(NU) : 2];
    float AS[SA::packed(NX) > 2 ? SA::packed(NX) : 2];
};
template <int NX, int NU, int NH, int NSL, int NIL, bool CONV, class SA>
inline void fill_const_pack3(ConstPack3<NX, NU, NH, NSL, NIL, CONV, SA>& c, const double* pk, const PackLayout& L) {
    fill_const_pack2(static_cast<ConstPack2<float, NX, NU, NH, false>&>(c), pk, L);
    c.Alx[0] = c.blx[0] = c.inx[0] = c.Alu[0] = c.blu[0] = c.inu[0] = 0.f;
    c.NG[0] = c.NG[1] = c.NQ[0] = c.NQ[1] = 0.f;
    c.AS[0] = c.AS[1] = 0.f;
    if constexpr (!SA::DENSE) SA::pack(c.AS, c.A, NX);
    if constexpr (CONV) {
        constexpr int NUP = pad2(NU);
        double G[NU * NX], Gn[NU * NX];                 // row-major NU x NX, double
        for (int a = 0; a < NU; ++a)
            for (int cc = 0; cc < NX; ++cc) {           // G_0 = Quu_inv B'
                double acc = 0.0;
                for (int b = 0; b < NU; ++b) acc += pk[L.Quu_inv + a * NU + b] * pk[L.B + cc * NU + b];
                G[a * NX + cc] = acc;
            }
        for (int k = 0; k < NH - 1; ++k) {
            for (int a = 0; a < NU; ++a) for (int cc = 0; cc < NX; ++cc) c.NG[k * NX * NUP + cc * NUP + a] = static_cast<float>(-G[a * NX + cc]);
            for (int a = 0; a < NU; ++a)                // G_{k+1} = G_k AmBKt
                for (int cc = 0; cc < NX; ++cc) {
                    double acc = 0.0;
                    for (int r = 0; r < NX; ++r) acc += G[a * NX + r] * pk[L.AmBKt + r * NX + cc];
                    Gn[a * NX + cc] = acc;
                }
            for (int e = 0; e < NU * NX; ++e) G[e] = Gn[e];
        }
        for (int a = 0; a < NU; ++a) for (int b = 0; b < NU; ++b) c.NQ[b * NUP + a] = static_cast<float>(-pk[L.Quu_inv + a * NU + b]);
    }
    for (int k = 0; k < NSL; ++k) {
        for (int j = 0; j < NX; ++j) c.Alx[k * NX + j] = static_cast<float>(pk[L.Alin_x + k * NX + j]);
        c.blx[k] = static_cast<float>(pk[L.blin_x + k]);
        c.inx[k] = static_cast<float>(1.0 / pk[L.nrm_x + k]);
    }
    for (int k = 0; k < NIL; ++k) {
        for (int j = 0; j < NU; ++j) c.Alu[k * NU + j] = static_cast<float>(pk[L.Alin_u + k * NU + j]);
        c.blu[k] = static_cast<float>(pk[L.blin_u + k]);
        c.inu[k] = static_cast<float>(1.0 / pk[L.nrm_u + k]);
    }
}

template <int NX_, int NU_, int NH_, int BLOCK_, bool REFS_, bool PPB_, bool FB_, bool AFF_, bool OPQ_, bool TIB_, int FEAT_ = FEAT_BOX,
          int SCS_ = 0, int SCD_ = 0, int UCS_ = 0, int UCD_ = 0, int NSL_ = 0, int NIL_ = 0, int TTM_ = -1, int CONV_ = -1,
          class SA_ = SparsePairs<>>
struct Tpp3Cfg {
    using T = float;
    static_assert(FEAT_ == FEAT_BOX || FEAT_ == FEAT_CONSTR, "the incremental form covers box and box + cone + half-space families");
    static constexpr int NX = NX_, NU = NU_, NH = NH_, FEAT = FEAT_, BLOCK = BLOCK_, MINB = 1;
    static constexpr bool CONSTR = FEAT_ == FEAT_CONSTR;   // + second-order cones and linear inequalities (admm.cpp:102-173)
    // The cone blocks are part of the instance: at most one state cone on elements [SCS, SCS + SCD) and one input cone on
    // [UCS, UCS + UCD) (dim 0 = none), so that the projection is straight-line register code.  Families with any other cone
    // list run the direct-form kernel (tmpc_tpp2.cuh), whose cones are run-time tables.  So are the numbers of linear rows
    // (NSL state rows, NIL input rows); their coefficients ride in the constant bank next to the matrices.
    static constexpr int SCS = SCS_, SCD = SCD_, UCS = UCS_, UCD = UCD_, NSL = NSL_, NIL = NIL_;
    static_assert(SCS_ >= 0 && SCS_ + SCD_ <= NX_ && UCS_ >= 0 && UCS_ + UCD_ <= NU_, "cone block outside the vector");
    static constexpr int REFMODE = REFS_ ? REFS_STATE : REFS_NONE;
    static constexpr bool REFS = REFS_;
    static constexpr bool PPB = PPB_;
    static constexpr bool FB = FB_ && !PPB_;
    static constexpr bool AFF = AFF_;
    static constexpr bool OPQ = OPQ_;
    static constexpr bool TIB = TIB_ && FB_ && !PPB_ && !OPQ_;
    static constexpr int SX = NX * NH, SU = NU * (NH - 1);
    // IMPULSE-RESPONSE form of the backward pass (CONV).  The costate recursion p_i = q_i + AmBKt p_{i+1} - Kinf' r_i followed by
    // d_i = Quu_inv (B' p_{i+1} + r_i) (admm.cpp:13-20) is the ill-conditioned step of the iteration in float32: on the quadrotor
    // the costates are ~13x their right-hand sides and B' p cancels to ~1 % of its terms, so d carries 2.6e-6 of relative rounding
    // error per sweep -- the drift of ~6e-5 the fp32 iterates pick up over a solve.  Unrolling the recursion,
    //     d_i = Quu_inv r_i + sum_{j > i} G_{j-i-1} s_j,    s_j = q_j - Kinf' r_j (j <= N-2),  s_{N-1} = p_N,    G_k = Quu_inv B' AmBKt^k,
    // with the small matrices G_k (|G_k| <= 9e-3 on the quadrotor) formed once on the host in double: no large intermediate, no
    // cancellation -- 1.6e-7 relative error in d, 16x better, for N (N-1) / 2 products of nu x nx instead of N-1 steps of
    // (nx x nx + 2 nu x nx + nu x nu), i.e. 2 160 against 2 304 multiply-adds on the quadrotor shape.  Column j of the sweep
    // scatters -G_k s_j into the -dd slots of the steps before it.  The cost grows with N^2 nu nx against N nx^2, so the form is
    // the default where it matters and is cheap (nx >= 6); the nx = 4 shapes keep the recursion, which is well conditioned there.
    static constexpr bool CONV = CONV_ < 0 ? (NX_ >= 12 && FEAT_ == FEAT_BOX) : (CONV_ != 0);
    // SPARSE-A instances (SA_ non-empty): the nonzero pattern of A, at row-pair granularity, compiled in.  The forward rollout's
    // product A dx then issues an FFMA2 only for the pairs of the pattern (26 of 72 on the quadrotor shape), fed from a packed table;
    // the dispatcher (tmpc_capi.cu find_kernel) runs such an instance only for a family whose float32 A has no nonzero outside it.
    using SA = SA_;
    static_assert(SA_::DENSE || SA_::NCOL == NX_, "A pattern of another shape");
    using CPack = ConstPack3<NX_, NU_, NH_, NSL_, NIL_, CONV, SA_>;
    // HYBRID state layout (TTM_ >= 0, box instances): the 2 nx N columns of x and t per thread cap the quadrotor shape at 8 warps
    // per SM (2 per scheduler, 61 % issue utilisation).  Three observations buy a third warp per scheduler:
    //   * x_0 is the problem's x0, which the lane holds in registers anyway -- column 0 of X is never stored;
    //   * column N-1 of X and T is produced last by the forward pass / first sweep column and consumed first by the sweep:
    //     it lives in registers across the iteration (2 nx of the ~40 registers the 12-warp budget leaves free);
    //   * the columns of T that no longer fit the tensor-memory share of the warp (TTM_ of them do) go to shared memory.
    static constexpr bool HYB = TTM_ >= 0;
    // The time loops stay rolled where a step is hundreds of instructions (the body must fit the instruction cache); the small
    // shapes unroll them partially -- with nx = 4 a step is ~85 instructions and loop control was 28 % of the cartpole kernel
    // (measured on the N = 20 cartpole batch: rolled 119.9, x4 137.6, x10 148.5, fully unrolled 145.0 M solves/s; the rocket
    // instance with its ~600-instruction column loses 4 % when unrolled x3 and stays rolled).
    static constexpr int TUNROLL = (NX_ <= 4 && FEAT_ == FEAT_BOX) ? TMPC_TUNROLL_SMALL : 1;
    static constexpr int TTM = HYB ? TTM_ : NH_;
    static_assert(!HYB || (FEAT_ == FEAT_BOX && NH_ >= 3 && TTM_ <= NH_ - 1), "hybrid layout: box instances only");
    // shared memory: u, u + y_prev, -dd (+ the pre-projection input slacks of the cone and half-space families; + the T columns
    // TTM .. N-2 of the hybrid layout)
    static constexpr int oU = 0, oTZ = SU, oD = 2 * SU, oTZC = 3 * SU, oTZL = 4 * SU, oTS = 3 * SU;
    static constexpr int TS_STEPS = HYB ? (NH_ - 1 - TTM) : 0;
    static constexpr int COLS = (CONSTR ? 5 : 3) * SU + TS_STEPS * NX;
    // tensor memory: x, t (+ the pre-projection state slacks tc = x + gc_prev, tl = x + gl_prev); hybrid: x_1 .. x_{N-2}, t_0 .. t_{TTM-1}
    static constexpr int TM_COLS_PER_THREAD = HYB ? ((NH_ - 2) + TTM) * NX : (CONSTR ? 4 : 2) * SX;
    static_assert(((BLOCK_ / 32 + 3) / 4) * TM_COLS_PER_THREAD <= 512, "the state does not fit the 512 tensor-memory columns");
};

__device__ __forceinline__ float2 sel0(bool c, float2 a) { return make_float2(c ? 0.f : a.x, c ? 0.f : a.y); }   // c ? 0 : a
__device__ __forceinline__ float sel0(bool c, float a) { return c ? 0.f : a; }

// Second-order-cone projection (admm.cpp:39-60) of the block [S, S + D) of a register vector, in place; S and D are
// compile-time, so this is straight-line code on registers.  mu is the reference's float mu; the norm and the two
// quotients use the approximate SFU forms (sqrt.approx, x * rcp(y): <= 2 ulp) -- the fp32 path is compared to the
// reference within a tolerance, the fp64 parity kernels keep the IEEE forms.
template <int S, int D, int N>
__device__ __forceinline__ void project_soc_fixed(Vec<float, N>& v, float mu, float inv_mu) {
    if constexpr (D > 0) {
        float ss = 0.f;
#pragma unroll
        for (int e = S; e < S + D - 1; ++e) ss = fmaf(v.get(e), v.get(e), ss);
        const float lv = v.get(S + D - 1);
        float a;
        asm("sqrt.approx.f32 %0, %1;" : "=f"(a) : "f"(ss));
        const float u0 = lv * mu;
        const bool zero = a <= -u0, inside = a <= u0;
        const float fct = fmaf(0.5f, __fdividef(u0, a), 0.5f);
        const float sc = zero ? 0.f : (inside ? 1.f : fct);
        const float ln = zero ? 0.f : (inside ? lv : fct * (a * inv_mu));
#pragma unroll
        for (int e = S; e < S + D - 1; ++e) v.set(e, sc * v.get(e));
        v.set(S + D - 1, ln);
    }
}

// Half-space projections (admm.cpp:70-73), row after row in place (:148-159 / :162-173); NR rows of N coefficients, their
// offsets b and 1 / ||a||^2, all in the constant bank: straight-line FFMAs with constant operands.
template <int NR, int N>
__device__ __forceinline__ void project_rows_fixed(Vec<float, N>& v, const float* __restrict__ A, const float* __restrict__ b, const float* __restrict__ inv) {
#pragma unroll
    for (int c = 0; c < NR; ++c) {
        float val = 0.f;
#pragma unroll
        for (int e = 0; e < N; ++e) val = fmaf(A[c * N + e], v.get(e), val);
        const float dist = (val > b[c]) ? (val - b[c]) * inv[c] : 0.f;
#pragma unroll
        for (int e = 0; e < N; ++e) v.set(e, fmaf(-dist, A[c * N + e], v.get(e)));
    }
}

template <class C>
__global__ void __launch_bounds__(C::BLOCK, 1)
tpp3_kernel(const __grid_constant__ SolveParams prm, const __grid_constant__ typename C::CPack cp) {
    using T = float;
    using N = Num<T>;
    using P = float2;
    using SP = StaticPack<C::NX, C::NU, C::NH>;
    using VX = Vec<T, C::NX>;
    using VU = Vec<T, C::NU>;
    constexpr int NX = C::NX, NU = C::NU, NH = C::NH, BLOCK = C::BLOCK, SXL = C::SX, SUL = C::SU;
    constexpr int NXP = pad2(NX), NUP = pad2(NU);
    constexpr unsigned FULL = 0xffffffffu;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t pack_bar;
    __shared__ uint32_t tmem_base_s;
    T* pack = reinterpret_cast<T*>(smem_raw);
    const uint32_t pack_bytes = static_cast<uint32_t>(prm.pack_elems) * sizeof(T);

    // ---- cold family tables -> shared memory (one TMA bulk copy per CTA); all 512 tensor-memory columns for the state ----
    if (threadIdx.x == 0) {
        mbar_init(&pack_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(&pack_bar, pack_bytes);
        tma_bulk_g2s(pack, prm.pack, pack_bytes, &pack_bar);
    }
    if (threadIdx.x < 32) tmem_alloc(&tmem_base_s, 512);
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    mbar_wait(&pack_bar, 0);

    T* cta_cols = pack + ((prm.pack_elems + 31) & ~31);
    const int tid = threadIdx.x;
    const uint32_t w_id = static_cast<uint32_t>(tid) >> 5;
    const uint32_t tm_base = tmem_base_s + ((32u * (w_id & 3u)) << 16) + (w_id >> 2) * C::TM_COLS_PER_THREAD;
    // hybrid layout: X.base is biased by one column block (step i at base + i NX for i = 1 .. N-2), T follows the N-2 blocks of X
    const TmemTraj<NX, NH> X{C::HYB ? tm_base - NX : tm_base};                       // x(k)
    const TmemTraj<NX, NH> TT{C::HYB ? tm_base + (NH - 2) * NX : tm_base + SXL};     // t(k) = x(k) + g(k-1)
    Traj<T, NX, (C::TS_STEPS > 0 ? C::TS_STEPS : 1), C::oTS, BLOCK> TS(cta_cols, tid);   // hybrid: t columns TTM .. N-2
    VX xlast, tlast;                              // hybrid: column N-1 of x and t
    xlast.fill(T(0));
    tlast.fill(T(0));
    Traj<T, NU, NH - 1, C::oU, BLOCK> U(cta_cols, tid);      // u(k)
    Traj<T, NU, NH - 1, C::oTZ, BLOCK> TZ(cta_cols, tid);    // u(k) + y(k-1)
    Traj<T, NU, NH - 1, C::oD, BLOCK> ND(cta_cols, tid);     // -dd of the last sweep
    // cone / half-space families (CONSTR): pre-projection slacks, vc = proj(tc), gc = tc - vc (admm.cpp:103-122,191)
    const TmemTraj<NX, NH> TC{tm_base + 2 * SXL};            // x(k) + gc(k-1)
    const TmemTraj<NX, NH> TL{tm_base + 3 * SXL};            // x(k) + gl(k-1)
    Traj<T, NU, NH - 1, C::oTZC, BLOCK> TZC(cta_cols, tid);  // u(k) + yc(k-1)
    Traj<T, NU, NH - 1, C::oTZL, BLOCK> TZL(cta_cols, tid);  // u(k) + yl(k-1)
    const float mu_x = prm.cx[0], mu_u = prm.cu[0], imu_x = 1.f / mu_x, imu_u = 1.f / mu_u;   // the instance's cones (C::SCD, C::UCD)
    // An instance with rows serves only families that enable them (tmpc_capi.cu find_kernel), so its row families are
    // unconditional straight-line code next to the box and the cone of the column.  With zero rows an enabled family still
    // contributes vl - gl = x to the linear cost (admm.cpp:138-140, 223-225): that rare case is a run-time branch.
    const bool lin_x = C::CONSTR && prm.en_state_linear;
    const bool lin_u = C::CONSTR && prm.en_input_linear;

    const T* cP = pack + SP::Pinf;
    const T rho0 = static_cast<T>(prm.rho);
    const T tol_pri = static_cast<T>(prm.abs_pri_tol), tol_dua = static_cast<T>(prm.abs_dua_tol);
    const int max_iter = prm.max_iter, check_every = prm.check_termination;
    const bool en_sb = prm.en_state_bound != 0, en_ib = prm.en_input_bound != 0;
    (void)en_sb; (void)en_ib;

    const int lane = tid & 31;
    const int n_items = prm.batch_ptr ? min(*prm.batch_ptr, prm.batch) : prm.batch;
    const bool producer = prm.q_tail != nullptr;   // exact-count mode: undecidable problems are queued for the fp64 consumer launch
    int prob = 0;
    bool active = false, exhausted = false;
    bool pending = false;   // holds a claimed problem (claim) whose inputs have not landed yet (streamed host pipeline)
    int last_k = 32;        // iterations of the last problem this lane finished (batched refill)
    int claim = 0, seen = 0, unpub = -1;   // seen: cached arrival watermark; unpub: finished problem not yet counted for its chunk
    int k = 0;
    int next_check = check_every;
    T res_px = 0, res_dx = 0, res_pu = 0, res_du = 0;
    VX x0v;
    x0v.fill(T(0));

    // ---- state accessors (one code path for both layouts; i is warp-uniform, so the hybrid branches are uniform) ----
    auto bits_of = [](const VX& v, uint32_t (&r)[NX]) {
#pragma unroll
        for (int e = 0; e < NX; ++e) r[e] = __float_as_uint(v.get(e));
    };
    auto t_issue = [&](int i, uint32_t (&r)[NX]) {
        if constexpr (!C::HYB) { TT.issue(i, r); }
        else {
            if (i < C::TTM) TT.issue(i, r);
            else if (i == NH - 1) bits_of(tlast, r);
            else { VX v; TS.load(i - C::TTM, v); bits_of(v, r); }
        }
    };
    // t column c of the lanes with mine := vals, all other lanes keep theirs.  tcgen05.st has no lane mask: tensor-memory columns
    // are read - select - written warp-wide; shared-memory and register columns are predicated per lane.
    auto t_park = [&](int c, const VX& vals, bool mine) {
        if (!C::HYB || c < C::TTM) {
            uint32_t r[NX];
            TmemSpan<NX>::ld(TT.base + c * NX, r);
            TmemSpan<NX>::wait(r);
#pragma unroll
            for (int e = 0; e < NX; ++e) r[e] = mine ? __float_as_uint(vals.get(e)) : r[e];
            TmemSpan<NX>::st(TT.base + c * NX, r);
        } else if (c == NH - 1) {
#pragma unroll
            for (int e = 0; e < NX; ++e) tlast.set(e, mine ? vals.get(e) : tlast.get(e));
        } else if (mine) {
            TS.store(c - C::TTM, vals);
        }
    };

    auto bt = [](int i) { return C::TIB ? 0 : i; };
    auto xb_pair = [&](int i, int j, size_t pb, P& lo, P& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NX + 2 * j;
            lo = en_sb ? mk2(__ldg(prm.x_min + e), __ldg(prm.x_min + e + 1)) : mk2(-N::inf(), -N::inf());
            hi = en_sb ? mk2(__ldg(prm.x_max + e), __ldg(prm.x_max + e + 1)) : mk2(N::inf(), N::inf());
        } else {
            lo = mk2(cp.xmin[bt(i) * NXP + 2 * j], cp.xmin[bt(i) * NXP + 2 * j + 1]); hi = mk2(cp.xmax[bt(i) * NXP + 2 * j], cp.xmax[bt(i) * NXP + 2 * j + 1]);
        }
    };
    auto xb_tail = [&](int i, size_t pb, T& lo, T& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NX + NX - 1;
            lo = en_sb ? __ldg(prm.x_min + e) : -N::inf();
            hi = en_sb ? __ldg(prm.x_max + e) : N::inf();
        } else { lo = cp.xmin[bt(i) * NXP + NX - 1]; hi = cp.xmax[bt(i) * NXP + NX - 1]; }
    };
    auto ub_pair = [&](int i, int j, size_t pb, P& lo, P& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NU + 2 * j;
            lo = en_ib ? mk2(__ldg(prm.u_min + e), __ldg(prm.u_min + e + 1)) : mk2(-N::inf(), -N::inf());
            hi = en_ib ? mk2(__ldg(prm.u_max + e), __ldg(prm.u_max + e + 1)) : mk2(N::inf(), N::inf());
        } else {
            lo = mk2(cp.umin[bt(i) * NUP + 2 * j], cp.umin[bt(i) * NUP + 2 * j + 1]); hi = mk2(cp.umax[bt(i) * NUP + 2 * j], cp.umax[bt(i) * NUP + 2 * j + 1]);
        }
    };
    auto ub_tail = [&](int i, size_t pb, T& lo, T& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NU + NU - 1;
            lo = en_ib ? __ldg(prm.u_min + e) : -N::inf();
            hi = en_ib ? __ldg(prm.u_max + e) : N::inf();
        } else { lo = cp.umin[bt(i) * NUP + NU - 1]; hi = cp.umax[bt(i) * NUP + NU - 1]; }
    };

    for (;;) {
        // ------------------------------------------------------------------ refill idle lanes
        {
            const bool want = !active && !exhausted && !pending;
            unsigned mw = __ballot_sync(FULL, want);
            // Batched refill: wait until a few lanes are free, unless nothing else keeps the warp busy.  One refill pass costs the
            // warp R ~ 0.23 iterations whatever the number of lanes it serves; with I iterations per problem 32 / I lanes finish
            // per iteration, so a threshold m costs 32 R / (I m) in passes and (m - 1) / 64 in idle lanes: m* = sqrt(2048 R / I)
            // (3 for the hard quadrotor batch, 7 for the easy one; measured optimum 3-4 and >= 8).  I is the warp's mean over
            // the last problem of each lane.  refill_min > 0 fixes the threshold instead.
            if (mw && __any_sync(FULL, active)) {
                int m = prm.refill_min;
                if (m <= 0) {
                    const int sum_k = __reduce_add_sync(FULL, last_k);
                    m = __float2int_rn(sqrtf(__fdividef(471.f * 32.f, (float)max(sum_k, 32))));
                    m = min(max(m, 1), 12);
                }
                if (__popc(mw) < m) mw = 0;
            }
            if (mw) {   // claim the next problem indices (one atomic per warp)
                const int leader = __ffs(mw) - 1;
                int base = 0;
                if (lane == leader) base = atomicAdd(prm.work_counter, __popc(mw));
                base = __shfl_sync(FULL, base, leader);
                if (want) {
                    claim = base + __popc(mw & ((1u << lane) - 1u));
                    if (claim >= n_items) {
                        exhausted = true;
                        prob = 0;
                    } else {
                        if (prm.index_list && prm.order_from == 0) claim = __ldg(prm.index_list + claim);
                        pending = true;
                    }
                }
            }
            // a claimed work item starts once the watermark covers it (always, unless the host streams the batch in): its inputs have
            // landed and, in the ordered part of a streamed batch (SolveParams::order_from), its list entry is written
            const bool listed = prm.order_from > 0 && claim >= prm.order_from;
            const bool mine = pending && problem_ready(prm, claim, seen);
            const unsigned m = __ballot_sync(FULL, mine);
            if (m) {
                if (mine) {
                    prob = listed ? ld_relaxed_gpu(prm.index_list + (claim - prm.order_from)) : claim;
                    pending = false;
                    active = true;
                    k = 0;
                    next_check = check_every;
                    res_px = res_dx = res_pu = res_du = 0;
                }
                const bool have_xref = C::REFS && prm.Xref != nullptr, have_uref = C::REFS && prm.Uref != nullptr;
                // compact reference input (SolveParams::xref_const): one state per problem stands for every column of the horizon
                const bool xconst = have_xref && prm.xref_const != 0;
                if (mine) {
                    if (have_xref && !xconst) {   // pull the whole problem towards L2 first: the blocks below then cost one DRAM round trip
                        const char* s = reinterpret_cast<const char*>(prm.Xref + (size_t)prob * SXL);
#pragma unroll
                        for (int b = 0; b <= (SXL * 4 + 127) / 128; ++b) prefetch_l2(s + (b * 128 < SXL * 4 ? b * 128 : SXL * 4 - 4));
                    }
                    if (have_uref) {
                        const char* s = reinterpret_cast<const char*>(prm.Uref + (size_t)prob * SUL);
#pragma unroll
                        for (int b = 0; b <= (SUL * 4 + 127) / 128; ++b) prefetch_l2(s + (b * 128 < SUL * 4 ? b * 128 : SUL * 4 - 4));
                    }
                    load_span<NX, vec_width(NX, NX)>(prm.x0 + (size_t)prob * NX, [&](int i, float v) { x0v.set(i, v); });
                }
                // T columns of the refilled lanes := -(Xref .* Q) (column N-1: -(xref_N' Pinf)'), all other lanes keep theirs
                // (tcgen05.st has no lane mask: read - select - write, warp-wide)
                if (have_xref) {
                    constexpr int GX = steps_per_block(NH, NX, 64);
                    const float* src = prm.Xref + (size_t)prob * (xconst ? NX : SXL);
                    T xr_last[NX];
#pragma unroll
                    for (int r = 0; r < NX; ++r) xr_last[r] = 0;
#pragma unroll 1
                    for (int b = 0; b < NH / GX; ++b) {
                        float buf[GX * NX];
#pragma unroll
                        for (int e = 0; e < GX * NX; ++e) buf[e] = 0.f;
                        if (mine) {
                            if (xconst) {
                                load_span<NX, vec_width(NX, NX)>(src, [&](int e, float v) {
#pragma unroll
                                    for (int g = 0; g < GX; ++g) buf[g * NX + e] = v;
                                });
                            } else {
                                load_span<GX * NX, vec_width(SXL, GX * NX)>(src + b * GX * NX, [&](int e, float v) { buf[e] = v; });
                            }
                        }
#pragma unroll
                        for (int r = 0; r < NX; ++r) xr_last[r] = buf[(GX - 1) * NX + r];   // after the last block: xref_N
#pragma unroll
                        for (int g = 0; g < GX; ++g) {
                            VX vals;
#pragma unroll
                            for (int e = 0; e < NX; ++e) vals.set(e, -(buf[g * NX + e] * cp.Qd[e]));
                            t_park(b * GX + g, vals, mine);
                        }
                    }
                    {   // PT = -(xref_N' Pinf)' as row pairs of Pinf' (Pinf is row-major in the staged pack)
                        VX acc;
                        acc.fill(T(0));
#pragma unroll
                        for (int r = 0; r < NX; ++r) {
                            const T nxr = -xr_last[r];
#pragma unroll
                            for (int j = 0; j < NX / 2; ++j) acc.p[j] = fmas(mk2(cP[r * NX + 2 * j], cP[r * NX + 2 * j + 1]), nxr, acc.p[j]);
                            if constexpr (NX & 1) acc.t = fmas(cP[r * NX + NX - 1], nxr, acc.t);
                        }
                        t_park(NH - 1, acc, mine);
                    }
                    tmem_wait_st();
                } else {
                    if constexpr (!C::HYB) {
                        TT.reset(mine);
                    } else {
                        VX zero;
                        zero.fill(T(0));
#pragma unroll 1
                        for (int c = 0; c < NH; ++c) t_park(c, zero, mine);
                        tmem_wait_st();
                    }
                }
                // x := 0, u := 0 for the refilled lanes: the first forward pass then ADDS the full affine map like every later
                // increment (no per-element select on "first iteration" in the rollout, 2 % of the instructions), and nothing of the
                // previous problem -- not even a NaN -- survives into the new one.  Tensor-memory columns: read - select - write.
                if constexpr (C::HYB) {
#pragma unroll 1
                    for (int c = 1; c < NH - 1; ++c) {
                        uint32_t r[NX];
                        TmemSpan<NX>::ld(X.base + c * NX, r);
                        TmemSpan<NX>::wait(r);
#pragma unroll
                        for (int e = 0; e < NX; ++e) r[e] = mine ? 0u : r[e];
                        TmemSpan<NX>::st(X.base + c * NX, r);
                    }
                    tmem_wait_st();
#pragma unroll
                    for (int e = 0; e < NX; ++e) xlast.set(e, mine ? T(0) : xlast.get(e));
                } else {
                    X.reset(mine);
                }
                if (mine) {
#pragma unroll 1
                    for (int i = 0; i < NH - 1; ++i) {
#pragma unroll
                        for (int j = 0; j < NU / 2; ++j) U.setp(i, j, mk2(T(0), T(0)));
                        if constexpr (NU & 1) U.sett(i, T(0));
                    }
                }
                if (mine) {
                    // TZ := -(Uref .* R), -dd := -d0 (first backward pass on the zero workspace, tiny_api.cpp:68-105 + admm.cpp:13-20)
                    if (have_uref) {
                        constexpr int GU = steps_per_block(NH - 1, NU, 64);
                        const float* src = prm.Uref + (size_t)prob * SUL;
#pragma unroll 1
                        for (int b = 0; b < (NH - 1) / GU; ++b) {
                            float buf[GU * NU];
                            load_span<GU * NU, vec_width(SUL, GU * NU)>(src + b * GU * NU, [&](int e, float v) { buf[e] = v; });
#pragma unroll
                            for (int g = 0; g < GU; ++g) {
#pragma unroll
                                for (int j = 0; j < NU / 2; ++j)
                                    TZ.setp(b * GU + g, j, mk2(-(buf[g * NU + 2 * j] * cp.Rd[2 * j]), -(buf[g * NU + 2 * j + 1] * cp.Rd[2 * j + 1])));
                                if constexpr (NU & 1) TZ.sett(b * GU + g, -(buf[g * NU + NU - 1] * cp.Rd[NU - 1]));
                            }
                        }
                    }
#pragma unroll 1
                    for (int i = 0; i < NH - 1; ++i) {
#pragma unroll
                        for (int j = 0; j < NU / 2; ++j) {
                            if (!have_uref) TZ.setp(i, j, mk2(T(0), T(0)));
                            ND.setp(i, j, mk2(-pack[SP::d0 + i * NU + 2 * j], -pack[SP::d0 + i * NU + 2 * j + 1]));
                        }
                        if constexpr (NU & 1) {
                            if (!have_uref) TZ.sett(i, T(0));
                            ND.sett(i, -pack[SP::d0 + i * NU + NU - 1]);
                        }
                    }
                }
            }
            if (!__any_sync(FULL, active)) {
                publish_done(prm, unpub);
                if (!__any_sync(FULL, pending)) break;
                __nanosleep(256);   // the whole warp is waiting for the copy engine
                continue;
            }
        }

        const size_t pbx = (size_t)prob * SXL, pbu = (size_t)prob * SUL;

        // ------------------------------------------------- forward rollout of the increment: X += dx, U += du
        {
            const bool ff = (k == 0);                                  // first iteration: the full affine map from x0
            const bool anyff = __any_sync(FULL, active && ff);
            VX dx;
#pragma unroll
            for (int j = 0; j < NX / 2; ++j) dx.p[j] = ff ? x0v.p[j] : mk2(T(0), T(0));
            dx.t = ff ? x0v.t : T(0);
            uint32_t xr[NX];
            if constexpr (!C::HYB) X.issue(0, xr);
            // hybrid layout: x_0 = x0 is not stored (its update is the identity), x_{N-1} is a register column updated after the loop
            constexpr int FEND = C::HYB ? NH - 1 : NH;
#pragma unroll C::TUNROLL
            for (int i = 0; i < FEND; ++i) {
                const int zf = C::OPQ ? opaque_zero4() : 0;
                if (!C::HYB || i >= 1) {
                    VX xo;
                    TmemTraj<NX, NH>::complete(xr, xo);
#pragma unroll
                    for (int j = 0; j < NX / 2; ++j) xo.p[j] = addv(xo.p[j], dx.p[j]);   // a new problem's columns were zeroed at refill
                    if constexpr (NX & 1) xo.t = xo.t + dx.t;
                    X.store(i, xo);
                }
                if (i < NH - 1) {
                    if (!C::HYB || i + 1 <= NH - 2) X.issue(i + 1, xr);   // lands behind the mat-vecs of this step
                    // du_i = -Kinf dx_i - dd_i (admm.cpp:29)
                    VU du;
                    ND.load(i, du);
                    if constexpr (C::CONV) {   // the sweep accumulates the next -dd in this slot
#pragma unroll
                        for (int j = 0; j < NU / 2; ++j) ND.setp(i, j, mk2(T(0), T(0)));
                        if constexpr (NU & 1) ND.sett(i, T(0));
                    }
                    if (i > 0 || anyff) mv_acc<NU, NX>(cp.NK, zf, dx, du);     // dx_0 = 0 unless this is a first iteration
                    VU un;
                    U.load(i, un);
#pragma unroll
                    for (int j = 0; j < NU / 2; ++j) un.p[j] = addv(un.p[j], du.p[j]);
                    if constexpr (NU & 1) un.t = un.t + du.t;
                    U.store(i, un);
                    // dx_{i+1} = A dx_i + B du_i (+ f on the first iteration, admm.cpp:30)
                    VX dxn;
                    if constexpr (C::AFF) {
#pragma unroll
                        for (int j = 0; j < NX / 2; ++j) dxn.p[j] = ff ? mk2(cp.f[2 * j], cp.f[2 * j + 1]) : mk2(T(0), T(0));
                        if constexpr (NX & 1) dxn.t = ff ? cp.f[NX - 1] : T(0);
                    } else {
                        dxn.fill(T(0));
                    }
                    if (i > 0 || anyff) {
                        if constexpr (C::SA::DENSE) mv_acc<NX, NX>(cp.A, zf, dx, dxn);
                        else mv_acc_masked<typename C::SA, NX, NX>(cp.AS, zf, dx, dxn);
                    }
                    mv_acc<NX, NU>(cp.B, zf, du, dxn);
                    dx = dxn;
                }
            }
            if constexpr (C::HYB) {
#pragma unroll
                for (int j = 0; j < NX / 2; ++j) xlast.p[j] = addv(xlast.p[j], dx.p[j]);
                if constexpr (NX & 1) xlast.t = xlast.t + dx.t;
            }
            X.stores_done();
        }
        publish_done(prm, unpub);   // the solution stores of the previous finish are half an iteration old by now
        k += 1;   // work->iter += 1 (admm.cpp:328)

        // ------------------------------------------------- reverse sweep: slack + dual + residuals fused with the Riccati step
        const bool first = (k == 1);
        const T nrho = -rho0;
        T rpx = 0, rdx = 0, rpu = 0, rdu = 0;
        // one trajectory element (pair or scalar tail).  traw: stored pre-clamp slack t(k-1) (on the first sweep: the parked
        // reference term, t(0) = 0).  vo = clamp(t_old), g = t_old - vo, t_new = x + g, vn = clamp(t_new)  (admm.cpp:85,92,184);
        // increment of (slack - dual) = (2 vn - t_new) - (2 vo - t_old) = 2 (vn - vo) - (t_new - t_old) = (vn - vo) - (x - vn); dq = ref - rho dw
        auto slack = [&](auto traw, auto xv, auto lo, auto hi, T& rp, T& rd, auto& tnew, auto& dq) {
            const auto told = sel0(first, traw);
            const auto ref = subv(traw, told);                 // first ? traw : 0
            auto vo = clampv(told, lo, hi);
            if constexpr (!C::FB) vo = sel0(first, vo);        // cold start: v = 0 whatever the bounds are (FB: clamp(0) = 0 already)
            const auto go = subv(told, vo);
            tnew = addv(xv, go);
            const auto vn = clampv(tnew, lo, hi);
            const auto a = subv(xv, vn);                       // primal residual of the element
            rp = amaxv(rp, a);
            const auto e = subv(vn, vo);                       // dual residual / rho
            rd = amaxv(rd, e);
            // t_new - t_old = x - v_old, hence dw = 2 e - (x - v_old) = e - a: the increment of (slack - dual) is the
            // difference of the two residuals
            dq = fmas(subv(e, a), nrho, ref);
        };
        // one more constraint family of a column (cone or half-space): traw = stored pre-projection value x(k-1) + dual(k-2)
        // (garbage of the previous problem on the first sweep, where the cold value is 0 and so is its projection,
        // tiny_api.cpp:88-100).  Same algebra as the box: vo = proj(t_old), dual = t_old - vo, t_new = x + dual,
        // vn = proj(t_new), dq -= rho (2 (vn - vo) - (t_new - t_old)).  The projection is recomputed instead of stored:
        // it is a handful of instructions per column.
        auto family = [&](auto& tv, const auto& xv, auto& dq, auto&& proj) {
            using V = std::decay_t<decltype(tv)>;
            V to, vo, vn;
#pragma unroll
            for (int j = 0; j < V::NP; ++j) to.p[j] = sel0(first, tv.p[j]);
            to.t = V::TAIL ? sel0(first, tv.t) : T(0);
            vo = to;
            proj(vo);
#pragma unroll
            for (int j = 0; j < V::NP; ++j) { vo.p[j] = sel0(first, vo.p[j]); tv.p[j] = addv(xv.p[j], subv(to.p[j], vo.p[j])); }
            if constexpr (V::TAIL) { vo.t = sel0(first, vo.t); tv.t = xv.t + (to.t - vo.t); }
            vn = tv;
            proj(vn);
#pragma unroll
            for (int j = 0; j < V::NP; ++j) dq.p[j] = fmas(twice_minus(subv(vn.p[j], vo.p[j]), subv(tv.p[j], to.p[j])), nrho, dq.p[j]);
            if constexpr (V::TAIL) dq.t = fmas(twice_minus(vn.t - vo.t, tv.t - to.t), nrho, dq.t);
        };
        auto cones_x = [&](VX& v) { project_soc_fixed<C::SCS, C::SCD>(v, mu_x, imu_x); };
        auto cones_u = [&](VU& v) { project_soc_fixed<C::UCS, C::UCD>(v, mu_u, imu_u); };
        auto rows_x = [&](VX& v) { project_rows_fixed<C::NSL>(v, cp.Alx, cp.blx, cp.inx); };
        auto rows_u = [&](VU& v) { project_rows_fixed<C::NIL>(v, cp.Alu, cp.blu, cp.inu); };
        // the state-sized loads of column i are ISSUED at the top of the column (x, t, tc, tl: tensor memory) and completed
        // after the input column's work, which hides their latency
        constexpr bool HAS_TC = C::CONSTR && C::SCD > 0, HAS_TL = C::CONSTR;
        uint32_t rx[NX], rt[NX], rc[HAS_TC ? NX : 1], rl[HAS_TL ? NX : 1];
        auto issue_x = [&](int i, auto col0) {   // every issued load is completed below (column 0 has no cone / half-space work)
            if constexpr (!C::HYB) {
                X.issue(i, rx);
                TT.issue(i, rt);
            } else {   // loop columns N-2 .. 0 only: x_i from tensor memory (x_0 = x0 is taken from registers at the point of use),
                       // t_i from tensor memory or, beyond the warp's share of it, from shared memory
                if constexpr (!decltype(col0)::value) X.issue(i, rx);
                if (i < C::TTM) {
                    TT.issue(i, rt);
                } else {
#pragma unroll
                    for (int j = 0; j < NX / 2; ++j) {
                        const P v = TS.getp(i - C::TTM, j);
                        rt[2 * j] = __float_as_uint(v.x); rt[2 * j + 1] = __float_as_uint(v.y);
                    }
                    if constexpr (NX & 1) rt[NX - 1] = __float_as_uint(TS.gett(i - C::TTM));
                }
            }
            if constexpr (HAS_TC) { if (i > 0) TC.issue(i, rc); }
            if constexpr (HAS_TL) { if (i > 0 && (C::NSL > 0 || lin_x)) TL.issue(i, rl); }
        };
        auto extra_x = [&](int i, const VX& xv, VX& dq) {
            if constexpr (HAS_TC) { VX tc; TmemTraj<NX, NH>::complete(rc, tc); family(tc, xv, dq, cones_x); TC.store(i, tc); }
            if constexpr (HAS_TL) { if (C::NSL > 0 || lin_x) { VX tl; TmemTraj<NX, NH>::complete(rl, tl); family(tl, xv, dq, rows_x); TL.store(i, tl); } }
        };
        auto extra_u = [&](int i, const VU& uv, VU& dr) {
            if constexpr (C::CONSTR) {
                if constexpr (C::UCD > 0) { VU tc; TZC.load(i, tc); family(tc, uv, dr, cones_u); TZC.store(i, tc); }
                if (C::NIL > 0 || lin_u) { VU tl; TZL.load(i, tl); family(tl, uv, dr, rows_u); TZL.store(i, tl); }
            }
        };
        // impulse-response form (C::CONV): -dd_t += -G_k s_j for the steps t = j-1-k before column j.  The slots were zeroed by the
        // forward pass when it consumed them.  Two accumulator chains per product (columns split in halves); the blocks of one
        // call are independent.  Called at the top of column j-1, so that the products run under the latency of that column's
        // state loads, and so that the terminal column needs no copy of this code (the hot loop must fit the 32 KB instruction cache).
        auto scatter = [&](int j, const VX& sv) {
            constexpr int NG1 = NX * NUP, H = NX / 2;
#pragma unroll
            for (int kk = NH - 2; kk >= 0; --kk) {
                if (kk < j) {
                    const int t = j - 1 - kk;
                    VU a, b;
                    ND.load(t, a);
                    b.fill(T(0));
                    const T* __restrict__ M = cp.NG + kk * NG1;
#pragma unroll
                    for (int c = 0; c < H; ++c) {
                        const T x0c = sv.get(c), x1c = sv.get(c + H);
#pragma unroll
                        for (int jj = 0; jj < NU / 2; ++jj) {
                            a.p[jj] = fmas(mk2(M[c * NUP + 2 * jj], M[c * NUP + 2 * jj + 1]), x0c, a.p[jj]);
                            b.p[jj] = fmas(mk2(M[(c + H) * NUP + 2 * jj], M[(c + H) * NUP + 2 * jj + 1]), x1c, b.p[jj]);
                        }
                        if constexpr (NU & 1) { a.t = fmas(M[c * NUP + NU - 1], x0c, a.t); b.t = fmas(M[(c + H) * NUP + NU - 1], x1c, b.t); }
                    }
                    if constexpr (NX & 1) {
                        const T xc = sv.get(NX - 1);
#pragma unroll
                        for (int jj = 0; jj < NU / 2; ++jj) a.p[jj] = fmas(mk2(M[(NX - 1) * NUP + 2 * jj], M[(NX - 1) * NUP + 2 * jj + 1]), xc, a.p[jj]);
                        if constexpr (NU & 1) a.t = fmas(M[(NX - 1) * NUP + NU - 1], xc, a.t);
                    }
#pragma unroll
                    for (int jj = 0; jj < NU / 2; ++jj) a.p[jj] = addv(a.p[jj], b.p[jj]);
                    if constexpr (NU & 1) a.t = a.t + b.t;
                    ND.store(t, a);
                }
            }
        };
        VX dp;
        {   // column N-1: dp_N = -(xref_N' Pinf)' [first sweep] - rho dw_N   (admm.cpp:238-246)
            VX xv, traw, tnew;
            if constexpr (C::HYB) {
                xv = xlast;
                traw = tlast;
            } else {
                issue_x(NH - 1, std::false_type{});
                TmemTraj<NX, NH>::complete(rx, xv);
                TmemTraj<NX, NH>::complete(rt, traw);
            }
#pragma unroll
            for (int j = 0; j < NX / 2; ++j) {
                P lo, hi;
                xb_pair(NH - 1, j, pbx, lo, hi);
                slack(traw.p[j], xv.p[j], lo, hi, rpx, rdx, tnew.p[j], dp.p[j]);
            }
            if constexpr (NX & 1) {
                T lo, hi;
                xb_tail(NH - 1, pbx, lo, hi);
                slack(traw.t, xv.t, lo, hi, rpx, rdx, tnew.t, dp.t);
            }
            if constexpr (C::HYB) tlast = tnew; else TT.store(NH - 1, tnew);
            extra_x(NH - 1, xv, dp);
        }
        // One column of the sweep.  col0 (compile-time): the peeled column 0 of the hybrid layout -- x_0 = x0 comes from registers,
        // and the Riccati step is skipped altogether (p_0 and q_0 are never used, admm.cpp:17 reads p_{i+1}).
        auto sweep_col = [&](int i, auto col0) {
            constexpr bool COL0 = decltype(col0)::value;
            const int zb = C::OPQ ? opaque_zero4() : 0;
            issue_x(i, col0);
            if constexpr (C::CONV) scatter(COL0 ? 1 : i + 1, dp);   // s_{i+1} -> the -dd slots of the steps 0 .. i
            // The two products with dp_{i+1} start from zero and are added to their right-hand sides afterwards: they depend on
            // nothing of this column, so they run under the latency of the column's tensor-/shared-memory loads and the scheduler
            // is free to weave the slack updates (ALU pipe) into their FFMA2 stream (FMA pipe).  Measured: rocket +6 %,
            // quadrotor +1 %; the 4-state shapes lose 1 % to the extra additions and keep the chained form.
            constexpr bool SPLIT = NX >= 6 && !C::CONV;
            VX akp;
            VU btp;
            akp.fill(T(0));
            btp.fill(T(0));
            if constexpr (SPLIT) {
                if constexpr (!COL0) mv_acc<NX, NX>(cp.AK, zb, dp, akp);
                mv_acc<NU, NX>(cp.BT, zb, dp, btp);
            }
            // ---- input column i: dr_i = -(Uref .* R) [first sweep] - rho dw   (admm.cpp:227-236)
            VU uv, dr;
            U.load(i, uv);
#pragma unroll
            for (int j = 0; j < NU / 2; ++j) {
                P lo, hi, tn;
                ub_pair(i, j, pbu, lo, hi);
                slack(TZ.getp(i, j), uv.p[j], lo, hi, rpu, rdu, tn, dr.p[j]);
                TZ.setp(i, j, tn);
            }
            if constexpr (NU & 1) {
                T lo, hi, tn;
                ub_tail(i, pbu, lo, hi);
                slack(TZ.gett(i), uv.t, lo, hi, rpu, rdu, tn, dr.t);
                TZ.sett(i, tn);
            }
            extra_u(i, uv, dr);
            // dd_i = Quu_inv (B' dp + dr)   (admm.cpp:17; BPf cancels in the increment)
            if constexpr (C::CONV) {   // the products with the later columns are already in the slot: -dd_i = slot - Quu_inv dr_i
                VU a;
                ND.load(i, a);
                mv_acc<NU, NU>(cp.NQ, zb, dr, a);
                ND.store(i, a);
            } else {
            VU t = dr;
            if constexpr (SPLIT) {
#pragma unroll
                for (int j = 0; j < NU / 2; ++j) t.p[j] = addv(btp.p[j], dr.p[j]);
                if constexpr (NU & 1) t.t = btp.t + dr.t;
            } else {
                mv_acc<NU, NX>(cp.BT, zb, dp, t);
            }
            VU d;
            d.fill(T(0));
            mv_acc<NU, NU>(cp.Quu, zb, t, d);
            {
                VU nd;
#pragma unroll
                for (int j = 0; j < NU / 2; ++j) nd.p[j] = negv(d.p[j]);
                if constexpr (NU & 1) nd.t = -d.t;
                ND.store(i, nd);
            }
            }
            // ---- state column i: dq_i = -(Xref .* Q) [first sweep] - rho dw;  dp_i = dq_i + AmBKt dp - Kinf' dr   (admm.cpp:18)
            VX xv, traw, tnew, dq;
            if constexpr (C::HYB) {
                TmemTraj<NX, NH>::complete(rt, traw);
                if constexpr (COL0) xv = x0v; else TmemTraj<NX, NH>::complete(rx, xv);
            } else {
                TmemTraj<NX, NH>::complete(rx, xv);
                TmemTraj<NX, NH>::complete(rt, traw);
            }
#pragma unroll
            for (int j = 0; j < NX / 2; ++j) {
                P lo, hi;
                xb_pair(i, j, pbx, lo, hi);
                slack(traw.p[j], xv.p[j], lo, hi, rpx, rdx, tnew.p[j], dq.p[j]);
            }
            if constexpr (NX & 1) {
                T lo, hi;
                xb_tail(i, pbx, lo, hi);
                slack(traw.t, xv.t, lo, hi, rpx, rdx, tnew.t, dq.t);
            }
            if constexpr (C::HYB) {
                if (i < C::TTM) TT.store(i, tnew); else TS.store(i - C::TTM, tnew);
            } else {
                TT.store(i, tnew);
            }
            // p_0 is never used (admm.cpp:17 reads p_{i+1}), hence neither are q_0 and the cone / half-space slacks of x_0; in the
            // rolled loop the Riccati step of column 0 is computed all the same, which keeps the loop body one basic block.
            if (C::CONSTR && i > 0) extra_x(i, xv, dq);
            if constexpr (!COL0) {
                if constexpr (C::CONV) {
                    // s_i = dq_i - Kinf' dr_i, scattered to the steps before i at the top of the next column
                    mv_acc<NX, NU>(cp.NKT, zb, dr, dq);
                    dp = dq;
                } else {
                if constexpr (SPLIT) {
#pragma unroll
                    for (int j = 0; j < NX / 2; ++j) dq.p[j] = addv(dq.p[j], akp.p[j]);
                    if constexpr (NX & 1) dq.t += akp.t;
                } else {
                    mv_acc<NX, NX>(cp.AK, zb, dp, dq);
                }
                mv_acc<NX, NU>(cp.NKT, zb, dr, dq);
                dp = dq;
                }
            }
        };
#pragma unroll C::TUNROLL
        for (int i = NH - 2; i >= (C::HYB ? 1 : 0); --i) sweep_col(i, std::false_type{});
        if constexpr (C::HYB) sweep_col(0, std::true_type{});
        TT.stores_done();

        // ------------------------------------------------- termination (admm.cpp:253-271, 364-388)
        bool finish = false;
        int st = 11;
        if (k == next_check) {   // iter % check_termination == 0
            next_check += check_every;
            res_px = rpx; res_dx = rdx * rho0; res_pu = rpu; res_du = rdu * rho0;
            if (res_px < tol_pri && res_pu < tol_pri && res_dx < tol_dua && res_du < tol_dua) { finish = true; st = 1; }
            if (prm.amb_band > 0.f) {   // mixed mode, see tmpc_tpp2.cuh
                const T up = T(1) + prm.amb_band, dn = T(1) - prm.amb_band;
                const bool below_up = res_px < tol_pri * up && res_pu < tol_pri * up && res_dx < tol_dua * up && res_du < tol_dua * up;
                const bool below_dn = res_px < tol_pri * dn && res_pu < tol_pri * dn && res_dx < tol_dua * dn && res_du < tol_dua * dn;
                if (below_up && !below_dn) { finish = true; st = kAmbiguousBit | 11; }
            }
        }
        if (k >= max_iter) finish = true;
        bool fin = active && finish;
        if (producer) {   // (tmpc_tpp2.cuh, queue_push) no result and no completion count from this lane: the consumer delivers both
            const bool amb = fin && (st & kAmbiguousBit);
            queue_push(prm, amb, prob, lane);
            if (amb) { fin = false; active = false; last_k = k; }
        }
        const bool u0_only = prm.u0 != nullptr;   // compact output (SolveParams::u0): x and u are not written
        if (!u0_only && __any_sync(FULL, fin)) {
            // solution = (vnew, znew) = clamp of the stored pre-clamp values (the T read is warp-collective)
#pragma unroll 1
            for (int i = 0; i < NH; ++i) {
                VX v;
                {
                    uint32_t r[NX];
                    t_issue(i, r);
                    TmemTraj<NX, NH>::complete(r, v);
                }
                if (fin) {
#pragma unroll
                    for (int j = 0; j < NX / 2; ++j) { P lo, hi; xb_pair(i, j, pbx, lo, hi); v.p[j] = clampv(v.p[j], lo, hi); }
                    if constexpr (NX & 1) { T lo, hi; xb_tail(i, pbx, lo, hi); v.t = clampv(v.t, lo, hi); }
                    store_span<NX, vec_width(SXL, NX)>(prm.x + pbx + i * NX, [&](int r) { return v.get(r); });
                }
            }
        }
        if (fin) {
#pragma unroll 1
            for (int i = 0; i < (u0_only ? 1 : NH - 1); ++i) {
                VU z;
#pragma unroll
                for (int j = 0; j < NU / 2; ++j) { P lo, hi; ub_pair(i, j, pbu, lo, hi); z.p[j] = clampv(TZ.getp(i, j), lo, hi); }
                if constexpr (NU & 1) { T lo, hi; ub_tail(i, pbu, lo, hi); z.t = clampv(TZ.gett(i), lo, hi); }
                if (u0_only) store_span<NU, vec_width(NU, NU)>(prm.u0 + (size_t)prob * NU, [&](int a) { return z.get(a); });
                else store_span<NU, vec_width(SUL, NU)>(prm.u + pbu + i * NU, [&](int a) { return z.get(a); });
            }
            prm.iter[prob] = k;
            prm.status[prob] = st;
            if (prm.residuals) *reinterpret_cast<float4*>(prm.residuals + 4 * (size_t)prob) = make_float4(res_px, res_dx, res_pu, res_du);
            if (prm.rho_out) prm.rho_out[prob] = rho0;
            if (prm.done_counters) unpub = prob;
            active = false;
            last_k = k;
        }
    }
    tmem_fence_before_sync();
    __syncthreads();
    if (producer && threadIdx.x == 0) queue_producer_exit(prm);
    if (threadIdx.x < 32) tmem_dealloc(tmem_base_s, 512);
}

template <class C>
inline size_t tpp3_smem_bytes(int pack_elems) {
    return ((size_t)((pack_elems + 31) & ~31) + (size_t)C::COLS * C::BLOCK) * sizeof(float);
}

}  // namespace tmpc
