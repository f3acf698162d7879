// tmpc_tpp2.cuh -- the batched ADMM throughput kernel for sm_100a ("thread per problem", packed-pair form).
//
// Path implemented (reference: tinympc/TinyMPC/src/tinympc/admm.cpp):
//   solve                 :274-389   loop driver, termination, status codes
//   backward_pass_grad    :13-20     d_i = Quu_inv (B' p_{i+1} + r_i + BPf);  p_i = q_i + AmBKt p_{i+1} - Kinf' r_i + APf
//   forward_pass          :25-32     u_i = -Kinf x_i - d_i;  x_{i+1} = A x_i + B u_i + f
//   update_slack          :81-175    box clamp, second-order-cone projection (:39-60), half-space projection (:70-73)
//   update_dual           :181-208
//   update_linear_cost    :214-247   (never materialised: q, r, p_N are recomputed inside the backward sweep)
//   termination_condition :253-271
//   adaptive rho          rho_benchmark.cpp:44-250 in closed block form (SURVEY.md section 8a-8)
//
// Mapping.  One CUDA thread owns one MPC problem for all of its ADMM iterations; a mat-vec is then a
// pure FMA stream with no shuffles.  The kernel is bound by instruction issue and the FP32 pipe, so
// everything is arranged to retire two flops-pairs per issued instruction:
//   * every vector (state, input, costate, slack) is held as PAIRS of adjacent elements and all
//     arithmetic on them is packed f32x2 (FFMA2 / FADD2; fp64 instances run the same code with scalar
//     pairs);
//   * a mat-vec y = M x accumulates column by column into ROW pairs: y(2j,2j+1) += M(2j..2j+1, c) * x_c.
//     ptxas encodes the broadcast of x_c as an operand modifier of FFMA2 (R.F32), so there is no pair-sum,
//     no zero initialisation and no register shuffling; the summation order is Eigen's gemv order;
//   * the family matrices ride in the kernel-parameter constant bank, stored column-major so that the
//     coefficient pair of one FFMA2 is adjacent, and reach the FMA pipe as uniform registers
//     (LDCU.128 = two FFMA2 operands).  A shared-memory broadcast would cap the kernel at 25 % of the
//     FP32 pipe (profiles/microbench/RESULTS.md);
//   * per-problem state lives in conflict-free shared-memory pair columns ([pair][thread], 64-bit
//     accesses) for the whole solve; HBM is touched only to read x0/Xref/Uref once and to write the
//     solution once.  The cold tables (Pinf, d0, linear rows) are staged once per CTA with a TMA bulk
//     copy (cp.async.bulk + mbarrier).
// Problems need 1..max_iter iterations, so lanes are refilled: a lane that finishes claims the next
// problem from a global counter (warp-aggregated atomic) while its neighbours keep iterating.  The
// refill issues all of a problem's loads back to back behind an L2 prefetch, so it costs about one
// DRAM round trip.
//
// State compression.  For the box constraint the reference keeps four arrays per variable: slack
// vnew, previous slack v, dual g (and the trajectory x).  Since vnew = clamp(x + g) and
// g_new = (g + x) - vnew (admm.cpp:85,92,184), the single pre-clamp value t = x + g determines both:
// vnew = clamp(t), g_new = t - vnew.  Only t is stored (TV / TZ).
//
// Loop rotation.  The reference runs backward -> forward -> slack -> dual -> linear cost -> check.
// On a cold workspace (q = r = p = 0) the first backward pass is problem independent, so its result
// d0 is precomputed on the host; each iteration here is forward+slack+dual -> check -> backward (for
// the next iteration): the same sequence of values, without the backward pass of the last iteration.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cstring>
#include <type_traits>

#include "tmpc_common.h"

namespace tmpc {

enum : int { FEAT_BOX = 0, FEAT_CONSTR = 1, FEAT_ADAPT = 2 };
enum : int { REFS_NONE = 0, REFS_L2 = 2 };

// ----------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA bulk copy (global -> shared), L2 prefetch
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Streamed host pipeline (SolveParams::avail_ptr / done_counters).
// problem_ready: has the copy engine delivered problem `prob`?  The watermark is written in stream order behind the chunk's
// H2D copies; it is read from L2 (strong load, no L1 involvement) only when the lane's cached copy does not cover `prob`, and
// the problem's own lines cannot be in this SM's L1 before that (chunk boundaries fall on 128-byte lines, nobody reads ahead
// of the watermark).  A lane whose claimed problem has not landed stays PENDING and re-checks at its warp's next refill
// point while the other lanes keep iterating.
// publish_done: count a finished problem for its chunk's D2H copy.  Called well after the lane stored its solution (half an
// ADMM iteration later), so the release fence finds those stores already acknowledged by L2 and costs next to nothing; the
// copy engine and the stream wait both read through L2, hence device scope.
__device__ __forceinline__ bool problem_ready(const SolveParams& prm, int prob, int& seen) {
    if (prm.avail_ptr == nullptr || seen > prob) return true;
    // acquire: the problem's inputs (written by the copy engine before the watermark) are read after this load
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(prm.avail_ptr) : "memory");
    return seen > prob;
}

// ---- exact-count mode queue (SolveParams::q_*) -----------------------------------------------------------------------
__device__ __forceinline__ int ld_relaxed_gpu(const int* p) { int v; asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ int ld_acquire_gpu(const int* p) { int v; asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void st_release_gpu(int* p, int v) { asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// Producer, warp-collective: the lanes with push == true append their problem (one reservation per warp).
__device__ __forceinline__ void queue_push(const SolveParams& prm, bool push, int prob, int lane) {
    const unsigned m = __ballot_sync(0xffffffffu, push);
    if (!m) return;
    const int leader = __ffs(m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(prm.q_tail, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (push) st_release_gpu(prm.q_list + base + __popc(m & ((1u << lane) - 1u)), prob);
}
// Consumer: is ticket t filled?  none = the producers are gone and the queue ends before t.
__device__ __forceinline__ bool queue_take(const SolveParams& prm, int t, int& prob, bool& none) {
    none = false;
    if (t < ld_relaxed_gpu(prm.q_tail)) {
        const int e = ld_acquire_gpu(prm.q_list + t);
        if (e >= 0) { prob = e; return true; }
        return false;                                            // reserved, not written yet
    }
    if (ld_acquire_gpu(prm.q_prod_done) >= prm.q_prod_total) none = t >= ld_relaxed_gpu(prm.q_tail);
    return false;
}
// Producer CTA exit (after its last push): call from one thread behind a __syncthreads().
__device__ __forceinline__ void queue_producer_exit(const SolveParams& prm) {
    __threadfence();
    atomicAdd(prm.q_prod_done, 1);
}
__device__ __forceinline__ void publish_done(const SolveParams& prm, int& unpub) {
    if (unpub >= 0) {
        asm volatile("fence.release.gpu;" ::: "memory");
        atomicAdd(prm.done_counters + prm.done_map[unpub / prm.done_chunk], 1);
        unpub = -1;
    }
}

// A warp-uniform value that is always 0 but that the compiler cannot prove to be: bit 31 of the upper clock word
// (set only after 2^63 cycles).  Added to the constant-bank index of the matrix tables once per time step, it
// makes their LDCU loads loop-variant.  Without it ptxas hoists ~60 loop-invariant coefficients into the 63
// uniform registers for the whole solve and streams the remaining ~200 per step through a 2-deep window, so every
// FFMA2 waits a full LDCU latency (measured: 50 % issue utilisation, FFMA2 stalled on the short scoreboard).
__device__ __forceinline__ int opaque_zero4() {
    unsigned h;
    asm volatile("mov.u32 %0, %%clock_hi;" : "=r"(h));
    return static_cast<int>((h >> 31) << 2);
}

// ----------------------------------------------------------------------------------------------
// pair arithmetic: float -> packed f32x2 instructions, double -> two scalar operations.
// The same overload names exist for scalars so that generic lambdas serve a vector's odd tail.
// ----------------------------------------------------------------------------------------------
template <typename T> struct PairOf;
template <> struct PairOf<float> { using type = float2; };
template <> struct PairOf<double> { using type = double2; };

__device__ __forceinline__ float2 mk2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ double2 mk2(double a, double b) { return make_double2(a, b); }

// a * s + c with the scalar s broadcast
__device__ __forceinline__ float2 fmas(float2 a, float s, float2 c) { return __ffma2_rn(a, make_float2(s, s), c); }
__device__ __forceinline__ double2 fmas(double2 a, double s, double2 c) { return make_double2(::fma(a.x, s, c.x), ::fma(a.y, s, c.y)); }
__device__ __forceinline__ float fmas(float a, float s, float c) { return fmaf(a, s, c); }
__device__ __forceinline__ double fmas(double a, double s, double c) { return ::fma(a, s, c); }
// a + b, a - b, -a
__device__ __forceinline__ float2 addv(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ double2 addv(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float addv(float a, float b) { return a + b; }
__device__ __forceinline__ double addv(double a, double b) { return a + b; }
__device__ __forceinline__ float2 subv(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ double2 subv(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float subv(float a, float b) { return a - b; }
__device__ __forceinline__ double subv(double a, double b) { return a - b; }
__device__ __forceinline__ float2 negv(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ double2 negv(double2 a) { return make_double2(-a.x, -a.y); }
__device__ __forceinline__ float negv(float a) { return -a; }
__device__ __forceinline__ double negv(double a) { return -a; }
// a * s (scalar broadcast)
__device__ __forceinline__ float2 muls(float2 a, float s) { return __fmul2_rn(a, make_float2(s, s)); }
__device__ __forceinline__ double2 muls(double2 a, double s) { return make_double2(a.x * s, a.y * s); }
__device__ __forceinline__ float muls(float a, float s) { return a * s; }
__device__ __forceinline__ double muls(double a, double s) { return a * s; }
// element-wise product
__device__ __forceinline__ float2 mulv(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ double2 mulv(double2 a, double2 b) { return make_double2(a.x * b.x, a.y * b.y); }
__device__ __forceinline__ float mulv(float a, float b) { return a * b; }
__device__ __forceinline__ double mulv(double a, double b) { return a * b; }
// min(hi, max(lo, t))  (admm.cpp:91-98 order: max with the lower bound first)
__device__ __forceinline__ float2 clampv(float2 t, float2 lo, float2 hi) { return make_float2(fminf(hi.x, fmaxf(lo.x, t.x)), fminf(hi.y, fmaxf(lo.y, t.y))); }
__device__ __forceinline__ double2 clampv(double2 t, double2 lo, double2 hi) { return make_double2(::fmin(hi.x, ::fmax(lo.x, t.x)), ::fmin(hi.y, ::fmax(lo.y, t.y))); }
__device__ __forceinline__ float clampv(float t, float lo, float hi) { return fminf(hi, fmaxf(lo, t)); }
__device__ __forceinline__ double clampv(double t, double lo, double hi) { return ::fmin(hi, ::fmax(lo, t)); }
// 2 v - t
__device__ __forceinline__ float2 twice_minus(float2 v, float2 t) { return __ffma2_rn(v, make_float2(2.f, 2.f), make_float2(-t.x, -t.y)); }
__device__ __forceinline__ double2 twice_minus(double2 v, double2 t) { return make_double2(::fma(2.0, v.x, -t.x), ::fma(2.0, v.y, -t.y)); }
__device__ __forceinline__ float twice_minus(float v, float t) { return fmaf(2.f, v, -t); }
__device__ __forceinline__ double twice_minus(double v, double t) { return ::fma(2.0, v, -t); }
// running infinity norm: max(r, |a|)
__device__ __forceinline__ float amaxv(float r, float2 a) { return fmaxf(r, fmaxf(fabsf(a.x), fabsf(a.y))); }
__device__ __forceinline__ double amaxv(double r, double2 a) { return ::fmax(r, ::fmax(::fabs(a.x), ::fabs(a.y))); }
__device__ __forceinline__ float amaxv(float r, float a) { return fmaxf(r, fabsf(a)); }
__device__ __forceinline__ double amaxv(double r, double a) { return ::fmax(r, ::fabs(a)); }
__device__ __forceinline__ float2 zero_like(float2) { return make_float2(0.f, 0.f); }
__device__ __forceinline__ double2 zero_like(double2) { return make_double2(0.0, 0.0); }
__device__ __forceinline__ float zero_like(float) { return 0.f; }
__device__ __forceinline__ double zero_like(double) { return 0.0; }

template <typename T> struct Num;
template <> struct Num<float> {
    static __device__ __forceinline__ float fma(float a, float b, float c) { return fmaf(a, b, c); }
    static __device__ __forceinline__ float abs(float a) { return fabsf(a); }
    static __device__ __forceinline__ float max(float a, float b) { return fmaxf(a, b); }
    static __device__ __forceinline__ float min(float a, float b) { return fminf(a, b); }
    static __device__ __forceinline__ float sqrt(float a) { return sqrtf(a); }
    static __device__ __forceinline__ float inf() { return CUDART_INF_F; }
};
template <> struct Num<double> {
    static __device__ __forceinline__ double fma(double a, double b, double c) { return ::fma(a, b, c); }
    static __device__ __forceinline__ double abs(double a) { return ::fabs(a); }
    static __device__ __forceinline__ double max(double a, double b) { return ::fmax(a, b); }
    static __device__ __forceinline__ double min(double a, double b) { return ::fmin(a, b); }
    static __device__ __forceinline__ double sqrt(double a) { return ::sqrt(a); }
    static __device__ __forceinline__ double inf() { return CUDART_INF; }
};

// ----------------------------------------------------------------------------------------------
// a length-N vector in registers: N/2 pairs + a scalar tail when N is odd
// ----------------------------------------------------------------------------------------------
template <typename T, int N>
struct Vec {
    using P = typename PairOf<T>::type;
    static constexpr int NP = N / 2;
    static constexpr bool TAIL = (N & 1) != 0;
    P p[NP > 0 ? NP : 1];
    T t;
    __device__ __forceinline__ T get(int r) const {
        if (TAIL && r == N - 1) return t;
        return (r & 1) ? p[r >> 1].y : p[r >> 1].x;
    }
    __device__ __forceinline__ void set(int r, T v) {
        if (TAIL && r == N - 1) { t = v; return; }
        if (r & 1) p[r >> 1].y = v; else p[r >> 1].x = v;
    }
    __device__ __forceinline__ void fill(T v) {
#pragma unroll
        for (int j = 0; j < NP; ++j) p[j] = mk2(v, v);
        t = v;
    }
};

// v[j] = f(j-th pair index, is_tail) helpers: apply a generic lambda to every pair and to the tail.
// f receives (j, element_index_of_first, pair_or_scalar references...) through captured Vec's.
#define TMPC_FOR_PAIRS(VecType, j) _Pragma("unroll") for (int j = 0; j < VecType::NP; ++j)

// padded row count of a column-major constant table
__host__ __device__ constexpr int pad2(int n) { return (n + 1) & ~1; }

// acc += M x for a ROWS x COLS matrix stored column-major with padded column stride pad2(ROWS) in the
// constant bank: M[c * pad2(ROWS) + r].  Column by column into row pairs (gemv order).
template <int ROWS, int COLS, typename T>
__device__ __forceinline__ void mv_acc(const T* __restrict__ M0, int z, const Vec<T, COLS>& x, Vec<T, ROWS>& acc) {
    constexpr int RP = pad2(ROWS);
    const T* __restrict__ M = M0 + z;
#pragma unroll
    for (int c = 0; c < COLS; ++c) {
        const T xc = x.get(c);
#pragma unroll
        for (int j = 0; j < ROWS / 2; ++j) acc.p[j] = fmas(mk2(M[c * RP + 2 * j], M[c * RP + 2 * j + 1]), xc, acc.p[j]);
        if constexpr (ROWS & 1) acc.t = fmas(M[c * RP + ROWS - 1], xc, acc.t);
    }
}

// Compile-time sparsity pattern of a square matrix at row-pair granularity: M = one mask per column, bit j = row pair (2j, 2j+1),
// bit ROWS / 2 = the odd tail row; an empty list means dense.  A masked product skips the pairs whose coefficients are both zero.
template <unsigned... M>
struct SparsePairs {
    static constexpr int NCOL = static_cast<int>(sizeof...(M));
    static constexpr bool DENSE = NCOL == 0;
    static constexpr unsigned kCols[NCOL + 1] = {M..., 0u};   // host side: the registry's copy of the pattern
    __host__ __device__ static constexpr unsigned col(int c) {
        unsigned r = 0;
        int i = 0;
        ((r |= (i++ == c ? M : 0u)), ...);
        return r;
    }
    // packed coefficients (SparsePairs::pack): the masked pairs column by column, then the masked tail entries
    __host__ __device__ static constexpr int pairs(int rows) {
        int n = 0;
        for (int c = 0; c < NCOL; ++c)
            for (int j = 0; j < rows / 2; ++j) n += (col(c) >> j) & 1u;
        return n;
    }
    __host__ __device__ static constexpr int packed(int rows) {
        int n = 2 * pairs(rows);
        if (rows & 1)
            for (int c = 0; c < NCOL; ++c) n += (col(c) >> (rows / 2)) & 1u;
        return n;
    }
    template <typename T>
    static void pack(T* dst, const T* M0, int rows) {   // M0 column-major with stride pad2(rows), as mv_acc reads it
        const int rp = pad2(rows);
        int k = 0;
        for (int c = 0; c < NCOL; ++c)
            for (int j = 0; j < rows / 2; ++j)
                if ((col(c) >> j) & 1u) { dst[k++] = M0[c * rp + 2 * j]; dst[k++] = M0[c * rp + 2 * j + 1]; }
        if (rows & 1)
            for (int c = 0; c < NCOL; ++c)
                if ((col(c) >> (rows / 2)) & 1u) dst[k++] = M0[c * rp + rows - 1];
    }
};

// acc += M x as mv_acc computes it, for a matrix with the nonzero pattern S, from its packed coefficients MP (SparsePairs::pack):
// the products of the masked pairs in mv_acc's order, so that the result equals mv_acc's for finite x up to the sign of an
// exact zero (fma(0, x, acc) = acc).
template <class S, int ROWS, int COLS, typename T>
__device__ __forceinline__ void mv_acc_masked(const T* __restrict__ MP, int z, const Vec<T, COLS>& x, Vec<T, ROWS>& acc) {
    static_assert(S::NCOL == COLS, "pattern of another shape");
    constexpr int NPAIR = S::pairs(ROWS);
    const T* __restrict__ M = MP + z;
    int k = 0, kt = 2 * NPAIR;
#pragma unroll
    for (int c = 0; c < COLS; ++c) {
        const T xc = x.get(c);
#pragma unroll
        for (int j = 0; j < ROWS / 2; ++j)
            if ((S::col(c) >> j) & 1u) { acc.p[j] = fmas(mk2(M[2 * k], M[2 * k + 1]), xc, acc.p[j]); ++k; }
        if constexpr (ROWS & 1) {
            if ((S::col(c) >> (ROWS / 2)) & 1u) { acc.t = fmas(M[kt], xc, acc.t); ++kt; }
        }
    }
}

// ----------------------------------------------------------------------------------------------
// family tables in the kernel-parameter constant bank.  Every matrix is stored COLUMN-major with an
// even (padded) column stride: the coefficient pair (M[2j][c], M[2j+1][c]) of one FFMA2 is adjacent.
// ----------------------------------------------------------------------------------------------
template <typename T, int NX, int NU, int NH, bool ADAPT>
struct alignas(16) ConstPack2 {
    static constexpr int NXP = pad2(NX), NUP = pad2(NU);
    T A[NX * NXP];       // A            (x_next = A x + B u + f)
    T B[NU * NXP];       // B
    T NK[NX * NUP];      // -Kinf        (u = -Kinf x - d)
    T BT[NX * NUP];      // B'           (backward: B' p)
    T Quu[NU * NUP];     // Quu_inv
    T AK[NX * NXP];      // AmBKt
    T NKT[NU * NXP];     // -Kinf'       (backward: - Kinf' r)
    T f[NXP], APf[NXP], BPf[NUP];
    T Qd[NXP], Rd[NUP];
    // shared bounds, padded time-major [i][NXP] / [i][NUP].  Always indexed by the time step, also when they
    // are constant over the horizon: a loop-invariant bound would be hoisted into uniform registers for the
    // whole solve (32 of the 63 there are), which starves the LDCU stream that feeds the FFMA2 operands.
    T xmin[NXP * NH], xmax[NXP * NH];
    T umin[NUP * (NH - 1)], umax[NUP * (NH - 1)];
    // adaptive rho: -dKinf, -dKinf', A' (A' g of the dual residual)
    T NdK[ADAPT ? NX * NUP : 2], NdKT[ADAPT ? NU * NXP : 2], AT[ADAPT ? NX * NXP : 2];
};

template <typename T, int NX, int NU, int NH, bool ADAPT>
inline void fill_const_pack2(ConstPack2<T, NX, NU, NH, ADAPT>& c, const double* pk, const PackLayout& L) {
    constexpr int NXP = pad2(NX), NUP = pad2(NU);
    std::memset(&c, 0, sizeof(c));
    // src row-major (rows x cols) -> dst column-major with stride RP, scaled by sgn
    auto colmajor = [&](T* dst, int at, int rows, int cols, int RP, double sgn) {
        for (int r = 0; r < rows; ++r) for (int k = 0; k < cols; ++k) dst[k * RP + r] = static_cast<T>(sgn * pk[at + r * cols + k]);
    };
    // dst = column-major of the TRANSPOSE of the row-major (rows x cols) source: dst[(r) * RP + k] = src[r][k]
    auto colmajor_t = [&](T* dst, int at, int rows, int cols, int RP, double sgn) {
        for (int r = 0; r < rows; ++r) for (int k = 0; k < cols; ++k) dst[r * RP + k] = static_cast<T>(sgn * pk[at + r * cols + k]);
    };
    auto vec = [&](T* dst, int at, int n) { for (int i = 0; i < n; ++i) dst[i] = static_cast<T>(pk[at + i]); };
    colmajor(c.A, L.A, NX, NX, NXP, 1.0);
    colmajor(c.B, L.B, NX, NU, NXP, 1.0);
    colmajor(c.NK, L.Kinf, NU, NX, NUP, -1.0);
    colmajor_t(c.BT, L.B, NX, NU, NUP, 1.0);          // (B')[a][r] = B[r][a], stored at [r * NUP + a]
    colmajor(c.Quu, L.Quu_inv, NU, NU, NUP, 1.0);
    colmajor(c.AK, L.AmBKt, NX, NX, NXP, 1.0);
    colmajor_t(c.NKT, L.Kinf, NU, NX, NXP, -1.0);     // (-Kinf')[c][a] = -Kinf[a][c], stored at [a * NXP + c]
    vec(c.f, L.f, NX); vec(c.APf, L.APf, NX); vec(c.BPf, L.BPf, NU); vec(c.Qd, L.Qd, NX); vec(c.Rd, L.Rd, NU);
    const int steps_x = NH, steps_u = NH - 1;
    for (int i = 0; i < steps_x; ++i) for (int r = 0; r < NX; ++r) { c.xmin[i * NXP + r] = static_cast<T>(pk[L.xmin + i * NX + r]); c.xmax[i * NXP + r] = static_cast<T>(pk[L.xmax + i * NX + r]); }
    for (int i = 0; i < steps_u; ++i) for (int a = 0; a < NU; ++a) { c.umin[i * NUP + a] = static_cast<T>(pk[L.umin + i * NU + a]); c.umax[i * NUP + a] = static_cast<T>(pk[L.umax + i * NU + a]); }
    if (ADAPT) {
        colmajor(c.NdK, L.dKinf, NU, NX, NUP, -1.0);
        colmajor_t(c.NdKT, L.dKinf, NU, NX, NXP, -1.0);
        colmajor_t(c.AT, L.A, NX, NX, NXP, 1.0);      // (A')[c][r] = A[r][c], stored at [r * NXP + c]
    }
}

// ----------------------------------------------------------------------------------------------
// per-thread trajectory in shared memory: S steps of N elements, as S*(N/2) pair columns
// ([pair][thread], 64-bit per lane, conflict free) followed by S scalar columns when N is odd.
// OFF is in scalar columns from the CTA's column base.
// ----------------------------------------------------------------------------------------------
template <typename T, int N, int S, int OFF, int BLOCK>
struct Traj {
    using P = typename PairOf<T>::type;
    static constexpr int NP = N / 2;
    static constexpr int COLS = S * N;   // scalar columns occupied
    P* pp;
    T* tp;
    __device__ __forceinline__ explicit Traj(T* cta_cols, int tid)
        : pp(reinterpret_cast<P*>(cta_cols + (size_t)OFF * BLOCK) + tid), tp(cta_cols + (size_t)(OFF + S * NP * 2) * BLOCK + tid) {}
    __device__ __forceinline__ P getp(int i, int j) const { return pp[(i * NP + j) * BLOCK]; }
    __device__ __forceinline__ void setp(int i, int j, P v) { pp[(i * NP + j) * BLOCK] = v; }
    __device__ __forceinline__ T gett(int i) const { return tp[i * BLOCK]; }
    __device__ __forceinline__ void sett(int i, T v) { tp[i * BLOCK] = v; }
    __device__ __forceinline__ void load(int i, Vec<T, N>& v) const {
#pragma unroll
        for (int j = 0; j < NP; ++j) v.p[j] = getp(i, j);
        if constexpr (N & 1) v.t = gett(i);
    }
    __device__ __forceinline__ void store(int i, const Vec<T, N>& v) {
#pragma unroll
        for (int j = 0; j < NP; ++j) setp(i, j, v.p[j]);
        if constexpr (N & 1) sett(i, v.t);
    }
};

template <typename T, int OFF, int BLOCK>
struct Col {
    T* base;
    __device__ __forceinline__ explicit Col(T* cta_cols, int tid) : base(cta_cols + (size_t)OFF * BLOCK + tid) {}
    __device__ __forceinline__ T get(int i) const { return base[i * BLOCK]; }
    __device__ __forceinline__ void set(int i, T v) { base[i * BLOCK] = v; }
};


// ----------------------------------------------------------------------------------------------
// Tensor memory as a per-thread scratchpad.  TMEM is 128 lanes x 512 columns x 32 bit per SM; warp w of a CTA
// may touch lanes 32 (w % 4) .. +31, and the 32x32b shape of tcgen05.ld / tcgen05.st gives every thread N
// consecutive columns of "its" lane -- exactly the [element][thread] column layout of the shared-memory
// state, in a second 256 KB memory that this (tensor-core free) kernel would otherwise leave idle.  Holding
// the largest state array (TV) there doubles the number of resident problems per SM.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// NC consecutive columns -> registers.  The loaded registers are threaded through the wait so that no consumer
// can be scheduled above it.
template <int NC> struct TmemIO;
template <> struct TmemIO<1> {
    static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) { asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(a)); }
    static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) { asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(a), "r"(r[0]) : "memory"); }
    static __device__ __forceinline__ void wait(uint32_t* r) { asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0])::"memory"); }
};
template <> struct TmemIO<2> {
    static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) { asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a)); }
    static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) { asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(a), "r"(r[0]), "r"(r[1]) : "memory"); }
    static __device__ __forceinline__ void wait(uint32_t* r) { asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1])::"memory"); }
};
template <> struct TmemIO<4> {
    static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
    }
    static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
    }
    static __device__ __forceinline__ void wait(uint32_t* r) { asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3])::"memory"); }
};
template <> struct TmemIO<8> {
    static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(a));
    }
    static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                     ::"r"(a), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
    }
    static __device__ __forceinline__ void wait(uint32_t* r) {
        asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7])::"memory");
    }
};
template <> struct TmemIO<16> {
    static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                       "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(a));
    }
    static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                     ::"r"(a), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
                       "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
    }
    static __device__ __forceinline__ void wait(uint32_t* r) {
        asm volatile("tcgen05.wait::ld.sync.aligned;"
                     : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                       "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])::"memory");
    }
};
// N columns as a sum of power-of-two chunks (largest first)
template <int N, int CH = 16>
struct TmemSpan {
    static constexpr int K = (N >= CH) ? CH : 0;
    static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
        if constexpr (K > 0) { TmemIO<K>::ld(a, r); TmemSpan<N - K, CH>::ld(a + K, r + K); }
        else if constexpr (N > 0) TmemSpan<N, CH / 2>::ld(a, r);
    }
    static __device__ __forceinline__ void wait(uint32_t* r) {   // one wait per chunk keeps every register behind a wait
        if constexpr (K > 0) { TmemIO<K>::wait(r); TmemSpan<N - K, CH>::wait(r + K); }
        else if constexpr (N > 0) TmemSpan<N, CH / 2>::wait(r);
    }
    static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
        if constexpr (K > 0) { TmemIO<K>::st(a, r); TmemSpan<N - K, CH>::st(a + K, r + K); }
        else if constexpr (N > 0) TmemSpan<N, CH / 2>::st(a, r);
    }
};
template <int CH> struct TmemSpan<0, CH> {
    static __device__ __forceinline__ void ld(uint32_t, uint32_t*) {}
    static __device__ __forceinline__ void wait(uint32_t*) {}
    static __device__ __forceinline__ void st(uint32_t, const uint32_t*) {}
};

// S steps of N float elements in this thread's TMEM lane, starting at column `base` (fp32 instances only).
// Every member is warp-collective (.sync.aligned): call them from warp-uniform control flow only.
template <int N, int S>
struct TmemTraj {
    uint32_t base;   // TMEM address: (first lane of the warp's quarter) << 16 | first column of this warp
    __device__ __forceinline__ void load(int i, Vec<float, N>& v) const {
        uint32_t r[N];
        TmemSpan<N>::ld(base + i * N, r);
        TmemSpan<N>::wait(r);
#pragma unroll
        for (int e = 0; e < N; ++e) v.set(e, __uint_as_float(r[e]));
    }
    // split form: issue the load of step i early (no wait), complete it right before the first use -- the tensor-memory
    // latency then overlaps whatever sits in between.  tcgen05.wait::ld covers every load issued before it.
    __device__ __forceinline__ void issue(int i, uint32_t (&r)[N]) const { TmemSpan<N>::ld(base + i * N, r); }
    static __device__ __forceinline__ void complete(uint32_t (&r)[N], Vec<float, N>& v) {
        TmemSpan<N>::wait(r);
#pragma unroll
        for (int e = 0; e < N; ++e) v.set(e, __uint_as_float(r[e]));
    }
    __device__ __forceinline__ void store(int i, const Vec<float, N>& v) const {
        uint32_t r[N];
#pragma unroll
        for (int e = 0; e < N; ++e) r[e] = __float_as_uint(v.get(e));
        TmemSpan<N>::st(base + i * N, r);
    }
    // zero the whole trajectory of the lanes with mine == true, keep the others (tcgen05.st has no lane mask)
    __device__ __forceinline__ void reset(bool mine) const {
#pragma unroll 1
        for (int i = 0; i < S; ++i) {
            uint32_t r[N];
            TmemSpan<N>::ld(base + i * N, r);
            TmemSpan<N>::wait(r);
#pragma unroll
            for (int e = 0; e < N; ++e) r[e] = mine ? 0u : r[e];
            TmemSpan<N>::st(base + i * N, r);
        }
        tmem_wait_st();
    }
    __device__ __forceinline__ void stores_done() const { tmem_wait_st(); }
};

// the same interface over shared-memory pair columns
template <typename T, int N, int S, int OFF, int BLOCK>
struct SmemTraj : Traj<T, N, S, OFF, BLOCK> {
    using Base = Traj<T, N, S, OFF, BLOCK>;
    __device__ __forceinline__ SmemTraj(T* cta_cols, int tid) : Base(cta_cols, tid) {}
    __device__ __forceinline__ void reset(bool mine) {
        if (mine) {
#pragma unroll 1
            for (int i = 0; i < S; ++i) {
#pragma unroll
                for (int j = 0; j < N / 2; ++j) Base::setp(i, j, mk2(T(0), T(0)));
                if constexpr (N & 1) Base::sett(i, T(0));
            }
        }
    }
    __device__ __forceinline__ void stores_done() const {}
};

template <typename T_, int NX_, int NU_, int NH_, int FEAT_, int BLOCK_, int REFS_, bool PPB_, int MINB_ = 1, bool FB_ = false, bool AFF_ = true, int NTM_ = 0, bool OPQ_ = true, bool TIB_ = false>
struct Tpp2Cfg {
    using T = T_;
    static constexpr int NX = NX_, NU = NU_, NH = NH_, FEAT = FEAT_, BLOCK = BLOCK_, MINB = MINB_;
    static constexpr int REFMODE = REFS_;
    static constexpr bool REFS = REFS_ != REFS_NONE;        // per-problem Xref/Uref present
    static constexpr bool PPB = PPB_;                       // per-problem bounds read from global memory
    static constexpr bool FB = FB_ && !PPB_;                // "fast box": every shared box contains 0 (cold start needs no special case)
    static constexpr bool AFF = AFF_;                       // affine dynamics term: f, APf, BPf may be non-zero
    static constexpr bool TIB = TIB_ && FB_ && !PPB_ && !OPQ_;   // fast-box bounds read from time row 0 with immediate addresses
    static constexpr bool OPQ = OPQ_;                       // loop-variant (opaque) constant-bank offsets: see opaque_zero4()
    // number of state-sized arrays held in tensor memory instead of shared memory, in the order TV, GC, GL, SXT
    // (the last three exist only with cones / linear rows); one CTA per SM owns all 512 columns
    static constexpr int NTM = (sizeof(T_) == 4) ? ((FEAT_ == FEAT_CONSTR) ? NTM_ : (NTM_ > 0 ? 1 : 0)) : 0;
    static constexpr bool TM = NTM > 0;
    static constexpr bool CONSTR = FEAT_ == FEAT_CONSTR;
    static constexpr bool ADAPT = FEAT_ == FEAT_ADAPT;
    static constexpr int SX = NX * NH, SU = NU * (NH - 1);
    using CPack = ConstPack2<T_, NX_, NU_, NH_, ADAPT>;
    static constexpr int VX = (NX_ % 4 == 0) ? 4 : ((NX_ % 2 == 0) ? 2 : 1);   // elements per vector load of the reference scratch
    static constexpr int VU = (NU_ % 4 == 0) ? 4 : ((NU_ % 2 == 0) ? 2 : 1);
    // scalar-column offsets of the shared-memory state
    static constexpr int oTV = 0;
    static constexpr int oTZ = oTV + (NTM >= 1 ? 0 : SX);
    static constexpr int oD = oTZ + SU;
    static constexpr int oGC = oD + SU;
    static constexpr int oGL = oGC + (CONSTR && NTM < 2 ? SX : 0);
    static constexpr int oSX = oGL + (CONSTR && NTM < 3 ? SX : 0);
    static constexpr int oYC = oSX + (CONSTR && NTM < 4 ? SX : 0);
    static constexpr int oYL = oYC + (CONSTR ? SU : 0);
    static constexpr int oSU = oYL + (CONSTR ? SU : 0);
    static constexpr int oSCR = oSU + (CONSTR ? SU : 0);
    static constexpr int COLS = oSCR + (CONSTR ? (NX > NU ? NX : NU) : 0);   // + cone scratch column
    // tensor-memory columns per thread: warps w, w+4, w+8, ... share a lane quarter
    static constexpr int TM_COLS_PER_THREAD = NTM * SX;
    static_assert(((BLOCK_ / 32 + 3) / 4) * TM_COLS_PER_THREAD <= 512, "the state does not fit the 512 tensor-memory columns");
};

// second-order-cone projection of scr[start .. start+dim) in place (admm.cpp:39-60).
// mu and the norm are float in the reference (:39,:42); a/mu is a float division (:54).
template <typename T, int BLOCK>
__device__ __forceinline__ void project_soc_col2(T* scr, int start, int dim, float mu) {
    using N = Num<T>;
    T* s = scr + start * BLOCK;
    const T last = s[(dim - 1) * BLOCK];
    const T u0 = last * static_cast<T>(mu);
    T ss = 0;
    for (int j = 0; j < dim - 1; ++j) { T e = s[j * BLOCK]; ss = N::fma(e, e, ss); }
    const float a = static_cast<float>(N::sqrt(ss));
    const T aT = static_cast<T>(a);
    if (aT <= -u0) {
        for (int j = 0; j < dim; ++j) s[j * BLOCK] = T(0);
    } else if (aT <= u0) {
        // inside the cone
    } else {
        const T fct = T(0.5) * (T(1) + u0 / aT);
        for (int j = 0; j < dim - 1; ++j) s[j * BLOCK] = fct * s[j * BLOCK];
        s[(dim - 1) * BLOCK] = fct * static_cast<T>(a / mu);
    }
}

// largest vector width (in floats: 4, 2 or 1) that divides both a and b
__host__ __device__ constexpr int vec_width(int a, int b) { return (a % 4 == 0 && b % 4 == 0) ? 4 : ((a % 2 == 0 && b % 2 == 0) ? 2 : 1); }

// vectorised read-only load of LEN contiguous floats starting at src, which is aligned to AL floats
// (AL = 4, 2 or 1 and divides LEN); all loads are issued before the first use
template <int LEN, int AL, typename F>
__device__ __forceinline__ void load_span(const float* __restrict__ src, F&& sink) {
    static_assert(LEN % AL == 0, "span length must be a multiple of its alignment");
    if constexpr (AL == 4) {
        float4 t[LEN / 4];
#pragma unroll
        for (int k = 0; k < LEN / 4; ++k) t[k] = __ldg(reinterpret_cast<const float4*>(src) + k);
#pragma unroll
        for (int k = 0; k < LEN / 4; ++k) { sink(4 * k + 0, t[k].x); sink(4 * k + 1, t[k].y); sink(4 * k + 2, t[k].z); sink(4 * k + 3, t[k].w); }
    } else if constexpr (AL == 2) {
        float2 t[LEN / 2];
#pragma unroll
        for (int k = 0; k < LEN / 2; ++k) t[k] = __ldg(reinterpret_cast<const float2*>(src) + k);
#pragma unroll
        for (int k = 0; k < LEN / 2; ++k) { sink(2 * k + 0, t[k].x); sink(2 * k + 1, t[k].y); }
    } else {
        float t[LEN];
#pragma unroll
        for (int k = 0; k < LEN; ++k) t[k] = __ldg(src + k);
#pragma unroll
        for (int k = 0; k < LEN; ++k) sink(k, t[k]);
    }
}
template <int LEN, int AL, typename F>
__device__ __forceinline__ void store_span(float* __restrict__ dst, F&& src) {
    static_assert(LEN % AL == 0, "span length must be a multiple of its alignment");
    if constexpr (AL == 4) {
        float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
        for (int k = 0; k < LEN / 4; ++k) d4[k] = make_float4(src(4 * k), src(4 * k + 1), src(4 * k + 2), src(4 * k + 3));
    } else if constexpr (AL == 2) {
        float2* d2 = reinterpret_cast<float2*>(dst);
#pragma unroll
        for (int k = 0; k < LEN / 2; ++k) d2[k] = make_float2(src(2 * k), src(2 * k + 1));
    } else {
#pragma unroll
        for (int k = 0; k < LEN; ++k) dst[k] = src(k);
    }
}

// largest number of whole steps (of N elements) per refill block with at most `cap` elements in flight
__host__ __device__ constexpr int steps_per_block(int steps, int n, int cap) {
    int best = 1;
    for (int g = 1; g <= steps; ++g) if (steps % g == 0 && g * n <= cap) best = g;
    return best;
}

// vector type of V elements of T for the lane-interleaved reference scratch
template <typename T, int V> struct VecOf;
template <> struct VecOf<float, 4> { using type = float4; };
template <> struct VecOf<float, 2> { using type = float2; };
template <> struct VecOf<float, 1> { using type = float; };
template <> struct VecOf<double, 4> { using type = double4; };
template <> struct VecOf<double, 2> { using type = double2; };
template <> struct VecOf<double, 1> { using type = double; };

// A register copy the compiler cannot coalesce away (volatile mov): keeps the destination of a prefetch and the
// value still in use in DIFFERENT registers, so that the prefetch can be issued at the top of a loop body.
__device__ __forceinline__ float pinned_copy(float s) { float d; asm volatile("mov.b32 %0, %1;" : "=f"(d) : "f"(s)); return d; }
__device__ __forceinline__ double pinned_copy(double s) { double d; asm volatile("mov.b64 %0, %1;" : "=d"(d) : "d"(s)); return d; }
template <typename T, int N>
__device__ __forceinline__ void pinned_copy(Vec<T, N>& d, const Vec<T, N>& s) {
#pragma unroll
    for (int j = 0; j < N / 2; ++j) d.p[j] = mk2(pinned_copy(s.p[j].x), pinned_copy(s.p[j].y));
    d.t = (N & 1) ? pinned_copy(s.t) : s.t;
}

// store V consecutive elements as one vector (two 16-byte halves for four doubles)
template <typename T, int V>
__device__ __forceinline__ void store_vec(T* dst, const T (&v)[V]) {
    if constexpr (V == 1) dst[0] = v[0];
    else if constexpr (V == 2) *reinterpret_cast<typename PairOf<T>::type*>(dst) = mk2(v[0], v[1]);
    else if constexpr (sizeof(T) == 4) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    else { *reinterpret_cast<double2*>(dst) = make_double2(v[0], v[1]); *reinterpret_cast<double2*>(dst + 2) = make_double2(v[2], v[3]); }
}

// Load LEN contiguous floats (aligned to AL), transform element e with f(e, value) and store the results as
// LEN / V vectors of V elements, vector g at dst + g * stride (the lane-interleaved scratch layout).
template <int LEN, int AL, int V, typename T, typename F>
__device__ __forceinline__ void load_transform_scatter(const float* __restrict__ src, T* dst, uint32_t stride, F&& f) {
    static_assert(LEN % V == 0, "block length must be a whole number of vectors");
    float buf[LEN];
    load_span<LEN, AL>(src, [&](int e, float v) { buf[e] = v; });
#pragma unroll
    for (int g = 0; g < LEN / V; ++g) {
        T out[V];
#pragma unroll
        for (int k = 0; k < V; ++k) out[k] = f(g * V + k, buf[g * V + k]);
        store_vec<T, V>(dst + (size_t)g * stride, out);
    }
}

template <class C>
__global__ void __launch_bounds__(C::BLOCK, C::MINB)
tpp2_kernel(const __grid_constant__ SolveParams prm, const __grid_constant__ typename C::CPack cp) {
    using T = typename C::T;
    using N = Num<T>;
    using P = typename PairOf<T>::type;
    using SP = StaticPack<C::NX, C::NU, C::NH>;
    using VX = Vec<T, C::NX>;
    using VU = Vec<T, C::NU>;
    constexpr int NX = C::NX, NU = C::NU, NH = C::NH, BLOCK = C::BLOCK, SXL = C::SX, SUL = C::SU;
    constexpr int NXP = pad2(NX), NUP = pad2(NU);
    constexpr unsigned FULL = 0xffffffffu;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t pack_bar;
    T* pack = reinterpret_cast<T*>(smem_raw);
    const uint32_t pack_bytes = static_cast<uint32_t>(prm.pack_elems) * sizeof(T);

    // ---- stage the cold family tables into shared memory: one TMA bulk copy per CTA ----
    if (threadIdx.x == 0) {
        mbar_init(&pack_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(&pack_bar, pack_bytes);
        tma_bulk_g2s(pack, prm.pack, pack_bytes, &pack_bar);
    }
    // ---- tensor memory for the TV columns: warp 0 allocates all 512 columns (this CTA owns the SM) ----
    __shared__ uint32_t tmem_base_s;
    if constexpr (C::TM) {
        if (threadIdx.x < 32) tmem_alloc(&tmem_base_s, 512);
        tmem_fence_before_sync();
    }
    __syncthreads();
    if constexpr (C::TM) tmem_fence_after_sync();
    mbar_wait(&pack_bar, 0);

    T* cta_cols = pack + ((prm.pack_elems + 31) & ~31);
    const int tid = threadIdx.x;
    // t = x + g (pre-clamp state slack): shared-memory pair columns, or this thread's tensor-memory columns
    // array number A of the state-sized arrays (TV, GC, GL, SXT) lives in tensor memory iff A < NTM
    const uint32_t tm_thread_base = [&]() -> uint32_t {
        if constexpr (C::TM) {
            const uint32_t w = static_cast<uint32_t>(tid) >> 5;
            return tmem_base_s + ((32u * (w & 3u)) << 16) + (w >> 2) * C::TM_COLS_PER_THREAD;
        } else {
            return 0u;
        }
    }();
    auto make_x = [&](auto a_tag, auto off_tag) {
        constexpr int A = decltype(a_tag)::value, OFF = decltype(off_tag)::value;
        if constexpr (A < C::NTM) return TmemTraj<NX, NH>{tm_thread_base + A * SXL};
        else return SmemTraj<T, NX, NH, OFF, BLOCK>(cta_cols, tid);
    };
    auto TV = make_x(std::integral_constant<int, 0>{}, std::integral_constant<int, C::oTV>{});
    auto GC = make_x(std::integral_constant<int, 1>{}, std::integral_constant<int, C::oGC>{});    // cone duals (state)
    auto GL = make_x(std::integral_constant<int, 2>{}, std::integral_constant<int, C::oGL>{});    // linear duals (state)
    auto SXT = make_x(std::integral_constant<int, 3>{}, std::integral_constant<int, C::oSX>{});   // (vc - gc) + (vl - gl)
    Traj<T, NU, NH - 1, C::oTZ, BLOCK> TZ(cta_cols, tid);    // t = u + y   (pre-clamp input slack)
    Traj<T, NU, NH - 1, C::oD, BLOCK> ND(cta_cols, tid);     // -d of the backward pass
    Col<T, C::oYC, BLOCK> YC(cta_cols, tid);
    Col<T, C::oYL, BLOCK> YL(cta_cols, tid);
    Col<T, C::oSU, BLOCK> SUT(cta_cols, tid);
    T* scr = cta_cols + (size_t)C::oSCR * BLOCK + tid;   // cone scratch column (CONSTR only)

    // Reference terms in a global scratch laid out [element / V][slot][V] (V = 4/2/1 elements per lane and
    // load): coalesced across lanes, one vector load per V elements, re-read every iteration out of L2.
    // Stored pre-combined: SQ = APf - Xref .* Q (state) and SR = -(Uref .* R) (input).
    // All index arithmetic is 32 bit (the scratch has gridDim * BLOCK * (SX + SU) < 2^32 elements).
    const uint32_t slots = gridDim.x * BLOCK;
    const uint32_t slot = blockIdx.x * BLOCK + tid;
    const uint32_t qstride = slots * C::VX, ustride = slots * C::VU;   // elements between consecutive vectors of a lane
    T* const gxr = static_cast<T*>(prm.ref_scratch) + slot * C::VX;
    T* const gur = static_cast<T*>(prm.ref_scratch) + (size_t)SXL * slots + slot * C::VU;
    auto sq_step = [&](int i, VX& dst) {   // fetch the NX state reference terms of time step i
        using V = typename VecOf<T, C::VX>::type;
#pragma unroll
        for (int k = 0; k < NX / C::VX; ++k) {
            const V v = *reinterpret_cast<const V*>(gxr + static_cast<uint32_t>(i * (NX / C::VX) + k) * qstride);
            if constexpr (C::VX == 4) { dst.p[2 * k] = mk2(v.x, v.y); dst.p[2 * k + 1] = mk2(v.z, v.w); }
            else if constexpr (C::VX == 2) { dst.p[k] = mk2(v.x, v.y); }
            else { dst.set(k, v); }
        }
    };
    auto sr_step = [&](int i, VU& dst) {
        using V = typename VecOf<T, C::VU>::type;
#pragma unroll
        for (int k = 0; k < NU / C::VU; ++k) {
            const V v = *reinterpret_cast<const V*>(gur + static_cast<uint32_t>(i * (NU / C::VU) + k) * ustride);
            if constexpr (C::VU == 4) { dst.p[2 * k] = mk2(v.x, v.y); dst.p[2 * k + 1] = mk2(v.z, v.w); }
            else if constexpr (C::VU == 2) { dst.p[k] = mk2(v.x, v.y); }
            else { dst.set(k, v); }
        }
    };
    (void)qstride; (void)ustride;

    const T* cP = pack + SP::Pinf;
    const T* cdP = pack + SP::dPinf;

    const T rho0 = static_cast<T>(prm.rho);
    const T tol_pri = static_cast<T>(prm.abs_pri_tol), tol_dua = static_cast<T>(prm.abs_dua_tol);
    const int max_iter = prm.max_iter, check_every = prm.check_termination;
    const bool soc_x = C::CONSTR && prm.en_state_soc && prm.n_state_cones > 0;
    const bool soc_u = C::CONSTR && prm.en_input_soc && prm.n_input_cones > 0;
    const bool lin_x = C::CONSTR && prm.en_state_linear;
    const bool lin_u = C::CONSTR && prm.en_input_linear;
    const int nsl = prm.nsl, nil = prm.nil;
    const T* cAlx = pack + SP::lin;
    const T* cblx = cAlx + nsl * NX;
    const T* cnrx = cblx + nsl;
    const T* cAlu = cnrx + nsl;
    const T* cblu = cAlu + nil * NU;
    const T* cnru = cblu + nil;
    const bool en_sb = prm.en_state_bound != 0, en_ib = prm.en_input_bound != 0;
    (void)en_sb; (void)en_ib;

    const int lane = tid & 31;
    const int n_items = prm.batch_ptr ? min(*prm.batch_ptr, prm.batch) : prm.batch;   // work items (mixed mode: the marked problems)
    const bool consumer = prm.q_tail != nullptr && prm.q_consume != 0;   // exact-count mode: this launch drains the queue
    const bool producer = prm.q_tail != nullptr && prm.q_consume == 0;   //                   this launch feeds it
    int prob = 0;           // problem owned by this lane
    bool active = false;    // lane holds an unfinished problem
    int last_k = 32;        // iterations of the last problem this lane finished (batched refill)
    bool exhausted = false; // the work counter ran past the batch
    bool pending = false;   // holds a claimed problem (claim) whose inputs have not landed yet (streamed host pipeline)
    int claim = 0, seen = 0, unpub = -1;   // seen: cached arrival watermark; unpub: finished problem not yet counted for its chunk
    int k = 0;              // ADMM iterations done on the current problem
    int wit = 0;            // passes of this warp since it last was idle (warp-uniform): start phase of the adaptive-rho instances
    int next_check = check_every;   // next iteration count at which termination is evaluated (iter % check == 0)
    T res_px = 0, res_dx = 0, res_pu = 0, res_du = 0;   // last evaluated residuals (admm.cpp:257-260)
    // adaptive rho state (cache->rho and the Taylor offset of Kinf/Pinf); *_lc are the values
    // update_linear_cost saw (it runs BEFORE the adaptation inside an iteration)
    T rho = rho0, rho_lc = rho0, dlt = 0, dlt_lc = 0;
    VX x0v, ptv, ptv1;      // x0, the terminal term -(xref_N' Pinf)' and its rho-derivative (ADAPT)
    x0v.fill(T(0)); ptv.fill(T(0)); ptv1.fill(T(0));

    // box bounds of state pair j (elements 2j, 2j+1) / tail element of time step i
    // time row of the shared bound tables: fast-box families have time-invariant bounds (tmpc_capi.cu); TIB instances
    // read row 0 with immediate addresses (LDCU.128, hoistable).  Measured: +10 % cartpole, +5 % adaptive quadrotor,
    // -7 % on the plain quadrotor kernel (the bounds then compete with the matrix coefficients for the uniform
    // registers), so build.py sets it per instance.
    auto bt = [](int i) { return C::TIB ? 0 : i; };
    auto xb_pair = [&](int i, int j, size_t pb, P& lo, P& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NX + 2 * j;
            lo = en_sb ? mk2(static_cast<T>(__ldg(prm.x_min + e)), static_cast<T>(__ldg(prm.x_min + e + 1))) : mk2(-N::inf(), -N::inf());
            hi = en_sb ? mk2(static_cast<T>(__ldg(prm.x_max + e)), static_cast<T>(__ldg(prm.x_max + e + 1))) : mk2(N::inf(), N::inf());
        } else {
            lo = mk2(cp.xmin[bt(i) * NXP + 2 * j], cp.xmin[bt(i) * NXP + 2 * j + 1]); hi = mk2(cp.xmax[bt(i) * NXP + 2 * j], cp.xmax[bt(i) * NXP + 2 * j + 1]);
        }
    };
    auto xb_tail = [&](int i, size_t pb, T& lo, T& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NX + NX - 1;
            lo = en_sb ? static_cast<T>(__ldg(prm.x_min + e)) : -N::inf();
            hi = en_sb ? static_cast<T>(__ldg(prm.x_max + e)) : N::inf();
        } else { lo = cp.xmin[bt(i) * NXP + NX - 1]; hi = cp.xmax[bt(i) * NXP + NX - 1]; }
    };
    auto ub_pair = [&](int i, int j, size_t pb, P& lo, P& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NU + 2 * j;
            lo = en_ib ? mk2(static_cast<T>(__ldg(prm.u_min + e)), static_cast<T>(__ldg(prm.u_min + e + 1))) : mk2(-N::inf(), -N::inf());
            hi = en_ib ? mk2(static_cast<T>(__ldg(prm.u_max + e)), static_cast<T>(__ldg(prm.u_max + e + 1))) : mk2(N::inf(), N::inf());
        } else {
            lo = mk2(cp.umin[bt(i) * NUP + 2 * j], cp.umin[bt(i) * NUP + 2 * j + 1]); hi = mk2(cp.umax[bt(i) * NUP + 2 * j], cp.umax[bt(i) * NUP + 2 * j + 1]);
        }
    };
    auto ub_tail = [&](int i, size_t pb, T& lo, T& hi) {
        if constexpr (C::PPB) {
            const size_t e = pb + (size_t)i * NU + NU - 1;
            lo = en_ib ? static_cast<T>(__ldg(prm.u_min + e)) : -N::inf();
            hi = en_ib ? static_cast<T>(__ldg(prm.u_max + e)) : N::inf();
        } else { lo = cp.umin[bt(i) * NUP + NU - 1]; hi = cp.umax[bt(i) * NUP + NU - 1]; }
    };

    for (;;) {
        // ------------------------------------------------------------------ refill idle lanes
        {
            publish_done(prm, unpub);
            const bool want = !active && !exhausted && !pending;
            unsigned mw = __ballot_sync(FULL, want);
            // Adaptive rho: problems start only on every 5th pass of the warp.  The adaptation (rho_benchmark.cpp:146-250 in
            // block form: ~96 extra FFMA2 per time step) is due at the problem's own iterations 5, 10, ... (admm.cpp:339); with
            // lanes at arbitrary phases some lane is due on practically every pass and the whole warp pays for it every time,
            // with aligned phases it pays on one pass in five.  A lane waits 2.5 passes on average, about what the batched refill
            // makes it wait anyway.
            if (!__any_sync(FULL, active)) wit = 0;     // nobody to stay aligned with
            const bool phase_ok = !(C::ADAPT && prm.adaptive_rho) || (wit % 5 == 0);
            if (!phase_ok) mw = 0;
            // batched refill (SolveParams::refill_min; the model behind the adaptive threshold is spelled out in tmpc_tpp3.cuh)
            if (mw && __any_sync(FULL, active) && !(C::ADAPT && prm.adaptive_rho)) {
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
                    if (consumer) {
                        pending = true;      // claim is a queue ticket: resolved below, once the producer has filled it
                    } else if (claim >= n_items) {
                        exhausted = true;
                        prob = 0;   // keeps the (unused) per-problem reads of an idle lane in range
                    } else {
                        if (prm.index_list) claim = __ldg(prm.index_list + claim);
                        pending = true;
                    }
                }
            }
            // a claimed problem starts once its inputs have landed (always, unless the host streams the batch in)
            bool mine;
            if (consumer) {
                bool none = false;
                int qp = 0;
                mine = pending && queue_take(prm, claim, qp, none) && phase_ok;
                if (mine) claim = qp;
                if (pending && none) { pending = false; exhausted = true; prob = 0; }
            } else {
                mine = phase_ok && pending && problem_ready(prm, claim, seen);
            }
            const unsigned m = __ballot_sync(FULL, mine);
            if (m) {
                if (mine) {
                    {
                        prob = claim;
                        pending = false;
                        active = true;
                        k = 0;
                        next_check = check_every;
                        res_px = res_dx = res_pu = res_du = 0;
                        rho = rho_lc = rho0; dlt = dlt_lc = 0;
                        if constexpr (C::REFS) {
                            // pull the whole problem towards L2 first: the blocks below then cost one DRAM round trip in total
                            if (prm.Xref) {
                                const char* s = reinterpret_cast<const char*>(prm.Xref + (size_t)prob * SXL);
#pragma unroll
                                for (int b = 0; b <= (SXL * 4 + 127) / 128; ++b) prefetch_l2(s + (b * 128 < SXL * 4 ? b * 128 : SXL * 4 - 4));
                            }
                            if (prm.Uref) {
                                const char* s = reinterpret_cast<const char*>(prm.Uref + (size_t)prob * SUL);
#pragma unroll
                                for (int b = 0; b <= (SUL * 4 + 127) / 128; ++b) prefetch_l2(s + (b * 128 < SUL * 4 ? b * 128 : SUL * 4 - 4));
                            }
                        }
                        load_span<NX, vec_width(NX, NX)>(prm.x0 + (size_t)prob * NX, [&](int i, float v) { x0v.set(i, static_cast<T>(v)); });
                        // Xref -> SQ = APf - Xref .* Q (work->Q = diag(Q)+rho, admm.cpp:218) and the terminal
                        // term PT = -(xref_N' Pinf)' (admm.cpp:238)
                        if constexpr (C::REFS) {
                            constexpr int GX = steps_per_block(NH, NX, 64), GU = steps_per_block(NH - 1, NU, 64);
                            T xr_last[NX];
#pragma unroll
                            for (int r = 0; r < NX; ++r) xr_last[r] = 0;
                            if (prm.Xref) {
                                const float* src = prm.Xref + (size_t)prob * SXL;
#pragma unroll 1
                                for (int b = 0; b < NH / GX; ++b)
                                    load_transform_scatter<GX * NX, vec_width(SXL, GX * NX), C::VX>(
                                        src + b * GX * NX, gxr + static_cast<uint32_t>(b * (GX * NX / C::VX)) * qstride, qstride, [&](int e, float v) {
                                            const int r = e % NX;
                                            if (e / NX == GX - 1) xr_last[r] = static_cast<T>(v);   // after the last block: xref_N
                                            return (C::AFF ? cp.APf[r] : T(0)) - static_cast<T>(v) * cp.Qd[r];
                                        });
                            } else {
#pragma unroll 1
                                for (int i = 0; i < NH; ++i) {
#pragma unroll
                                    for (int g = 0; g < NX / C::VX; ++g) {
                                        T out[C::VX];
#pragma unroll
                                        for (int k = 0; k < C::VX; ++k) out[k] = C::AFF ? cp.APf[g * C::VX + k] : T(0);
                                        store_vec<T, C::VX>(gxr + static_cast<uint32_t>(i * (NX / C::VX) + g) * qstride, out);
                                    }
                                }
                            }
                            {   // PT = -(xref_N' Pinf)' as row pairs of Pinf' (Pinf is row-major in the staged pack)
                                VX acc, acc1;
                                acc.fill(T(0)); acc1.fill(T(0));
#pragma unroll
                                for (int r = 0; r < NX; ++r) {
                                    const T nxr = -xr_last[r];
#pragma unroll
                                    for (int j = 0; j < NX / 2; ++j) {
                                        acc.p[j] = fmas(mk2(cP[r * NX + 2 * j], cP[r * NX + 2 * j + 1]), nxr, acc.p[j]);
                                        if constexpr (C::ADAPT) acc1.p[j] = fmas(mk2(cdP[r * NX + 2 * j], cdP[r * NX + 2 * j + 1]), nxr, acc1.p[j]);
                                    }
                                    if constexpr (NX & 1) {
                                        acc.t = fmas(cP[r * NX + NX - 1], nxr, acc.t);
                                        if constexpr (C::ADAPT) acc1.t = fmas(cdP[r * NX + NX - 1], nxr, acc1.t);
                                    }
                                }
                                ptv = acc;
                                if constexpr (C::ADAPT) ptv1 = acc1;
                            }
                            if (prm.Uref) {
                                const float* src = prm.Uref + (size_t)prob * SUL;
#pragma unroll 1
                                for (int b = 0; b < (NH - 1) / GU; ++b)
                                    load_transform_scatter<GU * NU, vec_width(SUL, GU * NU), C::VU>(
                                        src + b * GU * NU, gur + static_cast<uint32_t>(b * (GU * NU / C::VU)) * ustride, ustride,
                                        [&](int e, float v) { return -(static_cast<T>(v) * cp.Rd[e % NU]); });
                            } else {
#pragma unroll 1
                                for (int i = 0; i < NH - 1; ++i) {
#pragma unroll
                                    for (int g = 0; g < NU / C::VU; ++g) {
                                        T out[C::VU];
#pragma unroll
                                        for (int k = 0; k < C::VU; ++k) out[k] = T(0);
                                        store_vec<T, C::VU>(gur + static_cast<uint32_t>(i * (NU / C::VU) + g) * ustride, out);
                                    }
                                }
                            }
                        }
                        // cold workspace (tiny_api.cpp:68-105): duals and slacks zero, d = d0 (TV: below, warp-wide)
#pragma unroll 1
                        for (int i = 0; i < NH - 1; ++i) {
#pragma unroll
                            for (int j = 0; j < NU / 2; ++j) {
                                TZ.setp(i, j, mk2(T(0), T(0)));
                                ND.setp(i, j, mk2(-pack[SP::d0 + i * NU + 2 * j], -pack[SP::d0 + i * NU + 2 * j + 1]));
                            }
                            if constexpr (NU & 1) { TZ.sett(i, T(0)); ND.sett(i, -pack[SP::d0 + i * NU + NU - 1]); }
                        }
                        if constexpr (C::CONSTR) {
#pragma unroll 4
                            for (int e = 0; e < SUL; ++e) { YC.set(e, T(0)); YL.set(e, T(0)); SUT.set(e, T(0)); }
                        }
                    }
                }
                TV.reset(mine);   // warp-collective when TV lives in tensor memory
                if constexpr (C::CONSTR) { GC.reset(mine); GL.reset(mine); }   // SXT is written before it is read
            }
            if (!__any_sync(FULL, active)) {
                if (!__any_sync(FULL, pending)) break;
                __nanosleep(256);   // the whole warp is waiting for the copy engine
                continue;
            }
        }

        // ------------------------------------------------- forward rollout + slack + dual + residuals
        T rpx = 0, rdx = 0, rpu = 0, rdu = 0;
        // adaptive-rho accumulators (rho_benchmark.cpp:146-173); only evaluated on sweeps where some
        // lane of the warp is at an adaptation iteration (i > 0 && i % 5 == 0, admm.cpp:339)
        const bool do_adapt = C::ADAPT && prm.adaptive_rho && __any_sync(FULL, active && k > 0 && k % 5 == 0);
        T a_pri = 0, a_prin = 0, a_dua = 0, a_duan = 0;
        const bool first = (k == 0);   // cold start: v = 0, g = 0 whatever the bounds are
        VX x = x0v;
        VX xprev, gprev; VU uprev, yprev;   // ADAPT: lagged column for the A'g terms
        xprev.fill(T(0)); gprev.fill(T(0)); uprev.fill(T(0)); yprev.fill(T(0));
        const size_t pbx = (size_t)prob * SXL, pbu = (size_t)prob * SUL;

        // one trajectory element (pair or scalar tail): vnew = clamp(x + g), g += x - vnew (admm.cpp:85,92,184)
        auto slack_dual = [&](auto told, auto xv, auto lo, auto hi, T& rp, T& rd, auto& tnew, auto& vn, auto& gn) {
            auto vo = clampv(told, lo, hi);
            auto g = subv(told, vo);
            if constexpr (!C::FB) { if (first) { vo = zero_like(vo); g = zero_like(g); } }   // FB: 0 is inside the box, clamp(0) = 0 already
            tnew = addv(xv, g);
            vn = clampv(tnew, lo, hi);
            rp = amaxv(rp, subv(xv, vn));
            rd = amaxv(rd, subv(vo, vn));
            gn = subv(tnew, vn);
        };

#pragma unroll 1
        for (int i = 0; i < NH; ++i) {
            const int zf = C::OPQ ? opaque_zero4() : 0;
            // ---- state column i
            VX gnew, vnx, tvo, tvn;
            TV.load(i, tvo);
#pragma unroll
            for (int j = 0; j < NX / 2; ++j) {
                P lo, hi;
                xb_pair(i, j, pbx, lo, hi);
                slack_dual(tvo.p[j], x.p[j], lo, hi, rpx, rdx, tvn.p[j], vnx.p[j], gnew.p[j]);
            }
            if constexpr (NX & 1) {
                T lo, hi;
                xb_tail(i, pbx, lo, hi);
                slack_dual(tvo.t, x.t, lo, hi, rpx, rdx, tvn.t, vnx.t, gnew.t);
            }
            TV.store(i, tvn);
            if constexpr (C::ADAPT) {
                if (do_adapt && i > 0) {   // dynamics rows of A_matrix: (A x + B u - x_next) - vnew_next = -f - vnew
#pragma unroll
                    for (int r = 0; r < NX; ++r) {
                        const T vn = vnx.get(r);
                        const T fr = C::AFF ? cp.f[r] : T(0);
                        a_pri = N::max(a_pri, N::abs(fr + vn));
                        a_prin = N::max(a_prin, N::max(N::abs(vn), N::abs(fr)));
                    }
                }
            }
            if constexpr (C::CONSTR) {
                VX extra;
                extra.fill(T(0));
                if (soc_x) {   // admm.cpp:103,112-122,191
                    VX gcv;
                    GC.load(i, gcv);
#pragma unroll
                    for (int r = 0; r < NX; ++r) scr[r * BLOCK] = x.get(r) + gcv.get(r);
                    for (int c = 0; c < prm.n_state_cones; ++c) project_soc_col2<T, BLOCK>(scr, prm.Acx[c], prm.qcx[c], prm.cx[c]);
#pragma unroll
                    for (int r = 0; r < NX; ++r) {
                        const T vc = scr[r * BLOCK];
                        const T gcn = (gcv.get(r) + x.get(r)) - vc;
                        gcv.set(r, gcn);
                        extra.set(r, extra.get(r) + (vc - gcn));
                    }
                    GC.store(i, gcv);
                }
                if (lin_x) {   // admm.cpp:139,148-159,201
                    T vl[NX];
                    VX glv;
                    GL.load(i, glv);
#pragma unroll
                    for (int r = 0; r < NX; ++r) vl[r] = x.get(r) + glv.get(r);
                    for (int c = 0; c < nsl; ++c) {
                        T val = 0;
#pragma unroll
                        for (int r = 0; r < NX; ++r) val = N::fma(cAlx[c * NX + r], vl[r], val);
                        if (val > cblx[c]) {
                            const T dist = (val - cblx[c]) / cnrx[c];
#pragma unroll
                            for (int r = 0; r < NX; ++r) vl[r] = vl[r] - dist * cAlx[c * NX + r];
                        }
                    }
#pragma unroll
                    for (int r = 0; r < NX; ++r) {
                        const T gln = (glv.get(r) + x.get(r)) - vl[r];
                        glv.set(r, gln);
                        extra.set(r, extra.get(r) + (vl[r] - gln));
                    }
                    GL.store(i, glv);
                }
                SXT.store(i, extra);
            }
            if constexpr (C::ADAPT) {
                // dual residual blocks of column i-1 need g_i (post update): x-block A'g_i - g_{i-1}, u-block y_{i-1} + B'g_i
                if (do_adapt && i > 0) {
                    VX atx; atx.fill(T(0));
                    mv_acc<NX, NX>(cp.AT, zf, gnew, atx);
                    VU atu = yprev;
                    mv_acc<NU, NX>(cp.BT, zf, gnew, atu);
#pragma unroll
                    for (int c = 0; c < NX; ++c) {
                        T aty = atx.get(c);
                        if (i > 1) aty -= gprev.get(c);
                        const T qx = cp.Qd[c] * xprev.get(c);   // Px = qv = Q .* x for columns < N-1
                        a_dua = N::max(a_dua, N::abs(qx + qx + aty));
                        a_duan = N::max(a_duan, N::max(N::abs(qx), N::abs(aty)));
                    }
#pragma unroll
                    for (int a = 0; a < NU; ++a) {
                        const T aty = atu.get(a);
                        const T ru = cp.Rd[a] * uprev.get(a);
                        a_dua = N::max(a_dua, N::abs(ru + ru + aty));
                        a_duan = N::max(a_duan, N::max(N::abs(ru), N::abs(aty)));
                    }
                }
                if (do_adapt && i == NH - 1) {   // last state block: Px = Pinf x_N, qv = Q .* x_N, ATy = -g_N
#pragma unroll
                    for (int r = 0; r < NX; ++r) {
                        T px = 0;
#pragma unroll
                        for (int c = 0; c < NX; ++c) px = N::fma(N::fma(dlt, cdP[r * NX + c], cP[r * NX + c]), x.get(c), px);
                        const T qx = cp.Qd[r] * x.get(r);
                        const T aty = -gnew.get(r);
                        a_dua = N::max(a_dua, N::abs(px + qx + aty));
                        a_duan = N::max(a_duan, N::max(N::max(N::abs(px), N::abs(qx)), N::abs(aty)));
                    }
                }
            }
            if (i < NH - 1) {
                // ---- u_i = -Kinf x_i - d_i (admm.cpp:29); Kinf = Kinf0 + dlt * dKinf under adaptive rho
                VU u;
                if constexpr (C::ADAPT) {
                    VU a0, a1; a0.fill(T(0)); a1.fill(T(0));
                    mv_acc<NU, NX>(cp.NK, zf, x, a0);
                    mv_acc<NU, NX>(cp.NdK, zf, x, a1);
                    VU nd; ND.load(i, nd);
#pragma unroll
                    for (int j = 0; j < NU / 2; ++j) u.p[j] = addv(fmas(a1.p[j], dlt, a0.p[j]), nd.p[j]);
                    if constexpr (NU & 1) u.t = addv(fmas(a1.t, dlt, a0.t), nd.t);
                } else {
                    VU a0; a0.fill(T(0));
                    mv_acc<NU, NX>(cp.NK, zf, x, a0);
                    VU nd; ND.load(i, nd);
#pragma unroll
                    for (int j = 0; j < NU / 2; ++j) u.p[j] = addv(a0.p[j], nd.p[j]);
                    if constexpr (NU & 1) u.t = addv(a0.t, nd.t);
                }
                // ---- input column i: znew = clamp(u + y), y += u - znew (admm.cpp:88,97,187)
                VU ynew, znu;
#pragma unroll
                for (int j = 0; j < NU / 2; ++j) {
                    P lo, hi, tn;
                    ub_pair(i, j, pbu, lo, hi);
                    slack_dual(TZ.getp(i, j), u.p[j], lo, hi, rpu, rdu, tn, znu.p[j], ynew.p[j]);
                    TZ.setp(i, j, tn);
                }
                if constexpr (NU & 1) {
                    T lo, hi, tn;
                    ub_tail(i, pbu, lo, hi);
                    slack_dual(TZ.gett(i), u.t, lo, hi, rpu, rdu, tn, znu.t, ynew.t);
                    TZ.sett(i, tn);
                }
                if constexpr (C::ADAPT) {
                    if (do_adapt) {
#pragma unroll
                        for (int a = 0; a < NU; ++a) a_prin = N::max(a_prin, N::max(N::abs(u.get(a)), N::abs(znu.get(a))));
                    }
                }
                if constexpr (C::CONSTR) {
                    T extra[NU];
#pragma unroll
                    for (int a = 0; a < NU; ++a) extra[a] = 0;
                    if (soc_u) {
#pragma unroll
                        for (int a = 0; a < NU; ++a) scr[a * BLOCK] = u.get(a) + YC.get(i * NU + a);
                        for (int c = 0; c < prm.n_input_cones; ++c) project_soc_col2<T, BLOCK>(scr, prm.Acu[c], prm.qcu[c], prm.cu[c]);
#pragma unroll
                        for (int a = 0; a < NU; ++a) {
                            const T zc = scr[a * BLOCK];
                            const T ycn = (YC.get(i * NU + a) + u.get(a)) - zc;
                            YC.set(i * NU + a, ycn);
                            extra[a] += zc - ycn;
                        }
                    }
                    if (lin_u) {
                        T zl[NU];
#pragma unroll
                        for (int a = 0; a < NU; ++a) zl[a] = u.get(a) + YL.get(i * NU + a);
                        for (int c = 0; c < nil; ++c) {
                            T val = 0;
#pragma unroll
                            for (int a = 0; a < NU; ++a) val = N::fma(cAlu[c * NU + a], zl[a], val);
                            if (val > cblu[c]) {
                                const T dist = (val - cblu[c]) / cnru[c];
#pragma unroll
                                for (int a = 0; a < NU; ++a) zl[a] = zl[a] - dist * cAlu[c * NU + a];
                            }
                        }
#pragma unroll
                        for (int a = 0; a < NU; ++a) {
                            const T yln = (YL.get(i * NU + a) + u.get(a)) - zl[a];
                            YL.set(i * NU + a, yln);
                            extra[a] += zl[a] - yln;
                        }
                    }
#pragma unroll
                    for (int a = 0; a < NU; ++a) SUT.set(i * NU + a, extra[a]);
                }
                // ---- x_{i+1} = A x_i + B u_i + f (admm.cpp:30)
                VX xn;
                if constexpr (C::AFF) {
#pragma unroll
                    for (int j = 0; j < NX / 2; ++j) xn.p[j] = mk2(cp.f[2 * j], cp.f[2 * j + 1]);
                    if constexpr (NX & 1) xn.t = cp.f[NX - 1];
                } else {
                    xn.fill(T(0));
                }
                mv_acc<NX, NX>(cp.A, zf, x, xn);
                mv_acc<NX, NU>(cp.B, zf, u, xn);
                if constexpr (C::ADAPT) { xprev = x; gprev = gnew; uprev = u; yprev = ynew; }
                x = xn;
            }
        }
        TV.stores_done();
        k += 1;   // work->iter += 1 (admm.cpp:328)
        wit += 1;

        // ------------------------------------------------- adaptive rho (admm.cpp:331-357), i = k-1
        rho_lc = rho; dlt_lc = dlt;   // update_linear_cost of this iteration ran with the pre-adaptation cache
        if constexpr (C::ADAPT) {
            if (do_adapt && (k - 1) > 0 && (k - 1) % 5 == 0) {
                a_pri = N::max(a_pri, rpu);                       // input rows: u - znew
                const T eps = T(1e-10);
                const T npri = a_pri / (a_prin + eps), ndua = a_dua / (a_duan + eps);
                T nr = rho * N::sqrt(npri / (ndua + eps));
                if (prm.rho_clip) nr = N::min(N::max(nr, static_cast<T>(prm.rho_min)), static_cast<T>(prm.rho_max));
                dlt += nr - rho;      // Kinf, Pinf += (rho' - rho) * d/drho (rho_benchmark.cpp:199-212)
                rho = nr;
            }
        }

        // ------------------------------------------------- termination (admm.cpp:253-271, 364-388)
        bool finish = false;
        int st = 11;
        if (k == next_check) {   // iter % check_termination == 0
            next_check += check_every;
            res_px = rpx; res_dx = rdx * rho; res_pu = rpu; res_du = rdu * rho;
            if (res_px < tol_pri && res_pu < tol_pri && res_dx < tol_dua && res_du < tol_dua) { finish = true; st = 1; }
            if constexpr (sizeof(T) == 4) {
                // Mixed mode: this decision is a threshold crossing on values carrying fp32 rounding noise.  If the largest
                // residual/tolerance ratio lies inside [1 - band, 1 + band] the fp64 arithmetic of the reference may decide
                // the other way: stop here and hand the problem to the fp64 pass.
                if (prm.amb_band > 0.f) {
                    const T up = T(1) + prm.amb_band, dn = T(1) - prm.amb_band;
                    const bool below_up = res_px < tol_pri * up && res_pu < tol_pri * up && res_dx < tol_dua * up && res_du < tol_dua * up;
                    const bool below_dn = res_px < tol_pri * dn && res_pu < tol_pri * dn && res_dx < tol_dua * dn && res_du < tol_dua * dn;
                    if (below_up && !below_dn) { finish = true; st = kAmbiguousBit | 11; }
                }
            }
        }
        if (k >= max_iter) finish = true;
        bool fin = active && finish;
        if (producer) {   // undecidable problems go to the fp64 consumer: no result, no completion count from this lane
            const bool amb = fin && (st & kAmbiguousBit);
            queue_push(prm, amb, prob, lane);
            if (amb) { fin = false; active = false; last_k = k; }
        }
        if (__any_sync(FULL, fin)) {
            // solution = (vnew, znew) = clamp of the stored pre-clamp values (the TV read is warp-collective)
#pragma unroll 1
            for (int i = 0; i < NH; ++i) {
                VX v;
                TV.load(i, v);
                if (fin) {
#pragma unroll
                    for (int j = 0; j < NX / 2; ++j) { P lo, hi; xb_pair(i, j, pbx, lo, hi); v.p[j] = clampv(v.p[j], lo, hi); }
                    if constexpr (NX & 1) { T lo, hi; xb_tail(i, pbx, lo, hi); v.t = clampv(v.t, lo, hi); }
                    store_span<NX, vec_width(SXL, NX)>(prm.x + pbx + i * NX, [&](int r) { return static_cast<float>(v.get(r)); });
                }
            }
        }
        if (fin) {
#pragma unroll 1
            for (int i = 0; i < NH - 1; ++i) {
                VU z;
#pragma unroll
                for (int j = 0; j < NU / 2; ++j) { P lo, hi; ub_pair(i, j, pbu, lo, hi); z.p[j] = clampv(TZ.getp(i, j), lo, hi); }
                if constexpr (NU & 1) { T lo, hi; ub_tail(i, pbu, lo, hi); z.t = clampv(TZ.gett(i), lo, hi); }
                store_span<NU, vec_width(SUL, NU)>(prm.u + pbu + i * NU, [&](int a) { return static_cast<float>(z.get(a)); });
            }
            prm.iter[prob] = k;
            prm.status[prob] = st;
            if (prm.residuals) {
                float4 rr = make_float4(static_cast<float>(res_px), static_cast<float>(res_dx), static_cast<float>(res_pu), static_cast<float>(res_du));
                *reinterpret_cast<float4*>(prm.residuals + 4 * (size_t)prob) = rr;
            }
            if (prm.rho_out) prm.rho_out[prob] = static_cast<float>(rho);
            if (prm.done_counters) unpub = prob;
            active = false;
            last_k = k;
        }
        if (!__any_sync(FULL, active)) continue;   // whole warp idle: go refill (or exit) without a backward sweep

        // ------------------------------------------------- backward Riccati sweep for the next iteration
        // q, r, p_N of update_linear_cost (admm.cpp:214-247) are formed on the fly with the rho / Pinf
        // that update_linear_cost saw; Kinf' uses the current (possibly adapted) Kinf.
        // v - g = 2 clamp(t) - t for the box slack/dual pair.
        const T nrho = -rho_lc;
        // reference terms of step i are fetched one step ahead (they live in L2)
        VX sq_nx; VU sr_nx;
        if constexpr (C::AFF) {
#pragma unroll
            for (int j = 0; j < NX / 2; ++j) sq_nx.p[j] = mk2(cp.APf[2 * j], cp.APf[2 * j + 1]);
            if constexpr (NX & 1) sq_nx.t = cp.APf[NX - 1];
        } else {
            sq_nx.fill(T(0));
        }
        sr_nx.fill(T(0));
        if constexpr (C::REFS) { sq_step(NH - 2, sq_nx); sr_step(NH - 2, sr_nx); }

        // box slack minus dual of one element: w = 2 clamp(t) - t (+ cone / linear terms)
        auto w_of = [&](auto t, auto lo, auto hi) { return twice_minus(clampv(t, lo, hi), t); };

        VX p, tvv, sxv;
        {   // p_N = -(xref_N' Pinf)' - rho (vnew_N - g_N) ...  (admm.cpp:238-246)
            TV.load(NH - 1, tvv);
            if constexpr (C::CONSTR) SXT.load(NH - 1, sxv);
#pragma unroll
            for (int j = 0; j < NX / 2; ++j) {
                P lo, hi;
                xb_pair(NH - 1, j, pbx, lo, hi);
                P w = w_of(tvv.p[j], lo, hi);
                if constexpr (C::CONSTR) w = addv(w, sxv.p[j]);
                P pt = ptv.p[j];
                if constexpr (C::ADAPT) pt = fmas(ptv1.p[j], dlt_lc, pt);
                p.p[j] = fmas(w, nrho, pt);
            }
            if constexpr (NX & 1) {
                T lo, hi;
                xb_tail(NH - 1, pbx, lo, hi);
                T w = w_of(tvv.t, lo, hi);
                if constexpr (C::CONSTR) w += sxv.t;
                T pt = ptv.t;
                if constexpr (C::ADAPT) pt = fmas(ptv1.t, dlt_lc, pt);
                p.t = fmas(w, nrho, pt);
            }
        }
#pragma unroll 1
        for (int i = NH - 2; i >= 0; --i) {
            const int zb = C::OPQ ? opaque_zero4() : 0;
            TV.load(i, tvv);
            if constexpr (C::CONSTR) SXT.load(i, sxv);
            // The terms of step i move to their own registers with copies the compiler cannot remove, and the fetch
            // for step i-1 is issued at once: a whole step of distance to the L2.  (With plain copies the register
            // allocator coalesces both buffers and sinks the loads to the end of the loop body: distance zero, 8 % of
            // all stall samples on the first consumer.)
            VX sq_cur; VU sr_cur;
            if constexpr (C::REFS) {
                pinned_copy(sq_cur, sq_nx); pinned_copy(sr_cur, sr_nx);
                const int inx = i > 0 ? i - 1 : 0;   // no branch: a conditional fetch block gets laid out at the loop end
                sq_step(inx, sq_nx); sr_step(inx, sr_nx);
            } else {
                sq_cur = sq_nx; sr_cur = sr_nx;
            }
            // r_i = -(Uref .* R) - rho (znew - y) ...  (admm.cpp:227-236)
            VU rr;
#pragma unroll
            for (int j = 0; j < NU / 2; ++j) {
                P lo, hi;
                ub_pair(i, j, pbu, lo, hi);
                P w = w_of(TZ.getp(i, j), lo, hi);
                if constexpr (C::CONSTR) w = addv(w, mk2(SUT.get(i * NU + 2 * j), SUT.get(i * NU + 2 * j + 1)));
                rr.p[j] = fmas(w, nrho, sr_cur.p[j]);
            }
            if constexpr (NU & 1) {
                T lo, hi;
                ub_tail(i, pbu, lo, hi);
                T w = w_of(TZ.gett(i), lo, hi);
                if constexpr (C::CONSTR) w += SUT.get(i * NU + NU - 1);
                rr.t = fmas(w, nrho, sr_cur.t);
            }
            // d_i = Quu_inv (B' p + r + BPf)   (admm.cpp:17)
            VU t = rr;
            if constexpr (C::AFF) {
#pragma unroll
                for (int j = 0; j < NU / 2; ++j) t.p[j] = addv(rr.p[j], mk2(cp.BPf[2 * j], cp.BPf[2 * j + 1]));
                if constexpr (NU & 1) t.t = rr.t + cp.BPf[NU - 1];
            }
            mv_acc<NU, NX>(cp.BT, zb, p, t);
            VU d; d.fill(T(0));
            mv_acc<NU, NU>(cp.Quu, zb, t, d);
            {
                VU nd;
#pragma unroll
                for (int j = 0; j < NU / 2; ++j) nd.p[j] = negv(d.p[j]);
                if constexpr (NU & 1) nd.t = -d.t;
                ND.store(i, nd);
            }
            // p_i = q_i + AmBKt p - Kinf' r + APf   (admm.cpp:18), q_i = -(Xref .* Q) - rho (vnew - g) ...
            VX pn;
#pragma unroll
            for (int j = 0; j < NX / 2; ++j) {
                P lo, hi;
                xb_pair(i, j, pbx, lo, hi);
                P w = w_of(tvv.p[j], lo, hi);
                if constexpr (C::CONSTR) w = addv(w, sxv.p[j]);
                pn.p[j] = fmas(w, nrho, sq_cur.p[j]);
            }
            if constexpr (NX & 1) {
                T lo, hi;
                xb_tail(i, pbx, lo, hi);
                T w = w_of(tvv.t, lo, hi);
                if constexpr (C::CONSTR) w += sxv.t;
                pn.t = fmas(w, nrho, sq_cur.t);
            }
            mv_acc<NX, NX>(cp.AK, zb, p, pn);
            mv_acc<NX, NU>(cp.NKT, zb, rr, pn);
            if constexpr (C::ADAPT) {
                VX ak; ak.fill(T(0));
                mv_acc<NX, NU>(cp.NdKT, zb, rr, ak);
#pragma unroll
                for (int j = 0; j < NX / 2; ++j) pn.p[j] = fmas(ak.p[j], dlt, pn.p[j]);
                if constexpr (NX & 1) pn.t = fmas(ak.t, dlt, pn.t);
            }
            p = pn;
        }
    }
    if (producer) {
        __syncthreads();
        if (threadIdx.x == 0) queue_producer_exit(prm);
    }
    if constexpr (C::TM) {   // every warp is done with its columns: give the tensor memory back
        tmem_fence_before_sync();
        __syncthreads();
        if (threadIdx.x < 32) tmem_dealloc(tmem_base_s, 512);
    }
}

template <class C>
inline size_t tpp2_smem_bytes(int pack_elems) {
    return ((size_t)((pack_elems + 31) & ~31) + (size_t)C::COLS * C::BLOCK) * sizeof(typename C::T);
}

}  // namespace tmpc
