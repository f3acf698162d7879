// tmpc_capi.cu -- implementation of the C ABI declared in include/tinympc_b200.h.
//
// Host side of the drop-in boundary: validates and packs the family data a TinySolver holds
// (reference types.hpp:43-187), shards batches contiguously by problem index over the devices of
// one box (no collective: problems are independent), moves host buffers through pinned-speed
// async copies in a chunked H2D -> kernel -> D2H pipeline, and launches the sm_100a kernels.
// There is no CPU fallback anywhere in this file: without a device every call fails.
#include "../../include/tinympc_b200.h"

#include <cuda.h>            // types of the two stream memory operations only; the entry points come from cudaGetDriverEntryPoint
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "tmpc_common.h"
#include "tmpc_devptr.h"
#include "tmpc_registry.h"
#include "tmpc_sparse_a.h"
#include "tmpc_wpp.h"

using namespace tmpc;

namespace {

constexpr int kFeatBox = 0, kFeatConstr = 1, kFeatAdapt = 2;
constexpr int kMaxChunks = 64;
constexpr int kStreams = 3;
constexpr int kLatencyVariant = 9;        // registry variant of the plain-layout (latency) instances, see enqueue()
constexpr int kMaxStreamChunks = 256;    // streamed pipeline: [0] work counter, [1] arrival watermark, [2 + c] finished problems of chunk c

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct DeviceCtx {
    int device = 0;
    int sm_count = 0;
    void* pack32 = nullptr;
    void* pack64 = nullptr;
    int* stream_ctl = nullptr;          // 2 + kMaxStreamChunks ints (see kMaxStreamChunks)
    cudaEvent_t ev_ctl = nullptr;
    int* counters = nullptr;            // 3 * kMaxChunks ints: work counters of the first pass, of the fp64 re-solve pass, marked-problem counts
    cudaStream_t streams[kStreams] = {nullptr, nullptr, nullptr};
    cudaEvent_t k0[kMaxChunks], k1[kMaxChunks];
    bool events = false;
    DevBuf x0, Xref, Uref, xmin, xmax, umin, umax, x, u, iter, status, res, rho, xrc, u0;
    DevBuf exp_xref[kStreams + 1], exp_x[kStreams + 1], exp_u[kStreams + 1];   // compact I/O: device-side expansion / full trajectories per slot
    DevBuf ref_scratch[kStreams + 1];   // REFS_L2 kernels: per-slot reference terms
    DevBuf wpp_scratch[kStreams + 1];   // warp-per-problem workspaces (one per pipeline stream + the device/workspace entry)
    DevBuf ref_scratch64[kStreams + 1]; // mixed mode: reference terms of the fp64 re-solve pass
    DevBuf marked[kStreams + 1];        // mixed mode: indices of the problems the fp32 pass marked ambiguous (two-pass form) / the queue
    DevBuf order_buf;                   // claim order of the device-resident entry: 256 histogram words, n list words, n bucket bytes
    DevBuf models[14];                  // model batches through the host entry: one buffer per field of tinympc_cuda_models (model_fields)
    cudaEvent_t ev_pass = nullptr, ev_copied = nullptr;   // compact streamed pipeline: end of the first pass / of the early result copies
    // exact-count mode, concurrent form: per slot {q_tail, producer CTAs done, consumer ticket counter, pad}
    int* qctl = nullptr;                // 4 * kMaxChunks ints, indexed like the work counters (chunk index; the last one = device entry)
    cudaStream_t fix_stream[kStreams + 1] = {nullptr, nullptr, nullptr, nullptr};   // the fp64 consumer launches
    cudaEvent_t ev_fork[kStreams + 1] = {nullptr, nullptr, nullptr, nullptr}, ev_join[kStreams + 1] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_p0 = nullptr, ev_p1 = nullptr, ev_p2 = nullptr;   // option "pass_timing": around the fp32 pass and the fp64 pass of a device-resident exact-count solve
    bool pass_timed = false;
};

struct Family {
    bool set = false;
    int nx = 0, nu = 0, N = 0;
    int feat = kFeatBox;
    bool shared_bounds_ok = false;     // every enabled bound has shared arrays
    bool fastbox = false;              // shared bounds are constant over the horizon and contain 0
    bool affine = false;               // fdyn (hence APf, BPf) is not identically zero
    std::vector<unsigned> a_pairs;     // nonzero pattern of the float32 A, as KernelEntry::a_pairs (one row-pair mask per column)
    PackLayout L{};
    std::vector<double> pack;          // double master copy
    SolveParams base{};                // settings + cone specs, pointers empty
};

}  // namespace

struct tinympc_cuda_session;
struct tinympc_cuda_solver {
    std::vector<DeviceCtx> devs;
    Family fam;
    int precision = 32;
    int ctas_per_sm = 0;
    int chunks = 0;                    // 0 = auto
    int variant = 0;
    int force_wpp = 0;                 // option "kernel": 0 auto, 1 always the warp-per-problem kernel
    int refill_min = 0;                // option "refill_min": free lanes a warp collects before it claims new problems (tmpc_tpp3.cuh); 0 = adaptive
    int dense_a = 0;                   // option "dense_a": 1 = never the sparse-A instances (Tpp3Cfg::SA), always their dense twins
    int streamed = 1;                  // option "streamed": 1 = single-launch streamed host pipeline where it applies, 0 = chunked launches
    int compact_streamed = 1;          // option "compact_streamed": compact host I/O through one launch chain behind an arrival watermark
                                       // (run_shard_compact_streamed); 0 = the chunked pipeline
    int compact_early_d2h = 1;         // option "compact_early_d2h": exact-count mode of that pipeline with pinned result arrays -- the results
                                       // of the first pass are copied back under the fp64 pass, whose results a kernel then writes over them
    int order = 1;                     // option "order": 1 = device-resident batches of box families are claimed hardest-first (counting sort by
                                       // the expected difficulty, see order_count_kernel), 0 = in index order
    int order_sms = 1, order_from_div = 2;   // options "order_sms", "order_from_div": the compact streamed pipeline leaves that many SMs to the
                                       // ordering kernels and claims the first 1 / order_from_div of a shard in index order (measured,
                                       // profiles/r02/order_streamed_*.jsonl: 1 SM and the second half ordered is the best pair)
    int compact_in_kernel = 1;         // option "compact_in_kernel": kernels read tinympc_cuda_batch_in::xref_const in place where they can;
                                       // 0 = always replicate it over the horizon on the device first
    double mixed_band = 0;             // option "mixed": > 0 = fp32 pass + fp64 re-solve of the problems whose termination decision
                                       // falls within this relative band of the tolerances (exact iteration counts at ~fp32 speed)
    int pass_timing = 0;               // option "pass_timing": 1 = record CUDA events around the two passes of the sequential exact-count form
    int fixer_sms = -2;                // option "fixer_sms", exact-count mode: > 0 SMs the fp32 producer leaves to the concurrent fp64 consumer, 0 =
                                       // 13 % of the device; -1 = always the sequential two-pass form (fp32 pass, compaction, fp64 pass);
                                       // -2 (default) = the two-pass form for device-resident and chunked batches (its fp64 pass is the
                                       // lane-group kernel, ~1 ms per 2^20 problems), the concurrent pair inside the streamed host pipeline
    long long mixed_marked = 0;        // problems re-solved in fp64 by the last mixed solve (host entry: filled by the call)
    int mixed_pending_dev = -1;        // device entry: the count still sits in that device's counter slot
    // err, last_kernel and launches are written by the per-device worker threads of tinympc_cuda_solve_batch: the strings
    // only under `mu` (fail(), note_kernel()), the counter atomically.  Everything else a worker touches is its own DeviceCtx.
    std::mutex mu;
    std::vector<tinympc_cuda_session*> sessions;   // live sessions; orphaned (their s set to null, buffers freed) by tinympc_cuda_destroy
    std::string err;
    std::string last_kernel;
    std::atomic<long long> launches{0};
    double t_total_ms = 0, t_kernel_ms = 0;
    int t_chunks = 0;
};

struct tinympc_cuda_session {
    tinympc_cuda_solver* s = nullptr;
    int dev = 0, batch = 0, bits = 64;
    Family fam;                        // the family at creation time (a later set_family does not disturb a live session)
    WppLayout W{};
    DevBuf ws, pack, x, u, iter, status;
    std::vector<unsigned char> stage;
    // model sessions (tinympc_cuda_session_create_models): every solver's model, resident in double (one buffer per field of
    // tinympc_cuda_models, model_fields), and `dm`, the device view of them; the warp-per-problem kernels read the copy that
    // wpp_session_models writes into the model block of every workspace
    bool models = false;
    DevBuf mdl[14];
    tinympc_cuda_models dm{};
    // the device-resident entries (tinympc_cuda_session_*_device) order their work on streams[0] against the caller's stream with
    // these: ev_in recorded on the caller's stream, ev_out on streams[0]
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
};

namespace {

int fail(tinympc_cuda_solver* s, int code, const std::string& msg) {
    if (s) {
        std::lock_guard<std::mutex> lk(s->mu);
        s->err = msg;
    }
    return code;
}
void note_kernel(tinympc_cuda_solver* s, const std::string& name) {
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->last_kernel != name) s->last_kernel = name;
}
int cuda_fail(tinympc_cuda_solver* s, cudaError_t e, const char* what) {
    return fail(s, TINYMPC_CUDA_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
struct DeviceGuard {
    int prev = 0;
    DeviceGuard() { cudaGetDevice(&prev); }
    ~DeviceGuard() { cudaSetDevice(prev); }
};
#define CU(s, call)                                              \
    do {                                                         \
        cudaError_t e__ = (call);                                \
        if (e__ != cudaSuccess) return cuda_fail(s, e__, #call); \
    } while (0)

// column-major (rows x cols) double -> row-major into the pack
void put_rowmajor(std::vector<double>& pk, int at, const double* src, int rows, int cols) {
    for (int r = 0; r < rows; ++r)
        for (int c = 0; c < cols; ++c) pk[at + r * cols + c] = src ? src[(size_t)c * rows + r] : 0.0;
}
void put_vec(std::vector<double>& pk, int at, const double* src, int n) {
    for (int i = 0; i < n; ++i) pk[at + i] = src ? src[i] : 0.0;
}

// dense_a: skip the sparse-A instances (option "dense_a")
const KernelEntry* find_kernel(const Family& f, int bits, bool ppb, bool refs, int variant, bool dense_a = false) {
    int n = 0;
    const KernelEntry* const* tab = kernel_table(&n);
    for (int pass = 0; pass < 2; ++pass) {   // pass 1: a reference-storing kernel also serves a reference-free batch
        for (int i = 0; i < n; ++i) {
            const KernelEntry* e = tab[i];
            if (e->models) continue;                               // model-batch instances: model_kernel()
            if (e->fastbox && (!f.fastbox || ppb)) continue;      // table order puts the fast-box instances first
            if (f.affine && !e->affine) continue;
            if (e->a_cols && (dense_a || !a_pattern_covers(e->a_pairs, e->a_cols, f.a_pairs.data(), (int)f.a_pairs.size())))
                continue;                                          // table order puts the sparse-A instances before their dense twins
            if (e->cone_fixed) {   // cones compiled into the instance: the family's cone list must be exactly that
                const SolveParams& b = f.base;
                const bool fsx = b.en_state_soc && b.n_state_cones > 0, fsu = b.en_input_soc && b.n_input_cones > 0;
                const bool okx = e->scd > 0 ? (fsx && b.n_state_cones == 1 && b.Acx[0] == e->scs && b.qcx[0] == e->scd) : !fsx;
                const bool oku = e->ucd > 0 ? (fsu && b.n_input_cones == 1 && b.Acu[0] == e->ucs && b.qcu[0] == e->ucd) : !fsu;
                if (!okx || !oku || f.L.nsl != e->nsl || f.L.nil != e->nil) continue;
                if ((e->nsl > 0 && !b.en_state_linear) || (e->nil > 0 && !b.en_input_linear)) continue;   // rows present but switched off
            }
            if (e->family == KF_TPP && e->nx == f.nx && e->nu == f.nu && e->N == f.N && e->feat == f.feat && e->dtype_bits == bits &&
                e->ppb == (ppb ? 1 : 0) && e->variant == variant && ((e->refs != 0) == refs || (pass == 1 && e->refs != 0)))
                return e;
        }
    }
    if (variant != 0) return find_kernel(f, bits, ppb, refs, 0, dense_a);
    return nullptr;
}

// Model batches (tinympc_cuda_solve_batch_models): the model form of the lane-group fp64 kernel where it applies -- precision 64, a box
// family without adaptive rho, shared bounds, a compiled shape -- else nullptr: the warp-per-problem kernel in the solver's precision.
// max_iter <= 0 also takes the warp-per-problem kernel, which runs the reference's zero iterations (the lane-group kernel runs one).
const KernelEntry* model_kernel(const tinympc_cuda_solver* s, const Family& f, bool ppb, int bits) {
    if (s->force_wpp || bits != 64 || f.feat != kFeatBox || ppb || !f.shared_bounds_ok || f.base.max_iter <= 0) return nullptr;
    int n = 0;
    const KernelEntry* const* tab = kernel_table(&n);
    for (int i = 0; i < n; ++i)
        if (tab[i]->models && tab[i]->nx == f.nx && tab[i]->nu == f.nu && tab[i]->N == f.N) return tab[i];
    return nullptr;
}

// the arrays of tinympc_cuda_models and their doubles per problem
struct ModelField {
    const double* tinympc_cuda_models::*field;
    const char* name;
    int per_problem;
    bool required;        // dKinf_drho, dPinf_drho: required with adaptive rho
};
constexpr int kModelFields = 14;
void model_fields(int nx, int nu, bool adaptive, ModelField out[kModelFields]) {
    using M = tinympc_cuda_models;
    const ModelField f[kModelFields] = {
        {&M::Adyn, "Adyn", nx * nx, true}, {&M::Bdyn, "Bdyn", nx * nu, true}, {&M::fdyn, "fdyn", nx, false}, {&M::Q, "Q", nx, true},
        {&M::R, "R", nu, true}, {&M::rho, "rho", 1, true}, {&M::Kinf, "Kinf", nu * nx, true}, {&M::Pinf, "Pinf", nx * nx, true},
        {&M::Quu_inv, "Quu_inv", nu * nu, true}, {&M::AmBKt, "AmBKt", nx * nx, true}, {&M::APf, "APf", nx, false}, {&M::BPf, "BPf", nu, false},
        {&M::dKinf_drho, "dKinf_drho", nu * nx, adaptive}, {&M::dPinf_drho, "dPinf_drho", nx * nx, adaptive}};
    for (int k = 0; k < kModelFields; ++k) out[k] = f[k];
}

// mixed mode: gather the indices of the problems whose status carries kAmbiguousBit (order is irrelevant)
__global__ void collect_marked_kernel(const int* __restrict__ status, int n, int* __restrict__ list, int* __restrict__ count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool hit = i < n && (status[i] & kAmbiguousBit);
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (!m) return;
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(count, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (hit) list[base + __popc(m & ((1u << lane) - 1u))] = i;
}

// compact I/O (tinympc_cuda_batch_in::xref_const, tinympc_cuda_batch_out::u0): the set point replicated over the horizon,
// the first control picked out of the solution.  One thread per float4 / per element; pure HBM traffic (~0.1 ms per 2^20 problems).
__global__ void expand_xref_kernel(const float* __restrict__ xc, float* __restrict__ Xref, size_t total, int nx, int sx) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const size_t b = i / sx;
    const int e = (int)(i - b * sx) % nx;
    Xref[i] = __ldg(xc + b * nx + e);
}
__global__ void gather_u0_kernel(const float* __restrict__ u, float* __restrict__ u0, size_t total, int nu, int su) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const size_t b = i / nu;
    u0[i] = u[b * su + (i - b * nu)];
}

// compact streamed pipeline, exact-count mode: the results of the fp64 pass (the marked problems) written straight into the caller's
// pinned host arrays, over the copies of the first pass's results that are already there (hu0 / hiter / hstatus: device aliases of
// those host arrays).  ~1 % of the batch, one thread per marked problem.
__global__ void scatter_marked_to_host_kernel(const int* __restrict__ list, const int* __restrict__ count, const int* __restrict__ iter,
                                              const int* __restrict__ status, const float* __restrict__ u0, int nu,
                                              int* __restrict__ hiter, int* __restrict__ hstatus, float* __restrict__ hu0) {
    const int n = *count;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const int i = list[k];
        hiter[i] = iter[i];
        hstatus[i] = status[i];
        for (int a = 0; a < nu; ++a) hu0[(size_t)i * nu + a] = u0[(size_t)i * nu + a];
    }
}

// ---- claim order: hardest problems first -----------------------------------------------------------------------------------
// The thread-per-problem kernels hold one problem per lane until it converges, and problems take anything from one check
// interval to max_iter iterations.  In claim order = index order a warp's lanes hold problems of all lengths (its refill passes
// serve one or two lanes at a time) and the launch ends with a tail in which every lane finishes whatever it happened to hold.
// How far the unconstrained feedback -Kinf (x0 - xref_0) leaves the input bounds predicts the iteration count well (rank
// correlation 0.9 on the quadrotor batch): key = max_a |Kinf (x0 - xref_0)|_a / min(-u_min_a, u_max_a).  The three kernels below
// bucket the batch by that key (256 buckets, hardest first; counting sort: count, scan, scatter) into an index list the solve
// kernel claims from.  Lanes of a warp then hold problems of similar length and the tail consists of the shortest ones:
// 15.2 -> 13.9 ms on the 2^20 quadrotor batch (profiles/r02/order_study.jsonl) for ~0.05 ms of pre-pass.  Scheduling only:
// every problem is solved by the same code whatever its position (the permutation test holds the results to bit identity).
constexpr int kOrderBuckets = 256, kOrderBlock = 256, kOrderItems = 4;
struct OrderParams {
    float K[8 * 16];      // Kinf, row-major nu x nx
    float inv_ub[8];      // 1 / min(-u_min_a, u_max_a)
    int nx, nu, xref_stride;   // xref_stride: floats between the reference states of consecutive problems (nx: compact, nx*N: full, 0: none)
};
__device__ __forceinline__ int order_bucket(const OrderParams& op, const float* __restrict__ x0, const float* __restrict__ xref, int i) {
    // d = x0 - xref_0 in registers (nx <= 16): 128-bit loads when the rows are 16-byte multiples (every compiled shape but nx = 6)
    float d[16];
    const int nx = op.nx;
    const float* px = x0 + (size_t)i * nx;
    const float* pr = xref ? xref + (size_t)i * op.xref_stride : nullptr;
    if (((nx | op.xref_stride) & 3) == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (4 * q < nx) {
                v = __ldg(reinterpret_cast<const float4*>(px) + q);
                if (pr) {
                    const float4 r = __ldg(reinterpret_cast<const float4*>(pr) + q);
                    v.x -= r.x; v.y -= r.y; v.z -= r.z; v.w -= r.w;
                }
            }
            d[4 * q] = v.x; d[4 * q + 1] = v.y; d[4 * q + 2] = v.z; d[4 * q + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int c = 0; c < 16; ++c) d[c] = c < nx ? __ldg(px + c) - (pr ? __ldg(pr + c) : 0.f) : 0.f;
    }
    float key = 0.f;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        if (a < op.nu) {
            float acc = 0.f;
#pragma unroll
            for (int c = 0; c < 16; ++c) if (c < nx) acc = fmaf(op.K[a * nx + c], d[c], acc);
            key = fmaxf(key, fabsf(acc) * op.inv_ub[a]);
        }
    }
    // 64 buckets per unit of key: everything beyond 4x the bound is "hardest"; bucket 0 of the LIST is the hardest
    const int b = min(kOrderBuckets - 1, __float2int_rd(key * 64.f));
    return kOrderBuckets - 1 - (b < 0 ? kOrderBuckets - 1 : b);      // NaN / negative: treat as hardest
}
// problems first .. first + n - 1 of the arrays; bucket[] and the list positions are relative to `first`, the list ENTRIES are problem indices
__global__ void __launch_bounds__(kOrderBlock) order_count_kernel(const __grid_constant__ OrderParams op, const float* __restrict__ x0,
                                                                  const float* __restrict__ xref, int first, int n,
                                                                  unsigned char* __restrict__ bucket, int* __restrict__ hist) {
    __shared__ int sh[kOrderBuckets];
    for (int b = threadIdx.x; b < kOrderBuckets; b += kOrderBlock) sh[b] = 0;
    __syncthreads();
#pragma unroll 2
    for (int k = 0; k < kOrderItems; ++k) {
        const int i = (blockIdx.x * kOrderItems + k) * kOrderBlock + threadIdx.x;
        if (i < n) {
            const int b = order_bucket(op, x0, xref, first + i);
            bucket[i] = (unsigned char)b;
            atomicAdd(&sh[b], 1);
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kOrderBuckets; b += kOrderBlock) if (sh[b]) atomicAdd(&hist[b], sh[b]);
}
__global__ void order_scan_kernel(int* __restrict__ hist) {   // one block of kOrderBuckets threads: exclusive prefix sum in place
    __shared__ int sh[kOrderBuckets];
    const int t = threadIdx.x;
    sh[t] = hist[t];
    __syncthreads();
    for (int o = 1; o < kOrderBuckets; o <<= 1) {
        const int v = t >= o ? sh[t - o] : 0;
        __syncthreads();
        sh[t] += v;
        __syncthreads();
    }
    hist[t] = sh[t] - hist[t];
}
__global__ void __launch_bounds__(kOrderBlock) order_scatter_kernel(const unsigned char* __restrict__ bucket, int first, int n,
                                                                    int* __restrict__ offset, int* __restrict__ list) {
    __shared__ int cnt[kOrderBuckets], base[kOrderBuckets];
    for (int b = threadIdx.x; b < kOrderBuckets; b += kOrderBlock) cnt[b] = 0;
    __syncthreads();
    int bk[kOrderItems], rk[kOrderItems];
    for (int k = 0; k < kOrderItems; ++k) {
        const int i = (blockIdx.x * kOrderItems + k) * kOrderBlock + threadIdx.x;
        bk[k] = i < n ? bucket[i] : -1;
        rk[k] = bk[k] >= 0 ? atomicAdd(&cnt[bk[k]], 1) : 0;          // rank inside the block's share of the bucket
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kOrderBuckets; b += kOrderBlock) base[b] = cnt[b] ? atomicAdd(&offset[b], cnt[b]) : 0;
    __syncthreads();
    for (int k = 0; k < kOrderItems; ++k) {
        const int i = (blockIdx.x * kOrderItems + k) * kOrderBlock + threadIdx.x;
        if (bk[k] >= 0) list[base[bk[k]] + rk[k]] = first + i;
    }
}

// device alias of a pinned (page-locked, mapped) host pointer; false for pageable memory
bool host_alias(const void* p, void** alias) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type != cudaMemoryTypeHost || a.devicePointer == nullptr) return false;
    *alias = a.devicePointer;
    return true;
}

int upload_family(tinympc_cuda_solver* s) {
    const Family& f = s->fam;
    std::vector<float> p32(f.pack.size());
    for (size_t i = 0; i < f.pack.size(); ++i) p32[i] = static_cast<float>(f.pack[i]);
    for (auto& d : s->devs) {
        CU(s, cudaSetDevice(d.device));
        if (d.pack32) cudaFree(d.pack32);
        if (d.pack64) cudaFree(d.pack64);
        d.pack32 = d.pack64 = nullptr;
        CU(s, cudaMalloc(&d.pack32, p32.size() * sizeof(float)));
        CU(s, cudaMalloc(&d.pack64, f.pack.size() * sizeof(double)));
        CU(s, cudaMemcpy(d.pack32, p32.data(), p32.size() * sizeof(float), cudaMemcpyHostToDevice));
        CU(s, cudaMemcpy(d.pack64, f.pack.data(), f.pack.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    return TINYMPC_CUDA_OK;
}

// Launch one thread-per-problem kernel instance (persistent grid, a multiple of the SM count).
// find_kernel + the small-batch rule: where the default instance uses the hybrid state layout (more resident warps, more
// instructions per iteration), a batch that fits one wave of the plain-layout instance is latency bound and runs that one.
const KernelEntry* pick_kernel(const tinympc_cuda_solver* s, const DeviceCtx& d, const Family& f, int bits, bool ppb, bool refs, int batch) {
    const KernelEntry* ke = find_kernel(f, bits, ppb, refs, s->variant, s->dense_a);
    if (ke && s->variant == 0 && bits == 32) {
        const KernelEntry* kl = find_kernel(f, bits, ppb, refs, kLatencyVariant, s->dense_a);
        if (kl && kl->variant == kLatencyVariant && kl->block < ke->block && batch <= d.sm_count * kl->block) ke = kl;
    }
    return ke;
}

int launch_tpp(tinympc_cuda_solver* s, DeviceCtx& d, const KernelEntry* ke, SolveParams& p, DevBuf& rb, int bits, int* counter, cudaStream_t st,
               int reserve_sms = 0, int* grid_out = nullptr, int max_sms = 0, const tinympc_cuda_models* models = nullptr) {
    const Family& f = s->fam;
    const size_t smem = ke->smem_bytes(f.L.cold_size);
    if (smem > 227u * 1024u) return fail(s, TINYMPC_CUDA_EUNSUPPORTED, std::string("kernel ") + ke->name + " needs more shared memory than an SM has");
    CU(s, ke->prepare(smem));
    int occ = 0;
    CU(s, ke->occupancy(&occ, smem));
    if (occ < 1) return fail(s, TINYMPC_CUDA_EUNSUPPORTED, std::string("kernel ") + ke->name + " does not fit on an SM");
    if (s->ctas_per_sm > 0 && s->ctas_per_sm < occ) occ = s->ctas_per_sm;
    int grid = std::max(1, d.sm_count - reserve_sms) * occ;   // persistent CTAs: a multiple of the SM count (minus the SMs left to a concurrent launch)
    if (max_sms > 0) grid = std::min(grid, max_sms * occ);
    const int per_cta = ke->lanes_per_problem > 1 ? ke->block / ke->lanes_per_problem : ke->block;   // problems a CTA holds at a time
    const int need = (p.batch + per_cta - 1) / per_cta;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    if (ke->refs == 2) {   // reference terms live in a lane-interleaved global scratch that stays L2 resident
        const size_t esz = bits == 64 ? sizeof(double) : sizeof(float);
        CU(s, rb.reserve((size_t)grid * ke->block * ((size_t)f.nx * f.N + (size_t)f.nu * (f.N - 1)) * esz));
        p.ref_scratch = rb.p;
    }
    p.work_counter = counter;
    p.refill_min = s->refill_min;
    CU(s, cudaMemsetAsync(counter, 0, sizeof(int), st));
    CU(s, models ? ke->models_launch(p, grid, smem, st, f.pack.data(), f.L, *models) : ke->launch(p, grid, smem, st, f.pack.data(), f.L));
    s->launches += 1;
    if (grid_out) *grid_out = grid;
    return TINYMPC_CUDA_OK;
}

int auto_fixer_sms(const tinympc_cuda_solver* s, const DeviceCtx& d) {
    if (s->fixer_sms > 0) return std::min(s->fixer_sms, d.sm_count / 2);
    // The consumer re-solves ~2 % of the problems at ~1/7 of the producer's per-SM rate: ~13 % of the SMs balances the two
    // launches (measured optimum on the quadrotor batch, profiles/r02/fixer_sweep.jsonl).
    return std::max(2, (d.sm_count * 13 + 50) / 100);
}

// Exact-count mode, concurrent form: the fp32 producer on `st` over all but R SMs, the fp64 consumer on the slot's own stream over
// exactly R.  The two grids together never exceed the device, so whichever of them the hardware starts first leaves room for
// the other: a consumer that waits on the queue can never keep the producer from running.  p32 / p64 arrive with their in/out
// pointers (and, for the streamed pipeline, the watermark / completion fields) set.  The producer is launched FIRST: if something
// serialises the two launches (profilers), the queue is simply complete before the consumer starts.
int launch_exact_pair(tinympc_cuda_solver* s, DeviceCtx& d, const KernelEntry* ke, const KernelEntry* ke64, SolveParams p32, SolveParams p64, int batch,
                      int counter_slot, int slot, int* counter, cudaStream_t st) {
    const Family& f = s->fam;
    int* q = d.qctl + 4 * counter_slot;
    DevBuf& list = d.marked[slot];
    CU(s, list.reserve(sizeof(int) * (size_t)batch));
    CU(s, cudaMemsetAsync(q, 0, sizeof(int) * 4, st));
    CU(s, cudaMemsetAsync(list.p, 0xFF, sizeof(int) * (size_t)batch, st));      // every entry -1 = "not written yet"
    CU(s, cudaEventRecord(d.ev_fork[slot], st));
    p32.amb_band = static_cast<float>(s->mixed_band);
    p32.q_tail = q; p32.q_list = static_cast<int*>(list.p); p32.q_prod_done = q + 1; p32.q_consume = 0; p32.q_prod_total = 0;
    int grid32 = 0;
    const int R = auto_fixer_sms(s, d);
    int rc = launch_tpp(s, d, ke, p32, d.ref_scratch[slot], 32, counter, st, R, &grid32);
    if (rc) return rc;
    p64.pack = (const void*)((const double*)d.pack64 + f.L.cold);
    p64.amb_band = 0.f;
    p64.avail_ptr = nullptr;                 // whatever the producer queued has landed
    p64.q_tail = q; p64.q_list = static_cast<int*>(list.p); p64.q_prod_done = q + 1; p64.q_consume = 1; p64.q_prod_total = grid32;
    cudaStream_t fs = d.fix_stream[slot];
    CU(s, cudaStreamWaitEvent(fs, d.ev_fork[slot], 0));
    rc = launch_tpp(s, d, ke64, p64, d.ref_scratch64[slot], 64, q + 2, fs, 0, nullptr, R);
    if (rc) return rc;
    CU(s, cudaEventRecord(d.ev_join[slot], fs));
    CU(s, cudaStreamWaitEvent(st, d.ev_join[slot], 0));
    note_kernel(s, std::string(ke->name) + "|" + ke64->name);
    return TINYMPC_CUDA_OK;
}

// Do the kernels that will serve the batch do compact I/O themselves (SolveParams::xref_const / u0, KernelEntry::compact_ok)?
// Mirrors the kernel choice of enqueue(): the first-pass kernel and, in the exact-count mode, the fp64 kernel of the second pass.
bool compact_in_kernel(const tinympc_cuda_solver* s, const DeviceCtx& d, bool ppb, bool refs, int batch, const KernelEntry** ke_out = nullptr,
                       const KernelEntry** ke64_out = nullptr, bool models = false) {
    const Family& f = s->fam;
    if (ke_out) *ke_out = nullptr;
    if (ke64_out) *ke64_out = nullptr;
    if (models) {
        const KernelEntry* ke = model_kernel(s, f, ppb, s->precision);
        return s->compact_in_kernel && ke && ke->compact_ok;
    }
    if (s->force_wpp) return false;
    const KernelEntry* ke = pick_kernel(s, d, f, s->precision, ppb, refs, batch);
    const bool mixed = s->mixed_band > 0 && s->precision == 32;
    const KernelEntry* ke64 = mixed ? find_kernel(f, 64, ppb, refs, 0) : nullptr;
    if (ke_out) *ke_out = ke;
    if (ke64_out) *ke64_out = ke64;
    return s->compact_in_kernel && ke && ke->compact_ok && (!mixed || (ke64 && ke64->compact_ok));
}

constexpr int kDirectXref = 1, kDirectU0 = 2;   // enqueue(): compact I/O handed to the kernels as it is

// Claim order (order_count_kernel): problems first .. first + n - 1 bucketed hardest-first into list[0 .. n) (entries = problem
// indices), on `st`.  hist: kOrderBuckets ints, bucket: n bytes of scratch.
int build_order_range(tinympc_cuda_solver* s, const SolveParams& p, int first, int n, int* hist, int* list, unsigned char* bucket, cudaStream_t st) {
    const Family& f = s->fam;
    OrderParams op{};
    op.nx = f.nx; op.nu = f.nu;
    op.xref_stride = p.Xref ? (p.xref_const ? f.nx : f.nx * f.N) : 0;
    for (int a = 0; a < f.nu; ++a) {
        for (int c = 0; c < f.nx; ++c) op.K[a * f.nx + c] = static_cast<float>(f.pack[f.L.Kinf + a * f.nx + c]);
        const double ub = std::min(-f.pack[f.L.umin + a], f.pack[f.L.umax + a]);     // the bounds of the first step
        op.inv_ub[a] = (ub > 0 && std::isfinite(ub)) ? static_cast<float>(1.0 / ub) : 0.f;
    }
    const int blocks = (n + kOrderBlock * kOrderItems - 1) / (kOrderBlock * kOrderItems);
    CU(s, cudaMemsetAsync(hist, 0, sizeof(int) * kOrderBuckets, st));
    order_count_kernel<<<blocks, kOrderBlock, 0, st>>>(op, p.x0, p.Xref, first, n, bucket, hist);
    order_scan_kernel<<<1, kOrderBuckets, 0, st>>>(hist);
    order_scatter_kernel<<<blocks, kOrderBlock, 0, st>>>(bucket, first, n, hist, list);
    CU(s, cudaGetLastError());
    s->launches += 3;
    return TINYMPC_CUDA_OK;
}
// ... of a whole device-resident batch; order_buf: hist per range (kMaxGranules of them) | list | bucket bytes
int reserve_order(tinympc_cuda_solver* s, DeviceCtx& d, int n, int** hist, int** list, unsigned char** bucket) {
    CU(s, d.order_buf.reserve(sizeof(int) * ((size_t)kOrderBuckets * kMaxGranules + (size_t)n) + (size_t)n));
    *hist = static_cast<int*>(d.order_buf.p);
    *list = *hist + kOrderBuckets * kMaxGranules;
    *bucket = reinterpret_cast<unsigned char*>(*list + n);
    return TINYMPC_CUDA_OK;
}
int build_order(tinympc_cuda_solver* s, DeviceCtx& d, const SolveParams& p, int n, cudaStream_t st, const int** list_out) {
    int *hist, *list;
    unsigned char* bucket;
    int rc = reserve_order(s, d, n, &hist, &list, &bucket);
    if (rc) return rc;
    rc = build_order_range(s, p, 0, n, hist, list, bucket, st);
    *list_out = list;
    return rc;
}

// Enqueue the solve of `in`/`out` (device pointers) on `st`.  slot selects the work counters and scratch buffers
// (one set per pipeline stream + one for the device-resident entry point).  models (device pointers): a model batch.
int enqueue(tinympc_cuda_solver* s, DeviceCtx& d, const tinympc_cuda_batch_in& in, const tinympc_cuda_batch_out& out, int counter_slot,
            cudaStream_t st, int scratch_slot, int direct = 0, const tinympc_cuda_models* models = nullptr) {
    const Family& f = s->fam;
    const bool ppb = in.x_min || in.x_max || in.u_min || in.u_max;
    if (ppb && !(in.x_min && in.x_max && in.u_min && in.u_max))
        return fail(s, TINYMPC_CUDA_EINVAL, "per-problem bounds need all four of x_min, x_max, u_min, u_max");
    if (!ppb && !f.shared_bounds_ok)
        return fail(s, TINYMPC_CUDA_EINVAL, "bound constraints are enabled but neither the family nor the batch supplies bounds");
    if (in.xref_const && in.Xref) return fail(s, TINYMPC_CUDA_EINVAL, "give Xref or xref_const, not both");
    const bool full_out = out.x && out.u;
    if (!full_out && !out.u0) return fail(s, TINYMPC_CUDA_EINVAL, "x and u are required unless u0 is given");
    if (!direct && (in.xref_const || !full_out)) {
        // compact I/O.  Kernels with KernelEntry::compact_ok read the one reference state per problem in place of every column and
        // write the first control alone; for any other kernel the reference is replicated over the horizon first and the
        // trajectories go to this slot's device scratch, from which u0 is gathered.
        const size_t sx = (size_t)f.nx * f.N, su = (size_t)f.nu * (f.N - 1);
        const bool in_kernel = compact_in_kernel(s, d, ppb, in.xref_const || in.Xref || in.Uref, in.batch, nullptr, nullptr, models != nullptr);
        tinympc_cuda_batch_in in2 = in;
        tinympc_cuda_batch_out out2 = out;
        in2.xref_const = nullptr;
        int dir = 0;
        if (in.xref_const) {
            if (in_kernel) {
                in2.Xref = in.xref_const;
                dir |= kDirectXref;
            } else {
                DevBuf& xb = d.exp_xref[scratch_slot];
                CU(s, xb.reserve(sizeof(float) * sx * in.batch));
                const size_t total = sx * in.batch;
                expand_xref_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in.xref_const, static_cast<float*>(xb.p), total, f.nx, (int)sx);
                CU(s, cudaGetLastError());
                s->launches += 1;
                in2.Xref = static_cast<const float*>(xb.p);
            }
        }
        const bool u0_direct = in_kernel && out.u0 && !out.x && !out.u;
        if (u0_direct) {
            dir |= kDirectU0;
        } else {
            out2.u0 = nullptr;
            if (!out.x) { CU(s, d.exp_x[scratch_slot].reserve(sizeof(float) * sx * in.batch)); out2.x = static_cast<float*>(d.exp_x[scratch_slot].p); }
            if (!out.u) { CU(s, d.exp_u[scratch_slot].reserve(sizeof(float) * su * in.batch)); out2.u = static_cast<float*>(d.exp_u[scratch_slot].p); }
        }
        if (dir == 0) dir = -1;   // plain trajectories from here on: do not come back into this branch
        int rc = enqueue(s, d, in2, out2, counter_slot, st, scratch_slot, dir, models);
        if (rc) return rc;
        if (out.u0 && !u0_direct) {
            const size_t total = (size_t)f.nu * in.batch;
            gather_u0_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(out2.u, out.u0, total, f.nu, (int)su);
            CU(s, cudaGetLastError());
            s->launches += 1;
        }
        return TINYMPC_CUDA_OK;
    }
    if (direct < 0) direct = 0;
    const bool refs = in.Xref || in.Uref;
    int bits = s->precision;
    const KernelEntry* ke = models ? model_kernel(s, f, ppb, s->precision) : s->force_wpp ? nullptr : pick_kernel(s, d, f, bits, ppb, refs, in.batch);
    // mixed mode needs the specialised kernels in both precisions; any other shape runs entirely in fp64 (exact as well)
    const KernelEntry* ke64 = nullptr;
    const bool mixed = !models && s->mixed_band > 0 && bits == 32;   // model batches: refused by solve_batch_common
    if (mixed) {
        ke64 = s->force_wpp ? nullptr : find_kernel(f, 64, ppb, refs, 0);
        if (!ke || !ke64) { ke = nullptr; bits = 64; }
    }
    SolveParams p = f.base;
    p.pack = bits == 64 ? (const void*)((const double*)d.pack64 + f.L.cold) : (const void*)((const float*)d.pack32 + f.L.cold);
    p.pack_elems = f.L.cold_size;
    p.batch = in.batch;
    p.x0 = in.x0; p.Xref = in.Xref; p.Uref = in.Uref;
    p.xref_const = (direct & kDirectXref) ? 1 : 0;
    p.x_min = in.x_min; p.x_max = in.x_max; p.u_min = in.u_min; p.u_max = in.u_max;
    p.x = out.x; p.u = out.u; p.iter = out.iter; p.status = out.status; p.residuals = out.residuals; p.rho_out = out.rho;
    p.u0 = (direct & kDirectU0) ? out.u0 : nullptr;

    if (direct && !(ke && ke->compact_ok && (!mixed || ke64->compact_ok)))
        return fail(s, TINYMPC_CUDA_EUNSUPPORTED, "internal: compact I/O handed to a kernel that does not do it");
    if (!ke) {
        // no specialised thread-per-problem kernel for this shape / feature mix: general warp-per-problem kernel
        const WppLayout W = WppLayout::make(f.nx, f.nu, f.N, models != nullptr);
        const int warps = std::max(1, std::min(in.batch, d.sm_count * 16));
        const size_t esz = bits == 64 ? sizeof(double) : sizeof(float);
        DevBuf& sb = d.wpp_scratch[scratch_slot];
        CU(s, sb.reserve((size_t)warps * W.size * esz));
        const void* full_pack = bits == 64 ? d.pack64 : d.pack32;
        if (bits == 64) CU(s, wpp_launch<double>(p, f.L, full_pack, W, sb.p, warps, 0, st, models));
        else CU(s, wpp_launch<float>(p, f.L, full_pack, W, sb.p, warps, 0, st, models));
        note_kernel(s, models ? (bits == 64 ? "wpp_f64_mdl_generic" : "wpp_f32_mdl_generic") : (bits == 64 ? "wpp_f64_generic" : "wpp_f32_generic"));
        s->launches += 1;
        return TINYMPC_CUDA_OK;
    }
    int* const counter = d.counters + counter_slot;
    // device-resident batches of a few waves: the fp32 thread-per-problem kernels claim the hardest problems first (build_order)
    if (!models && s->order && scratch_slot == kStreams && bits == 32 && f.feat == kFeatBox && !ppb && f.shared_bounds_ok && p.en_input_bound &&
        ke->lanes_per_problem <= 1 && f.nx <= 16 && f.nu <= 8 && (long long)in.batch >= 2LL * d.sm_count * ke->block) {
        int rc = build_order(s, d, p, in.batch, st, &p.index_list);
        if (rc) return rc;
    }
    if (!mixed) {
        int rc = launch_tpp(s, d, ke, p, d.ref_scratch[scratch_slot], bits, counter, st, 0, nullptr, 0, models);
        if (rc) return rc;
        note_kernel(s, ke->name);
        return TINYMPC_CUDA_OK;
    }
    if (s->fixer_sms >= 0) {
        SolveParams p64 = p;
        p64.index_list = nullptr;          // the consumer takes its problems from the queue
        return launch_exact_pair(s, d, ke, ke64, p, p64, in.batch, counter_slot, scratch_slot, counter, st);
    }
    // ---- mixed mode, sequential form: fp32 pass that marks the ambiguous problems, compaction, fp64 re-solve of the marked ones ----
    int* const counter2 = d.counters + kMaxChunks + counter_slot;
    int* const n_marked = d.counters + 2 * kMaxChunks + counter_slot;
    DevBuf& list = d.marked[scratch_slot];
    CU(s, list.reserve(sizeof(int) * (size_t)in.batch));
    p.amb_band = static_cast<float>(s->mixed_band);
    const bool timed = s->pass_timing != 0 && scratch_slot == kStreams;     // the device-resident entry point only
    if (timed) CU(s, cudaEventRecord(d.ev_p0, st));
    int rc = launch_tpp(s, d, ke, p, d.ref_scratch[scratch_slot], 32, counter, st);
    if (rc) return rc;
    if (timed) CU(s, cudaEventRecord(d.ev_p1, st));
    CU(s, cudaMemsetAsync(n_marked, 0, sizeof(int), st));
    collect_marked_kernel<<<(in.batch + 255) / 256, 256, 0, st>>>(out.status, in.batch, static_cast<int*>(list.p), n_marked);
    CU(s, cudaGetLastError());
    s->launches += 1;
    SolveParams p2 = p;
    p2.pack = (const void*)((const double*)d.pack64 + f.L.cold);
    p2.amb_band = 0.f;
    p2.index_list = static_cast<const int*>(list.p);
    p2.batch_ptr = n_marked;
    rc = launch_tpp(s, d, ke64, p2, d.ref_scratch64[scratch_slot], 64, counter2, st);
    if (rc) return rc;
    if (timed) { CU(s, cudaEventRecord(d.ev_p2, st)); d.pass_timed = true; }
    note_kernel(s, std::string(ke->name) + "+" + ke64->name);
    return TINYMPC_CUDA_OK;
}

int check_ptr16(tinympc_cuda_solver* s, const void* p, const char* name) {
    if (p && (reinterpret_cast<uintptr_t>(p) & 15u)) return fail(s, TINYMPC_CUDA_EINVAL, std::string(name) + " must be 16-byte aligned");
    return TINYMPC_CUDA_OK;
}

// max_iter <= 0: the reference loop body never runs (admm.cpp:312); solution = zero workspace, iter 0, status 11
int zero_iteration_result(tinympc_cuda_solver* s, const Family& f, const tinympc_cuda_batch_out& out, int batch, cudaStream_t st, bool device) {
    const size_t sx = (size_t)f.nx * f.N, su = (size_t)f.nu * (f.N - 1);
    if (device) {
        if (out.x) CU(s, cudaMemsetAsync(out.x, 0, sizeof(float) * sx * batch, st));
        if (out.u) CU(s, cudaMemsetAsync(out.u, 0, sizeof(float) * su * batch, st));
        if (out.u0) CU(s, cudaMemsetAsync(out.u0, 0, sizeof(float) * f.nu * batch, st));
        CU(s, cudaMemsetAsync(out.iter, 0, sizeof(int) * batch, st));
        std::vector<int> st11(batch, 11);
        CU(s, cudaMemcpyAsync(out.status, st11.data(), sizeof(int) * batch, cudaMemcpyHostToDevice, st));
        CU(s, cudaStreamSynchronize(st));
        if (out.residuals) CU(s, cudaMemsetAsync(out.residuals, 0, sizeof(float) * 4 * batch, st));
        if (out.rho) {
            std::vector<float> r(batch, (float)f.base.rho);
            CU(s, cudaMemcpyAsync(out.rho, r.data(), sizeof(float) * batch, cudaMemcpyHostToDevice, st));
            CU(s, cudaStreamSynchronize(st));
        }
    } else {
        if (out.x) std::memset(out.x, 0, sizeof(float) * sx * batch);
        if (out.u) std::memset(out.u, 0, sizeof(float) * su * batch);
        if (out.u0) std::memset(out.u0, 0, sizeof(float) * f.nu * batch);
        for (int b = 0; b < batch; ++b) { out.iter[b] = 0; out.status[b] = 11; }
        if (out.residuals) std::memset(out.residuals, 0, sizeof(float) * 4 * batch);
        if (out.rho) for (int b = 0; b < batch; ++b) out.rho[b] = (float)f.base.rho;
    }
    return TINYMPC_CUDA_OK;
}

// ---- streamed pipeline -------------------------------------------------------------------------------------------------
// The two stream memory operations of the driver API, resolved at run time (no link-time dependency on libcuda).
using StreamMemOp32 = CUresult (*)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
struct StreamMemOps {
    StreamMemOp32 wait = nullptr, write = nullptr;
    bool ok = false;
};
const StreamMemOps& stream_memops() {
    static const StreamMemOps ops = [] {
        StreamMemOps o;
        void* fw = nullptr; void* fr = nullptr;
        cudaDriverEntryPointQueryResult q1, q2;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fw, cudaEnableDefault, &q1) == cudaSuccess && q1 == cudaDriverEntryPointSuccess &&
            cudaGetDriverEntryPoint("cuStreamWriteValue32", &fr, cudaEnableDefault, &q2) == cudaSuccess && q2 == cudaDriverEntryPointSuccess && fw && fr) {
            o.wait = reinterpret_cast<StreamMemOp32>(fw);
            o.write = reinterpret_cast<StreamMemOp32>(fr);
            o.ok = true;
        }
        cudaGetLastError();
        return o;
    }();
    return ops;
}

// One device's share of a host batch as ONE persistent launch that consumes the problems while the copy engine is still
// delivering them: stream 0 carries the H2D chunks, each followed by a write of the arrival watermark; stream 1 carries the
// kernel, whose lanes wait on the watermark before they read a claimed problem and count every finished problem per chunk;
// stream 2 waits (cuStreamWaitValue32) for a chunk's count and copies its results back.  No launch boundaries, hence no
// per-chunk tails of idle lanes, and the three engines (H2D DMA, SMs, D2H DMA) overlap for the whole batch.
int run_shard_streamed(tinympc_cuda_solver* s, DeviceCtx& d, const KernelEntry* ke, const KernelEntry* ke64, const tinympc_cuda_batch_in& in,
                       const tinympc_cuda_batch_out& out, int lo, int hi, int nch, double* kernel_ms, int* nchunks_out, long long* marked_out) {
    const Family& f = s->fam;
    const StreamMemOps& ops = stream_memops();
    const int n = hi - lo;
    const size_t sx = (size_t)f.nx * f.N, su = (size_t)f.nu * (f.N - 1);
    const bool ppb = in.x_min != nullptr;
    // Granules of a multiple of 32 problems: every array's granule boundary then falls on a 128-byte line for any shape, so
    // no line holds data of two chunks (a lane reads its problem with non-coherent loads once the watermark covers it).
    // Chunks are runs of granules.  nch > 0: nch equal chunks.  nch == 0 (auto): 1, 1, 2, 4, 4, ..., 4, 2, 1, 1 sixty-fourths
    // of the shard -- the kernel starts after 1/64 of the H2D time and the last D2H copy is 1/64 of the results.
    std::vector<int> bounds;   // chunk c = problems [bounds[c], bounds[c + 1])
    int gran;
    {
        const bool ramp = nch <= 0;
        const int ng_target = ramp ? kMaxGranules : std::min(nch, kMaxGranules);
        gran = (((n + ng_target - 1) / ng_target) + 31) & ~31;
        const int ng = (n + gran - 1) / gran;
        std::vector<int> runs;
        if (ramp && ng >= 16) {
            const int head[3] = {1, 1, 2};
            int left = ng - 8;
            for (int h : head) runs.push_back(h);
            while (left > 0) { runs.push_back(std::min(4, left)); left -= 4; }
            runs.push_back(2); runs.push_back(1); runs.push_back(1);
        } else {
            runs.assign(ng, 1);
        }
        int g = 0;
        bounds.push_back(0);
        for (size_t c = 0; c < runs.size(); ++c) {
            g += runs[c];
            bounds.push_back(std::min(n, g * gran));
        }
    }
    nch = (int)bounds.size() - 1;
    cudaStream_t s_in = d.streams[0], s_k = d.streams[1], s_out = d.streams[2];
    int* ctl = d.stream_ctl;
    CU(s, cudaMemsetAsync(ctl, 0, sizeof(int) * (2 + nch), s_k));
    CU(s, cudaEventRecord(d.ev_ctl, s_k));
    CU(s, cudaStreamWaitEvent(s_in, d.ev_ctl, 0));
    CU(s, cudaStreamWaitEvent(s_out, d.ev_ctl, 0));

    SolveParams p = f.base;
    p.pack = (const void*)((const float*)d.pack32 + f.L.cold);
    if (ke->dtype_bits == 64) p.pack = (const void*)((const double*)d.pack64 + f.L.cold);
    p.pack_elems = f.L.cold_size;
    p.batch = n;
    p.x0 = (const float*)d.x0.p; p.Xref = in.Xref ? (const float*)d.Xref.p : nullptr; p.Uref = in.Uref ? (const float*)d.Uref.p : nullptr;
    if (ppb) { p.x_min = (const float*)d.xmin.p; p.x_max = (const float*)d.xmax.p; p.u_min = (const float*)d.umin.p; p.u_max = (const float*)d.umax.p; }
    p.x = (float*)d.x.p; p.u = (float*)d.u.p; p.iter = (int*)d.iter.p; p.status = (int*)d.status.p;
    p.residuals = out.residuals ? (float*)d.res.p : nullptr;
    p.rho_out = out.rho ? (float*)d.rho.p : nullptr;
    p.avail_ptr = ctl + 1;
    p.done_counters = ctl + 2;
    p.done_chunk = gran;
    for (int c = 0; c < nch; ++c)
        for (int g = bounds[c] / gran; g * gran < bounds[c + 1]; ++g) p.done_map[g] = (unsigned char)c;
    // Order of the enqueues: ALL the input copies and their watermark writes first, then the kernel, then the result copies.
    // Nothing the kernel waits for is enqueued after its launch, so the pipeline also completes when something serialises
    // kernel launches on the host (ncu / compute-sanitizer replay, CUDA_LAUNCH_BLOCKING=1): the launch call may block until the
    // kernel has finished, and the copy engine keeps delivering meanwhile.  The copies are asynchronous (pinned memory), so
    // the launch is delayed only by the ~100 enqueue calls, less than the arrival time of the first chunk.
    auto sync_fail = [&](int rc) -> int { cudaDeviceSynchronize(); return rc; };
#define RT(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return sync_fail(cuda_fail(s, e__, #call)); } while (0)
#define DRV(call, what) do { CUresult r__ = (call); if (r__ != CUDA_SUCCESS) return sync_fail(fail(s, TINYMPC_CUDA_ECUDA, std::string(what) + " failed with CUresult " + std::to_string((int)r__))); } while (0)
    for (int c = 0; c < nch; ++c) {
        const int c0 = bounds[c], c1 = bounds[c + 1], cn = c1 - c0;
        const size_t g0 = (size_t)lo + c0;
        auto h2d = [&](DevBuf& dst, const float* src, size_t per_problem) -> cudaError_t {
            return cudaMemcpyAsync((float*)dst.p + per_problem * c0, src + per_problem * g0, sizeof(float) * per_problem * cn, cudaMemcpyHostToDevice, s_in);
        };
        RT(h2d(d.x0, in.x0, f.nx));
        if (in.Xref) RT(h2d(d.Xref, in.Xref, sx));
        if (in.Uref) RT(h2d(d.Uref, in.Uref, su));
        if (ppb) { RT(h2d(d.xmin, in.x_min, sx)); RT(h2d(d.xmax, in.x_max, sx)); RT(h2d(d.umin, in.u_min, su)); RT(h2d(d.umax, in.u_max, su)); }
        DRV(ops.write(reinterpret_cast<CUstream>(s_in), reinterpret_cast<CUdeviceptr>(ctl + 1), (cuuint32_t)c1, 0), "cuStreamWriteValue32");
    }
    RT(cudaEventRecord(d.k0[0], s_k));
    if (ke64) {
        // exact-count mode: producer (streamed fp32) + concurrent fp64 consumer; a problem counts for its chunk when whichever
        // of the two finishes it
        int rc = launch_exact_pair(s, d, ke, ke64, p, p, n, 0, 0, ctl, s_k);
        if (rc) return sync_fail(rc);
    } else {
        // launch_tpp zeroes the work counter itself (ctl[0], on s_k, before the kernel)
        int rc = launch_tpp(s, d, ke, p, d.ref_scratch[0], ke->dtype_bits, ctl, s_k);
        if (rc) return sync_fail(rc);
        note_kernel(s, ke->name);
    }
    RT(cudaEventRecord(d.k1[0], s_k));
    for (int c = 0; c < nch; ++c) {
        const int c0 = bounds[c], c1 = bounds[c + 1], cn = c1 - c0;
        const size_t g0 = (size_t)lo + c0;
        DRV(ops.wait(reinterpret_cast<CUstream>(s_out), reinterpret_cast<CUdeviceptr>(ctl + 2 + c), (cuuint32_t)cn, CU_STREAM_WAIT_VALUE_GEQ), "cuStreamWaitValue32");
        RT(cudaMemcpyAsync(out.x + sx * g0, (float*)d.x.p + sx * c0, sizeof(float) * sx * cn, cudaMemcpyDeviceToHost, s_out));
        RT(cudaMemcpyAsync(out.u + su * g0, (float*)d.u.p + su * c0, sizeof(float) * su * cn, cudaMemcpyDeviceToHost, s_out));
        RT(cudaMemcpyAsync(out.iter + g0, (int*)d.iter.p + c0, sizeof(int) * cn, cudaMemcpyDeviceToHost, s_out));
        RT(cudaMemcpyAsync(out.status + g0, (int*)d.status.p + c0, sizeof(int) * cn, cudaMemcpyDeviceToHost, s_out));
        if (out.residuals) RT(cudaMemcpyAsync(out.residuals + 4 * g0, (float*)d.res.p + 4 * (size_t)c0, sizeof(float) * 4 * cn, cudaMemcpyDeviceToHost, s_out));
        if (out.rho) RT(cudaMemcpyAsync(out.rho + g0, (float*)d.rho.p + c0, sizeof(float) * cn, cudaMemcpyDeviceToHost, s_out));
    }
#undef DRV
#undef RT
    for (int k = 0; k < kStreams; ++k) CU(s, cudaStreamSynchronize(d.streams[k]));
    float ms = 0;
    CU(s, cudaEventElapsedTime(&ms, d.k0[0], d.k1[0]));
    *kernel_ms = ms;
    *nchunks_out = nch;
    if (ke64) {
        int q = 0;
        CU(s, cudaMemcpy(&q, d.qctl, sizeof(int), cudaMemcpyDeviceToHost));
        *marked_out = q;
    }
    return TINYMPC_CUDA_OK;
}

// Upload plan of the compact streamed pipeline for a shard of n problems.  bounds: chunk c = problems [bounds[c], bounds[c + 1]),
// runs of granules of a multiple of 32 problems (no 128-byte line holds inputs of two chunks, see run_shard_streamed); chunks <= 0
// (auto): 1, 1, 2, 4, 8, ... sixty-fourths of the shard, so that the kernel starts after 1/64 of the upload; chunks = k > 1: k equal
// chunks.  Returns the first chunk that is claimed through an ordered list when claim order applies: the chunks before it cover
// at most n / div problems (but always the first chunk).
int plan_compact_chunks(int n, int chunks, int div, std::vector<int>& bounds) {
    const bool ramp = chunks <= 0;
    const int ng_target = ramp ? kMaxGranules : std::min(chunks, kMaxGranules);
    const int gran = (((n + ng_target - 1) / ng_target) + 31) & ~31;
    const int ng = (n + gran - 1) / gran;
    bounds.clear();
    bounds.push_back(0);
    int g = 0, run = 1;
    while (g < ng) {
        g = std::min(ng, g + run);
        bounds.push_back(std::min(n, g * gran));
        if (ramp && bounds.size() > 2) run *= 2;
    }
    const int nch = (int)bounds.size() - 1;
    int first_ordered = 1;
    while (first_ordered < nch - 1 && bounds[first_ordered + 1] <= n / std::max(2, div)) ++first_ordered;
    return first_ordered;
}

// Compact host I/O (x0 + one reference state per problem in, u0 + iter + status out: ~120 bytes per problem) as ONE launch chain.
// The chunked pipeline pays for every chunk a partial last wave of the persistent kernel and the latency-bound end of its fp64
// pass, and its first launch waits for the first chunk's upload; here stream 0 uploads the inputs in a few chunks of doubling
// size, each followed by a write of the arrival watermark, and stream 1 runs the solve over the WHOLE shard -- first kernel
// (lanes start a claimed problem once the watermark covers it), then, in the exact-count mode, compaction + fp64 pass, then the
// result copies.  Kernels with KernelEntry::compact_ok read the compact reference in place and write the first control alone,
// so no expansion kernel has to find room next to a persistent launch that waits for it, and there is no trajectory scratch and
// no gather.  The link delivers ~55 GB/s, the kernel consumes ~7: after the first chunk (1/64 of the shard) the upload is
// hidden, and what is left of the bus is the 24 bytes per problem that come back (0.45 ms per 2^20 problems).  Enqueue order as
// in run_shard_streamed: every copy the kernel waits for is enqueued before its launch.
// Measured (quadrotor, 2^20 problems, exact-count mode, profiles/r02/e2e_compact_sweep*.jsonl): chunked pipeline with expansion /
// gather kernels 17.1 ms end to end -> 15.1 ms as one launch chain -> 14.8 ms with the result copies under the fp64 pass (below)
// -> 14.4 ms with the second half of the shard claimed hardest-first (below), against 14.1 ms of kernels.
int run_shard_compact_streamed(tinympc_cuda_solver* s, DeviceCtx& d, const KernelEntry* ke, const KernelEntry* ke64, const tinympc_cuda_batch_in& in,
                               const tinympc_cuda_batch_out& out, int lo, int hi, double* kernel_ms, int* nchunks_out, long long* marked_out) {
    const Family& f = s->fam;
    const StreamMemOps& ops = stream_memops();
    const int n = hi - lo;
    const size_t sx = (size_t)f.nx * f.N, su = (size_t)f.nu * (f.N - 1);
    const bool ppb = in.x_min != nullptr;
    const bool mixed = ke64 != nullptr;
    std::vector<int> bounds;
    const int plan_first_ordered = plan_compact_chunks(n, s->chunks, s->order_from_div, bounds);
    const int nch = (int)bounds.size() - 1;
    cudaStream_t s_in = d.streams[0], s_k = d.streams[1];
    int* ctl = d.stream_ctl;   // [0] work counter of the first kernel, [1] arrival watermark
    CU(s, cudaMemsetAsync(ctl, 0, sizeof(int) * 2, s_k));
    CU(s, cudaEventRecord(d.ev_ctl, s_k));
    CU(s, cudaStreamWaitEvent(s_in, d.ev_ctl, 0));
    // kernels that write the first control alone (KernelEntry::compact_ok) need no trajectory scratch and no gather
    const bool u0_direct = s->compact_in_kernel && out.u0 && !out.x && !out.u && ke->compact_ok && (!mixed || ke64->compact_ok);
    if (!u0_direct) {
        if (!out.x) CU(s, d.exp_x[0].reserve(sizeof(float) * sx * n));
        if (!out.u) CU(s, d.exp_u[0].reserve(sizeof(float) * su * n));
    }
    DevBuf& list = d.marked[0];
    if (mixed) CU(s, list.reserve(sizeof(int) * (size_t)n));
    // Exact-count mode with compact output into PINNED host arrays: all but the ~1 % of marked problems is final after the first
    // pass, so the result copies (the whole D2H volume) start then, on the third stream, under the fp64 pass; once both are done a
    // small kernel writes the fp64 pass's results over them through the device alias of the host arrays.  (Scattering a packed
    // result list on the host instead was tried: ~14 000 entries over three 4-17 MB arrays cost more than the copies hide.)
    void *hu0 = nullptr, *hiter = nullptr, *hstatus = nullptr;
    const bool early = mixed && u0_direct && s->compact_early_d2h && !out.residuals && !out.rho &&
                       host_alias(out.u0, &hu0) && host_alias(out.iter, &hiter) && host_alias(out.status, &hstatus);
    const int bits = ke->dtype_bits;
    SolveParams p = f.base;
    p.pack = bits == 64 ? (const void*)((const double*)d.pack64 + f.L.cold) : (const void*)((const float*)d.pack32 + f.L.cold);
    p.pack_elems = f.L.cold_size;
    p.batch = n;
    p.x0 = (const float*)d.x0.p;
    p.Xref = in.xref_const ? (const float*)d.xrc.p : (in.Xref ? (const float*)d.Xref.p : nullptr);
    p.xref_const = in.xref_const ? 1 : 0;
    p.Uref = in.Uref ? (const float*)d.Uref.p : nullptr;
    if (ppb) { p.x_min = (const float*)d.xmin.p; p.x_max = (const float*)d.xmax.p; p.u_min = (const float*)d.umin.p; p.u_max = (const float*)d.umax.p; }
    if (u0_direct) {
        p.x = nullptr; p.u = nullptr; p.u0 = (float*)d.u0.p;
    } else {
        p.x = out.x ? (float*)d.x.p : (float*)d.exp_x[0].p;
        p.u = out.u ? (float*)d.u.p : (float*)d.exp_u[0].p;
    }
    p.iter = (int*)d.iter.p; p.status = (int*)d.status.p;
    p.residuals = out.residuals ? (float*)d.res.p : nullptr;
    p.rho_out = out.rho ? (float*)d.rho.p : nullptr;
    p.avail_ptr = ctl + 1;

    auto sync_fail = [&](int rc) -> int { cudaDeviceSynchronize(); return rc; };
#define RT(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return sync_fail(cuda_fail(s, e__, #call)); } while (0)
    // Claim order (option "order", order_count_kernel): the chunks of the first half of the shard are claimed in index order as they
    // arrive; a later chunk is bucketed by expected difficulty as soon as it has landed -- on the third stream, on the SM the
    // persistent launch leaves free for it -- and claimed hardest-first through its part of the list (SolveParams::order_from); the
    // watermark moves past such a chunk when its list is written.  With the default chunks that is the last chunk, half the shard:
    // listed ~1.5 ms after it landed, long before the lanes get there, and ending on its easiest problems, the tail of the launch.
    // Measured on 2^20 problems (profiles/r02/order_streamed_*.jsonl): quadrotor 14.80 -> 14.35 ms end to end; the 4-state cartpole
    // loses 1 % (its solve is too short for the ordered half to pay for the SM), hence nx >= 8.  The device-resident entry orders
    // the whole batch before the launch and gains 7-9 % on both.
    int reserve = 0, first_ordered = nch;
    int *ohist = nullptr, *olist = nullptr;
    unsigned char* obucket = nullptr;
    if (s->order && ke->order_from_ok && bits == 32 && f.feat == kFeatBox && !ppb && f.shared_bounds_ok && p.en_input_bound &&
        f.nx >= 8 && f.nx <= 16 && f.nu <= 8 && n >= (1 << 18) && nch >= 3 && nch <= kMaxGranules) {
        first_ordered = plan_first_ordered;
        int rc = reserve_order(s, d, n, &ohist, &olist, &obucket);
        if (rc) return sync_fail(rc);
        p.index_list = olist;                       // entry (c - order_from) for work item c
        p.order_from = bounds[first_ordered];
        reserve = std::max(1, s->order_sms);        // SMs for the ordering kernels
    }
    cudaStream_t s_ord = d.streams[2];
    for (int c = 0; c < nch; ++c) {
        const int c0 = bounds[c], c1 = bounds[c + 1], cn = c1 - c0;
        const size_t g0 = (size_t)lo + c0;
        auto h2d = [&](DevBuf& dst, const float* src, size_t per_problem) -> cudaError_t {
            return cudaMemcpyAsync((float*)dst.p + per_problem * c0, src + per_problem * g0, sizeof(float) * per_problem * cn, cudaMemcpyHostToDevice, s_in);
        };
        RT(h2d(d.x0, in.x0, f.nx));
        if (in.xref_const) RT(h2d(d.xrc, in.xref_const, f.nx));
        if (in.Xref) RT(h2d(d.Xref, in.Xref, sx));
        if (in.Uref) RT(h2d(d.Uref, in.Uref, su));
        if (ppb) { RT(h2d(d.xmin, in.x_min, sx)); RT(h2d(d.xmax, in.x_max, sx)); RT(h2d(d.umin, in.u_min, su)); RT(h2d(d.umax, in.u_max, su)); }
        cudaStream_t s_w = s_in;                    // the stream that publishes the chunk
        if (c >= first_ordered) {
            // (the events of the chunked pipeline are idle here; the watermark writes of the ordered chunks follow those of the
            // chunks before them: s_ord waits for an event recorded behind them)
            RT(cudaEventRecord(d.k1[c], s_in));
            RT(cudaStreamWaitEvent(s_ord, d.k1[c], 0));
            int rc = build_order_range(s, p, c0, cn, ohist + (size_t)kOrderBuckets * c, olist + (c0 - p.order_from), obucket + c0, s_ord);
            if (rc) return sync_fail(rc);
            s_w = s_ord;
        }
        CUresult r = ops.write(reinterpret_cast<CUstream>(s_w), reinterpret_cast<CUdeviceptr>(ctl + 1), (cuuint32_t)c1, 0);
        if (r != CUDA_SUCCESS) return sync_fail(fail(s, TINYMPC_CUDA_ECUDA, "cuStreamWriteValue32 failed with CUresult " + std::to_string((int)r)));
    }
    RT(cudaEventRecord(d.k0[0], s_k));
    int* const n_marked = d.counters + 2 * kMaxChunks;
    if (!mixed) {
        int rc = launch_tpp(s, d, ke, p, d.ref_scratch[0], bits, ctl, s_k, reserve);
        if (rc) return sync_fail(rc);
        note_kernel(s, ke->name);
    } else {   // sequential exact-count form (enqueue()): fp32 pass that marks, compaction, fp64 re-solve of the marked problems
        p.amb_band = static_cast<float>(s->mixed_band);
        int rc = launch_tpp(s, d, ke, p, d.ref_scratch[0], 32, ctl, s_k, reserve);
        if (rc) return sync_fail(rc);
        if (early) {
            cudaStream_t s_out = d.streams[2];
            RT(cudaEventRecord(d.ev_pass, s_k));
            RT(cudaStreamWaitEvent(s_out, d.ev_pass, 0));
            RT(cudaMemcpyAsync(out.u0 + (size_t)f.nu * lo, d.u0.p, sizeof(float) * f.nu * n, cudaMemcpyDeviceToHost, s_out));
            RT(cudaMemcpyAsync(out.iter + lo, d.iter.p, sizeof(int) * n, cudaMemcpyDeviceToHost, s_out));
            RT(cudaMemcpyAsync(out.status + lo, d.status.p, sizeof(int) * n, cudaMemcpyDeviceToHost, s_out));
            RT(cudaEventRecord(d.ev_copied, s_out));
        }
        RT(cudaMemsetAsync(n_marked, 0, sizeof(int), s_k));
        collect_marked_kernel<<<(n + 255) / 256, 256, 0, s_k>>>(p.status, n, static_cast<int*>(list.p), n_marked);
        RT(cudaGetLastError());
        s->launches += 1;
        SolveParams p2 = p;
        p2.pack = (const void*)((const double*)d.pack64 + f.L.cold);
        p2.amb_band = 0.f;
        p2.avail_ptr = nullptr;            // the first pass has seen every problem
        p2.order_from = 0;
        p2.index_list = static_cast<const int*>(list.p);
        p2.batch_ptr = n_marked;
        rc = launch_tpp(s, d, ke64, p2, d.ref_scratch64[0], 64, d.counters + kMaxChunks, s_k);
        if (rc) return sync_fail(rc);
        note_kernel(s, std::string(ke->name) + "+" + ke64->name);
    }
    if (out.u0 && !u0_direct) {
        const size_t total = (size_t)f.nu * n;
        gather_u0_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s_k>>>(p.u, (float*)d.u0.p, total, f.nu, (int)su);
        RT(cudaGetLastError());
        s->launches += 1;
    }
    RT(cudaEventRecord(d.k1[0], s_k));
    if (early) {
        RT(cudaStreamWaitEvent(s_k, d.ev_copied, 0));
        scatter_marked_to_host_kernel<<<32, 256, 0, s_k>>>(static_cast<const int*>(list.p), n_marked, p.iter, p.status, p.u0, f.nu,
                                                           static_cast<int*>(hiter) + lo, static_cast<int*>(hstatus) + lo,
                                                           static_cast<float*>(hu0) + (size_t)f.nu * lo);
        RT(cudaGetLastError());
        s->launches += 1;
    } else {
        if (out.x) RT(cudaMemcpyAsync(out.x + sx * lo, d.x.p, sizeof(float) * sx * n, cudaMemcpyDeviceToHost, s_k));
        if (out.u) RT(cudaMemcpyAsync(out.u + su * lo, d.u.p, sizeof(float) * su * n, cudaMemcpyDeviceToHost, s_k));
        if (out.u0) RT(cudaMemcpyAsync(out.u0 + (size_t)f.nu * lo, d.u0.p, sizeof(float) * f.nu * n, cudaMemcpyDeviceToHost, s_k));
        RT(cudaMemcpyAsync(out.iter + lo, d.iter.p, sizeof(int) * n, cudaMemcpyDeviceToHost, s_k));
        RT(cudaMemcpyAsync(out.status + lo, d.status.p, sizeof(int) * n, cudaMemcpyDeviceToHost, s_k));
        if (out.residuals) RT(cudaMemcpyAsync(out.residuals + 4 * (size_t)lo, d.res.p, sizeof(float) * 4 * n, cudaMemcpyDeviceToHost, s_k));
        if (out.rho) RT(cudaMemcpyAsync(out.rho + lo, d.rho.p, sizeof(float) * n, cudaMemcpyDeviceToHost, s_k));
    }
#undef RT
    for (int k = 0; k < kStreams; ++k) CU(s, cudaStreamSynchronize(d.streams[k]));
    float ms = 0;
    CU(s, cudaEventElapsedTime(&ms, d.k0[0], d.k1[0]));
    *kernel_ms = ms;
    *nchunks_out = nch;
    if (mixed) {
        int q = 0;
        CU(s, cudaMemcpy(&q, n_marked, sizeof(int), cudaMemcpyDeviceToHost));
        *marked_out = q;
    }
    return TINYMPC_CUDA_OK;
}

// Host batch calls are serialised per device within the process.  Every pipeline below ends in a persistent launch that wants the
// whole GPU, so two of them on one device (two solver handles, or one handle created with the same device twice) gain nothing from
// running together -- and the compact streamed pipeline with claim order relies on the SM its launch leaves free staying free
// for its ordering kernels: another persistent launch of ours would take it and both would wait for ordering kernels that can
// never be scheduled.
std::mutex& device_call_mutex(int device) {
    static std::mutex mu[64];
    return mu[device & 63];
}

// One device's share of a host batch: chunked H2D -> kernel -> D2H pipeline over kStreams streams.  models (host pointers): a model
// batch, whose model arrays travel chunk by chunk with the inputs.
int run_shard(tinympc_cuda_solver* s, DeviceCtx& d, const tinympc_cuda_batch_in& in, const tinympc_cuda_batch_out& out, int lo, int hi,
              double* kernel_ms, int* nchunks_out, long long* marked_out, const tinympc_cuda_models* models) {
    const Family& f = s->fam;
    const int n = hi - lo;
    *kernel_ms = 0; *nchunks_out = 0; *marked_out = 0;
    if (n <= 0) return TINYMPC_CUDA_OK;
    std::lock_guard<std::mutex> one_call_per_device(device_call_mutex(d.device));
    CU(s, cudaSetDevice(d.device));
    const size_t sx = (size_t)f.nx * f.N, su = (size_t)f.nu * (f.N - 1);
    const bool ppb = in.x_min != nullptr;
    CU(s, d.x0.reserve(sizeof(float) * f.nx * (size_t)n));
    if (in.Xref) CU(s, d.Xref.reserve(sizeof(float) * sx * n));
    if (in.Uref) CU(s, d.Uref.reserve(sizeof(float) * su * n));
    if (ppb) {
        CU(s, d.xmin.reserve(sizeof(float) * sx * n)); CU(s, d.xmax.reserve(sizeof(float) * sx * n));
        CU(s, d.umin.reserve(sizeof(float) * su * n)); CU(s, d.umax.reserve(sizeof(float) * su * n));
    }
    const bool compact = in.xref_const || !(out.x && out.u);   // compact I/O goes through the chunked pipeline (the bus is no longer the limit)
    if (in.xref_const) CU(s, d.xrc.reserve(sizeof(float) * f.nx * (size_t)n));
    if (out.x) CU(s, d.x.reserve(sizeof(float) * sx * n));
    if (out.u) CU(s, d.u.reserve(sizeof(float) * su * n));
    if (out.u0) CU(s, d.u0.reserve(sizeof(float) * f.nu * (size_t)n));
    CU(s, d.iter.reserve(sizeof(int) * (size_t)n)); CU(s, d.status.reserve(sizeof(int) * (size_t)n));
    if (out.residuals) CU(s, d.res.reserve(sizeof(float) * 4 * (size_t)n));
    if (out.rho) CU(s, d.rho.reserve(sizeof(float) * (size_t)n));
    ModelField mf[kModelFields];
    if (models) {
        model_fields(f.nx, f.nu, f.base.adaptive_rho != 0, mf);
        for (int k = 0; k < kModelFields; ++k)
            if (models->*mf[k].field) CU(s, d.models[k].reserve(sizeof(double) * mf[k].per_problem * (size_t)n));
    }

    // single-launch streamed pipeline: a thread-per-problem kernel that honours the watermark; in the exact-count mode the
    // concurrent producer / consumer pair (both count completions per chunk)
    const bool mixed = s->mixed_band > 0 && s->precision == 32;
    if (!models && s->streamed && !compact && !(mixed && s->fixer_sms == -1) && !s->force_wpp && stream_memops().ok) {
        const KernelEntry* ke = pick_kernel(s, d, f, s->precision, ppb, in.Xref || in.Uref, n);
        const KernelEntry* ke64 = mixed ? find_kernel(f, 64, ppb, in.Xref || in.Uref, 0) : nullptr;
        // auto (0): the ramped chunk layout for shards of >= 2^16 problems, else equal chunks of >= 2^14 problems
        int nst = s->chunks > 0 ? std::min(s->chunks, kMaxGranules) : (n >= (1 << 16) ? 0 : n / 16384);
        if (ke && ke->streaming && (!mixed || (ke64 && ke64->streaming)) && (nst == 0 || nst >= 2) && (ppb || f.shared_bounds_ok))
            return run_shard_streamed(s, d, ke, ke64, in, out, lo, hi, nst, kernel_ms, nchunks_out, marked_out);
    }
    // compact I/O: one launch chain behind an arrival watermark, when the kernels of the batch wait for the watermark and read
    // the compact reference in place (chunks = 1 keeps the single chunked launch, fixer_sms >= 0 the concurrent exact-count pair)
    if (!models && compact && s->compact_streamed && !s->force_wpp && stream_memops().ok && !(mixed && s->fixer_sms >= 0) &&
        (s->chunks >= 2 || (s->chunks <= 0 && n >= (1 << 16))) && (ppb || f.shared_bounds_ok)) {
        const KernelEntry *ke = nullptr, *ke64 = nullptr;
        const bool refs = in.xref_const || in.Xref || in.Uref;
        // a compact reference must be read in place: an expansion kernel could not run next to the persistent launch that waits for it
        const bool ck = compact_in_kernel(s, d, ppb, refs, n, &ke, &ke64);
        const bool ok = in.xref_const ? ck : (ke && (!mixed || ke64));
        if (ok && ke->streaming && ke->family == KF_TPP)
            return run_shard_compact_streamed(s, d, ke, mixed ? ke64 : nullptr, in, out, lo, hi, kernel_ms, nchunks_out, marked_out);
    }
    // chunking: enough chunks to overlap copies with compute, each still many waves of the GPU.  Compact I/O moves ~120 bytes per
    // problem, so there is next to nothing to overlap and every extra chunk costs a partial last wave of the persistent kernel plus
    // the latency-bound end of its fp64 pass: two chunks, a short first one (its upload is all that precedes the first launch).
    std::vector<int> cuts;   // chunk c = [cuts[c], cuts[c + 1])
    if (s->chunks <= 0 && compact) {
        cuts.push_back(0);
        if (n >= (1 << 17)) cuts.push_back((n / 8 + 3) & ~3);
        cuts.push_back(n);
    } else {
        int nch0 = s->chunks > 0 ? s->chunks : (n >= (1 << 17) ? 8 : (n >= (1 << 15) ? 4 : 1));
        nch0 = std::min(nch0, kMaxChunks);
        int per = (n + nch0 - 1) / nch0;
        per = (per + 3) & ~3;                     // keeps every chunk's arrays 16 B aligned for all shapes
        for (int c0 = 0; c0 < n; c0 += per) cuts.push_back(c0);
        cuts.push_back(n);
    }
    const int nch = (int)cuts.size() - 1;
    for (int c = 0; c < nch; ++c) {
        const int c0 = cuts[c], c1 = cuts[c + 1], cn = c1 - c0;
        cudaStream_t st = d.streams[c % kStreams];
        const size_t g0 = (size_t)lo + c0;    // global problem index of the chunk start
        auto h2d = [&](DevBuf& dst, const float* src, size_t per_problem) -> cudaError_t {
            return cudaMemcpyAsync((float*)dst.p + per_problem * c0, src + per_problem * g0, sizeof(float) * per_problem * cn,
                                   cudaMemcpyHostToDevice, st);
        };
        CU(s, h2d(d.x0, in.x0, f.nx));
        if (in.Xref) CU(s, h2d(d.Xref, in.Xref, sx));
        if (in.xref_const) CU(s, h2d(d.xrc, in.xref_const, f.nx));
        if (in.Uref) CU(s, h2d(d.Uref, in.Uref, su));
        if (ppb) { CU(s, h2d(d.xmin, in.x_min, sx)); CU(s, h2d(d.xmax, in.x_max, sx)); CU(s, h2d(d.umin, in.u_min, su)); CU(s, h2d(d.umax, in.u_max, su)); }
        tinympc_cuda_batch_in din{};
        din.batch = cn;
        din.x0 = (float*)d.x0.p + (size_t)f.nx * c0;
        din.Xref = in.Xref ? (float*)d.Xref.p + sx * c0 : nullptr;
        din.xref_const = in.xref_const ? (float*)d.xrc.p + (size_t)f.nx * c0 : nullptr;
        din.Uref = in.Uref ? (float*)d.Uref.p + su * c0 : nullptr;
        if (ppb) {
            din.x_min = (float*)d.xmin.p + sx * c0; din.x_max = (float*)d.xmax.p + sx * c0;
            din.u_min = (float*)d.umin.p + su * c0; din.u_max = (float*)d.umax.p + su * c0;
        }
        tinympc_cuda_batch_out dout{};
        dout.x = out.x ? (float*)d.x.p + sx * c0 : nullptr; dout.u = out.u ? (float*)d.u.p + su * c0 : nullptr;
        dout.u0 = out.u0 ? (float*)d.u0.p + (size_t)f.nu * c0 : nullptr;
        dout.iter = (int*)d.iter.p + c0; dout.status = (int*)d.status.p + c0;
        dout.residuals = out.residuals ? (float*)d.res.p + 4 * (size_t)c0 : nullptr;
        dout.rho = out.rho ? (float*)d.rho.p + c0 : nullptr;
        tinympc_cuda_models dm{};
        if (models)
            for (int k = 0; k < kModelFields; ++k)
                if (const double* src = models->*mf[k].field) {
                    const size_t per_problem = mf[k].per_problem;
                    double* dst = static_cast<double*>(d.models[k].p) + per_problem * c0;
                    CU(s, cudaMemcpyAsync(dst, src + per_problem * g0, sizeof(double) * per_problem * cn, cudaMemcpyHostToDevice, st));
                    dm.*mf[k].field = dst;
                }
        CU(s, cudaEventRecord(d.k0[c], st));
        int rc = enqueue(s, d, din, dout, c, st, c % kStreams, 0, models ? &dm : nullptr);
        if (rc) return rc;
        CU(s, cudaEventRecord(d.k1[c], st));
        if (out.x) CU(s, cudaMemcpyAsync(out.x + sx * g0, dout.x, sizeof(float) * sx * cn, cudaMemcpyDeviceToHost, st));
        if (out.u) CU(s, cudaMemcpyAsync(out.u + su * g0, dout.u, sizeof(float) * su * cn, cudaMemcpyDeviceToHost, st));
        if (out.u0) CU(s, cudaMemcpyAsync(out.u0 + (size_t)f.nu * g0, dout.u0, sizeof(float) * f.nu * cn, cudaMemcpyDeviceToHost, st));
        CU(s, cudaMemcpyAsync(out.iter + g0, dout.iter, sizeof(int) * cn, cudaMemcpyDeviceToHost, st));
        CU(s, cudaMemcpyAsync(out.status + g0, dout.status, sizeof(int) * cn, cudaMemcpyDeviceToHost, st));
        if (out.residuals) CU(s, cudaMemcpyAsync(out.residuals + 4 * g0, dout.residuals, sizeof(float) * 4 * cn, cudaMemcpyDeviceToHost, st));
        if (out.rho) CU(s, cudaMemcpyAsync(out.rho + g0, dout.rho, sizeof(float) * cn, cudaMemcpyDeviceToHost, st));
    }
    for (int k = 0; k < kStreams; ++k) CU(s, cudaStreamSynchronize(d.streams[k]));
    for (int c = 0; c < nch; ++c) {
        float ms = 0;
        CU(s, cudaEventElapsedTime(&ms, d.k0[c], d.k1[c]));
        *kernel_ms += ms;
    }
    *nchunks_out = nch;
    if (s->mixed_band > 0 && s->precision == 32) {
        long long tot = 0;
        if (s->fixer_sms >= 0) {
            int q[4 * kMaxChunks];
            CU(s, cudaMemcpy(q, d.qctl, sizeof(int) * 4 * nch, cudaMemcpyDeviceToHost));
            for (int c = 0; c < nch; ++c) tot += q[4 * c];
        } else {
            int counts[kMaxChunks];
            CU(s, cudaMemcpy(counts, d.counters + 2 * kMaxChunks, sizeof(int) * nch, cudaMemcpyDeviceToHost));
            for (int c = 0; c < nch; ++c) tot += counts[c];
        }
        *marked_out = tot;
    }
    return TINYMPC_CUDA_OK;
}

}  // namespace

extern "C" {

int tinympc_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char* tinympc_cuda_version(void) { return "tinympc-b200 0.1 (sm_100a)"; }

int tinympc_cuda_create(tinympc_cuda_solver** out, const int* devices, int n_devices) {
    if (!out) return TINYMPC_CUDA_EINVAL;
    *out = nullptr;
    const int have = tinympc_cuda_device_count();
    if (have <= 0) return TINYMPC_CUDA_ENODEVICE;
    auto* s = new tinympc_cuda_solver();
    // environment override of the "streamed" option (0 = one launch per chunk), e.g. for tools that cannot follow a kernel
    // that consumes data while it is still arriving
    if (const char* e = std::getenv("TINYMPC_B200_STREAMED")) s->streamed = std::atoi(e) != 0;
    std::vector<int> ids;
    if (n_devices <= 0 || !devices) {
        int cur = 0;
        cudaGetDevice(&cur);
        ids.push_back(cur);
    } else {
        for (int i = 0; i < n_devices; ++i) {
            if (devices[i] < 0 || devices[i] >= have) { delete s; return TINYMPC_CUDA_EINVAL; }
            ids.push_back(devices[i]);
        }
    }
    int prev = 0;
    cudaGetDevice(&prev);
    for (int id : ids) {
        DeviceCtx d;
        d.device = id;
        if (cudaSetDevice(id) != cudaSuccess) { delete s; return TINYMPC_CUDA_ECUDA; }
        cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, id);
        if (cudaMalloc(&d.counters, sizeof(int) * 3 * kMaxChunks) != cudaSuccess) { delete s; return TINYMPC_CUDA_ECUDA; }
        if (cudaMalloc(&d.stream_ctl, sizeof(int) * (2 + kMaxStreamChunks)) != cudaSuccess) { delete s; return TINYMPC_CUDA_ECUDA; }
        if (cudaMalloc(&d.qctl, sizeof(int) * 4 * kMaxChunks) != cudaSuccess) { delete s; return TINYMPC_CUDA_ECUDA; }
        for (int k = 0; k <= kStreams; ++k) {
            cudaStreamCreateWithFlags(&d.fix_stream[k], cudaStreamNonBlocking);
            cudaEventCreateWithFlags(&d.ev_fork[k], cudaEventDisableTiming);
            cudaEventCreateWithFlags(&d.ev_join[k], cudaEventDisableTiming);
        }
        cudaEventCreateWithFlags(&d.ev_ctl, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&d.ev_pass, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&d.ev_copied, cudaEventDisableTiming);
        cudaEventCreate(&d.ev_p0); cudaEventCreate(&d.ev_p1); cudaEventCreate(&d.ev_p2);
        for (int k = 0; k < kStreams; ++k) cudaStreamCreateWithFlags(&d.streams[k], cudaStreamNonBlocking);
        for (int c = 0; c < kMaxChunks; ++c) { cudaEventCreate(&d.k0[c]); cudaEventCreate(&d.k1[c]); }
        d.events = true;
        s->devs.push_back(d);
    }
    cudaSetDevice(prev);
    *out = s;
    return TINYMPC_CUDA_OK;
}

int tinympc_cuda_destroy(tinympc_cuda_solver* s) {
    if (!s) return TINYMPC_CUDA_OK;
    int prev = 0;
    cudaGetDevice(&prev);
    // a session outliving its solver keeps its handle but loses its device state: every later call on it fails with
    // TINYMPC_CUDA_ENOTREADY instead of dereferencing the freed solver, and session_destroy still releases the handle
    for (tinympc_cuda_session* ss : s->sessions) {
        cudaSetDevice(s->devs[ss->dev].device);
        cudaStreamSynchronize(s->devs[ss->dev].streams[0]);   // work a device-resident session entry left queued
        for (DevBuf* b : {&ss->ws, &ss->pack, &ss->x, &ss->u, &ss->iter, &ss->status}) b->release();
        for (DevBuf& b : ss->mdl) b.release();
        for (cudaEvent_t* ev : {&ss->ev_in, &ss->ev_out}) if (*ev) { cudaEventDestroy(*ev); *ev = nullptr; }
        ss->s = nullptr;
    }
    s->sessions.clear();
    for (auto& d : s->devs) {
        cudaSetDevice(d.device);
        for (int k = 0; k < kStreams; ++k) if (d.streams[k]) { cudaStreamSynchronize(d.streams[k]); cudaStreamDestroy(d.streams[k]); }
        if (d.events) for (int c = 0; c < kMaxChunks; ++c) { cudaEventDestroy(d.k0[c]); cudaEventDestroy(d.k1[c]); }
        if (d.pack32) cudaFree(d.pack32);
        if (d.pack64) cudaFree(d.pack64);
        if (d.counters) cudaFree(d.counters);
        if (d.stream_ctl) cudaFree(d.stream_ctl);
        if (d.qctl) cudaFree(d.qctl);
        for (int k = 0; k <= kStreams; ++k) {
            if (d.fix_stream[k]) { cudaStreamSynchronize(d.fix_stream[k]); cudaStreamDestroy(d.fix_stream[k]); }
            if (d.ev_fork[k]) cudaEventDestroy(d.ev_fork[k]);
            if (d.ev_join[k]) cudaEventDestroy(d.ev_join[k]);
        }
        if (d.ev_ctl) cudaEventDestroy(d.ev_ctl);
        if (d.ev_pass) cudaEventDestroy(d.ev_pass);
        if (d.ev_copied) cudaEventDestroy(d.ev_copied);
        for (DevBuf* b : {&d.x0, &d.Xref, &d.Uref, &d.xmin, &d.xmax, &d.umin, &d.umax, &d.x, &d.u, &d.iter, &d.status, &d.res, &d.rho, &d.xrc, &d.u0}) b->release();
        for (auto& b : d.models) b.release();
        for (auto& b : d.exp_xref) b.release();
        for (auto& b : d.exp_x) b.release();
        for (auto& b : d.exp_u) b.release();
        for (auto& b : d.wpp_scratch) b.release();
        for (auto& b : d.ref_scratch) b.release();
        for (auto& b : d.ref_scratch64) b.release();
        for (auto& b : d.marked) b.release();
        d.order_buf.release();
    }
    cudaSetDevice(prev);
    delete s;
    return TINYMPC_CUDA_OK;
}

int tinympc_cuda_set_family(tinympc_cuda_solver* s, const tinympc_cuda_family* fm) {
    if (!s || !fm) return TINYMPC_CUDA_EINVAL;
    const int nx = fm->nx, nu = fm->nu, N = fm->N;
    if (nx < 1 || nu < 1 || N < 2) return fail(s, TINYMPC_CUDA_EINVAL, "need nx >= 1, nu >= 1, N >= 2");
    if (!fm->Adyn || !fm->Bdyn || !fm->Q || !fm->R || !fm->Kinf || !fm->Pinf || !fm->Quu_inv || !fm->AmBKt)
        return fail(s, TINYMPC_CUDA_EINVAL, "Adyn, Bdyn, Q, R, Kinf, Pinf, Quu_inv, AmBKt are required");
    if (fm->check_termination <= 0)
        return fail(s, TINYMPC_CUDA_EINVAL, "check_termination must be >= 1 (the reference divides by it, admm.cpp:255)");
    if (fm->numStateCones < 0 || fm->numInputCones < 0 || fm->numStateCones > TINYMPC_MAX_CONES || fm->numInputCones > TINYMPC_MAX_CONES)
        return fail(s, TINYMPC_CUDA_EINVAL, "at most TINYMPC_MAX_CONES cones per kind");
    for (int k = 0; k < fm->numStateCones; ++k)
        if (fm->qcx[k] < 1 || fm->Acx[k] < 0 || fm->Acx[k] + fm->qcx[k] > nx) return fail(s, TINYMPC_CUDA_EINVAL, "state cone outside [0, nx)");
    for (int k = 0; k < fm->numInputCones; ++k)
        if (fm->qcu[k] < 1 || fm->Acu[k] < 0 || fm->Acu[k] + fm->qcu[k] > nu) return fail(s, TINYMPC_CUDA_EINVAL, "input cone outside [0, nu)");
    if (fm->numStateLinear < 0 || fm->numInputLinear < 0) return fail(s, TINYMPC_CUDA_EINVAL, "negative linear row count");
    if (fm->en_state_linear && fm->numStateLinear > 0 && (!fm->Alin_x || !fm->blin_x)) return fail(s, TINYMPC_CUDA_EINVAL, "Alin_x/blin_x missing");
    if (fm->en_input_linear && fm->numInputLinear > 0 && (!fm->Alin_u || !fm->blin_u)) return fail(s, TINYMPC_CUDA_EINVAL, "Alin_u/blin_u missing");
    if (fm->adaptive_rho && (!fm->dKinf_drho || !fm->dPinf_drho)) return fail(s, TINYMPC_CUDA_EINVAL, "adaptive_rho needs dKinf_drho and dPinf_drho");

    Family f;
    f.nx = nx; f.nu = nu; f.N = N;
    const int nsl = fm->en_state_linear ? fm->numStateLinear : 0, nil = fm->en_input_linear ? fm->numInputLinear : 0;
    f.L = PackLayout::make(nx, nu, N, nsl, nil);
    const PackLayout& L = f.L;
    f.pack.assign(L.size, 0.0);
    put_rowmajor(f.pack, L.A, fm->Adyn, nx, nx);
    put_rowmajor(f.pack, L.B, fm->Bdyn, nx, nu);
    put_rowmajor(f.pack, L.Kinf, fm->Kinf, nu, nx);
    put_rowmajor(f.pack, L.AmBKt, fm->AmBKt, nx, nx);
    put_rowmajor(f.pack, L.Quu_inv, fm->Quu_inv, nu, nu);
    put_rowmajor(f.pack, L.Pinf, fm->Pinf, nx, nx);
    put_vec(f.pack, L.f, fm->fdyn, nx);
    put_vec(f.pack, L.APf, fm->APf, nx);
    put_vec(f.pack, L.BPf, fm->BPf, nu);
    put_vec(f.pack, L.Qd, fm->Q, nx);
    put_vec(f.pack, L.Rd, fm->R, nu);
    if (fm->adaptive_rho) {
        put_rowmajor(f.pack, L.dKinf, fm->dKinf_drho, nu, nx);
        put_rowmajor(f.pack, L.dPinf, fm->dPinf_drho, nx, nx);
    }
    // d0: backward_pass_grad (admm.cpp:13-20) on the zero workspace tiny_setup leaves (q = r = p = 0)
    {
        std::vector<double> p(nx, 0.0), pn(nx), t(nu);
        for (int i = N - 2; i >= 0; --i) {
            for (int a = 0; a < nu; ++a) {
                double acc = 0;
                for (int r = 0; r < nx; ++r) acc += f.pack[L.B + r * nu + a] * p[r];
                t[a] = acc + f.pack[L.BPf + a];
            }
            for (int a = 0; a < nu; ++a) {
                double acc = 0;
                for (int b = 0; b < nu; ++b) acc += f.pack[L.Quu_inv + a * nu + b] * t[b];
                f.pack[L.d0 + i * nu + a] = acc;
            }
            for (int c = 0; c < nx; ++c) {
                double acc = 0;
                for (int r = 0; r < nx; ++r) acc += f.pack[L.AmBKt + c * nx + r] * p[r];
                pn[c] = acc + f.pack[L.APf + c];
            }
            p = pn;
        }
    }
    // bounds: a disabled bound is an infinite box (clamping with +-inf is the identity)
    const double inf = std::numeric_limits<double>::infinity();
    const bool sb = fm->en_state_bound != 0, ib = fm->en_input_bound != 0;
    const bool have_sb = fm->x_min && fm->x_max, have_ib = fm->u_min && fm->u_max;
    for (int e = 0; e < nx * N; ++e) {
        f.pack[L.xmin + e] = (sb && have_sb) ? fm->x_min[e] : -inf;
        f.pack[L.xmax + e] = (sb && have_sb) ? fm->x_max[e] : inf;
    }
    for (int e = 0; e < nu * (N - 1); ++e) {
        f.pack[L.umin + e] = (ib && have_ib) ? fm->u_min[e] : -inf;
        f.pack[L.umax + e] = (ib && have_ib) ? fm->u_max[e] : inf;
    }
    f.shared_bounds_ok = (!sb || have_sb) && (!ib || have_ib);
    for (int r = 0; r < nx; ++r) f.affine = f.affine || f.pack[L.f + r] != 0.0 || f.pack[L.APf + r] != 0.0;
    for (int a = 0; a < nu; ++a) f.affine = f.affine || f.pack[L.BPf + a] != 0.0;
    f.a_pairs.assign(nx, 0u);
    a_pairs_of(f.pack.data() + L.A, nx, f.a_pairs.data());
    f.fastbox = true;
    for (int e = 0; e < nx * N && f.fastbox; ++e)
        f.fastbox = f.pack[L.xmin + e] == f.pack[L.xmin + e % nx] && f.pack[L.xmax + e] == f.pack[L.xmax + e % nx] &&
                    f.pack[L.xmin + e] <= 0.0 && f.pack[L.xmax + e] >= 0.0;
    for (int e = 0; e < nu * (N - 1) && f.fastbox; ++e)
        f.fastbox = f.pack[L.umin + e] == f.pack[L.umin + e % nu] && f.pack[L.umax + e] == f.pack[L.umax + e % nu] &&
                    f.pack[L.umin + e] <= 0.0 && f.pack[L.umax + e] >= 0.0;
    // linear rows + squared norms (project_hyperplane, admm.cpp:70-73)
    for (int k = 0; k < nsl; ++k) {
        double nr = 0;
        for (int j = 0; j < nx; ++j) { double a = fm->Alin_x[(size_t)j * fm->numStateLinear + k]; f.pack[L.Alin_x + k * nx + j] = a; nr += a * a; }
        f.pack[L.blin_x + k] = fm->blin_x[k];
        f.pack[L.nrm_x + k] = nr;
    }
    for (int k = 0; k < nil; ++k) {
        double nr = 0;
        for (int j = 0; j < nu; ++j) { double a = fm->Alin_u[(size_t)j * fm->numInputLinear + k]; f.pack[L.Alin_u + k * nu + j] = a; nr += a * a; }
        f.pack[L.blin_u + k] = fm->blin_u[k];
        f.pack[L.nrm_u + k] = nr;
    }

    SolveParams& b = f.base;
    b = SolveParams{};
    b.rho = fm->rho;
    b.abs_pri_tol = fm->abs_pri_tol; b.abs_dua_tol = fm->abs_dua_tol;
    b.max_iter = fm->max_iter; b.check_termination = fm->check_termination;
    b.en_state_bound = fm->en_state_bound; b.en_input_bound = fm->en_input_bound;
    b.en_state_soc = fm->en_state_soc; b.en_input_soc = fm->en_input_soc;
    b.adaptive_rho = fm->adaptive_rho;
    b.rho_min = fm->adaptive_rho_min; b.rho_max = fm->adaptive_rho_max; b.rho_clip = fm->adaptive_rho_enable_clipping;
    b.n_state_cones = fm->numStateCones; b.n_input_cones = fm->numInputCones;
    for (int k = 0; k < fm->numStateCones; ++k) { b.Acx[k] = fm->Acx[k]; b.qcx[k] = fm->qcx[k]; b.cx[k] = (float)fm->cx[k]; }
    for (int k = 0; k < fm->numInputCones; ++k) { b.Acu[k] = fm->Acu[k]; b.qcu[k] = fm->qcu[k]; b.cu[k] = (float)fm->cu[k]; }
    b.nsl = nsl; b.nil = nil;
    // NB: with en_*_linear set but zero rows the reference still adds the (vl - gl) = x term to q
    // (admm.cpp:138-140, 223-225); keep that by leaving the flag on with zero rows.
    b.en_state_linear = fm->en_state_linear; b.en_input_linear = fm->en_input_linear;

    const bool soc = (fm->en_state_soc && fm->numStateCones > 0) || (fm->en_input_soc && fm->numInputCones > 0);
    const bool lin = fm->en_state_linear || fm->en_input_linear;
    // adaptive rho together with cones / linear rows has no specialised kernel: feat 3 matches none, so the
    // general warp-per-problem kernel takes it
    f.feat = fm->adaptive_rho ? ((soc || lin) ? 3 : kFeatAdapt) : ((soc || lin) ? kFeatConstr : kFeatBox);
    f.set = true;
    s->fam = std::move(f);
    return upload_family(s);
}

}  // extern "C"

namespace {

// every required array of the family `f` present (adaptive rho: the two sensitivities too); device pointers 16-byte aligned
int check_model_arrays(tinympc_cuda_solver* s, const Family& f, const tinympc_cuda_models* m, bool device, const char* what) {
    ModelField mf[kModelFields];
    model_fields(f.nx, f.nu, f.base.adaptive_rho != 0, mf);
    for (int k = 0; k < kModelFields; ++k) {
        const double* p = m->*mf[k].field;
        if (mf[k].required && !p)
            return fail(s, TINYMPC_CUDA_EINVAL, std::string(what) + ": " + mf[k].name + " is required" +
                                                    (k >= 12 ? " (the family has adaptive_rho)" : ""));
        if (device && check_ptr16(s, p, mf[k].name)) return TINYMPC_CUDA_EINVAL;
    }
    return TINYMPC_CUDA_OK;
}
// model batches
int check_models(tinympc_cuda_solver* s, const tinympc_cuda_models* m, bool device) {
    if (!m) return TINYMPC_CUDA_OK;
    if (s->mixed_band > 0 && s->precision == 32)
        return fail(s, TINYMPC_CUDA_EUNSUPPORTED, "model batches have no exact-count (\"mixed\") form: use \"precision\" 64, which is exact for them");
    return check_model_arrays(s, s->fam, m, device, "model batch");
}

int solve_batch_device_common(tinympc_cuda_solver* s, int dev_index, const tinympc_cuda_models* m, const tinympc_cuda_batch_in* in,
                              const tinympc_cuda_batch_out* out, void* stream) {
    if (!s || !in || !out) return TINYMPC_CUDA_EINVAL;
    if (!s->fam.set) return fail(s, TINYMPC_CUDA_ENOTREADY, "tinympc_cuda_set_family has not been called");
    if (dev_index < 0 || dev_index >= (int)s->devs.size()) return fail(s, TINYMPC_CUDA_EINVAL, "dev_index out of range");
    if (in->batch < 0) return fail(s, TINYMPC_CUDA_EINVAL, "negative batch");
    if (in->batch == 0) return TINYMPC_CUDA_OK;
    if (!in->x0 || !out->iter || !out->status || !((out->x && out->u) || out->u0))
        return fail(s, TINYMPC_CUDA_EINVAL, "x0, iter, status and either (x, u) or u0 are required");
    int rc = check_models(s, m, true);
    if (rc) return rc;
    rc |= check_ptr16(s, in->xref_const, "xref_const"); rc |= check_ptr16(s, out->u0, "u0");
    rc |= check_ptr16(s, in->x0, "x0"); rc |= check_ptr16(s, in->Xref, "Xref"); rc |= check_ptr16(s, in->Uref, "Uref");
    rc |= check_ptr16(s, in->x_min, "x_min"); rc |= check_ptr16(s, in->x_max, "x_max"); rc |= check_ptr16(s, in->u_min, "u_min");
    rc |= check_ptr16(s, in->u_max, "u_max"); rc |= check_ptr16(s, out->x, "x"); rc |= check_ptr16(s, out->u, "u");
    rc |= check_ptr16(s, out->residuals, "residuals");
    if (rc) return TINYMPC_CUDA_EINVAL;
    DeviceCtx& d = s->devs[dev_index];
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DeviceGuard guard;                 // restores the caller's current device on every return path
    CU(s, cudaSetDevice(d.device));
    if (s->fam.base.max_iter <= 0 && !m) {   // a model batch runs the zero iterations in the kernel: every problem keeps its own rho
        rc = zero_iteration_result(s, s->fam, *out, in->batch, st, true);
    } else {
        // The last counter / scratch slot belongs to the device-resident entry point: ONE call in flight per device context
        // (include/tinympc_b200.h).  A second call on another stream would share the work counter and the scratch buffers.
        rc = enqueue(s, d, *in, *out, kMaxChunks - 1, st, kStreams, 0, m);
        s->mixed_pending_dev = (s->mixed_band > 0 && s->precision == 32) ? dev_index : -1;
    }
    return rc;
}

int solve_batch_common(tinympc_cuda_solver* s, const tinympc_cuda_models* m, const tinympc_cuda_batch_in* in, const tinympc_cuda_batch_out* out) {
    if (!s || !in || !out) return TINYMPC_CUDA_EINVAL;
    if (!s->fam.set) return fail(s, TINYMPC_CUDA_ENOTREADY, "tinympc_cuda_set_family has not been called");
    if (in->batch < 0) return fail(s, TINYMPC_CUDA_EINVAL, "negative batch");
    if (in->batch == 0) return TINYMPC_CUDA_OK;
    if (!in->x0 || !out->iter || !out->status || !((out->x && out->u) || out->u0))
        return fail(s, TINYMPC_CUDA_EINVAL, "x0, iter, status and either (x, u) or u0 are required");
    if (in->xref_const && in->Xref) return fail(s, TINYMPC_CUDA_EINVAL, "give Xref or xref_const, not both");
    const bool ppb = in->x_min || in->x_max || in->u_min || in->u_max;
    if (ppb && !(in->x_min && in->x_max && in->u_min && in->u_max))
        return fail(s, TINYMPC_CUDA_EINVAL, "per-problem bounds need all four of x_min, x_max, u_min, u_max");
    if (int rc = check_models(s, m, false)) return rc;
    if (s->fam.base.max_iter <= 0 && !m) return zero_iteration_result(s, s->fam, *out, in->batch, nullptr, false);

    const auto t0 = std::chrono::steady_clock::now();
    const int G = (int)s->devs.size();
    int prev = 0;
    cudaGetDevice(&prev);
    std::vector<int> rcs(G, 0), nch(G, 0);
    std::vector<double> kms(G, 0.0);
    std::vector<long long> marked(G, 0);
    // contiguous split by problem index (multiples of 4 keep every shard 16 B aligned), remainder to the last
    int per = ((in->batch + G - 1) / G + 3) & ~3;
    auto work = [&](int g) {
        const int lo = std::min(in->batch, g * per), hi = (g == G - 1) ? in->batch : std::min(in->batch, lo + per);
        rcs[g] = run_shard(s, s->devs[g], *in, *out, lo, hi, &kms[g], &nch[g], &marked[g], m);
    };
    if (G == 1) {
        work(0);
    } else {
        std::vector<std::thread> th;
        for (int g = 0; g < G; ++g) th.emplace_back(work, g);
        for (auto& t : th) t.join();
    }
    cudaSetDevice(prev);
    for (int g = 0; g < G; ++g) if (rcs[g]) return rcs[g];
    s->mixed_marked = 0;
    for (int g = 0; g < G; ++g) s->mixed_marked += marked[g];
    s->mixed_pending_dev = -1;
    s->t_kernel_ms = *std::max_element(kms.begin(), kms.end());
    s->t_chunks = *std::max_element(nch.begin(), nch.end());
    s->t_total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return TINYMPC_CUDA_OK;
}

}  // namespace

extern "C" {

int tinympc_cuda_solve_batch_device(tinympc_cuda_solver* s, int dev_index, const tinympc_cuda_batch_in* in, const tinympc_cuda_batch_out* out,
                                    void* stream) {
    return solve_batch_device_common(s, dev_index, nullptr, in, out, stream);
}

int tinympc_cuda_solve_batch(tinympc_cuda_solver* s, const tinympc_cuda_batch_in* in, const tinympc_cuda_batch_out* out) {
    return solve_batch_common(s, nullptr, in, out);
}

int tinympc_cuda_solve_batch_models_device(tinympc_cuda_solver* s, int dev_index, const tinympc_cuda_models* m, const tinympc_cuda_batch_in* in,
                                           const tinympc_cuda_batch_out* out, void* stream) {
    if (!m) return s ? fail(s, TINYMPC_CUDA_EINVAL, "model batch: models is NULL") : TINYMPC_CUDA_EINVAL;
    return solve_batch_device_common(s, dev_index, m, in, out, stream);
}

int tinympc_cuda_solve_batch_models(tinympc_cuda_solver* s, const tinympc_cuda_models* m, const tinympc_cuda_batch_in* in,
                                    const tinympc_cuda_batch_out* out) {
    if (!m) return s ? fail(s, TINYMPC_CUDA_EINVAL, "model batch: models is NULL") : TINYMPC_CUDA_EINVAL;
    return solve_batch_common(s, m, in, out);
}

int tinympc_cuda_solve_workspace(tinympc_cuda_solver* s, const tinympc_cuda_workspace* w) {
    if (!s || !w) return TINYMPC_CUDA_EINVAL;
    if (!s->fam.set) return fail(s, TINYMPC_CUDA_ENOTREADY, "tinympc_cuda_set_family has not been called");
    if (!w->x || !w->u || !w->q || !w->r || !w->p || !w->d || !w->v || !w->vnew || !w->z || !w->znew || !w->g || !w->y || !w->iter || !w->status)
        return fail(s, TINYMPC_CUDA_EINVAL, "workspace arrays x,u,q,r,p,d,v,vnew,z,znew,g,y and iter,status are required");
    const Family& f = s->fam;
    const int nx = f.nx, nu = f.nu, N = f.N, sx = nx * N, su = nu * (N - 1);
    const WppLayout W = WppLayout::make(nx, nu, N);
    std::vector<double> h(W.size, 0.0);
    auto put = [&](int at, const double* src, int n) { if (src) std::memcpy(h.data() + at, src, sizeof(double) * n); };
    put(W.x, w->x, sx); put(W.u, w->u, su); put(W.q, w->q, sx); put(W.r, w->r, su); put(W.p, w->p, sx); put(W.d, w->d, su);
    put(W.v, w->v, sx); put(W.vnew, w->vnew, sx); put(W.z, w->z, su); put(W.znew, w->znew, su); put(W.g, w->g, sx); put(W.y, w->y, su);
    put(W.vcnew, w->vcnew, sx); put(W.zcnew, w->zcnew, su); put(W.gc, w->gc, sx); put(W.yc, w->yc, su);
    put(W.vlnew, w->vlnew, sx); put(W.zlnew, w->zlnew, su); put(W.gl, w->gl, sx); put(W.yl, w->yl, su);
    put(W.Xref, w->Xref, sx); put(W.Uref, w->Uref, su);
    put(W.xmin, f.pack.data() + f.L.xmin, sx); put(W.xmax, f.pack.data() + f.L.xmax, sx);
    put(W.umin, f.pack.data() + f.L.umin, su); put(W.umax, f.pack.data() + f.L.umax, su);
    if (w->Kinf) { for (int a = 0; a < nu; ++a) for (int c = 0; c < nx; ++c) h[W.Kinf + a * nx + c] = w->Kinf[(size_t)c * nu + a]; }
    else put(W.Kinf, f.pack.data() + f.L.Kinf, nu * nx);
    if (w->Pinf) { for (int r = 0; r < nx; ++r) for (int c = 0; c < nx; ++c) h[W.Pinf + r * nx + c] = w->Pinf[(size_t)c * nx + r]; }
    else put(W.Pinf, f.pack.data() + f.L.Pinf, nx * nx);
    h[W.scalars + 0] = w->rho ? *w->rho : f.base.rho;
    if (w->residuals) for (int k = 0; k < 4; ++k) h[W.scalars + 3 + k] = w->residuals[k];

    DeviceCtx& d = s->devs[0];
    int prev = 0;
    cudaGetDevice(&prev);
    CU(s, cudaSetDevice(d.device));
    DevBuf& sb = d.wpp_scratch[kStreams];
    CU(s, sb.reserve(sizeof(double) * W.size));
    cudaStream_t st = d.streams[0];
    CU(s, cudaMemcpyAsync(sb.p, h.data(), sizeof(double) * W.size, cudaMemcpyHostToDevice, st));
    SolveParams p = f.base;
    p.batch = 1;
    if (w->rho) p.rho = *w->rho;
    // A box family of a compiled shape whose live cache is the family's own (no adaptive rho, no set_cache_terms override) runs the
    // lane-group kernel in session mode on this one workspace: ~2.5 us per ADMM iteration instead of ~10 (tmpc_gpp.cuh); every member
    // of the workspace comes back as the reference would leave it.
    auto same = [&](const double* a, int at, int rows, int cols) {   // a: column-major (Eigen) vs the row-major pack
        if (!a) return true;
        for (int r = 0; r < rows; ++r) for (int c = 0; c < cols; ++c) if (a[(size_t)c * rows + r] != f.pack[at + r * cols + c]) return false;
        return true;
    };
    const KernelEntry* kg = (!s->force_wpp && f.feat == kFeatBox && f.shared_bounds_ok && p.max_iter > 0 && p.rho == f.base.rho &&
                             same(w->Kinf, f.L.Kinf, nu, nx) && same(w->Pinf, f.L.Pinf, nx, nx)) ? find_kernel(f, 64, false, true, 0) : nullptr;
    if (kg && kg->session_launch) {
        const size_t smem = kg->smem_bytes(f.L.cold_size);
        p.work_counter = d.counters + kMaxChunks - 1;
        p.x = nullptr; p.u = nullptr;
        CU(s, cudaMemsetAsync(p.work_counter, 0, sizeof(int), st));
        CU(s, d.iter.reserve(sizeof(int) * 4));
        p.iter = static_cast<int*>(d.iter.p); p.status = p.iter + 1;
        CU(s, kg->session_launch(p, 1, smem, st, f.pack.data(), f.L, static_cast<double*>(sb.p), W, 1));
        note_kernel(s, std::string(kg->name) + "_workspace");
    } else {
        CU(s, wpp_launch<double>(p, f.L, d.pack64, W, sb.p, 1, 1, st));
        note_kernel(s, "wpp_f64_workspace");
    }
    CU(s, cudaMemcpyAsync(h.data(), sb.p, sizeof(double) * W.size, cudaMemcpyDeviceToHost, st));
    CU(s, cudaStreamSynchronize(st));
    cudaSetDevice(prev);
    s->launches += 1;

    auto get = [&](double* dst, int at, int n) { if (dst) std::memcpy(dst, h.data() + at, sizeof(double) * n); };
    get(w->x, W.x, sx); get(w->u, W.u, su); get(w->q, W.q, sx); get(w->r, W.r, su); get(w->p, W.p, sx); get(w->d, W.d, su);
    get(w->v, W.v, sx); get(w->vnew, W.vnew, sx); get(w->z, W.z, su); get(w->znew, W.znew, su); get(w->g, W.g, sx); get(w->y, W.y, su);
    get(w->vcnew, W.vcnew, sx); get(w->zcnew, W.zcnew, su); get(w->gc, W.gc, sx); get(w->yc, W.yc, su);
    get(w->vlnew, W.vlnew, sx); get(w->zlnew, W.zlnew, su); get(w->gl, W.gl, sx); get(w->yl, W.yl, su);
    get(w->sol_x, W.vnew, sx); get(w->sol_u, W.znew, su);     // solution = (vnew, znew), admm.cpp:370-371, 386-387
    if (w->Kinf) for (int a = 0; a < nu; ++a) for (int c = 0; c < nx; ++c) w->Kinf[(size_t)c * nu + a] = h[W.Kinf + a * nx + c];
    if (w->Pinf) for (int r = 0; r < nx; ++r) for (int c = 0; c < nx; ++c) w->Pinf[(size_t)c * nx + r] = h[W.Pinf + r * nx + c];
    if (w->rho) *w->rho = h[W.scalars + 0];
    *w->iter = (int)h[W.scalars + 1];
    *w->status = (int)h[W.scalars + 2];
    if (w->solved) *w->solved = (int)h[W.scalars + 7];
    if (w->residuals) for (int k = 0; k < 4; ++k) w->residuals[k] = h[W.scalars + 3 + k];
    return TINYMPC_CUDA_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// sessions: persistent per-problem workspaces iterated in place by the warp-per-problem kernel (exact tiny_solve
// warm-start semantics, tmpc_wpp.cu mode 2)
// ---------------------------------------------------------------------------------------------------------------
namespace {
// Stream contract of the device-resident session entries (include/tinympc_b200.h): the session's stream waits for the work the
// caller queued on `caller` before the call; after the entry has queued its own work there, `caller` waits for that.  The host
// entries copy on the legacy stream, which does not order against the non-blocking streams[0]: they call session_wait first.
cudaError_t session_begin(tinympc_cuda_session* ss, cudaStream_t caller) {
    cudaError_t e = cudaEventRecord(ss->ev_in, caller);
    return e == cudaSuccess ? cudaStreamWaitEvent(ss->s->devs[ss->dev].streams[0], ss->ev_in, 0) : e;
}
cudaError_t session_end(tinympc_cuda_session* ss, cudaStream_t caller) {
    cudaError_t e = cudaEventRecord(ss->ev_out, ss->s->devs[ss->dev].streams[0]);
    return e == cudaSuccess ? cudaStreamWaitEvent(caller, ss->ev_out, 0) : e;
}
// host entries: whatever a device-resident entry left queued on the session's stream has finished (the session's device is current)
cudaError_t session_wait(tinympc_cuda_session* ss) { return cudaStreamSynchronize(ss->s->devs[ss->dev].streams[0]); }

// device entries: every array of `m` is 16-byte aligned device (or managed) memory of `device`, on top of check_model_arrays
int check_device_models(tinympc_cuda_solver* s, const Family& f, const tinympc_cuda_models* m, int device, const char* what) {
    if (int rc = check_model_arrays(s, f, m, true, what)) return rc;
    ModelField mf[kModelFields];
    model_fields(f.nx, f.nu, f.base.adaptive_rho != 0, mf);
    for (int k = 0; k < kModelFields; ++k) {
        const double* p = m->*mf[k].field;
        if (p && !device_ptr_on(p, device))
            return fail(s, TINYMPC_CUDA_EINVAL, std::string(what) + ": " + mf[k].name + " is not device memory of device " + std::to_string(device));
    }
    return TINYMPC_CUDA_OK;
}

// models (the tinympc_cuda_models layout, checked; host arrays, or device arrays with `device`) -> the session's resident copy,
// then into every workspace's model block, Kinf, Pinf and rho.  The rest of each workspace stays as it is.  The host form copies
// and waits; the device form copies device to device on the session's stream under the stream contract and does not wait.
int session_upload_models(tinympc_cuda_session* ss, const tinympc_cuda_models* m, bool device = false, cudaStream_t caller = nullptr) {
    tinympc_cuda_solver* s = ss->s;
    DeviceCtx& d = s->devs[ss->dev];
    DeviceGuard guard;                       // restores the caller's current device on every return path
    CU(s, cudaSetDevice(d.device));
    cudaStream_t st = d.streams[0];
    if (!device) CU(s, session_wait(ss));
    ModelField mf[kModelFields];
    model_fields(ss->fam.nx, ss->fam.nu, ss->fam.base.adaptive_rho != 0, mf);
    for (int k = 0; k < kModelFields; ++k)   // the buffers exist from the first upload of each field on
        if (m->*mf[k].field) CU(s, ss->mdl[k].reserve(sizeof(double) * mf[k].per_problem * (size_t)ss->batch));
    if (device) CU(s, session_begin(ss, caller));
    for (int k = 0; k < kModelFields; ++k) {
        const double* src = m->*mf[k].field;
        const size_t bytes = sizeof(double) * mf[k].per_problem * (size_t)ss->batch;
        if (src) {
            if (device) CU(s, cudaMemcpyAsync(ss->mdl[k].p, src, bytes, cudaMemcpyDeviceToDevice, st));
            else CU(s, cudaMemcpy(ss->mdl[k].p, src, bytes, cudaMemcpyHostToDevice));
        }
        ss->dm.*mf[k].field = src ? static_cast<const double*>(ss->mdl[k].p) : nullptr;
    }
    const int adaptive = ss->fam.base.adaptive_rho != 0;
    CU(s, ss->bits == 64 ? wpp_session_models<double>(ss->W, ss->ws.p, ss->batch, ss->fam.nx, ss->fam.nu, ss->dm, adaptive, st)
                         : wpp_session_models<float>(ss->W, ss->ws.p, ss->batch, ss->fam.nx, ss->fam.nu, ss->dm, adaptive, st));
    s->launches += 1;
    if (device) CU(s, session_end(ss, caller));
    else CU(s, cudaStreamSynchronize(st));
    return TINYMPC_CUDA_OK;
}

int session_create_common(tinympc_cuda_solver* s, int dev_index, int batch, const tinympc_cuda_models* m, tinympc_cuda_session** out,
                          bool device = false, cudaStream_t caller = nullptr) {
    if (!s || !out) return TINYMPC_CUDA_EINVAL;
    *out = nullptr;
    if (!s->fam.set) return fail(s, TINYMPC_CUDA_ENOTREADY, "tinympc_cuda_set_family has not been called");
    if (dev_index < 0 || dev_index >= (int)s->devs.size()) return fail(s, TINYMPC_CUDA_EINVAL, "dev_index out of range");
    if (batch < 1) return fail(s, TINYMPC_CUDA_EINVAL, "session batch must be >= 1");
    if (!s->fam.shared_bounds_ok) return fail(s, TINYMPC_CUDA_EINVAL, "bound constraints are enabled but the family has no bounds");
    if (m && !device) if (int rc = check_model_arrays(s, s->fam, m, false, "model session")) return rc;
    if (m && device) if (int rc = check_device_models(s, s->fam, m, s->devs[dev_index].device, "model session")) return rc;
    auto* ss = new tinympc_cuda_session();
    ss->s = s; ss->dev = dev_index; ss->batch = batch; ss->bits = s->precision;
    ss->fam = s->fam;
    ss->models = m != nullptr;
    ss->W = WppLayout::make(ss->fam.nx, ss->fam.nu, ss->fam.N, ss->models);
    DeviceCtx& d = s->devs[dev_index];
    int prev = 0;
    cudaGetDevice(&prev);
    auto bail = [&](cudaError_t e, const char* what) { cudaSetDevice(prev); tinympc_cuda_session_destroy(ss); return cuda_fail(s, e, what); };
    cudaError_t e = cudaSetDevice(d.device);
    if (e != cudaSuccess) return bail(e, "cudaSetDevice");
    if ((e = cudaEventCreateWithFlags(&ss->ev_in, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "session event");
    if ((e = cudaEventCreateWithFlags(&ss->ev_out, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "session event");
    const size_t esz = ss->bits == 64 ? sizeof(double) : sizeof(float);
    const size_t sx = (size_t)ss->fam.nx * ss->fam.N, su = (size_t)ss->fam.nu * (ss->fam.N - 1);
    if ((e = ss->ws.reserve((size_t)batch * ss->W.size * esz)) != cudaSuccess) return bail(e, "session workspace allocation");
    if ((e = ss->x.reserve(sizeof(float) * sx * batch)) != cudaSuccess) return bail(e, "session buffer");
    if ((e = ss->u.reserve(sizeof(float) * su * batch)) != cudaSuccess) return bail(e, "session buffer");
    if ((e = ss->iter.reserve(sizeof(int) * (size_t)batch)) != cudaSuccess) return bail(e, "session buffer");
    if ((e = ss->status.reserve(sizeof(int) * (size_t)batch)) != cudaSuccess) return bail(e, "session buffer");
    // the family pack in the session's precision lives with the solver (re-uploaded by set_family); keep our own copy
    if ((e = ss->pack.reserve(ss->fam.pack.size() * esz)) != cudaSuccess) return bail(e, "session pack");
    if (ss->bits == 64) {
        e = cudaMemcpy(ss->pack.p, ss->fam.pack.data(), ss->fam.pack.size() * sizeof(double), cudaMemcpyHostToDevice);
    } else {
        std::vector<float> p32(ss->fam.pack.size());
        for (size_t i = 0; i < p32.size(); ++i) p32[i] = static_cast<float>(ss->fam.pack[i]);
        e = cudaMemcpy(ss->pack.p, p32.data(), p32.size() * sizeof(float), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) return bail(e, "session pack upload");
    cudaStream_t st = d.streams[0];
    e = ss->bits == 64 ? wpp_session_init<double>(ss->fam.base, ss->fam.L, ss->pack.p, ss->W, ss->ws.p, batch, st)
                       : wpp_session_init<float>(ss->fam.base, ss->fam.L, ss->pack.p, ss->W, ss->ws.p, batch, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return bail(e, "session init");
    s->launches += 1;
    cudaSetDevice(prev);
    s->sessions.push_back(ss);
    if (m) {
        if (int rc = session_upload_models(ss, m, device, caller)) { tinympc_cuda_session_destroy(ss); return rc; }
    }
    *out = ss;
    return TINYMPC_CUDA_OK;
}

// the workspace member (WppLayout offset) and width per solver of a session field: with `write` the fields the setters write, else
// the fields session_read reads.  false for an unknown name.
bool session_field(const tinympc_cuda_session* ss, const std::string& f, bool write, int* at, int* width) {
    const WppLayout& W = ss->W;
    const int nx = ss->fam.nx, nu = ss->fam.nu, N = ss->fam.N;
    struct F { const char* name; int at, width; bool read, write; };
    const F fields[] = {
        {"x0", W.x, nx, true, true}, {"Xref", W.Xref, nx * N, false, true}, {"Uref", W.Uref, nu * (N - 1), false, true},
        {"x", W.x, nx * N, true, false}, {"u", W.u, nu * (N - 1), true, false},
        {"sol_x", W.vnew, nx * N, true, false}, {"sol_u", W.znew, nu * (N - 1), true, false},   // solution->x = work->vnew, admm.cpp:370, 386
        {"rho", W.scalars + 0, 1, true, false}, {"iter", W.scalars + 1, 1, true, false}, {"status", W.scalars + 2, 1, true, false},
        {"residuals", W.scalars + 3, 4, true, false}};
    for (const F& x : fields)
        if (f == x.name && (write ? x.write : x.read)) { *at = x.at; *width = x.width; return true; }
    return false;
}
}  // namespace

int tinympc_cuda_session_create(tinympc_cuda_solver* s, int dev_index, int batch, tinympc_cuda_session** out) {
    return session_create_common(s, dev_index, batch, nullptr, out);
}

int tinympc_cuda_session_create_models(tinympc_cuda_solver* s, int dev_index, int batch, const tinympc_cuda_models* m,
                                       tinympc_cuda_session** out) {
    if (out) *out = nullptr;
    if (!m) return s ? fail(s, TINYMPC_CUDA_EINVAL, "model session: models is NULL") : TINYMPC_CUDA_EINVAL;
    return session_create_common(s, dev_index, batch, m, out);
}

int tinympc_cuda_session_create_models_device(tinympc_cuda_solver* s, int dev_index, int batch, const tinympc_cuda_models* m, void* stream,
                                              tinympc_cuda_session** out) {
    if (out) *out = nullptr;
    if (!m) return s ? fail(s, TINYMPC_CUDA_EINVAL, "model session: models is NULL") : TINYMPC_CUDA_EINVAL;
    return session_create_common(s, dev_index, batch, m, out, true, static_cast<cudaStream_t>(stream));
}

int tinympc_cuda_session_set_models(tinympc_cuda_session* ss, const tinympc_cuda_models* m) {
    if (!ss) return TINYMPC_CUDA_EINVAL;
    tinympc_cuda_solver* s = ss->s;
    if (!s) return TINYMPC_CUDA_ENOTREADY;   // the solver was destroyed under the session
    if (!m) return fail(s, TINYMPC_CUDA_EINVAL, "model session: models is NULL");
    if (!ss->models) return fail(s, TINYMPC_CUDA_EINVAL, "set_models needs a session created with models (tinympc_cuda_session_create_models)");
    if (int rc = check_model_arrays(s, ss->fam, m, false, "model session")) return rc;
    return session_upload_models(ss, m);
}

int tinympc_cuda_session_set_models_device(tinympc_cuda_session* ss, const tinympc_cuda_models* m, void* stream) {
    if (!ss) return TINYMPC_CUDA_EINVAL;
    tinympc_cuda_solver* s = ss->s;
    if (!s) return TINYMPC_CUDA_ENOTREADY;   // the solver was destroyed under the session
    if (!m) return fail(s, TINYMPC_CUDA_EINVAL, "model session: models is NULL");
    if (!ss->models) return fail(s, TINYMPC_CUDA_EINVAL, "set_models needs a session created with models (tinympc_cuda_session_create_models)");
    if (int rc = check_device_models(s, ss->fam, m, s->devs[ss->dev].device, "model session")) return rc;
    return session_upload_models(ss, m, true, static_cast<cudaStream_t>(stream));
}

int tinympc_cuda_session_destroy(tinympc_cuda_session* ss) {
    if (!ss) return TINYMPC_CUDA_OK;
    if (ss->s) {   // (an orphan's buffers went with its solver)
        int prev = 0;
        cudaGetDevice(&prev);
        cudaSetDevice(ss->s->devs[ss->dev].device);
        if (ss->ev_in) session_wait(ss);     // (a session that failed in creation may have no events and nothing queued)
        for (DevBuf* b : {&ss->ws, &ss->pack, &ss->x, &ss->u, &ss->iter, &ss->status}) b->release();
        for (DevBuf& b : ss->mdl) b.release();
        for (cudaEvent_t ev : {ss->ev_in, ss->ev_out}) if (ev) cudaEventDestroy(ev);
        cudaSetDevice(prev);
        auto& v = ss->s->sessions;
        v.erase(std::remove(v.begin(), v.end(), ss), v.end());
    }
    delete ss;
    return TINYMPC_CUDA_OK;
}

namespace {
// host doubles (rows of `width` elements, `rows_src` of them or ONE broadcast row) -> member `at` of every workspace
int session_scatter(tinympc_cuda_session* ss, int at, int width, const double* src, bool broadcast) {
    tinympc_cuda_solver* s = ss->s;
    if (!s) return TINYMPC_CUDA_ENOTREADY;
    const size_t esz = ss->bits == 64 ? sizeof(double) : sizeof(float);
    const size_t n = (size_t)ss->batch * width;
    ss->stage.resize(n * esz);
    for (size_t k = 0; k < n; ++k) {
        const double v = src ? src[broadcast ? k % width : k] : 0.0;
        if (ss->bits == 64) reinterpret_cast<double*>(ss->stage.data())[k] = v;
        else reinterpret_cast<float*>(ss->stage.data())[k] = static_cast<float>(v);
    }
    int prev = 0;
    cudaGetDevice(&prev);
    CU(s, cudaSetDevice(s->devs[ss->dev].device));
    CU(s, session_wait(ss));
    CU(s, cudaMemcpy2D(static_cast<char*>(ss->ws.p) + (size_t)at * esz, (size_t)ss->W.size * esz, ss->stage.data(), (size_t)width * esz,
                       (size_t)width * esz, ss->batch, cudaMemcpyHostToDevice));
    cudaSetDevice(prev);
    return TINYMPC_CUDA_OK;
}
int session_gather(tinympc_cuda_session* ss, int at, int width, double* dst) {
    tinympc_cuda_solver* s = ss->s;
    if (!s) return TINYMPC_CUDA_ENOTREADY;
    const size_t esz = ss->bits == 64 ? sizeof(double) : sizeof(float);
    const size_t n = (size_t)ss->batch * width;
    ss->stage.resize(n * esz);
    int prev = 0;
    cudaGetDevice(&prev);
    CU(s, cudaSetDevice(s->devs[ss->dev].device));
    CU(s, session_wait(ss));
    CU(s, cudaMemcpy2D(ss->stage.data(), (size_t)width * esz, static_cast<char*>(ss->ws.p) + (size_t)at * esz, (size_t)ss->W.size * esz,
                       (size_t)width * esz, ss->batch, cudaMemcpyDeviceToHost));
    cudaSetDevice(prev);
    for (size_t k = 0; k < n; ++k)
        dst[k] = ss->bits == 64 ? reinterpret_cast<double*>(ss->stage.data())[k] : static_cast<double>(reinterpret_cast<float*>(ss->stage.data())[k]);
    return TINYMPC_CUDA_OK;
}
}  // namespace

int tinympc_cuda_session_set_x0(tinympc_cuda_session* ss, const double* x0) {
    if (!ss || !x0) return TINYMPC_CUDA_EINVAL;
    return session_scatter(ss, ss->W.x, ss->fam.nx, x0, false);     // work->x.col(0) = x0, tiny_api.cpp:383
}
int tinympc_cuda_session_set_x_ref(tinympc_cuda_session* ss, const double* Xref, int broadcast) {
    if (!ss) return TINYMPC_CUDA_EINVAL;
    return session_scatter(ss, ss->W.Xref, ss->fam.nx * ss->fam.N, Xref, broadcast != 0);
}
int tinympc_cuda_session_set_u_ref(tinympc_cuda_session* ss, const double* Uref, int broadcast) {
    if (!ss) return TINYMPC_CUDA_EINVAL;
    return session_scatter(ss, ss->W.Uref, ss->fam.nu * (ss->fam.N - 1), Uref, broadcast != 0);
}

int tinympc_cuda_session_solve(tinympc_cuda_session* ss) {
    if (!ss) return TINYMPC_CUDA_EINVAL;
    tinympc_cuda_solver* s = ss->s;
    if (!s) return TINYMPC_CUDA_ENOTREADY;   // the solver was destroyed under the session
    DeviceCtx& d = s->devs[ss->dev];
    int prev = 0;
    cudaGetDevice(&prev);
    CU(s, cudaSetDevice(d.device));
    SolveParams p = ss->fam.base;
    p.batch = ss->batch;
    p.x = static_cast<float*>(ss->x.p); p.u = static_cast<float*>(ss->u.p);
    p.iter = static_cast<int*>(ss->iter.p); p.status = static_cast<int*>(ss->status.p);
    const int warps = std::max(1, std::min(ss->batch, d.sm_count * 16));
    cudaStream_t st = d.streams[0];
    // fp64 sessions of a box family with a compiled shape run the lane-group kernel on the same workspaces (tmpc_gpp.cuh, session
    // mode): the reference's warm-start semantics at ~4x the rate of the warp-per-problem kernel; option "kernel" = 1 keeps the latter
    // Model sessions: the session form of the lane-group kernel's model mode where model batches take the model mode
    const KernelEntry* kg = ss->models ? model_kernel(s, ss->fam, false, ss->bits)
                          : (ss->bits == 64 && !s->force_wpp && ss->fam.feat == kFeatBox && ss->fam.shared_bounds_ok) ? find_kernel(ss->fam, 64, false, true, 0) : nullptr;
    if (kg && !(ss->models ? kg->models_session_launch != nullptr : kg->session_launch != nullptr)) kg = nullptr;
    if (ss->fam.base.max_iter > 0 && kg) {
        const size_t smem = kg->smem_bytes(ss->fam.L.cold_size);
        int occ = 1;
        CU(s, kg->prepare(smem));
        CU(s, kg->occupancy(&occ, smem));
        const int per_cta = kg->block / std::max(1, kg->lanes_per_problem);
        const int grid = std::max(1, std::min(d.sm_count * std::max(1, occ), (ss->batch + per_cta - 1) / per_cta));
        p.work_counter = d.counters + kMaxChunks - 1;
        CU(s, cudaMemsetAsync(p.work_counter, 0, sizeof(int), st));
        if (ss->models) CU(s, kg->models_session_launch(p, grid, smem, st, ss->fam.pack.data(), ss->fam.L, static_cast<double*>(ss->ws.p), ss->W, ss->dm));
        else CU(s, kg->session_launch(p, grid, smem, st, ss->fam.pack.data(), ss->fam.L, static_cast<double*>(ss->ws.p), ss->W, 0));
        s->launches += 1;
        note_kernel(s, std::string(kg->name) + "_session");
    } else if (ss->fam.base.max_iter > 0) {
        const tinympc_cuda_models* mdl = ss->models ? &ss->dm : nullptr;
        CU(s, ss->bits == 64 ? wpp_launch<double>(p, ss->fam.L, ss->pack.p, ss->W, ss->ws.p, warps, 2, st, mdl)
                             : wpp_launch<float>(p, ss->fam.L, ss->pack.p, ss->W, ss->ws.p, warps, 2, st, mdl));
        s->launches += 1;
        note_kernel(s, ss->models ? (ss->bits == 64 ? "wpp_f64_mdl_session" : "wpp_f32_mdl_session")
                                  : (ss->bits == 64 ? "wpp_f64_session" : "wpp_f32_session"));
    }
    CU(s, cudaStreamSynchronize(st));
    cudaSetDevice(prev);
    return TINYMPC_CUDA_OK;
}

int tinympc_cuda_session_step(tinympc_cuda_session* ss, int use_solution) {
    if (!ss) return TINYMPC_CUDA_EINVAL;
    tinympc_cuda_solver* s = ss->s;
    if (!s) return TINYMPC_CUDA_ENOTREADY;   // the solver was destroyed under the session
    if (ss->fam.nx > 32)                     // the step kernel gives each state row one lane of a warp
        return fail(s, TINYMPC_CUDA_EUNSUPPORTED, "session step needs nx <= 32 (one lane per state); the session has nx = " +
                                                      std::to_string(ss->fam.nx));
    DeviceCtx& d = s->devs[ss->dev];
    DeviceGuard guard;                       // restores the caller's current device on every return path
    CU(s, cudaSetDevice(d.device));
    cudaStream_t st = d.streams[0];
    const int nx = ss->fam.nx, nu = ss->fam.nu;
    if (ss->models)
        CU(s, ss->bits == 64 ? wpp_session_step_models<double>(ss->W, ss->ws.p, ss->batch, nx, nu, use_solution, st)
                             : wpp_session_step_models<float>(ss->W, ss->ws.p, ss->batch, nx, nu, use_solution, st));
    else
        CU(s, ss->bits == 64 ? wpp_session_step<double>(ss->fam.L, ss->pack.p, ss->W, ss->ws.p, ss->batch, use_solution, st)
                             : wpp_session_step<float>(ss->fam.L, ss->pack.p, ss->W, ss->ws.p, ss->batch, use_solution, st));
    s->launches += 1;
    CU(s, cudaStreamSynchronize(st));
    return TINYMPC_CUDA_OK;
}

int tinympc_cuda_session_read(tinympc_cuda_session* ss, const char* field, double* host) {
    if (!ss || !field || !host) return TINYMPC_CUDA_EINVAL;
    if (!ss->s) return TINYMPC_CUDA_ENOTREADY;
    int at = 0, width = 0;
    if (!session_field(ss, field, false, &at, &width)) return fail(ss->s, TINYMPC_CUDA_EINVAL, std::string("unknown session field ") + field);
    return session_gather(ss, at, width, host);
}

namespace {
// the two device-resident I/O entries: `p` (16-byte aligned device memory of the session's device), a packed [batch][width] array of
// doubles (or one row, write with broadcast) <-> member `at` of every workspace, under the stream contract
int session_io_device(tinympc_cuda_session* ss, const char* field, bool write, const double* src, double* dst, int broadcast, void* stream) {
    if (!ss || !field) return TINYMPC_CUDA_EINVAL;
    tinympc_cuda_solver* s = ss->s;
    if (!s) return TINYMPC_CUDA_ENOTREADY;   // the solver was destroyed under the session
    DeviceCtx& d = s->devs[ss->dev];
    int at = 0, width = 0;
    if (!session_field(ss, field, write, &at, &width))
        return fail(s, TINYMPC_CUDA_EINVAL, std::string("unknown session field for ") + (write ? "write_device: " : "read_device: ") + field);
    const void* p = write ? static_cast<const void*>(src) : static_cast<const void*>(dst);
    if (!p || !device_ptr_on(p, d.device))
        return fail(s, TINYMPC_CUDA_EINVAL, std::string(field) + ": the array must be 16-byte aligned device memory of device " + std::to_string(d.device));
    const cudaStream_t caller = static_cast<cudaStream_t>(stream);
    DeviceGuard guard;                       // restores the caller's current device on every return path
    CU(s, cudaSetDevice(d.device));
    CU(s, session_begin(ss, caller));
    if (write)
        CU(s, ss->bits == 64 ? wpp_session_scatter<double>(ss->W, ss->ws.p, ss->batch, at, width, src, broadcast != 0, d.streams[0])
                             : wpp_session_scatter<float>(ss->W, ss->ws.p, ss->batch, at, width, src, broadcast != 0, d.streams[0]));
    else
        CU(s, ss->bits == 64 ? wpp_session_gather<double>(ss->W, ss->ws.p, ss->batch, at, width, dst, d.streams[0])
                             : wpp_session_gather<float>(ss->W, ss->ws.p, ss->batch, at, width, dst, d.streams[0]));
    s->launches += 1;
    CU(s, session_end(ss, caller));
    return TINYMPC_CUDA_OK;
}
}  // namespace

int tinympc_cuda_session_write_device(tinympc_cuda_session* ss, const char* field, const double* src, int broadcast, void* stream) {
    return session_io_device(ss, field, true, src, nullptr, broadcast, stream);
}
int tinympc_cuda_session_read_device(tinympc_cuda_session* ss, const char* field, double* dst, void* stream) {
    return session_io_device(ss, field, false, nullptr, dst, 0, stream);
}

int tinympc_cuda_set_option(tinympc_cuda_solver* s, const char* name, double value) {
    if (!s || !name) return TINYMPC_CUDA_EINVAL;
    const std::string n(name);
    if (n == "precision") {
        if (value != 32 && value != 64) return fail(s, TINYMPC_CUDA_EINVAL, "precision must be 32 or 64");
        s->precision = (int)value;
    } else if (n == "ctas_per_sm") {
        s->ctas_per_sm = (int)value;
    } else if (n == "chunks") {
        s->chunks = (int)value;
    } else if (n == "variant") {
        s->variant = (int)value;
    } else if (n == "mixed") {
        if (!(value >= 0 && value < 1)) return fail(s, TINYMPC_CUDA_EINVAL, "mixed (relative band) must be in [0, 1)");
        s->mixed_band = value;
    } else if (n == "pass_timing") {
        s->pass_timing = (int)value;
    } else if (n == "fixer_sms") {
        s->fixer_sms = (int)value;
    } else if (n == "force_wpp") {
        s->force_wpp = (int)value;
    } else if (n == "streamed") {
        s->streamed = value != 0;
    } else if (n == "compact_streamed") {
        s->compact_streamed = value != 0;
    } else if (n == "compact_early_d2h") {
        s->compact_early_d2h = value != 0;
    } else if (n == "order") {
        s->order = value != 0;
    } else if (n == "order_sms") {
        s->order_sms = (int)value;
    } else if (n == "order_from_div") {
        s->order_from_div = (int)value;
    } else if (n == "compact_in_kernel") {
        s->compact_in_kernel = value != 0;
    } else if (n == "refill_min") {
        s->refill_min = (int)value;
    } else if (n == "dense_a") {
        s->dense_a = value != 0;
    } else {
        return fail(s, TINYMPC_CUDA_EINVAL, "unknown option " + n);
    }
    return TINYMPC_CUDA_OK;
}

int tinympc_cuda_num_devices(const tinympc_cuda_solver* s) { return s ? (int)s->devs.size() : 0; }
const char* tinympc_cuda_last_kernel(const tinympc_cuda_solver* s) { return s ? s->last_kernel.c_str() : ""; }
long long tinympc_cuda_launch_count(const tinympc_cuda_solver* s) { return s ? s->launches.load() : 0; }
int tinympc_cuda_last_timing(const tinympc_cuda_solver* s, double ms[3]) {
    if (!s || !ms) return TINYMPC_CUDA_EINVAL;
    ms[0] = s->t_total_ms; ms[1] = s->t_kernel_ms; ms[2] = (double)s->t_chunks;
    return TINYMPC_CUDA_OK;
}
int tinympc_cuda_last_pass_ms(tinympc_cuda_solver* s, double ms[2]) {
    if (!s || !ms) return TINYMPC_CUDA_EINVAL;
    ms[0] = ms[1] = 0.0;
    DeviceCtx& d = s->devs[0];
    if (!d.pass_timed) return TINYMPC_CUDA_ENOTREADY;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(d.device);
    float a = 0.f, b = 0.f;
    cudaError_t e = cudaEventSynchronize(d.ev_p2);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&a, d.ev_p0, d.ev_p1);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&b, d.ev_p1, d.ev_p2);
    cudaSetDevice(prev);
    if (e != cudaSuccess) return cuda_fail(s, e, "pass timing");
    ms[0] = a; ms[1] = b;
    return TINYMPC_CUDA_OK;
}
long long tinympc_cuda_last_marked(tinympc_cuda_solver* s) {
    if (!s) return 0;
    if (s->mixed_pending_dev >= 0) {   // device entry: blocking read of the count its fp64 pass consumed
        DeviceCtx& d = s->devs[s->mixed_pending_dev];
        int prev = 0, n = 0;
        cudaGetDevice(&prev);
        cudaSetDevice(d.device);
        cudaDeviceSynchronize();
        cudaMemcpy(&n, s->fixer_sms >= 0 ? d.qctl + 4 * (kMaxChunks - 1) : d.counters + 3 * kMaxChunks - 1, sizeof(int), cudaMemcpyDeviceToHost);
        cudaSetDevice(prev);
        s->mixed_marked = n;
        s->mixed_pending_dev = -1;
    }
    return s->mixed_marked;
}
int tinympc_cuda_plan_compact_chunks(int n, int chunks, int order_from_div, int* bounds, int max_bounds, int* first_ordered) {
    if (n <= 0 || !bounds || max_bounds < 2) return -1;
    std::vector<int> b;
    const int fo = plan_compact_chunks(n, chunks, order_from_div, b);
    if ((int)b.size() > max_bounds) return -1;
    for (size_t k = 0; k < b.size(); ++k) bounds[k] = b[k];
    if (first_ordered) *first_ordered = fo;
    return (int)b.size() - 1;
}
const char* tinympc_cuda_last_error(const tinympc_cuda_solver* s) { return s ? s->err.c_str() : "null solver"; }

void* tinympc_cuda_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void tinympc_cuda_host_free(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
