// tmpc_common.h -- data shared by the host C-ABI layer and the sm_100a kernels.
//
// "Family" data = everything a TinySolver holds that is identical for every problem of a batch
// (reference: TinyCache types.hpp:43-59, the matrices/bounds/constraint specs of TinyWorkspace
// types.hpp:114-173 and TinySettings types.hpp:63-80).  The host converts it once to the kernel's
// scalar type and lays it out as one contiguous "pack" that every CTA stages into shared memory
// with a single TMA bulk copy.
#pragma once
#include <cstddef>
#include <cstdint>

#include "tinympc_b200.h"   // tinympc_cuda_models: the per-problem model arrays the model kernels read on the device

namespace tmpc {

constexpr int kMaxCones = 4;     // per family (state cones) and (input cones)
constexpr int kMaxGranules = 64; // streamed host pipeline: the batch is cut into at most this many equal granules

// Offsets (in elements) of the tables inside the family's master pack (host, double).
// All small matrices are stored ROW-major: M[r * cols + c].  The "hot" tables are converted into the
// kernel-parameter constant pack at launch; the "cold" tail [cold, cold + cold_size) is what each CTA
// stages into shared memory with one TMA bulk copy.
struct PackLayout {
    int nx, nu, N;
    int nsl, nil;                 // linear rows (state / input)
    // hot
    int A, B, Kinf, AmBKt, Quu_inv, f, APf, BPf, Qd, Rd;
    int xmin, xmax, umin, umax;   // shared bounds nx*N / nu*(N-1) (time-major)
    int dKinf;
    // cold (shared-memory staged)
    int cold;                     // start of the cold tail (multiple of 4 elements)
    int Pinf, dPinf;
    int d0;                       // nu*(N-1): d of the first backward pass on a zero workspace
    int Alin_x, blin_x, nrm_x;    // nsl*nx, nsl, nsl (||a||^2)
    int Alin_u, blin_u, nrm_u;
    int cold_size;                // elements in the cold tail, multiple of 4
    int size;                     // total elements

    static PackLayout make(int nx, int nu, int N, int nsl, int nil) {
        PackLayout L{};
        L.nx = nx; L.nu = nu; L.N = N; L.nsl = nsl; L.nil = nil;
        int o = 0;
        auto take = [&](int n) { int at = o; o += n; return at; };
        L.A = take(nx * nx); L.B = take(nx * nu); L.Kinf = take(nu * nx); L.AmBKt = take(nx * nx);
        L.Quu_inv = take(nu * nu); L.f = take(nx); L.APf = take(nx); L.BPf = take(nu);
        L.Qd = take(nx); L.Rd = take(nu);
        L.xmin = take(nx * N); L.xmax = take(nx * N); L.umin = take(nu * (N - 1)); L.umax = take(nu * (N - 1));
        L.dKinf = take(nu * nx);
        o = (o + 3) & ~3;
        L.cold = o;
        L.Pinf = take(nx * nx); L.dPinf = take(nx * nx); L.d0 = take(nu * (N - 1));
        L.Alin_x = take(nsl * nx); L.blin_x = take(nsl); L.nrm_x = take(nsl);
        L.Alin_u = take(nil * nu); L.blin_u = take(nil); L.nrm_u = take(nil);
        o = (o + 3) & ~3;         // multiple of 4 elements -> 16 B multiple for float and double
        L.cold_size = o - L.cold;
        L.size = o;
        return L;
    }
};

// compile-time offsets inside the COLD tail (relative to PackLayout::cold) used by the kernels
template <int NX, int NU, int NH>
struct StaticPack {
    static constexpr int Pinf = 0;
    static constexpr int dPinf = Pinf + NX * NX;
    static constexpr int d0 = dPinf + NX * NX;
    static constexpr int lin = d0 + NU * (NH - 1);   // linear rows start here (runtime sized)
};

// Kernel launch parameters (passed by value; plain data only).
struct SolveParams {
    const void* pack;          // device pointer to the cold tail of the pack, 16 B aligned
    int pack_elems;            // PackLayout::cold_size
    int batch;
    int* work_counter;         // device int, zeroed before launch: next unclaimed problem index
    void* ref_scratch;         // REFS_L2 kernels: grid*block*(nx*N+nu*(N-1)) elements of the kernel scalar type
    // per-problem inputs (device pointers, float32); NULL where noted
    const float* x0;           // batch*nx
    const float* Xref;         // batch*nx*N      or NULL (zeros)
    const float* Uref;         // batch*nu*(N-1)  or NULL (zeros)
    const float* x_min;        // per-problem bounds or NULL (use the family's shared bounds)
    const float* x_max;
    const float* u_min;
    const float* u_max;
    // outputs
    float* x;                  // batch*nx*N      solution->x (= vnew)
    float* u;                  // batch*nu*(N-1)  solution->u (= znew)
    int* iter;                 // batch
    int* status;               // batch (1 solved / 11 unsolved)
    float* residuals;          // batch*4 or NULL  (pri_state, dua_state, pri_input, dua_input)
    float* rho_out;            // batch or NULL
    // settings (TinySettings) + cache->rho
    double rho;
    double abs_pri_tol, abs_dua_tol;
    int max_iter, check_termination;
    int en_state_bound, en_input_bound;
    int en_state_soc, en_input_soc;
    int en_state_linear, en_input_linear;
    int adaptive_rho;
    double rho_min, rho_max;
    int rho_clip;
    // cones as they sit in the workspace
    int n_state_cones, n_input_cones;
    int Acx[kMaxCones], qcx[kMaxCones], Acu[kMaxCones], qcu[kMaxCones];
    float cx[kMaxCones], cu[kMaxCones];     // the reference's project_soc takes `float mu` (admm.cpp:39)
    int nsl, nil;
    // mixed-precision exact-count mode (tmpc_capi.cu, option "mixed"): the fp32 pass marks a problem whose termination
    // decision falls inside the relative band around the tolerances (status |= kAmbiguousBit) and stops iterating it;
    // the fp64 pass re-solves exactly the marked problems through index_list / batch_ptr.
    float amb_band;            // 0 = off
    const int* index_list;     // NULL, or problem index of work item k (the kernel then runs over *batch_ptr items)
    const int* batch_ptr;      // NULL, or device int holding the number of work items (<= batch)
    // Exact-count mode as a producer / consumer pair running CONCURRENTLY (tmpc_capi.cu enqueue_exact): the fp32 kernel
    // (producer, q_consume = 0) pushes every problem it cannot decide onto a device queue instead of finishing it; the fp64
    // kernel (consumer, q_consume = 1) runs on the SMs the producer's grid leaves free, takes tickets from work_counter, waits
    // for its ticket to be filled, and exits once every producer CTA has left and the queue is drained.
    //   q_tail       entries reserved so far (producer: atomicAdd; consumer: how far it may look)
    //   q_list       problem index per entry, preset to -1, written with release semantics after the reservation
    //   q_prod_done  producer CTAs that have exited; the queue is complete when it reaches q_prod_total
    int* q_tail;               // NULL = no queue (plain solve, or the two-pass form with index_list)
    int* q_list;
    int* q_prod_done;
    int q_prod_total;
    int q_consume;
    // streamed host pipeline (tmpc_capi.cu run_shard_streamed): ONE persistent launch consumes the batch while the copy engines
    // are still delivering it.  avail_ptr counts the problems whose inputs have landed (written in stream order behind each
    // H2D chunk); a lane that claims problem p starts it once *avail_ptr > p.  done_counters[chunk of p] counts finished
    // problems per chunk (release): the D2H stream waits on it (cuStreamWaitValue32) before copying that chunk.
    const int* avail_ptr;      // NULL = the whole batch is resident
    int* done_counters;        // NULL = nobody is waiting
    int done_chunk;            // problems per granule; chunk of problem p = done_map[p / done_chunk]
    unsigned char done_map[kMaxGranules];   // chunks are runs of granules: short ones first (early start) and last (short tail)
    // Batched lane refill (tmpc_tpp3.cuh): a warp claims new problems only once at least refill_min of its lanes are free (or
    // none is busy).  Claim + input loads + tensor-memory parking are warp-wide code executed for however few lanes need it,
    // so sharing one pass between several lanes trades a little idle lane time for fewer passes.  1: refill at once; 0: adaptive.
    int refill_min;
    // Compact I/O in the kernel, honoured by the kernels whose KernelEntry::compact_ok is set (for the others the library expands /
    // gathers on the device around the launch and leaves these 0 / NULL):
    //   xref_const  1: Xref holds ONE state per problem (batch*nx), which stands for every column of the horizon
    //               (tinympc_cuda_batch_in::xref_const)
    //   u0          not NULL: the only solution output is the first control, batch*nu (tinympc_cuda_batch_out::u0); x and u are
    //               then not written (and may be NULL)
    int xref_const;
    float* u0;
    // Streamed batch with an ordered part (tmpc_capi.cu run_shard_compact_streamed): work items below order_from are problem
    // indices; item c >= order_from is problem index_list[c - order_from].  The list is built on the device chunk by chunk, as
    // the chunks arrive and while earlier items are being solved; the arrival watermark moves past a chunk only when its part of
    // the list is written too, so a lane waits for item c exactly as it waits for problem c.  0 = index_list, if any, covers every
    // work item.  Honoured by the incremental fp32 kernel (tmpc_tpp3.cuh).
    int order_from;
};

constexpr int kAmbiguousBit = 0x100;

}  // namespace tmpc
