/*
 * tinympc_b200.h -- thin C ABI of the B200-native batched TinyMPC ADMM solver.
 *
 * This is the drop-in boundary for the reference's hot path: everything between tiny_solve()
 * being entered (tinympc/TinyMPC/src/tinympc/tiny_api.cpp:321-323) and solve() returning
 * (tinympc/TinyMPC/src/tinympc/admm.cpp:274-389).  The reference's own "extern C" API passes Eigen
 * objects by value (tiny_api.hpp:10-50) and is therefore not a C ABI; the host C++ mirror of that
 * API (tinympc-matlab_b200/csrc/host/tiny_api.hpp) and the MEX layer call THIS interface, which
 * uses only plain pointers, ints and doubles.  INTEGRATION.md shows the binding a maintainer of the
 * reference would add.
 *
 * Conventions
 *   - "family" data (dynamics, cache, settings, shared constraints) is what one TinySolver holds
 *     (types.hpp:43-187): column-major double arrays on the HOST, copied at set_family time.
 *   - batch data is float32, one contiguous chunk per problem: x0[b][nx], Xref[b][N][nx]
 *     (= column-major nx x N per problem, as TinyWorkspace::Xref), Uref[b][N-1][nu], etc.
 *   - every entry point returns 0 on success, a TINYMPC_CUDA_E* code otherwise;
 *     tinympc_cuda_last_error() gives the text.  There is NO CPU fallback: without a usable CUDA
 *     device every solve call fails with TINYMPC_CUDA_ENODEVICE.
 *   - cold-start semantics per problem: workspace as tiny_setup leaves it (tiny_api.cpp:68-105) and
 *     the pristine cache, i.e. exactly what a fresh tiny_setup + tiny_set_x0/x_ref/u_ref +
 *     tiny_solve produces.  solution = (vnew, znew) (admm.cpp:370-371, 386-387), status 1 solved /
 *     11 unsolved (admm.cpp:279, 365), iter = work->iter.
 */
#ifndef TINYMPC_B200_H
#define TINYMPC_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TINYMPC_CUDA_OK          0
#define TINYMPC_CUDA_EINVAL      1   /* bad argument / dimension mismatch (cf. check_dimension, tiny_api.cpp:13-19) */
#define TINYMPC_CUDA_ENODEVICE   2   /* no CUDA device / driver: the product never falls back to the CPU */
#define TINYMPC_CUDA_ECUDA       3   /* a CUDA runtime call failed */
#define TINYMPC_CUDA_EUNSUPPORTED 4  /* problem shape has no compiled kernel */
#define TINYMPC_CUDA_ENOTREADY   5   /* solve before set_family */

#define TINYMPC_MAX_CONES 4

typedef struct tinympc_cuda_solver tinympc_cuda_solver;   /* opaque */

/* What one TinySolver holds after tiny_setup + the constraint setters (replaces reading
 * solver->work / solver->cache / solver->settings directly, types.hpp:43-197). */
typedef struct {
    int nx, nu, N;
    /* TinyWorkspace dynamics and cost diagonals (types.hpp:165-169); Q, R are work->Q, work->R,
       i.e. diag(Q)+rho, diag(R)+rho as tiny_setup stores them (tiny_api.cpp:107-108) */
    const double *Adyn, *Bdyn, *fdyn, *Q, *R;
    /* TinyCache (types.hpp:43-59) */
    double rho;
    const double *Kinf, *Pinf, *Quu_inv, *AmBKt, *APf, *BPf;
    const double *dKinf_drho, *dPinf_drho;   /* read only when adaptive_rho != 0; C1/C2 are dead on the
                                                iteration path (admm.cpp:17-18) and are not needed */
    /* TinySettings (types.hpp:63-80) */
    double abs_pri_tol, abs_dua_tol;
    int max_iter, check_termination;
    int en_state_bound, en_input_bound, en_state_soc, en_input_soc, en_state_linear, en_input_linear;
    int adaptive_rho;
    double adaptive_rho_min, adaptive_rho_max;
    int adaptive_rho_enable_clipping;
    /* shared bounds (types.hpp:115-118), nx*N and nu*(N-1) column-major; may be NULL when the
       matching en_* flag is 0 or when every batch supplies per-problem bounds */
    const double *x_min, *x_max, *u_min, *u_max;
    /* cones as they sit in the workspace (types.hpp:122-129) */
    int numStateCones, numInputCones;
    const int *Acx, *qcx; const double *cx;
    const int *Acu, *qcu; const double *cu;
    /* linear inequality rows (types.hpp:143-150), Alin_x is numStateLinear x nx column-major */
    int numStateLinear, numInputLinear;
    const double *Alin_x, *blin_x, *Alin_u, *blin_u;
} tinympc_cuda_family;

/* One batch of independent problems of the family.  Pointers are HOST pointers for
 * tinympc_cuda_solve_batch and DEVICE pointers (16-byte aligned) for tinympc_cuda_solve_batch_device. */
typedef struct {
    int batch;
    const float *x0;      /* batch*nx                        replaces tiny_set_x0   (tiny_api.cpp:375-385) */
    const float *Xref;    /* batch*nx*N      or NULL = zeros replaces tiny_set_x_ref (tiny_api.cpp:387-397) */
    const float *Uref;    /* batch*nu*(N-1)  or NULL = zeros replaces tiny_set_u_ref (tiny_api.cpp:399-409) */
    const float *x_min, *x_max;   /* optional per-problem bounds, batch*nx*N     (all four or none) */
    const float *u_min, *u_max;   /*                              batch*nu*(N-1)                    */
    /* Compact input (instead of Xref): ONE reference state per problem, held over the whole horizon -- what
       tiny_set_x_ref receives in the closed-loop examples, where every column of Xref is the same set point
       (tinympc/TinyMPC/examples/quadrotor_hovering.cpp:60-66).  batch*nx; Xref must then be NULL.  4 nx bytes cross the
       bus per problem instead of 4 nx N; the incremental fp32 kernels and the lane-group fp64 kernels read the state in
       place of every column, for any other kernel the library replicates it over the horizon on the device first. */
    const float *xref_const;
} tinympc_cuda_batch_in;

typedef struct {
    float *x;           /* batch*nx*N      solution->x */
    float *u;           /* batch*nu*(N-1)  solution->u */
    int   *iter;        /* batch           solution->iter */
    int   *status;      /* batch           work->status (1 / 11) */
    float *residuals;   /* batch*4 or NULL: primal_residual_state, dual_residual_state,
                           primal_residual_input, dual_residual_input (types.hpp:181-184) */
    float *rho;         /* batch or NULL: cache->rho at exit (adaptive rho) */
    /* Compact output: the first control of every problem, solution->u.col(0) -- all a closed-loop user applies
       (quadrotor_hovering.cpp:85-88).  batch*nu or NULL.  With u0 given, x and u may be NULL: the trajectories then
       stay on the device and 4 nu + 8 bytes come back per problem instead of 4 (nx N + nu (N-1)) + 8. */
    float *u0;
} tinympc_cuda_batch_out;

/* ---- life cycle ---------------------------------------------------------------------------- */
/* devices: list of CUDA ordinals to shard batches over (contiguous split by problem index, no
   collective); n_devices <= 0 means "the current device only". */
int  tinympc_cuda_create(tinympc_cuda_solver **out, const int *devices, int n_devices);
int  tinympc_cuda_destroy(tinympc_cuda_solver *s);
/* replaces tiny_setup's workspace/cache hand-over + tiny_set_bound/cone/linear_constraints +
   tiny_update_settings for the batched path (tiny_api.cpp:21-242, 325-345) */
int  tinympc_cuda_set_family(tinympc_cuda_solver *s, const tinympc_cuda_family *fam);

/* ---- the hot path -------------------------------------------------------------------------- */
/* replaces a loop of { tiny_set_x0; tiny_set_x_ref; tiny_set_u_ref; tiny_solve } over `batch` fresh
   solvers (tiny_api.cpp:321-323 -> admm.cpp:274-389).  Host buffers; H2D, kernel and D2H inside. */
int  tinympc_cuda_solve_batch(tinympc_cuda_solver *s, const tinympc_cuda_batch_in *in, const tinympc_cuda_batch_out *out);
/* same, data already resident on device `dev_index` (index into the create() list); enqueued on
   `stream` (a cudaStream_t, NULL = default stream) and asynchronous with respect to the host.
   ONE call in flight per (solver, dev_index): the call uses that device context's work counter and
   scratch buffers, so issue the next call on the same stream, or after the previous one has
   completed.  Independent concurrent batches need one solver handle each. */
int  tinympc_cuda_solve_batch_device(tinympc_cuda_solver *s, int dev_index, const tinympc_cuda_batch_in *in,
                                     const tinympc_cuda_batch_out *out, void *stream);

/* ---- batches in which every problem brings its own model ---------------------------------------- */
/* Per-problem models: double, one contiguous COLUMN-MAJOR chunk per problem (the layout of tinympc_cuda_family and of
 * tinympc_cuda_precompute_out, so precompute results plug in unchanged).  HOST pointers for _solve_batch_models, DEVICE
 * pointers (16-byte aligned) for _solve_batch_models_device. */
typedef struct {
    const double *Adyn, *Bdyn;            /* batch*nx*nx, batch*nx*nu */
    const double *fdyn;                   /* batch*nx or NULL = 0 */
    const double *Q, *R;                  /* batch*nx, batch*nu: work->Q, work->R (diag + rho), exactly as tinympc_cuda_family */
    const double *rho;                    /* batch: cache->rho */
    const double *Kinf, *Pinf, *Quu_inv, *AmBKt;   /* batch*(nu*nx | nx*nx | nu*nu | nx*nx) */
    const double *APf, *BPf;              /* batch*nx, batch*nu, or NULL = 0 */
    const double *dKinf_drho, *dPinf_drho;   /* batch*(nu*nx | nx*nx); required when the family has adaptive_rho */
} tinympc_cuda_models;
/* replaces a loop of { tiny_setup(A_b, B_b, Q_b, R_b, rho_b); tiny_set_x0; tiny_set_x_ref; tiny_set_u_ref; tiny_solve } over
 * `batch` solvers whose models differ.  The family set by tinympc_cuda_set_family still supplies nx, nu, N, the settings, the
 * shared bounds, the cones, the linear rows and the adaptive-rho flags; its matrices and cache are not read.  Each problem gets a
 * cold start with ITS OWN model and pristine cache, i.e. what a fresh tiny_setup with that model produces.  Per-problem bounds,
 * compact I/O (xref_const, u0), residuals and rho work as in tinympc_cuda_solve_batch.
 * The host entry shards contiguously over the solver's devices like tinympc_cuda_solve_batch and runs the chunked H2D -> kernel
 * -> D2H pipeline, the model arrays of each chunk travelling with its inputs; the streamed pipeline, the compact launch chain and
 * the claim order (option "order") do not apply to model batches.  The device entry has the rule of
 * tinympc_cuda_solve_batch_device: ONE call in flight per (solver, dev_index).
 * Kernels: with "precision" 64, a box family without adaptive rho, shared bounds and a shape that has a compiled lane-group fp64
 * kernel, its model form; otherwise the warp-per-problem kernel in the arithmetic "precision" selects.  The exact-count mode
 * ("precision" 32 with "mixed" > 0) has no model form: TINYMPC_CUDA_EUNSUPPORTED ("precision" 64 is exact for model batches).
 * A missing required array, adaptive rho without the two sensitivities or (device entry) a misaligned pointer: TINYMPC_CUDA_EINVAL. */
int  tinympc_cuda_solve_batch_models(tinympc_cuda_solver *s, const tinympc_cuda_models *m, const tinympc_cuda_batch_in *in,
                                     const tinympc_cuda_batch_out *out);
int  tinympc_cuda_solve_batch_models_device(tinympc_cuda_solver *s, int dev_index, const tinympc_cuda_models *m,
                                            const tinympc_cuda_batch_in *in, const tinympc_cuda_batch_out *out, void *stream);

/* Full-workspace solve of ONE problem with the reference's warm-start semantics: replaces
 * tiny_solve(solver) on a live TinySolver (tiny_api.cpp:321-323 -> admm.cpp:274-389).  All arrays are HOST,
 * column-major double, exactly the TinyWorkspace members (types.hpp:92-160); the solve starts from whatever
 * they hold (q, r, p, d, duals, slacks of the previous solve) and leaves them as the reference would.
 * Always computed in fp64. */
typedef struct {
    double *x, *u, *q, *r, *p, *d, *v, *vnew, *z, *znew, *g, *y;   /* in-out; x[:,0] is x0 */
    double *vcnew, *zcnew, *gc, *yc;     /* in-out; may be NULL when the cone flags are off */
    double *vlnew, *zlnew, *gl, *yl;     /* in-out; may be NULL when the linear flags are off */
    const double *Xref, *Uref;           /* NULL = zeros */
    double *rho, *Kinf, *Pinf;           /* in-out cache fields adaptive rho mutates persistently (NULL = family values,
                                            not written back); Kinf nu x nx, Pinf nx x nx column-major */
    double *sol_x, *sol_u;               /* out: solution->x, solution->u */
    int *iter, *status, *solved;         /* out */
    double *residuals;                   /* out, 4 values or NULL */
} tinympc_cuda_workspace;
int  tinympc_cuda_solve_workspace(tinympc_cuda_solver *s, const tinympc_cuda_workspace *w);

/* ---- batched cache precompute + rho-sensitivities on the device ------------------------------------ */
/* replaces tiny_precompute_and_set_cache (tinympc/TinyMPC/src/tinympc/tiny_api.cpp:244-318) looped over problems that each
 * bring their OWN dynamics and costs, and TinyMPC.compute_sensitivity_autograd (src/TinyMPC.m:223-241: forward difference in rho,
 * h = 1e-6, both ends solved to 1e-10) for the derivatives adaptive rho needs.  All arrays are HOST, double, one contiguous
 * column-major chunk per problem (Eigen's layout); Q and R are the user's diagonals (before "+ rho").  Runs on the current device. */
typedef struct {
    int batch, nx, nu;                 /* nx <= 16, nu <= 8 */
    const double *Adyn, *Bdyn;         /* batch*nx*nx, batch*nx*nu */
    const double *fdyn;                /* batch*nx or NULL = 0 */
    const double *Q, *R;               /* batch*nx, batch*nu (diagonals) */
    const double *rho;                 /* batch */
} tinympc_cuda_precompute_in;
typedef struct {
    double *Kinf, *Pinf, *Quu_inv, *AmBKt, *APf, *BPf;   /* batch*(nu*nx | nx*nx | nu*nu | nx*nx | nx | nu), required */
    double *dKinf_drho, *dPinf_drho, *dC1_drho, *dC2_drho;   /* optional (give the first two to get any); C1 = Quu_inv, C2 = AmBKt */
    int *iters;                        /* batch or NULL: Riccati iterations until max|Kinf - Kprev| < 1e-5 (at most 1000) */
} tinympc_cuda_precompute_out;
int  tinympc_cuda_precompute_batch(const tinympc_cuda_precompute_in *in, const tinympc_cuda_precompute_out *out);

/* ---- sessions: a batch of warm-started solvers resident on the device ------------------------- */
/* The closed-loop pattern of the reference (tinympc/TinyMPC/examples/quadrotor_hovering.cpp:73-93,
 * examples/cartpole_example_mpc.m:36-44): { tiny_set_x0; tiny_solve; x0 = A x0 + B u0 } repeated on ONE solver whose
 * workspace persists between solves (admm.cpp starts from the q, r, p, d, duals and slacks of the previous solve).
 * A session is `batch` such solvers of the family, each with its own complete TinyWorkspace and cache copy
 * (types.hpp:43-187) in device memory; every call below acts on all of them.  Arithmetic follows the "precision" option
 * at creation (64 reproduces the reference's iteration counts exactly).  All array arguments are HOST pointers. */
typedef struct tinympc_cuda_session tinympc_cuda_session;
/* `batch` solvers as tiny_setup + the constraint setters leave them (cold workspaces, pristine cache), on device `dev_index` */
int  tinympc_cuda_session_create(tinympc_cuda_solver *s, int dev_index, int batch, tinympc_cuda_session **out);
int  tinympc_cuda_session_destroy(tinympc_cuda_session *ss);
/* tiny_set_x0 / tiny_set_x_ref / tiny_set_u_ref on every solver (tiny_api.cpp:375-409).  x0: batch*nx doubles.
 * Xref: batch*nx*N (broadcast 0) or one nx*N array shared by all (broadcast 1); Uref likewise with nu*(N-1). */
int  tinympc_cuda_session_set_x0(tinympc_cuda_session *ss, const double *x0);
int  tinympc_cuda_session_set_x_ref(tinympc_cuda_session *ss, const double *Xref, int broadcast);
int  tinympc_cuda_session_set_u_ref(tinympc_cuda_session *ss, const double *Uref, int broadcast);
/* tiny_solve on every solver, warm start (tiny_api.cpp:321-323 -> admm.cpp:274-389) */
int  tinympc_cuda_session_solve(tinympc_cuda_session *ss);
/* x0 <- Adyn x0 + Bdyn u0 + fdyn on the device; u0 = work->u.col(0) (use_solution 0, quadrotor_hovering.cpp:91) or
 * solution->u.col(0) (use_solution 1, cartpole_example_mpc.m:40-41).  TINYMPC_CUDA_EUNSUPPORTED for nx > 32, x0 untouched. */
int  tinympc_cuda_session_step(tinympc_cuda_session *ss, int use_solution);
/* read one member of every solver into host memory (doubles; iter/status as doubles too):
 * "x0" batch*nx | "x", "sol_x" batch*nx*N (work->x, solution->x) | "u", "sol_u" batch*nu*(N-1) |
 * "iter", "status", "rho" batch | "residuals" batch*4 */
int  tinympc_cuda_session_read(tinympc_cuda_session *ss, const char *field, double *host);

/* ---- knobs and introspection ----------------------------------------------------------------- */
/* option names: "precision" (32 = fp32 arithmetic [default], 64 = fp64 parity mode),
   "mixed" (relative band b in [0,1), 0 = off [default]; with precision 32 and b > 0 the fp32 kernel stops and marks every
   problem whose termination decision (admm.cpp:262-265) has its largest residual/tolerance ratio inside [1-b, 1+b], and an
   fp64 pass re-solves exactly the marked problems: the reference's iteration counts and status codes at close to fp32 speed),
   "refill_min" (a warp of the thread-per-problem kernel claims new problems once that many of its lanes are free; 0 [default]:
   chosen by the kernel from the iterations its problems take),
   "streamed" (1 [default]: tinympc_cuda_solve_batch runs each device's shard as ONE persistent launch that consumes the
   problems while the H2D copies are still arriving and returns results chunk by chunk while it is still solving;
   0: one launch per chunk),
   "compact_streamed" (1 [default]: a host batch with compact I/O -- xref_const in and / or u0 out -- of >= 2^16 problems per
   device runs as one launch chain over the whole shard while its inputs are still arriving in a few chunks of doubling size
   behind an arrival watermark; 0: the chunked pipeline), "compact_in_kernel" (1 [default]: kernels read xref_const in place
   where they can; 0: always replicate it on the device first),
   "compact_early_d2h" (1 [default]: in the exact-count mode of that chain, with PINNED result arrays, the results of the fp32 pass are
   copied back under the fp64 pass and a kernel writes the fp64 results over them through the device alias of the host arrays),
   "order" (1 [default]: a device-resident batch of a box-constrained family, from a few waves of the persistent grid on, is
   bucketed on the device by its expected difficulty |Kinf (x0 - xref_0)| / u_bound and the fp32 kernel claims the hardest
   problems first -- lanes of a warp then hold problems of similar length and the launch ends on the shortest ones, ~9 % on the
   2^20 quadrotor batch; the compact streamed host pipeline orders the later half of a shard of >= 2^18 problems with >= 8 states
   the same way, on "order_sms" [1] SMs the persistent launch leaves free, while the first 1 / "order_from_div" [2] of the shard is
   being solved; scheduling only, the results do not depend on it; 0: index order.  Host batch calls are serialised per device
   within the process, so that SM stays free; a device-resident call or another process that runs a persistent launch on the same
   device at the same time can take it and delay the ordered half -- set "order" 0 for such use),
   "ctas_per_sm" (0 = occupancy API), "chunks" (host pipeline depth, 0 = auto),
   "fixer_sms" (how the exact-count mode schedules its fp64 pass: -2 [default] the sequential two-pass form for device-resident and
   chunked batches, the concurrent producer / consumer pair inside the streamed host pipeline; -1 always sequential; 0 always the
   pair with 13 % of the SMs left to the consumer; n > 0 the pair with n SMs),
   "variant" (kernel tuning variant, 0 = default; 7 = costate recursion instead of the impulse-response backward pass of the
   fp32 quadrotor kernels, 5 = direct-form fp32 kernels, 6 = thread-per-problem fp64 kernels, 9 = plain state layout) */
int  tinympc_cuda_set_option(tinympc_cuda_solver *s, const char *name, double value);
int  tinympc_cuda_device_count(void);
int  tinympc_cuda_num_devices(const tinympc_cuda_solver *s);
/* name of the kernel the last solve launched, and the number of kernel launches so far */
const char *tinympc_cuda_last_kernel(const tinympc_cuda_solver *s);
long long tinympc_cuda_launch_count(const tinympc_cuda_solver *s);
/* last tinympc_cuda_solve_batch(): ms[0] host wall time of the call, ms[1] summed device time of its kernels
   (CUDA events, max over devices), ms[2] number of pipeline chunks */
int  tinympc_cuda_last_timing(const tinympc_cuda_solver *s, double ms[3]);
/* option "pass_timing" = 1: a device-resident exact-count solve (sequential form) records CUDA events around its two passes on the
   caller's stream; ms[0] = fp32 pass, ms[1] = compaction + fp64 pass of the LAST such solve (synchronises on its end).
   TINYMPC_CUDA_ENOTREADY if none was timed. */
int  tinympc_cuda_last_pass_ms(tinympc_cuda_solver *s, double ms[2]);
/* number of problems the last "mixed" solve re-solved in fp64 (after a device-resident solve this synchronises the device) */
long long tinympc_cuda_last_marked(tinympc_cuda_solver *s);
/* upload plan of the compact streamed host pipeline for a shard of n problems (no device needed): chunk c = problems
   [bounds[c], bounds[c+1]); *first_ordered = the first chunk claimed hardest-first when option "order" applies.  Returns the
   number of chunks, -1 if `bounds` (max_bounds ints) is too small. */
int  tinympc_cuda_plan_compact_chunks(int n, int chunks, int order_from_div, int *bounds, int max_bounds, int *first_ordered);
const char *tinympc_cuda_last_error(const tinympc_cuda_solver *s);
const char *tinympc_cuda_version(void);

/* pinned host memory helpers for callers that want full-rate H2D/D2H */
void *tinympc_cuda_host_alloc(size_t bytes);
void  tinympc_cuda_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* TINYMPC_B200_H */
