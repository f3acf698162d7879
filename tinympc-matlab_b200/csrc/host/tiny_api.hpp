// tiny_api.hpp -- drop-in mirror of the reference C++ API (tinympc/TinyMPC/src/tinympc/tiny_api.hpp:10-50)
// on top of the B200 C ABI (include/tinympc_b200.h).  Same function names, argument meaning and
// error behaviour; tiny_solve() and the new tiny_solve_batch() run on the GPU -- there is no CPU
// solver in this library.
#pragma once
#include "types.hpp"

extern "C" {

// tiny_api.cpp:21-137.  Allocates the five structs, zeroes the workspace, stores diag(Q)+rho / diag(R)+rho,
// precomputes the cache (Riccati fixed point, tiny_api.cpp:244-318) on the host.  0 on success.
int tiny_setup(TinySolver** solverp, tinyMatrix Adyn, tinyMatrix Bdyn, tinyMatrix fdyn, tinyMatrix Q, tinyMatrix R,
               tinytype rho, int nx, int nu, int N, int verbose);
// tiny_api.cpp:139-164 (dimension mismatches are reported on stdout and, like the reference, do not fail the call)
int tiny_set_bound_constraints(TinySolver* solver, tinyMatrix x_min, tinyMatrix x_max, tinyMatrix u_min, tinyMatrix u_max);
// tiny_api.cpp:166-198.  POSITIONAL meaning follows the reference DEFINITION: the first triple lands in
// work->Acx/qcx/cx (state cones), the second in work->Acu/qcu/cu (input cones).  The reference header
// names them the other way round and its callers follow the header (SURVEY.md quirk Q3); callers that
// are ported verbatim therefore keep their behaviour.
int tiny_set_cone_constraints(TinySolver* solver, VectorXi Acx, VectorXi qcx, tinyVector cx, VectorXi Acu, VectorXi qcu, tinyVector cu);
// tiny_api.cpp:200-242
int tiny_set_linear_constraints(TinySolver* solver, tinyMatrix Alin_x, tinyVector blin_x, tinyMatrix Alin_u, tinyVector blin_u);
// tiny_api.cpp:244-318 (adds rho to Q, R once more: with tiny_setup's Q+rho this is the reference's Q+2rho, quirk Q1)
int tiny_precompute_and_set_cache(TinyCache* cache, tinyMatrix Adyn, tinyMatrix Bdyn, tinyMatrix fdyn, tinyMatrix Q, tinyMatrix R,
                                  int nx, int nu, tinytype rho, int verbose);
// tiny_api.cpp:321-323 -> admm.cpp:274-389, executed on the GPU with the full warm-start semantics of the
// workspace.  Returns 0 (converged) / 1 (max_iter), sets work->status 1 / 11; negative on a backend error.
int tiny_solve(TinySolver* solver);
// tiny_api.cpp:325-345
int tiny_update_settings(TinySettings* settings, tinytype abs_pri_tol, tinytype abs_dua_tol, int max_iter, int check_termination,
                         int en_state_bound, int en_input_bound, int en_state_soc, int en_input_soc, int en_state_linear,
                         int en_input_linear);
// tiny_api.cpp:347-373
int tiny_set_default_settings(TinySettings* settings);
// tiny_api.cpp:375-409
int tiny_set_x0(TinySolver* solver, tinyVector x0);
int tiny_set_x_ref(TinySolver* solver, tinyMatrix x_ref);
int tiny_set_u_ref(TinySolver* solver, tinyMatrix u_ref);
// tiny_api.cpp:411-472 (hard-coded 12 x 4 quadrotor tables, stored exactly as the reference maps them)
void tiny_initialize_sensitivity_matrices(TinySolver* solver);

// ---------------------------------------------------------------------------------- new entry points
// Solve `in->batch` independent problems of this solver's family (cache, settings, shared constraints
// taken from `solver` as it is NOW) that differ in x0 / Xref / Uref / bounds; cold start per problem.
// 0 on success, a TINYMPC_CUDA_E* code otherwise.  Validates its arguments (unlike quirk Q8).
int tiny_solve_batch(TinySolver* solver, const TinyBatchIn* in, const TinyBatchOut* out);
// The same for problems that each bring their OWN model (dynamics, costs, cache, rho: TinyModelBatch, e.g. from
// tinympc_cuda_precompute_batch): replaces a loop of { tiny_setup(A_b, B_b, Q_b, R_b, rho_b); tiny_set_x0; tiny_solve } over solvers.
// `solver` supplies the shape, settings, shared bounds, cones and linear rows; its own matrices and cache are not used.
int tiny_solve_batch_models(TinySolver* solver, const TinyModelBatch* models, const TinyBatchIn* in, const TinyBatchOut* out);
// devices to shard batches over (default: the current CUDA device); precision 32 / 64 and other knobs of
// tinympc_cuda_set_option
int tiny_b200_set_devices(TinySolver* solver, const int* devices, int n_devices);
int tiny_b200_set_option(TinySolver* solver, const char* name, double value);
const char* tiny_b200_last_error(const TinySolver* solver);
void* tiny_b200_cuda_handle(TinySolver* solver);   // the tinympc_cuda_solver* (family uploaded), for device-resident batches
// the reference has no destructor for what tiny_setup allocates (SURVEY.md section 8b "Ownership"); this one frees all of it
void tiny_free(TinySolver* solver);

}  // extern "C"
