// bindings.cpp -- MEX gateway `tinympc_matlab('<command>', args...)` of the B200 build.
//
// Mirrors the command surface of the reference gateway (src/bindings.cpp:641-692: 17 string-dispatched
// commands, one global solver, real-double inputs, int32-or-double index vectors, auto-enabling of the
// constraint flags, errors as mexErrMsgIdAndTxt("TinyMPC:<Id>", ...)) and adds 'solve_batch', 'set_option' and 'session_*'.  All solves
// run on the GPU through the host C++ mirror (csrc/host/tiny_api.hpp) -> C ABI (include/tinympc_b200.h).
// Build inside MATLAB:  mex -I<repo>/tinympc-matlab_b200/csrc/host bindings.cpp -L<repo>/tinympc-matlab_b200 -ltinympc_b200
// (tests build it against tests/stub_mex/mex.h, since neither MATLAB nor mex.h exist in the build image).
#include <cmath>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "mex.h"
#include "tiny_api.hpp"
#include "codegen.hpp"
#include "tinympc_b200.h"

namespace {

TinySolver* g_solver = nullptr;   // one solver per MEX module, like the reference (src/bindings.cpp:17)
tinympc_cuda_session* g_session = nullptr;   // NEW: a batch of warm-started copies of that solver, resident on the GPU
int g_session_batch = 0;

[[noreturn]] void fail(const char* id, const std::string& msg) {
    mexErrMsgIdAndTxt((std::string("TinyMPC:") + id).c_str(), "%s", msg.c_str());
    throw std::runtime_error(msg);   // not reached inside MATLAB
}
void need_solver() { if (!g_solver) fail("NotInitialized", "Solver not initialized"); }
void need_args(int nrhs, int n, const char* cmd) {
    if (nrhs != n) fail("InvalidInput", std::string(cmd) + " requires " + std::to_string(n) + " input arguments");
}

// real double mxArray -> column-major tinyMatrix (MATLAB and the API agree on the layout)
tinyMatrix to_matrix(const mxArray* a) {
    if (!mxIsDouble(a) || mxIsComplex(a)) fail("InvalidInput", "Input must be a real double array");
    const int r = (int)mxGetM(a), c = (int)mxGetN(a);
    tinyMatrix m = tinyMatrix::Zero(r, c);
    if (r * c) std::memcpy(m.data(), mxGetPr(a), sizeof(double) * (size_t)r * c);
    return m;
}
tinyMatrix to_column(const mxArray* a) {   // 1xK or Kx1 -> Kx1
    tinyMatrix m = to_matrix(a);
    tinyMatrix v = tinyMatrix::Zero((int)m.size(), 1);
    for (int i = 0; i < (int)m.size(); ++i) v(i) = m.data()[i];
    return v;
}
VectorXi to_index_vector(const mxArray* a) {
    const size_t n = mxGetM(a) * mxGetN(a);
    VectorXi v((int)n, 1);
    if (mxIsInt32(a)) {
        const int* p = static_cast<const int*>(mxGetData(a));
        for (size_t i = 0; i < n; ++i) v((int)i) = p[i];
    } else if (mxIsDouble(a)) {
        const double* p = mxGetPr(a);
        for (size_t i = 0; i < n; ++i) v((int)i) = (int)std::lround(p[i]);
    } else {
        fail("InvalidInput", "Input must be int32 or double array");
    }
    return v;
}
mxArray* from_matrix(const tinyMatrix& m) {
    mxArray* a = mxCreateDoubleMatrix(m.rows(), m.cols(), mxREAL);
    if (m.size()) std::memcpy(mxGetPr(a), m.data(), sizeof(double) * m.size());
    return a;
}
int scalar_int(const mxArray* a) { return (int)mxGetScalar(a); }

// ---- per-problem float32 chunk from a MATLAB array dim x steps x B (double: converted; single: used in place)
struct FloatView {
    const float* ptr = nullptr;
    std::vector<float> owned;
};
FloatView float_view(const mxArray* a, size_t expect) {
    FloatView v;
    const size_t n = mxGetNumberOfElements(a);
    if (n == 0) return v;
    if (n != expect) fail("InvalidInput", "batched array has " + std::to_string(n) + " elements, expected " + std::to_string(expect));
    if (mxIsSingle(a)) { v.ptr = static_cast<const float*>(mxGetData(a)); return v; }
    if (!mxIsDouble(a) || mxIsComplex(a)) fail("InvalidInput", "batched inputs must be real double or single");
    const double* p = mxGetPr(a);
    v.owned.resize(n);
    for (size_t i = 0; i < n; ++i) v.owned[i] = (float)p[i];
    v.ptr = v.owned.data();
    return v;
}

// ------------------------------------------------------------------------------------------ commands
void drop_session();
void cmd_setup(int, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 10, "setup");   // A, B, fdyn, Q, R, rho, nx, nu, N, verbose
    const double rho = mxGetScalar(prhs[5]);
    const int nx = scalar_int(prhs[6]), nu = scalar_int(prhs[7]), N = scalar_int(prhs[8]), verbose = scalar_int(prhs[9]);
    if (verbose) mexPrintf("Setting up TinyMPC solver with nx=%d, nu=%d, N=%d, rho=%f\n", nx, nu, N, rho);
    TinySolver* s = nullptr;
    const int status = tiny_setup(&s, to_matrix(prhs[0]), to_matrix(prhs[1]), to_matrix(prhs[2]), to_matrix(prhs[3]), to_matrix(prhs[4]), rho,
                                  nx, nu, N, verbose);
    if (status != 0) { tiny_free(s); fail("SetupFailed", "tiny_setup failed with status " + std::to_string(status)); }
    drop_session();      // a live session belongs to the solver that is about to go
    tiny_free(g_solver);
    g_solver = s;
    plhs[0] = mxCreateDoubleScalar(0);
}
void cmd_set_x0(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 2, "set_x0"); need_solver();
    if (tiny_set_x0(g_solver, to_column(prhs[0])) != 0) fail("SetX0Failed", "tiny_set_x0 failed");
}
void cmd_set_x_ref(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 2, "set_x_ref"); need_solver();
    if (tiny_set_x_ref(g_solver, to_matrix(prhs[0])) != 0) fail("SetXRefFailed", "tiny_set_x_ref failed");
}
void cmd_set_u_ref(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 2, "set_u_ref"); need_solver();
    if (tiny_set_u_ref(g_solver, to_matrix(prhs[0])) != 0) fail("SetURefFailed", "tiny_set_u_ref failed");
}
void cmd_set_bound_constraints(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 5, "set_bound_constraints"); need_solver();
    const int status = tiny_set_bound_constraints(g_solver, to_matrix(prhs[0]), to_matrix(prhs[1]), to_matrix(prhs[2]), to_matrix(prhs[3]));
    if (status != 0) fail("SetBoundConstraintsFailed", "status " + std::to_string(status));
    g_solver->settings->en_state_bound = 1;   // auto-enable, src/bindings.cpp:206-207
    g_solver->settings->en_input_bound = 1;
}
void cmd_solve(int, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 1, "solve"); need_solver();
    const int rc = tiny_solve(g_solver);
    if (rc < 0) fail("SolveFailed", std::string("GPU solve failed: ") + tiny_b200_last_error(g_solver));
    if (scalar_int(prhs[0])) mexPrintf("Solve completed with status: %d\n", rc);
    plhs[0] = mxCreateDoubleScalar(0);        // the reference always reports 0 (src/bindings.cpp:230-231)
}
void cmd_get_solution(int, mxArray* plhs[], int nrhs, const mxArray*[]) {
    need_args(nrhs, 1, "get_solution"); need_solver();
    plhs[0] = from_matrix(g_solver->solution->x);
    plhs[1] = from_matrix(g_solver->solution->u);
}
void cmd_get_stats(int, mxArray* plhs[], int nrhs, const mxArray*[]) {
    need_args(nrhs, 1, "get_stats"); need_solver();
    plhs[0] = mxCreateDoubleScalar(g_solver->work->iter);
    plhs[1] = mxCreateDoubleScalar(g_solver->work->status);
    plhs[2] = mxCreateDoubleScalar(g_solver->work->primal_residual_state);
    plhs[3] = mxCreateDoubleScalar(g_solver->work->primal_residual_input);
}
// status = tinympc_matlab('codegen', output_dir, verbose)                                  (src/bindings.cpp:288-309)
void cmd_codegen(int, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 2, "codegen"); need_solver();
    char* dir = mxArrayToString(prhs[0]);
    if (!dir) fail("InvalidInput", "output_dir must be a string");
    const int status = tiny_codegen(g_solver, dir, scalar_int(prhs[1]));
    mxFree(dir);
    plhs[0] = mxCreateDoubleScalar(status);
}
// status = tinympc_matlab('codegen_with_sensitivity', output_dir, dK, dP, dC1, dC2, verbose)   (src/bindings.cpp:481-520)
void cmd_codegen_with_sensitivity(int, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 6, "codegen_with_sensitivity"); need_solver();
    char* dir = mxArrayToString(prhs[0]);
    if (!dir) fail("InvalidInput", "output_dir must be a string");
    tinyMatrix dK = to_matrix(prhs[1]), dP = to_matrix(prhs[2]), dC1 = to_matrix(prhs[3]), dC2 = to_matrix(prhs[4]);
    const int status = tiny_codegen_with_sensitivity(g_solver, dir, &dK, &dP, &dC1, &dC2, scalar_int(prhs[5]));
    mxFree(dir);
    plhs[0] = mxCreateDoubleScalar(status);
}
void drop_session() {
    if (g_session) tinympc_cuda_session_destroy(g_session);
    g_session = nullptr;
    g_session_batch = 0;
}
void cmd_reset(int, mxArray*[], int nrhs, const mxArray*[]) {
    need_args(nrhs, 1, "reset");
    drop_session();
    tiny_free(g_solver);
    g_solver = nullptr;
}
void cmd_set_sensitivity_matrices(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 5, "set_sensitivity_matrices"); need_solver();
    // the reference command validates and then stores nothing (src/bindings.cpp:319-361); here the matrices
    // really reach the cache so that adaptive rho works from MATLAB
    g_solver->cache->dKinf_drho = to_matrix(prhs[0]);
    g_solver->cache->dPinf_drho = to_matrix(prhs[1]);
    g_solver->cache->dC1_drho = to_matrix(prhs[2]);
    g_solver->cache->dC2_drho = to_matrix(prhs[3]);
}
void cmd_set_cache_terms(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 5, "set_cache_terms"); need_solver();
    TinyCache* c = g_solver->cache;
    c->Kinf = to_matrix(prhs[0]); c->Pinf = to_matrix(prhs[1]); c->Quu_inv = to_matrix(prhs[2]); c->AmBKt = to_matrix(prhs[3]);
    c->C1 = c->Quu_inv; c->C2 = c->AmBKt;      // src/bindings.cpp:364-405
}
void cmd_update_settings(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 15, "update_settings"); need_solver();
    TinySettings* st = g_solver->settings;
    tiny_update_settings(st, mxGetScalar(prhs[0]), mxGetScalar(prhs[1]), scalar_int(prhs[2]), scalar_int(prhs[3]), scalar_int(prhs[4]),
                         scalar_int(prhs[5]), scalar_int(prhs[6]), scalar_int(prhs[7]), scalar_int(prhs[8]), scalar_int(prhs[9]));
    st->adaptive_rho = scalar_int(prhs[10]);
    st->adaptive_rho_min = mxGetScalar(prhs[11]);
    st->adaptive_rho_max = mxGetScalar(prhs[12]);
    st->adaptive_rho_enable_clipping = scalar_int(prhs[13]);
}
void cmd_print_problem_data(int, mxArray*[], int nrhs, const mxArray*[]) {
    need_args(nrhs, 0, "print_problem_data"); need_solver();
    const TinySolver* s = g_solver;
    mexPrintf("solution iter: %d\nsolution solved: %d\n", s->solution->iter, s->solution->solved);
    mexPrintf("cache rho: %f\n", s->cache->rho);
    mexPrintf("abs_pri_tol: %f\nabs_dua_tol: %f\nmax_iter: %d\ncheck_termination: %d\n", s->settings->abs_pri_tol, s->settings->abs_dua_tol,
              s->settings->max_iter, s->settings->check_termination);
    mexPrintf("en_state_bound: %d\nen_input_bound: %d\n", s->settings->en_state_bound, s->settings->en_input_bound);
    mexPrintf("nx: %d\nnu: %d\niter: %d\nstatus: %d\n", s->work->nx, s->work->nu, s->work->iter, s->work->status);
}
void cmd_set_linear_constraints(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 4) fail("InvalidInput", "set_linear_constraints requires Alin_x, blin_x, Alin_u, blin_u");
    need_solver();
    tinyMatrix Ax = to_matrix(prhs[0]), Au = to_matrix(prhs[2]);
    tinyMatrix bx = to_column(prhs[1]), bu = to_column(prhs[3]);
    const int status = tiny_set_linear_constraints(g_solver, Ax, bx, Au, bu);
    if (status != 0) fail("SetLinearConstraintsFailed", "status " + std::to_string(status));
    if (Ax.rows() > 0 && bx.rows() > 0) g_solver->settings->en_state_linear = 1;    // src/bindings.cpp:423-430
    if (Au.rows() > 0 && bu.rows() > 0) g_solver->settings->en_input_linear = 1;
}
void cmd_set_cone_constraints(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 6) fail("InvalidInput", "set_cone_constraints requires Acx, qcx, cx, Acu, qcu, cu");
    need_solver();
    // MATLAB order is state-first.  The reference gateway hands (Acu,qcu,cu, Acx,qcx,cx) to a core whose definition is
    // state-first (src/bindings.cpp:465-466 vs tiny_api.cpp:166-168, SURVEY quirk Q3); kept, so MATLAB scripts behave identically.
    VectorXi Acx = to_index_vector(prhs[0]), qcx = to_index_vector(prhs[1]), Acu = to_index_vector(prhs[3]), qcu = to_index_vector(prhs[4]);
    tinyMatrix cx = to_column(prhs[2]), cu = to_column(prhs[5]);
    // The swap is harmless only when both sides carry cones (the rocket example).  With cones on one side only, the reference
    // stores them on the OTHER side and then enables the flag of the side that is empty: they are silently not applied.
    // Reproduced for parity, but said out loud.
    if ((Acx.size() > 0) != (Acu.size() > 0))
        mexPrintf("Warning [TinyMPC:ConeSwap]: cones were given on one side only; like the reference gateway (src/bindings.cpp:465-477) "
                  "this build stores them on the other side and they will NOT be applied. Use the C++ API or solve_batch families for one-sided cones.\n");
    const int status = tiny_set_cone_constraints(g_solver, Acu, qcu, cu, Acx, qcx, cx);
    if (status != 0) fail("SetConeConstraintsFailed", "status " + std::to_string(status));
    if (Acx.size() > 0 && qcx.size() > 0 && cx.size() > 0) g_solver->settings->en_state_soc = 1;   // un-swapped names, :470-477
    if (Acu.size() > 0 && qcu.size() > 0 && cu.size() > 0) g_solver->settings->en_input_soc = 1;
}

// NEW.  [X, U, iter, status, residuals, rho] = tinympc_matlab('solve_batch', X0, Xref, Uref, xmin, xmax, umin, umax, verbose)
//   X0 nx x B; Xref nx x N x B or []; Uref nu x (N-1) x B or []; per-problem bounds in the same shapes or [].
//   double or single inputs (single is passed to the GPU library without a copy); outputs are single.
void cmd_solve_batch(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 8, "solve_batch"); need_solver();
    const TinyWorkspace* w = g_solver->work;
    const size_t nx = w->nx, nu = w->nu, N = w->N;
    if (mxGetM(prhs[0]) != nx) fail("InvalidInput", "X0 must be nx x B");
    const size_t B = mxGetN(prhs[0]);
    const size_t sx = nx * N * B, su = nu * (N - 1) * B;
    FloatView x0 = float_view(prhs[0], nx * B), Xr = float_view(prhs[1], sx), Ur = float_view(prhs[2], su);
    FloatView xl = float_view(prhs[3], sx), xh = float_view(prhs[4], sx), ul = float_view(prhs[5], su), uh = float_view(prhs[6], su);
    const mwSize dx[3] = {(mwSize)nx, (mwSize)N, (mwSize)B}, du[3] = {(mwSize)nu, (mwSize)(N - 1), (mwSize)B};
    plhs[0] = mxCreateNumericArray(3, dx, mxSINGLE_CLASS, mxREAL);
    mxArray* U = mxCreateNumericArray(3, du, mxSINGLE_CLASS, mxREAL);
    const mwSize d1[2] = {(mwSize)B, 1}, d4[2] = {4, (mwSize)B};
    mxArray* it = mxCreateNumericArray(2, d1, mxINT32_CLASS, mxREAL);
    mxArray* st = mxCreateNumericArray(2, d1, mxINT32_CLASS, mxREAL);
    mxArray* rs = mxCreateNumericArray(2, d4, mxSINGLE_CLASS, mxREAL);
    mxArray* rh = mxCreateNumericArray(2, d1, mxSINGLE_CLASS, mxREAL);
    TinyBatchIn in{(int)B, x0.ptr, Xr.ptr, Ur.ptr, xl.ptr, xh.ptr, ul.ptr, uh.ptr};
    TinyBatchOut out{static_cast<float*>(mxGetData(plhs[0])), static_cast<float*>(mxGetData(U)), static_cast<int*>(mxGetData(it)),
                     static_cast<int*>(mxGetData(st)), static_cast<float*>(mxGetData(rs)), static_cast<float*>(mxGetData(rh))};
    const int rc = tiny_solve_batch(g_solver, &in, &out);
    if (rc != 0) fail("SolveBatchFailed", std::string("tiny_solve_batch failed: ") + tiny_b200_last_error(g_solver));
    mxArray* outs[6] = {plhs[0], U, it, st, rs, rh};
    for (int k = 1; k < 6; ++k) { if (k < nlhs || k == 0) plhs[k] = outs[k]; else mxDestroyArray(outs[k]); }
    if (scalar_int(prhs[7])) mexPrintf("solve_batch: %d problems\n", (int)B);
}
// NEW.  [X, U, iter, status, residuals, rho] = tinympc_matlab('solve_batch_models', X0, Xref, Uref, A, B, f, Q, R, rho, Kinf, Pinf,
//                                                                Quu_inv, AmBKt, APf, BPf, dKinf, dPinf, verbose)
//   Problems that each bring their own model (tiny_solve_batch_models).  X0, Xref, Uref as for solve_batch; the model arrays are
//   double, one MATLAB page per problem: A nx x nx x B, B nx x nu x B, Kinf nu x nx x B, Pinf / AmBKt nx x nx x B, Quu_inv nu x nu x B,
//   Q nx x B, R nu x B (diag + rho, as setup stores them), rho B; f, APf, BPf (nx x B, nx x B, nu x B), dKinf, dPinf may be [].
void cmd_solve_batch_models(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 18, "solve_batch_models"); need_solver();
    const TinyWorkspace* w = g_solver->work;
    const size_t nx = w->nx, nu = w->nu, N = w->N;
    if (mxGetM(prhs[0]) != nx) fail("InvalidInput", "X0 must be nx x B");
    const size_t B = mxGetN(prhs[0]);
    const size_t sx = nx * N * B, su = nu * (N - 1) * B;
    FloatView x0 = float_view(prhs[0], nx * B), Xr = float_view(prhs[1], sx), Ur = float_view(prhs[2], su);
    const char* names[14] = {"A", "B", "f", "Q", "R", "rho", "Kinf", "Pinf", "Quu_inv", "AmBKt", "APf", "BPf", "dKinf", "dPinf"};
    const size_t per[14] = {nx * nx, nx * nu, nx, nx, nu, 1, nu * nx, nx * nx, nu * nu, nx * nx, nx, nu, nu * nx, nx * nx};
    const double* p[14];
    for (int k = 0; k < 14; ++k) {
        const mxArray* a = prhs[3 + k];
        p[k] = nullptr;
        if (mxGetNumberOfElements(a) == 0) continue;
        if (!mxIsDouble(a) || mxIsComplex(a)) fail("InvalidInput", std::string(names[k]) + " must be a real double array");
        if (mxGetNumberOfElements(a) != per[k] * B)
            fail("InvalidInput", std::string(names[k]) + " must hold " + std::to_string(per[k]) + " x B values");
        p[k] = mxGetPr(a);
    }
    TinyModelBatch m{p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7], p[8], p[9], p[10], p[11], p[12], p[13]};
    const mwSize dx[3] = {(mwSize)nx, (mwSize)N, (mwSize)B}, du[3] = {(mwSize)nu, (mwSize)(N - 1), (mwSize)B};
    plhs[0] = mxCreateNumericArray(3, dx, mxSINGLE_CLASS, mxREAL);
    mxArray* U = mxCreateNumericArray(3, du, mxSINGLE_CLASS, mxREAL);
    const mwSize d1[2] = {(mwSize)B, 1}, d4[2] = {4, (mwSize)B};
    mxArray* it = mxCreateNumericArray(2, d1, mxINT32_CLASS, mxREAL);
    mxArray* st = mxCreateNumericArray(2, d1, mxINT32_CLASS, mxREAL);
    mxArray* rs = mxCreateNumericArray(2, d4, mxSINGLE_CLASS, mxREAL);
    mxArray* rh = mxCreateNumericArray(2, d1, mxSINGLE_CLASS, mxREAL);
    TinyBatchIn in{(int)B, x0.ptr, Xr.ptr, Ur.ptr, nullptr, nullptr, nullptr, nullptr};
    TinyBatchOut out{static_cast<float*>(mxGetData(plhs[0])), static_cast<float*>(mxGetData(U)), static_cast<int*>(mxGetData(it)),
                     static_cast<int*>(mxGetData(st)), static_cast<float*>(mxGetData(rs)), static_cast<float*>(mxGetData(rh))};
    const int rc = tiny_solve_batch_models(g_solver, &m, &in, &out);
    if (rc != 0) fail("SolveBatchFailed", std::string("tiny_solve_batch_models failed: ") + tiny_b200_last_error(g_solver));
    mxArray* outs[6] = {plhs[0], U, it, st, rs, rh};
    for (int k = 1; k < 6; ++k) { if (k < nlhs) plhs[k] = outs[k]; else mxDestroyArray(outs[k]); }
    if (scalar_int(prhs[17])) mexPrintf("solve_batch_models: %d problems\n", (int)B);
}
// NEW.  tinympc_matlab('set_option', name, value): 'precision' 32|64, 'chunks', 'ctas_per_sm', 'force_wpp'
void cmd_set_option(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 2, "set_option"); need_solver();
    char* name = mxArrayToString(prhs[0]);
    const int rc = tiny_b200_set_option(g_solver, name, mxGetScalar(prhs[1]));
    mxFree(name);
    if (rc != 0) fail("SetOptionFailed", tiny_b200_last_error(g_solver));
}

// NEW.  Sessions: B warm-started copies of the solver on the GPU, the closed loop of examples/cartpole_example_mpc.m:36-44 /
// quadrotor_hovering.cpp:73-93 for B systems at once (include/tinympc_b200.h, tinympc_cuda_session_*).
//   tinympc_matlab('session_create', B)            cold workspaces + pristine cache of the current solver (constraints, settings,
//                                                  options as set so far; 'precision' 64 reproduces the reference's iteration counts)
//   tinympc_matlab('session_set_x0', X0)           nx x B
//   tinympc_matlab('session_set_x_ref', Xref)      nx x N (shared) or nx x N x B;   'session_set_u_ref' likewise with nu x (N-1)
//   tinympc_matlab('session_solve')                tiny_solve on every copy, warm start
//   tinympc_matlab('session_step', use_solution)   x0 <- A x0 + B u0 + f on the device (u0 = work.u(:,1) or solution.u(:,1))
//   v = tinympc_matlab('session_read', field)      'x0' nx x B | 'x','sol_x' nx x N x B | 'u','sol_u' nu x (N-1) x B |
//                                                  'iter','status','rho' B x 1 | 'residuals' 4 x B      (doubles)
//   tinympc_matlab('session_destroy')
void need_session() { if (!g_session) fail("NotInitialized", "No session: call session_create first"); }
void session_check(int rc, const char* what) {
    if (rc != 0) fail("SessionFailed", std::string(what) + ": " + tinympc_cuda_last_error(static_cast<tinympc_cuda_solver*>(tiny_b200_cuda_handle(g_solver))));
}
const double* session_doubles(const mxArray* a, size_t per_problem, int* broadcast) {
    if (!mxIsDouble(a) || mxIsComplex(a)) fail("InvalidInput", "Input must be a real double array");
    const size_t n = mxGetNumberOfElements(a);
    if (n == per_problem * (size_t)g_session_batch) { if (broadcast) *broadcast = 0; }
    else if (broadcast && n == per_problem) *broadcast = 1;
    else fail("InvalidInput", "array has " + std::to_string(n) + " elements, expected " + std::to_string(per_problem) + " per problem");
    return mxGetPr(a);
}
void cmd_session_create(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 1, "session_create"); need_solver();
    const int B = scalar_int(prhs[0]);
    if (B < 1) fail("InvalidInput", "session_create requires a positive number of problems");
    drop_session();
    auto* h = static_cast<tinympc_cuda_solver*>(tiny_b200_cuda_handle(g_solver));   // uploads the family (cache, constraints, settings)
    if (!h) fail("SessionFailed", std::string("no GPU backend: ") + tiny_b200_last_error(g_solver));
    const int rc = tinympc_cuda_session_create(h, 0, B, &g_session);
    if (rc != 0) { g_session = nullptr; fail("SessionFailed", std::string("session_create: ") + tinympc_cuda_last_error(h)); }
    g_session_batch = B;
}
void cmd_session_destroy(int, mxArray*[], int, const mxArray*[]) { drop_session(); }
void cmd_session_set_x0(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 1, "session_set_x0"); need_solver(); need_session();
    session_check(tinympc_cuda_session_set_x0(g_session, session_doubles(prhs[0], g_solver->work->nx, nullptr)), "session_set_x0");
}
void cmd_session_set_x_ref(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 1, "session_set_x_ref"); need_solver(); need_session();
    int bc = 0;
    const double* p = session_doubles(prhs[0], (size_t)g_solver->work->nx * g_solver->work->N, &bc);
    session_check(tinympc_cuda_session_set_x_ref(g_session, p, bc), "session_set_x_ref");
}
void cmd_session_set_u_ref(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 1, "session_set_u_ref"); need_solver(); need_session();
    int bc = 0;
    const double* p = session_doubles(prhs[0], (size_t)g_solver->work->nu * (g_solver->work->N - 1), &bc);
    session_check(tinympc_cuda_session_set_u_ref(g_session, p, bc), "session_set_u_ref");
}
void cmd_session_solve(int, mxArray*[], int, const mxArray*[]) {
    need_solver(); need_session();
    session_check(tinympc_cuda_session_solve(g_session), "session_solve");
}
void cmd_session_step(int, mxArray*[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 1, "session_step"); need_solver(); need_session();
    session_check(tinympc_cuda_session_step(g_session, scalar_int(prhs[0]) ? 1 : 0), "session_step");
}
void cmd_session_read(int, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    need_args(nrhs, 1, "session_read"); need_solver(); need_session();
    char* raw = mxArrayToString(prhs[0]);
    const std::string f = raw ? raw : "";
    mxFree(raw);
    const mwSize nx = g_solver->work->nx, nu = g_solver->work->nu, N = g_solver->work->N, B = (mwSize)g_session_batch;
    mxArray* a = nullptr;
    if (f == "x0") a = mxCreateDoubleMatrix(nx, B, mxREAL);
    else if (f == "x" || f == "sol_x") { const mwSize d[3] = {nx, N, B}; a = mxCreateNumericArray(3, d, mxDOUBLE_CLASS, mxREAL); }
    else if (f == "u" || f == "sol_u") { const mwSize d[3] = {nu, N - 1, B}; a = mxCreateNumericArray(3, d, mxDOUBLE_CLASS, mxREAL); }
    else if (f == "iter" || f == "status" || f == "rho") a = mxCreateDoubleMatrix(B, 1, mxREAL);
    else if (f == "residuals") a = mxCreateDoubleMatrix(4, B, mxREAL);
    else fail("InvalidInput", "unknown session field: " + f);
    plhs[0] = a;
    session_check(tinympc_cuda_session_read(g_session, f.c_str(), mxGetPr(a)), "session_read");
}

struct Command { const char* name; void (*fn)(int, mxArray*[], int, const mxArray*[]); };
const Command kCommands[] = {
    {"setup", cmd_setup}, {"set_x0", cmd_set_x0}, {"set_x_ref", cmd_set_x_ref}, {"set_u_ref", cmd_set_u_ref}, {"solve", cmd_solve},
    {"get_solution", cmd_get_solution}, {"get_stats", cmd_get_stats}, {"codegen", cmd_codegen}, {"reset", cmd_reset},
    {"set_bound_constraints", cmd_set_bound_constraints}, {"set_sensitivity_matrices", cmd_set_sensitivity_matrices},
    {"set_cache_terms", cmd_set_cache_terms}, {"codegen_with_sensitivity", cmd_codegen_with_sensitivity}, {"update_settings", cmd_update_settings},
    {"print_problem_data", cmd_print_problem_data}, {"set_linear_constraints", cmd_set_linear_constraints},
    {"set_cone_constraints", cmd_set_cone_constraints}, {"solve_batch", cmd_solve_batch}, {"solve_batch_models", cmd_solve_batch_models}, {"set_option", cmd_set_option},
    {"session_create", cmd_session_create}, {"session_destroy", cmd_session_destroy}, {"session_set_x0", cmd_session_set_x0},
    {"session_set_x_ref", cmd_session_set_x_ref}, {"session_set_u_ref", cmd_session_set_u_ref}, {"session_solve", cmd_session_solve},
    {"session_step", cmd_session_step}, {"session_read", cmd_session_read},
};

}  // namespace

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 1) fail("InvalidInput", "At least one input argument required");
    char* raw = mxArrayToString(prhs[0]);
    const std::string cmd = raw ? raw : "";
    mxFree(raw);
    for (const Command& c : kCommands)
        if (cmd == c.name) {
            try {
                c.fn(nlhs, plhs, nrhs - 1, prhs + 1);
            } catch (const std::runtime_error&) {
                throw;                                   // already reported through mexErrMsgIdAndTxt (stub build)
            } catch (const std::exception& e) {
                fail("Exception", std::string("Error: ") + e.what());
            }
            return;
        }
    fail("InvalidFunction", "Unknown function: " + cmd);
}
