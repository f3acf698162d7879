// tmpc_wpp.h -- host-visible interface of the warp-per-problem kernel (tmpc_wpp.cu)
#pragma once
#include <cuda_runtime.h>

#include "tmpc_common.h"

namespace tmpc {

// Element offsets of one problem's explicit workspace (the TinyWorkspace members, types.hpp:86-187)
struct WppLayout {
    int x, u, q, r, p, d, v, vnew, z, znew, g, y;
    int vcnew, zcnew, gc, yc, vlnew, zlnew, gl, yl;
    int tmp, scalars;      // scalars: [0] rho, [1] iter, [2] status, [3] pri_state, [4] dua_state, [5] pri_input, [6] dua_input, [7] solved
    int zero_end;          // [0, zero_end) is zeroed on a cold start
    int Xref, Uref, xmin, xmax, umin, umax;
    int Kinf, Pinf;        // per-problem cache copies (adaptive rho mutates them), row-major
    int size;
    // models: room for the claimed problem's own model (WppModelBlock) behind Pinf (tinympc_cuda_solve_batch_models)
    static WppLayout make(int nx, int nu, int N, bool models = false);
};

// Element offsets of the model block of a model-batch workspace: the claimed problem's matrices and cache converted to the
// kernel's scalar type, row-major like the family pack (Kinf, Pinf go to WppLayout::Kinf / Pinf).  Starts right behind Pinf.
struct WppModelBlock {
    int A, B, f, Qd, Rd, AmBKt, Quu_inv, APf, BPf, dKinf, dPinf, end;
    __host__ __device__ static WppModelBlock make(const WppLayout& W, int nx, int nu) {
        WppModelBlock M{};
        int o = W.Pinf + nx * nx;
        auto take = [&](int n) { int at = o; o += n; return at; };
        M.A = take(nx * nx); M.B = take(nx * nu); M.f = take(nx); M.Qd = take(nx); M.Rd = take(nu);
        M.AmBKt = take(nx * nx); M.Quu_inv = take(nu * nu); M.APf = take(nx); M.BPf = take(nu);
        M.dKinf = take(nu * nx); M.dPinf = take(nx * nx);
        M.end = o;
        return M;
    }
};

// explicit_workspace = 1: `scratch` holds ONE fully initialised workspace that is iterated in place
// (tiny_solve semantics); 0: cold start per problem from p.x0/Xref/Uref, `warps` scratch workspaces;
// 2: `scratch` holds p.batch persistent workspaces (a session of warm-started solvers), each iterated in place.
// models (device pointers, explicit_workspace 0): every problem iterates with its own model, copied into the model block of
// the warp's workspace (W made with models = true) when the warp claims it; the family pack then supplies the bounds and rows only.
// explicit_workspace 2 with models non-NULL: a model session, every solver's model already in the model block of its workspace
// (wpp_session_models; the pointers are not read)
template <typename T>
cudaError_t wpp_launch(const SolveParams& p, const PackLayout& L, const void* pack, const WppLayout& W, void* scratch, int warps,
                       int explicit_workspace, cudaStream_t st, const tinympc_cuda_models* models = nullptr);

// session helpers: cold workspaces for `batch` solvers; x0 <- A x0 + B u0 + f on every workspace
template <typename T>
cudaError_t wpp_session_init(const SolveParams& p, const PackLayout& L, const void* pack, const WppLayout& W, void* wsp, int batch, cudaStream_t st);
template <typename T>
cudaError_t wpp_session_step(const PackLayout& L, const void* pack, const WppLayout& W, void* wsp, int batch, int use_solution, cudaStream_t st);
// model sessions (W made with models = true): every solver's model m (device pointers, column-major double) -> the model block,
// Kinf, Pinf and rho of its workspace; x0 <- A_b x0 + B_b u0 + f_b with the model block
template <typename T>
cudaError_t wpp_session_models(const WppLayout& W, void* wsp, int batch, int nx, int nu, const tinympc_cuda_models& m, int adaptive,
                               cudaStream_t st);
template <typename T>
cudaError_t wpp_session_step_models(const WppLayout& W, void* wsp, int batch, int nx, int nu, int use_solution, cudaStream_t st);

// device-resident session I/O: packed doubles [batch][width] (src: or one row shared by all, broadcast 1) <-> member `at` (a WppLayout
// offset) of every workspace, in the workspace's type T
template <typename T>
cudaError_t wpp_session_scatter(const WppLayout& W, void* wsp, int batch, int at, int width, const double* src, int broadcast, cudaStream_t st);
template <typename T>
cudaError_t wpp_session_gather(const WppLayout& W, const void* wsp, int batch, int at, int width, double* dst, cudaStream_t st);

}  // namespace tmpc
