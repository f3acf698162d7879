// tmpc_wpp.cu -- "warp per problem" ADMM kernel: the general, faithful form of the hot path.
//
// One warp owns one problem; lanes split the rows of every mat-vec and the elements of every
// element-wise update, the four residual infinity-norms and the adaptive-rho norms are warp-shuffle
// max-reductions, and cone / half-space projections run one time step per lane.  Shapes, constraint
// counts and all feature flags are runtime values, and the complete TinyWorkspace of the reference
// (types.hpp:86-187) is kept explicitly, in the reference's own order of operations
// (admm.cpp:274-389: backward -> forward -> slack -> dual -> linear cost -> iter++ -> adaptive rho ->
// termination -> v = vnew).  It serves
//   (A) tiny_solve(): one solver, full warm-start semantics -- the workspace is uploaded, iterated on
//       and downloaded, so a closed-loop MPC written against the reference API behaves identically;
//   (B) batches whose shape has no specialised thread-per-problem kernel (cold start per problem, one
//       scratch workspace per resident warp).
// The throughput path for the BASELINE shapes is tmpc_tpp3.cuh / tmpc_tpp2.cuh.
#include <cuda_runtime.h>
#include <math_constants.h>

#include "tmpc_common.h"
#include "tmpc_wpp.h"

namespace tmpc {

namespace {

constexpr unsigned FULL = 0xffffffffu;

template <typename T> __device__ __forceinline__ T tabs(T a) { return a < 0 ? -a : a; }
template <typename T> __device__ __forceinline__ T tmax(T a, T b) { return a > b ? a : b; }
template <typename T> __device__ __forceinline__ T tmin(T a, T b) { return a < b ? a : b; }
__device__ __forceinline__ float tsqrt(float a) { return sqrtf(a); }
__device__ __forceinline__ double tsqrt(double a) { return sqrt(a); }

template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = tmax(v, __shfl_xor_sync(FULL, v, o));
    return v;
}

// out[r] = sum_c M[r*C + c] * x[c]   (row-major M, lanes over rows)
// With compile-time shapes (wpp_kernel<T, NX, NU>) the loops below unroll completely: the 2 C loads of a dot product are then
// issued back to back ahead of the dependent FMA chain instead of one load-use round trip per term (the run-time-shaped
// kernel spends ~19 us per ADMM iteration on exactly that).  Same summation order either way.
template <typename T, int UNR>
__device__ __forceinline__ T row_dot(const T* __restrict__ M, int r, int C, const T* x) {
    T acc = 0;
#pragma unroll UNR
    for (int c = 0; c < C; ++c) acc = fma(M[r * C + c], x[c], acc);
    return acc;
}
// out[c] = sum_r M[r*C + c] * x[r]   (transposed product, lanes over columns)
template <typename T, int UNR>
__device__ __forceinline__ T col_dot(const T* __restrict__ M, int c, int R, int C, const T* x) {
    T acc = 0;
#pragma unroll UNR
    for (int r = 0; r < R; ++r) acc = fma(M[r * C + c], x[r], acc);
    return acc;
}

// admm.cpp:39-60 on a contiguous block s[0..dim)
template <typename T>
__device__ void project_soc(T* s, int dim, float mu) {
    const T u0 = s[dim - 1] * static_cast<T>(mu);
    T ss = 0;
    for (int j = 0; j < dim - 1; ++j) ss = fma(s[j], s[j], ss);
    const float a = static_cast<float>(tsqrt(ss));
    const T aT = static_cast<T>(a);
    if (aT <= -u0) {
        for (int j = 0; j < dim; ++j) s[j] = 0;
    } else if (aT <= u0) {
    } else {
        const T fct = T(0.5) * (T(1) + u0 / aT);
        for (int j = 0; j < dim - 1; ++j) s[j] = fct * s[j];
        s[dim - 1] = fct * static_cast<T>(a / mu);
    }
}

}  // namespace

// NXC, NUC > 0: the state / input dimensions are compile-time (instances for the shipped shapes); 0: run-time shapes
template <typename T, int NXC, int NUC>
__global__ void __launch_bounds__(128) wpp_kernel(const SolveParams prm, const PackLayout L, const T* __restrict__ pack,
                                                  const WppLayout W, T* __restrict__ scratch, const int explicit_workspace,
                                                  const int ws_in_smem) {
    constexpr bool MODELS = false;
    [[maybe_unused]] const tinympc_cuda_models M{};
#include "tmpc_wpp_body.inc"
}

// model batches (tinympc_cuda_solve_batch_models): cold start per problem, one scratch workspace per warp with a model block
// (WppLayout::make(..., true))
template <typename T, int NXC, int NUC>
__global__ void __launch_bounds__(128) wpp_mdl_kernel(const SolveParams prm, const PackLayout L, const T* __restrict__ pack,
                                                      const WppLayout W, T* __restrict__ scratch, const int ws_in_smem,
                                                      const tinympc_cuda_models M) {
    constexpr bool MODELS = true;
    constexpr int explicit_workspace = 0;
#include "tmpc_wpp_body.inc"
}

// model sessions (tinympc_cuda_session_create_models): a persistent workspace per solver (WppLayout::make(..., true)), iterated in
// place, whose model block holds the solver's own model
template <typename T, int NXC, int NUC>
__global__ void __launch_bounds__(128) wpp_mdl_session_kernel(const SolveParams prm, const PackLayout L, const T* __restrict__ pack,
                                                              const WppLayout W, T* __restrict__ scratch, const int ws_in_smem) {
    constexpr bool MODELS = true;
    constexpr int explicit_workspace = 2;
    [[maybe_unused]] const tinympc_cuda_models M{};
#include "tmpc_wpp_body.inc"
}

// ---- session helpers (persistent per-problem workspaces) -------------------------------------------------------
// cold workspaces as tiny_setup + the constraint setters leave them (tiny_api.cpp:68-105) with the pristine cache
template <typename T>
__global__ void wpp_session_init_kernel(const SolveParams prm, const PackLayout L, const T* __restrict__ pack, const WppLayout W,
                                        T* __restrict__ wsp, int batch) {
    const int sx = L.nx * L.N, su = L.nu * (L.N - 1);
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < (size_t)batch * W.size; k += (size_t)gridDim.x * blockDim.x) {
        const int e = static_cast<int>(k % W.size);
        T v = 0;
        if (e >= W.xmin && e < W.xmin + sx) v = pack[L.xmin + (e - W.xmin)];
        else if (e >= W.xmax && e < W.xmax + sx) v = pack[L.xmax + (e - W.xmax)];
        else if (e >= W.umin && e < W.umin + su) v = pack[L.umin + (e - W.umin)];
        else if (e >= W.umax && e < W.umax + su) v = pack[L.umax + (e - W.umax)];
        else if (e >= W.Kinf && e < W.Kinf + L.nu * L.nx) v = pack[L.Kinf + (e - W.Kinf)];
        else if (e >= W.Pinf && e < W.Pinf + L.nx * L.nx) v = pack[L.Pinf + (e - W.Pinf)];
        else if (e == W.scalars) v = static_cast<T>(prm.rho);
        else if (e == W.scalars + 2) v = T(11);
        wsp[k] = v;
    }
}
// x0 <- A x0 + B u0 + f for every problem (the "simulate forward" line of quadrotor_hovering.cpp:91); u0 = work->u.col(0)
// (use_solution 0) or solution->u.col(0) = znew.col(0) (use_solution 1, cartpole_example_mpc.m:40-41)
template <typename T>
__global__ void wpp_session_step_kernel(const PackLayout L, const T* __restrict__ pack, const WppLayout W, T* __restrict__ wsp, int batch,
                                        int use_solution) {
    const int nx = L.nx, nu = L.nu;
    constexpr int UNR = 1;
    const int prob = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (prob >= batch) return;
    T* ws = wsp + (size_t)prob * W.size;
    const T* x0 = ws + W.x;
    const T* u0 = ws + (use_solution ? W.znew : W.u);
    T xn = 0;
    if (lane < nx) xn = row_dot<T, UNR>(pack + L.A, lane, nx, x0) + row_dot<T, UNR>(pack + L.B, lane, nu, u0) + pack[L.f + lane];
    __syncwarp();
    if (lane < nx) ws[W.x + lane] = xn;
}

// every solver's model (column-major double, device) -> the model block, Kinf, Pinf and rho of its workspace, row-major T as
// set_family packs a family (the conversion wpp_mdl_kernel makes at claim); one warp per solver
template <typename T>
__global__ void wpp_session_models_kernel(const WppLayout W, T* __restrict__ wsp, int batch, int nx, int nu, const tinympc_cuda_models M,
                                          int adaptive) {
    const int lane = threadIdx.x & 31;
    const WppModelBlock MB = WppModelBlock::make(W, nx, nu);
    for (int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < batch; b += (gridDim.x * blockDim.x) >> 5) {
        T* ws = wsp + (size_t)b * W.size;
        auto cm = [&](int at, const double* src, int rows, int cols) {
            for (int e = lane; e < rows * cols; e += 32)
                ws[at + e] = static_cast<T>(src[(size_t)b * rows * cols + (size_t)(e % cols) * rows + e / cols]);
        };
        auto vec = [&](int at, const double* src, int n) {
            for (int e = lane; e < n; e += 32) ws[at + e] = src ? static_cast<T>(src[(size_t)b * n + e]) : T(0);
        };
        cm(MB.A, M.Adyn, nx, nx); cm(MB.B, M.Bdyn, nx, nu); cm(W.Kinf, M.Kinf, nu, nx); cm(W.Pinf, M.Pinf, nx, nx);
        cm(MB.AmBKt, M.AmBKt, nx, nx); cm(MB.Quu_inv, M.Quu_inv, nu, nu);
        vec(MB.f, M.fdyn, nx); vec(MB.APf, M.APf, nx); vec(MB.BPf, M.BPf, nu); vec(MB.Qd, M.Q, nx); vec(MB.Rd, M.R, nu);
        if (adaptive) { cm(MB.dKinf, M.dKinf_drho, nu, nx); cm(MB.dPinf, M.dPinf_drho, nx, nx); }
        if (lane == 0) ws[W.scalars] = static_cast<T>(M.rho[b]);
    }
}
// x0 <- A_b x0 + B_b u0 + f_b with every solver's own model (the model block)
template <typename T>
__global__ void wpp_session_step_models_kernel(const WppLayout W, T* __restrict__ wsp, int batch, int nx, int nu, int use_solution) {
    constexpr int UNR = 1;
    const int prob = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (prob >= batch) return;
    T* ws = wsp + (size_t)prob * W.size;
    const WppModelBlock MB = WppModelBlock::make(W, nx, nu);
    const T* x0 = ws + W.x;
    const T* u0 = ws + (use_solution ? W.znew : W.u);
    T xn = 0;
    if (lane < nx) xn = row_dot<T, UNR>(ws + MB.A, lane, nx, x0) + row_dot<T, UNR>(ws + MB.B, lane, nu, u0) + ws[MB.f + lane];
    __syncwarp();
    if (lane < nx) ws[W.x + lane] = xn;
}

template <typename T>
cudaError_t wpp_session_models(const WppLayout& W, void* wsp, int batch, int nx, int nu, const tinympc_cuda_models& m, int adaptive,
                               cudaStream_t st) {
    wpp_session_models_kernel<T><<<592, 256, 0, st>>>(W, static_cast<T*>(wsp), batch, nx, nu, m, adaptive);
    return cudaGetLastError();
}
template <typename T>
cudaError_t wpp_session_step_models(const WppLayout& W, void* wsp, int batch, int nx, int nu, int use_solution, cudaStream_t st) {
    if (nx > 32) return cudaErrorInvalidValue;
    wpp_session_step_models_kernel<T><<<(batch + 3) / 4, 128, 0, st>>>(W, static_cast<T*>(wsp), batch, nx, nu, use_solution);
    return cudaGetLastError();
}
template cudaError_t wpp_session_models<float>(const WppLayout&, void*, int, int, int, const tinympc_cuda_models&, int, cudaStream_t);
template cudaError_t wpp_session_models<double>(const WppLayout&, void*, int, int, int, const tinympc_cuda_models&, int, cudaStream_t);
template cudaError_t wpp_session_step_models<float>(const WppLayout&, void*, int, int, int, int, cudaStream_t);
template cudaError_t wpp_session_step_models<double>(const WppLayout&, void*, int, int, int, int, cudaStream_t);

template <typename T>
cudaError_t wpp_session_init(const SolveParams& p, const PackLayout& L, const void* pack, const WppLayout& W, void* wsp, int batch, cudaStream_t st) {
    wpp_session_init_kernel<T><<<592, 256, 0, st>>>(p, L, static_cast<const T*>(pack), W, static_cast<T*>(wsp), batch);
    return cudaGetLastError();
}
template <typename T>
cudaError_t wpp_session_step(const PackLayout& L, const void* pack, const WppLayout& W, void* wsp, int batch, int use_solution, cudaStream_t st) {
    if (L.nx > 32) return cudaErrorInvalidValue;
    wpp_session_step_kernel<T><<<(batch + 3) / 4, 128, 0, st>>>(L, static_cast<const T*>(pack), W, static_cast<T*>(wsp), batch, use_solution);
    return cudaGetLastError();
}
template cudaError_t wpp_session_init<float>(const SolveParams&, const PackLayout&, const void*, const WppLayout&, void*, int, cudaStream_t);
template cudaError_t wpp_session_init<double>(const SolveParams&, const PackLayout&, const void*, const WppLayout&, void*, int, cudaStream_t);
template cudaError_t wpp_session_step<float>(const PackLayout&, const void*, const WppLayout&, void*, int, int, cudaStream_t);
template cudaError_t wpp_session_step<double>(const PackLayout&, const void*, const WppLayout&, void*, int, int, cudaStream_t);

WppLayout WppLayout::make(int nx, int nu, int N, bool models) {
    WppLayout W{};
    const int sx = nx * N, su = nu * (N - 1);
    int o = 0;
    auto take = [&](int n) { int at = o; o += n; return at; };
    // zero-initialised on a cold start: everything up to zero_end
    W.x = take(sx); W.u = take(su); W.q = take(sx); W.r = take(su); W.p = take(sx); W.d = take(su);
    W.v = take(sx); W.vnew = take(sx); W.z = take(su); W.znew = take(su); W.g = take(sx); W.y = take(su);
    W.vcnew = take(sx); W.zcnew = take(su); W.gc = take(sx); W.yc = take(su);
    W.vlnew = take(sx); W.zlnew = take(su); W.gl = take(sx); W.yl = take(su);
    W.tmp = take(nu);
    W.scalars = take(8);
    W.zero_end = o;
    W.Xref = take(sx); W.Uref = take(su);
    W.xmin = take(sx); W.xmax = take(sx); W.umin = take(su); W.umax = take(su);
    W.Kinf = take(nu * nx); W.Pinf = take(nx * nx);
    if (models) o = WppModelBlock::make(W, nx, nu).end;
    W.size = (o + 3) & ~3;
    return W;
}

template <typename T>
cudaError_t wpp_launch(const SolveParams& p, const PackLayout& L, const void* pack, const WppLayout& W, void* scratch, int warps,
                       int explicit_workspace, cudaStream_t st, const tinympc_cuda_models* models) {
    const int block = 128;                       // 4 warps per CTA
    int grid = (warps * 32 + block - 1) / block;
    if (grid < 1) grid = 1;
    const int threads = warps * 32 < block ? warps * 32 : block;
    const T* pk = static_cast<const T*>(pack);
    T* sc = static_cast<T*>(scratch);
    const size_t smem = (size_t)(threads / 32) * W.size * sizeof(T);
    // fp32 workspaces that fit are iterated in shared memory (measured on 65 536 warm-started quadrotor solvers: 15.0 -> 19.9 M
    // solves/s); fp64 ones stay in global memory, where the smaller footprint per CTA keeps more warps resident (13.2 M against
    // 9.2 M solves/s), and so do long horizons that do not fit
    const int in_smem = (sizeof(T) == 4 && smem <= 200 * 1024) ? 1 : 0;
    auto go = [&](auto kernel, auto... args) -> cudaError_t {
        if (in_smem && smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kernel<<<grid, threads, in_smem ? smem : 0, st>>>(p, L, pk, W, sc, args...);
        return cudaGetLastError();
    };
    if (models && explicit_workspace == 2) {
        if (L.nx == 12 && L.nu == 4) return go(wpp_mdl_session_kernel<T, 12, 4>, in_smem);
        if (L.nx == 4 && L.nu == 1) return go(wpp_mdl_session_kernel<T, 4, 1>, in_smem);
        if (L.nx == 6 && L.nu == 3) return go(wpp_mdl_session_kernel<T, 6, 3>, in_smem);
        return go(wpp_mdl_session_kernel<T, 0, 0>, in_smem);
    }
    if (models) {
        if (L.nx == 12 && L.nu == 4) return go(wpp_mdl_kernel<T, 12, 4>, in_smem, *models);
        if (L.nx == 4 && L.nu == 1) return go(wpp_mdl_kernel<T, 4, 1>, in_smem, *models);
        if (L.nx == 6 && L.nu == 3) return go(wpp_mdl_kernel<T, 6, 3>, in_smem, *models);
        return go(wpp_mdl_kernel<T, 0, 0>, in_smem, *models);
    }
    if (L.nx == 12 && L.nu == 4) return go(wpp_kernel<T, 12, 4>, explicit_workspace, in_smem);
    if (L.nx == 4 && L.nu == 1) return go(wpp_kernel<T, 4, 1>, explicit_workspace, in_smem);
    if (L.nx == 6 && L.nu == 3) return go(wpp_kernel<T, 6, 3>, explicit_workspace, in_smem);
    return go(wpp_kernel<T, 0, 0>, explicit_workspace, in_smem);
}
template cudaError_t wpp_launch<float>(const SolveParams&, const PackLayout&, const void*, const WppLayout&, void*, int, int, cudaStream_t,
                                       const tinympc_cuda_models*);
template cudaError_t wpp_launch<double>(const SolveParams&, const PackLayout&, const void*, const WppLayout&, void*, int, int, cudaStream_t,
                                        const tinympc_cuda_models*);

}  // namespace tmpc
