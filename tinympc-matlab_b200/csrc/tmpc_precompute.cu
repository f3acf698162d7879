// tmpc_precompute.cu -- batched cache precompute + rho-sensitivities on the device (SURVEY 8f-2).
//
// Reference: tiny_precompute_and_set_cache, tinympc/TinyMPC/src/tinympc/tiny_api.cpp:244-318 (the Riccati recursion that gives
// Kinf, Pinf, Quu_inv, AmBKt, APf, BPf for one (A, B, f, Q, R, rho)), and TinyMPC.m:223-241 compute_sensitivity_autograd (the
// derivatives dKinf/drho, dPinf/drho, dC1/drho, dC2/drho by a forward difference with h = 1e-6, src/TinyMPC.m:336-366 solve_lqr).
// Here every problem of a batch brings its OWN (A, B, f, Q, R, rho): one warp per problem, all matrices of the recursion in
// shared memory in double, lanes over the elements of each product, the nu x nu inverse by Gauss-Jordan with partial pivoting
// on lane 0's say-so (nu <= 8 in every shipped model).  The recursion is strictly sequential in its iterations (<= 1000, each a
// handful of <= 12 x 12 products), so the parallelism is the batch -- and the elements of a product inside the warp.
#include <cuda_runtime.h>

#include <algorithm>

#include "../../include/tinympc_b200.h"
#include "tmpc_devptr.h"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kMaxNx = 16, kMaxNu = 8;

struct PreParams {
    int batch, nx, nu, max_iter, want_sens;
    double tol, h;
    const double *A, *B, *f, *Q, *R, *rho;           // per problem: nx*nx, nx*nu (column-major), nx, nx (diagonal), nu (diagonal), 1
    double *Kinf, *Pinf, *Quu_inv, *AmBKt, *APf, *BPf;   // per problem, column-major (the tinympc_cuda_models layout)
    double *dKinf, *dPinf, *dC1, *dC2;                // per problem or NULL
    int* iters;                                       // per problem or NULL: Riccati iterations used
};

// C (m x n) = op(X) (m x k) * Y (k x n), all row-major in shared memory; TX: X is stored k x m and used transposed
template <bool TX>
__device__ __forceinline__ void mm(double* C, const double* X, const double* Y, int m, int k, int n, int lane) {
    for (int e = lane; e < m * n; e += 32) {
        const int r = e / n, c = e - r * n;
        double acc = 0;
        for (int j = 0; j < k; ++j) acc = fma(TX ? X[j * m + r] : X[r * k + j], Y[j * n + c], acc);
        C[e] = acc;
    }
    __syncwarp();
}

// G (n x n, row-major) -> Ginv by Gauss-Jordan on the augmented [G | I] in W (n x 2n); every lane owns columns
__device__ void inverse(double* Ginv, const double* G, double* W, int n, int lane) {
    const int n2 = 2 * n;
    for (int e = lane; e < n * n2; e += 32) {
        const int r = e / n2, c = e - r * n2;
        W[e] = c < n ? G[r * n + c] : (c - n == r ? 1.0 : 0.0);
    }
    __syncwarp();
    for (int col = 0; col < n; ++col) {
        int piv = col;                                      // partial pivoting (every lane computes the same answer)
        double best = fabs(W[col * n2 + col]);
        for (int r = col + 1; r < n; ++r) { const double v = fabs(W[r * n2 + col]); if (v > best) { best = v; piv = r; } }
        __syncwarp();
        if (piv != col) for (int c = lane; c < n2; c += 32) { const double t = W[col * n2 + c]; W[col * n2 + c] = W[piv * n2 + c]; W[piv * n2 + c] = t; }
        __syncwarp();
        const double ip = 1.0 / W[col * n2 + col];
        __syncwarp();
        for (int c = lane; c < n2; c += 32) W[col * n2 + c] *= ip;
        __syncwarp();
        for (int e = lane; e < n * n2; e += 32) {
            const int r = e / n2, c = e - r * n2;
            if (r != col && c != col) W[e] = fma(-W[r * n2 + col], W[col * n2 + c], W[e]);
        }
        __syncwarp();
        for (int r = lane; r < n; r += 32) if (r != col) W[r * n2 + col] = 0.0;
        __syncwarp();
    }
    for (int e = lane; e < n * n; e += 32) Ginv[e] = W[(e / n) * n2 + n + (e % n)];
    __syncwarp();
}

struct WarpMem {
    double *A, *B, *P, *Pn, *K, *Kp, *T1, *T2, *G, *Gi, *W, *M, *T3, *Q1, *R1, *f;
    __device__ WarpMem(double* base, int nx, int nu) {
        auto take = [&](int n) { double* p = base; base += n; return p; };
        A = take(nx * nx); B = take(nx * nu); P = take(nx * nx); Pn = take(nx * nx); K = take(nu * nx); Kp = take(nu * nx);
        T1 = take(nu * nx); T2 = take(nu * nx); G = take(nu * nu); Gi = take(nu * nu); W = take(2 * nu * nu); M = take(nx * nx); T3 = take(nx * nx);
        Q1 = take(nx); R1 = take(nu); f = take(nx);
    }
    static __host__ __device__ int size(int nx, int nu) { return 5 * nx * nx + nx * nu + 4 * nu * nx + 4 * nu * nu + 2 * nx + nu; }
};

// One Riccati solve for the warp's (A, B, Q + rho, R + rho): Kinf -> m.K, Pinf -> m.Pn, Quu_inv -> m.Gi, (A - B Kinf) -> m.M.
// stop: max|K - K_prev| < tol (tiny_api.cpp:274: 1e-5, at most 1000 iterations; the sensitivities use the tighter setting of
// TinyMPC.m:350-356).  Returns the iterations used.
__device__ int riccati(const WarpMem& m, int nx, int nu, double rho, const double* Qd, const double* Rd, int max_iter, double tol, int lane) {
    for (int e = lane; e < nx; e += 32) m.Q1[e] = Qd[e] + rho;
    for (int e = lane; e < nu; e += 32) m.R1[e] = Rd[e] + rho;
    for (int e = lane; e < nx * nx; e += 32) m.P[e] = (e / nx == e % nx) ? rho : 0.0;      // Ptp1 = rho I (tiny_api.cpp:265)
    for (int e = lane; e < nu * nx; e += 32) m.Kp[e] = 0.0;
    __syncwarp();
    int it = 0;
    for (; it < max_iter; ++it) {
        // Kinf = (R1 + B' P B)^-1 B' P A
        mm<true>(m.T1, m.B, m.P, nu, nx, nx, lane);                     // B' P
        mm<false>(m.G, m.T1, m.B, nu, nx, nu, lane);                    // B' P B
        for (int e = lane; e < nu; e += 32) m.G[e * nu + e] += m.R1[e];
        __syncwarp();
        inverse(m.Gi, m.G, m.W, nu, lane);
        mm<false>(m.T2, m.T1, m.A, nu, nx, nx, lane);                   // B' P A
        mm<false>(m.K, m.Gi, m.T2, nu, nu, nx, lane);
        // Pinf = Q1 + A' P (A - B Kinf)
        mm<false>(m.M, m.B, m.K, nx, nu, nx, lane);
        for (int e = lane; e < nx * nx; e += 32) m.M[e] = m.A[e] - m.M[e];
        __syncwarp();
        mm<true>(m.T3, m.A, m.P, nx, nx, nx, lane);                     // A' P
        mm<false>(m.Pn, m.T3, m.M, nx, nx, nx, lane);
        for (int e = lane; e < nx; e += 32) m.Pn[e * nx + e] += m.Q1[e];
        double dmax = 0;
        for (int e = lane; e < nu * nx; e += 32) dmax = fmax(dmax, fabs(m.K[e] - m.Kp[e]));
        for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(FULL, dmax, o));
        __syncwarp();
        if (dmax < tol) { ++it; break; }
        for (int e = lane; e < nu * nx; e += 32) m.Kp[e] = m.K[e];
        for (int e = lane; e < nx * nx; e += 32) m.P[e] = m.Pn[e];
        __syncwarp();
    }
    // cached terms from the FINAL Pinf (tiny_api.cpp:286-287): Quu_inv = (R1 + B' Pinf B)^-1, A - B Kinf
    mm<true>(m.T1, m.B, m.Pn, nu, nx, nx, lane);
    mm<false>(m.G, m.T1, m.B, nu, nx, nu, lane);
    for (int e = lane; e < nu; e += 32) m.G[e * nu + e] += m.R1[e];
    __syncwarp();
    inverse(m.Gi, m.G, m.W, nu, lane);
    mm<false>(m.M, m.B, m.K, nx, nu, nx, lane);
    for (int e = lane; e < nx * nx; e += 32) m.M[e] = m.A[e] - m.M[e];
    __syncwarp();
    return it;
}

// Between the column-major arrays of one problem in global memory (element e = row e % rows, column e / rows) and the row-major
// matrices the recursion keeps in shared memory; lanes walk the global side contiguously.
__device__ __forceinline__ void load_cm(double* S, const double* G, int rows, int cols, int lane) {
    for (int e = lane; e < rows * cols; e += 32) S[(e % rows) * cols + e / rows] = G[e];
}
__device__ __forceinline__ void store_cm(double* G, const double* S, int rows, int cols, int lane) {
    for (int e = lane; e < rows * cols; e += 32) G[e] = S[(e % rows) * cols + e / rows];
}
// G <- (S - G) / h, the forward difference of the sensitivities over the base point G holds
__device__ __forceinline__ void diff_cm(double* G, const double* S, int rows, int cols, double ih, int lane) {
    for (int e = lane; e < rows * cols; e += 32) G[e] = (S[(e % rows) * cols + e / rows] - G[e]) * ih;
}

__global__ void __launch_bounds__(128) precompute_kernel(const PreParams p) {
    extern __shared__ __align__(16) double pre_smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nx = p.nx, nu = p.nu;
    const WarpMem m(pre_smem + (size_t)wib * WarpMem::size(nx, nu), nx, nu);
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < p.batch; b += nwarps) {
        load_cm(m.A, p.A + (size_t)b * nx * nx, nx, nx, lane);
        load_cm(m.B, p.B + (size_t)b * nx * nu, nx, nu, lane);
        for (int e = lane; e < nx; e += 32) m.f[e] = p.f ? p.f[(size_t)b * nx + e] : 0.0;
        __syncwarp();
        const double rho = p.rho[b];
        const double* Qd = p.Q + (size_t)b * nx;
        const double* Rd = p.R + (size_t)b * nu;
        const int it = riccati(m, nx, nu, rho, Qd, Rd, p.max_iter, p.tol, lane);
        if (p.iters && lane == 0) p.iters[b] = it;
        double* oK = p.Kinf + (size_t)b * nu * nx; double* oP = p.Pinf + (size_t)b * nx * nx;
        double* oQ = p.Quu_inv + (size_t)b * nu * nu; double* oA = p.AmBKt + (size_t)b * nx * nx;
        store_cm(oK, m.K, nu, nx, lane);
        store_cm(oP, m.Pn, nx, nx, lane);
        for (int e = lane; e < nx * nx; e += 32) oA[e] = m.M[e];     // AmBKt = (A - B K)': column-major AmBKt is row-major A - B K
        store_cm(oQ, m.Gi, nu, nu, lane);
        // APf = AmBKt Pinf f, BPf = B' Pinf f   (tiny_api.cpp:290-291)
        for (int r = lane; r < nx; r += 32) { double acc = 0; for (int c = 0; c < nx; ++c) acc = fma(m.Pn[r * nx + c], m.f[c], acc); m.T3[r] = acc; }
        __syncwarp();
        for (int r = lane; r < nx; r += 32) { double acc = 0; for (int c = 0; c < nx; ++c) acc = fma(m.M[c * nx + r], m.T3[c], acc); p.APf[(size_t)b * nx + r] = acc; }
        for (int a = lane; a < nu; a += 32) { double acc = 0; for (int c = 0; c < nx; ++c) acc = fma(m.B[c * nu + a], m.T3[c], acc); p.BPf[(size_t)b * nu + a] = acc; }
        __syncwarp();
        if (p.want_sens) {
            // forward difference in rho (TinyMPC.m:223-241), both ends solved to the tight tolerance of its iterative branch
            // (TinyMPC.m:350-356: norm(K - K_prev) < 1e-10, at most 5000 iterations).  The base point is re-solved with that
            // tolerance too -- differencing a 1e-5-converged K against a 1e-10-converged one would swamp h = 1e-6.
            double* dK = p.dKinf + (size_t)b * nu * nx; double* dP = p.dPinf + (size_t)b * nx * nx;
            double* d1 = p.dC1 ? p.dC1 + (size_t)b * nu * nu : nullptr; double* d2 = p.dC2 ? p.dC2 + (size_t)b * nx * nx : nullptr;
            riccati(m, nx, nu, rho, Qd, Rd, 5000, 1e-10, lane);
            store_cm(dK, m.K, nu, nx, lane);
            store_cm(dP, m.Pn, nx, nx, lane);
            if (d2) for (int e = lane; e < nx * nx; e += 32) d2[e] = m.M[e];
            if (d1) store_cm(d1, m.Gi, nu, nu, lane);
            __syncwarp();
            riccati(m, nx, nu, rho + p.h, Qd, Rd, 5000, 1e-10, lane);
            const double ih = 1.0 / p.h;
            diff_cm(dK, m.K, nu, nx, ih, lane);
            diff_cm(dP, m.Pn, nx, nx, ih, lane);
            if (d2) for (int e = lane; e < nx * nx; e += 32) d2[e] = (m.M[e] - d2[e]) * ih;
            if (d1) diff_cm(d1, m.Gi, nu, nu, ih, lane);
            __syncwarp();
        }
    }
}

struct Dev {
    void* p = nullptr;
    cudaError_t put(const void* h, size_t bytes) {
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess && h) e = cudaMemcpy(p, h, bytes, cudaMemcpyHostToDevice);
        return e;
    }
    ~Dev() { if (p) cudaFree(p); }
};

// shape and required arrays, the same for both entries
int check_args(const tinympc_cuda_precompute_in* in, const tinympc_cuda_precompute_out* out) {
    if (!in || !out) return TINYMPC_CUDA_EINVAL;
    if (in->batch < 0 || in->nx < 1 || in->nu < 1 || in->nx > kMaxNx || in->nu > kMaxNu) return TINYMPC_CUDA_EINVAL;
    if (in->batch == 0) return TINYMPC_CUDA_OK;
    if (!in->Adyn || !in->Bdyn || !in->Q || !in->R || !in->rho) return TINYMPC_CUDA_EINVAL;
    if (!out->Kinf || !out->Pinf || !out->Quu_inv || !out->AmBKt || !out->APf || !out->BPf) return TINYMPC_CUDA_EINVAL;
    return TINYMPC_CUDA_OK;
}

PreParams params_of(const tinympc_cuda_precompute_in* in, const tinympc_cuda_precompute_out* out) {
    PreParams p{};
    p.batch = in->batch; p.nx = in->nx; p.nu = in->nu; p.max_iter = 1000; p.tol = 1e-5; p.h = 1e-6;
    p.want_sens = out->dKinf_drho && out->dPinf_drho ? 1 : 0;
    p.A = in->Adyn; p.B = in->Bdyn; p.f = in->fdyn; p.Q = in->Q; p.R = in->R; p.rho = in->rho;
    p.Kinf = out->Kinf; p.Pinf = out->Pinf; p.Quu_inv = out->Quu_inv; p.AmBKt = out->AmBKt; p.APf = out->APf; p.BPf = out->BPf;
    if (p.want_sens) { p.dKinf = out->dKinf_drho; p.dPinf = out->dPinf_drho; p.dC1 = out->dC1_drho; p.dC2 = out->dC2_drho; }
    p.iters = out->iters;
    return p;
}

// the kernel on `stream` over device arrays (p's pointers); no allocation, copy or synchronisation
cudaError_t enqueue(const PreParams& p, cudaStream_t stream) {
    const int warps_per_cta = 4;
    const size_t smem = sizeof(double) * WarpMem::size(p.nx, p.nu) * warps_per_cta;
    cudaError_t e = cudaFuncSetAttribute(precompute_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int sms = 0, dev = 0;
    if (e == cudaSuccess) e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const int grid = std::max(1, std::min((p.batch + warps_per_cta - 1) / warps_per_cta, sms * 4));
    precompute_kernel<<<grid, warps_per_cta * 32, smem, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace

extern "C" int tinympc_cuda_precompute_batch(const tinympc_cuda_precompute_in* in, const tinympc_cuda_precompute_out* out) {
    if (int rc = check_args(in, out)) return rc;
    const int B = in->batch, nx = in->nx, nu = in->nu;
    if (B == 0) return TINYMPC_CUDA_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return TINYMPC_CUDA_ENODEVICE; }
    const size_t nxx = (size_t)nx * nx, nxu = (size_t)nx * nu, nuu = (size_t)nu * nu;
    const bool sens = out->dKinf_drho && out->dPinf_drho;
    // the kernel reads and writes the host entry's column-major layout as it is: upload, kernel, download
    Dev dA, dB, df, dQ, dR, drho, oK, oP, oQ, oA, oAPf, oBPf, sK, sP, s1, s2, dit;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    ok(dA.put(in->Adyn, sizeof(double) * B * nxx)); ok(dB.put(in->Bdyn, sizeof(double) * B * nxu));
    if (in->fdyn) ok(df.put(in->fdyn, sizeof(double) * B * nx));
    ok(dQ.put(in->Q, sizeof(double) * B * nx)); ok(dR.put(in->R, sizeof(double) * B * nu)); ok(drho.put(in->rho, sizeof(double) * B));
    ok(oK.put(nullptr, sizeof(double) * B * nxu)); ok(oP.put(nullptr, sizeof(double) * B * nxx)); ok(oQ.put(nullptr, sizeof(double) * B * nuu));
    ok(oA.put(nullptr, sizeof(double) * B * nxx)); ok(oAPf.put(nullptr, sizeof(double) * B * nx)); ok(oBPf.put(nullptr, sizeof(double) * B * nu));
    ok(dit.put(nullptr, sizeof(int) * B));
    if (sens) {
        ok(sK.put(nullptr, sizeof(double) * B * nxu)); ok(sP.put(nullptr, sizeof(double) * B * nxx));
        if (out->dC1_drho) ok(s1.put(nullptr, sizeof(double) * B * nuu));
        if (out->dC2_drho) ok(s2.put(nullptr, sizeof(double) * B * nxx));
    }
    if (e != cudaSuccess) return TINYMPC_CUDA_ECUDA;
    const tinympc_cuda_precompute_in din{B, nx, nu, (const double*)dA.p, (const double*)dB.p, (const double*)df.p, (const double*)dQ.p,
                                         (const double*)dR.p, (const double*)drho.p};
    const tinympc_cuda_precompute_out dout{(double*)oK.p, (double*)oP.p, (double*)oQ.p, (double*)oA.p, (double*)oAPf.p, (double*)oBPf.p,
                                           (double*)sK.p, (double*)sP.p, (double*)s1.p, (double*)s2.p, (int*)dit.p};
    ok(enqueue(params_of(&din, &dout), nullptr));
    ok(cudaDeviceSynchronize());
    if (e != cudaSuccess) return TINYMPC_CUDA_ECUDA;
    auto fetch = [&](const Dev& d, void* dst, size_t bytes) { if (dst) ok(cudaMemcpy(dst, d.p, bytes, cudaMemcpyDeviceToHost)); };
    fetch(oK, out->Kinf, sizeof(double) * B * nxu); fetch(oP, out->Pinf, sizeof(double) * B * nxx);
    fetch(oQ, out->Quu_inv, sizeof(double) * B * nuu); fetch(oA, out->AmBKt, sizeof(double) * B * nxx);
    fetch(oAPf, out->APf, sizeof(double) * B * nx); fetch(oBPf, out->BPf, sizeof(double) * B * nu);
    fetch(dit, out->iters, sizeof(int) * B);
    if (sens) {
        fetch(sK, out->dKinf_drho, sizeof(double) * B * nxu); fetch(sP, out->dPinf_drho, sizeof(double) * B * nxx);
        fetch(s1, out->dC1_drho, sizeof(double) * B * nuu); fetch(s2, out->dC2_drho, sizeof(double) * B * nxx);
    }
    return e == cudaSuccess ? TINYMPC_CUDA_OK : TINYMPC_CUDA_ECUDA;
}

extern "C" int tinympc_cuda_precompute_batch_device(const tinympc_cuda_precompute_in* in, const tinympc_cuda_precompute_out* out,
                                                    void* stream) {
    if (int rc = check_args(in, out)) return rc;
    if (in->batch == 0) return TINYMPC_CUDA_OK;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return TINYMPC_CUDA_ENODEVICE; }
    const PreParams p = params_of(in, out);
    // every array the kernel will touch: 16-byte aligned device memory of the current device
    for (const void* a : {(const void*)p.A, (const void*)p.B, (const void*)p.f, (const void*)p.Q, (const void*)p.R, (const void*)p.rho,
                          (const void*)p.Kinf, (const void*)p.Pinf, (const void*)p.Quu_inv, (const void*)p.AmBKt, (const void*)p.APf,
                          (const void*)p.BPf, (const void*)p.dKinf, (const void*)p.dPinf, (const void*)p.dC1, (const void*)p.dC2,
                          (const void*)p.iters})
        if (a && !tmpc::device_ptr_on(a, dev)) return TINYMPC_CUDA_EINVAL;
    return enqueue(p, static_cast<cudaStream_t>(stream)) == cudaSuccess ? TINYMPC_CUDA_OK : TINYMPC_CUDA_ECUDA;
}
