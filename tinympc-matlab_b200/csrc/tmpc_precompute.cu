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

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kMaxNx = 16, kMaxNu = 8;

struct PreParams {
    int batch, nx, nu, max_iter, want_sens;
    double tol, h;
    const double *A, *B, *f, *Q, *R, *rho;           // per problem: nx*nx, nx*nu (row-major), nx, nx (diagonal), nu (diagonal), 1
    double *Kinf, *Pinf, *Quu_inv, *AmBKt, *APf, *BPf;   // per problem, row-major
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

__global__ void __launch_bounds__(128) precompute_kernel(const PreParams p) {
    extern __shared__ __align__(16) double pre_smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nx = p.nx, nu = p.nu;
    const WarpMem m(pre_smem + (size_t)wib * WarpMem::size(nx, nu), nx, nu);
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < p.batch; b += nwarps) {
        for (int e = lane; e < nx * nx; e += 32) m.A[e] = p.A[(size_t)b * nx * nx + e];
        for (int e = lane; e < nx * nu; e += 32) m.B[e] = p.B[(size_t)b * nx * nu + e];
        for (int e = lane; e < nx; e += 32) m.f[e] = p.f ? p.f[(size_t)b * nx + e] : 0.0;
        __syncwarp();
        const double rho = p.rho[b];
        const double* Qd = p.Q + (size_t)b * nx;
        const double* Rd = p.R + (size_t)b * nu;
        const int it = riccati(m, nx, nu, rho, Qd, Rd, p.max_iter, p.tol, lane);
        if (p.iters && lane == 0) p.iters[b] = it;
        double* oK = p.Kinf + (size_t)b * nu * nx; double* oP = p.Pinf + (size_t)b * nx * nx;
        double* oQ = p.Quu_inv + (size_t)b * nu * nu; double* oA = p.AmBKt + (size_t)b * nx * nx;
        for (int e = lane; e < nu * nx; e += 32) oK[e] = m.K[e];
        for (int e = lane; e < nx * nx; e += 32) { oP[e] = m.Pn[e]; oA[e] = m.M[(e % nx) * nx + e / nx]; }     // AmBKt = (A - B K)'
        for (int e = lane; e < nu * nu; e += 32) oQ[e] = m.Gi[e];
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
            for (int e = lane; e < nu * nx; e += 32) dK[e] = m.K[e];
            for (int e = lane; e < nx * nx; e += 32) { dP[e] = m.Pn[e]; if (d2) d2[e] = m.M[(e % nx) * nx + e / nx]; }
            for (int e = lane; e < nu * nu; e += 32) if (d1) d1[e] = m.Gi[e];
            __syncwarp();
            riccati(m, nx, nu, rho + p.h, Qd, Rd, 5000, 1e-10, lane);
            const double ih = 1.0 / p.h;
            for (int e = lane; e < nu * nx; e += 32) dK[e] = (m.K[e] - dK[e]) * ih;
            for (int e = lane; e < nx * nx; e += 32) { dP[e] = (m.Pn[e] - dP[e]) * ih; if (d2) d2[e] = (m.M[(e % nx) * nx + e / nx] - d2[e]) * ih; }
            for (int e = lane; e < nu * nu; e += 32) if (d1) d1[e] = (m.Gi[e] - d1[e]) * ih;
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

}  // namespace

extern "C" int tinympc_cuda_precompute_batch(const tinympc_cuda_precompute_in* in, const tinympc_cuda_precompute_out* out) {
    if (!in || !out) return TINYMPC_CUDA_EINVAL;
    const int B = in->batch, nx = in->nx, nu = in->nu;
    if (B < 0 || nx < 1 || nu < 1 || nx > kMaxNx || nu > kMaxNu) return TINYMPC_CUDA_EINVAL;
    if (B == 0) return TINYMPC_CUDA_OK;
    if (!in->Adyn || !in->Bdyn || !in->Q || !in->R || !in->rho) return TINYMPC_CUDA_EINVAL;
    if (!out->Kinf || !out->Pinf || !out->Quu_inv || !out->AmBKt || !out->APf || !out->BPf) return TINYMPC_CUDA_EINVAL;
    const bool sens = out->dKinf_drho && out->dPinf_drho;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return TINYMPC_CUDA_ENODEVICE; }
    const size_t nxx = (size_t)nx * nx, nxu = (size_t)nx * nu, nuu = (size_t)nu * nu;
    // host arrays are column-major per problem (the reference's Eigen layout); the kernel works row-major: transpose on the way
    auto to_rowmajor = [&](const double* src, int rows, int cols, double* dst) {
        for (int b = 0; b < B; ++b)
            for (int r = 0; r < rows; ++r)
                for (int c = 0; c < cols; ++c) dst[(size_t)b * rows * cols + r * cols + c] = src[(size_t)b * rows * cols + (size_t)c * rows + r];
    };
    auto to_colmajor = [&](const double* src, int rows, int cols, double* dst) {
        for (int b = 0; b < B; ++b)
            for (int r = 0; r < rows; ++r)
                for (int c = 0; c < cols; ++c) dst[(size_t)b * rows * cols + (size_t)c * rows + r] = src[(size_t)b * rows * cols + r * cols + c];
    };
    double* hA = new double[B * nxx]; double* hB = new double[B * nxu];
    to_rowmajor(in->Adyn, nx, nx, hA);
    to_rowmajor(in->Bdyn, nx, nu, hB);
    Dev dA, dB, df, dQ, dR, drho, oK, oP, oQ, oA, oAPf, oBPf, sK, sP, s1, s2, dit;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    ok(dA.put(hA, sizeof(double) * B * nxx)); ok(dB.put(hB, sizeof(double) * B * nxu));
    delete[] hA; delete[] hB;
    if (in->fdyn) ok(df.put(in->fdyn, sizeof(double) * B * nx));
    ok(dQ.put(in->Q, sizeof(double) * B * nx)); ok(dR.put(in->R, sizeof(double) * B * nu)); ok(drho.put(in->rho, sizeof(double) * B));
    ok(oK.put(nullptr, sizeof(double) * B * nxu)); ok(oP.put(nullptr, sizeof(double) * B * nxx)); ok(oQ.put(nullptr, sizeof(double) * B * nuu));
    ok(oA.put(nullptr, sizeof(double) * B * nxx)); ok(oAPf.put(nullptr, sizeof(double) * B * nx)); ok(oBPf.put(nullptr, sizeof(double) * B * nu));
    ok(dit.put(nullptr, sizeof(int) * B));
    if (sens) {
        ok(sK.put(nullptr, sizeof(double) * B * nxu)); ok(sP.put(nullptr, sizeof(double) * B * nxx));
        ok(s1.put(nullptr, sizeof(double) * B * nuu)); ok(s2.put(nullptr, sizeof(double) * B * nxx));
    }
    if (e != cudaSuccess) return TINYMPC_CUDA_ECUDA;
    PreParams p{};
    p.batch = B; p.nx = nx; p.nu = nu; p.max_iter = 1000; p.tol = 1e-5; p.h = 1e-6; p.want_sens = sens ? 1 : 0;
    p.A = (const double*)dA.p; p.B = (const double*)dB.p; p.f = (const double*)df.p; p.Q = (const double*)dQ.p; p.R = (const double*)dR.p;
    p.rho = (const double*)drho.p;
    p.Kinf = (double*)oK.p; p.Pinf = (double*)oP.p; p.Quu_inv = (double*)oQ.p; p.AmBKt = (double*)oA.p; p.APf = (double*)oAPf.p; p.BPf = (double*)oBPf.p;
    p.dKinf = (double*)sK.p; p.dPinf = (double*)sP.p; p.dC1 = (double*)s1.p; p.dC2 = (double*)s2.p; p.iters = (int*)dit.p;
    const int warps_per_cta = 4;
    const size_t smem = sizeof(double) * WarpMem::size(nx, nu) * warps_per_cta;
    cudaFuncSetAttribute(precompute_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int sms = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = std::max(1, std::min((B + warps_per_cta - 1) / warps_per_cta, sms * 4));
    precompute_kernel<<<grid, warps_per_cta * 32, smem>>>(p);
    ok(cudaGetLastError());
    ok(cudaDeviceSynchronize());
    if (e != cudaSuccess) return TINYMPC_CUDA_ECUDA;
    // back to the host, column-major per problem; the staging buffer holds the largest block fetched (nu x nx or nu x nu when nu > nx)
    double* h = new double[B * std::max({nxx, nxu, nuu})];
    auto fetch = [&](const Dev& d, double* dst, int rows, int cols) {
        if (!dst) return;
        ok(cudaMemcpy(h, d.p, sizeof(double) * B * rows * cols, cudaMemcpyDeviceToHost));
        to_colmajor(h, rows, cols, dst);
    };
    fetch(oK, out->Kinf, nu, nx); fetch(oP, out->Pinf, nx, nx); fetch(oQ, out->Quu_inv, nu, nu); fetch(oA, out->AmBKt, nx, nx);
    ok(cudaMemcpy(out->APf, oAPf.p, sizeof(double) * B * nx, cudaMemcpyDeviceToHost));
    ok(cudaMemcpy(out->BPf, oBPf.p, sizeof(double) * B * nu, cudaMemcpyDeviceToHost));
    if (out->iters) ok(cudaMemcpy(out->iters, dit.p, sizeof(int) * B, cudaMemcpyDeviceToHost));
    if (sens) {
        fetch(sK, out->dKinf_drho, nu, nx); fetch(sP, out->dPinf_drho, nx, nx); fetch(s1, out->dC1_drho, nu, nu); fetch(s2, out->dC2_drho, nx, nx);
    }
    delete[] h;
    return e == cudaSuccess ? TINYMPC_CUDA_OK : TINYMPC_CUDA_ECUDA;
}
