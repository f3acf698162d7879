// Drives the gateway's 'solve_batch_models' command (tinympc-matlab_b200/matlab/bindings.cpp) the way TinyMPC.m's solve_batch_models
// does, with two cartpole models: the G2 model of examples/cartpole_example_one_solve.m and one with a 30 % larger input gain and
// doubled state weights.  Each model's cache comes from tiny_setup of the host API mirror.  Prints lines that
// tests/test_mex_models.py parses.  Usage: mex_models_driver host|gpu
#include <cstdio>
#include <string>
#include <vector>

#include "mex.h"
#include "tiny_api.hpp"

static mxArray* M(int r, int c, std::initializer_list<double> rowmajor) {
    mxArray* a = mxCreateDoubleMatrix(r, c, mxREAL);
    int k = 0;
    for (double v : rowmajor) { int i = k / c, j = k % c; mxGetPr(a)[j * r + i] = v; ++k; }
    return a;
}
static mxArray* S(double v) { return mxCreateDoubleScalar(v); }
static mxArray* F(int r, int c, double v) { mxArray* a = mxCreateDoubleMatrix(r, c, mxREAL); for (int i = 0; i < r * c; ++i) mxGetPr(a)[i] = v; return a; }
static mxArray* E() { return mxCreateDoubleMatrix(0, 0, mxREAL); }

static std::vector<mxArray*> call(const char* cmd, std::vector<mxArray*> args, int nlhs = 1) {
    std::vector<const mxArray*> in{mxCreateString(cmd)};
    for (auto* a : args) in.push_back(a);
    std::vector<mxArray*> out(8, nullptr);
    mexFunction(nlhs, out.data(), (int)in.size(), in.data());
    return out;
}

int main(int argc, char** argv) {
    const bool gpu = argc > 1 && std::string(argv[1]) == "gpu";
    const int nx = 4, nu = 1, N = 20, NB = 4;   // problems 0, 2: model 0 (G2); 1, 3: model 1
    const double A[16] = {1, 0, 0, 0, 0.01, 1, 0, 0, 0, 0.039, 1.002, 0.458, 0, 0, 0.01, 1.002};   // column-major
    const double B0[4] = {0, 0.02, 0, 0.067}, Qd0[4] = {10, 1, 10, 1};
    mxArray* Am = M(4, 4, {1, 0.01, 0, 0, 0, 1, 0.039, 0, 0, 0, 1.002, 0.01, 0, 0, 0.458, 1.002});
    auto o = call("setup", {Am, M(4, 1, {0, 0.02, 0, 0.067}), F(4, 1, 0), M(4, 4, {10, 0, 0, 0, 0, 1, 0, 0, 0, 0, 10, 0, 0, 0, 0, 1}),
                            M(1, 1, {1}), S(1.0), S(4), S(1), S(20), S(0)});
    std::printf("setup_status %g\n", mxGetScalar(o[0]));
    call("set_bound_constraints", {F(4, 20, -1e17), F(4, 20, 1e17), F(1, 19, -0.5), F(1, 19, 0.5), S(0)}, 0);
    call("update_settings", {S(1e-4), S(1e-4), S(100), S(1), S(1), S(1), S(0), S(0), S(0), S(0), S(0), S(0.1), S(10), S(1), S(0)}, 0);
    // per-problem model arrays, one MATLAB page per problem
    mxArray *mA = F(nx * nx, NB, 0), *mB = F(nx * nu, NB, 0), *mQ = F(nx, NB, 0), *mR = F(nu, NB, 0), *mrho = F(1, NB, 0);
    mxArray *mK = F(nu * nx, NB, 0), *mP = F(nx * nx, NB, 0), *mQi = F(nu * nu, NB, 0), *mAK = F(nx * nx, NB, 0);
    for (int b = 0; b < NB; ++b) {
        const int model = b % 2;
        tinyMatrix a = tinyMatrix::Zero(nx, nx), bm = tinyMatrix::Zero(nx, nu), f = tinyMatrix::Zero(nx, 1), q = tinyMatrix::Zero(nx, nx),
                   r = tinyMatrix::Zero(nu, nu);
        for (int i = 0; i < 16; ++i) a.data()[i] = A[i];
        for (int i = 0; i < 4; ++i) { bm.data()[i] = B0[i] * (model ? 1.3 : 1.0); q(i, i) = Qd0[i] * (model ? 2.0 : 1.0); }
        r(0, 0) = 1.0;
        TinySolver* s = nullptr;
        if (tiny_setup(&s, a, bm, f, q, r, 1.0, nx, nu, N, 0) != 0) { std::printf("tiny_setup_failed\n"); return 1; }
        auto put = [&](mxArray* dst, const double* src, int n) { for (int i = 0; i < n; ++i) mxGetPr(dst)[b * n + i] = src[i]; };
        put(mA, a.data(), nx * nx); put(mB, bm.data(), nx * nu); put(mQ, s->work->Q.data(), nx); put(mR, s->work->R.data(), nu);
        put(mrho, &s->cache->rho, 1); put(mK, s->cache->Kinf.data(), nu * nx); put(mP, s->cache->Pinf.data(), nx * nx);
        put(mQi, s->cache->Quu_inv.data(), nu * nu); put(mAK, s->cache->AmBKt.data(), nx * nx);
        tiny_free(s);
    }
    mxArray* X0 = F(nx, NB, 0);
    for (int b = 0; b < NB; ++b) mxGetPr(X0)[nx * b] = 0.5;
    auto models = [&](mxArray* K) { return std::vector<mxArray*>{X0, E(), E(), mA, mB, E(), mQ, mR, mrho, K, mP, mQi, mAK, E(), E(), E(), E(), S(0)}; };
    try { call("solve_batch_models", {X0, E(), E()}, 0); } catch (const MexError& e) { std::printf("error_id %s\n", e.id.c_str()); }
    try { auto a = models(F(2, NB, 0)); call("solve_batch_models", a, 0); } catch (const MexError& e) { std::printf("error_id %s\n", e.id.c_str()); }
    if (!gpu) { std::printf("host_only_done\n"); return 0; }
    try { call("solve_batch_models", models(E()), 0); } catch (const MexError& e) { std::printf("error_id %s\n", e.id.c_str()); }
    call("set_option", {mxCreateString("precision"), S(64)}, 0);
    o = call("solve_batch_models", models(mK), 4);
    const int* it = static_cast<const int*>(mxGetData(o[2]));
    const int* st = static_cast<const int*>(mxGetData(o[3]));
    const float* U = static_cast<const float*>(mxGetData(o[1]));
    std::printf("models_iter %d %d %d %d\n", it[0], it[1], it[2], it[3]);
    std::printf("models_status %d %d %d %d\n", st[0], st[1], st[2], st[3]);
    std::printf("models_u0 %.7f %.7f %.7f %.7f\n", U[0], U[(N - 1)], U[2 * (N - 1)], U[3 * (N - 1)]);
    std::printf("models_done\n");
    return 0;
}
