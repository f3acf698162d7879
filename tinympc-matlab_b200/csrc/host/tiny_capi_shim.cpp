// tiny_capi_shim.cpp -- plain-C handles over the C++ API mirror, for hosts that cannot pass C++ objects
// (Python ctypes in tests/bench, the MEX gateway).  One function per tiny_* entry point; matrices are
// column-major double like MATLAB's mxArray data (src/bindings.cpp:20-30 copies exactly such arrays).
#include <cstring>

#include "../../../include/tinympc_b200.h"
#include "tiny_api.hpp"
#include "codegen.hpp"

namespace {
tinyMatrix mat(const double* p, int r, int c) {
    tinyMatrix m = tinyMatrix::Zero(r, c);
    if (p) std::memcpy(m.data(), p, sizeof(double) * (size_t)r * c);
    return m;
}
VectorXi ivec(const int* p, int n) {
    VectorXi v(n > 0 ? n : 0, 1);
    for (int i = 0; i < n; ++i) v(i) = p[i];
    return v;
}
TinySolver* S(void* h) { return static_cast<TinySolver*>(h); }
}  // namespace

extern "C" {

void* tinympc_host_setup(const double* A, const double* B, const double* f, const double* Q, const double* R, double rho, int nx, int nu, int N,
                         int verbose, int* status) {
    TinySolver* s = nullptr;
    int rc = tiny_setup(&s, mat(A, nx, nx), mat(B, nx, nu), mat(f, nx, 1), mat(Q, nx, nx), mat(R, nu, nu), rho, nx, nu, N, verbose);
    if (status) *status = rc;
    if (rc) { tiny_free(s); return nullptr; }
    return s;
}
void tinympc_host_free(void* h) { tiny_free(S(h)); }
/* tiny_codegen / tiny_codegen_with_sensitivity (codegen.hpp); sensitivities column-major or all NULL */
int tinympc_host_codegen(void* h, const char* output_dir, const double* dK, const double* dP, const double* dC1, const double* dC2, int verbose) {
    const TinyWorkspace* w = S(h)->work;
    if (!dK || !dP || !dC1 || !dC2) return tiny_codegen(S(h), output_dir, verbose);
    tinyMatrix a = mat(dK, w->nu, w->nx), b = mat(dP, w->nx, w->nx), c = mat(dC1, w->nu, w->nu), d = mat(dC2, w->nx, w->nx);
    return tiny_codegen_with_sensitivity(S(h), output_dir, &a, &b, &c, &d, verbose);
}

int tinympc_host_set_bound_constraints(void* h, const double* xmin, const double* xmax, const double* umin, const double* umax) {
    const TinyWorkspace* w = S(h)->work;
    return tiny_set_bound_constraints(S(h), mat(xmin, w->nx, w->N), mat(xmax, w->nx, w->N), mat(umin, w->nu, w->N - 1), mat(umax, w->nu, w->N - 1));
}
/* positional order of the reference DEFINITION: first triple = state cones (work->Acx...), second = input cones */
int tinympc_host_set_cone_constraints(void* h, int n_first, const int* A1, const int* q1, const double* c1, int n_second, const int* A2,
                                      const int* q2, const double* c2) {
    return tiny_set_cone_constraints(S(h), ivec(A1, n_first), ivec(q1, n_first), mat(c1, n_first, 1), ivec(A2, n_second), ivec(q2, n_second),
                                     mat(c2, n_second, 1));
}
int tinympc_host_set_linear_constraints(void* h, int nsl, const double* Alin_x, const double* blin_x, int nil, const double* Alin_u,
                                        const double* blin_u) {
    const TinyWorkspace* w = S(h)->work;
    return tiny_set_linear_constraints(S(h), mat(Alin_x, nsl, w->nx), mat(blin_x, nsl, 1), mat(Alin_u, nil, w->nu), mat(blin_u, nil, 1));
}
/* the 15-scalar update_settings of the MEX layer (src/bindings.cpp:548-603) minus `verbose` */
int tinympc_host_update_settings(void* h, double abs_pri_tol, double abs_dua_tol, int max_iter, int check_termination, int en_state_bound,
                                 int en_input_bound, int en_state_soc, int en_input_soc, int en_state_linear, int en_input_linear,
                                 int adaptive_rho, double adaptive_rho_min, double adaptive_rho_max, int adaptive_rho_enable_clipping) {
    TinySettings* st = S(h)->settings;
    int rc = tiny_update_settings(st, abs_pri_tol, abs_dua_tol, max_iter, check_termination, en_state_bound, en_input_bound, en_state_soc,
                                  en_input_soc, en_state_linear, en_input_linear);
    st->adaptive_rho = adaptive_rho; st->adaptive_rho_min = adaptive_rho_min; st->adaptive_rho_max = adaptive_rho_max;
    st->adaptive_rho_enable_clipping = adaptive_rho_enable_clipping;
    return rc;
}
int tinympc_host_get_settings(void* h, double* d3 /* pri, dua, rho_min, rho_max */, int* i11) {
    const TinySettings* st = S(h)->settings;
    d3[0] = st->abs_pri_tol; d3[1] = st->abs_dua_tol; d3[2] = st->adaptive_rho_min; d3[3] = st->adaptive_rho_max;
    const int v[11] = {st->max_iter, st->check_termination, st->en_state_bound, st->en_input_bound, st->en_state_soc, st->en_input_soc,
                       st->en_state_linear, st->en_input_linear, st->adaptive_rho, st->adaptive_rho_enable_clipping, 0};
    std::memcpy(i11, v, sizeof v);
    return 0;
}
int tinympc_host_set_x0(void* h, const double* x0) { return tiny_set_x0(S(h), mat(x0, S(h)->work->nx, 1)); }
int tinympc_host_set_x_ref(void* h, const double* xr) { return tiny_set_x_ref(S(h), mat(xr, S(h)->work->nx, S(h)->work->N)); }
int tinympc_host_set_u_ref(void* h, const double* ur) { return tiny_set_u_ref(S(h), mat(ur, S(h)->work->nu, S(h)->work->N - 1)); }
int tinympc_host_solve(void* h) { return tiny_solve(S(h)); }
int tinympc_host_get_solution(void* h, double* x, double* u) {
    const TinySolver* s = S(h);
    if (x) std::memcpy(x, s->solution->x.data(), sizeof(double) * s->solution->x.size());
    if (u) std::memcpy(u, s->solution->u.data(), sizeof(double) * s->solution->u.size());
    return 0;
}
/* iter, status, primal_residual_state, primal_residual_input as get_stats (src/bindings.cpp:264-285) + the two dual residuals + rho */
int tinympc_host_get_stats(void* h, int* iter, int* status, double* res5) {
    const TinyWorkspace* w = S(h)->work;
    *iter = w->iter; *status = w->status;
    res5[0] = w->primal_residual_state; res5[1] = w->primal_residual_input; res5[2] = w->dual_residual_state; res5[3] = w->dual_residual_input;
    res5[4] = S(h)->cache->rho;
    return 0;
}
int tinympc_host_get_work_u0(void* h, double* u0) { std::memcpy(u0, S(h)->work->u.data(), sizeof(double) * S(h)->work->nu); return 0; }
int tinympc_host_get_cache(void* h, double* Kinf, double* Pinf, double* Quu_inv, double* AmBKt, double* APf, double* BPf) {
    const TinyCache* c = S(h)->cache;
    auto cp = [](double* d, const tinyMatrix& m) { if (d) std::memcpy(d, m.data(), sizeof(double) * m.size()); };
    cp(Kinf, c->Kinf); cp(Pinf, c->Pinf); cp(Quu_inv, c->Quu_inv); cp(AmBKt, c->AmBKt); cp(APf, c->APf); cp(BPf, c->BPf);
    return 0;
}
/* set_cache_terms of the MEX layer (src/bindings.cpp:364-405): also sets C1 = Quu_inv, C2 = AmBKt */
int tinympc_host_set_cache_terms(void* h, const double* Kinf, const double* Pinf, const double* Quu_inv, const double* AmBKt) {
    TinySolver* s = S(h);
    const int nx = s->work->nx, nu = s->work->nu;
    s->cache->Kinf = mat(Kinf, nu, nx); s->cache->Pinf = mat(Pinf, nx, nx);
    s->cache->Quu_inv = mat(Quu_inv, nu, nu); s->cache->AmBKt = mat(AmBKt, nx, nx);
    s->cache->C1 = s->cache->Quu_inv; s->cache->C2 = s->cache->AmBKt;
    return 0;
}
int tinympc_host_init_sensitivity(void* h) { tiny_initialize_sensitivity_matrices(S(h)); return 0; }
int tinympc_host_set_sensitivity(void* h, const double* dK, const double* dP, const double* dC1, const double* dC2) {
    TinySolver* s = S(h);
    const int nx = s->work->nx, nu = s->work->nu;
    s->cache->dKinf_drho = mat(dK, nu, nx); s->cache->dPinf_drho = mat(dP, nx, nx);
    s->cache->dC1_drho = mat(dC1, nu, nu); s->cache->dC2_drho = mat(dC2, nx, nx);
    return 0;
}
/* cold reset of the workspace to the state tiny_setup leaves (tiny_api.cpp:68-105) */
int tinympc_host_reset_workspace(void* h) {
    TinyWorkspace* w = S(h)->work;
    for (tinyMatrix* m : {&w->x, &w->u, &w->q, &w->r, &w->p, &w->d, &w->v, &w->vnew, &w->z, &w->znew, &w->g, &w->y, &w->vc, &w->vcnew, &w->zc,
                          &w->zcnew, &w->gc, &w->yc, &w->vl, &w->vlnew, &w->zl, &w->zlnew, &w->gl, &w->yl})
        m->setZero();
    return 0;
}
int tinympc_host_solve_batch(void* h, const tinympc_cuda_batch_in* in, const tinympc_cuda_batch_out* out) {
    TinyBatchIn bi{in->batch, in->x0, in->Xref, in->Uref, in->x_min, in->x_max, in->u_min, in->u_max};
    TinyBatchOut bo{out->x, out->u, out->iter, out->status, out->residuals, out->rho};
    return tiny_solve_batch(S(h), &bi, &bo);
}
int tinympc_host_solve_batch_models(void* h, const tinympc_cuda_models* m, const tinympc_cuda_batch_in* in, const tinympc_cuda_batch_out* out) {
    TinyBatchIn bi{in->batch, in->x0, in->Xref, in->Uref, in->x_min, in->x_max, in->u_min, in->u_max, in->xref_const};
    TinyBatchOut bo{out->x, out->u, out->iter, out->status, out->residuals, out->rho, out->u0};
    return tiny_solve_batch_models(S(h), m, &bi, &bo);
}
int tinympc_host_set_devices(void* h, const int* devices, int n) { return tiny_b200_set_devices(S(h), devices, n); }
int tinympc_host_set_option(void* h, const char* name, double value) { return tiny_b200_set_option(S(h), name, value); }
const char* tinympc_host_last_error(void* h) { return tiny_b200_last_error(S(h)); }
void* tinympc_host_cuda_handle(void* h) { return tiny_b200_cuda_handle(S(h)); }

}  // extern "C"
