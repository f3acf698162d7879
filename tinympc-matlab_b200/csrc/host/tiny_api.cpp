// tiny_api.cpp -- host implementation of the drop-in C++ API (see tiny_api.hpp).
//
// Everything here is O(1) per problem FAMILY (setup, cache precompute, setters); the per-problem
// work -- the ADMM loop -- is handed to the CUDA library through the C ABI of
// include/tinympc_b200.h.  There is deliberately no CPU solve loop in this file.
#include "tiny_api.hpp"

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <iostream>
#include <string>
#include <vector>

#include "../../../include/tinympc_b200.h"
#include "quadrotor_sensitivity_tables.hpp"

struct TinyB200Backend {
    tinympc_cuda_solver* cuda = nullptr;
    std::vector<int> devices;
    uint64_t family_hash = 0;
    bool family_set = false;
    int precision = 32;
    std::string err;
};

namespace {

// reference defaults, tiny_api_constants.hpp:5-14
constexpr double kDefAbsPriTol = 1e-3, kDefAbsDuaTol = 1e-3;
constexpr int kDefMaxIter = 1000, kDefCheckTermination = 1;

int check_dimension(const char* name, const char* what, int actual, int expected) {
    if (actual != expected) {
        std::cout << name << " has " << actual << " " << what << ". Expected " << expected << "." << std::endl;
        return 1;
    }
    return 0;
}

tinyMatrix zeros(int r, int c) { return tinyMatrix::Zero(r, c); }

// dense inverse by LU with partial pivoting (what a dynamic-size Eigen .inverse() computes)
bool invert(const tinyMatrix& A, tinyMatrix& Ainv) {
    const int n = (int)A.rows();
    tinyMatrix a = A;
    Ainv = tinyMatrix::Identity(n, n);
    for (int k = 0; k < n; ++k) {
        int piv = k;
        for (int i = k + 1; i < n; ++i) if (std::fabs(a(i, k)) > std::fabs(a(piv, k))) piv = i;
        if (a(piv, k) == 0.0) return false;
        if (piv != k)
            for (int j = 0; j < n; ++j) { std::swap(a(k, j), a(piv, j)); std::swap(Ainv(k, j), Ainv(piv, j)); }
        const double dinv = 1.0 / a(k, k);
        for (int j = 0; j < n; ++j) { a(k, j) *= dinv; Ainv(k, j) *= dinv; }
        for (int i = 0; i < n; ++i) {
            if (i == k) continue;
            const double f = a(i, k);
            if (f == 0.0) continue;
            for (int j = 0; j < n; ++j) { a(i, j) -= f * a(k, j); Ainv(i, j) -= f * Ainv(k, j); }
        }
    }
    return true;
}

tinyMatrix mul(const tinyMatrix& a, const tinyMatrix& b) {
    tinyMatrix c = zeros((int)a.rows(), (int)b.cols());
    for (int j = 0; j < (int)b.cols(); ++j)
        for (int i = 0; i < (int)a.rows(); ++i) {
            double s = 0;
            for (int k = 0; k < (int)a.cols(); ++k) s += a(i, k) * b(k, j);
            c(i, j) = s;
        }
    return c;
}
tinyMatrix tr(const tinyMatrix& a) {
    tinyMatrix t = zeros((int)a.cols(), (int)a.rows());
    for (int i = 0; i < (int)a.rows(); ++i) for (int j = 0; j < (int)a.cols(); ++j) t(j, i) = a(i, j);
    return t;
}
tinyMatrix add(const tinyMatrix& a, const tinyMatrix& b, double sb = 1.0) {
    tinyMatrix c = a;
    for (int j = 0; j < (int)a.cols(); ++j) for (int i = 0; i < (int)a.rows(); ++i) c(i, j) = a(i, j) + sb * b(i, j);
    return c;
}
void print_matrix(const char* name, const tinyMatrix& m) {
    std::cout << name << " = ";
    for (int i = 0; i < (int)m.rows(); ++i) {
        std::cout << "[";
        for (int j = 0; j < (int)m.cols(); ++j) std::cout << m(i, j) << (j + 1 < (int)m.cols() ? ", " : "");
        std::cout << "]" << std::endl;
    }
}

uint64_t fnv(uint64_t h, const void* p, size_t n) {
    const unsigned char* b = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; }
    return h;
}
template <typename M> uint64_t fnv_m(uint64_t h, const M& m) {
    const int rc[2] = {(int)m.rows(), (int)m.cols()};
    h = fnv(h, rc, sizeof rc);
    return m.size() ? fnv(h, m.data(), sizeof(*m.data()) * m.size()) : h;
}

TinyB200Backend* backend_of(TinySolver* s) {
    if (!s->backend) s->backend = new TinyB200Backend();
    return s->backend;
}

int ensure_cuda(TinySolver* s) {
    TinyB200Backend* b = backend_of(s);
    if (b->cuda) return 0;
    int rc = tinympc_cuda_create(&b->cuda, b->devices.empty() ? nullptr : b->devices.data(), (int)b->devices.size());
    if (rc) { b->err = "tinympc_cuda_create failed (no usable CUDA device: this library has no CPU fallback)"; return rc; }
    tinympc_cuda_set_option(b->cuda, "precision", b->precision);
    return 0;
}

// (Re)upload the family data whenever anything in solver->{work,cache,settings} that the GPU path reads has
// changed -- callers of the reference API poke these structs directly between solves.
int sync_family(TinySolver* s) {
    int rc = ensure_cuda(s);
    if (rc) return rc;
    TinyB200Backend* b = s->backend;
    const TinyWorkspace* w = s->work;
    const TinyCache* c = s->cache;
    const TinySettings* st = s->settings;
    uint64_t h = 1469598103934665603ull;
    const int dims[3] = {w->nx, w->nu, w->N};
    h = fnv(h, dims, sizeof dims);
    h = fnv_m(h, w->Adyn); h = fnv_m(h, w->Bdyn); h = fnv_m(h, w->fdyn); h = fnv_m(h, w->Q); h = fnv_m(h, w->R);
    h = fnv(h, &c->rho, sizeof c->rho);
    h = fnv_m(h, c->Kinf); h = fnv_m(h, c->Pinf); h = fnv_m(h, c->Quu_inv); h = fnv_m(h, c->AmBKt); h = fnv_m(h, c->APf); h = fnv_m(h, c->BPf);
    h = fnv_m(h, c->dKinf_drho); h = fnv_m(h, c->dPinf_drho);
    h = fnv(h, st, sizeof *st);
    h = fnv_m(h, w->x_min); h = fnv_m(h, w->x_max); h = fnv_m(h, w->u_min); h = fnv_m(h, w->u_max);
    h = fnv(h, &w->numStateCones, sizeof(int)); h = fnv(h, &w->numInputCones, sizeof(int));
    h = fnv_m(h, w->Acx); h = fnv_m(h, w->qcx); h = fnv_m(h, w->cx); h = fnv_m(h, w->Acu); h = fnv_m(h, w->qcu); h = fnv_m(h, w->cu);
    h = fnv(h, &w->numStateLinear, sizeof(int)); h = fnv(h, &w->numInputLinear, sizeof(int));
    h = fnv_m(h, w->Alin_x); h = fnv_m(h, w->blin_x); h = fnv_m(h, w->Alin_u); h = fnv_m(h, w->blin_u);
    if (b->family_set && h == b->family_hash) return 0;

    tinympc_cuda_family f;
    std::memset(&f, 0, sizeof f);
    f.nx = w->nx; f.nu = w->nu; f.N = w->N;
    f.Adyn = w->Adyn.data(); f.Bdyn = w->Bdyn.data(); f.fdyn = w->fdyn.size() ? w->fdyn.data() : nullptr;
    f.Q = w->Q.data(); f.R = w->R.data();
    f.rho = c->rho;
    f.Kinf = c->Kinf.data(); f.Pinf = c->Pinf.data(); f.Quu_inv = c->Quu_inv.data(); f.AmBKt = c->AmBKt.data();
    f.APf = c->APf.size() ? c->APf.data() : nullptr; f.BPf = c->BPf.size() ? c->BPf.data() : nullptr;
    const bool have_sens = (int)c->dKinf_drho.size() == w->nu * w->nx && (int)c->dPinf_drho.size() == w->nx * w->nx;
    f.dKinf_drho = have_sens ? c->dKinf_drho.data() : nullptr;
    f.dPinf_drho = have_sens ? c->dPinf_drho.data() : nullptr;
    f.abs_pri_tol = st->abs_pri_tol; f.abs_dua_tol = st->abs_dua_tol; f.max_iter = st->max_iter; f.check_termination = st->check_termination;
    const bool have_xb = (int)w->x_min.size() == w->nx * w->N && (int)w->x_max.size() == w->nx * w->N;
    const bool have_ub = (int)w->u_min.size() == w->nu * (w->N - 1) && (int)w->u_max.size() == w->nu * (w->N - 1);
    // The C++ defaults enable the bound flags before any bounds exist (tiny_api_constants.hpp:9-10); the
    // reference would then read empty matrices.  Missing bounds are treated as "no bound" here.
    f.en_state_bound = st->en_state_bound && have_xb; f.en_input_bound = st->en_input_bound && have_ub;
    f.en_state_soc = st->en_state_soc; f.en_input_soc = st->en_input_soc;
    f.en_state_linear = st->en_state_linear; f.en_input_linear = st->en_input_linear;
    f.adaptive_rho = st->adaptive_rho; f.adaptive_rho_min = st->adaptive_rho_min; f.adaptive_rho_max = st->adaptive_rho_max;
    f.adaptive_rho_enable_clipping = st->adaptive_rho_enable_clipping;
    if (have_xb) { f.x_min = w->x_min.data(); f.x_max = w->x_max.data(); }
    if (have_ub) { f.u_min = w->u_min.data(); f.u_max = w->u_max.data(); }
    f.numStateCones = w->numStateCones; f.numInputCones = w->numInputCones;
    if (w->numStateCones > 0) { f.Acx = w->Acx.data(); f.qcx = w->qcx.data(); f.cx = w->cx.data(); }
    if (w->numInputCones > 0) { f.Acu = w->Acu.data(); f.qcu = w->qcu.data(); f.cu = w->cu.data(); }
    f.numStateLinear = w->numStateLinear; f.numInputLinear = w->numInputLinear;
    if (w->numStateLinear > 0) { f.Alin_x = w->Alin_x.data(); f.blin_x = w->blin_x.data(); }
    if (w->numInputLinear > 0) { f.Alin_u = w->Alin_u.data(); f.blin_u = w->blin_u.data(); }
    rc = tinympc_cuda_set_family(b->cuda, &f);
    if (rc) { b->err = tinympc_cuda_last_error(b->cuda); return rc; }
    b->family_hash = h;
    b->family_set = true;
    return 0;
}

}  // namespace

extern "C" {

int tiny_set_default_settings(TinySettings* settings) {
    if (!settings) { std::cout << "Error in tiny_set_default_settings: settings is nullptr" << std::endl; return 1; }
    settings->abs_pri_tol = kDefAbsPriTol;
    settings->abs_dua_tol = kDefAbsDuaTol;
    settings->max_iter = kDefMaxIter;
    settings->check_termination = kDefCheckTermination;
    settings->en_state_bound = 1;      // C++ defaults: bounds on, everything else off (tiny_api_constants.hpp:9-14)
    settings->en_input_bound = 1;
    settings->en_state_soc = 0;
    settings->en_input_soc = 0;
    settings->en_state_linear = 0;
    settings->en_input_linear = 0;
    settings->adaptive_rho = 0;
    settings->adaptive_rho_min = 1.0;
    settings->adaptive_rho_max = 100.0;
    settings->adaptive_rho_enable_clipping = 1;
    return 0;
}

int tiny_update_settings(TinySettings* settings, tinytype abs_pri_tol, tinytype abs_dua_tol, int max_iter, int check_termination,
                         int en_state_bound, int en_input_bound, int en_state_soc, int en_input_soc, int en_state_linear,
                         int en_input_linear) {
    if (!settings) { std::cout << "Error in tiny_update_settings: settings is nullptr" << std::endl; return 1; }
    settings->abs_pri_tol = abs_pri_tol; settings->abs_dua_tol = abs_dua_tol;
    settings->max_iter = max_iter; settings->check_termination = check_termination;
    settings->en_state_bound = en_state_bound; settings->en_input_bound = en_input_bound;
    settings->en_state_soc = en_state_soc; settings->en_input_soc = en_input_soc;
    settings->en_state_linear = en_state_linear; settings->en_input_linear = en_input_linear;
    return 0;
}

int tiny_precompute_and_set_cache(TinyCache* cache, tinyMatrix Adyn, tinyMatrix Bdyn, tinyMatrix fdyn, tinyMatrix Q, tinyMatrix R,
                                  int nx, int nu, tinytype rho, int verbose) {
    if (!cache) { std::cout << "Error in tiny_precompute_and_set_cache: cache is nullptr" << std::endl; return 1; }
    tinyMatrix Q1 = add(Q, tinyMatrix::Identity(nx, nx), rho);
    tinyMatrix R1 = add(R, tinyMatrix::Identity(nu, nu), rho);
    if (verbose) { print_matrix("A", Adyn); print_matrix("B", Bdyn); print_matrix("Q", Q1); print_matrix("R", R1); std::cout << "rho = " << rho << std::endl; }
    const tinyMatrix At = tr(Adyn), Bt = tr(Bdyn);
    tinyMatrix Ktp1 = zeros(nu, nx), Ptp1 = zeros(nx, nx), Kinf = zeros(nu, nx), Pinf = zeros(nx, nx), Sinv;
    for (int i = 0; i < nx; ++i) Ptp1(i, i) = rho;
    for (int it = 0; it < 1000; ++it) {     // infinite-horizon Riccati fixed point, tiny_api.cpp:272-286
        const tinyMatrix BtP = mul(Bt, Ptp1);
        if (!invert(add(R1, mul(BtP, Bdyn)), Sinv)) { std::cout << "tiny_precompute_and_set_cache: R + B'PB is singular" << std::endl; return 1; }
        Kinf = mul(mul(mul(Sinv, Bt), Ptp1), Adyn);
        Pinf = add(Q1, mul(mul(At, Ptp1), add(Adyn, mul(Bdyn, Kinf), -1.0)));
        double md = 0;
        for (int j = 0; j < nx; ++j) for (int a = 0; a < nu; ++a) md = std::fmax(md, std::fabs(Kinf(a, j) - Ktp1(a, j)));
        if (md < 1e-5) { if (verbose) std::cout << "Kinf converged after " << it + 1 << " iterations" << std::endl; break; }
        Ktp1 = Kinf; Ptp1 = Pinf;
    }
    tinyMatrix Quu_inv;
    if (!invert(add(R1, mul(mul(Bt, Pinf), Bdyn)), Quu_inv)) return 1;
    const tinyMatrix AmBKt = tr(add(Adyn, mul(Bdyn, Kinf), -1.0));
    const tinyMatrix APf = mul(mul(AmBKt, Pinf), fdyn), BPf = mul(mul(Bt, Pinf), fdyn);
    if (verbose) {
        print_matrix("Kinf", Kinf); print_matrix("Pinf", Pinf); print_matrix("Quu_inv", Quu_inv); print_matrix("AmBKt", AmBKt);
        print_matrix("APf", APf); print_matrix("BPf", BPf);
        std::cout << "\nPrecomputation finished!\n" << std::endl;
    }
    cache->rho = rho;
    cache->Kinf = Kinf; cache->Pinf = Pinf; cache->Quu_inv = Quu_inv; cache->AmBKt = AmBKt;
    cache->C1 = Quu_inv; cache->C2 = AmBKt;
    cache->APf = APf; cache->BPf = BPf;
    return 0;
}

int tiny_setup(TinySolver** solverp, tinyMatrix Adyn, tinyMatrix Bdyn, tinyMatrix fdyn, tinyMatrix Q, tinyMatrix R,
               tinytype rho, int nx, int nu, int N, int verbose) {
    if (!solverp) return 1;
    TinySolver* solver = new TinySolver();
    solver->solution = new TinySolution();
    solver->cache = new TinyCache();
    solver->settings = new TinySettings();
    solver->work = new TinyWorkspace();
    solver->backend = nullptr;
    *solverp = solver;
    TinyWorkspace* work = solver->work;

    solver->solution->iter = 0; solver->solution->solved = 0;
    solver->solution->x = zeros(nx, N); solver->solution->u = zeros(nu, N - 1);
    tiny_set_default_settings(solver->settings);
    work->nx = nx; work->nu = nu; work->N = N;

    int status = 0;
    status |= check_dimension("State transition matrix (A)", "rows", (int)Adyn.rows(), nx);
    status |= check_dimension("State transition matrix (A)", "columns", (int)Adyn.cols(), nx);
    status |= check_dimension("Input matrix (B)", "rows", (int)Bdyn.rows(), nx);
    status |= check_dimension("Input matrix (B)", "columns", (int)Bdyn.cols(), nu);
    status |= check_dimension("Affine vector (f)", "rows", (int)fdyn.rows(), nx);
    status |= check_dimension("Affine vector (f)", "columns", (int)fdyn.cols(), 1);
    status |= check_dimension("State stage cost (Q)", "rows", (int)Q.rows(), nx);
    status |= check_dimension("State stage cost (Q)", "columns", (int)Q.cols(), nx);
    status |= check_dimension("State input cost (R)", "rows", (int)R.rows(), nu);
    status |= check_dimension("State input cost (R)", "columns", (int)R.cols(), nu);
    if (status) return status;

    for (tinyMatrix* m : {&work->x, &work->q, &work->p, &work->v, &work->vnew, &work->g, &work->vc, &work->vcnew, &work->gc, &work->vl,
                          &work->vlnew, &work->gl, &work->Xref})
        *m = zeros(nx, N);
    for (tinyMatrix* m : {&work->u, &work->r, &work->d, &work->z, &work->znew, &work->y, &work->zc, &work->zcnew, &work->yc, &work->zl,
                          &work->zlnew, &work->yl, &work->Uref})
        *m = zeros(nu, N - 1);
    work->numStateCones = work->numInputCones = 0;
    work->numStateLinear = work->numInputLinear = 0;
    work->Q = tinyVector::Zero(nx, 1); work->R = tinyVector::Zero(nu, 1);
    for (int i = 0; i < nx; ++i) work->Q(i) = Q(i, i) + rho;     // tiny_api.cpp:107
    for (int i = 0; i < nu; ++i) work->R(i) = R(i, i) + rho;     // tiny_api.cpp:108
    work->Adyn = Adyn; work->Bdyn = Bdyn;
    work->fdyn = tinyVector::Zero(nx, 1);
    for (int i = 0; i < nx; ++i) work->fdyn(i) = fdyn(i, 0);
    work->Qu = tinyVector::Zero(nu, 1);
    work->primal_residual_state = work->primal_residual_input = 0;
    work->dual_residual_state = work->dual_residual_input = 0;
    work->status = 0; work->iter = 0;

    // the cache sees diag(Q)+rho and adds rho again (tiny_api.cpp:126, 254-255; SURVEY.md quirk Q1)
    tinyMatrix Qw = zeros(nx, nx), Rw = zeros(nu, nu);
    for (int i = 0; i < nx; ++i) Qw(i, i) = work->Q(i);
    for (int i = 0; i < nu; ++i) Rw(i, i) = work->R(i);
    status = tiny_precompute_and_set_cache(solver->cache, Adyn, Bdyn, fdyn, Qw, Rw, nx, nu, rho, verbose);
    if (status) return status;
    if (solver->settings->adaptive_rho) tiny_initialize_sensitivity_matrices(solver);
    return 0;
}

int tiny_set_bound_constraints(TinySolver* solver, tinyMatrix x_min, tinyMatrix x_max, tinyMatrix u_min, tinyMatrix u_max) {
    if (!solver) { std::cout << "Error in tiny_set_bound_constraints: solver is nullptr" << std::endl; return 1; }
    const TinyWorkspace* w = solver->work;
    int status = 0;
    status |= check_dimension("Lower state bounds (x_min)", "rows", (int)x_min.rows(), w->nx);
    status |= check_dimension("Lower state bounds (x_min)", "cols", (int)x_min.cols(), w->N);
    status |= check_dimension("Lower state bounds (x_max)", "rows", (int)x_max.rows(), w->nx);
    status |= check_dimension("Lower state bounds (x_max)", "cols", (int)x_max.cols(), w->N);
    status |= check_dimension("Lower input bounds (u_min)", "rows", (int)u_min.rows(), w->nu);
    status |= check_dimension("Lower input bounds (u_min)", "cols", (int)u_min.cols(), w->N - 1);
    status |= check_dimension("Lower input bounds (u_max)", "rows", (int)u_max.rows(), w->nu);
    status |= check_dimension("Lower input bounds (u_max)", "cols", (int)u_max.cols(), w->N - 1);
    (void)status;   // like the reference (tiny_api.cpp:148-163, quirk Q8) a mismatch is reported, not returned
    solver->work->x_min = x_min; solver->work->x_max = x_max; solver->work->u_min = u_min; solver->work->u_max = u_max;
    return 0;
}

int tiny_set_cone_constraints(TinySolver* solver, VectorXi Acx, VectorXi qcx, tinyVector cx, VectorXi Acu, VectorXi qcu, tinyVector cu) {
    if (!solver) { std::cout << "Error in tiny_set_cone_constraints: solver is nullptr" << std::endl; return 1; }
    const int nsc = (int)Acx.rows(), nic = (int)Acu.rows();
    int status = 0;
    status |= check_dimension("Cone state size (qcx)", "rows", (int)qcx.rows(), nsc);
    status |= check_dimension("Cone mu value for state (cx)", "rows", (int)cx.rows(), nsc);
    status |= check_dimension("Cone input size (qcu)", "rows", (int)qcu.rows(), nic);
    status |= check_dimension("Cone mu value for input (cu)", "rows", (int)cu.rows(), nic);
    if (status) return status;
    TinyWorkspace* w = solver->work;
    w->numStateCones = nsc; w->numInputCones = nic;
    w->Acx = Acx; w->qcx = qcx; w->cx = cx;
    w->Acu = Acu; w->qcu = qcu; w->cu = cu;
    return 0;
}

int tiny_set_linear_constraints(TinySolver* solver, tinyMatrix Alin_x, tinyVector blin_x, tinyMatrix Alin_u, tinyVector blin_u) {
    if (!solver) { std::cout << "Error in tiny_set_linear_constraints: solver is nullptr" << std::endl; return 1; }
    const int nsl = (int)Alin_x.rows(), nil = (int)Alin_u.rows();
    int status = 0;
    if (nsl > 0) {
        status |= check_dimension("State linear constraint matrix (Alin_x)", "columns", (int)Alin_x.cols(), solver->work->nx);
        status |= check_dimension("State linear constraint vector (blin_x)", "rows", (int)blin_x.rows(), nsl);
        status |= check_dimension("State linear constraint vector (blin_x)", "columns", (int)blin_x.cols(), 1);
    }
    if (nil > 0) {
        status |= check_dimension("Input linear constraint matrix (Alin_u)", "columns", (int)Alin_u.cols(), solver->work->nu);
        status |= check_dimension("Input linear constraint vector (blin_u)", "rows", (int)blin_u.rows(), nil);
        status |= check_dimension("Input linear constraint vector (blin_u)", "columns", (int)blin_u.cols(), 1);
    }
    if (status) return status;
    TinyWorkspace* w = solver->work;
    w->numStateLinear = nsl; w->numInputLinear = nil;
    w->Alin_x = Alin_x; w->blin_x = blin_x; w->Alin_u = Alin_u; w->blin_u = blin_u;
    return 0;
}

int tiny_set_x0(TinySolver* solver, tinyVector x0) {
    if (!solver) { std::cout << "Error in tiny_set_x0: solver is nullptr" << std::endl; return 1; }
    if ((int)x0.rows() != solver->work->nx) { perror("Error in tiny_set_x0: x0 is not the correct length"); return 0; }
    for (int i = 0; i < solver->work->nx; ++i) solver->work->x(i, 0) = x0(i);
    return 0;
}

int tiny_set_x_ref(TinySolver* solver, tinyMatrix x_ref) {
    if (!solver) { std::cout << "Error in tiny_set_x_ref: solver is nullptr" << std::endl; return 1; }
    int status = 0;
    status |= check_dimension("State reference trajectory (x_ref)", "rows", (int)x_ref.rows(), solver->work->nx);
    status |= check_dimension("State reference trajectory (x_ref)", "columns", (int)x_ref.cols(), solver->work->N);
    (void)status;
    solver->work->Xref = x_ref;
    return 0;
}

int tiny_set_u_ref(TinySolver* solver, tinyMatrix u_ref) {
    if (!solver) { std::cout << "Error in tiny_set_u_ref: solver is nullptr" << std::endl; return 1; }
    int status = 0;
    status |= check_dimension("Control/input reference trajectory (u_ref)", "rows", (int)u_ref.rows(), solver->work->nu);
    status |= check_dimension("Control/input reference trajectory (u_ref)", "columns", (int)u_ref.cols(), solver->work->N - 1);
    (void)status;
    solver->work->Uref = u_ref;
    return 0;
}

void tiny_initialize_sensitivity_matrices(TinySolver* solver) {
    const int nu = solver->work->nu, nx = solver->work->nx;
    TinyCache* c = solver->cache;
    c->dKinf_drho = zeros(nu, nx); c->dPinf_drho = zeros(nx, nx); c->dC1_drho = zeros(nu, nu); c->dC2_drho = zeros(nx, nx);
    if (nx != 12 || nu != 4) return;   // the tables exist for the 12-state / 4-input quadrotor only (tiny_api.cpp:366 note)
    for (int i = 0; i < 48; ++i) c->dKinf_drho.data()[i] = (double)tmpc_tables::dKinf_flat[i];
    for (int i = 0; i < 144; ++i) { c->dPinf_drho.data()[i] = (double)tmpc_tables::dPinf_flat[i]; c->dC2_drho.data()[i] = (double)tmpc_tables::dC2_flat[i]; }
}

namespace {
int solve_batch_impl(TinySolver* solver, const TinyModelBatch* models, const TinyBatchIn* in, const TinyBatchOut* out) {
    if (!solver || !in || !out) return TINYMPC_CUDA_EINVAL;
    int rc = sync_family(solver);
    if (rc) return rc;
    tinympc_cuda_batch_in ci{};
    ci.batch = in->batch; ci.x0 = in->x0; ci.Xref = in->Xref; ci.Uref = in->Uref;
    ci.x_min = in->x_min; ci.x_max = in->x_max; ci.u_min = in->u_min; ci.u_max = in->u_max; ci.xref_const = in->xref_const;
    tinympc_cuda_batch_out co{};
    co.x = out->x; co.u = out->u; co.iter = out->iter; co.status = out->status; co.residuals = out->residuals; co.rho = out->rho; co.u0 = out->u0;
    rc = models ? tinympc_cuda_solve_batch_models(solver->backend->cuda, models, &ci, &co) : tinympc_cuda_solve_batch(solver->backend->cuda, &ci, &co);
    if (rc) solver->backend->err = tinympc_cuda_last_error(solver->backend->cuda);
    return rc;
}
}  // namespace

int tiny_solve_batch(TinySolver* solver, const TinyBatchIn* in, const TinyBatchOut* out) { return solve_batch_impl(solver, nullptr, in, out); }

int tiny_solve_batch_models(TinySolver* solver, const TinyModelBatch* models, const TinyBatchIn* in, const TinyBatchOut* out) {
    if (!models) return TINYMPC_CUDA_EINVAL;
    return solve_batch_impl(solver, models, in, out);
}

int tiny_b200_set_devices(TinySolver* solver, const int* devices, int n_devices) {
    if (!solver) return TINYMPC_CUDA_EINVAL;
    TinyB200Backend* b = backend_of(solver);
    if (b->cuda) { tinympc_cuda_destroy(b->cuda); b->cuda = nullptr; b->family_set = false; }
    b->devices.assign(devices, devices + (n_devices > 0 ? n_devices : 0));
    return 0;
}

int tiny_b200_set_option(TinySolver* solver, const char* name, double value) {
    if (!solver || !name) return TINYMPC_CUDA_EINVAL;
    TinyB200Backend* b = backend_of(solver);
    if (std::string(name) == "precision") b->precision = (int)value;
    int rc = ensure_cuda(solver);
    if (rc) return rc;
    rc = tinympc_cuda_set_option(b->cuda, name, value);
    if (rc) b->err = tinympc_cuda_last_error(b->cuda);
    return rc;
}

const char* tiny_b200_last_error(const TinySolver* solver) { return (solver && solver->backend) ? solver->backend->err.c_str() : ""; }

void* tiny_b200_cuda_handle(TinySolver* solver) {
    if (!solver || sync_family(solver)) return nullptr;
    return solver->backend->cuda;
}

void tiny_free(TinySolver* solver) {
    if (!solver) return;
    if (solver->backend) { if (solver->backend->cuda) tinympc_cuda_destroy(solver->backend->cuda); delete solver->backend; }
    delete solver->solution; delete solver->cache; delete solver->settings; delete solver->work;
    delete solver;
}

int tiny_solve(TinySolver* solver) {
    if (!solver) return -TINYMPC_CUDA_EINVAL;
    int rc = sync_family(solver);
    if (rc) return -rc;
    TinyWorkspace* w = solver->work;
    TinyCache* c = solver->cache;
    const TinySettings* st = solver->settings;
    const int nx = w->nx, nu = w->nu, N = w->N;
    auto ensure = [](tinyMatrix& m, int r, int cc) { if ((int)m.rows() != r || (int)m.cols() != cc) m = tinyMatrix::Zero(r, cc); };
    ensure(w->vcnew, nx, N); ensure(w->zcnew, nu, N - 1); ensure(w->gc, nx, N); ensure(w->yc, nu, N - 1);
    ensure(w->vlnew, nx, N); ensure(w->zlnew, nu, N - 1); ensure(w->gl, nx, N); ensure(w->yl, nu, N - 1);
    ensure(w->Xref, nx, N); ensure(w->Uref, nu, N - 1);
    solver->solution->x = tinyMatrix::Zero(nx, N);
    solver->solution->u = tinyMatrix::Zero(nu, N - 1);

    tinympc_cuda_workspace ws;
    std::memset(&ws, 0, sizeof ws);
    ws.x = w->x.data(); ws.u = w->u.data(); ws.q = w->q.data(); ws.r = w->r.data(); ws.p = w->p.data(); ws.d = w->d.data();
    ws.v = w->v.data(); ws.vnew = w->vnew.data(); ws.z = w->z.data(); ws.znew = w->znew.data(); ws.g = w->g.data(); ws.y = w->y.data();
    ws.vcnew = w->vcnew.data(); ws.zcnew = w->zcnew.data(); ws.gc = w->gc.data(); ws.yc = w->yc.data();
    ws.vlnew = w->vlnew.data(); ws.zlnew = w->zlnew.data(); ws.gl = w->gl.data(); ws.yl = w->yl.data();
    ws.Xref = w->Xref.data(); ws.Uref = w->Uref.data();
    const tinytype rho_before = c->rho;
    ws.rho = &c->rho; ws.Kinf = c->Kinf.data(); ws.Pinf = c->Pinf.data();
    ws.sol_x = solver->solution->x.data(); ws.sol_u = solver->solution->u.data();
    int iter = 0, status = 11, solved = 0;
    double res[4] = {w->primal_residual_state, w->dual_residual_state, w->primal_residual_input, w->dual_residual_input};
    ws.iter = &iter; ws.status = &status; ws.solved = &solved; ws.residuals = res;
    rc = tinympc_cuda_solve_workspace(solver->backend->cuda, &ws);
    if (rc) { solver->backend->err = tinympc_cuda_last_error(solver->backend->cuda); return -rc; }
    w->iter = iter; w->status = status;
    w->primal_residual_state = res[0]; w->dual_residual_state = res[1]; w->primal_residual_input = res[2]; w->dual_residual_input = res[3];
    solver->solution->iter = iter; solver->solution->solved = solved;
    if (st->adaptive_rho && c->rho != rho_before) {
        // the reference also drags C1/C2 along (rho_benchmark.cpp:206-207); they are never read by the iteration
        const tinytype dr = c->rho - rho_before;
        if (c->dC1_drho.size() == c->C1.size()) for (size_t i = 0; i < c->C1.size(); ++i) c->C1.data()[i] += dr * c->dC1_drho.data()[i];
        if (c->dC2_drho.size() == c->C2.size()) for (size_t i = 0; i < c->C2.size(); ++i) c->C2.data()[i] += dr * c->dC2_drho.data()[i];
    }
    return solved ? 0 : 1;    // admm.cpp:375 / :388
}

}  // extern "C"
