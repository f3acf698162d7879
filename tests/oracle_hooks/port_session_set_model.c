/*
 * Test-only hook on the C port of the reference (oracle/tinympc_oracle.c, compiled into this file unchanged): replace the model of a
 * live session solver between two solves, as a user of the reference does to a live TinySolver.  It writes work->Adyn, Bdyn, fdyn,
 * Q and R and the cache fields (rho, Kinf, Pinf, Quu_inv, AmBKt, APf, BPf, C1, C2 and the sensitivities), taken from a fresh
 * tiny_setup of the new model (solver_create), and keeps the rest of the workspace: x, u, q, r, p, d, slacks, duals, references.
 * Only the model half of `d` is read; the shape and the settings must be those of the session.
 */
#include "tinympc_oracle.c"

int port_session_set_model(void* h, const oracle_problem* d) {
    Solver* s = (Solver*)h;
    Solver* t = solver_create(d);
    if (!s || !t || t->nx != s->nx || t->nu != s->nu) { solver_free(t); return 1; }
    const size_t nx = (size_t)s->nx, nu = (size_t)s->nu;
#define TAKE(field, n) memcpy(s->field, t->field, sizeof(double) * (n))
    TAKE(A, nx * nx); TAKE(B, nx * nu); TAKE(f, nx); TAKE(Q, nx); TAKE(R, nu);
    TAKE(Kinf, nu * nx); TAKE(Pinf, nx * nx); TAKE(Quu_inv, nu * nu); TAKE(AmBKt, nx * nx); TAKE(APf, nx); TAKE(BPf, nu);
    TAKE(C1, nu * nu); TAKE(C2, nx * nx); TAKE(dK, nu * nx); TAKE(dP, nx * nx); TAKE(dC1, nu * nu); TAKE(dC2, nx * nx);
    TAKE(Kinf0, nu * nx); TAKE(Pinf0, nx * nx); TAKE(C10, nu * nu); TAKE(C20, nx * nx);
#undef TAKE
    s->rho = t->rho;
    s->rho0 = t->rho0;
    solver_free(t);
    return 0;
}

/* cache->rho of a live session solver (adaptive rho moves it) */
double port_session_rho(void* h) { return ((Solver*)h)->rho; }
