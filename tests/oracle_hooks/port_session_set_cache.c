/*
 * Test-only hook on the C port of the reference: port_session_set_model (port_session_set_model.c, included unchanged), then the
 * cache of the live session solver replaced by GIVEN arrays instead of the port's own precompute -- so that a reference session runs
 * with exactly the cache the device computed.  Kinf, Pinf, Quu_inv, AmBKt column-major (nu x nx, nx x nx, nu x nu, nx x nx), APf nx,
 * BPf nu.  C1 = Quu_inv and C2 = AmBKt as tiny_precompute_and_set_cache sets them (tiny_api.cpp:312-313); the pristine copies too.
 */
#include "port_session_set_model.c"

int port_session_set_cache(void* h, const oracle_problem* d, const double* Kinf, const double* Pinf, const double* Quu_inv,
                           const double* AmBKt, const double* APf, const double* BPf) {
    if (port_session_set_model(h, d)) return 1;
    Solver* s = (Solver*)h;
    const size_t nx = (size_t)s->nx, nu = (size_t)s->nu;
    memcpy(s->Kinf, Kinf, sizeof(double) * nu * nx); memcpy(s->Pinf, Pinf, sizeof(double) * nx * nx);
    memcpy(s->Quu_inv, Quu_inv, sizeof(double) * nu * nu); memcpy(s->AmBKt, AmBKt, sizeof(double) * nx * nx);
    memcpy(s->APf, APf, sizeof(double) * nx); memcpy(s->BPf, BPf, sizeof(double) * nu);
    memcpy(s->C1, Quu_inv, sizeof(double) * nu * nu); memcpy(s->C2, AmBKt, sizeof(double) * nx * nx);
    memcpy(s->Kinf0, Kinf, sizeof(double) * nu * nx); memcpy(s->Pinf0, Pinf, sizeof(double) * nx * nx);
    memcpy(s->C10, Quu_inv, sizeof(double) * nu * nu); memcpy(s->C20, AmBKt, sizeof(double) * nx * nx);
    return 0;
}
