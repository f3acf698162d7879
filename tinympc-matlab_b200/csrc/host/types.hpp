// types.hpp -- the solver data model of the drop-in C++ API.
//
// Field-for-field the same names as the reference's structs (tinympc/TinyMPC/src/tinympc/types.hpp:
// TinySolution :32-37, TinyCache :43-59, TinySettings :63-80, TinyWorkspace :86-187, TinySolver
// :192-197), because reference user code reads and writes them directly (e.g.
// T/examples/quadrotor_hovering.cpp:54,66, rocket_landing_mpc.cpp:97-134).  One member is added at the
// END of TinySolver: the opaque B200 backend that tiny_solve / tiny_solve_batch run on.
#pragma once
#include "../../../include/tinympc_b200.h"
#include "tiny_linalg.hpp"

struct TinySolution {
    int iter;        // ADMM iterations of the last solve
    int solved;      // 1 if the termination test passed
    tinyMatrix x;    // nx x N    (= vnew at exit)
    tinyMatrix u;    // nu x N-1  (= znew at exit)
};

struct TinyCache {
    tinytype rho;
    tinyMatrix Kinf;      // nu x nx
    tinyMatrix Pinf;      // nx x nx
    tinyMatrix Quu_inv;   // nu x nu
    tinyMatrix AmBKt;     // nx x nx
    tinyVector APf;       // nx
    tinyVector BPf;       // nu
    tinyMatrix C1;        // = Quu_inv at setup; only moved by adaptive rho, never read by the iteration
    tinyMatrix C2;        // = AmBKt  at setup; idem
    tinyMatrix dKinf_drho, dPinf_drho, dC1_drho, dC2_drho;   // adaptive-rho sensitivities
};

struct TinySettings {
    tinytype abs_pri_tol;
    tinytype abs_dua_tol;
    int max_iter;
    int check_termination;
    int en_state_bound;
    int en_input_bound;
    int en_state_soc;
    int en_input_soc;
    int en_state_linear;
    int en_input_linear;
    int adaptive_rho;
    tinytype adaptive_rho_min;
    tinytype adaptive_rho_max;
    int adaptive_rho_enable_clipping;
};

struct TinyWorkspace {
    int nx, nu, N;
    tinyMatrix x, u;             // trajectory            nx x N, nu x N-1
    tinyMatrix q, r;             // linear cost terms
    tinyMatrix p, d;             // Riccati backward-pass terms
    tinyMatrix v, vnew, z, znew; // box slacks (previous / current)
    tinyMatrix g, y;             // box duals
    tinyMatrix x_min, x_max, u_min, u_max;
    int numStateCones, numInputCones;
    tinyVector cx, cu;           // cone coefficients mu
    VectorXi Acx, Acu;           // cone start indices
    VectorXi qcx, qcu;           // cone dimensions
    tinyMatrix vc, vcnew, zc, zcnew;   // cone slacks
    tinyMatrix gc, yc;                 // cone duals
    int numStateLinear, numInputLinear;
    tinyMatrix Alin_x; tinyVector blin_x;
    tinyMatrix Alin_u; tinyVector blin_u;
    tinyMatrix vl, vlnew, zl, zlnew;   // linear-constraint slacks
    tinyMatrix gl, yl;                 // linear-constraint duals
    tinyVector Q, R;             // diag(Q)+rho, diag(R)+rho
    tinyMatrix Adyn, Bdyn;
    tinyVector fdyn;
    tinyMatrix Xref, Uref;
    tinyVector Qu;
    tinytype primal_residual_state;
    tinytype primal_residual_input;
    tinytype dual_residual_state;
    tinytype dual_residual_input;
    int status;                  // 1 solved, 11 unsolved
    int iter;
};

struct TinyB200Backend;          // opaque: CUDA handle + cached family fingerprint

struct TinySolver {
    TinySolution* solution;
    TinySettings* settings;
    TinyCache* cache;
    TinyWorkspace* work;
    TinyB200Backend* backend;    // added by the B200 build (NULL until the first GPU call)
};

// ---- new: the batched entry point's argument blocks (float32, one contiguous chunk per problem) ----
struct TinyBatchIn {
    int batch;
    const float* x0;      // batch x nx
    const float* Xref;    // batch x (nx*N)      column-major nx x N per problem, or NULL = zeros
    const float* Uref;    // batch x (nu*(N-1))  or NULL = zeros
    const float* x_min;   // optional per-problem bounds (all four or none)
    const float* x_max;
    const float* u_min;
    const float* u_max;
    const float* xref_const = nullptr;   // batch x nx: one reference state per problem, held over the horizon (instead of Xref)
};
struct TinyBatchOut {
    float* x;             // batch x (nx*N)
    float* u;             // batch x (nu*(N-1))
    int* iter;            // batch
    int* status;          // batch (1 / 11)
    float* residuals;     // batch x 4 or NULL
    float* rho;           // batch or NULL
    float* u0 = nullptr;  // batch x nu: first control only; with it x and u may be NULL (the trajectories stay on the device)
};
// per-problem models of tiny_solve_batch_models: the C ABI's struct itself (double, one column-major chunk per problem)
typedef tinympc_cuda_models TinyModelBatch;
