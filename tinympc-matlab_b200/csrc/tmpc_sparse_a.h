// tmpc_sparse_a.h -- nonzero patterns of A at row-pair granularity, the dispatcher's side of the sparse-A fp32 instances
// (Tpp3Cfg::SA, tmpc_tpp3.cuh).  A pattern is one mask per column: bit j = rows 2j, 2j+1; bit nx / 2 = the odd tail row
// (SparsePairs, tmpc_tpp2.cuh).  Plain C++: no CUDA header.
#pragma once

namespace tmpc {

// pattern of the float32 conversion of a row-major nx x nx matrix (the kernels' A: fill_const_pack2 converts with the same cast)
inline void a_pairs_of(const double* A_rowmajor, int nx, unsigned* cols) {
    for (int c = 0; c < nx; ++c) cols[c] = 0u;
    for (int r = 0; r < nx; ++r)
        for (int c = 0; c < nx; ++c)
            if (static_cast<float>(A_rowmajor[r * nx + c]) != 0.f) cols[c] |= 1u << (r / 2);   // odd nx: row nx - 1 -> bit nx / 2
}

// a family with pattern fam (nx columns) may run an instance compiled for pattern inst (inst_cols columns; 0 = dense): every nonzero
// of the family lies inside the compiled pattern
inline bool a_pattern_covers(const unsigned* inst, int inst_cols, const unsigned* fam, int nx) {
    if (inst_cols == 0) return true;
    if (inst_cols != nx) return false;
    for (int c = 0; c < nx; ++c)
        if (fam[c] & ~inst[c]) return false;
    return true;
}

}  // namespace tmpc
