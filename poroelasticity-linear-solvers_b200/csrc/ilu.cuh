// ilu.cuh -- ILU(0) of one inner block on the device (-<prefix>pc_type ilu, and the sub-PC of -<prefix>pc_type bjacobi).
#pragma once
#include "solver.cuh"

namespace poro {

// Level sets of the dependency graph of a CSR pattern with sorted columns: level(i) = 1 + max level(j) over the stored j < i
// (lower) or j > i (upper), 0 without such j.  Rows are grouped contiguously per level: level l holds rows[ptr[l] .. ptr[l+1]).
void ilu_level_sets(int n, const int* rowptr, const int* col, bool upper, std::vector<int>& ptr, std::vector<int>& rows);

// PETSc's ILU(0): natural ordering, fill pattern = the block's stored pattern (explicit zeros included), unit-diagonal L,
// y = U^-1 L^-1 x.  Symbolic set-up on the host, IKJ factorisation on the device (one launch per lower level, one warp per
// row, no atomics: bitwise reproducible), level-scheduled triangular solves (one launch per level and direction, a fixed
// launch sequence without host synchronisation, captured in the preconditioner's CUDA graph).
struct PCIlu : PC {
    Ctx* ctx;
    int n = 0;
    bool bjacobi = false;             // the block is this rank's owned diagonal block of a row-partitioned matrix
    Csr L, U;                         // strictly lower / strictly upper parts of the factor (L has a unit diagonal)
    DBuf<double> dinv;                // 1 / u_ii
    DBuf<int> lrows, urows;           // rows grouped by lower / upper level
    std::vector<int> lptr, uptr;      // level boundaries (host: the launch sequence)
    int gl = 32, gu = 32;             // lanes per row of the lower / upper solve
    // ilu_info
    double min_pivot = 0.0;
    int64_t device_bytes = 0, apply_bytes = 0;
    // `opt` is the prefix of the factor keys: "<prefix>" for ilu, "<prefix>sub_" for bjacobi
    PCIlu(Ctx* c, const Csr& A, const std::string& prefix, const std::string& opt, bool bjacobi);
    void apply(const double* x, double* y) override;
    const char* kind() const override { return bjacobi ? "bjacobi" : "ilu"; }
};

}  // namespace poro
