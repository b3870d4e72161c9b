// Host harness for csrc/lu_symbolic.h (the symbolic analysis of the device sparse LU), for tests/test_lu_symbolic_host.py.
#include <stdint.h>

#include "lu_symbolic.h"

extern "C" {

void* lusym_analyse(int n, const int64_t* rowptr, const int32_t* col) {
    try {
        return new poro::lusym::Symbolic(poro::lusym::analyse(n, rowptr, col));
    } catch (...) {
        return nullptr;
    }
}

// n, supernodes, levels, total front rows, nnz(L), nnz(U), amalgamation zeros, largest front
void lusym_sizes(void* h, int64_t* out) {
    const auto& S = *static_cast<poro::lusym::Symbolic*>(h);
    out[0] = S.n;
    out[1] = S.nsuper;
    out[2] = S.nlevels;
    out[3] = S.row_ptr[S.nsuper];
    out[4] = S.nnz_l;
    out[5] = S.nnz_u;
    out[6] = S.amalg_zeros;
    out[7] = S.max_front;
}

// perm (n), first (nsuper + 1), parent (nsuper), row_ptr (nsuper + 1), row_idx (total front rows), level of each supernode
void lusym_copy(void* h, int32_t* perm, int32_t* first, int32_t* parent, int64_t* row_ptr, int32_t* row_idx, int32_t* level) {
    const auto& S = *static_cast<poro::lusym::Symbolic*>(h);
    for (int i = 0; i < S.n; ++i) perm[i] = S.perm[i];
    for (int s = 0; s <= S.nsuper; ++s) { first[s] = S.first[s]; row_ptr[s] = S.row_ptr[s]; }
    for (int s = 0; s < S.nsuper; ++s) parent[s] = S.parent[s];
    for (int64_t q = 0; q < S.row_ptr[S.nsuper]; ++q) row_idx[q] = S.row_idx[q];
    for (int l = 0; l < S.nlevels; ++l)
        for (int q = S.level_ptr[l]; q < S.level_ptr[l + 1]; ++q) level[S.level_sn[q]] = l;
}

void lusym_free(void* h) { delete static_cast<poro::lusym::Symbolic*>(h); }
}
