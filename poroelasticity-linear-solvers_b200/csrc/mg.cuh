// mg.cuh -- geometric transfer between a generated field block and the same block generated at N/2 (mg.cu), the pieces of
// `-<prefix>pc_type mg`.  The levels are linked by poro_mat_set_coarse (StencilData::coarse); the transfer is pure geometry
// (mg_transfer.h), so it has no matrix: columns come from the lattice position, the Dirichlet flags from the two levels.
#pragma once
#include "common.cuh"
#include "mg_transfer.h"
#include "stencil.cuh"

namespace poro {

// P~ = diag(1 - bc_fine) P diag(1 - bc_coarse) and R~ = P~^T (unscaled: with it the coarse generated block is the Galerkin
// product R~ B P~ on the free dofs) of one field
struct MgTransfer {
    StencilOp fine, coarse;          // diagonal field blocks (fr == fc) of the two levels
    int dim = 0, kind = 0, br = 0, Nc = 0;
    int64_t nf = 0, nc = 0;          // nodes of the fine / coarse lattice
    const uint8_t* bcf = nullptr;    // Dirichlet flags of the field's rows on each level, or null
    const uint8_t* bcc = nullptr;
    DBuf<int> pptr, rptr;
    DBuf<poromg::Entry> pent, rent;
    int64_t ptab_bytes = 0, rtab_bytes = 0;
};

// number of coarse levels attached below the matrix of `s` (poro_mat_set_coarse)
int mg_attached_levels(const StencilOp& s);
// the same field block of the next level, cut out of its generated matrix (carries its descriptor: products run k_stencil)
void mg_coarse_block(Ctx& c, const StencilOp& s, Csr& out);
void mg_transfer_init(Ctx& c, MgTransfer& t, const StencilOp& fine, const StencilOp& coarse);
// y = P~ e (add = false) or y += P~ e (add = true); e on the coarse level, y on the fine level
void mg_prolong(Ctx& c, const MgTransfer& t, const double* e, double* y, bool add);
// y = R~ r; r on the fine level, y on the coarse level
void mg_restrict(Ctx& c, const MgTransfer& t, const double* r, double* y);
// coarse near-nullspace: the fine rows of the coinciding nodes (fine lattice index = 2 x coarse), n_c x k
void mg_inject(Ctx& c, const MgTransfer& t, const double* B, int k, DBuf<double>& Bc);
// algorithmic bytes of one launch: the vectors it reads and writes, the flags it reads, the tables
int64_t mg_prolong_bytes(const MgTransfer& t, bool add);
int64_t mg_restrict_bytes(const MgTransfer& t);

}  // namespace poro
