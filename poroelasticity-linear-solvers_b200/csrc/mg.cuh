// mg.cuh -- geometric transfer between a generated field block and the same block generated at N/2 (mg.cu), the pieces of
// `-<prefix>pc_type mg`.  The levels are linked by poro_mat_set_coarse (StencilData::coarse); the transfer is pure geometry
// (mg_transfer.h), so it has no matrix: columns come from the lattice position, the Dirichlet flags from the two levels.
#pragma once
#include "common.cuh"
#include "mg_transfer.h"
#include "stencil.cuh"

namespace poro {

// the ghost nodes one transfer reads from a level vector stored [owned | ghost] (row-partitioned slabs): the owned nodes
// [o0, o1) map by arithmetic, the nodes of the ghost planes [g0, o0) and [o1, g1) through `tab` (index node - g0 below the
// owned nodes, o0 - g0 + node - o1 above them): the ghost dof of component 0, or -1 when the node is not held.  The
// components of a ghost node are consecutive.  Single rank: [0, n) owned, no table.
struct MgGhosts {
    int64_t o0 = 0, o1 = 0, g0 = 0, g1 = 0;
    DBuf<int> tab;
    DBuf<uint8_t> bc;                // Dirichlet flags of the ghost dofs (received from their owners), or empty
};

// P~ = diag(1 - bc_fine) P diag(1 - bc_coarse) and R~ = P~^T (unscaled: with it the coarse generated block is the Galerkin
// product R~ B P~ on the free dofs) of one field
struct MgTransfer {
    StencilOp fine, coarse;          // diagonal field blocks (fr == fc) of the two levels
    int dim = 0, kind = 0, br = 0, Nc = 0;
    int64_t nf = 0, nc = 0;          // owned nodes of the fine / coarse lattice (single rank: all of them)
    const uint8_t* bcf = nullptr;    // Dirichlet flags of the field's owned rows on each level, or null
    const uint8_t* bcc = nullptr;
    DBuf<int> pptr, rptr;
    DBuf<poromg::Entry> pent, rent;
    int64_t ptab_bytes = 0, rtab_bytes = 0;
    // row-partitioned slabs: prolongation reads coarse ghosts of the coarse level's plan (the cycle refreshes them), the
    // restriction reads fine ghosts of its own transfer plan `tplan` (received into `tghost` by each restriction)
    bool dist = false;
    MgGhosts cg, fg;
    std::unique_ptr<DistPlan> tplan;
    DBuf<double> tghost;
};

// number of coarse levels attached below the matrix of `s` (poro_mat_set_coarse)
int mg_attached_levels(const StencilOp& s);
// the same field block of the next level, cut out of its generated matrix (carries its descriptor: on one rank products run
// k_stencil).  A slab block has columns [owned | lower ghosts | upper ghosts] and gets its halo plan in `plan` (collective).
void mg_coarse_block(Ctx& c, const StencilOp& s, Csr& out, std::unique_ptr<DistPlan>* plan = nullptr);
// cplan: halo plan of the coarse block (slabs; collective: builds the transfer plan and exchanges the ghost flags)
void mg_transfer_init(Ctx& c, MgTransfer& t, const StencilOp& fine, const StencilOp& coarse, DistPlan* cplan = nullptr);
// y = P~ e (add = false) or y += P~ e (add = true); e on the coarse level (slabs: [owned | ghost], ghosts current), y on the
// fine level (owned rows)
void mg_prolong(Ctx& c, const MgTransfer& t, const double* e, double* y, bool add);
// y = R~ r; r on the fine level (owned rows; slabs: the transfer halo is exchanged first, collective), y on the coarse level
void mg_restrict(Ctx& c, MgTransfer& t, const double* r, double* y);
// coarse near-nullspace: the fine rows of the coinciding nodes (fine lattice index = 2 x coarse), n_c x k (owned nodes: the
// coinciding fine node of an owned coarse node is owned by the same rank, the slabs nest)
void mg_inject(Ctx& c, const MgTransfer& t, const double* B, int k, DBuf<double>& Bc);
// algorithmic bytes of one launch: the vectors it reads and writes, the flags it reads, the tables
int64_t mg_prolong_bytes(const MgTransfer& t, bool add);
int64_t mg_restrict_bytes(const MgTransfer& t);

}  // namespace poro
