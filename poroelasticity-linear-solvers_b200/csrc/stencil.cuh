// stencil.cuh -- generated structured-mesh operators applied from their class tables (stencil.cu).
//
// A matrix that poro_gen_matrix builds keeps what it was built from: the nine field-block tables (gen_stencil.cuh), the row
// layout and the Dirichlet row flags.  A block cut out of it along whole fields (one row field x one column field) carries
// the same description, and its products run k_stencil instead of streaming the assembled CSR: the kernel reads only the
// vectors the product touches (plus a few hundred KB of tables that stay in L1 / L2).  The CSR stays alongside for every
// consumer of the assembled form (AMG set-up, Schur assembly, poro_mat_copy, poro_mat_mult).
#pragma once
#include "common.cuh"
#include "gen_stencil.cuh"

namespace poro {

struct Epilogue;

// everything one generated matrix was built from.  A whole-lattice matrix (one rank, no ghosts) is applied from it; a
// row-partitioned slab (`slab`) keeps it for the geometry of its geometric transfers (mg.cuh) and stays assembled.
struct StencilData {
    int dim = 0, N = 0;
    // slab: per lattice (index kind - 1) the owned node range and the ghost node ranges of the lower / upper neighbour, and
    // per field the first local column of its lower / upper ghosts (columns [owned s f p | lower s f p | upper s f p])
    bool slab = false;
    int64_t o0[2] = {0, 0}, o1[2] = {0, 0}, gl0[2] = {0, 0}, gl1[2] = {0, 0}, gu0[2] = {0, 0}, gu1[2] = {0, 0};
    int64_t off_gl[3] = {0, 0, 0}, off_gu[3] = {0, 0, 0};
    porogen::BlockTable t[9];        // block (fr, fc) at fr * 3 + fc; device pointers into the buffers below
    int present[9] = {0};
    int diag_only[9] = {0};          // every entry of the table is a diagonal block (mass couplings M (x) I)
    int64_t table_bytes[9] = {0};
    DBuf<int32_t> cls[9];
    DBuf<int64_t> off[9];
    DBuf<double> val[9];
    DBuf<uint8_t> bc;                // one Dirichlet flag per row of the matrix, or empty
    int64_t row0[4] = {0};           // first row of each field; row0[3] = rows
    int bdim[3] = {0}, kind[3] = {0};
    // warps of the kernel per lattice (index kind - 1): {class, first node of the warp inside the class}; every lane of a
    // warp has the same class, so table reads are broadcasts and no warp diverges on the entry count
    DBuf<int2> wdesc[2];
    int nwarps[2] = {0};
    // next geometric level (poro_mat_set_coarse): the same matrix generated at N / 2, shared with its handle; its own
    // descriptor may link further down (mg.cuh)
    std::shared_ptr<const Csr> coarse;
};

// the operator of a Csr: row field `fr` against column field `fc` (a block extracted along whole fields), or against all
// column fields (fc = -1: the row field's slice of the whole matrix, used by the outer operator).  fr = -1 describes the
// whole matrix: it is never launched as such (poro_mat_mult stays on the assembled path).
struct StencilOp {
    std::shared_ptr<StencilData> d;
    int fr = -1, fc = -1;
};

// products of A run from the class tables: a field block of a whole-lattice descriptor
inline bool stencil_runs(const Csr& A) { return A.stencil && A.stencil->fr >= 0 && !A.stencil->d->slab; }

// builds the per-lattice warp descriptors of `d` (host work, once per generated matrix)
void stencil_build_warps(Ctx& c, StencilData& d);
// launches of row field `s.fr` (s.fc >= 0: x is field fc's vector; s.fc < 0: x is the whole [s | f | p] vector), y and the
// epilogue vectors indexed by the row field's rows.  Returns the grid (MODE 4 writes one partial per CTA).
template <int MODE>
int stencil_launch(Ctx& c, const StencilOp& s, const double* x, double* y, const Epilogue& ep, double* dot_partial);
int stencil_grid(const StencilOp& s);
// y = A x | y = z - A x | y = z + A x with the same argument conventions
void stencil_spmv(Ctx& c, const StencilOp& s, const double* x, double* y, SpmvMode mode, const double* z);
// algorithmic bytes of one plain product y = B x: 8 B per entry of x per column field, the tables, the Dirichlet flags and y
int64_t stencil_bytes(const StencilOp& s);

}  // namespace poro
