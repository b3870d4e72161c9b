// CPU harness of csrc/mg_transfer.h: expands the class tables of the geometric transfer into (row, column, value) triplets
// the way k_prolong / k_restrict (csrc/mg.cu) walk them, with the Dirichlet masks of both levels.  tests/test_mg_host.py
// compares the result with the scipy P~ of hostfem/mg.py.
#include "mg_transfer.h"

extern "C" {

// dir 0: P~ (rows fine dofs, columns coarse dofs); dir 1: R~ (rows coarse dofs, columns fine dofs).  bcf / bcc: one flag
// per dof of each level or null.  Returns the number of triplets (written only while below cap).
int64_t mg_expand(int dim, int kind, int Nc, int bs, const uint8_t* bcf, const uint8_t* bcc, int dir, int64_t* rows, int64_t* cols,
                  double* vals, int64_t cap) {
    const int M = poromg::fine_per_cell(kind), S = poromg::coarse_per_cell(kind);
    const int Lf = kind == 2 ? 4 * Nc + 1 : 2 * Nc + 1, Lc = kind == 2 ? 2 * Nc + 1 : Nc + 1;
    const poromg::Table T = dir == 0 ? poromg::prolong_table(kind, dim) : poromg::restrict_table(kind, dim);
    int64_t nf = 1, nc = 1;
    for (int m = 0; m < dim; ++m) { nf *= Lf; nc *= Lc; }
    int64_t n = 0;
    auto emit = [&](int64_t r, int64_t c, double v) {
        if (n < cap) { rows[n] = r; cols[n] = c; vals[n] = v; }
        ++n;
    };
    if (dir == 0) {
        for (int64_t node = 0; node < nf; ++node) {
            int base[3] = {0, 0, 0}, cls = 0, mul = 1;
            int64_t q = node;
            for (int m = 0; m < dim; ++m) {
                const int X = (int)(q % Lf);
                q /= Lf;
                cls += (X % M) * mul;
                mul *= M;
                base[m] = S * (X / M);
            }
            for (int p = T.ptr[cls]; p < T.ptr[cls + 1]; ++p) {
                int64_t cn = 0, mc = 1;
                for (int m = 0; m < dim; ++m) { cn += (int64_t)(base[m] + T.e[p].d[m]) * mc; mc *= Lc; }
                for (int i = 0; i < bs; ++i) {
                    if ((bcf && bcf[node * bs + i]) || (bcc && bcc[cn * bs + i])) continue;
                    emit(node * bs + i, cn * bs + i, T.e[p].w);
                }
            }
        }
    } else {
        for (int64_t node = 0; node < nc; ++node) {
            int Y[3] = {0, 0, 0}, cls = 0, mul = 1;
            int64_t q = node;
            for (int m = 0; m < dim; ++m) {
                Y[m] = (int)(q % Lc);
                q /= Lc;
                cls += (Y[m] % S) * mul;
                mul *= S;
            }
            for (int p = T.ptr[cls]; p < T.ptr[cls + 1]; ++p) {
                int64_t fn = 0, mf = 1;
                bool inside = true;
                for (int m = 0; m < dim; ++m) {
                    const int X = 2 * Y[m] + T.e[p].d[m];
                    inside = inside && X >= 0 && X < Lf;
                    fn += (int64_t)X * mf;
                    mf *= Lf;
                }
                if (!inside) continue;
                for (int i = 0; i < bs; ++i) {
                    if ((bcc && bcc[node * bs + i]) || (bcf && bcf[fn * bs + i])) continue;
                    emit(node * bs + i, fn * bs + i, T.e[p].w);
                }
            }
        }
    }
    return n;
}

}
