// mg_transfer.h -- class tables of the geometric transfer between the structured meshes at N/2 and N (host C++17; also
// compiled by g++ in tests/mg_transfer_harness.cpp).
//
// dolfin's UnitSquareMesh ("right" diagonal) and UnitCubeMesh (6 tets around the main diagonal) split every cell in the
// Kuhn way: the simplex holding a point t of the unit cell is {t_s1 >= t_s2 >= ...} for the permutation s that sorts t,
// and the mesh at N is the same triangulation refined once, so it is nested in the one at N/2.  The prolongation of a
// field is its coarse basis evaluated at the fine nodes.  Per axis a fine node sits at lattice index X = M c + r of coarse
// cell c (M = 4 on the P2 lattice, 2 on the P1 lattice), so its row is the table of class r (one per residue vector,
// M^dim classes) shifted to the cell: entries (coarse node 2 c + b on the P2 lattice, c + b on the P1 lattice, weight).
// The last plane X = M N_c is class r = 0 of the cell "N_c": only entries with b = 0 on that axis survive (the others have
// weight exactly 0 and are dropped), so no entry leaves the domain.  The weights are dyadic rationals, exact in binary.
//
// Restriction is the exact transpose: for a coarse node Y the fine node of entry (r, b) is X = 2 Y + (r - 2 b), and the
// entry belongs to the coarse class b mod S (S = 2 on the P2 lattice: vertex / edge node per axis; S = 1 on the P1 lattice).
// Fine nodes outside the domain are skipped by the caller.
#pragma once
#include <stdint.h>
#include <algorithm>
#include <vector>

namespace poromg {

struct Entry {
    int d[3];        // prolongation: coarse offset b per axis; restriction: fine offset r - 2 b per axis
    double w;
};

struct Table {
    int ncls = 0;
    std::vector<int> ptr;       // ncls + 1
    std::vector<Entry> e;
};

// fine lattice steps per coarse cell and coarse lattice steps per coarse cell
inline int fine_per_cell(int kind) { return kind == 2 ? 4 : 2; }
inline int coarse_per_cell(int kind) { return kind == 2 ? 2 : 1; }

// the nonzero coarse basis functions of a lattice (kind 2: P2, kind 1: P1) at the point t of the unit cell, in a fixed order
// (vertices of the Kuhn simplex, then its edges); b is the node offset inside the cell on the coarse lattice
inline void basis_at(int kind, int dim, const double* t, std::vector<Entry>& out) {
    out.clear();
    int s[3] = {0, 1, 2};
    std::stable_sort(s, s + dim, [&](int a, int b) { return t[a] > t[b]; });
    int v[4][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}};    // vertices of the simplex: v_k = v_{k-1} + e_{s_k}
    double lam[4];
    for (int k = 1; k <= dim; ++k) {
        for (int m = 0; m < 3; ++m) v[k][m] = v[k - 1][m];
        v[k][s[k - 1]] = 1;
    }
    lam[0] = 1.0 - t[s[0]];
    for (int k = 1; k < dim; ++k) lam[k] = t[s[k - 1]] - t[s[k]];
    lam[dim] = t[s[dim - 1]];
    auto push = [&](const int* b, int scale, const int* b2, double w) {
        if (w == 0.0) return;
        Entry e{{0, 0, 0}, w};
        for (int m = 0; m < dim; ++m) e.d[m] = scale * b[m] + (b2 ? b2[m] : 0);
        out.push_back(e);
    };
    if (kind == 1) {
        for (int k = 0; k <= dim; ++k) push(v[k], 1, nullptr, lam[k]);
        return;
    }
    for (int k = 0; k <= dim; ++k) push(v[k], 2, nullptr, lam[k] * (2.0 * lam[k] - 1.0));
    for (int i = 0; i <= dim; ++i)
        for (int j = i + 1; j <= dim; ++j) push(v[i], 1, v[j], 4.0 * lam[i] * lam[j]);
}

// prolongation: class id = sum_m r_m M^m, r_m = X_m mod M
inline Table prolong_table(int kind, int dim) {
    const int M = fine_per_cell(kind);
    Table T;
    T.ncls = 1;
    for (int m = 0; m < dim; ++m) T.ncls *= M;
    T.ptr.assign(1, 0);
    std::vector<Entry> row;
    for (int cls = 0; cls < T.ncls; ++cls) {
        double t[3] = {0, 0, 0};
        for (int m = 0, q = cls; m < dim; ++m, q /= M) t[m] = (double)(q % M) / M;
        basis_at(kind, dim, t, row);
        T.e.insert(T.e.end(), row.begin(), row.end());
        T.ptr.push_back((int)T.e.size());
    }
    return T;
}

// restriction: class id = sum_m (Y_m mod S) S^m; entry offsets are fine-lattice offsets from 2 Y
inline Table restrict_table(int kind, int dim) {
    const int M = fine_per_cell(kind), S = coarse_per_cell(kind);
    const Table P = prolong_table(kind, dim);
    Table T;
    T.ncls = 1;
    for (int m = 0; m < dim; ++m) T.ncls *= S;
    std::vector<std::vector<Entry>> per((size_t)T.ncls);
    for (int cls = 0; cls < P.ncls; ++cls) {
        int r[3] = {0, 0, 0};
        for (int m = 0, q = cls; m < dim; ++m, q /= M) r[m] = q % M;
        for (int p = P.ptr[cls]; p < P.ptr[cls + 1]; ++p) {
            const Entry& e = P.e[p];
            int qc = 0;
            Entry f{{0, 0, 0}, e.w};
            for (int m = dim - 1; m >= 0; --m) {
                qc = qc * S + e.d[m] % S;
                f.d[m] = r[m] - 2 * e.d[m];
            }
            per[qc].push_back(f);
        }
    }
    T.ptr.assign(1, 0);
    for (auto& v : per) {
        T.e.insert(T.e.end(), v.begin(), v.end());
        T.ptr.push_back((int)T.e.size());
    }
    return T;
}

// planes [lo, hi) of the target lattice that the rows of the planes [a, b) of the source lattice reach along axis dim - 1
// (the slab axis of a row partition): prolongation rows of fine planes Z reach coarse planes S (Z / M) + d, restriction
// rows of coarse planes Y fine planes 2 Y + d (planes outside [0, L_to) skipped, as the restriction kernel skips them).
// lo = hi = a when no row has an entry.
inline void plane_reach(const Table& T, int dim, bool prolong, int kind, int64_t a, int64_t b, int64_t L_to, int64_t& lo, int64_t& hi) {
    const int M = fine_per_cell(kind), S = coarse_per_cell(kind), R = prolong ? M : S;
    int stride = 1;
    for (int m = 0; m < dim - 1; ++m) stride *= R;
    lo = a; hi = a;
    bool any = false;
    for (int64_t Z = a; Z < b; ++Z)
        for (int cls = 0; cls < T.ncls; ++cls) {
            if ((cls / stride) % R != Z % R) continue;
            for (int p = T.ptr[cls]; p < T.ptr[cls + 1]; ++p) {
                const int64_t t = (prolong ? S * (Z / M) : 2 * Z) + T.e[p].d[dim - 1];
                if (t < 0 || t >= L_to) continue;
                lo = any ? std::min(lo, t) : t;
                hi = any ? std::max(hi, t + 1) : t + 1;
                any = true;
            }
        }
}

}  // namespace poromg
