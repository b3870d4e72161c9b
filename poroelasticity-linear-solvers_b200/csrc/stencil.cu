// stencil.cu -- products of generated structured-mesh blocks straight from their class tables (stencil.cuh).
//
// k_stencil: one thread per row node with all BR components of the node's block row.  The warps are laid out per row
// class (StencilData::wdesc), so that the class -- and with it the entry count, the column offsets and the values -- is
// the same on every lane: table reads are broadcasts through L1, no warp diverges.  Inside a class the lanes run along
// axis 0, so the gathers of x (one field vector, L2-resident) and the epilogue accesses are as contiguous as the class
// allows.  Columns are base + off[p] (no column indices in memory); a Dirichlet row applies DirichletBC.apply's
// semantics like porogen::row_item (unit diagonal in the diagonal field block, zero elsewhere); only boundary classes
// can hold one, so interior warps never read the flags.  No atomics: the sum order of a row is fixed (tables in column
// field order, entries in table order), so results are bitwise reproducible.  Entries whose block is all zero are
// dropped when the tables are uploaded (gen.cu); the zeros left inside a block are multiplied (cheaper than a test).
//
// Algorithmic bytes of a plain product: 8 B per entry of x per column field + the tables + 1 B per Dirichlet flag read
// + 8 B per row of y (the epilogues add their vectors, 56 B per row for the Chebyshev step).
#include "stencil.cuh"
#include "spmv_epilogue.cuh"

namespace poro {

static constexpr int kStBlock = 256;

struct StencilArgs {
    porogen::BlockTable t[3];    // the tables summed into each row, in column-field order
    int64_t xoff[3];             // offset of each table's column field inside x
    int diag_only[3];
    int nt;
    const uint8_t* bc;           // Dirichlet flags of the row field's rows, or null
    int unit_diag;               // x holds the row field itself: a Dirichlet row reads x[diag_xoff + row]
    int64_t diag_xoff;
    int dim, N, kr;
    const int2* wdesc;
    int nwarps;
};

// nodes of a lattice axis in one axis class (codes of porogen::axis_class) and the position of the i-th of them
__device__ __forceinline__ int st_axis_count(int kind, int N, int a) {
    if (kind == 2) return a == 0 ? N : (a == 3 ? N - 1 : 1);      // odd | first | last | even interior
    return a == 2 ? N - 1 : 1;                                     // first | last | interior
}
__device__ __forceinline__ int st_axis_pos(int kind, int N, int a, int i) {
    if (kind == 2) return a == 0 ? 2 * i + 1 : a == 1 ? 0 : a == 2 ? 2 * N : 2 * i + 2;
    return a == 0 ? 0 : a == 1 ? N : i + 1;
}

template <int BR, int BC>
__device__ __forceinline__ void st_accum(const porogen::BlockTable& t, int cls, int64_t base, const double* __restrict__ x, double (&acc)[BR]) {
    const int p0 = __ldg(t.cls_ptr + cls), p1 = __ldg(t.cls_ptr + cls + 1);
#pragma unroll 2
    for (int p = p0; p < p1; ++p) {
        const double* __restrict__ xc = x + (base + __ldg(t.off + p)) * BC;
        double xv[BC];
#pragma unroll
        for (int j = 0; j < BC; ++j) xv[j] = __ldg(xc + j);
        const double* __restrict__ v = t.vals + (int64_t)p * (BR * BC);
#pragma unroll
        for (int i = 0; i < BR; ++i)
#pragma unroll
            for (int j = 0; j < BC; ++j) acc[i] = fma(__ldg(v + i * BC + j), xv[j], acc[i]);
    }
}

// diagonal blocks (BR == BC): one value per component
template <int BR>
__device__ __forceinline__ void st_accum_diag(const porogen::BlockTable& t, int cls, int64_t base, const double* __restrict__ x, double (&acc)[BR]) {
    const int p0 = __ldg(t.cls_ptr + cls), p1 = __ldg(t.cls_ptr + cls + 1);
#pragma unroll 2
    for (int p = p0; p < p1; ++p) {
        const double* __restrict__ xc = x + (base + __ldg(t.off + p)) * BR;
        const double* __restrict__ v = t.vals + (int64_t)p * (BR * BR);
#pragma unroll
        for (int i = 0; i < BR; ++i) acc[i] = fma(__ldg(v + i * BR + i), __ldg(xc + i), acc[i]);
    }
}

template <int BR, int MODE>
__global__ void __launch_bounds__(kStBlock) k_stencil(StencilArgs a, const double* __restrict__ x, double* __restrict__ y, Epilogue ep,
                                                      double* __restrict__ dot_partial) {
    __shared__ double red[kStBlock / 32];
    const int warp = (int)(((int64_t)blockIdx.x * kStBlock + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    double contrib = 0.0;
    if (warp < a.nwarps) {
        const int2 wd = __ldg(a.wdesc + warp);
        const int cls = wd.x;
        const int ncl = a.kr == 2 ? 4 : 3;
        const int L = porogen::lattice_extent(a.kr, a.N);
        int k = wd.y + lane;
        int total = 1, rem = cls;
        int ac[3], cnt[3];
        bool boundary = false;
        // fixed trip counts (dim <= 3) keep ac / cnt / pos in registers
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            ac[m] = 0; cnt[m] = 1;
            if (m >= a.dim) continue;
            ac[m] = rem % ncl;
            rem /= ncl;
            cnt[m] = st_axis_count(a.kr, a.N, ac[m]);
            total *= cnt[m];
            boundary |= a.kr == 2 ? (ac[m] == 1 || ac[m] == 2) : ac[m] != 2;
        }
        if (k < total) {
            int pos[3];
            int64_t node = 0, mul = 1;
#pragma unroll
            for (int m = 0; m < 3; ++m) {
                pos[m] = 0;
                if (m >= a.dim) continue;
                const int i = k % cnt[m];
                k /= cnt[m];
                pos[m] = st_axis_pos(a.kr, a.N, ac[m], i);
                node += pos[m] * mul;
                mul *= L;
            }
            double acc[BR];
#pragma unroll
            for (int i = 0; i < BR; ++i) acc[i] = 0.0;
            for (int q = 0; q < a.nt; ++q) {
                const porogen::BlockTable& t = a.t[q];
                // base column node (porogen::row_info): the column-lattice node of the local origin of cell c0
                const int Lc = porogen::lattice_extent(t.kc, a.N), sc = t.kc == 2 ? 2 : 1;
                int64_t base = 0, mc = 1;
#pragma unroll
                for (int m = 0; m < 3; ++m) {
                    if (m >= a.dim) continue;
                    base += (int64_t)sc * (a.kr == 2 ? pos[m] / 2 : pos[m]) * mc;
                    mc *= Lc;
                }
                const double* xs = x + a.xoff[q];
                if (a.diag_only[q]) st_accum_diag<BR>(t, cls, base, xs, acc);      // only set when br == bc
                else if (t.bc == 3) st_accum<BR, 3>(t, cls, base, xs, acc);
                else if (t.bc == 2) st_accum<BR, 2>(t, cls, base, xs, acc);
                else st_accum<BR, 1>(t, cls, base, xs, acc);
            }
            const int64_t r0 = node * BR;
            if (boundary && a.bc) {
#pragma unroll
                for (int i = 0; i < BR; ++i)
                    if (a.bc[r0 + i]) acc[i] = a.unit_diag ? x[a.diag_xoff + r0 + i] : 0.0;
            }
#pragma unroll
            for (int i = 0; i < BR; ++i) contrib += apply_epilogue<MODE>(ep, (int)(r0 + i), acc[i], x, y);
        }
    }
    if (MODE == 4) {
        const double t = block_sum_256(contrib, red);
        if (threadIdx.x == 0) dot_partial[blockIdx.x] = t;
    }
}

void stencil_build_warps(Ctx& c, StencilData& d) {
    for (int kind = 1; kind <= 2; ++kind) {
        const int ncl = kind == 2 ? 4 : 3;
        int nclass = 1;
        for (int m = 0; m < d.dim; ++m) nclass *= ncl;
        auto count = [&](int a) { return kind == 2 ? (a == 0 ? d.N : (a == 3 ? d.N - 1 : 1)) : (a == 2 ? d.N - 1 : 1); };
        std::vector<int2> w;
        for (int cls = 0; cls < nclass; ++cls) {
            int64_t total = 1;
            for (int m = 0, r = cls; m < d.dim; ++m, r /= ncl) total *= count(r % ncl);
            for (int64_t f = 0; f < total; f += 32) w.push_back(make_int2(cls, (int)f));
        }
        d.nwarps[kind - 1] = (int)w.size();
        d.wdesc[kind - 1].alloc(w.size());
        if (!w.empty())
            PORO_CUDA(cudaMemcpyAsync(d.wdesc[kind - 1].p, w.data(), w.size() * sizeof(int2), cudaMemcpyHostToDevice, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
    }
}

static StencilArgs stencil_args(const StencilOp& s) {
    const StencilData& d = *s.d;
    StencilArgs a{};
    const int fr = s.fr;
    for (int fc = 0; fc < 3; ++fc) {
        if (s.fc >= 0 && fc != s.fc) continue;
        const int b = fr * 3 + fc;
        if (!d.present[b]) continue;
        a.t[a.nt] = d.t[b];
        a.xoff[a.nt] = s.fc >= 0 ? 0 : d.row0[fc];
        a.diag_only[a.nt] = d.diag_only[b];
        a.nt++;
    }
    a.bc = d.bc.p ? d.bc.p + d.row0[fr] : nullptr;
    a.unit_diag = s.fc < 0 || s.fc == fr;
    a.diag_xoff = s.fc >= 0 ? 0 : d.row0[fr];
    a.dim = d.dim;
    a.N = d.N;
    a.kr = d.kind[fr];
    a.wdesc = d.wdesc[a.kr - 1].p;
    a.nwarps = d.nwarps[a.kr - 1];
    return a;
}

int stencil_grid(const StencilOp& s) { return ceil_div((int64_t)s.d->nwarps[s.d->kind[s.fr] - 1] * 32, kStBlock); }

template <int MODE>
int stencil_launch(Ctx& c, const StencilOp& s, const double* x, double* y, const Epilogue& ep, double* dot_partial) {
    PORO_REQUIRE(!s.d->slab, "k_stencil: a row-partitioned slab has ghost columns and is applied assembled");
    const StencilArgs a = stencil_args(s);
    const int grid = stencil_grid(s);
    if (grid == 0) return 0;
    switch (s.d->bdim[s.fr]) {
        case 3: k_stencil<3, MODE><<<grid, kStBlock, 0, c.stream>>>(a, x, y, ep, dot_partial); break;
        case 2: k_stencil<2, MODE><<<grid, kStBlock, 0, c.stream>>>(a, x, y, ep, dot_partial); break;
        default: k_stencil<1, MODE><<<grid, kStBlock, 0, c.stream>>>(a, x, y, ep, dot_partial); break;
    }
    PORO_LAUNCH_CHECK(c);
    return grid;
}
template int stencil_launch<SPMV_SET>(Ctx&, const StencilOp&, const double*, double*, const Epilogue&, double*);
template int stencil_launch<SPMV_SUB>(Ctx&, const StencilOp&, const double*, double*, const Epilogue&, double*);
template int stencil_launch<SPMV_ADD>(Ctx&, const StencilOp&, const double*, double*, const Epilogue&, double*);
template int stencil_launch<3>(Ctx&, const StencilOp&, const double*, double*, const Epilogue&, double*);
template int stencil_launch<4>(Ctx&, const StencilOp&, const double*, double*, const Epilogue&, double*);

void stencil_spmv(Ctx& c, const StencilOp& s, const double* x, double* y, SpmvMode mode, const double* z) {
    Epilogue ep{};
    ep.mode = mode;
    ep.z = z;
    if (mode == SPMV_SET) stencil_launch<SPMV_SET>(c, s, x, y, ep, nullptr);
    else if (mode == SPMV_SUB) stencil_launch<SPMV_SUB>(c, s, x, y, ep, nullptr);
    else stencil_launch<SPMV_ADD>(c, s, x, y, ep, nullptr);
}

int64_t stencil_bytes(const StencilOp& s) {
    const StencilData& d = *s.d;
    const int fr = s.fr;
    const int64_t rows = d.row0[fr + 1] - d.row0[fr];
    int64_t b = 8 * rows + (d.bc.p ? rows : 0);
    for (int fc = 0; fc < 3; ++fc) {
        if ((s.fc >= 0 && fc != s.fc) || !d.present[fr * 3 + fc]) continue;
        b += 8 * (d.row0[fc + 1] - d.row0[fc]) + d.table_bytes[fr * 3 + fc];
    }
    return b;
}

}  // namespace poro
