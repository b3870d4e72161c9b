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
// k_stencil_brick: the same products for a 3-D P2 row field (s, f) in one launch, with its interior rows -- odd or
// even-interior on every axis, 8 of the 64 classes and most of the nodes -- applied from shared-memory bricks of x (see
// st_brick) and the boundary classes on the per-class warps.  `-poro_stencil_brick 0` at generation keeps every row on
// k_stencil; lattices too small for one box, P1 rows and dim 2 always are.
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
    // brick path (BR == 3 on the P2 lattice of a 3-D field): bricks, boxes per axis and their extent, and per table the
    // staged layout and the shared-memory offsets of the entries
    int nbrick, nb[3], bext[3];
    BrickGeom bg[3];
    const int32_t* soff[3];
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

// ---- brick path (3-D P2 row fields, interior classes) ------------------------------------------------------------------
//
// A CTA owns a box of row positions [r0, r1) per axis, inside the interior range [1, 2N - 1] of the P2 lattice, where
// every row class is odd or even-interior on every axis.  The nodes of one parity triple (= one row class) inside the box
// are numbered axis 0 fastest and cut into chunks of 64; a warp takes chunks w, w + 8, ... and a lane handles nodes k and
// k + 32 of its chunk, so each table value it loads feeds two rows.  Per table, in column-field order, the CTA stages the
// column region the box reaches (StencilData::bg: reach from the tables, clamped to the lattice) in shared memory with
// coalesced asynchronous copies, then sums from there.  The sums of the box then pass through shared memory, so that the
// epilogue runs over contiguous rows.  The per-row sum order is that of the per-class warps.
static constexpr int kBrickX = 68;       // largest box extent along axis 0 (whole interior up to N = 34)
static constexpr int kBrickYZ = 4;       // box extent along axes 1 and 2
static constexpr int kBrickCPW = 3;      // chunks of 64 nodes per warp: a box holds at most 8 classes x 3 chunks
static constexpr int kBrickSmem = 112 * 1024;    // two CTAs per SM

__host__ __device__ __forceinline__ int st_cb(int kc, int r) { return kc == 2 ? (r & ~1) : (r >> 1); }
// first staged column of axis m for the rows [r0, r1) (rows of one parity: the lowest reach is at the first of them)
__host__ __device__ __forceinline__ int brick_origin(const BrickGeom& g, int kc, int m, int r0, int r1) {
    int o = st_cb(kc, r0) + g.lo[m][r0 & 1];
    if (r1 > r0 + 1) o = min(o, st_cb(kc, r0 + 1) + g.lo[m][(r0 + 1) & 1]);
    return m == 0 && kc == 2 ? (o & ~1) : o;       // parity-split rows start at an even column
}
__host__ __device__ __forceinline__ int brick_top(const BrickGeom& g, int kc, int m, int r0, int r1) {
    int t = st_cb(kc, r1 - 1) + g.hi[m][(r1 - 1) & 1];
    if (r1 > r0 + 1) t = max(t, st_cb(kc, r1 - 2) + g.hi[m][(r1 - 2) & 1]);
    return t;
}
// nodes of parity `par` in [r0, r1) and the first of them
__host__ __device__ __forceinline__ int brick_count(int r0, int r1, int par, int& first) {
    first = r0 + ((r0 ^ par) & 1);
    return r1 > first ? (r1 - first + 1) / 2 : 0;
}

template <int BC>
__device__ __forceinline__ void brick_stage(const BrickGeom& g, int kc, int Lc, const int (&o)[3], const double* __restrict__ x,
                                            double* sm) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rowlen = g.e[0] * BC;
    const int c0lo = max(0, -o[0]) * BC, c0hi = min(g.e[0], Lc - o[0]) * BC;
    for (int row = warp; row < g.e[1] * g.e[2]; row += kStBlock / 32) {
        const int u1 = row % g.e[1], u2 = row / g.e[1];
        const int c1 = o[1] + u1, c2 = o[2] + u2;
        if (c1 < 0 || c1 >= Lc || c2 < 0 || c2 >= Lc) continue;
        const double* __restrict__ xr = x + ((int64_t)o[0] + Lc * ((int64_t)c1 + (int64_t)Lc * c2)) * BC;
        double* __restrict__ sr = sm + g.W0 * (u1 + g.e[1] * u2);
        // asynchronous copies (cp.async, no register round trip): every copy of the region is in flight at once
        for (int w = c0lo + lane; w < c0hi && w < rowlen; w += 32) {
            const int u0 = w / BC, j = w - u0 * BC;
            const unsigned d = (unsigned)__cvta_generic_to_shared(sr + j * g.cs + (g.H ? (u0 & 1) * g.H + (u0 >> 1) : u0));
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(__cvta_generic_to_global(xr + w)) : "memory");
        }
    }
    asm volatile("cp.async.wait_all;\n" ::: "memory");
}

template <int BC>
__device__ __forceinline__ void brick_accum(const porogen::BlockTable& t, const int32_t* __restrict__ soff, int cls, int cs,
                                            const double* sm, int rp0, int rp1, double (&a0)[3], double (&a1)[3]) {
    const int p0 = __ldg(t.cls_ptr + cls), p1 = __ldg(t.cls_ptr + cls + 1);
#pragma unroll 2
    for (int p = p0; p < p1; ++p) {
        const int so = __ldg(soff + p);
        const double* xa = sm + rp0 + so;
        const double* xb = sm + rp1 + so;
        double xva[BC], xvb[BC];
#pragma unroll
        for (int j = 0; j < BC; ++j) { xva[j] = xa[j * cs]; xvb[j] = xb[j * cs]; }
        const double* __restrict__ v = t.vals + (int64_t)p * (3 * BC);
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < BC; ++j) {
                const double vv = __ldg(v + i * BC + j);
                a0[i] = fma(vv, xva[j], a0[i]);
                a1[i] = fma(vv, xvb[j], a1[i]);
            }
    }
}

__device__ __forceinline__ void brick_accum_diag(const porogen::BlockTable& t, const int32_t* __restrict__ soff, int cls, int cs,
                                                 const double* sm, int rp0, int rp1, double (&a0)[3], double (&a1)[3]) {
    const int p0 = __ldg(t.cls_ptr + cls), p1 = __ldg(t.cls_ptr + cls + 1);
#pragma unroll 2
    for (int p = p0; p < p1; ++p) {
        const int so = __ldg(soff + p);
        const double* __restrict__ v = t.vals + (int64_t)p * 9;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double vv = __ldg(v + i * 4);
            a0[i] = fma(vv, sm[rp0 + so + i * cs], a0[i]);
            a1[i] = fma(vv, sm[rp1 + so + i * cs], a1[i]);
        }
    }
}

// offset of a row's base column inside the staged region (packed position: 10 bits per axis)
__device__ __forceinline__ int brick_rowpart(const BrickGeom& g, int kc, const int (&o)[3], int pk) {
    const int a0 = st_cb(kc, pk & 1023) - o[0];
    return (g.H ? a0 >> 1 : a0) + g.W0 * ((st_cb(kc, (pk >> 10) & 1023) - o[1]) + g.e[1] * (st_cb(kc, (pk >> 20) & 1023) - o[2]));
}

template <int MODE>
__device__ __forceinline__ double st_brick(const StencilArgs& a, const double* __restrict__ x, double* __restrict__ y,
                                           const Epilogue& ep, double* sm) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int r0[3], r1[3];
    {
        int b = blockIdx.x;
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const int bi = b % a.nb[m];
            b /= a.nb[m];
            r0[m] = 1 + bi * a.bext[m];
            r1[m] = min(r0[m] + a.bext[m], 2 * a.N);
        }
    }
    // this warp's chunks: class (-1: none) and the packed positions of its two nodes (bit 30: the node exists)
    int scls[kBrickCPW], spk[kBrickCPW][2];
    double acc[kBrickCPW][2][3];
#pragma unroll
    for (int s = 0; s < kBrickCPW; ++s) {
        scls[s] = -1;
        spk[s][0] = spk[s][1] = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int i = 0; i < 3; ++i) acc[s][h][i] = 0.0;
        int j = warp + s * (kStBlock / 32);      // chunk index, then inside its class
        for (int c = 0; c < 8; ++c) {
            int f[3], n[3];
#pragma unroll
            for (int m = 0; m < 3; ++m) n[m] = brick_count(r0[m], r1[m], (c >> m) & 1, f[m]);
            const int nc = n[0] * n[1] * n[2], ch = (nc + 63) >> 6;
            if (j >= ch) { j -= ch; continue; }
            // class id of porogen::axis_class: odd -> 0, even interior -> 3 per axis
            scls[s] = ((c & 1) ? 0 : 3) + 4 * ((c & 2) ? 0 : 3) + 16 * ((c & 4) ? 0 : 3);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k = j * 64 + h * 32 + lane;
                const int kk = min(k, nc - 1);
                const int i0 = kk % n[0], i1 = (kk / n[0]) % n[1], i2 = kk / (n[0] * n[1]);
                spk[s][h] = (f[0] + 2 * i0) | ((f[1] + 2 * i1) << 10) | ((f[2] + 2 * i2) << 20) | (k < nc ? 1 << 30 : 0);
            }
            break;
        }
    }
    for (int q = 0; q < a.nt; ++q) {
        const porogen::BlockTable& t = a.t[q];
        const BrickGeom& g = a.bg[q];
        const int kc = t.kc, Lc = porogen::lattice_extent(kc, a.N);
        int o[3];
#pragma unroll
        for (int m = 0; m < 3; ++m) o[m] = brick_origin(g, kc, m, r0[m], r1[m]);
        const double* xs = x + a.xoff[q];
        if (t.bc == 3) brick_stage<3>(g, kc, Lc, o, xs, sm);
        else brick_stage<1>(g, kc, Lc, o, xs, sm);
        __syncthreads();
#pragma unroll
        for (int s = 0; s < kBrickCPW; ++s) {
            if (scls[s] < 0) continue;
            const int rp0 = brick_rowpart(g, kc, o, spk[s][0]), rp1 = brick_rowpart(g, kc, o, spk[s][1]);
#ifdef PORO_DEBUG_STENCIL
            // an interior row reaches only columns inside the staged region and the lattice
            assert(rp0 >= 0 && rp1 >= 0 && rp0 < g.cs && rp1 < g.cs);
#endif
            if (a.diag_only[q]) brick_accum_diag(t, a.soff[q], scls[s], g.cs, sm, rp0, rp1, acc[s][0], acc[s][1]);
            else if (t.bc == 3) brick_accum<3>(t, a.soff[q], scls[s], g.cs, sm, rp0, rp1, acc[s][0], acc[s][1]);
            else brick_accum<1>(t, a.soff[q], scls[s], g.cs, sm, rp0, rp1, acc[s][0], acc[s][1]);
        }
        __syncthreads();
    }
    // epilogue over contiguous rows: the sums go to shared memory (the staging buffer is free after the last barrier)
    // laid out like the rows of the box in y, then each (axis 1, axis 2) line of the box is a run of 3 (r1 - r0) rows
    const int w0 = 3 * (r1[0] - r0[0]), n1 = r1[1] - r0[1], nrun = n1 * (r1[2] - r0[2]);
#pragma unroll
    for (int s = 0; s < kBrickCPW; ++s)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int pk = spk[s][h];
            if (scls[s] < 0 || !(pk & (1 << 30))) continue;
            double* o = sm + ((((pk >> 10) & 1023) - r0[1]) + n1 * (((pk >> 20) & 1023) - r0[2])) * w0 + 3 * ((pk & 1023) - r0[0]);
#pragma unroll
            for (int i = 0; i < 3; ++i) o[i] = acc[s][h][i];
        }
    __syncthreads();
    const int L = porogen::lattice_extent(2, a.N);
    double contrib = 0.0;
    for (int e = threadIdx.x; e < nrun * w0; e += kStBlock) {
        const int run = e / w0, k = e - run * w0;
        const int64_t node = r0[0] + (int64_t)L * ((r0[1] + run % n1) + (int64_t)L * (r0[2] + run / n1));
        contrib += apply_epilogue<MODE>(ep, (int)(node * 3 + k), sm[e], x, y);
    }
    return contrib;
}

// ---- per-class warps (every row field; with bricks, the boundary classes of the P2 row fields) ------------------------
template <int BR, int MODE>
__device__ __forceinline__ double st_warps(const StencilArgs& a, int cta, const double* __restrict__ x, double* __restrict__ y,
                                           const Epilogue& ep) {
    const int warp = (int)(((int64_t)cta * kStBlock + threadIdx.x) >> 5);
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
    return contrib;
}

template <int BR, int MODE>
__global__ void __launch_bounds__(kStBlock) k_stencil(StencilArgs a, const double* __restrict__ x, double* __restrict__ y, Epilogue ep,
                                                      double* __restrict__ dot_partial) {
    __shared__ double red[kStBlock / 32];
    const double contrib = st_warps<BR, MODE>(a, (int)blockIdx.x, x, y, ep);
    if (MODE == 4) {
        const double t = block_sum_256(contrib, red);
        if (threadIdx.x == 0) dot_partial[blockIdx.x] = t;
    }
}

// one launch for a 3-D P2 row field: CTAs [0, nbrick) are bricks, the rest run the warps of the boundary classes
template <int MODE>
__global__ void __launch_bounds__(kStBlock, 2) k_stencil_brick(StencilArgs a, const double* __restrict__ x, double* __restrict__ y,
                                                               Epilogue ep, double* __restrict__ dot_partial) {
    extern __shared__ double st_sm[];
    __shared__ double red[kStBlock / 32];
    const double contrib = (int)blockIdx.x < a.nbrick ? st_brick<MODE>(a, x, y, ep, st_sm)
                                                      : st_warps<3, MODE>(a, (int)blockIdx.x - a.nbrick, x, y, ep);
    if (MODE == 4) {
        const double t = block_sum_256(contrib, red);
        if (threadIdx.x == 0) dot_partial[blockIdx.x] = t;
    }
}

static std::vector<int2> class_warps(const StencilData& d, int kind, bool boundary_only) {
    const int ncl = kind == 2 ? 4 : 3;
    int nclass = 1;
    for (int m = 0; m < d.dim; ++m) nclass *= ncl;
    auto count = [&](int a) { return kind == 2 ? (a == 0 ? d.N : (a == 3 ? d.N - 1 : 1)) : (a == 2 ? d.N - 1 : 1); };
    std::vector<int2> w;
    for (int cls = 0; cls < nclass; ++cls) {
        int64_t total = 1;
        bool interior = true;
        for (int m = 0, r = cls; m < d.dim; ++m, r /= ncl) {
            total *= count(r % ncl);
            interior = interior && (r % ncl == 0 || r % ncl == 3);
        }
        if (boundary_only && interior) continue;
        for (int64_t f = 0; f < total; f += 32) w.push_back(make_int2(cls, (int)f));
    }
    return w;
}

template <int MODE>
static void brick_smem_attr(int bytes) {
    PORO_CUDA(cudaFuncSetAttribute(k_stencil_brick<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
}

// the brick path of the 3-D P2 row fields: box layout, per-table reach and staged layout, entry offsets in shared memory.
// Leaves d.brick = 0 (every row on the per-class warps) when a table reaches further than the layout assumes.
static void stencil_build_bricks(Ctx& c, StencilData& d) {
    const int N = d.N, nint = 2 * N - 1;
    if (d.dim != 3 || nint < kBrickYZ) return;
    int nb[3], bext[3];
    for (int m = 0; m < 3; ++m) {
        const int cap = m == 0 ? kBrickX : kBrickYZ;
        bext[m] = (int)ceil_div(nint, ceil_div(nint, cap));
        nb[m] = (int)ceil_div(nint, bext[m]);
    }
    BrickGeom bg[9]{};
    std::vector<std::vector<int32_t>> soff(9);
    for (int b = 0; b < 9; ++b) {
        const int fr = b / 3;
        if (!d.present[b] || d.kind[fr] != 2 || d.bdim[fr] != 3) continue;
        const porogen::BlockTable& t = d.t[b];
        const int kc = t.kc, Lc = porogen::lattice_extent(kc, N);
        if (Lc < 5) return;                         // offsets of +-2 along an axis would not decompose uniquely
        std::vector<int32_t> cp(65);
        PORO_CUDA(cudaMemcpyAsync(cp.data(), t.cls_ptr, cp.size() * 4, cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        std::vector<int64_t> off((size_t)cp[64]);
        if (!off.empty()) PORO_CUDA(cudaMemcpyAsync(off.data(), t.off, off.size() * 8, cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        BrickGeom& g = bg[b];
        std::vector<int> dd(off.size() * 3, 0);
        for (int m = 0; m < 3; ++m)
            for (int par = 0; par < 2; ++par) { g.lo[m][par] = 0; g.hi[m][par] = 0; }
        for (int cls = 0; cls < 64; ++cls) {
            int ac[3] = {cls & 3, (cls >> 2) & 3, cls >> 4};
            if ((ac[0] != 0 && ac[0] != 3) || (ac[1] != 0 && ac[1] != 3) || (ac[2] != 0 && ac[2] != 3)) continue;
            for (int p = cp[cls]; p < cp[cls + 1]; ++p) {
                // off = d0 + Lc d1 + Lc^2 d2 with |dm| <= 2 < Lc / 2: round to the nearest multiple, axis 2 first
                int64_t r = off[p];
                const int64_t L2 = (int64_t)Lc * Lc;
                const int64_t d2 = (r >= 0 ? r + L2 / 2 : r - L2 / 2) / L2;
                r -= d2 * L2;
                const int64_t d1 = (r >= 0 ? r + Lc / 2 : r - Lc / 2) / Lc;
                const int64_t d0 = r - d1 * Lc;
                const int64_t dv[3] = {d0, d1, d2};
                for (int m = 0; m < 3; ++m) {
                    if (dv[m] < -2 || dv[m] > 2) return;
                    const int par = ac[m] == 0 ? 1 : 0;
                    g.lo[m][par] = std::min(g.lo[m][par], (int)dv[m]);
                    g.hi[m][par] = std::max(g.hi[m][par], (int)dv[m]);
                    dd[(size_t)p * 3 + m] = (int)dv[m];
                }
            }
        }
        // staged extents: the largest over the boxes; interior rows must stay inside the lattice
        for (int m = 0; m < 3; ++m) {
            g.e[m] = 0;
            for (int k = 0; k < nb[m]; ++k) {
                const int a0 = 1 + k * bext[m], a1 = std::min(a0 + bext[m], 2 * N);
                const int o = brick_origin(g, kc, m, a0, a1), top = brick_top(g, kc, m, a0, a1);
                g.e[m] = std::max(g.e[m], top - o + 1);
                int lo_used = top;
                for (int par = 0; par < 2; ++par) {
                    int f;
                    if (brick_count(a0, a1, par, f)) lo_used = std::min(lo_used, st_cb(kc, f) + g.lo[m][par]);
                }
                if (lo_used < 0 || top >= Lc) return;
            }
        }
        g.H = kc == 2 ? (g.e[0] + 1) / 2 : 0;
        g.W0 = kc == 2 ? 2 * g.H : g.e[0];
        g.cs = g.W0 * g.e[1] * g.e[2];
        if ((int64_t)g.cs * t.bc * 8 > kBrickSmem) return;
        soff[b].assign(off.size(), 0);
        for (size_t p = 0; p < off.size(); ++p) {
            const int d0 = dd[p * 3], d1 = dd[p * 3 + 1], d2 = dd[p * 3 + 2];
            soff[b][p] = (kc == 2 ? (d0 & 1) * g.H + (d0 >> 1) : d0) + g.W0 * (d1 + g.e[1] * d2);
        }
    }
    for (int b = 0; b < 9; ++b) {
        d.bg[b] = bg[b];
        if (soff[b].empty()) continue;
        d.soff[b].alloc(soff[b].size());
        PORO_CUDA(cudaMemcpyAsync(d.soff[b].p, soff[b].data(), soff[b].size() * 4, cudaMemcpyHostToDevice, c.stream));
    }
    for (int m = 0; m < 3; ++m) { d.nb[m] = nb[m]; d.bext[m] = bext[m]; }
    std::vector<int2> w = class_warps(d, 2, true);
    d.nwbnd = (int)w.size();
    d.wbnd.alloc(w.size());
    if (!w.empty())
        PORO_CUDA(cudaMemcpyAsync(d.wbnd.p, w.data(), w.size() * sizeof(int2), cudaMemcpyHostToDevice, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    brick_smem_attr<SPMV_SET>(kBrickSmem);
    brick_smem_attr<SPMV_SUB>(kBrickSmem);
    brick_smem_attr<SPMV_ADD>(kBrickSmem);
    brick_smem_attr<3>(kBrickSmem);
    brick_smem_attr<4>(kBrickSmem);
    d.brick = 1;
}

void stencil_build_warps(Ctx& c, StencilData& d) {
    for (int kind = 1; kind <= 2; ++kind) {
        std::vector<int2> w = class_warps(d, kind, false);
        d.nwarps[kind - 1] = (int)w.size();
        d.wdesc[kind - 1].alloc(w.size());
        if (!w.empty())
            PORO_CUDA(cudaMemcpyAsync(d.wdesc[kind - 1].p, w.data(), w.size() * sizeof(int2), cudaMemcpyHostToDevice, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
    }
    if (c.opt_i("-poro_stencil_brick", 1)) stencil_build_bricks(c, d);
}

// the launch of `s` takes the brick path: a 3-D P2 row field of a descriptor whose bricks were built
static bool stencil_bricks(const StencilOp& s) { return s.d->brick && s.d->kind[s.fr] == 2 && s.d->bdim[s.fr] == 3; }

static StencilArgs stencil_args(const StencilOp& s, int* smem) {
    const StencilData& d = *s.d;
    StencilArgs a{};
    const int fr = s.fr;
    const bool bricks = stencil_bricks(s);
    *smem = 0;
    for (int fc = 0; fc < 3; ++fc) {
        if (s.fc >= 0 && fc != s.fc) continue;
        const int b = fr * 3 + fc;
        if (!d.present[b]) continue;
        a.t[a.nt] = d.t[b];
        a.xoff[a.nt] = s.fc >= 0 ? 0 : d.row0[fc];
        a.diag_only[a.nt] = d.diag_only[b];
        if (bricks) {
            a.bg[a.nt] = d.bg[b];
            a.soff[a.nt] = d.soff[b].p;
            *smem = std::max(*smem, d.bg[b].cs * d.t[b].bc * 8);
        }
        a.nt++;
    }
    a.bc = d.bc.p ? d.bc.p + d.row0[fr] : nullptr;
    a.unit_diag = s.fc < 0 || s.fc == fr;
    a.diag_xoff = s.fc >= 0 ? 0 : d.row0[fr];
    a.dim = d.dim;
    a.N = d.N;
    a.kr = d.kind[fr];
    a.wdesc = bricks ? d.wbnd.p : d.wdesc[a.kr - 1].p;
    a.nwarps = bricks ? d.nwbnd : d.nwarps[a.kr - 1];
    if (bricks) {
        *smem = std::max(*smem, 3 * d.bext[0] * d.bext[1] * d.bext[2] * 8);      // the box's sums before the epilogue
        a.nbrick = d.nb[0] * d.nb[1] * d.nb[2];
        for (int m = 0; m < 3; ++m) { a.nb[m] = d.nb[m]; a.bext[m] = d.bext[m]; }
    }
    return a;
}

int stencil_grid(const StencilOp& s) {
    const StencilData& d = *s.d;
    if (stencil_bricks(s)) return d.nb[0] * d.nb[1] * d.nb[2] + (int)ceil_div((int64_t)d.nwbnd * 32, kStBlock);
    return ceil_div((int64_t)d.nwarps[d.kind[s.fr] - 1] * 32, kStBlock);
}

template <int MODE>
int stencil_launch(Ctx& c, const StencilOp& s, const double* x, double* y, const Epilogue& ep, double* dot_partial) {
    PORO_REQUIRE(!s.d->slab, "k_stencil: a row-partitioned slab has ghost columns and is applied assembled");
    int smem = 0;
    const StencilArgs a = stencil_args(s, &smem);
    const int grid = stencil_grid(s);
    if (grid == 0) return 0;
    if (a.nbrick) k_stencil_brick<MODE><<<grid, kStBlock, smem, c.stream>>>(a, x, y, ep, dot_partial);
    else switch (s.d->bdim[s.fr]) {
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
