// spmv.cu -- fp64 CSR sparse matrix-vector products (the dominant kernel of the path).
//
// Takes over MatMult_SeqAIJ/MPIAIJ behind `A.mat()` as the KSP operator (lib/Solver.py:95),
// `self.matA * x` (lib/AAR.py:56,135), and the coupling products Mfp_s.mult / Mf_p.mult /
// Ms_f.mult / Ms_p.mult of the block sweeps (lib/Preconditioner.py:180,184,192-193,232).
// The reference's "mult then aypx(-1)" pairs are fused: y = z - A x in one pass.
//
// Primary kernel: "CSR stream".  The rows are packed (once, lazily) into row blocks of at most
// kCap nonzeros.  A CTA of 256 threads streams its block's val/col with perfectly coalesced,
// evict-first loads -- kNt independent loads of each per thread in flight before the first
// dependent gather of x -- writes the products val*x[col] to shared memory, and then sub-warps
// of G lanes reduce each row from shared memory (shuffle tree) and apply the epilogue.  No
// lane is idle on short rows and no row length leaves a warp partially filled in the
// streaming phase, which is what bounds the plain vector-CSR kernel (kept below as the
// fallback for matrices with a row longer than kCap).
// HBM-bound: algorithmic bytes = 12 nnz + 4 (nrows+1) + 8 nrows + 8 ncols.
#include "common.cuh"
#include "spmv_epilogue.cuh"
#include "stencil.cuh"
#include <algorithm>

namespace poro {

static constexpr int kSpmvBlock = 256;
static constexpr int kNt = 8;                       // nonzeros per thread in the streaming phase
static constexpr int kCap = kSpmvBlock * kNt;       // nonzeros per row block (16 KB of products)
static constexpr int kMaxRows = 1024;               // rows per row block (row pointers and row sums live in shared memory)

// ---------------------------------------------------------------------------------------------
// CSR stream
// ---------------------------------------------------------------------------------------------
template <int G, int MODE>
__global__ void __launch_bounds__(kSpmvBlock) k_spmv_stream(const int4* __restrict__ desc, const int* __restrict__ rowptr,
                                                            const int* __restrict__ col, const double* __restrict__ val,
                                                            const double* __restrict__ x, double* __restrict__ y, Epilogue ep,
                                                            double* __restrict__ dot_partial) {
    __shared__ double prod[kCap];
    __shared__ double rsum[kMaxRows];
    __shared__ int rp[kMaxRows + 1];
    __shared__ double red[kSpmvBlock / 32];
    // one 16-byte descriptor per row block {first row, rows, first nonzero, nonzeros}: the matrix loads depend on nothing else
    const int4 dsc = __ldg(desc + blockIdx.x);
    const int r0 = dsc.x, nr = dsc.y, p0 = dsc.z, cnt = dsc.w;
    const int* __restrict__ cb = col + p0;
    const double* __restrict__ vb = val + p0;
    // phase 1: stream the block's nonzeros; all matrix loads are issued before the first gather
    int cidx[kNt];
    double v[kNt];
#pragma unroll
    for (int t = 0; t < kNt; ++t) {
        const int i = threadIdx.x + t * kSpmvBlock;
        cidx[t] = i < cnt ? __ldcs(cb + i) : -1;
        v[t] = i < cnt ? __ldcs(vb + i) : 0.0;
    }
    // the block's slice of the row pointer, coalesced, once (needed after the barrier only)
    for (int i = threadIdx.x; i <= nr; i += kSpmvBlock) rp[i] = rowptr[r0 + i];
    double xv[kNt];
#pragma unroll
    for (int t = 0; t < kNt; ++t) xv[t] = cidx[t] >= 0 ? __ldg(x + cidx[t]) : 0.0;
#pragma unroll
    for (int t = 0; t < kNt; ++t) {
        const int i = threadIdx.x + t * kSpmvBlock;
        if (i < cnt) prod[i] = v[t] * xv[t];
    }
    __syncthreads();
    // phase 2: G lanes per row reduce the products from shared memory into rsum
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1)));
    for (int rl = threadIdx.x / G; rl < nr; rl += kSpmvBlock / G) {
        const int a = rp[rl] - p0, b = rp[rl + 1] - p0;
        double s = 0.0;
        for (int i = a + lane; i < b; i += G) s += prod[i];
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) s += __shfl_down_sync(gmask, s, o, G);
        if (lane == 0) rsum[rl] = s;
    }
    __syncthreads();
    // phase 3: epilogue with consecutive threads on consecutive rows (coalesced, all latencies overlapped)
    double contrib = 0.0;
    for (int rl = threadIdx.x; rl < nr; rl += kSpmvBlock) contrib += apply_epilogue<MODE>(ep, r0 + rl, rsum[rl], x, y);
    if (MODE == 4) {
        double t = block_sum_256(contrib, red);
        if (threadIdx.x == 0) dot_partial[blockIdx.x] = t;
    }
}

// ---------------------------------------------------------------------------------------------
// vector CSR (fallback): L lanes walk one row
// ---------------------------------------------------------------------------------------------
template <int L, int MODE>
__global__ void __launch_bounds__(kSpmvBlock) k_spmv(int nrows, const int* __restrict__ rowptr,
                                                     const int* __restrict__ col, const double* __restrict__ val,
                                                     const double* __restrict__ x, double* __restrict__ y, Epilogue ep,
                                                     double* __restrict__ dot_partial) {
    __shared__ double red[kSpmvBlock / 32];
    const int lane = threadIdx.x & (L - 1);
    const int row = (int)(((int64_t)blockIdx.x * kSpmvBlock + threadIdx.x) / L);
    double sum = 0.0;
    if (row < nrows) {
        const int start = rowptr[row], end = rowptr[row + 1];
        int k = start + lane;
        double s0 = 0.0, s1 = 0.0;
        for (; k + L < end; k += 2 * L) {
            const int c0 = __ldcs(col + k), c1 = __ldcs(col + k + L);
            const double v0 = __ldcs(val + k), v1 = __ldcs(val + k + L);
            s0 = fma(v0, __ldg(x + c0), s0);
            s1 = fma(v1, __ldg(x + c1), s1);
        }
        if (k < end) s0 = fma(__ldcs(val + k), __ldg(x + __ldcs(col + k)), s0);
        sum = s0 + s1;
    }
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, o, L);
    double contrib = 0.0;
    if (row < nrows && lane == 0) contrib = apply_epilogue<MODE>(ep, row, sum, x, y);
    if (MODE == 4) {
        double t = block_sum_256(contrib, red);
        if (threadIdx.x == 0) dot_partial[blockIdx.x] = t;
    }
}

void csr_choose_lanes(Csr& A) {
    double a = A.avg_row();
    A.lanes = a <= 3 ? 2 : a <= 6 ? 4 : a <= 12 ? 8 : a <= 24 ? 16 : 32;
    A.nblk = -1;     // row blocks are (re)built lazily at the first product
}

// packs whole rows into blocks of at most kCap nonzeros (host side, once per matrix)
static void build_row_blocks(Ctx& c, const Csr& A) {
    std::vector<int> rp((size_t)A.nrows + 1);
    PORO_CUDA(cudaMemcpyAsync(rp.data(), A.rowptr.p, rp.size() * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    std::vector<int> blk;
    blk.reserve((size_t)(A.nnz / kCap) * 2 + 16);
    int r = 0;
    bool ok = true;
    while (r < A.nrows) {
        blk.push_back(r);
        int start = r;
        const int limit = rp[r] + kCap;
        // largest r with rp[r] <= limit, but at most 8192 rows per block (keeps phase 2 short for empty rows)
        int hi = (int)(std::upper_bound(rp.begin() + r + 1, rp.end(), limit) - rp.begin()) - 1;
        hi = std::min(hi, start + kMaxRows);
        if (hi <= start) { ok = false; break; }      // a single row exceeds the block capacity
        r = hi;
    }
    blk.push_back(A.nrows);
    if (!ok || A.nrows == 0) { A.nblk = 0; return; }
    A.nblk = (int)blk.size() - 1;
    std::vector<int> dsc((size_t)A.nblk * 4);
    for (int b = 0; b < A.nblk; ++b) {
        dsc[4 * b] = blk[b];
        dsc[4 * b + 1] = blk[b + 1] - blk[b];
        dsc[4 * b + 2] = rp[blk[b]];
        dsc[4 * b + 3] = rp[blk[b + 1]] - rp[blk[b]];
    }
    A.blk_row.alloc(dsc.size());          // holds the descriptors {first row, rows, first nonzero, nonzeros}
    PORO_CUDA(cudaMemcpyAsync(A.blk_row.p, dsc.data(), dsc.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

static void try_bsr(Ctx& c, const Csr& A);

bool csr_ensure_bsr(Ctx& c, const Csr& A) {
    if (A.block_hint > 1 && A.bsr_state < 0 && A.nrows > 0) try_bsr(c, A);
    return A.bsr_state == 1;
}

bool csr_fuse_coupling(Ctx& c, const Csr& A, const Csr& C) {
    if (!csr_ensure_bsr(c, A)) return false;
    return bsr_fuse_coupling(c, *A.bsr, C);
}

void spmv_fused(Ctx& c, const Csr& A, const double* x, const double* x2, double* y, SpmvMode mode, const double* z) {
    PORO_REQUIRE(A.bsr_state == 1 && (A.bsr->t_fused || A.bsr->fused), "spmv_fused: no fused coupling on this matrix");
    Epilogue ep{};
    ep.mode = mode;
    ep.z = z;
    if (mode == SPMV_SET) bsr_launch<SPMV_SET>(c, *A.bsr, x, y, ep, nullptr, x2);
    else if (mode == SPMV_SUB) bsr_launch<SPMV_SUB>(c, *A.bsr, x, y, ep, nullptr, x2);
    else bsr_launch<SPMV_ADD>(c, *A.bsr, x, y, ep, nullptr, x2);
}

static void try_bsr(Ctx& c, const Csr& A) {
    {
        // node-blocked matrix: convert once to BSR unless the blocks are mostly empty (e.g. M (x) I couplings)
        auto B = std::make_shared<Bsr>();
        int BS = A.block_hint % 3 == 0 ? 3 : (A.block_hint % 2 == 0 ? 2 : 0);
        // break-even on bytes is a fill ratio of 12 / 8.44 = 1.42; below it BSR also wins on gather traffic
        if (BS && c.opt_i("-poro_use_bsr", 1) && bsr_from_csr(c, A, BS, *B, c.opt_d("-poro_bsr_max_fill", 1.42))) {
            A.bsr = B;
            A.bsr_state = 1;
        } else A.bsr_state = 0;
        if (c.has_opt("-poro_verbose"))
            fprintf(stderr, "    [spmv] %d x %d nnz=%lld hint=%d -> %s%s\n", A.nrows, A.ncols, (long long)A.nnz, A.block_hint,
                    A.bsr_state == 1 ? "BSR" : "CSR", A.bsr_state == 1 && A.bsr->t_ok ? " (TMA chunks)" : "");
    }
}

template <int MODE>
static int launch_spmv(Ctx& c, const Csr& A, const double* x, double* y, const Epilogue& ep, double* dot_partial) {
    if (A.nrows == 0) return 0;
    // a generated block along whole fields: apply its class tables (stencil.cu) instead of streaming the assembled matrix
    if (stencil_runs(A)) return stencil_launch<MODE>(c, *A.stencil, x, y, ep, dot_partial);
    if (A.block_hint > 1 && A.bsr_state < 0) try_bsr(c, A);
    if (A.bsr_state == 1) return bsr_launch<MODE>(c, *A.bsr, x, y, ep, dot_partial);
    if (A.nblk < 0) build_row_blocks(c, A);
    int grid;
    if (A.nblk > 0) {
        grid = A.nblk;
        const int G = row_group_lanes(A.avg_row());
#define GO(GG) k_spmv_stream<GG, MODE><<<grid, kSpmvBlock, 0, c.stream>>>(reinterpret_cast<const int4*>(A.blk_row.p), A.rowptr.p, A.col.p, A.val.p, x, y, ep, dot_partial)
        switch (G) {
            case 1: GO(1); break;
            case 2: GO(2); break;
            case 4: GO(4); break;
            case 8: GO(8); break;
            case 16: GO(16); break;
            default: GO(32); break;
        }
#undef GO
    } else {
        const int L = A.lanes ? A.lanes : 32;
        grid = ceil_div((int64_t)A.nrows * L, kSpmvBlock);
#define GO(LL) k_spmv<LL, MODE><<<grid, kSpmvBlock, 0, c.stream>>>(A.nrows, A.rowptr.p, A.col.p, A.val.p, x, y, ep, dot_partial)
        switch (L) {
            case 2: GO(2); break;
            case 4: GO(4); break;
            case 8: GO(8); break;
            case 16: GO(16); break;
            default: GO(32); break;
        }
#undef GO
    }
    PORO_LAUNCH_CHECK(c);
    return grid;
}

void spmv_kernel_info(Ctx& c, const Csr& A, int64_t* v) {
    std::fill(v, v + kSpmvInfoFields, (int64_t)0);
    v[7] = -1;
    if (stencil_runs(A)) { v[0] = 4; return; }
    if (A.nrows > 0 && csr_ensure_bsr(c, A)) {
        const Bsr& B = *A.bsr;
        const bool plain = !B.t_ok;
        v[0] = B.diag_only ? 2 : 1;
        v[1] = row_group_lanes(B.nbrows ? (double)B.nnzb / B.nbrows : 0.0);
        v[2] = B.bs;
        v[3] = plain && B.pref;
        v[4] = plain && B.coop && !B.fp32;      // bsr_launch has no cooperative variant for fp32 values
        v[5] = B.fp32;
        v[6] = B.t_ok;
        v[7] = B.t_ok ? B.t_cfg : -1;
        v[8] = B.t_ok ? B.t_fused : B.fused;
        v[9] = B.t_ok ? B.t_nchunk : B.nblk;
        v[10] = plain && B.pf_groups > 0;
        return;
    }
    if (A.nrows > 0 && A.nblk < 0) build_row_blocks(c, A);
    if (A.nrows == 0 || A.nblk > 0) {
        v[1] = row_group_lanes(A.avg_row());
        v[9] = std::max(A.nblk, 0);
    } else {
        v[0] = 5;
        v[1] = A.lanes ? A.lanes : 32;
    }
}

void spmv(Ctx& c, const Csr& A, const double* x, double* y, SpmvMode mode, const double* z) {
    Epilogue ep{};
    ep.mode = mode;
    ep.z = z;
    if (mode == SPMV_SET) launch_spmv<SPMV_SET>(c, A, x, y, ep, nullptr);
    else if (mode == SPMV_SUB) launch_spmv<SPMV_SUB>(c, A, x, y, ep, nullptr);
    else launch_spmv<SPMV_ADD>(c, A, x, y, ep, nullptr);
}

void spmv_cheb_step(Ctx& c, const Csr& A, const double* x_in, const double* d_old, double* d_new, double* r, double* x,
                    const double* dinv, double c1, double c2) {
    Epilogue ep{};
    ep.mode = 3;
    ep.d_old = d_old; ep.d_new = d_new; ep.r = r; ep.xv = x; ep.dinv = dinv; ep.c1 = c1; ep.c2 = c2;
    launch_spmv<3>(c, A, x_in, nullptr, ep, nullptr);      // x_in = d_old, or its [owned | halo] extension
}

__global__ void k_sum_to(const double* __restrict__ partial, int n, double* __restrict__ out) {
    __shared__ double sm[8];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) s += partial[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sm[w];
        *out = t;
    }
}

void spmv_dot(Ctx& c, const Csr& A, const double* p, double* w, double* d_dot) {
    Epilogue ep{};
    ep.mode = 4;
    const bool st = stencil_runs(A);
    if (!st && A.nblk < 0) build_row_blocks(c, A);
    const int L = A.lanes ? A.lanes : 32;
    const int64_t grid = st ? stencil_grid(*A.stencil)
                            : A.nblk > 0 ? A.nblk : ceil_div((int64_t)A.nrows * L, kSpmvBlock);   // upper bound for BSR too
    if (grid <= Ctx::kScal) {
        int g = launch_spmv<4>(c, A, p, w, ep, c.d_scal);
        k_sum_to<<<1, 256, 0, c.stream>>>(c.d_scal, g, d_dot);
        PORO_LAUNCH_CHECK(c);
    } else {
        launch_spmv<SPMV_SET>(c, A, p, w, ep, nullptr);
        const double* xs[1] = {p};
        const double* ys[1] = {w};
        vec_dots(c, 1, xs, ys, A.nrows, d_dot);
    }
}

}  // namespace poro
