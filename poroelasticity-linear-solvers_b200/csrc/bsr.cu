// bsr.cu -- block-CSR (BS x BS, BS = 2 or 3) SpMV for the node-blocked vector fields.
//
// The displacement and fluid-velocity blocks (A_ss, A_ff, P_ss, P_ff) and every level of their
// AMG hierarchies (prolongators included) consist of dense BS x BS node blocks.  Storing them
// as BSR cuts the matrix stream from 12 to (8 BS^2 + 4) / BS^2 = 8.44 bytes per nonzero (BS = 3)
// and -- what the ncu profile of the CSR kernel showed to be the real limiter (L1TEX wavefronts
// of the x gathers, profiles/r1_spmv_stream_csr.md) -- replaces 9 scattered 8-byte gathers by
// three loads of one contiguous 24-byte node vector.
//
// Layout: values are interleaved in groups of 32 blocks, val[((p / 32) * BS^2 + e) * 32 + p % 32]
// for entry e of block p, so that "one thread per block" reads every entry fully coalesced.
// Kernel: a CTA streams up to 256 * kNtb blocks of whole block rows (thread per block, kNtb blocks per
// thread in flight), writes BS partial sums per block to shared memory, then G lanes per block
// row reduce them and apply the same epilogues as the CSR kernel (y = Ax, z - Ax, z + Ax, fused
// Chebyshev step, fused p.Ap).
// Algorithmic bytes: (8 BS^2 + 4) nnzb + 4 (nbrows + 1) + 8 BS nbrows + 8 BS nbcols.
#include "common.cuh"
#include "spmv_epilogue.cuh"
#include <algorithm>

namespace poro {

static constexpr int kBlk = 256;
static constexpr int kMaxBRows = 256;     // block rows per chunk (row pointers and row sums live in shared memory)

// PREF: the chunk has at most kBlk scalar rows, so every thread owns at most one epilogue row and loads its operands
//       (z, or r / d / D^-1 / x of the Chebyshev step) at kernel START: they arrive while the blocks are streamed and
//       multiplied instead of trailing the CTA (the tail that cost the Chebyshev-step launches 0.160 vs 0.135 ms).
// FUSE: a mass coupling c M (x) I with the same block pattern rides along (one scalar per block in `mval`, a 3-bit row mask
//       in the top bits of the column word): y = A x + C x2 in one pass.
// VT: storage type of the matrix values (double; float for the opt-in fp32 storage of preconditioner matrices -- every value
//     is converted on load, all arithmetic and all vectors stay fp64)
// L2 prefetch (pf.groups > 0): the kernel is bound by its exposed DRAM latencies, not by a pipe (ncu: LSU 21 %, L1 wavefronts
//     55 %, issue 24 %; storing the values in fp32 moved 43 % fewer bytes in the SAME time).  One lane per CTA therefore asks
//     the TMA unit to pull the value / column / operand ranges of the chunk `pf.groups` groups further down the stream into
//     L2 (cp.async.bulk.prefetch.L2): consecutive chunks tile the arrays, so the shifted ranges tile them too, and by the
//     time that chunk's CTA is scheduled its loads are L2 hits.
struct BsrPrefetch {
    int groups;       // distance in groups of 32 blocks
    int ngroups;      // groups in the matrix (clip)
    int rows;         // distance in scalar rows
    int nrows;        // scalar rows (clip)
};
__device__ __forceinline__ void l2_prefetch(const void* p, unsigned bytes, bool evict_first = false) {
    if (evict_first) {
        // the matrix stream must not displace the gathered vectors from L2 (the demand loads are ld.global.cs for the same reason)
        unsigned long long pol;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
        asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(p), "r"(bytes), "l"(pol) : "memory");
    } else {
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
    }
}
// [lo, hi) in elements of `esz` bytes, widened to 16-byte boundaries (the arrays are allocated in 256-byte units)
__device__ __forceinline__ void l2_prefetch_range(const void* base, long long lo, long long hi, int esz, bool evict_first = false) {
    const unsigned long long a = ((unsigned long long)base + (unsigned long long)lo * esz) & ~15ull;
    const unsigned long long b = ((unsigned long long)base + (unsigned long long)hi * esz + 15ull) & ~15ull;
    if (b > a) l2_prefetch((const void*)a, (unsigned)(b - a), evict_first);
}
// COOP: the 32 x BS doubles of x a warp needs are gathered by (block, component) pairs laid out lane-contiguously -- lane l of
//     load k fetches component (32k + l) % BS of block (32k + l) / BS -- and handed to their owners through the warp's own
//     slice of `part`.  Thread-per-block gathers touch up to 32 nodes (~12 cache lines) per load instruction, and the L1
//     wavefront queue, not DRAM, is what the kernel saturates (ncu: 176 k wavefronts per SM in 313 k cycles at ~2 cycles per
//     replayed wavefront); the cooperative form touches 32 / BS nodes per instruction.
template <int BS, int MODE, bool DIAG, bool PREF, bool FUSE, typename VT = double, bool COOP = false>
__global__ void __launch_bounds__(kBlk, FUSE ? 3 : 4) k_bsr_stream(const int4* __restrict__ desc, const int* __restrict__ rowptr,
                                                     const int* __restrict__ col, const VT* __restrict__ val,
                                                     const double* __restrict__ mval, const double* __restrict__ x,
                                                     const double* __restrict__ x2, double* __restrict__ y, Epilogue ep,
                                                     double* __restrict__ dot_partial, int G, BsrPrefetch pf) {
    constexpr int kNtb = 2;
    __shared__ double part[kBlk * kNtb * BS];
    __shared__ double part2[(COOP && FUSE) ? kBlk * kNtb * BS : 1];
    __shared__ double eop[(COOP && PREF && MODE == 3) ? 2 * kBlk : 1];      // D^-1 and x of the Chebyshev step wait here, not in registers
    __shared__ double rsum[kMaxBRows * BS];
    __shared__ int rp[kMaxBRows + 1];
    __shared__ double red[kBlk / 32];
    // one 16-byte descriptor per chunk {first block row, block rows, first block, blocks}: the matrix loads below depend on
    // nothing else (the row pointers are only needed for the reduction and are fetched behind them)
    const int4 dsc = __ldg(desc + blockIdx.x);
    const int R0 = dsc.x, nbr = dsc.y, p0 = dsc.z, cnt = dsc.w;
    // epilogue operands of this thread's row, requested before anything else
    const bool has_row = PREF && (int)threadIdx.x < nbr * BS;
    const int myrow = R0 * BS + threadIdx.x;
    double e0 = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;
    if (has_row) {
        if (MODE == SPMV_SUB || MODE == SPMV_ADD) e0 = ep.z[myrow];
        else if (MODE == 3 && COOP) {
            e0 = ep.r[myrow]; e1 = ep.d_old[myrow];
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(eop + threadIdx.x)), "l"(ep.dinv + myrow) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(eop + kBlk + threadIdx.x)), "l"(ep.xv + myrow) : "memory");
        }
        else if (MODE == 3) { e0 = ep.r[myrow]; e1 = ep.d_old[myrow]; e2 = ep.dinv[myrow]; e3 = ep.xv[myrow]; }
        else if (MODE == 4) e0 = x[myrow];
    }
    if (pf.groups > 0 && threadIdx.x == kBlk - 32) {
        constexpr int NEs = DIAG ? BS : BS * BS;
        const int g0 = (p0 >> 5) + pf.groups, g1 = min(((p0 + cnt) >> 5) + pf.groups, pf.ngroups);
        if (g1 > g0) {
            l2_prefetch(val + (size_t)g0 * NEs * 32, (unsigned)((g1 - g0) * NEs * 32 * (int)sizeof(VT)), true);
            l2_prefetch_range(col, (long long)g0 * 32, (long long)g1 * 32, 4, true);
            if (FUSE) l2_prefetch_range(mval, (long long)g0 * 32, (long long)g1 * 32, 8, true);
        }
        if (PREF && MODE != SPMV_SET) {
            const long long r0 = (long long)R0 * BS + pf.rows, r1 = min((long long)(R0 + nbr) * BS + pf.rows, (long long)pf.nrows);
            if (r1 > r0) {
                if (MODE == SPMV_SUB || MODE == SPMV_ADD) l2_prefetch_range(ep.z, r0, r1, 8);
                else if (MODE == 3) {
                    l2_prefetch_range(ep.r, r0, r1, 8);
                    l2_prefetch_range(ep.d_old, r0, r1, 8);
                    l2_prefetch_range(ep.dinv, r0, r1, 8);
                    l2_prefetch_range(ep.xv, r0, r1, 8);
                }
            }
        }
    }
    // phase 1: one thread per block
    int c[kNtb];
    unsigned mk[kNtb];
    double m[kNtb];
#pragma unroll
    for (int t = 0; t < kNtb; ++t) {
        const int i = threadIdx.x + t * kBlk;
        c[t] = -1;
        mk[t] = 0u;
        m[t] = 0.0;
        if (i < cnt) {
            const int cw = __ldcs(col + p0 + i);          // FUSE: the top three bits carry the row mask (the word may be negative)
            c[t] = FUSE ? (cw & 0x1fffffff) : cw;
            if (FUSE) { mk[t] = (unsigned)cw >> 29; m[t] = __ldcs(mval + p0 + i); }
        }
    }
    constexpr int NE = DIAG ? BS : BS * BS;     // stored entries per block
    double v[kNtb][NE];
#pragma unroll
    for (int t = 0; t < kNtb; ++t) {
        const int p = p0 + threadIdx.x + t * kBlk;
        const VT* vb = val + ((size_t)(p >> 5) * NE) * 32 + (p & 31);
#pragma unroll
        for (int e = 0; e < NE; ++e) v[t][e] = c[t] >= 0 ? (double)__ldcs(vb + e * 32) : 0.0;
    }
    for (int i = threadIdx.x; i <= nbr; i += kBlk) rp[i] = rowptr[R0 + i];     // needed after the barrier only
    if (COOP) {
        const int ln = threadIdx.x & 31;
        // global -> shared without a register stop (LDGSTS): all kNtb * BS gathers of the warp are in flight at once and cost
        // no registers; a source size of 0 zero-fills the slots of absent blocks
#pragma unroll
        for (int t = 0; t < kNtb; ++t) {
            double* st = part + ((threadIdx.x & ~31) + t * kBlk) * BS;       // this warp's slice for its blocks of round t
            double* st2 = part2 + ((COOP && FUSE) ? ((threadIdx.x & ~31) + t * kBlk) * BS : 0);
#pragma unroll
            for (int k = 0; k < BS; ++k) {
                const int q = 32 * k + ln;
                const int bsrc = q / BS, j = q - bsrc * BS;
                const int cc = __shfl_sync(0xffffffffu, c[t], bsrc);
                const size_t off = cc >= 0 ? (size_t)cc * BS + j : 0;
                const unsigned sz = cc >= 0 ? 8u : 0u;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"((unsigned)__cvta_generic_to_shared(st + q)), "l"(x + off), "r"(sz) : "memory");
                if (FUSE)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"((unsigned)__cvta_generic_to_shared(st2 + q)), "l"(x2 + off), "r"(sz) : "memory");
            }
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncwarp();
        // each thread reads and then overwrites below only the BS slots of its own blocks
    }
#pragma unroll
    for (int t = 0; t < kNtb; ++t) {
        const int i = threadIdx.x + t * kBlk;
        if (c[t] >= 0) {
            double xv[BS], x2v[BS];
            if (COOP) {
#pragma unroll
                for (int j = 0; j < BS; ++j) { xv[j] = part[i * BS + j]; if (FUSE) x2v[j] = part2[i * BS + j]; }
            } else {
#pragma unroll
                for (int j = 0; j < BS; ++j) xv[j] = __ldg(x + (size_t)c[t] * BS + j);
                if (FUSE) {
#pragma unroll
                    for (int j = 0; j < BS; ++j) x2v[j] = __ldg(x2 + (size_t)c[t] * BS + j);
                }
            }
#pragma unroll
            for (int k = 0; k < BS; ++k) {
                double s = 0.0;
                if (DIAG) s = v[t][k] * xv[k];
                else {
#pragma unroll
                    for (int j = 0; j < BS; ++j) s = fma(v[t][DIAG ? 0 : k * BS + j], xv[j], s);
                }
                if (FUSE && ((mk[t] >> k) & 1u)) s = fma(m[t], x2v[k], s);
                part[i * BS + k] = s;
            }
        }
    }
    __syncthreads();
    // phase 2: G lanes per block row reduce the partial sums into rsum
    const int lg = 31 - __clz(G);           // G is a power of two
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1)));
    for (int Rl = threadIdx.x >> lg; Rl < nbr; Rl += kBlk >> lg) {
        const int a = rp[Rl] - p0, b = rp[Rl + 1] - p0;
        double s[BS];
#pragma unroll
        for (int k = 0; k < BS; ++k) s[k] = 0.0;
        for (int i = a + lane; i < b; i += G) {
#pragma unroll
            for (int k = 0; k < BS; ++k) s[k] += part[i * BS + k];
        }
#pragma unroll
        for (int k = 0; k < BS; ++k) {
            for (int o = G >> 1; o > 0; o >>= 1) s[k] += __shfl_down_sync(gmask, s[k], o, G);
        }
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < BS; ++k) rsum[Rl * BS + k] = s[k];
        }
    }
    __syncthreads();
    // phase 3: coalesced epilogue over the scalar rows of the chunk
    double contrib = 0.0;
    if (PREF) {
        if (has_row) {
            const double sum = rsum[threadIdx.x];
            if (MODE == SPMV_SET) y[myrow] = sum;
            else if (MODE == SPMV_SUB) y[myrow] = e0 - sum;
            else if (MODE == SPMV_ADD) y[myrow] = e0 + sum;
            else if (MODE == 3) {
                if (COOP) { e2 = eop[threadIdx.x]; e3 = eop[kBlk + threadIdx.x]; }      // own slots, completed by cp.async.wait_all above
                const double rn = e0 - sum;
                const double dn = ep.c1 * e1 + ep.c2 * e2 * rn;
                ep.r[myrow] = rn;
                ep.d_new[myrow] = dn;
                ep.xv[myrow] = e3 + dn;
            } else {
                y[myrow] = sum;
                contrib = sum * e0;
            }
        }
    } else {
        for (int rl = threadIdx.x; rl < nbr * BS; rl += kBlk) contrib += apply_epilogue<MODE>(ep, R0 * BS + rl, rsum[rl], x, y);
    }
    if (MODE == 4) {
        double t = block_sum_256(contrib, red);
        if (threadIdx.x == 0) dot_partial[blockIdx.x] = t;
    }
}

// ---------------------------------------------------------------------------------------------
// conversion CSR -> BSR on the device
// ---------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(256) k_for3(int64_t n, F f) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) f(i);
}
template <class F>
static void pfor(Ctx& c, int64_t n, F f) {
    if (n <= 0) return;
    int64_t g = (n + 255) / 256;
    int64_t cap = (int64_t)c.sm_count * 16;
    k_for3<<<(int)(g < cap ? g : cap), 256, 0, c.stream>>>(n, f);
    PORO_LAUNCH_CHECK(c);
}

bool bsr_from_csr(Ctx& c, const Csr& A, int BS, Bsr& out, double max_fill) {
    if (BS < 2 || BS > 3 || A.nrows % BS || A.ncols % BS || A.nnz == 0) return false;
    const int nbr = A.nrows / BS, nbc = A.ncols / BS;
    Csr Nb;
    {
        DBuf<uint64_t> keys((size_t)A.nnz);
        DBuf<double> vals((size_t)A.nnz);
        const int* rp = A.rowptr.p; const int* cc = A.col.p;
        uint64_t* kk = keys.p; double* vv = vals.p;
        pfor(c, A.nrows, [=] __device__(int64_t i) {
            for (int k = rp[i]; k < rp[i + 1]; ++k) {
                kk[k] = ((uint64_t)(uint32_t)((int)i / BS) << 32) | (uint32_t)(cc[k] / BS);
                vv[k] = 1.0;
            }
        });
        coo_to_csr(c, nbr, nbc, A.nnz, keys, vals, Nb, COMBINE_SUM);
    }
    const int64_t nnzb = Nb.nnz;
    // blocks with entries only on their diagonal (scalar matrix (x) I, rows possibly zeroed by BCs)?
    DBuf<int> offd(1);
    offd.zero(c.stream);
    {
        const int* rp = A.rowptr.p; const int* cc = A.col.p; int* od = offd.p;
        pfor(c, A.nrows, [=] __device__(int64_t i) {
            int n = 0;
            for (int k = rp[i]; k < rp[i + 1]; ++k) n += ((int)i % BS) != (cc[k] % BS);
            if (n) atomicAdd(od, n);
        });
    }
    int h_offd = 0;
    PORO_CUDA(cudaMemcpyAsync(&h_offd, offd.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    const bool diag = h_offd == 0;
    const int NE = diag ? BS : BS * BS;
    // byte break-even against CSR (12 B / nonzero): (8 NE + 4) nnzb <= max_fill-scaled budget
    if ((double)nnzb * (8.0 * NE + 4.0) > max_fill * 8.44 * (double)A.nnz) return false;
    out.bs = BS; out.nbrows = nbr; out.nbcols = nbc; out.nnzb = nnzb; out.diag_only = diag;
    out.rowptr = std::move(Nb.rowptr);
    out.col = std::move(Nb.col);
    const size_t ngroups = (size_t)((nnzb + 31) / 32);
    out.val.alloc(ngroups * 32 * NE);
    out.val.zero(c.stream);
    {
        const int* rp = A.rowptr.p; const int* cc = A.col.p; const double* av = A.val.p;
        const int* brp = out.rowptr.p; const int* bcc = out.col.p;
        double* bv = out.val.p;
        pfor(c, A.nrows, [=] __device__(int64_t i) {
            const int I = (int)i / BS, ri = (int)i % BS;
            const int b0 = brp[I], b1 = brp[I + 1];
            for (int k = rp[i]; k < rp[i + 1]; ++k) {
                const int J = cc[k] / BS, rj = cc[k] % BS;
                int lo = b0, hi = b1;
                while (lo < hi) { int mid = (lo + hi) >> 1; if (bcc[mid] < J) lo = mid + 1; else hi = mid; }
                const size_t p = (size_t)lo;
                // summed: an uploaded CSR may repeat an entry, and the CSR kernels add every copy
                bv[((p >> 5) * NE + (size_t)(diag ? ri : ri * BS + rj)) * 32 + (p & 31)] += av[k];
            }
        });
    }
    // pack whole block rows into chunks of at most 256 * ntb blocks
    std::vector<int> rp((size_t)nbr + 1);
    PORO_CUDA(cudaMemcpyAsync(rp.data(), out.rowptr.p, rp.size() * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    int max_row = 0;
    for (int i = 0; i < nbr; ++i) max_row = std::max(max_row, rp[i + 1] - rp[i]);
    // dense blocks: one block per thread keeps 7 CTAs per SM resident; long block rows (coarse levels) need two
    // measured on B200 (profiles/r1_spmv_kernels.md): 2 blocks per thread beats 1 (0.126 vs 0.140 ms on A_ss) and,
    // for diagonal blocks, 4 (0.086 vs 0.105 ms on A_sf)
    out.ntb = 2;
    (void)max_row;
    // long block rows (the field blocks and their AMG levels): at most kBlk scalar rows per chunk, so that every thread owns
    // one epilogue row and can request its operands up front (PREF); short rows (transfer operators) keep the wide chunks
    const bool pref = (double)nnzb >= 6.0 * nbr && c.opt_i("-poro_bsr_prefetch", 1) != 0;
    const int max_rows = pref ? kBlk / BS : kMaxBRows;
    out.pref = pref;
    out.coop = c.opt_i("-poro_bsr_coop_gather", 0) != 0;
    {
        // L2 prefetch distance in chunks (0 = off): further than the 4 x SM-count resident CTAs, short of what L2 holds
        const int64_t chunks = c.opt_i("-poro_bsr_l2_prefetch_chunks", 0);
        const int64_t total_chunks = (nnzb + kBlk * out.ntb - 1) / (kBlk * out.ntb);
        if (chunks > 0 && total_chunks > 2 * chunks) {
            out.pf_groups = (int)(chunks * (kBlk * out.ntb / 32));
            out.pf_rows = (int)((double)chunks * kBlk * out.ntb * nbr * BS / (double)nnzb) & ~1;
        }
    }
    std::vector<int> blk;
    int r = 0;
    while (r < nbr) {
        blk.push_back(r);
        const int limit = rp[r] + kBlk * out.ntb;
        int hi = (int)(std::upper_bound(rp.begin() + r + 1, rp.end(), limit) - rp.begin()) - 1;
        hi = std::min(hi, r + max_rows);
        if (hi <= r) return false;                 // one block row longer than a chunk
        r = hi;
    }
    blk.push_back(nbr);
    out.nblk = (int)blk.size() - 1;
    out.blk_row.alloc(blk.size());
    PORO_CUDA(cudaMemcpyAsync(out.blk_row.p, blk.data(), blk.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    {
        std::vector<int> dsc((size_t)out.nblk * 4);
        for (int b = 0; b < out.nblk; ++b) {
            dsc[4 * b] = blk[b];
            dsc[4 * b + 1] = blk[b + 1] - blk[b];
            dsc[4 * b + 2] = rp[blk[b]];
            dsc[4 * b + 3] = rp[blk[b + 1]] - rp[blk[b]];
        }
        out.blk_desc.alloc(dsc.size());
        PORO_CUDA(cudaMemcpyAsync(out.blk_desc.p, dsc.data(), dsc.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    if (A.fp32_hint) {
        // opt-in fp32 storage: 4 NE + 4 instead of 8 NE + 4 bytes per block; converted once, the fp64 copy is dropped
        const size_t nv = out.val.n;
        out.val32.alloc(nv);
        const double* src = out.val.p; float* dst = out.val32.p;
        pfor(c, (int64_t)nv, [=] __device__(int64_t i) { dst[i] = (float)src[i]; });
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        out.val.release();
        out.fp32 = true;
        return true;
    }
    // Blackwell path: chunked layout for the persistent TMA kernel; the plain arrays are only kept when it is unavailable
    if (c.opt_i("-poro_bsr_tma", 0) && bsr_build_tma(c, out, rp)) {
        out.val.release();
        out.col.release();
    }
    return true;
}

// ---------------------------------------------------------------------------------------------
// fused mass coupling on the plain layout: one scalar per block + 3-bit row mask in the column word
// ---------------------------------------------------------------------------------------------
static bool bsr_fuse_coupling_plain(Ctx& c, Bsr& B, const Csr& C) {
    if (B.diag_only || C.nrows != B.nbrows * B.bs || C.ncols != B.nbcols * B.bs || (int64_t)B.nbcols >= (1 << 29)) return false;
    const int BS = B.bs;
    DBuf<double> fm((size_t)B.nnzb);
    DBuf<int> fcol((size_t)B.nnzb);
    DBuf<unsigned long long> counters(2);      // [0] coupling entries matched, [1] violations of the c M_IJ I x mask form
    counters.zero(c.stream);
    {
        const int* brp = B.rowptr.p; const int* bc = B.col.p; int* oc = fcol.p; double* om = fm.p;
        const int* crp = C.rowptr.p; const int* ccol = C.col.p; const double* cv = C.val.p;
        unsigned long long* cnts = counters.p;
        pfor(c, (int64_t)B.nbrows * 32, [=] __device__(int64_t gt) {
            const int I = (int)(gt >> 5), ln = (int)(gt & 31);
            unsigned long long matched = 0, bad = 0;
            for (int p = brp[I] + ln; p < brp[I + 1]; p += 32) {
                const int J = bc[p];
                double m = 0.0;
                unsigned mask = 0u;
                for (int q = 0; q < BS; ++q) {
                    const int row = I * BS + q, want = J * BS + q;
                    int lo = crp[row], hi = crp[row + 1];
                    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ccol[mid] < want) lo = mid + 1; else hi = mid; }
                    if (lo < crp[row + 1] && ccol[lo] == want) {
                        const double v = cv[lo];
                        matched++;
                        if (v != 0.0) {
                            if (mask == 0u) m = v;
                            else if (v != m) bad++;
                            mask |= 1u << q;
                        }
                    }
                }
                om[p] = m;
                oc[p] = J | (int)(mask << 29);
            }
            if (matched) atomicAdd(cnts, matched);
            if (bad) atomicAdd(cnts + 1, bad);
        });
    }
    unsigned long long h[2] = {0, 0};
    PORO_CUDA(cudaMemcpyAsync(h, counters.p, sizeof h, cudaMemcpyDeviceToHost, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    if (h[1] != 0 || (int64_t)h[0] != C.nnz) return false;
    B.f_m = std::move(fm);
    B.f_col = std::move(fcol);
    B.fused = true;
    return true;
}

bool bsr_fuse_coupling(Ctx& c, Bsr& B, const Csr& C) {
    if (B.fp32) return false;          // the fused kernels read the fp64 values, which fp32 storage released
    return B.t_ok ? bsr_fuse_coupling_tma(c, B, C) : bsr_fuse_coupling_plain(c, B, C);
}

template <int MODE>
int bsr_launch(Ctx& c, const Bsr& B, const double* x, double* y, const Epilogue& ep, double* dot_partial, const double* x2) {
    if (B.t_ok) return bsr_tma_launch<MODE>(c, B, x, y, ep, dot_partial, x2);
    const int G = row_group_lanes(B.nbrows ? (double)B.nnzb / B.nbrows : 0.0);
    const bool fuse = x2 != nullptr && B.fused;
    const BsrPrefetch pf{B.pf_groups, (int)(B.nnzb >> 5), B.pf_rows, B.nbrows * B.bs};
#define GO(BSS, DG, PF, FS)                                                                                                     \
    do {                                                                                                                       \
        if (B.coop && !B.fp32)                                                                                                 \
            k_bsr_stream<BSS, MODE, DG, PF, FS, double, true><<<B.nblk, kBlk, 0, c.stream>>>(reinterpret_cast<const int4*>(B.blk_desc.p), B.rowptr.p, FS ? B.f_col.p : B.col.p, \
                                B.val.p, FS ? B.f_m.p : nullptr, x, x2, y, ep, dot_partial, G, pf);                             \
        else if (B.fp32 && !FS)                                                                                                \
            k_bsr_stream<BSS, MODE, DG, PF, false, float><<<B.nblk, kBlk, 0, c.stream>>>(reinterpret_cast<const int4*>(B.blk_desc.p), B.rowptr.p, \
                                B.col.p, B.val32.p, nullptr, x, x2, y, ep, dot_partial, G, pf);                                     \
        else                                                                                                                   \
            k_bsr_stream<BSS, MODE, DG, PF, FS><<<B.nblk, kBlk, 0, c.stream>>>(reinterpret_cast<const int4*>(B.blk_desc.p), B.rowptr.p, FS ? B.f_col.p : B.col.p, \
                                B.val.p, FS ? B.f_m.p : nullptr, x, x2, y, ep, dot_partial, G, pf);                                 \
    } while (0)
#define GOB(BSS)                                                                                   \
    do {                                                                                           \
        if (fuse) { if (B.pref) GO(BSS, false, true, true); else GO(BSS, false, false, true); }     \
        else if (B.diag_only) { if (B.pref) GO(BSS, true, true, false); else GO(BSS, true, false, false); } \
        else { if (B.pref) GO(BSS, false, true, false); else GO(BSS, false, false, false); }        \
    } while (0)
    if (B.bs == 3) GOB(3); else GOB(2);
#undef GOB
#undef GO
    PORO_LAUNCH_CHECK(c);
    return B.nblk;
}

template int bsr_launch<0>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_launch<1>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_launch<2>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_launch<3>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_launch<4>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);

}  // namespace poro
