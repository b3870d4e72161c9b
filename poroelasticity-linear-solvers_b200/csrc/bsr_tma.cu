// bsr_tma.cu -- Blackwell-native block-CSR SpMV: persistent CTAs fed by 1-D TMA bulk copies (cp.async.bulk + mbarrier).
//
// Same products as bsr.cu (A_ss, A_ff, P_ss, P_ff, the AMG levels of the vector fields, the M (x) I mass couplings), but
// the matrix streams no longer pass through the register file and L1TEX (the unit ncu showed saturated for the
// `ld.global.cs` kernel, profiles/r1_spmv_kernels.md): one elected thread per CTA posts bulk copies of the next chunk's
// values, block columns and row pointers into a 2-stage shared-memory ring and arms an mbarrier with the byte count; the
// 256 threads only gather x, multiply out of shared memory, reduce rows and run the epilogue -- while the TMA engine is
// already streaming the following chunk.  L1TEX carries nothing but the x gathers and the epilogue operands, which are
// loaded into registers at the START of a chunk (one scalar row per thread), so the Chebyshev-step epilogue
// (r, d, D^-1, x read; r, d, x written) overlaps the stream instead of trailing it.
//
// Layout ("chunked BSR"): whole block rows are packed into chunks of <= 512 blocks / <= 64 block rows; each chunk's
// blocks start at a multiple of 32 in the padded block index space so that its slice of the 32-interleaved value array
// val[((q / 32) * NE + e) * 32 + q % 32], its columns col[q] and its local row pointers are three contiguous,
// 16-byte-aligned byte ranges -- what cp.async.bulk needs.  Padding blocks carry value 0 / column 0.
// Fused coupling (FUSE): the outer operator's mass couplings A_sf, A_fs = c M (x) I have the block pattern of A_ss / A_ff;
// they ride along as ONE scalar per block plus a 3-bit row mask in the top bits of the column word (Dirichlet rows of the
// coupling are zero): y_s = A_ss x_s + (c M (x) I) x_f in a single pass, 84 instead of 76 + 28 bytes per block.
// Algorithmic bytes are those of bsr.cu; the padding adds about 1-2 % of traffic.
#include "common.cuh"
#include "spmv_epilogue.cuh"
#include <algorithm>

namespace poro {

namespace {

constexpr int kT = 256;        // threads per CTA
constexpr int kMaxR = 64;      // block rows per chunk (<= kT / 3 scalar rows: one epilogue row per thread)
// pipeline shapes (blocks per chunk, ring stages, resident CTAs per SM); the layout is built for one of them
// (-poro_bsr_tma_cfg): 0 = 512 / 2 / 2, 1 = 256 / 2 / 4, 2 = 256 / 3 / 3
constexpr int kNumCfg = 3;
constexpr int kCfgCap[kNumCfg] = {512, 256, 256};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t phase) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(phase) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// 1-D TMA: global -> shared, completion counted in bytes on the mbarrier; the matrix is streamed once per product, so it is
// marked evict-first in L2 and leaves the cache to the vectors
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}

template <int BS, bool DIAG, bool FUSE, int kCap, int kStages>
struct TmaSmem {
    static constexpr int NE = DIAG ? BS : BS * BS;
    static constexpr int VAL_BYTES = kCap * NE * 8;
    static constexpr int COL_BYTES = kCap * 4;
    static constexpr int RP_BYTES = (kMaxR + 4) * 4;
    static constexpr int M_BYTES = FUSE ? kCap * 8 : 0;
    static constexpr int STAGE_BYTES = VAL_BYTES + COL_BYTES + RP_BYTES + M_BYTES;
    static constexpr int PART_BYTES = kCap * BS * 8;
    static constexpr int RSUM_BYTES = kMaxR * BS * 8;
    static constexpr int RPL_BYTES = (kMaxR + 4) * 4;
    static constexpr int TOTAL = kStages * STAGE_BYTES + PART_BYTES + RSUM_BYTES + RPL_BYTES + 8 * 8 + kStages * 8;
    static_assert(STAGE_BYTES % 16 == 0 && VAL_BYTES % 16 == 0 && COL_BYTES % 16 == 0 && RP_BYTES % 16 == 0, "TMA alignment");
};

template <int BS, int MODE, bool DIAG, bool FUSE, int kCap, int kStages, int kMinB>
__global__ void __launch_bounds__(kT, kMinB)
k_bsr_tma(const int4* __restrict__ desc, int nchunk, const int* __restrict__ crp, const int* __restrict__ col,
          const double* __restrict__ val, const double* __restrict__ mval, const double* __restrict__ x,
          const double* __restrict__ x2, double* __restrict__ y, Epilogue ep, double* __restrict__ dot_partial, int G) {
    using L = TmaSmem<BS, DIAG, FUSE, kCap, kStages>;
    constexpr int NE = L::NE;
    extern __shared__ __align__(128) unsigned char smem[];
    double* part = reinterpret_cast<double*>(smem + kStages * L::STAGE_BYTES);
    double* rsum = part + kCap * BS;
    int* rpl = reinterpret_cast<int*>(rsum + kMaxR * BS);
    double* red = reinterpret_cast<double*>(rpl + kMaxR + 4);
    uint64_t* bars = reinterpret_cast<uint64_t*>(red + 8);

    const int tid = threadIdx.x;
    const int c0 = (int)(((int64_t)blockIdx.x * nchunk) / gridDim.x);
    const int c1 = (int)(((int64_t)(blockIdx.x + 1) * nchunk) / gridDim.x);
    const int nloc = c1 - c0;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) mbar_init(&bars[s], 1);
        fence_mbar_init();
        fence_proxy_async();
    }
    __syncthreads();
    uint64_t policy = 0;
    if (tid == 0) policy = policy_evict_first();
    // producer (thread 0): post the bulk copies of local chunk k into stage k % kStages
    auto issue = [&](int k) {
        const int4 d = __ldg(desc + c0 + k);
        const uint32_t nbr = (uint32_t)d.w & 0xffffu, cnt = (uint32_t)d.w >> 16;
        const int st = k % kStages;
        unsigned char* base = smem + st * L::STAGE_BYTES;
        const uint32_t groups = (cnt + 31u) >> 5;
        const uint32_t vb = groups * NE * 256u, cb = groups * 128u, rb = ((nbr + 1u + 3u) >> 2) * 16u, mb = FUSE ? groups * 256u : 0u;
        mbar_expect_tx(&bars[st], vb + cb + rb + mb);
        // a chunk of >= 64 empty block rows has no blocks: no zero-byte copies (the row pointers, rb >= 16, still arrive)
        if (cnt) {
            bulk_g2s(base, val + (size_t)(d.y >> 5) * NE * 32, vb, &bars[st], policy);
            bulk_g2s(base + L::VAL_BYTES, col + d.y, cb, &bars[st], policy);
            if (FUSE) bulk_g2s(base + L::VAL_BYTES + L::COL_BYTES + L::RP_BYTES, mval + d.y, mb, &bars[st], policy);
        }
        bulk_g2s(base + L::VAL_BYTES + L::COL_BYTES, crp + d.z, rb, &bars[st], policy);
    };
    if (tid == 0)
        for (int k = 0; k < kStages && k < nloc; ++k) issue(k);

    const int lg = 31 - __clz(G);
    const int lane = tid & (G - 1);
    const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << ((tid & 31) & ~(G - 1)));
    double contrib = 0.0;
    for (int k = 0; k < nloc; ++k) {
        const int st = k % kStages;
        const uint32_t ph = (uint32_t)(k / kStages) & 1u;
        const int4 d = __ldg(desc + c0 + k);
        const int R0 = d.x, nbr = d.w & 0xffff, cnt = (int)((uint32_t)d.w >> 16);
        // epilogue operands of this thread's scalar row: in flight while the chunk is multiplied and reduced
        const bool has_row = tid < nbr * BS;
        const int myrow = R0 * BS + tid;
        double e0 = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;
        if (has_row) {
            if (MODE == SPMV_SUB || MODE == SPMV_ADD) e0 = ep.z[myrow];
            else if (MODE == 3) { e0 = ep.r[myrow]; e1 = ep.d_old[myrow]; e2 = ep.dinv[myrow]; e3 = ep.xv[myrow]; }
            else if (MODE == 4) e0 = x[myrow];
        }
        while (!mbar_try_wait(&bars[st], ph)) {}
        const unsigned char* base = smem + st * L::STAGE_BYTES;
        const double* vs = reinterpret_cast<const double*>(base);
        const int* cs = reinterpret_cast<const int*>(base + L::VAL_BYTES);
        const int* rps = reinterpret_cast<const int*>(base + L::VAL_BYTES + L::COL_BYTES);
        const double* ms = reinterpret_cast<const double*>(base + L::VAL_BYTES + L::COL_BYTES + L::RP_BYTES);
        if (tid <= nbr) rpl[tid] = rps[tid];
        // phase 1: one thread per block, all gathers issued before the first use
        constexpr int NT = kCap / kT;
        int cc[NT];
        unsigned mk[NT];
        double xv[NT][BS], x2v[NT][BS];
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int i = tid + t * kT;
            cc[t] = -1;
            mk[t] = 0u;
            if (i < cnt) {
                int cw = cs[i];
                if (FUSE) { mk[t] = (unsigned)cw >> 29; cw &= 0x1fffffff; }
                cc[t] = cw;
#pragma unroll
                for (int j = 0; j < BS; ++j) xv[t][j] = __ldg(x + (size_t)cw * BS + j);
                if (FUSE) {
#pragma unroll
                    for (int j = 0; j < BS; ++j) x2v[t][j] = __ldg(x2 + (size_t)cw * BS + j);
                }
            }
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int i = tid + t * kT;
            if (cc[t] >= 0) {
                const double* vb = vs + (size_t)(i >> 5) * NE * 32 + (i & 31);
                const double m = FUSE ? ms[i] : 0.0;
#pragma unroll
                for (int q = 0; q < BS; ++q) {
                    double s = 0.0;
                    if (DIAG) s = vb[q * 32] * xv[t][q];
                    else {
#pragma unroll
                        for (int j = 0; j < BS; ++j) s = fma(vb[(DIAG ? 0 : q * BS + j) * 32], xv[t][j], s);
                    }
                    if (FUSE && ((mk[t] >> q) & 1u)) s = fma(m, x2v[t][q], s);
                    part[i * BS + q] = s;
                }
            }
        }
        __syncthreads();
        // the stage is consumed: refill it with chunk k + kStages while rows are reduced and the epilogue runs
        if (tid == 0 && k + kStages < nloc) { fence_proxy_async(); issue(k + kStages); }
        // phase 2: G lanes per block row
        for (int Rl = tid >> lg; Rl < nbr; Rl += kT >> lg) {
            const int a = rpl[Rl], b = rpl[Rl + 1];
            double s[BS];
#pragma unroll
            for (int q = 0; q < BS; ++q) s[q] = 0.0;
            for (int i = a + lane; i < b; i += G) {
#pragma unroll
                for (int q = 0; q < BS; ++q) s[q] += part[i * BS + q];
            }
#pragma unroll
            for (int q = 0; q < BS; ++q)
                for (int o = G >> 1; o > 0; o >>= 1) s[q] += __shfl_down_sync(gmask, s[q], o, G);
            if (lane == 0) {
#pragma unroll
                for (int q = 0; q < BS; ++q) rsum[Rl * BS + q] = s[q];
            }
        }
        __syncthreads();
        // phase 3: one scalar row per thread, operands already in registers
        if (has_row) {
            const double sum = rsum[tid];
            if (MODE == SPMV_SET) y[myrow] = sum;
            else if (MODE == SPMV_SUB) y[myrow] = e0 - sum;
            else if (MODE == SPMV_ADD) y[myrow] = e0 + sum;
            else if (MODE == 3) {
                const double rn = e0 - sum;
                const double dn = ep.c1 * e1 + ep.c2 * e2 * rn;
                ep.r[myrow] = rn;
                ep.d_new[myrow] = dn;
                ep.xv[myrow] = e3 + dn;
            } else {
                y[myrow] = sum;
                contrib = fma(sum, e0, contrib);
            }
        }
    }
    if (MODE == 4) {
        const double t = block_sum_256(contrib, red);
        if (tid == 0) dot_partial[blockIdx.x] = t;
    }
}

template <class F>
__global__ void __launch_bounds__(256) k_for_t(int64_t n, F f) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) f(i);
}
template <class F>
void pfor(Ctx& c, int64_t n, F f) {
    if (n <= 0) return;
    int64_t g = (n + 255) / 256, cap = (int64_t)c.sm_count * 16;
    k_for_t<<<(int)(g < cap ? g : cap), 256, 0, c.stream>>>(n, f);
    PORO_LAUNCH_CHECK(c);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// chunked layout from the plain BSR arrays (device copy, chunking on the host)
// ---------------------------------------------------------------------------------------------
bool bsr_build_tma(Ctx& c, Bsr& B, const std::vector<int>& rp) {
    if (B.bs != 2 && B.bs != 3) return false;
    B.t_cfg = std::max(0, std::min(kNumCfg - 1, c.opt_i("-poro_bsr_tma_cfg", 1)));
    const int kCap = kCfgCap[B.t_cfg];
    const int nbr = B.nbrows;
    const int NE = B.diag_only ? B.bs : B.bs * B.bs;
    std::vector<int> desc;            // 4 ints per chunk: R0, block offset (padded space), row-pointer offset, nbr | cnt << 16
    int64_t boff = 0, rpo = 0;
    int r = 0;
    while (r < nbr) {
        const int limit = rp[r] + kCap;
        int hi = (int)(std::upper_bound(rp.begin() + r + 1, rp.end(), limit) - rp.begin()) - 1;
        hi = std::min(hi, r + kMaxR);
        if (hi <= r) return false;                                  // a block row longer than a chunk: plain kernel
        // among the last few admissible row boundaries take the one that wastes the least padding per block
        int best = hi;
        double best_w = 1e300;
        for (int h = hi; h > r && h > hi - 4; --h) {
            const int cnt = rp[h] - rp[r];
            if (cnt <= 0) continue;
            const double w = (double)(((cnt + 31) & ~31) - cnt) / cnt + (h == hi ? 0.0 : 0.004 * (hi - h));
            if (w < best_w) { best_w = w; best = h; }
        }
        hi = best;
        const int cnt = rp[hi] - rp[r];
        desc.push_back(r);
        desc.push_back((int)boff);
        desc.push_back((int)rpo);
        desc.push_back((hi - r) | (cnt << 16));
        boff += (cnt + 31) & ~31;
        rpo += ((hi - r) + 1 + 3) & ~3;
        PORO_REQUIRE(boff < 2147483647LL, "chunked BSR: more than 2^31 padded blocks");
        r = hi;
    }
    B.t_nchunk = (int)(desc.size() / 4);
    if (B.t_nchunk == 0) return false;
    B.t_desc.alloc(desc.size());
    PORO_CUDA(cudaMemcpyAsync(B.t_desc.p, desc.data(), desc.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    B.t_col.alloc((size_t)boff);
    B.t_col.zero(c.stream);
    B.t_val.alloc((size_t)boff * NE);
    B.t_val.zero(c.stream);
    B.t_rp.alloc((size_t)rpo + 4);
    B.t_rp.zero(c.stream);
    {
        const int* dsc = B.t_desc.p; const int* brp = B.rowptr.p; const int* bc = B.col.p; const double* bv = B.val.p;
        int* tc = B.t_col.p; double* tv = B.t_val.p; int* trp = B.t_rp.p;
        const int ne = NE;
        // one warp per chunk walks its blocks
        pfor(c, (int64_t)B.t_nchunk * 32, [=] __device__(int64_t gt) {
            const int ch = (int)(gt >> 5), ln = (int)(gt & 31);
            const int R0 = dsc[4 * ch], bo = dsc[4 * ch + 1], ro = dsc[4 * ch + 2];
            const int nb = dsc[4 * ch + 3] & 0xffff, cnt = (int)((unsigned)dsc[4 * ch + 3] >> 16);
            const int p0 = brp[R0];
            for (int j = ln; j <= nb; j += 32) trp[ro + j] = brp[R0 + j] - p0;
            for (int i = ln; i < cnt; i += 32) {
                const size_t p = (size_t)p0 + i, q = (size_t)bo + i;
                tc[q] = bc[p];
                for (int e = 0; e < ne; ++e) tv[((q >> 5) * ne + e) * 32 + (q & 31)] = bv[((p >> 5) * ne + e) * 32 + (p & 31)];
            }
        });
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    B.t_blocks_padded = boff;
    B.t_ok = true;
    return true;
}

// ---------------------------------------------------------------------------------------------
// fused mass coupling: C (same block rows, diagonal blocks c M_IJ I with zeroed Dirichlet rows) rides along B
// ---------------------------------------------------------------------------------------------
bool bsr_fuse_coupling_tma(Ctx& c, Bsr& B, const Csr& C) {
    if (!B.t_ok || B.diag_only || C.nrows != B.nbrows * B.bs || C.ncols != B.nbcols * B.bs) return false;
    if ((int64_t)B.nbcols >= (1 << 29)) return false;
    const int BS = B.bs;
    B.t_m.alloc((size_t)B.t_blocks_padded);
    B.t_m.zero(c.stream);
    DBuf<int> colw((size_t)B.t_blocks_padded);
    PORO_CUDA(cudaMemcpyAsync(colw.p, B.t_col.p, (size_t)B.t_blocks_padded * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
    DBuf<unsigned long long> counters(2);      // [0] coupling nonzeros matched, [1] violations of the c M_IJ I x mask form
    counters.zero(c.stream);
    {
        const int* dsc = B.t_desc.p; const int* trp = B.t_rp.p; int* tc = colw.p; double* tm = B.t_m.p;
        const int* crp = C.rowptr.p; const int* ccol = C.col.p; const double* cv = C.val.p;
        unsigned long long* cnts = counters.p;
        pfor(c, (int64_t)B.t_nchunk * 32, [=] __device__(int64_t gt) {
            const int ch = (int)(gt >> 5), ln = (int)(gt & 31);
            const int R0 = dsc[4 * ch], bo = dsc[4 * ch + 1], ro = dsc[4 * ch + 2];
            const int nb = dsc[4 * ch + 3] & 0xffff;
            unsigned long long matched = 0, bad = 0;
            for (int Rl = 0; Rl < nb; ++Rl) {
                const int I = R0 + Rl;
                for (int i = trp[ro + Rl] + ln; i < trp[ro + Rl + 1]; i += 32) {
                    const int J = tc[bo + i];
                    double m = 0.0;
                    unsigned mask = 0u;
                    for (int q = 0; q < BS; ++q) {
                        // entry ((I, q), (J, q)) of the coupling by binary search in its (sorted) row
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
                    tm[bo + i] = m;
                    tc[bo + i] = J | (int)(mask << 29);
                }
            }
            if (matched) atomicAdd(cnts, matched);
            if (bad) atomicAdd(cnts + 1, bad);
        });
    }
    unsigned long long h[2] = {0, 0};
    PORO_CUDA(cudaMemcpyAsync(h, counters.p, sizeof h, cudaMemcpyDeviceToHost, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    // every stored entry of the coupling must sit on the diagonal of a block of B (its off-diagonal entries were excluded
    // by the caller: the coupling is `diag_only`), and within a block all non-zero diagonal entries must be equal
    if (h[1] != 0 || (int64_t)h[0] != C.nnz) { B.t_m.release(); return false; }
    B.t_colf = std::move(colw);
    B.t_fused = true;
    return true;
}

// ---------------------------------------------------------------------------------------------
// launch
// ---------------------------------------------------------------------------------------------
template <int BS, int MODE, bool DIAG, bool FUSE, int kCap, int kStages, int kMinB>
static void launch_cfg(Ctx& c, const Bsr& B, const double* x, const double* x2, double* y, const Epilogue& ep, double* dot_partial, int G,
                       int grid) {
    using L = TmaSmem<BS, DIAG, FUSE, kCap, kStages>;
    static bool configured = false;
    if (!configured) {
        PORO_CUDA(cudaFuncSetAttribute(k_bsr_tma<BS, MODE, DIAG, FUSE, kCap, kStages, kMinB>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
        configured = true;
    }
    k_bsr_tma<BS, MODE, DIAG, FUSE, kCap, kStages, kMinB><<<grid, kT, L::TOTAL, c.stream>>>(
        reinterpret_cast<const int4*>(B.t_desc.p), B.t_nchunk, B.t_rp.p, FUSE ? B.t_colf.p : B.t_col.p, B.t_val.p, FUSE ? B.t_m.p : nullptr,
        x, x2, y, ep, dot_partial, G);
}

template <int BS, int MODE, bool DIAG, bool FUSE>
static void launch_one(Ctx& c, const Bsr& B, const double* x, const double* x2, double* y, const Epilogue& ep, double* dot_partial, int G,
                       int grid) {
    if (B.t_cfg == 0) launch_cfg<BS, MODE, DIAG, FUSE, 512, 2, 2>(c, B, x, x2, y, ep, dot_partial, G, grid);
    else if (B.t_cfg == 1) launch_cfg<BS, MODE, DIAG, FUSE, 256, 2, 4>(c, B, x, x2, y, ep, dot_partial, G, grid);
    else launch_cfg<BS, MODE, DIAG, FUSE, 256, 3, 3>(c, B, x, x2, y, ep, dot_partial, G, grid);
}

template <int MODE>
int bsr_tma_launch(Ctx& c, const Bsr& B, const double* x, double* y, const Epilogue& ep, double* dot_partial, const double* x2) {
    const int G = row_group_lanes(B.nbrows ? (double)B.nnzb / B.nbrows : 0.0);
    const bool fuse = x2 != nullptr && B.t_fused;
    const int min_b = B.t_cfg == 0 ? 2 : (B.t_cfg == 1 ? 4 : 3);
    const int grid = std::min(B.t_nchunk, min_b * c.sm_count);
    if (B.bs == 3) {
        if (fuse) launch_one<3, MODE, false, true>(c, B, x, x2, y, ep, dot_partial, G, grid);
        else if (B.diag_only) launch_one<3, MODE, true, false>(c, B, x, x2, y, ep, dot_partial, G, grid);
        else launch_one<3, MODE, false, false>(c, B, x, x2, y, ep, dot_partial, G, grid);
    } else {
        if (fuse) launch_one<2, MODE, false, true>(c, B, x, x2, y, ep, dot_partial, G, grid);
        else if (B.diag_only) launch_one<2, MODE, true, false>(c, B, x, x2, y, ep, dot_partial, G, grid);
        else launch_one<2, MODE, false, false>(c, B, x, x2, y, ep, dot_partial, G, grid);
    }
    PORO_LAUNCH_CHECK(c);
    return grid;
}

template int bsr_tma_launch<0>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_tma_launch<1>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_tma_launch<2>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_tma_launch<3>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);
template int bsr_tma_launch<4>(Ctx&, const Bsr&, const double*, double*, const Epilogue&, double*, const double*);

}  // namespace poro
