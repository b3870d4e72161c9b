// amg.cu -- smoothed-aggregation AMG built and applied on the device.
//
// Stands where the reference uses hypre BoomerAMG behind `-*_pc_type hypre`
// (lib/Preconditioner.py:94-100, petsc-options-inexact:16-24, 32-40, 48-55, 62-69, 88-96).
// It is NOT BoomerAMG (classical RS-AMG, HMIS/ext+i): it is our own SA-AMG, specified in
// oracle/amg.py, which mirrors every deterministic choice made here (hash priorities,
// synchronous Luby rounds, per-aggregate modified Gram-Schmidt) so both build the same
// hierarchy.  Set-up: nodal strength graph -> MIS(2) aggregation -> tentative prolongator from
// the near-nullspace -> Jacobi-smoothed prolongator -> Galerkin triple product (SpGEMM).
// Apply: V-cycle with Chebyshev smoothing on D^-1 A (fused SpMV + update kernel), dense
// inverse on the coarsest level.
#include "amg.cuh"
#include "dist.cuh"
#include "distamg.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <chrono>
#include <cmath>

namespace poro {

static constexpr int kB = 256;

template <class F>
__global__ void __launch_bounds__(kB) k_for2(int64_t n, F f) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) f(i);
}
template <class F>
static void pfor(Ctx& c, int64_t n, F f) {
    if (n <= 0) return;
    int64_t g = (n + kB - 1) / kB;
    int64_t cap = (int64_t)c.sm_count * 16;
    k_for2<<<(int)(g < cap ? g : cap), kB, 0, c.stream>>>(n, f);
    PORO_LAUNCH_CHECK(c);
}

__host__ __device__ inline uint32_t hash32(uint32_t i) {
    uint32_t x = i + 0x9E3779B9u;
    x = (x ^ (x >> 16)) * 0x85EBCA6Bu;
    x = (x ^ (x >> 13)) * 0xC2B2AE35u;
    x = x ^ (x >> 16);
    return x;
}

static int64_t scan_i64(Ctx& c, const int64_t* in, int64_t* out, int64_t n) {
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, n, c.stream);
    DBuf<char> tmp(tb);
    cub::DeviceScan::ExclusiveSum(tmp.p, tb, in, out, n, c.stream);
    c.launches++;
    int64_t a = 0, b = 0;
    if (n > 0) {
        PORO_CUDA(cudaMemcpyAsync(&a, in + n - 1, 8, cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaMemcpyAsync(&b, out + n - 1, 8, cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
    }
    return a + b;
}

static void csr_rows_of(Ctx& c, const Csr& A, int* rows) {
    const int* rp = A.rowptr.p;
    pfor(c, A.nrows, [=] __device__(int64_t i) { for (int k = rp[i]; k < rp[i + 1]; ++k) rows[k] = (int)i; });
}

// ---- 1. symmetrised nodal strength graph; values = squared Frobenius norms of the blocks ----
static void strength_graph(Ctx& c, const Csr& A, int bs, double theta, Csr& S) {
    const int nn = A.nrows / bs;
    Csr N2;
    {
        DBuf<uint64_t> keys((size_t)A.nnz);
        DBuf<double> vals((size_t)A.nnz);
        DBuf<int> rows((size_t)A.nnz);
        csr_rows_of(c, A, rows.p);
        const int* r = rows.p; const int* cc = A.col.p; const double* v = A.val.p;
        uint64_t* kk = keys.p; double* vv = vals.p;
        pfor(c, A.nnz, [=] __device__(int64_t k) {
            kk[k] = ((uint64_t)(uint32_t)(r[k] / bs) << 32) | (uint32_t)(cc[k] / bs);
            vv[k] = v[k] * v[k];
        });
        coo_to_csr(c, nn, nn, A.nnz, keys, vals, N2, COMBINE_SUM);
    }
    DBuf<double> d((size_t)nn);
    csr_diag(c, N2, d.p);
    DBuf<int> rows((size_t)N2.nnz);
    csr_rows_of(c, N2, rows.p);
    DBuf<int64_t> keep((size_t)N2.nnz + 1), pos((size_t)N2.nnz + 1);
    {
        const int* r = rows.p; const int* cc = N2.col.p; const double* v = N2.val.p; const double* dd = d.p;
        int64_t* kp = keep.p;
        int64_t nz = N2.nnz;
        double t2 = theta * theta;
        pfor(c, N2.nnz + 1, [=] __device__(int64_t k) {
            int64_t f = 0;
            if (k < nz) {
                int i = r[k], j = cc[k];
                f = (i != j && v[k] > 0.0 && v[k] >= t2 * sqrt(dd[i] * dd[j])) ? 1 : 0;
            }
            kp[k] = f;
        });
    }
    int64_t ns = scan_i64(c, keep.p, pos.p, N2.nnz + 1);
    DBuf<uint64_t> keys((size_t)(2 * ns));
    DBuf<double> vals((size_t)(2 * ns));
    {
        const int* r = rows.p; const int* cc = N2.col.p; const double* v = N2.val.p;
        const int64_t* kp = keep.p; const int64_t* ps = pos.p;
        uint64_t* kk = keys.p; double* vv = vals.p;
        pfor(c, N2.nnz, [=] __device__(int64_t k) {
            if (kp[k]) {
                int64_t p = 2 * ps[k];
                kk[p] = ((uint64_t)(uint32_t)r[k] << 32) | (uint32_t)cc[k];
                kk[p + 1] = ((uint64_t)(uint32_t)cc[k] << 32) | (uint32_t)r[k];
                vv[p] = v[k];
                vv[p + 1] = v[k];
            }
        });
    }
    coo_to_csr(c, nn, nn, 2 * ns, keys, vals, S, COMBINE_MAX);
}

// ---- 2. MIS(2) aggregation ----------------------------------------------------------------------
static void nbr_max(Ctx& c, const Csr& S, const int64_t* key, int64_t* out) {
    const int* rp = S.rowptr.p; const int* cc = S.col.p;
    pfor(c, S.nrows, [=] __device__(int64_t i) {
        int64_t m = key[i];
        for (int k = rp[i]; k < rp[i + 1]; ++k) { int64_t v = key[cc[k]]; m = v > m ? v : m; }
        out[i] = m;
    });
}

static int aggregate_mis2(Ctx& c, const Csr& S, DBuf<int>& agg) {
    const int nn = S.nrows;
    DBuf<int> state((size_t)nn);
    DBuf<int64_t> key((size_t)nn), m1((size_t)nn), m2((size_t)nn), flag((size_t)nn);
    DBuf<int> undecided(1);
    {
        const int* rp = S.rowptr.p;
        int* st = state.p;
        pfor(c, nn, [=] __device__(int64_t i) { st[i] = (rp[i + 1] == rp[i]) ? 2 : 0; });
    }
    for (int round = 0; round < 1000; ++round) {
        {
            const int* st = state.p; int64_t* ky = key.p;
            pfor(c, nn, [=] __device__(int64_t i) {
                int64_t prio = ((int64_t)(hash32((uint32_t)i) >> 1) << 32) | (int64_t)(i + 1);
                ky[i] = st[i] == 0 ? prio : 0;
            });
        }
        nbr_max(c, S, key.p, m1.p);
        nbr_max(c, S, m1.p, m2.p);
        {
            int* st = state.p; const int64_t* ky = key.p; const int64_t* mm = m2.p; int64_t* fl = flag.p;
            pfor(c, nn, [=] __device__(int64_t i) {
                bool sel = st[i] == 0 && mm[i] == ky[i];
                if (sel) st[i] = 1;
                fl[i] = sel ? 1 : 0;
            });
        }
        nbr_max(c, S, flag.p, m1.p);
        nbr_max(c, S, m1.p, m2.p);
        undecided.zero(c.stream);
        {
            int* st = state.p; const int64_t* f2 = m2.p; int* un = undecided.p;
            pfor(c, nn, [=] __device__(int64_t i) {
                if (st[i] == 0) {
                    if (f2[i] > 0) st[i] = 2;
                    else *un = 1;
                }
            });
        }
        int h = 0;
        PORO_CUDA(cudaMemcpyAsync(&h, undecided.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        if (!h) break;
    }
    // roots numbered by ascending node id
    DBuf<int64_t> isroot((size_t)nn + 1), rid((size_t)nn + 1);
    {
        const int* st = state.p; int64_t* ir = isroot.p; int n_ = nn;
        pfor(c, (int64_t)nn + 1, [=] __device__(int64_t i) { ir[i] = (i < n_ && st[i] == 1) ? 1 : 0; });
    }
    int64_t n_agg = scan_i64(c, isroot.p, rid.p, (int64_t)nn + 1);
    agg.alloc((size_t)nn);
    DBuf<int> agg2((size_t)nn);
    {
        const int64_t* ir = isroot.p; const int64_t* id = rid.p; int* ag = agg.p;
        pfor(c, nn, [=] __device__(int64_t i) { ag[i] = ir[i] ? (int)id[i] : -1; });
    }
    for (int round = 0; round < 2; ++round) {
        const int* rp = S.rowptr.p; const int* cc = S.col.p; const double* w = S.val.p;
        const int* ain = agg.p; int* aout = agg2.p;
        pfor(c, nn, [=] __device__(int64_t i) {
            int a = ain[i];
            if (a < 0) {
                double bw = -1.0;
                int ba = -1;
                for (int k = rp[i]; k < rp[i + 1]; ++k) {
                    int aj = ain[cc[k]];
                    if (aj >= 0 && (w[k] > bw || (w[k] == bw && aj < ba))) { bw = w[k]; ba = aj; }
                }
                a = ba;
            }
            aout[i] = a;
        });
        std::swap(agg.p, agg2.p);
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    return (int)n_agg;
}

// ---- 3. tentative prolongator: per-aggregate modified Gram-Schmidt, one warp per aggregate -------
__global__ void __launch_bounds__(kB) k_mgs(int n_agg, const int* __restrict__ mstart, int bs, int k,
                                            double* __restrict__ Q, double* __restrict__ Bc) {
    const int a = (blockIdx.x * kB + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (a >= n_agg) return;
    const int r0 = mstart[a] * bs, r1 = mstart[a + 1] * bs;
    double* R = Bc + (size_t)a * k * k;
    for (int j = 0; j < k; ++j) {
        for (int i = 0; i < j; ++i) {
            double s = 0.0;
            for (int r = r0 + lane; r < r1; r += 32) s += Q[(size_t)r * k + i] * Q[(size_t)r * k + j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            for (int r = r0 + lane; r < r1; r += 32) Q[(size_t)r * k + j] -= s * Q[(size_t)r * k + i];
            if (lane == 0) R[i * k + j] = s;
            __syncwarp();
        }
        double s = 0.0;
        for (int r = r0 + lane; r < r1; r += 32) { double q = Q[(size_t)r * k + j]; s += q * q; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        double nrm = sqrt(s);
        bool ok = nrm > 1e-8;
        double inv = ok ? 1.0 / nrm : 0.0;
        for (int r = r0 + lane; r < r1; r += 32) Q[(size_t)r * k + j] *= inv;
        if (lane == 0) {
            R[j * k + j] = ok ? nrm : 0.0;
            for (int i = j + 1; i < k; ++i) R[i * k + j] = 0.0;
        }
        __syncwarp();
    }
}

static void tentative(Ctx& c, const DBuf<int>& agg, int n_agg, int nn, int bs, int k, const double* B, Csr& T,
                      DBuf<double>& Bc) {
    // members sorted by (aggregate, node id); non-members go to a trailing dummy row
    Csr mem;
    {
        DBuf<uint64_t> keys((size_t)nn);
        DBuf<double> vals((size_t)nn);
        const int* ag = agg.p; uint64_t* kk = keys.p; double* vv = vals.p; int na = n_agg;
        pfor(c, nn, [=] __device__(int64_t i) {
            int a = ag[i] >= 0 ? ag[i] : na;
            kk[i] = ((uint64_t)(uint32_t)a << 32) | (uint32_t)i;
            vv[i] = 1.0;
        });
        coo_to_csr(c, n_agg + 1, nn, nn, keys, vals, mem, COMBINE_SUM);
    }
    int nmem = 0;
    PORO_CUDA(cudaMemcpy(&nmem, mem.rowptr.p + n_agg, sizeof(int), cudaMemcpyDeviceToHost));
    DBuf<double> Q((size_t)nmem * bs * k);
    {
        const int* nodes = mem.col.p; double* q = Q.p;
        pfor(c, (int64_t)nmem * bs * k, [=] __device__(int64_t t) {
            int j = (int)(t % k);
            int64_t lr = t / k;
            int cpt = (int)(lr % bs);
            int p = (int)(lr / bs);
            q[t] = B[((size_t)nodes[p] * bs + cpt) * k + j];
        });
    }
    Bc.alloc((size_t)n_agg * k * k);
    Bc.zero(c.stream);
    k_mgs<<<ceil_div((int64_t)n_agg * 32, kB), kB, 0, c.stream>>>(n_agg, mem.rowptr.p, bs, k, Q.p, Bc.p);
    PORO_LAUNCH_CHECK(c);
    // T as triples
    int64_t nent = (int64_t)nmem * bs * k;
    DBuf<uint64_t> keys((size_t)nent);
    DBuf<double> vals((size_t)nent);
    {
        const int* nodes = mem.col.p; const int* ag = agg.p; const double* q = Q.p;
        uint64_t* kk = keys.p; double* vv = vals.p;
        pfor(c, nent, [=] __device__(int64_t t) {
            int j = (int)(t % k);
            int64_t lr = t / k;
            int cpt = (int)(lr % bs);
            int p = (int)(lr / bs);
            int node = nodes[p];
            kk[t] = ((uint64_t)(uint32_t)(node * bs + cpt) << 32) | (uint32_t)(ag[node] * k + j);
            vv[t] = q[t];
        });
    }
    coo_to_csr(c, nn * bs, n_agg * k, nent, keys, vals, T, COMBINE_SUM);
}

// ---- power iteration for lambda_max(D^-1 A) ----------------------------------------------------
static double power_lmax(Ctx& c, const Csr& A, const double* dinv, int its) {
    const int n = A.nrows;
    DBuf<double> v((size_t)n), w((size_t)n);
    {
        double* vv = v.p;
        pfor(c, n, [=] __device__(int64_t i) { vv[i] = (double)(hash32((uint32_t)i) % 2048u) / 1024.0 - 1.0; });
    }
    double nv = norm2_host(c, v.p, n);
    if (nv == 0) return 1.0;
    vec_scale(c, v.p, 1.0 / nv, n);
    double lam = 1.0;
    for (int it = 0; it < its; ++it) {
        spmv(c, A, v.p, w.p);
        vec_pmult(c, w.p, dinv, w.p, n);
        lam = norm2_host(c, w.p, n);
        if (lam == 0.0) return 1.0;
        vec_waxpby(c, v.p, 1.0 / lam, w.p, 0.0, w.p, n);
    }
    return lam;
}

static void make_dinv(Ctx& c, const Csr& A, DBuf<double>& dinv) {
    dinv.alloc((size_t)A.nrows);
    csr_diag(c, A, dinv.p);
    double* d = dinv.p;
    pfor(c, A.nrows, [=] __device__(int64_t i) { d[i] = d[i] != 0.0 ? 1.0 / d[i] : 1.0; });
}

struct Tick {
    Ctx& c; bool on; const char* what; std::chrono::steady_clock::time_point t0;
    Tick(Ctx& c_, const char* w) : c(c_), on(c_.has_opt("-poro_verbose")), what(w) {
        if (on) { cudaStreamSynchronize(c.stream); t0 = std::chrono::steady_clock::now(); }
    }
    ~Tick() {
        if (on) {
            cudaStreamSynchronize(c.stream);
            fprintf(stderr, "      [amg] %-22s %8.1f ms\n", what,
                    1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
        }
    }
};

// distributed power iteration: start vector hashed from GLOBAL ids, halo exchange before every product, all-reduced norms
static double power_lmax_dist(Ctx& c, const Csr& A, DistPlan& plan, const double* dinv, int its) {
    const int n = plan.n_owned, ng = plan.n_ghost;
    DBuf<double> v((size_t)n + ng), w((size_t)n);
    {
        double* vv = v.p; const uint32_t off = (uint32_t)plan.offset;
        pfor(c, n, [=] __device__(int64_t i) { vv[i] = (double)(hash32(off + (uint32_t)i) % 2048u) / 1024.0 - 1.0; });
    }
    double nv = norm2_host(c, v.p, n);
    if (nv == 0) return 1.0;
    vec_scale(c, v.p, 1.0 / nv, n);
    double lam = 1.0;
    for (int it = 0; it < its; ++it) {
        dist_halo_vec(c, plan, v.p, 1, v.p + n);
        spmv(c, A, v.p, w.p);
        vec_pmult(c, w.p, dinv, w.p, n);
        lam = norm2_host(c, w.p, n);
        if (lam == 0.0) return 1.0;
        vec_waxpby(c, v.p, 1.0 / lam, w.p, 0.0, w.p, n);
    }
    return lam;
}

// gathers a distributed level operator (local rows x [owned | ghost]) and its near-nullspace rows on EVERY rank
static void gather_level(Ctx& c, const Csr& A, const DistPlan& plan, const double* B, int k, Csr& Ag, DBuf<double>& Bg) {
    const int R = c.nranks;
    const int64_t ng = plan.offsets.back();
    Csr Al;
    csr_copy(c, A, Al);
    dist_globalize(c, Al, plan, ng);
    std::vector<int64_t> mine = {(int64_t)Al.nrows, Al.nnz}, all;
    dist_allgather_i64(c, mine.data(), 2, all);
    int64_t maxr = 1, maxz = 1, nnz_tot = 0;
    for (int r = 0; r < R; ++r) { maxr = std::max(maxr, all[2 * r]); maxz = std::max(maxz, all[2 * r + 1]); nnz_tot += all[2 * r + 1]; }
    PORO_REQUIRE(nnz_tot < 2147483647LL, "gathered level too large");
    DBuf<int> slen((size_t)maxr), glen((size_t)R * maxr), scol((size_t)maxz), gcol((size_t)R * maxz);
    DBuf<double> sval((size_t)maxz), gval((size_t)R * maxz), sB((size_t)maxr * k), gB((size_t)R * maxr * k);
    slen.zero(c.stream); scol.zero(c.stream); sval.zero(c.stream); sB.zero(c.stream);
    {
        const int* rp = Al.rowptr.p; int* L = slen.p;
        pfor(c, Al.nrows, [=] __device__(int64_t i) { L[i] = rp[i + 1] - rp[i]; });
    }
    if (Al.nnz) {
        PORO_CUDA(cudaMemcpyAsync(scol.p, Al.col.p, (size_t)Al.nnz * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
        PORO_CUDA(cudaMemcpyAsync(sval.p, Al.val.p, (size_t)Al.nnz * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
    }
    if (Al.nrows) PORO_CUDA(cudaMemcpyAsync(sB.p, B, (size_t)Al.nrows * k * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
    dist_allgather_bytes(c, slen.p, (size_t)maxr * sizeof(int), glen.p);
    dist_allgather_bytes(c, scol.p, (size_t)maxz * sizeof(int), gcol.p);
    dist_allgather_bytes(c, sval.p, (size_t)maxz * sizeof(double), gval.p);
    dist_allgather_bytes(c, sB.p, (size_t)maxr * k * sizeof(double), gB.p);
    Ag.nrows = (int)ng; Ag.ncols = (int)ng; Ag.nnz = nnz_tot;
    Ag.rowptr.alloc((size_t)ng + 1); Ag.col.alloc((size_t)nnz_tot); Ag.val.alloc((size_t)nnz_tot);
    Bg.alloc((size_t)ng * k);
    DBuf<int64_t> len64((size_t)ng + 1), ptr64((size_t)ng + 1);
    len64.zero(c.stream);
    int64_t zoff = 0;
    for (int r = 0; r < R; ++r) {
        const int64_t rows = all[2 * r], nz = all[2 * r + 1], ro = plan.offsets[r];
        {
            const int* src = glen.p + (size_t)r * maxr; int64_t* dst = len64.p + ro;
            pfor(c, rows, [=] __device__(int64_t i) { dst[i] = src[i]; });
        }
        if (nz) {
            PORO_CUDA(cudaMemcpyAsync(Ag.col.p + zoff, gcol.p + (size_t)r * maxz, (size_t)nz * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
            PORO_CUDA(cudaMemcpyAsync(Ag.val.p + zoff, gval.p + (size_t)r * maxz, (size_t)nz * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
        }
        if (rows) PORO_CUDA(cudaMemcpyAsync(Bg.p + (size_t)ro * k, gB.p + (size_t)r * maxr * k, (size_t)rows * k * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
        zoff += nz;
    }
    scan_i64(c, len64.p, ptr64.p, ng + 1);
    {
        const int64_t* s64 = ptr64.p; int* rp = Ag.rowptr.p;
        pfor(c, ng + 1, [=] __device__(int64_t i) { rp[i] = (int)s64[i]; });
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    csr_choose_lanes(Ag);
}

// ---- set-up ---------------------------------------------------------------------------------
void Amg::setup(Ctx& c, const Csr& A, int bs, const double* B_dev, int k, const AmgParams& p, DistPlan* plan0) {
    dist = plan0 != nullptr && c.nranks > 1;
    // a hierarchy without a plan is built on this rank's owned block: its reductions must not be collective
    struct LocalScope { Ctx& c; bool old; LocalScope(Ctx& c_, bool loc) : c(c_), old(c_.local_only) { if (loc) c.local_only = true; } ~LocalScope() { c.local_only = old; } } local_scope(c, !dist);
    ctx = &c;
    par = p;
    A0 = &A;
    levels.clear();
    // opt-in: fp32 STORAGE of every operator of the hierarchy (level operators incl. the block itself, P, R); the V-cycle stays a
    // fixed linear operator in fp64 arithmetic, so plain GMRES remains valid (profiles/r1_mixed_precision_study.md)
    const bool fp32m = c.opt_i("-poro_pc_fp32_matrices", 0) != 0;
    if (fp32m && A.bsr_state < 0) A.fp32_hint = true;
    DBuf<double> B;
    int n = A.nrows;
    if (B_dev) {
        B.alloc((size_t)n * k);
        PORO_CUDA(cudaMemcpyAsync(B.p, B_dev, (size_t)n * k * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
    } else {
        k = bs;
        B.alloc((size_t)n * k);
        double* b = B.p;
        pfor(c, (int64_t)n * k, [=] __device__(int64_t t) { b[t] = ((t / k) % bs == (t % k)) ? 1.0 : 0.0; });
    }
    Csr Anext;
    bool have_next = false;
    std::unique_ptr<DistPlan> next_plan;
    const bool verbose = c.has_opt("-poro_verbose");
    const bool keep = !dist && c.opt_i("-poro_amg_keep_setup", 0) != 0;
    auto keep_B = [&](AmgLevel& L) {
        L.keep_B.alloc((size_t)n * k);
        PORO_CUDA(cudaMemcpyAsync(L.keep_B.p, B.p, (size_t)n * k * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
        L.kept = true;
    };
    while (true) {
        auto L = std::make_unique<AmgLevel>();
        if (have_next) L->A = std::move(Anext);
        AmgLevel* Lp = L.get();
        const Csr* Acur = levels.empty() ? &A : &Lp->A;
        if (dist) {
            if (levels.empty()) Lp->plan = plan0;
            else { Lp->owned_plan = std::move(next_plan); Lp->plan = Lp->owned_plan.get(); }
            PORO_REQUIRE(Acur->ncols == Lp->plan->n_owned + Lp->plan->n_ghost && Acur->nrows == Lp->plan->n_owned,
                         "distributed level operator and its halo plan disagree");
        }
        levels.push_back(std::move(L));
        Lp->bs = bs;
        Lp->k = k;
        n = Acur->nrows;
        if (keep) keep_B(*Lp);
        const int n_gh = dist ? Lp->plan->n_ghost : 0;
        const int64_t n_glob = dist ? Lp->plan->offsets.back() : n;
        if (dist && levels.size() >= 2 && (int)levels.size() >= par.mg_levels && !par.smoother_only && n_glob > par.coarse_size &&
            n_glob <= c.opt_i("-poro_amg_replicate_below", 0)) {
            // latency-bound level: gather it once, build and cycle the rest of the hierarchy redundantly on every rank
            Tick t(c, "gathered tail hierarchy");
            DBuf<double> Bg;
            gather_level(c, *Acur, *Lp->plan, B.p, k, tail_A, Bg);
            tail_A.block_hint = bs;
            tail = std::make_unique<Amg>();
            AmgParams tp = par;
            tp.mg_levels = 0;                      // the gathered levels are algebraic (below the coarsest geometric one)
            tp.max_levels = std::max(1, par.max_levels - ((int)levels.size() - std::max(par.mg_levels - 1, 0)) + 1);
            tail->setup(c, tail_A, bs, Bg.p, k, tp, nullptr);
            tail_b.alloc((size_t)n_glob);
            tail_x.alloc((size_t)n_glob);
            Lp->replicated = true;
            Lp->x.alloc((size_t)n + n_gh);
            Lp->b.alloc(n);
            Lp->ext.alloc((size_t)n + n_gh);       // ext() of other vectors (poro_pc_mg_transfer onto this level)
            if (verbose && c.rank == 0)
                fprintf(stderr, "    [amg] level %d: %lld global rows gathered on every rank, %d redundant levels below\n", (int)levels.size() - 1,
                        (long long)n_glob, (int)tail->levels.size());
            break;
        }
        make_dinv(c, *Acur, Lp->dinv);
        {
            Tick t(c, "power iteration");
            Lp->lmax = 1.1 * (dist ? power_lmax_dist(c, *Acur, *Lp->plan, Lp->dinv.p, par.power_its) : power_lmax(c, *Acur, Lp->dinv.p, par.power_its));
        }
        if (verbose && c.rank == 0)
            fprintf(stderr, "    [amg] level %d: n=%d (global %lld) nnz=%lld bs=%d lmax=%.4f%s\n", (int)levels.size() - 1, n, (long long)n_glob,
                    (long long)Acur->nnz, bs, Lp->lmax, dist ? " distributed" : "");
        Lp->x.alloc((size_t)n + n_gh); Lp->b.alloc(n); Lp->r.alloc((size_t)n + n_gh); Lp->d0.alloc((size_t)n + n_gh); Lp->d1.alloc((size_t)n + n_gh);
        if (dist) Lp->ext.alloc((size_t)n + n_gh);
        // geometric levels are taken whatever their size; the algebraic ones count from the coarsest geometric level
        const bool geo_next = (int)levels.size() < par.mg_levels;
        if (!geo_next && (n_glob <= par.coarse_size || (int)levels.size() - std::max(par.mg_levels - 1, 0) >= par.max_levels)) break;
        // Dirichlet rows (diagonal only) carry no near-nullspace
        {
            const int* rp = Acur->rowptr.p; const int* cc = Acur->col.p; const double* v = Acur->val.p;
            double* b = B.p; int kk = k;
            pfor(c, n, [=] __device__(int64_t i) {
                double off = 0.0, d = 0.0;
                for (int q = rp[i]; q < rp[i + 1]; ++q) { if (cc[q] == (int)i) d += v[q]; else off += fabs(v[q]); }
                if (off <= 1e-14 * fabs(d)) for (int j = 0; j < kk; ++j) b[(size_t)i * kk + j] = 0.0;
            });
        }
        if (keep) keep_B(*Lp);
        if (geo_next) {
            // the same block generated at N/2 (rediscretisation = Galerkin product with the geometric transfer), the
            // near-nullspace injected at the coinciding nodes (exact for the rigid-body modes: the coarse space holds them).
            // Row-partitioned: the coarse slab block brings its halo plan, the next level's plan
            Tick t(c, "geometric level");
            Csr Ac;
            mg_coarse_block(c, *Acur->stencil, Ac, dist ? &next_plan : nullptr);
            Ac.block_hint = bs;
            Lp->mg = std::make_unique<MgTransfer>();
            mg_transfer_init(c, *Lp->mg, *Acur->stencil, *Ac.stencil, dist ? next_plan.get() : nullptr);
            DBuf<double> Bc;
            mg_inject(c, *Lp->mg, B.p, k, Bc);
            Anext = std::move(Ac);
            have_next = true;
            B = std::move(Bc);
            continue;
        }
        // aggregation sees the owned diagonal block only: aggregates never cross a rank boundary
        Csr sq;
        const Csr* Asq = Acur;
        if (dist) { csr_select(c, *Acur, 0, n, 0, n, true, sq); Asq = &sq; }
        Csr S;
        DBuf<int> agg;
        int n_agg = 0;
        if (n > 0) {
            { Tick t(c, "strength graph"); strength_graph(c, *Asq, bs, par.theta, S); }
            { Tick t(c, "MIS(2) aggregation"); n_agg = aggregate_mis2(c, S, agg); }
        }
        sq = Csr();
        std::vector<int64_t> coff;
        int64_t nc_glob = (int64_t)n_agg * k;
        if (dist) {
            std::vector<int64_t> sizes;
            const int64_t mine = (int64_t)n_agg * k;
            dist_allgather_i64(c, &mine, 1, sizes);
            coff.assign((size_t)c.nranks + 1, 0);
            for (int r = 0; r < c.nranks; ++r) coff[r + 1] = coff[r] + sizes[r];
            nc_glob = coff.back();
        }
        if (nc_glob == 0 || (double)nc_glob >= 0.8 * (double)n_glob) break;
        Csr T;
        DBuf<double> Bc;
        if (n_agg > 0) { Tick t(c, "tentative prolongator"); tentative(c, agg, n_agg, n / bs, bs, k, B.p, T, Bc); }
        else {
            T.nrows = n; T.ncols = 0; T.nnz = 0;
            T.rowptr.alloc((size_t)n + 1); T.rowptr.zero(c.stream); T.col.alloc(0); T.val.alloc(0);
        }
        double omega = 4.0 / (3.0 * Lp->lmax / 1.1);
        Csr Ac;
        if (!dist) {
            {
                Csr AT;
                { Tick t(c, "spgemm A*T"); csr_spgemm(c, *Acur, T, AT, &Lp->spgemm_chunks[0]); }
                csr_add_scaled(c, T, AT, -omega, Lp->dinv.p, Lp->P);
            }
            { Tick t(c, "transpose P"); csr_transpose(c, Lp->P, Lp->R); }
            {
                Csr AP;
                { Tick t(c, "spgemm A*P"); csr_spgemm(c, *Acur, Lp->P, AP, &Lp->spgemm_chunks[1]); }
                { Tick t(c, "spgemm R*(AP)"); csr_spgemm(c, Lp->R, AP, Ac, &Lp->spgemm_chunks[2]); }
            }
            // dead coarse dofs (rank-deficient aggregates): unit diagonal
            {
                const int* rp = Ac.rowptr.p; const int* cc = Ac.col.p; double* v = Ac.val.p;
                pfor(c, Ac.nrows, [=] __device__(int64_t i) {
                    for (int q = rp[i]; q < rp[i + 1]; ++q) if (cc[q] == (int)i && v[q] == 0.0) v[q] = 1.0;
                });
            }
        } else {
            Tick t(c, "distributed P, Galerkin");
            DistLevelOut o;
            dist_amg_level(c, *Acur, *Lp->plan, T, coff, Lp->dinv.p, omega, o);
            Lp->P = std::move(o.P);
            Lp->R = std::move(o.R);
            Ac = std::move(o.Ac);
            next_plan = std::make_unique<DistPlan>(std::move(o.coarse_plan));
        }
        Lp->n_agg = n_agg;
        if (keep) {
            Lp->keep_agg = std::move(agg);
            Lp->keep_T = std::move(T);
        }
        {
            // block structure of the transfer operators and of the coarse operator (k modes per aggregate)
            const int hint = (bs % 3 == 0 && k % 3 == 0) ? 3 : ((bs % 2 == 0 && k % 2 == 0) ? 2 : 0);
            Lp->P.block_hint = hint;
            Lp->R.block_hint = hint;
            Ac.block_hint = k;
            Lp->P.fp32_hint = Lp->R.fp32_hint = Ac.fp32_hint = fp32m;
        }
        Anext = std::move(Ac);
        have_next = true;
        B = std::move(Bc);
        bs = k;
    }
    if (tail) {                                    // the redundant tail owns the coarsest level
        coarse_direct = false;
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        return;
    }
    // coarsest level: dense inverse when small enough (gathered on every rank in a distributed hierarchy)
    const int lc = (int)levels.size() - 1;
    const Csr& Ac = op(lc);
    coarse_n_global = rows_global(lc);
    coarse_direct = !par.smoother_only && coarse_n_global <= c.opt_i("-poro_amg_dense_limit", 4096);
    if (coarse_direct && !dist) { Tick t(c, "dense coarse inverse"); dense_inverse(c, Ac, coarse_inv); }
    if (coarse_direct && dist) {
        Tick t(c, "gathered dense coarse inverse");
        const int ng = (int)coarse_n_global;
        DistPlan& pl = *levels[lc]->plan;
        DBuf<double> D((size_t)ng * ng);
        D.zero(c.stream);
        {
            const int* rp = Ac.rowptr.p; const int* cc = Ac.col.p; const double* v = Ac.val.p; const int* gid = pl.ghost_gid.p;
            double* d = D.p; const int no = pl.n_owned, off = (int)pl.offset;
            pfor(c, Ac.nrows, [=] __device__(int64_t i) {
                for (int q = rp[i]; q < rp[i + 1]; ++q) {
                    const int col = cc[q] < no ? off + cc[q] : gid[cc[q] - no];
                    d[(size_t)(off + (int)i) * ng + col] += v[q];
                }
            });
        }
        allreduce_sum(c, D.p, ng * ng);
        DBuf<double> full;
        dense_inverse_full(c, D.p, ng, full);
        coarse_inv.alloc((size_t)pl.n_owned * ng);                       // this rank applies its rows of the inverse
        if (pl.n_owned) PORO_CUDA(cudaMemcpyAsync(coarse_inv.p, full.p + (size_t)pl.offset * ng, (size_t)pl.n_owned * ng * sizeof(double),
                                                  cudaMemcpyDeviceToDevice, c.stream));
        coarse_full.alloc((size_t)ng);
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

double Amg::complexity() const {
    double s = 0.0;
    for (size_t l = 0; l < levels.size(); ++l) s += (double)op((int)l).nnz;
    return s / (double)op(0).nnz;
}

// ---- V-cycle --------------------------------------------------------------------------------
const double* Amg::ext(int l, const double* v) {
    if (!dist) return v;
    Ctx& c = *ctx;
    AmgLevel& L = *levels[l];
    const int n = L.plan->n_owned;
    if (L.replicated && v == L.x.p) return v;      // ghosts were taken from the replicated vector (cycle)
    double* dst;
    if (v == L.x.p || v == L.r.p || v == L.d0.p || v == L.d1.p) dst = const_cast<double*>(v);   // stored extended: halo lands in place
    else { vec_copy(c, L.ext.p, v, n); dst = L.ext.p; }
    dist_halo_vec(c, *L.plan, dst, 1, dst + n);
    return dst;
}

void Amg::cheby(int l, const double* b, double* x, bool zero_guess) {
    Ctx& c = *ctx;
    AmgLevel& L = *levels[l];
    const Csr& A = op(l);
    const int n = A.nrows;
    const double lmax = L.lmax, lmin = lmax / par.cheby_ratio;
    const double theta = 0.5 * (lmax + lmin), delta = 0.5 * (lmax - lmin);
    const double sigma = theta / delta;
    double rho = 1.0 / sigma;
    const int deg = par.cheby_degree;
    double* r = L.r.p;
    double* d_old = L.d0.p;
    double* d_new = L.d1.p;
    const double* dinv = L.dinv.p;
    const double it = 1.0 / theta;
    if (zero_guess) {
        bool need_r = deg > 1;
        pfor(c, n, [=] __device__(int64_t i) {
            double bi = b[i];
            double d = dinv[i] * bi * it;
            d_old[i] = d;
            x[i] = d;
            if (need_r) r[i] = bi;
        });
    } else {
        spmv(c, A, ext(l, x), r, SPMV_SUB, b);
        pfor(c, n, [=] __device__(int64_t i) {
            double d = dinv[i] * r[i] * it;
            d_old[i] = d;
            x[i] += d;
        });
    }
    for (int k = 1; k < deg; ++k) {
        double rho_new = 1.0 / (2.0 * sigma - rho);
        const double* din = ext(l, d_old);
        {
            ProfScope ps(c, (l == 0 && prof_base == 8) ? 37 : -1);       // the launch with the largest share of a solve
            spmv_cheb_step(c, A, din, d_old, d_new, r, x, dinv, rho_new * rho, 2.0 * rho_new / delta);
        }
        rho = rho_new;
        std::swap(d_old, d_new);
    }
}

void Amg::cycle(int l, const double* b, double* x) {
    Ctx& c = *ctx;
    ProfScope ps(c, prof_base >= 0 && l < 8 ? prof_base + l : -1);
    const Csr& A = op(l);
    const int last = (int)levels.size() - 1;
    if (levels[l]->replicated) {
        // one all-gather of the right-hand side, the redundant sub-cycle, then this rank's slice and its ghosts
        DistPlan& pl = *levels[l]->plan;
        dist_allgather_slices(c, b, pl.offsets, tail_b.p);
        tail->cycle(0, tail_b.p, tail_x.p);
        const double* full = tail_x.p; const int* gid = pl.ghost_gid.p; const int no = pl.n_owned; const int64_t off = pl.offset;
        pfor(c, (int64_t)no + pl.n_ghost, [=] __device__(int64_t i) { x[i] = i < no ? full[off + i] : full[gid[i - no]]; });
        return;
    }
    if (l == last) {
        if (coarse_direct && !dist) dense_gemv(c, coarse_inv.p, A.nrows, b, x);
        else if (coarse_direct) {
            // gather the coarsest right-hand side on every rank (one small all-reduce), apply this rank's rows of the inverse
            DistPlan& pl = *levels[l]->plan;
            const int ng = (int)coarse_n_global;
            coarse_full.zero(c.stream);
            vec_copy(c, coarse_full.p + pl.offset, b, pl.n_owned);
            allreduce_sum(c, coarse_full.p, ng);
            dense_gemv_rect(c, coarse_inv.p, pl.n_owned, ng, coarse_full.p, x);
        }
        else if (levels.size() == 1) cheby(l, b, x, true);            // `chebyshev` PC: one sweep of the full degree
        else { cheby(l, b, x, true); cheby(l, b, x, false); }
        return;
    }
    AmgLevel& L = *levels[l];
    AmgLevel& Ln = *levels[l + 1];
    cheby(l, b, x, true);
    spmv(c, A, ext(l, x), L.r.p, SPMV_SUB, b);
    if (L.mg) mg_restrict(c, *L.mg, L.r.p, Ln.b.p);
    else spmv(c, L.R, ext(l, L.r.p), Ln.b.p);                          // restriction reads the ghost residuals
    cycle(l + 1, Ln.b.p, Ln.x.p);
    if (L.mg) mg_prolong(c, *L.mg, ext(l + 1, Ln.x.p), x, true);      // the coarse ghosts the prolongation reads
    else spmv(c, L.P, ext(l + 1, Ln.x.p), x, SPMV_ADD, x);             // prolongation reads the ghost coarse values
    if (par.post_smooth) cheby(l, b, x, false);
}

void Amg::apply(const double* b, double* x) { cycle(0, b, x); }

}  // namespace poro
