// setup.cu -- device-side sparse set-up primitives (run once per solver set-up, not per iteration).
//
// Everything the reference delegates to MatCreateSubMatrix (lib/Preconditioner.py:60-75),
// PETSc's MatMatMult for the `selfp` Schur complement (petsc-options-inexact:80) and hypre's
// set-up (lib/Preconditioner.py:94-100) is expressed through ONE primitive: turn an unsorted
// list of (row, col, value) triples with duplicates into a CSR matrix with sorted unique
// columns (64-bit radix sort + deterministic segmented combine).  SpGEMM expands the
// products and feeds them to it (chunked over rows to bound memory); transpose, sub-matrix
// extraction and matrix addition only differ in how they emit the triples.
#include "common.cuh"
#include <cub/cub.cuh>
#include <algorithm>

namespace poro {

static constexpr int kB = 256;

template <class F>
__global__ void __launch_bounds__(kB) k_for(int64_t n, F f) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) f(i);
}
template <class F>
static void pfor(Ctx& c, int64_t n, F f) {
    if (n <= 0) return;
    int64_t g = (n + kB - 1) / kB;
    int64_t cap = (int64_t)c.sm_count * 16;
    k_for<<<(int)(g < cap ? g : cap), kB, 0, c.stream>>>(n, f);
    PORO_LAUNCH_CHECK(c);
}

static int64_t scan_exclusive_i64(Ctx& c, const int64_t* in, int64_t* out, int64_t n) {
    // out[i] = sum_{j<i} in[j]; returns total (synchronises)
    size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, in, out, n, c.stream);
    DBuf<char> tmp(tb);
    cub::DeviceScan::ExclusiveSum(tmp.p, tb, in, out, n, c.stream);
    c.launches++;
    int64_t last_in = 0, last_out = 0;
    if (n > 0) {
        PORO_CUDA(cudaMemcpyAsync(&last_in, in + n - 1, 8, cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaMemcpyAsync(&last_out, out + n - 1, 8, cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
    }
    return last_in + last_out;
}

// ------------------------------------------------------------------------------------------
// the primitive
// ------------------------------------------------------------------------------------------
void coo_to_csr(Ctx& c, int nrows, int ncols, int64_t nent, DBuf<uint64_t>& keys, DBuf<double>& vals, Csr& out,
                CombineOp op) {
    out.nrows = nrows;
    out.ncols = ncols;
    out.rowptr.alloc((size_t)nrows + 1);
    if (nent == 0) {
        out.nnz = 0;
        out.rowptr.zero(c.stream);
        out.col.alloc(0);
        out.val.alloc(0);
        csr_choose_lanes(out);
        return;
    }
    PORO_REQUIRE(nent < (int64_t)2147483647, "coo_to_csr: more than 2^31 entries in one call");
    // 1. sort by key (stable radix sort: duplicates keep their emission order -> deterministic sums)
    DBuf<uint64_t> keys2((size_t)nent);
    DBuf<double> vals2((size_t)nent);
    {
        cub::DoubleBuffer<uint64_t> kb(keys.p, keys2.p);
        cub::DoubleBuffer<double> vb(vals.p, vals2.p);
        int end_bit = 32;
        for (int64_t r = nrows; r > 1; r >>= 1) end_bit++;
        end_bit = std::min(64, end_bit + 1);
        size_t tb = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tb, kb, vb, (int)nent, 0, end_bit, c.stream);
        DBuf<char> tmp(tb);
        cub::DeviceRadixSort::SortPairs(tmp.p, tb, kb, vb, (int)nent, 0, end_bit, c.stream);
        c.launches++;
        if (kb.Current() != keys.p) { std::swap(keys.p, keys2.p); }
        if (vb.Current() != vals.p) { std::swap(vals.p, vals2.p); }
    }
    // 2. segment heads -> unique index
    DBuf<int64_t> head((size_t)nent), seg((size_t)nent);
    {
        const uint64_t* k = keys.p;
        int64_t* h = head.p;
        pfor(c, nent, [=] __device__(int64_t i) { h[i] = (i == 0 || k[i] != k[i - 1]) ? 1 : 0; });
    }
    int64_t nuniq = scan_exclusive_i64(c, head.p, seg.p, nent);
    PORO_REQUIRE(nuniq < (int64_t)2147483647, "matrix with more than 2^31 nonzeros");
    out.nnz = nuniq;
    out.col.alloc((size_t)nuniq);
    out.val.alloc((size_t)nuniq);
    DBuf<int64_t> segstart((size_t)nuniq + 1);
    {
        const int64_t* h = head.p;
        const int64_t* s = seg.p;
        int64_t* ss = segstart.p;
        int64_t ne = nent, nu = nuniq;
        pfor(c, nent, [=] __device__(int64_t i) {
            if (h[i]) ss[s[i]] = i;
            if (i == ne - 1) ss[nu] = ne;
        });
    }
    // 3. combine each run sequentially (fixed order), write col/val; 4. row pointers by binary search
    {
        const uint64_t* k = keys.p;
        const double* v = vals.p;
        const int64_t* ss = segstart.p;
        int* oc = out.col.p;
        double* ov = out.val.p;
        int cop = (int)op;
        pfor(c, nuniq, [=] __device__(int64_t u) {
            int64_t a = ss[u], b = ss[u + 1];
            double s = v[a];
            for (int64_t i = a + 1; i < b; ++i) s = cop == COMBINE_SUM ? s + v[i] : fmax(s, v[i]);
            oc[u] = (int)(k[a] & 0xffffffffu);
            ov[u] = s;
        });
        int* rp = out.rowptr.p;
        int64_t nu = nuniq;
        pfor(c, (int64_t)nrows + 1, [=] __device__(int64_t r) {
            // first unique entry whose row >= r
            int64_t lo = 0, hi = nu;
            while (lo < hi) {
                int64_t mid = (lo + hi) >> 1;
                int64_t row = (int64_t)(k[ss[mid]] >> 32);
                if (row < r) lo = mid + 1; else hi = mid;
            }
            rp[r] = (int)lo;
        });
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    keys.release();
    vals.release();
    csr_choose_lanes(out);
}

// ------------------------------------------------------------------------------------------
// SpGEMM by expansion, chunked over rows of A
// ------------------------------------------------------------------------------------------
void csr_spgemm(Ctx& c, const Csr& A, const Csr& B, Csr& C, int* chunks) {
    PORO_REQUIRE(A.ncols == B.nrows, "spgemm: inner dimensions differ");
    const int n = A.nrows;
    // products per row of A
    DBuf<int64_t> cnt((size_t)n + 1), off((size_t)n + 1);
    {
        const int* arp = A.rowptr.p; const int* ac = A.col.p; const int* brp = B.rowptr.p;
        int64_t* cn = cnt.p;
        int nn = n;
        pfor(c, (int64_t)n + 1, [=] __device__(int64_t i) {
            int64_t s = 0;
            if (i < nn) for (int k = arp[i]; k < arp[i + 1]; ++k) { int j = ac[k]; s += brp[j + 1] - brp[j]; }
            cn[i] = s;
        });
    }
    scan_exclusive_i64(c, cnt.p, off.p, (int64_t)n + 1);
    std::vector<int64_t> hoff((size_t)n + 1);
    PORO_CUDA(cudaMemcpy(hoff.data(), off.p, ((size_t)n + 1) * 8, cudaMemcpyDeviceToHost));
    const int64_t budget = (int64_t)c.opt_d("poro_spgemm_chunk", 3.0e8);
    std::vector<Csr> parts;
    std::vector<int> part_r0;
    int r0 = 0;
    while (r0 < n) {
        int r1 = r0 + 1;
        // largest r1 with products(r0..r1) <= budget
        {
            int64_t lim = hoff[r0] + budget;
            r1 = (int)(std::upper_bound(hoff.begin() + r0 + 1, hoff.end(), lim) - hoff.begin()) - 1;
            if (r1 <= r0) r1 = r0 + 1;
            if (r1 > n) r1 = n;
        }
        int64_t nent = hoff[r1] - hoff[r0];
        DBuf<uint64_t> keys((size_t)nent);
        DBuf<double> vals((size_t)nent);
        {
            const int* arp = A.rowptr.p; const int* ac = A.col.p; const double* av = A.val.p;
            const int* brp = B.rowptr.p; const int* bc = B.col.p; const double* bv = B.val.p;
            const int64_t* of = off.p;
            uint64_t* kk = keys.p; double* vv = vals.p;
            int64_t base = hoff[r0];
            int rr0 = r0;
            // one warp per row of the chunk; lanes stride over the row of B selected by each a_ik.  The
            // position of every product is a pure function of (i, k, q), so the emission is deterministic.
            int nrows_chunk = r1 - r0;
            pfor(c, (int64_t)nrows_chunk * 32, [=] __device__(int64_t gt) {
                int t = (int)(gt >> 5), lane = (int)(gt & 31);
                int i = rr0 + t;
                int64_t pos = of[i] - base;
                for (int k = arp[i]; k < arp[i + 1]; ++k) {
                    int j = ac[k];
                    double a = av[k];
                    int b0 = brp[j], b1 = brp[j + 1];
                    for (int q = b0 + lane; q < b1; q += 32) {
                        kk[pos + (q - b0)] = ((uint64_t)(uint32_t)t << 32) | (uint32_t)bc[q];
                        vv[pos + (q - b0)] = a * bv[q];
                    }
                    pos += b1 - b0;
                }
            });
        }
        Csr part;
        coo_to_csr(c, r1 - r0, B.ncols, nent, keys, vals, part, COMBINE_SUM);
        parts.push_back(std::move(part));
        part_r0.push_back(r0);
        r0 = r1;
    }
    if (chunks) *chunks = (int)parts.size();
    if (parts.size() == 1) {
        C = std::move(parts[0]);
        C.nrows = n;
        return;
    }
    if (parts.empty()) {                                   // no rows (a rank without coarse dofs)
        C.nrows = n; C.ncols = B.ncols; C.nnz = 0;
        C.rowptr.alloc((size_t)n + 1); C.rowptr.zero(c.stream); C.col.alloc(0); C.val.alloc(0);
        csr_choose_lanes(C);
        return;
    }
    // concatenate row chunks
    int64_t nnz = 0;
    for (auto& p : parts) nnz += p.nnz;
    PORO_REQUIRE(nnz < (int64_t)2147483647, "spgemm result has more than 2^31 nonzeros");
    C.nrows = n; C.ncols = B.ncols; C.nnz = nnz;
    C.rowptr.alloc((size_t)n + 1); C.col.alloc((size_t)nnz); C.val.alloc((size_t)nnz);
    int64_t base = 0;
    for (size_t pi = 0; pi < parts.size(); ++pi) {
        Csr& p = parts[pi];
        int* rp = C.rowptr.p + part_r0[pi];
        const int* prp = p.rowptr.p;
        int b = (int)base;
        bool last = pi + 1 == parts.size();
        pfor(c, (int64_t)p.nrows + (last ? 1 : 0), [=] __device__(int64_t i) { rp[i] = prp[i] + b; });
        if (p.nnz) {
            PORO_CUDA(cudaMemcpyAsync(C.col.p + base, p.col.p, p.nnz * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
            PORO_CUDA(cudaMemcpyAsync(C.val.p + base, p.val.p, p.nnz * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
        }
        base += p.nnz;
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    csr_choose_lanes(C);
}

// expands row index per nonzero
static void csr_rows(Ctx& c, const Csr& A, int* rows) {
    const int* rp = A.rowptr.p;
    pfor(c, A.nrows, [=] __device__(int64_t i) { for (int k = rp[i]; k < rp[i + 1]; ++k) rows[k] = (int)i; });
}

void csr_transpose(Ctx& c, const Csr& A, Csr& At) {
    DBuf<uint64_t> keys((size_t)A.nnz);
    DBuf<double> vals((size_t)A.nnz);
    DBuf<int> rows((size_t)A.nnz);
    csr_rows(c, A, rows.p);
    {
        const int* r = rows.p; const int* cc = A.col.p; const double* v = A.val.p;
        uint64_t* kk = keys.p; double* vv = vals.p;
        pfor(c, A.nnz, [=] __device__(int64_t k) { kk[k] = ((uint64_t)(uint32_t)cc[k] << 32) | (uint32_t)r[k]; vv[k] = v[k]; });
    }
    coo_to_csr(c, A.ncols, A.nrows, A.nnz, keys, vals, At, COMBINE_SUM);
}

void csr_extract(Ctx& c, const Csr& A, const int* row_map, const int* col_map, int new_rows, int new_cols, Csr& C) {
    // count kept entries, compact, then sort
    DBuf<int> rows((size_t)A.nnz);
    csr_rows(c, A, rows.p);
    DBuf<int64_t> keep((size_t)A.nnz + 1), pos((size_t)A.nnz + 1);
    {
        const int* r = rows.p; const int* cc = A.col.p;
        int64_t* kp = keep.p;
        int64_t nz = A.nnz;
        pfor(c, A.nnz + 1, [=] __device__(int64_t k) {
            kp[k] = (k < nz && row_map[r[k]] >= 0 && col_map[cc[k]] >= 0) ? 1 : 0;
        });
    }
    int64_t nkeep = scan_exclusive_i64(c, keep.p, pos.p, A.nnz + 1);
    DBuf<uint64_t> keys((size_t)nkeep);
    DBuf<double> vals((size_t)nkeep);
    {
        const int* r = rows.p; const int* cc = A.col.p; const double* v = A.val.p;
        const int64_t* kp = keep.p; const int64_t* ps = pos.p;
        uint64_t* kk = keys.p; double* vv = vals.p;
        pfor(c, A.nnz, [=] __device__(int64_t k) {
            if (kp[k]) {
                kk[ps[k]] = ((uint64_t)(uint32_t)row_map[r[k]] << 32) | (uint32_t)col_map[cc[k]];
                vv[ps[k]] = v[k];
            }
        });
    }
    coo_to_csr(c, new_rows, new_cols, nkeep, keys, vals, C, COMBINE_SUM);
}

// inside = true : C = A[r0:r1, c0:c1]  (rows and columns renumbered from 0)
// inside = false: C = A with the entries of the rectangle [r0:r1) x [c0:c1) removed (same shape)
// Order-preserving (count / scan / fill), no sort needed.
void csr_select(Ctx& c, const Csr& A, int r0, int r1, int c0, int c1, bool inside, Csr& C) {
    const int nr = inside ? r1 - r0 : A.nrows;
    const int rbase = inside ? r0 : 0;
    DBuf<int64_t> cnt((size_t)nr + 1), off((size_t)nr + 1);
    {
        const int* rp = A.rowptr.p; const int* cc = A.col.p;
        int64_t* cn = cnt.p;
        pfor(c, (int64_t)nr + 1, [=] __device__(int64_t t) {
            int64_t s = 0;
            if (t < nr) {
                const int i = rbase + (int)t;
                const bool rin = i >= r0 && i < r1;
                for (int k = rp[i]; k < rp[i + 1]; ++k) {
                    const bool in = rin && cc[k] >= c0 && cc[k] < c1;
                    s += (in == inside) ? 1 : 0;
                }
            }
            cn[t] = s;
        });
    }
    int64_t nnz = scan_exclusive_i64(c, cnt.p, off.p, (int64_t)nr + 1);
    PORO_REQUIRE(nnz < (int64_t)2147483647, "csr_select: too many nonzeros");
    C.nrows = nr;
    C.ncols = inside ? c1 - c0 : A.ncols;
    C.nnz = nnz;
    C.rowptr.alloc((size_t)nr + 1);
    C.col.alloc((size_t)nnz);
    C.val.alloc((size_t)nnz);
    {
        const int* rp = A.rowptr.p; const int* cc = A.col.p; const double* v = A.val.p;
        const int64_t* of = off.p;
        int* orp = C.rowptr.p; int* oc = C.col.p; double* ov = C.val.p;
        const int cshift = inside ? c0 : 0;
        pfor(c, (int64_t)nr + 1, [=] __device__(int64_t t) {
            orp[t] = (int)of[t];
            if (t < nr) {
                const int i = rbase + (int)t;
                const bool rin = i >= r0 && i < r1;
                int64_t p = of[t];
                for (int k = rp[i]; k < rp[i + 1]; ++k) {
                    const bool in = rin && cc[k] >= c0 && cc[k] < c1;
                    if (in == inside) { oc[p] = cc[k] - cshift; ov[p] = v[k]; ++p; }
                }
            }
        });
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    csr_choose_lanes(C);
}

void csr_diag(Ctx& c, const Csr& A, double* d) {
    const int* rp = A.rowptr.p; const int* cc = A.col.p; const double* v = A.val.p;
    pfor(c, A.nrows, [=] __device__(int64_t i) {
        double s = 0.0;
        for (int k = rp[i]; k < rp[i + 1]; ++k) if (cc[k] == (int)i) s += v[k];
        d[i] = s;
    });
}

void csr_copy(Ctx& c, const Csr& A, Csr& B) {
    B.nrows = A.nrows; B.ncols = A.ncols; B.nnz = A.nnz; B.lanes = A.lanes;
    B.rowptr.alloc((size_t)A.nrows + 1); B.col.alloc((size_t)A.nnz); B.val.alloc((size_t)A.nnz);
    PORO_CUDA(cudaMemcpyAsync(B.rowptr.p, A.rowptr.p, ((size_t)A.nrows + 1) * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
    if (A.nnz) {
        PORO_CUDA(cudaMemcpyAsync(B.col.p, A.col.p, A.nnz * sizeof(int), cudaMemcpyDeviceToDevice, c.stream));
        PORO_CUDA(cudaMemcpyAsync(B.val.p, A.val.p, A.nnz * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
    }
}

void csr_add_scaled(Ctx& c, const Csr& A, const Csr& B, double alpha, const double* s, Csr& C) {
    PORO_REQUIRE(A.nrows == B.nrows && A.ncols == B.ncols, "csr_add: shapes differ");
    int64_t nent = A.nnz + B.nnz;
    DBuf<uint64_t> keys((size_t)nent);
    DBuf<double> vals((size_t)nent);
    DBuf<int> ra((size_t)A.nnz), rb((size_t)B.nnz);
    csr_rows(c, A, ra.p);
    csr_rows(c, B, rb.p);
    {
        const int* r = ra.p; const int* cc = A.col.p; const double* v = A.val.p;
        uint64_t* kk = keys.p; double* vv = vals.p;
        pfor(c, A.nnz, [=] __device__(int64_t k) { kk[k] = ((uint64_t)(uint32_t)r[k] << 32) | (uint32_t)cc[k]; vv[k] = v[k]; });
    }
    {
        const int* r = rb.p; const int* cc = B.col.p; const double* v = B.val.p;
        uint64_t* kk = keys.p + A.nnz; double* vv = vals.p + A.nnz;
        pfor(c, B.nnz, [=] __device__(int64_t k) {
            kk[k] = ((uint64_t)(uint32_t)r[k] << 32) | (uint32_t)cc[k];
            vv[k] = alpha * (s ? s[r[k]] : 1.0) * v[k];
        });
    }
    coo_to_csr(c, A.nrows, A.ncols, nent, keys, vals, C, COMBINE_SUM);
}

void csr_scale_cols(Ctx& c, Csr& A, const double* s) {
    const int* cc = A.col.p; double* v = A.val.p;
    pfor(c, A.nnz, [=] __device__(int64_t k) { v[k] *= s[cc[k]]; });
}

void csr_to_host(const Csr& A, std::vector<int>& rp, std::vector<int>& ci, std::vector<double>& v) {
    rp.resize((size_t)A.nrows + 1); ci.resize((size_t)A.nnz); v.resize((size_t)A.nnz);
    PORO_CUDA(cudaMemcpy(rp.data(), A.rowptr.p, rp.size() * sizeof(int), cudaMemcpyDeviceToHost));
    if (A.nnz) {
        PORO_CUDA(cudaMemcpy(ci.data(), A.col.p, ci.size() * sizeof(int), cudaMemcpyDeviceToHost));
        PORO_CUDA(cudaMemcpy(v.data(), A.val.p, v.size() * sizeof(double), cudaMemcpyDeviceToHost));
    }
}

void csr_from_host(Ctx& c, int nrows, int ncols, const int64_t* rp, const int* ci, const double* v, Csr& out) {
    int64_t nnz = rp[nrows];
    PORO_REQUIRE(nnz < (int64_t)2147483647, "local matrix has more than 2^31 nonzeros: shard it over more GPUs");
    std::vector<int> rp32((size_t)nrows + 1);
    for (int i = 0; i <= nrows; ++i) rp32[i] = (int)rp[i];
    out.nrows = nrows; out.ncols = ncols; out.nnz = nnz;
    out.rowptr.alloc((size_t)nrows + 1); out.col.alloc((size_t)nnz); out.val.alloc((size_t)nnz);
    PORO_CUDA(cudaMemcpyAsync(out.rowptr.p, rp32.data(), rp32.size() * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    if (nnz) {
        PORO_CUDA(cudaMemcpyAsync(out.col.p, ci, nnz * sizeof(int), cudaMemcpyHostToDevice, c.stream));
        PORO_CUDA(cudaMemcpyAsync(out.val.p, v, nnz * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    csr_choose_lanes(out);
}

// ------------------------------------------------------------------------------------------
// dense inverse (coarsest AMG level, small `lu` blocks): Gauss-Jordan with partial pivoting
// on the augmented matrix [A | I], row-major, one column step = 3 small kernels.
// ------------------------------------------------------------------------------------------
__global__ void k_gj_pivot(const double* __restrict__ M, int n, int ld, int k, int* __restrict__ piv) {
    __shared__ double bv[256];
    __shared__ int bi[256];
    double best = -1.0;
    int idx = k;
    for (int i = k + threadIdx.x; i < n; i += 256) {
        double a = fabs(M[(size_t)i * ld + k]);
        if (a > best) { best = a; idx = i; }
    }
    bv[threadIdx.x] = best;
    bi[threadIdx.x] = idx;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            if (bv[threadIdx.x + s] > bv[threadIdx.x] ||
                (bv[threadIdx.x + s] == bv[threadIdx.x] && bi[threadIdx.x + s] < bi[threadIdx.x])) {
                bv[threadIdx.x] = bv[threadIdx.x + s];
                bi[threadIdx.x] = bi[threadIdx.x + s];
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) *piv = bi[0];
}

__global__ void k_gj_colk(const double* __restrict__ M, int n, int ld, int k, double* __restrict__ colk) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        colk[i] = i == k ? 0.0 : M[(size_t)i * ld + k];
}

__global__ void k_gj_swap(double* __restrict__ M, int ld, int k, const int* __restrict__ piv) {
    int p = *piv;
    if (p == k) return;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < ld; j += gridDim.x * blockDim.x) {
        double a = M[(size_t)k * ld + j];
        M[(size_t)k * ld + j] = M[(size_t)p * ld + j];
        M[(size_t)p * ld + j] = a;
    }
}

__global__ void k_gj_scale(double* __restrict__ M, int ld, int k, double* __restrict__ pivval) {
    // pivval holds M[k][k] read by a previous kernel
    double pv = *pivval;
    double inv = pv != 0.0 ? 1.0 / pv : 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < ld; j += gridDim.x * blockDim.x) M[(size_t)k * ld + j] *= inv;
}

__global__ void k_gj_readpiv(const double* __restrict__ M, int ld, int k, double* __restrict__ pivval) {
    *pivval = M[(size_t)k * ld + k];
}

__global__ void k_gj_elim(double* __restrict__ M, int n, int ld, int k, const double* __restrict__ colk) {
    // M[i,:] -= colk[i] * M[k,:] for all i != k (colk[k] == 0)
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ld) return;
    double rk = M[(size_t)k * ld + j];
    if (rk == 0.0) return;
    for (int i = blockIdx.y; i < n; i += gridDim.y) {
        double f = colk[i];
        if (f != 0.0) M[(size_t)i * ld + j] -= f * rk;
    }
}

static void gauss_jordan(Ctx& c, DBuf<double>& M, int n, DBuf<double>& inv);

void dense_inverse(Ctx& c, const Csr& A, DBuf<double>& inv) {
    const int n = A.nrows;
    PORO_REQUIRE(n == A.ncols, "dense_inverse: square matrix expected");
    const int ld = 2 * n;
    DBuf<double> M((size_t)n * ld);
    M.zero(c.stream);
    {
        const int* rp = A.rowptr.p; const int* cc = A.col.p; const double* v = A.val.p;
        double* m = M.p;
        int nn = n, l = ld;
        pfor(c, n, [=] __device__(int64_t i) {
            for (int k = rp[i]; k < rp[i + 1]; ++k) m[(size_t)i * l + cc[k]] += v[k];
            m[(size_t)i * l + nn + i] = 1.0;
        });
    }
    gauss_jordan(c, M, n, inv);
}

// same from a dense row-major n x n matrix (the gathered coarsest operator of a distributed hierarchy)
void dense_inverse_full(Ctx& c, const double* Ad, int n, DBuf<double>& inv) {
    const int ld = 2 * n;
    DBuf<double> M((size_t)n * ld);
    {
        double* m = M.p;
        int nn = n, l = ld;
        pfor(c, (int64_t)n * ld, [=] __device__(int64_t t) {
            const int i = (int)(t / l), j = (int)(t % l);
            m[t] = j < nn ? Ad[(size_t)i * nn + j] : (j - nn == i ? 1.0 : 0.0);
        });
    }
    gauss_jordan(c, M, n, inv);
}

static void gauss_jordan(Ctx& c, DBuf<double>& M, int n, DBuf<double>& inv) {
    const int ld = 2 * n;
    DBuf<int> piv(1);
    DBuf<double> colk((size_t)n), pivval(1);
    int gx = ceil_div(ld, 256);
    int gy = std::min(n, std::max(1, (c.sm_count * 8) / gx));
    for (int k = 0; k < n; ++k) {
        k_gj_pivot<<<1, 256, 0, c.stream>>>(M.p, n, ld, k, piv.p);
        k_gj_swap<<<gx, 256, 0, c.stream>>>(M.p, ld, k, piv.p);
        k_gj_readpiv<<<1, 1, 0, c.stream>>>(M.p, ld, k, pivval.p);
        k_gj_scale<<<gx, 256, 0, c.stream>>>(M.p, ld, k, pivval.p);
        k_gj_colk<<<ceil_div(n, 256), 256, 0, c.stream>>>(M.p, n, ld, k, colk.p);
        k_gj_elim<<<dim3(gx, gy), 256, 0, c.stream>>>(M.p, n, ld, k, colk.p);
        c.launches += 6;
    }
    PORO_CUDA(cudaGetLastError());
    inv.alloc((size_t)n * n);
    PORO_CUDA(cudaMemcpy2DAsync(inv.p, (size_t)n * sizeof(double), M.p + n, (size_t)ld * sizeof(double),
                                (size_t)n * sizeof(double), n, cudaMemcpyDeviceToDevice, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

// y = M x, M row-major nrows x n: one warp per row
__global__ void __launch_bounds__(256) k_gemv(const double* __restrict__ M, int nrows, int n, const double* __restrict__ x,
                                              double* __restrict__ y) {
    int row = (blockIdx.x * 256 + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (row >= nrows) return;
    const double* r = M + (size_t)row * n;
    double s = 0.0;
    for (int j = lane; j < n; j += 32) s = fma(r[j], x[j], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) y[row] = s;
}

void dense_gemv(Ctx& c, const double* M, int n, const double* x, double* y) { dense_gemv_rect(c, M, n, n, x, y); }

void dense_gemv_rect(Ctx& c, const double* M, int nrows, int ncols, const double* x, double* y) {
    if (nrows == 0) return;
    k_gemv<<<ceil_div((int64_t)nrows * 32, 256), 256, 0, c.stream>>>(M, nrows, ncols, x, y);
    PORO_LAUNCH_CHECK(c);
}

}  // namespace poro
