// ilu.cu -- PCIlu: ILU(0) of one inner block (ilu.cuh).
//
//   set-up   host: sorted-pattern check, diagonal positions, level sets of the lower and upper dependency graphs.
//            device: IKJ factorisation in place on a copy of the values, one launch per lower level, one warp per row:
//            for each stored k < i (ascending) a_ik /= u_kk, then the lanes walk row k's upper part and update a_ij wherever
//            (i, j) is stored (binary search in row i).  Each a_ij is updated in the fixed order of k and nothing is
//            accumulated across warps, so two set-ups give the same bits.  A pivot with |u_ii| <= zeropivot sets a flag
//            (the smallest such row) that the host reads once.  The factor is then split into L, U and 1/u_ii.
//   apply    forward substitution y = L^-1 x, one launch per lower level, then backward substitution y = U^-1 y in place,
//            one launch per upper level; a G-lane group per row sums its row in a fixed lane order and tree.
#include "ilu.cuh"
#include <climits>
#include <cmath>

namespace poro {

namespace {

constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads) k_ilu_factor_level(const int* __restrict__ rows, int count, const int* __restrict__ rp,
                                                               const int* __restrict__ ci, const int* __restrict__ dpos,
                                                               double* F, double tol, int* __restrict__ bad) {
    const int w = (int)(((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= count) return;                      // whole warps: every lane of a warp has the same row
    const int i = rows[w];
    const int e = rp[i + 1], di = dpos[i];
    for (int q = rp[i]; q < di; ++q) {
        const int k = ci[q];
        const double l = F[q] / F[dpos[k]];      // row k belongs to an earlier level: final
        __syncwarp();
        if (lane == 0) F[q] = l;
        for (int t = dpos[k] + 1 + lane; t < rp[k + 1]; t += 32) {
            const int j = ci[t];
            int lo = q + 1, hi = e - 1;
            while (lo <= hi) {
                const int mid = (lo + hi) >> 1, cm = ci[mid];
                if (cm == j) { F[mid] -= l * F[t]; break; }
                if (cm < j) lo = mid + 1; else hi = mid - 1;
            }
        }
        __syncwarp();                            // the next a_ik may just have been updated by another lane
    }
    if (lane == 0 && !(fabs(F[di]) > tol)) atomicMin(bad, i);
}

__global__ void __launch_bounds__(kThreads) k_ilu_split(int n, const int* __restrict__ rp, const int* __restrict__ dpos,
                                                        const double* __restrict__ F, const int* __restrict__ lrp,
                                                        double* __restrict__ lval, const int* __restrict__ urp,
                                                        double* __restrict__ uval, double* __restrict__ dinv) {
    const int i = blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    const int d = dpos[i];
    for (int q = rp[i]; q < d; ++q) lval[lrp[i] + q - rp[i]] = F[q];
    for (int q = d + 1; q < rp[i + 1]; ++q) uval[urp[i] + q - d - 1] = F[q];
    dinv[i] = 1.0 / F[d];
}

// one level of y_i = x_i - sum_j L_ij y_j (UPPER = false) or y_i = dinv_i (y_i - sum_j U_ij y_j) (UPPER = true, in place).
// y is read at other rows and written at this level's rows: no __restrict__ on it.
template <int G, bool UPPER>
__global__ void __launch_bounds__(kThreads) k_ilu_solve_level(const int* __restrict__ rows, int count, const int* __restrict__ rp,
                                                              const int* __restrict__ ci, const double* __restrict__ v,
                                                              const double* __restrict__ x, const double* __restrict__ dinv,
                                                              double* y) {
    const int g = (int)(((int64_t)blockIdx.x * kThreads + threadIdx.x) / G), lane = threadIdx.x & (G - 1);
    const bool on = g < count;                   // no early return: the shuffles below name the whole warp
    const int i = on ? rows[g] : 0;
    double s = 0.0;
    if (on)
        for (int q = rp[i] + lane; q < rp[i + 1]; q += G) s = fma(v[q], y[ci[q]], s);
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o, G);
    if (on && lane == 0) y[i] = UPPER ? dinv[i] * (y[i] - s) : x[i] - s;
}

int lanes_for(int64_t nnz, int n) {
    const double avg = n ? (double)nnz / n : 0.0;
    return avg <= 6.0 ? 4 : avg <= 12.0 ? 8 : avg <= 24.0 ? 16 : 32;
}

template <bool UPPER>
void solve_levels(Ctx& c, int G, const std::vector<int>& ptr, const int* rows, const Csr& T, const double* x, const double* dinv,
                  double* y) {
    for (size_t l = 0; l + 1 < ptr.size(); ++l) {
        const int cnt = ptr[l + 1] - ptr[l];
        const int grid = ceil_div((int64_t)cnt * G, kThreads);
        const int* r = rows + ptr[l];
        switch (G) {
            case 4: k_ilu_solve_level<4, UPPER><<<grid, kThreads, 0, c.stream>>>(r, cnt, T.rowptr.p, T.col.p, T.val.p, x, dinv, y); break;
            case 8: k_ilu_solve_level<8, UPPER><<<grid, kThreads, 0, c.stream>>>(r, cnt, T.rowptr.p, T.col.p, T.val.p, x, dinv, y); break;
            case 16: k_ilu_solve_level<16, UPPER><<<grid, kThreads, 0, c.stream>>>(r, cnt, T.rowptr.p, T.col.p, T.val.p, x, dinv, y); break;
            default: k_ilu_solve_level<32, UPPER><<<grid, kThreads, 0, c.stream>>>(r, cnt, T.rowptr.p, T.col.p, T.val.p, x, dinv, y); break;
        }
        PORO_LAUNCH_CHECK(c);
    }
}

template <class T>
void upload(DBuf<T>& d, const std::vector<T>& h) {
    d.alloc(h.size());
    if (!h.empty()) PORO_CUDA(cudaMemcpy(d.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
}

}  // namespace

void ilu_level_sets(int n, const int* rp, const int* ci, bool upper, std::vector<int>& ptr, std::vector<int>& rows) {
    std::vector<int> lev((size_t)n, 0);
    int nlev = n ? 1 : 0;
    for (int s = 0; s < n; ++s) {
        const int i = upper ? n - 1 - s : s;
        int m = -1;
        for (int q = rp[i]; q < rp[i + 1]; ++q)
            if (upper ? ci[q] > i : ci[q] < i) m = std::max(m, lev[ci[q]]);
        lev[i] = m + 1;
        nlev = std::max(nlev, m + 2);
    }
    ptr.assign((size_t)nlev + 1, 0);
    for (int i = 0; i < n; ++i) ptr[lev[i] + 1]++;
    for (int l = 0; l < nlev; ++l) ptr[l + 1] += ptr[l];
    rows.assign((size_t)n, 0);
    std::vector<int> fill(ptr.begin(), ptr.end() - 1);
    for (int i = 0; i < n; ++i) rows[fill[lev[i]]++] = i;          // ascending rows inside a level
}

PCIlu::PCIlu(Ctx* c_, const Csr& A, const std::string& prefix, const std::string& opt, bool bj) : ctx(c_), n(A.nrows), bjacobi(bj) {
    Ctx& c = *ctx;
    const std::string who = "-" + prefix + "pc_type " + (bj ? "bjacobi" : "ilu");
    auto key = [&](const char* k) { return "-" + opt + k; };
    if (c.has_opt(key("pc_factor_levels")) && c.opt_i(key("pc_factor_levels"), 0) != 0)
        throw Error(who + ": only ILU(0) is implemented; " + key("pc_factor_levels") + " " + c.opt(key("pc_factor_levels"), "") +
                    " is not supported");
    const std::string ord = c.opt(key("pc_factor_mat_ordering_type"), "natural");
    if (ord != "natural")
        throw Error(who + ": ILU(0) factors in the natural ordering only; " + key("pc_factor_mat_ordering_type") + " " + ord +
                    " is not supported");
    const std::string shift = c.opt(key("pc_factor_shift_type"), "none");
    if (shift != "none" && shift != "NONE")
        throw Error(who + ": pivot shifts are not implemented; " + key("pc_factor_shift_type") + " " + shift + " is not supported");
    // PETSc's default zero-pivot threshold as we understand it (100 x double epsilon; not checked against a PETSc build)
    const double tol = c.opt_d(key("pc_factor_zeropivot"), 2.220446049250313e-14);
    PORO_REQUIRE(A.nrows == A.ncols, who + ": the block must be square");

    // ---- symbolic, host ----
    std::vector<int> rp, ci;
    std::vector<double> val;
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    csr_to_host(A, rp, ci, val);
    std::vector<int> dpos((size_t)n, -1), lrp((size_t)n + 1, 0), urp((size_t)n + 1, 0);
    for (int i = 0; i < n; ++i) {
        for (int q = rp[i]; q < rp[i + 1]; ++q) {
            PORO_REQUIRE(q == rp[i] || ci[q] > ci[q - 1], who + ": the columns of row " + std::to_string(i) + " are not sorted");
            if (ci[q] == i) dpos[i] = q;
        }
        if (dpos[i] < 0)
            throw Error(who + ": row " + std::to_string(i) + " of the block has no stored diagonal entry (ILU(0) factors the "
                        "stored pattern and needs every diagonal)");
        lrp[i + 1] = lrp[i] + (dpos[i] - rp[i]);
        urp[i + 1] = urp[i] + (rp[i + 1] - dpos[i] - 1);
    }
    std::vector<int> lr, ur;
    ilu_level_sets(n, rp.data(), ci.data(), false, lptr, lr);
    ilu_level_sets(n, rp.data(), ci.data(), true, uptr, ur);
    std::vector<int> lc((size_t)lrp[n]), uc((size_t)urp[n]);
    for (int i = 0; i < n; ++i) {
        std::copy(ci.begin() + rp[i], ci.begin() + dpos[i], lc.begin() + lrp[i]);
        std::copy(ci.begin() + dpos[i] + 1, ci.begin() + rp[i + 1], uc.begin() + urp[i]);
    }
    L.nrows = L.ncols = U.nrows = U.ncols = n;
    L.nnz = lrp[n];
    U.nnz = urp[n];
    upload(L.rowptr, lrp); upload(L.col, lc); L.val.alloc((size_t)L.nnz);
    upload(U.rowptr, urp); upload(U.col, uc); U.val.alloc((size_t)U.nnz);
    upload(lrows, lr);
    upload(urows, ur);
    dinv.alloc((size_t)n);
    gl = lanes_for(L.nnz, n);
    gu = lanes_for(U.nnz, n);

    // ---- numeric, device ----
    if (n > 0) {
        DBuf<int> d_dpos, d_bad(1);
        upload(d_dpos, dpos);
        DBuf<double> F((size_t)A.nnz);
        if (A.nnz) PORO_CUDA(cudaMemcpyAsync(F.p, A.val.p, (size_t)A.nnz * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
        const int none = INT_MAX;
        PORO_CUDA(cudaMemcpyAsync(d_bad.p, &none, sizeof(int), cudaMemcpyHostToDevice, c.stream));
        for (size_t l = 0; l + 1 < lptr.size(); ++l) {
            const int cnt = lptr[l + 1] - lptr[l];
            k_ilu_factor_level<<<ceil_div((int64_t)cnt * 32, kThreads), kThreads, 0, c.stream>>>(
                lrows.p + lptr[l], cnt, A.rowptr.p, A.col.p, d_dpos.p, F.p, tol, d_bad.p);
            PORO_LAUNCH_CHECK(c);
        }
        k_ilu_split<<<ceil_div(n, kThreads), kThreads, 0, c.stream>>>(n, A.rowptr.p, d_dpos.p, F.p, L.rowptr.p, L.val.p, U.rowptr.p,
                                                                     U.val.p, dinv.p);
        PORO_LAUNCH_CHECK(c);
        int bad = none;
        PORO_CUDA(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        std::vector<double> hd((size_t)n);
        PORO_CUDA(cudaMemcpyAsync(hd.data(), dinv.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        if (bad != none) {
            char buf[160];
            snprintf(buf, sizeof buf, "|u_ii| = %.6e <= %.6g", std::fabs(1.0 / hd[bad]), tol);
            throw Error(who + ": zero pivot in row " + std::to_string(bad) + " of the block: " + buf + " (" +
                        key("pc_factor_zeropivot") + ")");
        }
        min_pivot = INFINITY;
        for (double d : hd) min_pivot = std::min(min_pivot, std::fabs(1.0 / d));
    }
    device_bytes = (int64_t)(L.nnz + U.nnz) * 12 + 8 * ((int64_t)n + 1) + 8 * (int64_t)n + 8 * (int64_t)n;
    // one application: L and U once (8 B value + 4 B column per entry, row pointers), the two row lists, 1/u_ii, x read once,
    // y written by both sweeps and read at its own row by the backward one, and the gathered y_j counted once per row (a lower
    // bound: each y_j is gathered by every row that stores column j)
    apply_bytes = (int64_t)(L.nnz + U.nnz) * 12 + 8 * ((int64_t)n + 1) + 8 * (int64_t)n + 8 * (int64_t)n + 5 * 8 * (int64_t)n;
}

void PCIlu::apply(const double* x, double* y) {
    Ctx& c = *ctx;
    if (n == 0) return;
    solve_levels<false>(c, gl, lptr, lrows.p, L, x, nullptr, y);
    solve_levels<true>(c, gu, uptr, urows.p, U, nullptr, dinv.p, y);
}

}  // namespace poro
