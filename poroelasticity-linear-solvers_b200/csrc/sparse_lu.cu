// sparse_lu.cu -- PCSparseLU: multifrontal sparse LU of one inner block, factorised once at set-up and applied by
// supernodal triangular solves (the exact-block `preonly + lu` of the reference above -poro_dense_lu_limit rows, selected
// by -<prefix>pc_factor_mat_solver_type poro).
//
//   set-up   host: lu_symbolic.h (ordering, supernodes, front maps, level schedule); device, per tree level, leaves first:
//            small fronts one CTA each (extend-add of the children in a fixed order + unblocked LU), large fronts by a blocked
//            right-looking LU (diagonal-block kernel, panel kernel, register-tiled fp64 GEMM for the trailing update).
//            No pivoting: the blocks are SPD or positive-real; a pivot below sqrt(eps) times the largest entry of its row and
//            column of B is replaced (static pivoting) and counted.  The scale is per pivot because the fp block mixes rows of
//            very different size (velocity rows ~1, pressure rows ~1e-5 in swelling): against max|B| the legitimate
//            pressure pivots would all count as tiny.  No floating-point atomics anywhere: two set-ups give bitwise identical factors.
//   apply    permute, forward substitution leaves up (one launch per level, one CTA per supernode; a supernode gathers its
//            children's update vectors in a fixed order), backward substitution root down (one launch per level), inverse
//            permutation.  A fixed launch sequence without host synchronisation: PCBlockCC captures it in its CUDA graph.
#include "lu_symbolic.h"
#include "solver.cuh"
#include <cmath>

namespace poro {

namespace {

constexpr int kThreads = 256;
constexpr int kSmallFront = 256;   // fronts with more rows take the blocked path
constexpr int kNB = 32;            // panel width of the blocked path
constexpr int kTile = 64;          // GEMM tile (kTile x kTile outputs per CTA, 4 x 4 per thread)

__global__ void __launch_bounds__(kThreads) k_scatter_entries(int64_t nnz, const double* __restrict__ val,
                                                              const int64_t* __restrict__ pos, double* __restrict__ F) {
    const int64_t q = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (q < nnz) F[pos[q]] = val[q];       // every entry has its own position: a store, not an accumulation
}

__device__ __forceinline__ double perturb(double p, double scale, int* npert) {
    const double tau = 1.4901161193847656e-08 * scale;     // sqrt(eps) scale
    if (fabs(p) < tau) {
        atomicAdd(npert, 1);
        return p < 0.0 ? -tau : tau;
    }
    return p;
}

// children's update blocks into the front of `S`, in the fixed order of the child list (one child at a time)
__device__ void extend_add_cta(const SluNode& S, const SluNode* __restrict__ sn, double* __restrict__ F_all,
                               const int* __restrict__ relmap, const int* __restrict__ child) {
    double* F = F_all + S.front;
    for (int ci = S.child_begin; ci < S.child_end; ++ci) {
        const SluNode C = sn[child[ci]];
        const int u = C.m - C.k;
        const double* Fc = F_all + C.front;
        const int* rel = relmap + C.upd;
        for (int64_t e = threadIdx.x; e < (int64_t)u * u; e += blockDim.x) {
            const int a = (int)(e % u), b = (int)(e / u);
            F[(int64_t)rel[b] * S.m + rel[a]] += Fc[(int64_t)(C.k + b) * C.m + C.k + a];
        }
        __syncthreads();
    }
}

// one CTA per small front of a level: extend-add, then right-looking LU of the k pivot columns (Schur update of F22 included)
__global__ void __launch_bounds__(kThreads) k_front_small(const int* __restrict__ list, const SluNode* __restrict__ sn,
                                                          double* __restrict__ F_all, const int* __restrict__ relmap,
                                                          const int* __restrict__ child, const double* __restrict__ pscale,
                                                          int* npert) {
    const SluNode S = sn[list[blockIdx.x]];
    extend_add_cta(S, sn, F_all, relmap, child);
    double* F = F_all + S.front;
    const int m = S.m;
    __shared__ double piv;
    for (int j = 0; j < S.k; ++j) {
        if (threadIdx.x == 0) {
            piv = perturb(F[(int64_t)j * m + j], pscale[S.first + j], npert);
            F[(int64_t)j * m + j] = piv;
        }
        __syncthreads();
        const double p = piv;
        for (int i = j + 1 + threadIdx.x; i < m; i += blockDim.x) F[(int64_t)j * m + i] /= p;
        __syncthreads();
        const int r = m - j - 1;
        for (int64_t e = threadIdx.x; e < (int64_t)r * r; e += blockDim.x) {
            const int i = j + 1 + (int)(e % r), c = j + 1 + (int)(e / r);
            F[(int64_t)c * m + i] -= F[(int64_t)j * m + i] * F[(int64_t)c * m + j];
        }
        __syncthreads();
    }
}

// large front: one child's update block (one launch per child keeps the accumulation order fixed)
__global__ void __launch_bounds__(kThreads) k_extend_add_one(double* __restrict__ F, int m, const double* __restrict__ Fc,
                                                             int cm, int ck, const int* __restrict__ rel) {
    const int u = cm - ck;
    const int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (e >= (int64_t)u * u) return;
    const int a = (int)(e % u), b = (int)(e / u);
    F[(int64_t)rel[b] * m + rel[a]] += Fc[(int64_t)(ck + b) * cm + ck + a];
}

// large front: LU of the nb x nb diagonal block at (j0, j0), in place
__global__ void __launch_bounds__(kThreads) k_panel_diag(double* __restrict__ F, int m, int j0, int nb,
                                                         const double* __restrict__ pscale, int* npert) {
    __shared__ double D[kNB][kNB + 1];       // D[col][row]
    for (int e = threadIdx.x; e < nb * nb; e += blockDim.x) D[e / nb][e % nb] = F[(int64_t)(j0 + e / nb) * m + j0 + e % nb];
    __syncthreads();
    for (int j = 0; j < nb; ++j) {
        if (threadIdx.x == 0) D[j][j] = perturb(D[j][j], pscale[j0 + j], npert);
        __syncthreads();
        for (int i = j + 1 + threadIdx.x; i < nb; i += blockDim.x) D[j][i] /= D[j][j];
        __syncthreads();
        const int r = nb - j - 1;
        for (int e = threadIdx.x; e < r * r; e += blockDim.x) {
            const int i = j + 1 + e % r, c = j + 1 + e / r;
            D[c][i] -= D[j][i] * D[c][j];
        }
        __syncthreads();
    }
    for (int e = threadIdx.x; e < nb * nb; e += blockDim.x) F[(int64_t)(j0 + e / nb) * m + j0 + e % nb] = D[e / nb][e % nb];
}

// large front: L21 = A21 U11^-1 (rows below the panel) and U12 = L11^-1 A12 (columns right of it), one thread per row / column
__global__ void __launch_bounds__(kThreads) k_panel_off(double* __restrict__ F, int m, int j0, int nb) {
    __shared__ double D[kNB][kNB + 1];
    for (int e = threadIdx.x; e < nb * nb; e += blockDim.x) D[e / nb][e % nb] = F[(int64_t)(j0 + e / nb) * m + j0 + e % nb];
    __syncthreads();
    const int rest = m - j0 - nb;
    const int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    double x[kNB];
    if (t < rest) {                               // row j0 + nb + t of L21
        double* row = F + (int64_t)j0 * m + j0 + nb + t;
#pragma unroll
        for (int c = 0; c < kNB; ++c) {
            if (c < nb) {
                double s = row[(int64_t)c * m];
#pragma unroll
                for (int q = 0; q < c; ++q) s -= x[q] * D[c][q];
                x[c] = s / D[c][c];
                row[(int64_t)c * m] = x[c];
            }
        }
    } else if (t < 2 * (int64_t)rest) {            // column j0 + nb + (t - rest) of U12
        double* colp = F + (int64_t)(j0 + nb + (t - rest)) * m + j0;
#pragma unroll
        for (int c = 0; c < kNB; ++c) {
            if (c < nb) {
                double s = colp[c];
#pragma unroll
                for (int q = 0; q < c; ++q) s -= D[q][c] * x[q];
                x[c] = s;
                colp[c] = s;
            }
        }
    }
}

// large front: trailing update F[r0:m, r0:m] -= F[r0:m, j0:j0+nb] F[j0:j0+nb, r0:m], r0 = j0 + nb (fp64 FFMA, 4 x 4 per thread)
__global__ void __launch_bounds__(kThreads) k_trailing_gemm(double* __restrict__ F, int m, int j0, int nb) {
    __shared__ double As[kNB][kTile];
    __shared__ double Bs[kNB][kTile];
    const int r0 = j0 + nb;
    const int row0 = r0 + blockIdx.x * kTile, col0 = r0 + blockIdx.y * kTile;
    for (int e = threadIdx.x; e < kTile * nb; e += kThreads) {
        const int i = e % kTile, kk = e / kTile;
        As[kk][i] = row0 + i < m ? F[(int64_t)(j0 + kk) * m + row0 + i] : 0.0;
    }
    for (int e = threadIdx.x; e < kTile * nb; e += kThreads) {
        const int kk = e % nb, jj = e / nb;
        Bs[kk][jj] = col0 + jj < m ? F[(int64_t)(col0 + jj) * m + j0 + kk] : 0.0;
    }
    __syncthreads();
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    double acc[4][4] = {};
    for (int kk = 0; kk < nb; ++kk) {
        double a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { a[i] = As[kk][tx + 16 * i]; b[i] = Bs[kk][ty + 16 * i]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = col0 + ty + 16 * j;
        if (c >= m) continue;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = row0 + tx + 16 * i;
            if (r < m) F[(int64_t)c * m + r] -= acc[i][j];
        }
    }
}

// factors out of the fronts: [L11\U11; L21] (m x k, column-major) then U12 (k x u, row-major: the backward solve reads rows)
__global__ void __launch_bounds__(kThreads) k_compact(const SluNode* __restrict__ sn, const double* __restrict__ F_all,
                                                      double* __restrict__ fac) {
    const SluNode S = sn[blockIdx.x];
    const double* F = F_all + S.front;
    double* L = fac + S.fac;
    const int u = S.m - S.k;
    for (int64_t e = threadIdx.x; e < (int64_t)S.m * S.k; e += blockDim.x) L[e] = F[e];
    double* U = L + (int64_t)S.m * S.k;
    for (int64_t e = threadIdx.x; e < (int64_t)S.k * u; e += blockDim.x) {
        const int r = (int)(e / u), c = (int)(e % u);
        U[e] = F[(int64_t)(S.k + c) * S.m + r];
    }
}

// forward substitution of one level: t = [x_piv; 0] + children's update vectors, t -= L (column sweep), y -> x_piv,
// t[k:m] -> this supernode's update vector
__global__ void __launch_bounds__(kThreads) k_forward(const int* __restrict__ list, const SluNode* __restrict__ sn,
                                                      const double* __restrict__ fac, const int* __restrict__ relmap,
                                                      const int* __restrict__ child, double* __restrict__ x,
                                                      double* __restrict__ w) {
    extern __shared__ double t[];
    const SluNode S = sn[list[blockIdx.x]];
    const int m = S.m, k = S.k;
    for (int i = threadIdx.x; i < m; i += blockDim.x) t[i] = i < k ? x[S.first + i] : 0.0;
    __syncthreads();
    for (int ci = S.child_begin; ci < S.child_end; ++ci) {
        const SluNode C = sn[child[ci]];
        const int u = C.m - C.k;
        for (int i = threadIdx.x; i < u; i += blockDim.x) t[relmap[C.upd + i]] += w[C.upd + i];
        __syncthreads();
    }
    // blocks of 32 pivot columns: warp 0 solves the unit-lower triangle in registers, then every row below takes the 32
    // columns at once (32 independent loads per thread: one memory latency per block instead of one per column)
    const double* L = fac + S.fac;
    const int lane = threadIdx.x % 32;
    for (int j0 = 0; j0 < k; j0 += 32) {
        const int nb = min(32, k - j0);
        if (threadIdx.x < 32) {
            double ti = lane < nb ? t[j0 + lane] : 0.0;
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                if (q >= nb) break;
                const double yq = __shfl_sync(0xffffffffu, ti, q);
                if (lane > q && lane < nb) ti -= L[(int64_t)(j0 + q) * m + j0 + lane] * yq;
            }
            if (lane < nb) t[j0 + lane] = ti;
        }
        __syncthreads();
        for (int i = j0 + nb + threadIdx.x; i < m; i += blockDim.x) {
            double s = t[i];
#pragma unroll
            for (int q = 0; q < 32; ++q)
                if (q < nb) s -= L[(int64_t)(j0 + q) * m + i] * t[j0 + q];
            t[i] = s;
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        if (i < k) x[S.first + i] = t[i];
        else w[S.upd + i - k] = t[i];
    }
}

// backward substitution of one level: x_piv = U11^-1 (y_piv - U12 x[update rows]); the update rows belong to ancestors,
// solved by earlier launches
__global__ void __launch_bounds__(kThreads) k_backward(const int* __restrict__ list, const SluNode* __restrict__ sn,
                                                       const double* __restrict__ fac, const int* __restrict__ row_idx,
                                                       double* __restrict__ x) {
    extern __shared__ double sh[];
    const SluNode S = sn[list[blockIdx.x]];
    const int m = S.m, k = S.k, u = m - k;
    double* t = sh;
    double* xu = sh + k;
    for (int i = threadIdx.x; i < u; i += blockDim.x) xu[i] = x[row_idx[S.rows + k + i]];
    __syncthreads();
    const double* L = fac + S.fac;
    const double* U12 = L + (int64_t)m * k;
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    for (int r = warp; r < k; r += kThreads / 32) {       // one warp per pivot row, fixed reduction tree
        const double* Ur = U12 + (int64_t)r * u;
        double s = 0.0;
        for (int c = lane; c < u; c += 32) s = fma(Ur[c], xu[c], s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) t[r] = x[S.first + r] - s;
    }
    __syncthreads();
    // blocks of 32 pivot rows from the bottom: warp 0 solves the upper triangle in registers, then the rows above take the
    // 32 solved values at once
    for (int j1 = k; j1 > 0; j1 -= 32) {
        const int j0 = max(0, j1 - 32), nb = j1 - j0;
        if (warp == 0) {
            double ti = lane < nb ? t[j0 + lane] : 0.0;
#pragma unroll
            for (int q = 31; q >= 0; --q) {
                if (q >= nb) continue;
                if (lane == q) ti /= L[(int64_t)(j0 + q) * m + j0 + q];
                const double xq = __shfl_sync(0xffffffffu, ti, q);
                if (lane < q) ti -= L[(int64_t)(j0 + q) * m + j0 + lane] * xq;
            }
            if (lane < nb) t[j0 + lane] = ti;
        }
        __syncthreads();
        for (int r = threadIdx.x; r < j0; r += blockDim.x) {
            double s = t[r];
#pragma unroll
            for (int q = 0; q < 32; ++q)
                if (q < nb) s -= L[(int64_t)(j0 + q) * m + r] * t[j0 + q];
            t[r] = s;
        }
        __syncthreads();
    }
    for (int r = threadIdx.x; r < k; r += blockDim.x) x[S.first + r] = t[r];
}

template <class T>
void upload(DBuf<T>& d, const std::vector<T>& h) {
    d.alloc(h.size());
    if (!h.empty()) PORO_CUDA(cudaMemcpy(d.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
}

}  // namespace

bool use_sparse_lu(const Ctx& c, const std::string& pc_type, const std::string& prefix, int64_t rows) {
    return (pc_type == "lu" || pc_type == "cholesky") && c.opt("-" + prefix + "pc_factor_mat_solver_type", "") == "poro" &&
           rows > c.opt_i("-poro_dense_lu_limit", 8192);
}

PCSparseLU::PCSparseLU(Ctx* c_, const Csr& A_, const std::string& prefix) : ctx(c_), n(A_.nrows) {
    Ctx& c = *ctx;
    PORO_REQUIRE(A_.nrows == A_.ncols, "sparse LU needs a square block");
    const std::string blk = "block '" + prefix + "' (" + std::to_string(n) + " rows)";
    // ---- symbolic (host) ----
    std::vector<int> rp, ci;
    std::vector<double> hv;
    csr_to_host(A_, rp, ci, hv);
    std::vector<int64_t> rp64(rp.begin(), rp.end());
    lusym::Symbolic S;
    try {
        S = lusym::analyse(n, rp64.data(), ci.data());
    } catch (const std::exception& e) {
        throw Error("sparse LU of " + blk + ": " + e.what());
    }
    // pivot scales: largest entry of the pivot's row and column of B, in the permuted numbering
    std::vector<double> pscale_h((size_t)n, 0.0);
    for (int i = 0; i < n; ++i)
        for (int q = rp[i]; q < rp[i + 1]; ++q) {
            const double a = std::fabs(hv[q]);
            double& si = pscale_h[S.iperm[i]];
            double& sj = pscale_h[S.iperm[ci[q]]];
            si = std::max(si, a);
            sj = std::max(sj, a);
        }
    const int ns = S.nsuper;
    std::vector<SluNode> nodes((size_t)ns);
    for (int s = 0; s < ns; ++s) {
        SluNode& d = nodes[s];
        d.first = S.first[s];
        d.k = S.first[s + 1] - S.first[s];
        d.m = S.m[s];
        d.child_begin = S.child_ptr[s];
        d.child_end = S.child_ptr[s + 1];
        d.rows = S.row_ptr[s];
        d.upd = S.upd_off[s];
        d.front = S.front_off[s];
        d.fac = S.fac_off[s];
    }
    // fronts of each level: small ones batched, large ones one by one
    std::vector<int> small_ids, small_ptr{0};
    std::vector<std::vector<int>> large((size_t)S.nlevels);
    for (int l = 0; l < S.nlevels; ++l) {
        for (int q = S.level_ptr[l]; q < S.level_ptr[l + 1]; ++q) {
            const int s = S.level_sn[q];
            if (S.m[s] <= kSmallFront) small_ids.push_back(s); else large[l].push_back(s);
        }
        small_ptr.push_back((int)small_ids.size());
    }
    // ---- memory: exact sizes, compared with what the device has free before anything is allocated ----
    const int64_t upd_total = S.upd_off[ns];
    const int64_t fac_bytes = 8 * S.fac_off[ns];
    const int64_t front_bytes = 8 * S.front_off[ns];              // set-up only: fronts incl. contribution blocks
    const int64_t idx_bytes = 4 * ((int64_t)n + upd_total + (int64_t)S.child.size() + ns + S.row_ptr[ns]) +
                              (int64_t)sizeof(SluNode) * ns + 8 * ((int64_t)n + upd_total);
    const int64_t setup_bytes = 8 * (int64_t)hv.size() + 4 * (int64_t)small_ids.size() + 8 * (int64_t)n;   // nz_pos, lists, scales
    {
        size_t fr = 0, tot = 0;
        PORO_CUDA(cudaMemGetInfo(&fr, &tot));
        const int64_t need = fac_bytes + front_bytes + idx_bytes + setup_bytes;
        if (need > (int64_t)fr) {
            char buf[512];
            snprintf(buf, sizeof buf, "sparse LU of %s needs %.3f GB on the device (factors %.3f GB, fronts %.3f GB during the "
                     "factorisation) but %.3f GB are free", blk.c_str(), need * 1e-9, fac_bytes * 1e-9, front_bytes * 1e-9, fr * 1e-9);
            throw Error(buf);
        }
    }
    int max_m = std::max(S.max_front, 1);
    smem = (size_t)max_m * 8;
    {
        int dev_max = 0;
        PORO_CUDA(cudaDeviceGetAttribute(&dev_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, c.device));
        if (smem > (size_t)dev_max)
            throw Error("sparse LU of " + blk + ": largest front (" + std::to_string(max_m) + " rows) exceeds the shared memory of one CTA");
        // the attribute is per kernel, shared by every factorised block: set it to the device limit, never to this block's need
        PORO_CUDA(cudaFuncSetAttribute(k_forward, cudaFuncAttributeMaxDynamicSharedMemorySize, dev_max));
        PORO_CUDA(cudaFuncSetAttribute(k_backward, cudaFuncAttributeMaxDynamicSharedMemorySize, dev_max));
    }
    upload(sn, nodes);
    upload(relmap, S.relmap);
    upload(child, S.child);
    upload(row_idx, S.row_idx);
    upload(level_sn, S.level_sn);
    upload(perm, S.perm);
    level_ptr = S.level_ptr;
    nlevels = S.nlevels;
    {
        DBuf<int64_t> nz_pos;
        upload(nz_pos, S.nz_pos);
        DBuf<int> small;
        upload(small, small_ids);
        DBuf<double> pscale;
        upload(pscale, pscale_h);
        DBuf<int> d_npert(1);
        d_npert.zero(c.stream);
        DBuf<double> F((size_t)S.front_off[ns]);
        fac.alloc((size_t)S.fac_off[ns]);
        cudaEvent_t e0, e1;
        PORO_CUDA(cudaEventCreate(&e0));
        PORO_CUDA(cudaEventCreate(&e1));
        PORO_CUDA(cudaEventRecord(e0, c.stream));
        // ---- numeric factorisation (device) ----
        F.zero(c.stream);
        if (A_.nnz) {
            k_scatter_entries<<<ceil_div(A_.nnz, kThreads), kThreads, 0, c.stream>>>(A_.nnz, A_.val.p, nz_pos.p, F.p);
            PORO_LAUNCH_CHECK(c);
        }
        for (int l = 0; l < S.nlevels; ++l) {
            const int cnt = small_ptr[l + 1] - small_ptr[l];
            if (cnt) {
                k_front_small<<<cnt, kThreads, 0, c.stream>>>(small.p + small_ptr[l], sn.p, F.p, relmap.p, child.p, pscale.p, d_npert.p);
                PORO_LAUNCH_CHECK(c);
            }
            for (int s : large[l]) {
                const SluNode& d = nodes[s];
                double* Fs = F.p + d.front;
                for (int q = d.child_begin; q < d.child_end; ++q) {
                    const SluNode& ch = nodes[S.child[q]];
                    const int64_t u = ch.m - ch.k;
                    if (!u) continue;
                    k_extend_add_one<<<ceil_div(u * u, kThreads), kThreads, 0, c.stream>>>(Fs, d.m, F.p + ch.front, ch.m, ch.k,
                                                                                          relmap.p + ch.upd);
                    PORO_LAUNCH_CHECK(c);
                }
                for (int j0 = 0; j0 < d.k; j0 += kNB) {
                    const int nb = std::min(kNB, d.k - j0), rest = d.m - j0 - nb;
                    k_panel_diag<<<1, kThreads, 0, c.stream>>>(Fs, d.m, j0, nb, pscale.p + d.first, d_npert.p);
                    PORO_LAUNCH_CHECK(c);
                    if (rest <= 0) continue;
                    k_panel_off<<<ceil_div(2 * (int64_t)rest, kThreads), kThreads, 0, c.stream>>>(Fs, d.m, j0, nb);
                    PORO_LAUNCH_CHECK(c);
                    const int tiles = ceil_div(rest, kTile);
                    k_trailing_gemm<<<dim3(tiles, tiles), kThreads, 0, c.stream>>>(Fs, d.m, j0, nb);
                    PORO_LAUNCH_CHECK(c);
                }
            }
        }
        if (ns) {
            k_compact<<<ns, kThreads, 0, c.stream>>>(sn.p, F.p, fac.p);
            PORO_LAUNCH_CHECK(c);
        }
        PORO_CUDA(cudaEventRecord(e1, c.stream));
        PORO_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        PORO_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        factor_ms = ms;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        int np_ = 0;
        PORO_CUDA(cudaMemcpy(&np_, d_npert.p, sizeof(int), cudaMemcpyDeviceToHost));
        npert = np_;
    }
    xw.alloc((size_t)n);
    wbuf.alloc((size_t)std::max<int64_t>(upd_total, 1));
    if (npert > 0) {
        // perturbed pivots: the factorisation is of a nearby matrix, so each application is refined once with the block
        csr_copy(c, A_, A);
        csr_choose_lanes(A);
        r.alloc((size_t)n);
        d.alloc((size_t)n);
        PORO_CUDA(cudaStreamSynchronize(c.stream));
    }
    nnz_l = S.nnz_l;
    nnz_u = S.nnz_u;
    amalg_zeros = S.amalg_zeros;
    nsuper = ns;
    max_front = S.max_front;
    flops = S.flops;
    device_bytes = (int64_t)(fac.bytes() + sn.bytes() + relmap.bytes() + child.bytes() + row_idx.bytes() + level_sn.bytes() +
                             perm.bytes() + xw.bytes() + wbuf.bytes() + A.rowptr.bytes() + A.col.bytes() + A.val.bytes() +
                             r.bytes() + d.bytes());
    // one application without refinement: factor entries once, the index and update-vector traffic, permutation and pivots
    apply_bytes = 8 * (nnz_l + nnz_u) + 32 * upd_total + 72 * (int64_t)n;
}

void PCSparseLU::solve(const double* b, double* x) {
    Ctx& c = *ctx;
    vec_gather(c, xw.p, b, perm.p, n);
    for (int l = 0; l < nlevels; ++l) {
        const int cnt = level_ptr[l + 1] - level_ptr[l];
        k_forward<<<cnt, kThreads, smem, c.stream>>>(level_sn.p + level_ptr[l], sn.p, fac.p, relmap.p, child.p, xw.p, wbuf.p);
        PORO_LAUNCH_CHECK(c);
    }
    for (int l = nlevels - 1; l >= 0; --l) {
        const int cnt = level_ptr[l + 1] - level_ptr[l];
        k_backward<<<cnt, kThreads, smem, c.stream>>>(level_sn.p + level_ptr[l], sn.p, fac.p, row_idx.p, xw.p);
        PORO_LAUNCH_CHECK(c);
    }
    vec_scatter(c, x, xw.p, perm.p, n);
}

void PCSparseLU::apply(const double* x, double* y) {
    solve(x, y);
    if (npert > 0) {
        spmv(*ctx, A, y, r.p, SPMV_SUB, x);          // r = x - B y
        solve(r.p, d.p);
        vec_axpy(*ctx, y, 1.0, d.p, n);
    }
}

}  // namespace poro
