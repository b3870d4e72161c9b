// spmv_epilogue.cuh -- row epilogues shared by the CSR and BSR SpMV kernels.
#pragma once
#include "common.cuh"

namespace poro {

struct Epilogue {
    int mode;                 // SpmvMode, or 3 = Chebyshev step, 4 = dot
    const double* z;          // SUB/ADD source
    // Chebyshev step: t = A d_old; r -= t; d_new = c1 d_old + c2 dinv.*r; x += d_new
    const double* d_old; double* d_new; double* r; double* xv; const double* dinv; double c1, c2;
};

template <int MODE>
__device__ __forceinline__ double apply_epilogue(const Epilogue& ep, int row, double sum, const double* __restrict__ x,
                                                 double* __restrict__ y) {
    if (MODE == SPMV_SET) y[row] = sum;
    else if (MODE == SPMV_SUB) y[row] = ep.z[row] - sum;
    else if (MODE == SPMV_ADD) y[row] = ep.z[row] + sum;
    else if (MODE == 3) {
        const double rn = ep.r[row] - sum;
        const double dn = ep.c1 * ep.d_old[row] + ep.c2 * ep.dinv[row] * rn;
        ep.r[row] = rn;
        ep.d_new[row] = dn;
        ep.xv[row] += dn;
    } else if (MODE == 4) {
        y[row] = sum;
        return sum * x[row];
    }
    return 0.0;
}

// lanes that reduce one row (CSR stream) or one block row (BSR), from the average row length in nonzeros or blocks
inline int row_group_lanes(double avg_row) {
    return avg_row <= 1.5 ? 1 : avg_row <= 4 ? 2 : avg_row <= 12 ? 4 : avg_row <= 48 ? 8 : avg_row <= 160 ? 16 : 32;
}

__device__ __forceinline__ double block_sum_256(double v, double* sm) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 0; w < 8; ++w) t += sm[w];
    }
    return t;
}

bool bsr_from_csr(Ctx& c, const Csr& A, int BS, Bsr& out, double max_fill);
// bsr_tma.cu: chunked layout + persistent TMA kernel; `rp` = host copy of the block row pointers
bool bsr_build_tma(Ctx& c, Bsr& B, const std::vector<int>& rp);
// lets the diagonal-block coupling C (same block rows/columns as B) ride along B: y = B x + C x2 in one pass
bool bsr_fuse_coupling(Ctx& c, Bsr& B, const Csr& C);
template <int MODE>
int bsr_tma_launch(Ctx& c, const Bsr& B, const double* x, double* y, const Epilogue& ep, double* dot_partial, const double* x2 = nullptr);
template <int MODE>
int bsr_launch(Ctx& c, const Bsr& B, const double* x, double* y, const Epilogue& ep, double* dot_partial, const double* x2 = nullptr);
bool bsr_fuse_coupling_tma(Ctx& c, Bsr& B, const Csr& C);

}  // namespace poro
