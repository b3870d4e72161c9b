// gen.cu -- device-side generator of the assembled three-field system on dolfin's structured meshes (SURVEY 8 f1).
//
// Stands where the reference assembles A, P, P_diff on the host with FEniCS (lib/Assembler.py:66-221) and applies the
// Dirichlet conditions (lib/Poromechanics.py:76-83).  With constant coefficients every field block is ONE macro-cell
// matrix scattered over all cells, so the block row of a node is one of <= 4^d (P2 rows) / 3^d (P1 rows) class stencils,
// shifted (gen_stencil.cuh; hostfem/stencil.py derives the tables from the element matrices and is the numpy statement).
// Here a rank generates the rows of ITS z-slab of nodes, for all three fields at once, straight into the local CSR the
// solver consumes: rows [s | f | p] of the owned nodes, columns renumbered to [owned | ghost of the lower neighbour |
// ghost of the upper neighbour] with analytic (contiguous plane range) maps -- no sort, no atomics, no host matrix.
//   k_gen_count : non-zeros per scalar row (structural zeros of the stencil tables are dropped, a Dirichlet row keeps
//                 its unit diagonal only: DirichletBC.apply + eliminate_zeros, like hostfem.fem.compose)
//   k_gen_fill  : one warp per scalar row; lanes run over the (entry, column component) items of the three blocks of
//                 the row and compact the non-zeros with a ballot, so stores are contiguous
#include "common.cuh"
#include "gen_stencil.cuh"
#include "stencil.cuh"
#include "../../include/poro.h"
#include <cub/cub.cuh>

namespace poro {

struct GenLayout {
    int dim, N;
    // per lattice (index 0: P1, 1: P2): owned node range and the ghost node ranges of the lower / upper neighbour
    int64_t o0[2], o1[2], gl0[2], gl1[2], gu0[2], gu1[2];
    int64_t off_owned[3], off_gl[3], off_gu[3];      // local dof offsets per field (s, f, p)
    int64_t row0[4];                                 // first local row of each field, row0[3] = number of owned rows
    int bdim[3], kind[3];                            // dofs per node and lattice of each field
};
struct GenTables {
    porogen::BlockTable t[9];
    int present[9];
};

__device__ __forceinline__ int gen_field_of(const GenLayout& g, int64_t r) { return r < g.row0[1] ? 0 : (r < g.row0[2] ? 1 : 2); }

// local column of (field fc, column node c, component j); -1 when the node is neither owned nor a ghost
__device__ __forceinline__ int64_t gen_local_col(const GenLayout& g, int fc, int64_t c, int j) {
    const int k = g.kind[fc] - 1, b = g.bdim[fc];
    if (c >= g.o0[k] && c < g.o1[k]) return g.off_owned[fc] + (c - g.o0[k]) * b + j;
    if (c >= g.gl0[k] && c < g.gl1[k]) return g.off_gl[fc] + (c - g.gl0[k]) * b + j;
    if (c >= g.gu0[k] && c < g.gu1[k]) return g.off_gu[fc] + (c - g.gu0[k]) * b + j;
    return -1;
}

__global__ void __launch_bounds__(256) k_gen_count(GenLayout g, GenTables T, const uint8_t* __restrict__ bc, int* __restrict__ counts) {
    const int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (r >= g.row0[3]) return;
    const int fr = gen_field_of(g, r);
    if (bc && bc[r]) { counts[r] = 1; return; }
    const int64_t lr = r - g.row0[fr];
    const int64_t node = g.o0[g.kind[fr] - 1] + lr / g.bdim[fr];
    const int i = (int)(lr % g.bdim[fr]);
    int cnt = 0;
    for (int fc = 0; fc < 3; ++fc) {
        if (!T.present[fr * 3 + fc]) continue;
        const porogen::BlockTable& t = T.t[fr * 3 + fc];
        int cls;
        int64_t base;
        porogen::row_info(t, node, cls, base);
        const int bsz = t.br * t.bc;
        for (int p = t.cls_ptr[cls]; p < t.cls_ptr[cls + 1]; ++p)
            for (int j = 0; j < t.bc; ++j) cnt += t.vals[(int64_t)p * bsz + i * t.bc + j] != 0.0;
    }
    counts[r] = cnt;
}

__global__ void __launch_bounds__(256) k_gen_fill(GenLayout g, GenTables T, const uint8_t* __restrict__ bc, const int* __restrict__ rowptr,
                                                  int* __restrict__ col, double* __restrict__ val, int* __restrict__ err) {
    const int lane = threadIdx.x & 31;
    const int64_t r = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (r >= g.row0[3]) return;
    const int fr = gen_field_of(g, r);
    const int64_t lr = r - g.row0[fr];
    const int64_t node = g.o0[g.kind[fr] - 1] + lr / g.bdim[fr];
    const int i = (int)(lr % g.bdim[fr]);
    int64_t dst = rowptr[r];
    if (bc && bc[r]) {                                             // Dirichlet row: unit diagonal (the row is owned)
        if (lane == 0) { col[dst] = (int)r; val[dst] = 1.0; }
        return;
    }
    for (int fc = 0; fc < 3; ++fc) {
        if (!T.present[fr * 3 + fc]) continue;
        const porogen::BlockTable& t = T.t[fr * 3 + fc];
        int cls;
        int64_t base;
        porogen::row_info(t, node, cls, base);
        const int p0 = t.cls_ptr[cls], items = (t.cls_ptr[cls + 1] - p0) * t.bc, bsz = t.br * t.bc;
        for (int q0 = 0; q0 < items; q0 += 32) {
            const int q = q0 + lane;
            double v = 0.0;
            int64_t lc = 0;
            if (q < items) {
                const int e = q / t.bc, j = q - e * t.bc;
                v = t.vals[(int64_t)(p0 + e) * bsz + i * t.bc + j];
                if (v != 0.0) {
                    lc = gen_local_col(g, fc, base + t.off[p0 + e], j);
                    if (lc < 0) { atomicExch(err, 1); lc = 0; }
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, v != 0.0);
            if (v != 0.0) {
                const int64_t pos = dst + __popc(m & ((1u << lane) - 1u));
                col[pos] = (int)lc;
                val[pos] = v;
            }
            dst += __popc(m);
        }
    }
}

__global__ void k_gen_widen(int64_t n, const int* __restrict__ ci, int64_t* __restrict__ co, int64_t nr) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n) co[i] = i < nr ? (int64_t)ci[i] : 0;
}
__global__ void k_gen_narrow(int64_t n, const int64_t* __restrict__ s, int* __restrict__ rp) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n) rp[i] = (int)s[i];
}

}  // namespace poro

using namespace poro;

// defined in capi.cu
poro_mat* poro_mat_adopt(poro_ctx* h, Csr&& A);
Ctx& poro_ctx_ref(poro_ctx* h);
void poro_set_error(const std::string& msg);

int poro_gen_matrix(poro_ctx* h, int dim, int N, const poro_gen_table* tables, const int64_t* layout, const uint8_t* bc_flags_host,
                    poro_mat** out) {
    try {
        Ctx& c = poro_ctx_ref(h);
        PORO_CUDA(cudaSetDevice(c.device));
        PORO_REQUIRE(dim == 2 || dim == 3, "dim must be 2 or 3");
        GenLayout g{};
        g.dim = dim; g.N = N;
        for (int k = 0; k < 2; ++k) {
            const int64_t* q = layout + 6 * k;
            g.o0[k] = q[0]; g.o1[k] = q[1]; g.gl0[k] = q[2]; g.gl1[k] = q[3]; g.gu0[k] = q[4]; g.gu1[k] = q[5];
        }
        for (int f = 0; f < 3; ++f) { g.off_owned[f] = layout[12 + f]; g.off_gl[f] = layout[15 + f]; g.off_gu[f] = layout[18 + f]; }
        const int64_t ncols = layout[21];
        g.bdim[0] = g.bdim[1] = dim; g.bdim[2] = 1;
        g.kind[0] = g.kind[1] = 2; g.kind[2] = 1;
        g.row0[0] = 0;
        for (int f = 0; f < 3; ++f) g.row0[f + 1] = g.row0[f] + (g.o1[g.kind[f] - 1] - g.o0[g.kind[f] - 1]) * g.bdim[f];
        const int64_t nrows = g.row0[3];
        PORO_REQUIRE(nrows < 2147483647LL && ncols < 2147483647LL, "local system too large for 32-bit indices");
        for (int f = 0; f < 3; ++f) PORO_REQUIRE(g.off_owned[f] == g.row0[f], "owned column offsets must equal the row offsets (field-major)");
        // tables to the device; entries whose block is all zero are dropped (they add nothing to the CSR and only cost the
        // stencil kernel work), and tables of diagonal blocks are marked for the stencil kernel
        GenTables T{};
        std::vector<DBuf<int32_t>> d_cls(9);
        std::vector<DBuf<int64_t>> d_off(9);
        std::vector<DBuf<double>> d_val(9);
        int diag_only[9] = {0};
        int64_t table_bytes[9] = {0};
        for (int b = 0; b < 9; ++b) {
            const poro_gen_table& s = tables[b];
            T.present[b] = s.cls_ptr != nullptr && s.ncls > 0 && s.cls_ptr[s.ncls] > 0;
            if (!T.present[b]) continue;
            const int fr = b / 3, fc = b % 3;
            PORO_REQUIRE(s.kr == g.kind[fr] && s.kc == g.kind[fc] && s.br == g.bdim[fr] && s.bc == g.bdim[fc], "block table does not match its field pair");
            const int bsz = s.br * s.bc;
            std::vector<int32_t> cp(1, 0);
            std::vector<int64_t> of;
            std::vector<double> va;
            bool diag = s.br == s.bc;
            for (int k = 0; k < s.ncls; ++k) {
                for (int p = s.cls_ptr[k]; p < s.cls_ptr[k + 1]; ++p) {
                    const double* v = s.vals + (int64_t)p * bsz;
                    bool nz = false;
                    for (int q = 0; q < bsz; ++q) {
                        nz = nz || v[q] != 0.0;
                        if (v[q] != 0.0 && q / s.bc != q % s.bc) diag = false;
                    }
                    if (!nz) continue;
                    of.push_back(s.off[p]);
                    va.insert(va.end(), v, v + bsz);
                }
                cp.push_back((int32_t)of.size());
            }
            diag_only[b] = diag;
            const int nent = (int)of.size();
            d_cls[b].alloc(cp.size()); d_off[b].alloc((size_t)nent); d_val[b].alloc(va.size());
            PORO_CUDA(cudaMemcpyAsync(d_cls[b].p, cp.data(), cp.size() * 4, cudaMemcpyHostToDevice, c.stream));
            if (nent) {
                PORO_CUDA(cudaMemcpyAsync(d_off[b].p, of.data(), of.size() * 8, cudaMemcpyHostToDevice, c.stream));
                PORO_CUDA(cudaMemcpyAsync(d_val[b].p, va.data(), va.size() * 8, cudaMemcpyHostToDevice, c.stream));
            }
            PORO_CUDA(cudaStreamSynchronize(c.stream));     // the host vectors go out of scope
            table_bytes[b] = (int64_t)cp.size() * 4 + (int64_t)nent * 8 + (int64_t)va.size() * 8;
            T.t[b] = porogen::BlockTable{dim, N, s.kr, s.kc, s.br, s.bc, s.diag_block, d_cls[b].p, d_off[b].p, d_val[b].p};
        }
        DBuf<uint8_t> d_bc;
        if (bc_flags_host) {
            d_bc.alloc((size_t)nrows);
            PORO_CUDA(cudaMemcpyAsync(d_bc.p, bc_flags_host, (size_t)nrows, cudaMemcpyHostToDevice, c.stream));
        }
        Csr A;
        A.nrows = (int)nrows;
        A.ncols = (int)ncols;
        A.rowptr.alloc((size_t)nrows + 1);
        DBuf<int> counts((size_t)nrows + 1);
        const int gridc = (int)((nrows + 255) / 256);
        if (nrows) k_gen_count<<<gridc, 256, 0, c.stream>>>(g, T, d_bc.p, counts.p);
        PORO_LAUNCH_CHECK(c);
        // exclusive scan in 64 bit (the local matrix must stay below 2^31 non-zeros)
        DBuf<int64_t> c64((size_t)nrows + 1), s64((size_t)nrows + 1);
        k_gen_widen<<<(int)((nrows + 1 + 255) / 256), 256, 0, c.stream>>>(nrows + 1, counts.p, c64.p, nrows);
        PORO_LAUNCH_CHECK(c);
        size_t tb = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tb, c64.p, s64.p, nrows + 1, c.stream);
        DBuf<char> tmp(tb);
        cub::DeviceScan::ExclusiveSum(tmp.p, tb, c64.p, s64.p, nrows + 1, c.stream);
        int64_t nnz = 0;
        PORO_CUDA(cudaMemcpyAsync(&nnz, s64.p + nrows, 8, cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        PORO_REQUIRE(nnz < 2147483647LL, "local matrix has more than 2^31 nonzeros: shard it over more GPUs");
        k_gen_narrow<<<(int)((nrows + 1 + 255) / 256), 256, 0, c.stream>>>(nrows + 1, s64.p, A.rowptr.p);
        PORO_LAUNCH_CHECK(c);
        A.nnz = nnz;
        A.col.alloc((size_t)nnz);
        A.val.alloc((size_t)nnz);
        DBuf<int> err(1);
        err.zero(c.stream);
        if (nrows) k_gen_fill<<<(int)((nrows * 32 + 255) / 256), 256, 0, c.stream>>>(g, T, d_bc.p, A.rowptr.p, A.col.p, A.val.p, err.p);
        PORO_LAUNCH_CHECK(c);
        int herr = 0;
        PORO_CUDA(cudaMemcpyAsync(&herr, err.p, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        PORO_REQUIRE(herr == 0, "generator: a stencil entry falls outside the owned and ghost node ranges of the layout");
        csr_choose_lanes(A);
        // single rank, whole lattices owned: keep the tables next to the CSR so that products run from them (stencil.cu).
        // Row-partitioned slabs order their ghost columns differently from the field blocks extracted later: their products
        // stay assembled, the descriptor only carries the geometry of `-<prefix>pc_type mg` (slab = true).
        const bool slab = c.nranks > 1 && dim == 3;
        bool whole = c.nranks == 1;
        for (int k = 0; k < 2; ++k)
            whole = whole && g.o0[k] == 0 && g.o1[k] == porogen::lattice_nodes(k + 1, N, dim) && g.gl0[k] == g.gl1[k] && g.gu0[k] == g.gu1[k];
        whole = whole && ncols == nrows;
        if (whole && bc_flags_host) {
            // the kernel reads the Dirichlet flags of boundary nodes only
            for (int64_t r = 0; r < nrows && whole; ++r) {
                if (!bc_flags_host[r]) continue;
                int f = r < g.row0[1] ? 0 : (r < g.row0[2] ? 1 : 2);
                int64_t node = (r - g.row0[f]) / g.bdim[f];
                const int L = porogen::lattice_extent(g.kind[f], N);
                bool bnd = false;
                for (int m = 0; m < dim; ++m, node /= L) bnd = bnd || node % L == 0 || node % L == L - 1;
                whole = bnd;
            }
        }
        if (whole || slab) {
            auto d = std::make_shared<StencilData>();
            d->dim = dim; d->N = N;
            d->slab = !whole;
            for (int k = 0; k < 2; ++k) {
                d->o0[k] = g.o0[k]; d->o1[k] = g.o1[k]; d->gl0[k] = g.gl0[k]; d->gl1[k] = g.gl1[k]; d->gu0[k] = g.gu0[k]; d->gu1[k] = g.gu1[k];
            }
            for (int f = 0; f < 3; ++f) { d->off_gl[f] = g.off_gl[f]; d->off_gu[f] = g.off_gu[f]; }
            for (int b = 0; b < 9; ++b) {
                d->t[b] = T.t[b]; d->present[b] = T.present[b]; d->diag_only[b] = diag_only[b]; d->table_bytes[b] = table_bytes[b];
                d->cls[b] = std::move(d_cls[b]); d->off[b] = std::move(d_off[b]); d->val[b] = std::move(d_val[b]);
            }
            d->bc = std::move(d_bc);
            for (int f = 0; f < 4; ++f) d->row0[f] = g.row0[f];
            for (int f = 0; f < 3; ++f) { d->bdim[f] = g.bdim[f]; d->kind[f] = g.kind[f]; }
            if (!d->slab) stencil_build_warps(c, *d);
            A.stencil = std::make_shared<StencilOp>();
            A.stencil->d = std::move(d);
        }
        *out = poro_mat_adopt(h, std::move(A));
        return 0;
    } catch (const std::exception& e) {
        poro_set_error(e.what());
        return -1;
    }
}
