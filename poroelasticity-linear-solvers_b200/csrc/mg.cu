// mg.cu -- matrix-free geometric transfer of `-<prefix>pc_type mg` (mg.cuh; tables in mg_transfer.h).
//
// k_prolong: one thread per fine node with all BR components; its class is the lattice index mod M per axis, its columns
// are the cell's coarse nodes plus the table offsets.  k_restrict: one thread per coarse node, gathering the fine residual
// of the transposed table (entries outside the domain skipped).  Both sum in table order without atomics, so results are
// bitwise reproducible.  Dirichlet flags of the fine and the coarse rows mask P on both sides.
#include "mg.cuh"

namespace poro {

static constexpr int kMgBlock = 256;

struct MgArgs {
    int dim, Lf, Lc, M, S;
    int64_t nf, nc;
    const int* ptr;
    const poromg::Entry* ent;
    const uint8_t* bcf;
    const uint8_t* bcc;
};

template <int BR, bool ADD>
__global__ void __launch_bounds__(kMgBlock) k_prolong(MgArgs a, const double* __restrict__ e, double* __restrict__ y) {
    const int64_t node = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (node >= a.nf) return;
    int base[3] = {0, 0, 0};
    int cls = 0;
    {
        int64_t q = node;
        int mul = 1;
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            if (m >= a.dim) continue;
            const int X = (int)(q % a.Lf);
            q /= a.Lf;
            cls += (X % a.M) * mul;
            mul *= a.M;
            base[m] = a.S * (X / a.M);
        }
    }
    double acc[BR];
#pragma unroll
    for (int i = 0; i < BR; ++i) acc[i] = 0.0;
    const int p0 = __ldg(a.ptr + cls), p1 = __ldg(a.ptr + cls + 1);
    for (int p = p0; p < p1; ++p) {
        const poromg::Entry& en = a.ent[p];
        const double w = __ldg(&en.w);
        int64_t cn = 0, mul = 1;
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            if (m >= a.dim) continue;
            cn += (int64_t)(base[m] + __ldg(&en.d[m])) * mul;
            mul *= a.Lc;
        }
#pragma unroll
        for (int i = 0; i < BR; ++i) {
            const double v = (a.bcc && a.bcc[cn * BR + i]) ? 0.0 : __ldg(e + cn * BR + i);
            acc[i] = fma(w, v, acc[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < BR; ++i) {
        const int64_t r = node * BR + i;
        const double v = (a.bcf && a.bcf[r]) ? 0.0 : acc[i];
        y[r] = ADD ? y[r] + v : v;
    }
}

template <int BR>
__global__ void __launch_bounds__(kMgBlock) k_restrict(MgArgs a, const double* __restrict__ rf, double* __restrict__ y) {
    const int64_t node = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (node >= a.nc) return;
    int Y[3] = {0, 0, 0};
    int cls = 0;
    {
        int64_t q = node;
        int mul = 1;
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            if (m >= a.dim) continue;
            Y[m] = (int)(q % a.Lc);
            q /= a.Lc;
            cls += (Y[m] % a.S) * mul;
            mul *= a.S;
        }
    }
    double acc[BR];
#pragma unroll
    for (int i = 0; i < BR; ++i) acc[i] = 0.0;
    const int p0 = __ldg(a.ptr + cls), p1 = __ldg(a.ptr + cls + 1);
    for (int p = p0; p < p1; ++p) {
        const poromg::Entry& en = a.ent[p];
        int64_t fn = 0, mul = 1;
        bool inside = true;
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            if (m >= a.dim) continue;
            const int X = 2 * Y[m] + __ldg(&en.d[m]);
            inside = inside && X >= 0 && X < a.Lf;
            fn += (int64_t)X * mul;
            mul *= a.Lf;
        }
        if (!inside) continue;
        const double w = __ldg(&en.w);
#pragma unroll
        for (int i = 0; i < BR; ++i) {
            const double v = (a.bcf && a.bcf[fn * BR + i]) ? 0.0 : __ldg(rf + fn * BR + i);
            acc[i] = fma(w, v, acc[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < BR; ++i) {
        const int64_t r = node * BR + i;
        y[r] = (a.bcc && a.bcc[r]) ? 0.0 : acc[i];
    }
}

int mg_attached_levels(const StencilOp& s) {
    int n = 0;
    for (const StencilData* d = s.d.get(); d && d->coarse; d = d->coarse->stencil->d.get()) ++n;
    return n;
}

void mg_coarse_block(Ctx& c, const StencilOp& s, Csr& out) {
    PORO_REQUIRE(s.d && s.d->coarse && s.fr >= 0 && s.fc == s.fr, "mg: the block has no coarse level attached");
    const Csr& M = *s.d->coarse;
    const StencilData& cd = *M.stencil->d;
    const int64_t r0 = cd.row0[s.fr], r1 = cd.row0[s.fr + 1];
    std::vector<int> rmap((size_t)M.nrows, -1), cmap((size_t)M.ncols, -1);
    for (int64_t i = r0; i < r1; ++i) rmap[i] = cmap[i] = (int)(i - r0);
    DBuf<int> d_r(rmap.size()), d_c(cmap.size());
    PORO_CUDA(cudaMemcpy(d_r.p, rmap.data(), rmap.size() * 4, cudaMemcpyHostToDevice));
    PORO_CUDA(cudaMemcpy(d_c.p, cmap.data(), cmap.size() * 4, cudaMemcpyHostToDevice));
    csr_extract(c, M, d_r.p, d_c.p, (int)(r1 - r0), (int)(r1 - r0), out);
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    csr_choose_lanes(out);
    out.stencil = std::make_shared<StencilOp>(StencilOp{M.stencil->d, s.fr, s.fr});
}

template <class T>
static void upload(Ctx& c, DBuf<T>& d, const std::vector<T>& h) {
    d.alloc(h.size());
    if (!h.empty()) PORO_CUDA(cudaMemcpyAsync(d.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

void mg_transfer_init(Ctx& c, MgTransfer& t, const StencilOp& fine, const StencilOp& coarse) {
    const StencilData& f = *fine.d;
    const StencilData& g = *coarse.d;
    const int fr = fine.fr;
    PORO_REQUIRE(fr >= 0 && fine.fc == fr && coarse.fr == fr && coarse.fc == fr, "mg: transfers link diagonal field blocks");
    PORO_REQUIRE(f.N == 2 * g.N && f.dim == g.dim && f.kind[fr] == g.kind[fr] && f.bdim[fr] == g.bdim[fr],
                 "mg: the coarse level is not the same field at N/2");
    t.fine = fine;
    t.coarse = coarse;
    t.dim = f.dim;
    t.kind = f.kind[fr];
    t.br = f.bdim[fr];
    t.Nc = g.N;
    t.nf = porogen::lattice_nodes(t.kind, f.N, t.dim);
    t.nc = porogen::lattice_nodes(t.kind, g.N, t.dim);
    t.bcf = f.bc.p ? f.bc.p + f.row0[fr] : nullptr;
    t.bcc = g.bc.p ? g.bc.p + g.row0[fr] : nullptr;
    const poromg::Table P = poromg::prolong_table(t.kind, t.dim), R = poromg::restrict_table(t.kind, t.dim);
    upload(c, t.pptr, P.ptr);
    upload(c, t.pent, P.e);
    upload(c, t.rptr, R.ptr);
    upload(c, t.rent, R.e);
    t.ptab_bytes = (int64_t)(P.ptr.size() * sizeof(int) + P.e.size() * sizeof(poromg::Entry));
    t.rtab_bytes = (int64_t)(R.ptr.size() * sizeof(int) + R.e.size() * sizeof(poromg::Entry));
}

static MgArgs mg_args(const MgTransfer& t, bool prolong) {
    MgArgs a{};
    a.dim = t.dim;
    a.Lf = porogen::lattice_extent(t.kind, 2 * t.Nc);
    a.Lc = porogen::lattice_extent(t.kind, t.Nc);
    a.M = prolong ? poromg::fine_per_cell(t.kind) : 0;
    a.S = poromg::coarse_per_cell(t.kind);
    a.nf = t.nf;
    a.nc = t.nc;
    a.ptr = prolong ? t.pptr.p : t.rptr.p;
    a.ent = prolong ? t.pent.p : t.rent.p;
    a.bcf = t.bcf;
    a.bcc = t.bcc;
    return a;
}

void mg_prolong(Ctx& c, const MgTransfer& t, const double* e, double* y, bool add) {
    const MgArgs a = mg_args(t, true);
    const int grid = (int)ceil_div(t.nf, kMgBlock);
    if (grid == 0) return;
#define PORO_MG_P(BR)                                                                             \
    if (add) k_prolong<BR, true><<<grid, kMgBlock, 0, c.stream>>>(a, e, y);                       \
    else k_prolong<BR, false><<<grid, kMgBlock, 0, c.stream>>>(a, e, y);
    switch (t.br) {
        case 3: PORO_MG_P(3) break;
        case 2: PORO_MG_P(2) break;
        default: PORO_MG_P(1) break;
    }
#undef PORO_MG_P
    PORO_LAUNCH_CHECK(c);
}

void mg_restrict(Ctx& c, const MgTransfer& t, const double* r, double* y) {
    const MgArgs a = mg_args(t, false);
    const int grid = (int)ceil_div(t.nc, kMgBlock);
    if (grid == 0) return;
    switch (t.br) {
        case 3: k_restrict<3><<<grid, kMgBlock, 0, c.stream>>>(a, r, y); break;
        case 2: k_restrict<2><<<grid, kMgBlock, 0, c.stream>>>(a, r, y); break;
        default: k_restrict<1><<<grid, kMgBlock, 0, c.stream>>>(a, r, y); break;
    }
    PORO_LAUNCH_CHECK(c);
}

__global__ void k_mg_inject(int dim, int Lf, int Lc, int64_t nc, int br, int k, const double* __restrict__ B, double* __restrict__ Bc) {
    const int64_t t = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (t >= nc * br * k) return;
    const int64_t row = t / k, node = row / br;
    int64_t q = node, fn = 0, mul = 1;
    for (int m = 0; m < dim; ++m) {
        fn += 2 * (q % Lc) * mul;
        q /= Lc;
        mul *= Lf;
    }
    Bc[t] = B[(fn * br + row % br) * k + t % k];
}

void mg_inject(Ctx& c, const MgTransfer& t, const double* B, int k, DBuf<double>& Bc) {
    const int64_t n = t.nc * t.br * k;
    Bc.alloc((size_t)n);
    if (n == 0) return;
    k_mg_inject<<<(int)ceil_div(n, kMgBlock), kMgBlock, 0, c.stream>>>(t.dim, porogen::lattice_extent(t.kind, 2 * t.Nc),
                                                                        porogen::lattice_extent(t.kind, t.Nc), t.nc, t.br, k, B, Bc.p);
    PORO_LAUNCH_CHECK(c);
}

int64_t mg_prolong_bytes(const MgTransfer& t, bool add) {
    const int64_t rf = t.nf * t.br, rc = t.nc * t.br;
    return 8 * rc + 8 * rf * (add ? 2 : 1) + (t.bcf ? rf : 0) + (t.bcc ? rc : 0) + t.ptab_bytes;
}

int64_t mg_restrict_bytes(const MgTransfer& t) {
    const int64_t rf = t.nf * t.br, rc = t.nc * t.br;
    return 8 * rf + 8 * rc + (t.bcf ? rf : 0) + (t.bcc ? rc : 0) + t.rtab_bytes;
}

}  // namespace poro
