// mg.cu -- matrix-free geometric transfer of `-<prefix>pc_type mg` (mg.cuh; tables in mg_transfer.h).
//
// k_prolong: one thread per fine node with all BR components; its class is the lattice index mod M per axis, its columns
// are the cell's coarse nodes plus the table offsets.  k_restrict: one thread per coarse node, gathering the fine residual
// of the transposed table (entries outside the domain skipped).  Both sum in table order without atomics, so results are
// bitwise reproducible.  Dirichlet flags of the fine and the coarse rows mask P on both sides.
#include "mg.cuh"
#include "dist.cuh"
#include "distamg.cuh"
#include <algorithm>

namespace poro {

static constexpr int kMgBlock = 256;

// device view of the vector a transfer reads (MgGhosts): owned flags `bc`, ghost flags `bcg`
struct MgSide {
    int64_t o0, o1, g0;
    const int* tab;
    const uint8_t* bc;
    const uint8_t* bcg;
};

struct MgArgs {
    int dim, Lf, Lc, M, S;
    int64_t nf, nc;
    const int* ptr;
    const poromg::Entry* ent;
    MgSide f, c;
};

// acc += w * v(node) for the BR components of lattice node `node` of a vector stored [owned (own) | ghost (gh)], Dirichlet
// components read as 0
template <int BR>
__device__ __forceinline__ void mg_gather(const MgSide& s, const double* __restrict__ own, const double* __restrict__ gh, int64_t node,
                                          double w, double (&acc)[BR]) {
    const double* v = own;
    const uint8_t* bc = s.bc;
    int64_t q;
    if (node >= s.o0 && node < s.o1) q = (node - s.o0) * BR;
    else {
        q = __ldg(s.tab + (node < s.o0 ? node - s.g0 : s.o0 - s.g0 + node - s.o1));
        v = gh;
        bc = s.bcg;
    }
#pragma unroll
    for (int i = 0; i < BR; ++i) {
        const double x = (bc && bc[q + i]) ? 0.0 : __ldg(v + q + i);
        acc[i] = fma(w, x, acc[i]);
    }
}

template <int BR, bool ADD>
__global__ void __launch_bounds__(kMgBlock) k_prolong(MgArgs a, const double* __restrict__ e, const double* __restrict__ eg,
                                                      double* __restrict__ y) {
    const int64_t node = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (node >= a.nf) return;
    int base[3] = {0, 0, 0};
    int cls = 0;
    {
        int64_t q = a.f.o0 + node;
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
        int64_t cn = 0, mul = 1;
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            if (m >= a.dim) continue;
            cn += (int64_t)(base[m] + __ldg(&en.d[m])) * mul;
            mul *= a.Lc;
        }
        mg_gather<BR>(a.c, e, eg, cn, __ldg(&en.w), acc);
    }
#pragma unroll
    for (int i = 0; i < BR; ++i) {
        const int64_t r = node * BR + i;
        const double v = (a.f.bc && a.f.bc[r]) ? 0.0 : acc[i];
        y[r] = ADD ? y[r] + v : v;
    }
}

template <int BR>
__global__ void __launch_bounds__(kMgBlock) k_restrict(MgArgs a, const double* __restrict__ rf, const double* __restrict__ rg,
                                                       double* __restrict__ y) {
    const int64_t node = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (node >= a.nc) return;
    int Y[3] = {0, 0, 0};
    int cls = 0;
    {
        int64_t q = a.c.o0 + node;
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
        mg_gather<BR>(a.f, rf, rg, fn, __ldg(&en.w), acc);
    }
#pragma unroll
    for (int i = 0; i < BR; ++i) {
        const int64_t r = node * BR + i;
        y[r] = (a.c.bc && a.c.bc[r]) ? 0.0 : acc[i];
    }
}

int mg_attached_levels(const StencilOp& s) {
    int n = 0;
    for (const StencilData* d = s.d.get(); d && d->coarse; d = d->coarse->stencil->d.get()) ++n;
    return n;
}

template <class T>
static void upload(Ctx& c, DBuf<T>& d, const std::vector<T>& h) {
    d.alloc(h.size());
    if (!h.empty()) PORO_CUDA(cudaMemcpyAsync(d.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

// rank-contiguous row offsets of a block whose ranks own `mine` rows each (collective)
static std::vector<int64_t> gather_offsets(Ctx& c, int64_t mine) {
    std::vector<int64_t> sizes, off((size_t)c.nranks + 1, 0);
    dist_allgather_i64(c, &mine, 1, sizes);
    for (int r = 0; r < c.nranks; ++r) off[r + 1] = off[r] + sizes[r];
    return off;
}

// a plan over the global dofs node * br + component of one field (the slabs own contiguous node ranges in rank order, so
// this is the rank-contiguous numbering); `gid` ascending (collective)
static void plan_of_dofs(Ctx& c, int64_t n_owned, std::vector<int>& gid, DistPlan& plan) {
    DBuf<int> d((size_t)gid.size());
    if (!gid.empty()) PORO_CUDA(cudaMemcpy(d.p, gid.data(), gid.size() * sizeof(int), cudaMemcpyHostToDevice));
    dist_plan_build(c, gather_offsets(c, n_owned), std::move(d), (int)gid.size(), plan);
}

void mg_coarse_block(Ctx& c, const StencilOp& s, Csr& out, std::unique_ptr<DistPlan>* plan) {
    PORO_REQUIRE(s.d && s.d->coarse && s.fr >= 0 && s.fc == s.fr, "mg: the block has no coarse level attached");
    const Csr& M = *s.d->coarse;
    const StencilData& cd = *M.stencil->d;
    const int fr = s.fr;
    const int64_t r0 = cd.row0[fr], r1 = cd.row0[fr + 1];
    std::vector<int> rmap((size_t)M.nrows, -1), cmap((size_t)M.ncols, -1);
    for (int64_t i = r0; i < r1; ++i) rmap[i] = cmap[i] = (int)(i - r0);
    int64_t ncols = r1 - r0;
    std::vector<int> gid;
    if (cd.slab) {
        // columns [owned | lower ghosts | upper ghosts] of the field: ascending global dofs node * b + component
        PORO_REQUIRE(plan != nullptr, "mg: a row-partitioned coarse level needs the distributed hierarchy");
        const int k = cd.kind[fr] - 1, b = cd.bdim[fr];
        const int64_t lo[2] = {cd.gl0[k], cd.gu0[k]}, hi[2] = {cd.gl1[k], cd.gu1[k]}, at[2] = {cd.off_gl[fr], cd.off_gu[fr]};
        for (int side = 0; side < 2; ++side)
            for (int64_t i = 0; i < (hi[side] - lo[side]) * b; ++i) {
                cmap[at[side] + i] = (int)ncols++;
                gid.push_back((int)(lo[side] * b + i));
            }
    }
    DBuf<int> d_r(rmap.size()), d_c(cmap.size());
    PORO_CUDA(cudaMemcpy(d_r.p, rmap.data(), rmap.size() * 4, cudaMemcpyHostToDevice));
    PORO_CUDA(cudaMemcpy(d_c.p, cmap.data(), cmap.size() * 4, cudaMemcpyHostToDevice));
    csr_extract(c, M, d_r.p, d_c.p, (int)(r1 - r0), (int)ncols, out);
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    csr_choose_lanes(out);
    out.stencil = std::make_shared<StencilOp>(StencilOp{M.stencil->d, fr, fr});
    if (cd.slab) {
        *plan = std::make_unique<DistPlan>();
        plan_of_dofs(c, r1 - r0, gid, **plan);
    }
}

__global__ void k_mg_flags_in(int64_t n, const uint8_t* __restrict__ bc, double* __restrict__ v) {
    const int64_t i = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (i < n) v[i] = bc[i] ? 1.0 : 0.0;
}
__global__ void k_mg_flags_out(int64_t n, const double* __restrict__ v, uint8_t* __restrict__ bc) {
    const int64_t i = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (i < n) bc[i] = v[i] != 0.0;
}

// G from the ghost ids of `plan` (global dof node * br + component): the table over the ghost planes, and the Dirichlet
// flags of the ghost dofs from their owners (collective when bc_owned is given on every rank)
static void mg_ghosts(Ctx& c, MgGhosts& G, DistPlan& plan, int br, int64_t o0, int64_t o1, const uint8_t* bc_owned) {
    PORO_REQUIRE(plan.offset == o0 * br && plan.n_owned == (o1 - o0) * br,
                 "mg: the halo plan of a slab block does not number its owned dofs node by node");
    std::vector<int> gid((size_t)plan.n_ghost);
    if (plan.n_ghost) PORO_CUDA(cudaMemcpy(gid.data(), plan.ghost_gid.p, gid.size() * sizeof(int), cudaMemcpyDeviceToHost));
    G.o0 = o0; G.o1 = o1; G.g0 = o0; G.g1 = o1;
    for (int q : gid) { G.g0 = std::min(G.g0, (int64_t)(q / br)); G.g1 = std::max(G.g1, (int64_t)(q / br) + 1); }
    std::vector<int> tab((size_t)(o0 - G.g0 + G.g1 - o1), -1);
    auto slot = [&](int64_t node) { return node < o0 ? node - G.g0 : o0 - G.g0 + node - o1; };
    for (size_t p = 0; p < gid.size(); ++p) {
        const int64_t node = gid[p] / br;
        PORO_REQUIRE(node < o0 || node >= o1, "mg: a ghost id of the halo plan is owned by this rank");
        if (gid[p] % br == 0) tab[slot(node)] = (int)p;
    }
    for (size_t p = 0; p < gid.size(); ++p)
        PORO_REQUIRE(tab[slot(gid[p] / br)] == (int)p - gid[p] % br, "mg: the components of a ghost node are not consecutive in the halo plan");
    upload(c, G.tab, tab);
    if (!bc_owned) return;
    const int64_t no = plan.n_owned, ng = plan.n_ghost;
    DBuf<double> v((size_t)(no + ng));
    if (no) k_mg_flags_in<<<(int)ceil_div(no, kMgBlock), kMgBlock, 0, c.stream>>>(no, bc_owned, v.p);
    PORO_LAUNCH_CHECK(c);
    dist_halo_vec(c, plan, v.p, 1, v.p + no);
    G.bc.alloc((size_t)ng);
    if (ng) k_mg_flags_out<<<(int)ceil_div(ng, kMgBlock), kMgBlock, 0, c.stream>>>(ng, v.p + no, G.bc.p);
    PORO_LAUNCH_CHECK(c);
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

void mg_transfer_init(Ctx& c, MgTransfer& t, const StencilOp& fine, const StencilOp& coarse, DistPlan* cplan) {
    const StencilData& f = *fine.d;
    const StencilData& g = *coarse.d;
    const int fr = fine.fr;
    PORO_REQUIRE(fr >= 0 && fine.fc == fr && coarse.fr == fr && coarse.fc == fr, "mg: transfers link diagonal field blocks");
    PORO_REQUIRE(f.N == 2 * g.N && f.dim == g.dim && f.kind[fr] == g.kind[fr] && f.bdim[fr] == g.bdim[fr],
                 "mg: the coarse level is not the same field at N/2");
    PORO_REQUIRE(f.slab == g.slab && f.slab == (cplan != nullptr), "mg: slab levels need the halo plan of the coarse level");
    t.fine = fine;
    t.coarse = coarse;
    t.dim = f.dim;
    t.kind = f.kind[fr];
    t.br = f.bdim[fr];
    t.Nc = g.N;
    t.dist = f.slab;
    const int k = t.kind - 1;
    t.nf = t.dist ? f.o1[k] - f.o0[k] : porogen::lattice_nodes(t.kind, f.N, t.dim);
    t.nc = t.dist ? g.o1[k] - g.o0[k] : porogen::lattice_nodes(t.kind, g.N, t.dim);
    t.bcf = f.bc.p ? f.bc.p + f.row0[fr] : nullptr;
    t.bcc = g.bc.p ? g.bc.p + g.row0[fr] : nullptr;
    t.fg.o1 = t.nf;
    t.cg.o1 = t.nc;
    const poromg::Table P = poromg::prolong_table(t.kind, t.dim), R = poromg::restrict_table(t.kind, t.dim);
    upload(c, t.pptr, P.ptr);
    upload(c, t.pent, P.e);
    upload(c, t.rptr, R.ptr);
    upload(c, t.rent, R.e);
    t.ptab_bytes = (int64_t)(P.ptr.size() * sizeof(int) + P.e.size() * sizeof(poromg::Entry));
    t.rtab_bytes = (int64_t)(R.ptr.size() * sizeof(int) + R.e.size() * sizeof(poromg::Entry));
    if (!t.dist) return;
    const int64_t Lf = porogen::lattice_extent(t.kind, f.N), Lc = porogen::lattice_extent(t.kind, g.N);
    const int64_t pf = Lf * Lf, pc = Lc * Lc;            // nodes per plane of the slab axis (the cube)
    PORO_REQUIRE(t.dim == 3, "mg: row-partitioned slabs are z-slabs of the cube");
    const int64_t fa = f.o0[k] / pf, fb = f.o1[k] / pf, ca = g.o0[k] / pc, cb = g.o1[k] / pc;
    // prolongation: the coarse ghosts are the coarse block's halo; every plane the rows reach must be held there
    mg_ghosts(c, t.cg, *cplan, t.br, g.o0[k], g.o1[k], t.bcc);
    {
        int64_t lo, hi;
        poromg::plane_reach(P, t.dim, true, t.kind, fa, fb, Lc, lo, hi);
        std::vector<int> tab((size_t)t.cg.tab.n);
        if (!tab.empty()) PORO_CUDA(cudaMemcpy(tab.data(), t.cg.tab.p, tab.size() * sizeof(int), cudaMemcpyDeviceToHost));
        for (int64_t z = lo; z < hi; ++z) {
            if (z >= ca && z < cb) continue;
            const bool held = z * pc >= t.cg.g0 && (z + 1) * pc <= t.cg.g1;
            for (int64_t node = z * pc; held && node < (z + 1) * pc; ++node)
                PORO_REQUIRE(tab[node < g.o0[k] ? node - t.cg.g0 : g.o0[k] - t.cg.g0 + node - g.o1[k]] >= 0, "mg: a coarse node the "
                             "prolongation reads is missing from the coarse halo");
            PORO_REQUIRE(held, "mg: the prolongation of fine planes [" + std::to_string(fa) + ", " + std::to_string(fb) + ") reads coarse plane " +
                                   std::to_string(z) + ", outside the coarse halo");
        }
    }
    // restriction: a transfer halo of the fine planes the rows of the owned coarse planes reach (its width follows from the
    // table: up to 3 P2 planes below a slab whose first plane is a multiple of 4), exchanged by every restriction
    {
        int64_t lo, hi;
        poromg::plane_reach(R, t.dim, false, t.kind, ca, cb, Lf, lo, hi);
        std::vector<int> gid;
        for (int64_t node = std::min(lo, fa) * pf; node < fa * pf; ++node)
            for (int i = 0; i < t.br; ++i) gid.push_back((int)(node * t.br + i));
        for (int64_t node = fb * pf; node < std::max(hi, fb) * pf; ++node)
            for (int i = 0; i < t.br; ++i) gid.push_back((int)(node * t.br + i));
        t.tplan = std::make_unique<DistPlan>();
        plan_of_dofs(c, t.nf * t.br, gid, *t.tplan);
        mg_ghosts(c, t.fg, *t.tplan, t.br, f.o0[k], f.o1[k], t.bcf);
        t.tghost.alloc((size_t)t.tplan->n_ghost);
    }
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
    a.f = MgSide{t.fg.o0, t.fg.o1, t.fg.g0, t.fg.tab.p, t.bcf, t.fg.bc.p};
    a.c = MgSide{t.cg.o0, t.cg.o1, t.cg.g0, t.cg.tab.p, t.bcc, t.cg.bc.p};
    return a;
}

void mg_prolong(Ctx& c, const MgTransfer& t, const double* e, double* y, bool add) {
    const MgArgs a = mg_args(t, true);
    const int grid = (int)ceil_div(t.nf, kMgBlock);
    if (grid == 0) return;
    const double* eg = e + t.nc * t.br;
#define PORO_MG_P(BR)                                                                             \
    if (add) k_prolong<BR, true><<<grid, kMgBlock, 0, c.stream>>>(a, e, eg, y);                   \
    else k_prolong<BR, false><<<grid, kMgBlock, 0, c.stream>>>(a, e, eg, y);
    switch (t.br) {
        case 3: PORO_MG_P(3) break;
        case 2: PORO_MG_P(2) break;
        default: PORO_MG_P(1) break;
    }
#undef PORO_MG_P
    PORO_LAUNCH_CHECK(c);
}

void mg_restrict(Ctx& c, MgTransfer& t, const double* r, double* y) {
    if (t.dist) dist_halo_vec(c, *t.tplan, r, 1, t.tghost.p);      // collective: also on a rank without coarse rows
    const MgArgs a = mg_args(t, false);
    const int grid = (int)ceil_div(t.nc, kMgBlock);
    if (grid == 0) return;
    switch (t.br) {
        case 3: k_restrict<3><<<grid, kMgBlock, 0, c.stream>>>(a, r, t.tghost.p, y); break;
        case 2: k_restrict<2><<<grid, kMgBlock, 0, c.stream>>>(a, r, t.tghost.p, y); break;
        default: k_restrict<1><<<grid, kMgBlock, 0, c.stream>>>(a, r, t.tghost.p, y); break;
    }
    PORO_LAUNCH_CHECK(c);
}

// coarse owned node -> its coinciding fine node (fine lattice index = 2 x coarse), local on both levels
__global__ void k_mg_inject(int dim, int Lf, int Lc, int64_t fo0, int64_t co0, int64_t nc, int br, int k, const double* __restrict__ B,
                            double* __restrict__ Bc) {
    const int64_t t = (int64_t)blockIdx.x * kMgBlock + threadIdx.x;
    if (t >= nc * br * k) return;
    const int64_t row = t / k, node = row / br;
    int64_t q = co0 + node, fn = 0, mul = 1;
    for (int m = 0; m < dim; ++m) {
        fn += 2 * (q % Lc) * mul;
        q /= Lc;
        mul *= Lf;
    }
    Bc[t] = B[((fn - fo0) * br + row % br) * k + t % k];
}

void mg_inject(Ctx& c, const MgTransfer& t, const double* B, int k, DBuf<double>& Bc) {
    const int64_t n = t.nc * t.br * k;
    Bc.alloc((size_t)n);
    if (n == 0) return;
    k_mg_inject<<<(int)ceil_div(n, kMgBlock), kMgBlock, 0, c.stream>>>(t.dim, porogen::lattice_extent(t.kind, 2 * t.Nc),
                                                                        porogen::lattice_extent(t.kind, t.Nc), t.fg.o0, t.cg.o0, t.nc,
                                                                        t.br, k, B, Bc.p);
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
