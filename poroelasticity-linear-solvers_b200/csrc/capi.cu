// capi.cu -- the extern "C" boundary (include/poro.h): object lifetimes, field permutation,
// block extraction and the wiring of inner solvers from the PETSc-style options database.
#include "../../include/poro.h"
#include "ilu.cuh"
#include "solver.cuh"
#include <algorithm>
#include <cmath>

using namespace poro;

static thread_local std::string g_err;
const char* poro_last_error(void) { return g_err.c_str(); }
int poro_version(void) { return 100; }

#define API_BEGIN try {
#define API_END                                   \
    return 0;                                     \
    }                                             \
    catch (const std::exception& e) {             \
        g_err = e.what();                         \
        return -1;                                \
    }                                             \
    catch (...) {                                 \
        g_err = "unknown error";                  \
        return -1;                                \
    }

struct poro_ctx {
    Ctx c;
    Fields fl;
    HaloField raw_halo;
};
struct poro_mat {
    poro_ctx* ctx;
    Csr raw;
    DBuf<double> xext;
    int fuse_state = -1;         // poro_mat_mult_fused: -1 not tried, 0 refused, 1 the coupling rides along
};
struct poro_pc {
    poro_ctx* ctx;
    PCBlockCC cc;
    Csr Pperm;                   // permuted P (dropped after block extraction unless identity)
    DBuf<double> xp, yp;         // permuted work vectors for the raw-ordering apply
};
struct poro_ksp {
    poro_ctx* ctx;
    poro_pc* pc;
    std::unique_ptr<MatOp> A;
    KSP ksp;
    DBuf<double> bp, xp, bdev, xdev;
};
struct poro_aar {
    poro_ctx* ctx;
    poro_pc* pc;
    std::unique_ptr<MatOp> A;
    AAR aar;
    DBuf<double> bp, xp;
};

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
int poro_ctx_create(int device, poro_ctx** out) {
    API_BEGIN
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw Error("no CUDA device: libporo has no CPU fallback (" + std::string(cudaGetErrorString(e)) + ")");
    PORO_REQUIRE(device >= 0 && device < ndev, "device index out of range");
    PORO_CUDA(cudaSetDevice(device));
    auto* h = new poro_ctx();
    Ctx& c = h->c;
    c.device = device;
    cudaDeviceProp prop;
    PORO_CUDA(cudaGetDeviceProperties(&prop, device));
    c.sm_count = prop.multiProcessorCount;
    // a BLOCKING stream on purpose: it orders itself against the legacy default stream, i.e. against
    // plain cudaMemcpy calls in the set-up code and against torch's default-stream work on the buffers
    // handed across the ABI (tensor creation / H2D copies before a solve, reads after it)
    PORO_CUDA(cudaStreamCreate(&c.stream));
    PORO_CUDA(cudaMallocHost(&c.h_pin, 8192 * sizeof(double)));
    PORO_CUDA(cudaMalloc(&c.d_scal, ((size_t)Ctx::kScal + 8192) * sizeof(double)));
    PORO_CUDA(cudaMemset(c.d_scal, 0, ((size_t)Ctx::kScal + 8192) * sizeof(double)));
    *out = h;
    API_END
}

int poro_ctx_destroy(poro_ctx* h) {
    API_BEGIN
    if (!h) return 0;
    Ctx& c = h->c;
    cudaSetDevice(c.device);
    dist_finalize(c);
    for (auto e : c.prof.ev) cudaEventDestroy(e);
    if (c.t0) { cudaEventDestroy(c.t0); cudaEventDestroy(c.t1); }
    if (c.h_pin) cudaFreeHost(c.h_pin);
    if (c.d_scal) cudaFree(c.d_scal);
    if (c.stream) cudaStreamDestroy(c.stream);
    delete h;
    API_END
}

int poro_nccl_unique_id(unsigned char* id128) {
    API_BEGIN
    dist_get_unique_id(id128);
    API_END
}

int poro_ctx_init_dist(poro_ctx* h, int rank, int nranks, const unsigned char* id128) {
    API_BEGIN
    dist_init(h->c, rank, nranks, id128);
    API_END
}

// CUDA-event stopwatch on the library's stream (bench.py: device-side time of the K timed steps)
int poro_timer_start(poro_ctx* h) {
    API_BEGIN
    Ctx& c = h->c;
    if (!c.t0) { PORO_CUDA(cudaEventCreate(&c.t0)); PORO_CUDA(cudaEventCreate(&c.t1)); }
    PORO_CUDA(cudaEventRecord(c.t0, c.stream));
    API_END
}
int poro_timer_stop(poro_ctx* h, double* ms) {
    API_BEGIN
    Ctx& c = h->c;
    PORO_REQUIRE(c.t0 != nullptr, "poro_timer_stop without poro_timer_start");
    PORO_CUDA(cudaEventRecord(c.t1, c.stream));
    PORO_CUDA(cudaEventSynchronize(c.t1));
    float f = 0.f;
    PORO_CUDA(cudaEventElapsedTime(&f, c.t0, c.t1));
    *ms = f;
    API_END
}

int poro_options_set(poro_ctx* h, const char* key, const char* val) {
    API_BEGIN
    PORO_REQUIRE(key && key[0], "empty option key");
    std::string k = key;
    if (k[0] != '-') k = "-" + k;
    h->c.opts[k] = val ? val : "";
    API_END
}
int poro_options_clear(poro_ctx* h) {
    API_BEGIN
    h->c.opts.clear();
    API_END
}
int64_t poro_launch_count(poro_ctx* h) { return h ? h->c.launches : 0; }
int poro_sync(poro_ctx* h) {
    API_BEGIN
    PORO_CUDA(cudaStreamSynchronize(h->c.stream));
    API_END
}

// ---------------------------------------------------------------------------------------------
// matrices
// ---------------------------------------------------------------------------------------------
int poro_mat_create_csr(poro_ctx* h, int64_t nrows, int64_t ncols, const int64_t* rowptr, const int32_t* col,
                        const double* val, int on_device, poro_mat** out) {
    API_BEGIN
    Ctx& c = h->c;
    PORO_CUDA(cudaSetDevice(c.device));
    PORO_REQUIRE(nrows >= 0 && ncols >= 0 && nrows < 2147483647LL && ncols < 2147483647LL, "matrix dimensions out of range");
    auto m = std::make_unique<poro_mat>();
    m->ctx = h;
    if (!on_device) {
        csr_from_host(c, (int)nrows, (int)ncols, rowptr, col, val, m->raw);
    } else {
        std::vector<int64_t> rp((size_t)nrows + 1);
        PORO_CUDA(cudaMemcpy(rp.data(), rowptr, rp.size() * 8, cudaMemcpyDeviceToHost));
        int64_t nnz = rp[nrows];
        PORO_REQUIRE(nnz < 2147483647LL, "local matrix has more than 2^31 nonzeros: shard it over more GPUs");
        std::vector<int> rp32(rp.size());
        for (size_t i = 0; i < rp.size(); ++i) rp32[i] = (int)rp[i];
        Csr& A = m->raw;
        A.nrows = (int)nrows; A.ncols = (int)ncols; A.nnz = nnz;
        A.rowptr.alloc(rp.size()); A.col.alloc((size_t)nnz); A.val.alloc((size_t)nnz);
        PORO_CUDA(cudaMemcpy(A.rowptr.p, rp32.data(), rp32.size() * 4, cudaMemcpyHostToDevice));
        PORO_CUDA(cudaMemcpy(A.col.p, col, (size_t)nnz * 4, cudaMemcpyDeviceToDevice));
        PORO_CUDA(cudaMemcpy(A.val.p, val, (size_t)nnz * 8, cudaMemcpyDeviceToDevice));
        csr_choose_lanes(A);
    }
    m->raw.block_hint = c.opt_i("-poro_mat_block_hint", 0);   // micro-benchmarks: treat the raw matrix as node-blocked
    m->raw.fp32_hint = c.opt_i("-poro_mat_fp32_values", 0) != 0;
    *out = m.release();
    API_END
}

// helpers for gen.cu (the handle types are private to this file)
poro_mat* poro_mat_adopt(poro_ctx* h, Csr&& A) {
    auto m = std::make_unique<poro_mat>();
    m->ctx = h;
    m->raw = std::move(A);
    m->raw.block_hint = h->c.opt_i("-poro_mat_block_hint", 0);
    m->raw.fp32_hint = h->c.opt_i("-poro_mat_fp32_values", 0) != 0;
    return m.release();
}
Ctx& poro_ctx_ref(poro_ctx* h) { return h->c; }
void poro_set_error(const std::string& msg) { g_err = msg; }

// copy of the raw local CSR to host arrays sized from poro_mat_info (tests of the device-side generator)
int poro_mat_copy(poro_mat* m, int64_t* rowptr, int32_t* col, double* val) {
    API_BEGIN
    std::vector<int> rp, ci;
    std::vector<double> v;
    PORO_CUDA(cudaStreamSynchronize(m->ctx->c.stream));
    csr_to_host(m->raw, rp, ci, v);
    for (size_t i = 0; i < rp.size(); ++i) rowptr[i] = rp[i];
    for (size_t i = 0; i < ci.size(); ++i) { col[i] = ci[i]; val[i] = v[i]; }
    API_END
}

int poro_mat_destroy(poro_mat* m) {
    API_BEGIN
    delete m;
    API_END
}

int poro_mat_info(poro_mat* m, int64_t* nrows, int64_t* ncols, int64_t* nnz) {
    API_BEGIN
    if (nrows) *nrows = m->raw.nrows;
    if (ncols) *ncols = m->raw.ncols;
    if (nnz) *nnz = m->raw.nnz;
    API_END
}

int poro_mat_mult(poro_mat* m, const double* x, double* y) {
    API_BEGIN
    Ctx& c = m->ctx->c;
    const double* xin = x;
    if (c.nranks > 1 && m->ctx->raw_halo.n_halo > 0) {
        if ((int64_t)m->xext.n < m->raw.ncols) m->xext.alloc((size_t)m->raw.ncols);
        vec_copy(c, m->xext.p, x, m->raw.nrows);
        dist_halo_exchange(c, m->ctx->raw_halo, x, m->xext.p + m->raw.nrows);
        xin = m->xext.p;
    }
    spmv(c, m->raw, xin, y);
    API_END
}

int poro_mat_set_coarse(poro_mat* fine, poro_mat* coarse) {
    API_BEGIN
    PORO_REQUIRE(fine && coarse && fine != coarse, "poro_mat_set_coarse: two distinct matrices are needed");
    PORO_REQUIRE(fine->ctx == coarse->ctx, "poro_mat_set_coarse: the matrices belong to different contexts");
    const Csr& F = fine->raw;
    const Csr& G = coarse->raw;
    auto generated = [](const Csr& M) { return M.stencil && M.stencil->fr < 0; };
    PORO_REQUIRE(generated(F), "poro_mat_set_coarse: the fine matrix was not generated by poro_gen_matrix (whole lattices on one "
                               "rank, or a z-slab of the cube on several)");
    PORO_REQUIRE(generated(G), "poro_mat_set_coarse: the coarse matrix was not generated by poro_gen_matrix (whole lattices on one "
                               "rank, or a z-slab of the cube on several)");
    const StencilData& f = *F.stencil->d;
    const StencilData& g = *G.stencil->d;
    PORO_REQUIRE(f.slab == g.slab, "poro_mat_set_coarse: one matrix is a row-partitioned slab, the other holds whole lattices");
    if (f.slab) {
        // nested slabs: coarse P2 plane k is fine P2 plane 2k, so the coarse slab of fine planes [a, b) is [ceil(a/2), ceil(b/2))
        const int64_t sf = (int64_t)(2 * f.N + 1) * (2 * f.N + 1), sg = (int64_t)(2 * g.N + 1) * (2 * g.N + 1);
        const int64_t a = f.o0[1] / sf, b = f.o1[1] / sf, ca = g.o0[1] / sg, cb = g.o1[1] / sg;
        PORO_REQUIRE(f.N == 2 * g.N && ca == (a + 1) / 2 && cb == (b + 1) / 2,
                     "poro_mat_set_coarse: the slabs do not nest: fine P2 planes [" + std::to_string(a) + ", " + std::to_string(b) +
                         ") need coarse planes [" + std::to_string((a + 1) / 2) + ", " + std::to_string((b + 1) / 2) + "), the coarse slab owns [" +
                         std::to_string(ca) + ", " + std::to_string(cb) + ")");
    }
    PORO_REQUIRE(f.dim == g.dim, "poro_mat_set_coarse: dim differs (fine " + std::to_string(f.dim) + ", coarse " + std::to_string(g.dim) + ")");
    PORO_REQUIRE(f.N == 2 * g.N, "poro_mat_set_coarse: N_fine must be 2 N_coarse (fine N = " + std::to_string(f.N) + ", coarse N = " +
                                     std::to_string(g.N) + ")");
    for (int b = 0; b < 9; ++b)
        PORO_REQUIRE(f.present[b] == g.present[b], "poro_mat_set_coarse: the present tables differ (field block " + std::to_string(b / 3) +
                                                       "," + std::to_string(b % 3) + ")");
    for (int fld = 0; fld < 3; ++fld)
        PORO_REQUIRE(f.kind[fld] == g.kind[fld] && f.bdim[fld] == g.bdim[fld],
                     "poro_mat_set_coarse: lattice kind or block size of field " + std::to_string(fld) + " differs");
    PORO_REQUIRE((f.bc.p != nullptr) == (g.bc.p != nullptr), "poro_mat_set_coarse: one matrix has Dirichlet flags, the other none");
    // the fine descriptor keeps its own reference to the coarse matrix: destroying the coarse handle afterwards is safe
    auto keep = std::make_shared<Csr>();
    csr_copy(coarse->ctx->c, G, *keep);
    PORO_CUDA(cudaStreamSynchronize(coarse->ctx->c.stream));
    csr_choose_lanes(*keep);
    keep->stencil = G.stencil;
    F.stencil->d->coarse = std::move(keep);
    API_END
}

// one product in epilogue mode `mode` (include/poro.h, poro_pc_block_mult); `op` applies modes 0..2 when given, else B does
static void mult_in_mode(Ctx& c, const Csr& B, MatOp* op, int mode, const double* x, double* y, const double* z, double* r,
                         double* d_new, double* xv, const double* dinv, double c1, double c2, double* dot) {
    PORO_REQUIRE(mode >= 0 && mode <= 4, "mode in 0..4");
    PORO_REQUIRE(mode <= 2 || B.nrows == B.ncols, "Chebyshev / dot modes need a square matrix");
    if (mode <= 2 && op) op->apply(x, y, (SpmvMode)mode, z);
    else if (mode <= 2) spmv(c, B, x, y, (SpmvMode)mode, z);
    else if (mode == 3) spmv_cheb_step(c, B, x, x, d_new, r, xv, dinv, c1, c2);
    else spmv_dot(c, B, x, y, dot);
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

int poro_mat_mult_mode(poro_mat* m, int mode, const double* x, double* y, const double* z, double* r, double* d_new, double* xv,
                       const double* dinv, double c1, double c2, double* dot) {
    API_BEGIN
    PORO_REQUIRE(m->ctx->c.nranks == 1, "poro_mat_mult_mode: single rank only");
    mult_in_mode(m->ctx->c, m->raw, nullptr, mode, x, y, z, r, d_new, xv, dinv, c1, c2, dot);
    API_END
}

int poro_mat_kernel_info(poro_mat* m, int64_t* out, int n) {
    API_BEGIN
    int64_t v[kSpmvInfoFields];
    spmv_kernel_info(m->ctx->c, m->raw, v);
    for (int i = 0; i < n; ++i) out[i] = i < kSpmvInfoFields ? v[i] : 0;
    API_END
}

int poro_mat_mult_fused(poro_mat* a, poro_mat* cpl, int mode, const double* x, const double* x2, double* y, const double* z, int* fused) {
    API_BEGIN
    Ctx& c = a->ctx->c;
    const Csr& A = a->raw;
    const Csr& C = cpl->raw;
    PORO_REQUIRE(mode >= 0 && mode <= 2, "mode in 0..2");
    PORO_REQUIRE(C.nrows == A.nrows, "the coupling must have the rows of the matrix");
    if (a->fuse_state < 0) a->fuse_state = csr_fuse_coupling(c, A, C) ? 1 : 0;
    if (a->fuse_state == 1) spmv_fused(c, A, x, x2, y, (SpmvMode)mode, z);
    else {
        spmv(c, A, x, y, (SpmvMode)mode, z);
        spmv(c, C, x2, y, mode == SPMV_SET ? SPMV_ADD : (SpmvMode)mode, y);
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    if (fused) *fused = a->fuse_state;
    API_END
}

// micro-benchmark of one matrix in one epilogue mode: 0 y = A x, 1 y = z - A x, 2 y = z + A x, 3 fused Chebyshev step,
// 4 w = A p with p.w; device time per launch by CUDA events on the library's stream (vectors are internal)
int poro_mat_bench(poro_mat* m, int mode, int reps, double* ms_per_launch) {
    API_BEGIN
    Ctx& c = m->ctx->c;
    const Csr& A = m->raw;
    PORO_REQUIRE(A.nrows == A.ncols || mode <= 2, "Chebyshev / dot modes need a square matrix");
    PORO_REQUIRE(mode >= 0 && mode <= 4 && reps > 0, "mode in 0..4, reps > 0");
    const int64_t n = A.nrows, nc = A.ncols;
    DBuf<double> x((size_t)nc), y((size_t)n), z((size_t)n), r((size_t)n), d1((size_t)n), dinv((size_t)n), xv((size_t)n);
    vec_set(c, x.p, 1.0, nc); vec_set(c, z.p, 0.5, n); vec_set(c, r.p, 0.25, n); vec_set(c, dinv.p, 1e-3, n); vec_set(c, xv.p, 0.0, n);
    auto once = [&]() {
        if (mode == 0) spmv(c, A, x.p, y.p);
        else if (mode == 1) spmv(c, A, x.p, y.p, SPMV_SUB, z.p);
        else if (mode == 2) spmv(c, A, x.p, y.p, SPMV_ADD, z.p);
        else if (mode == 3) spmv_cheb_step(c, A, x.p, x.p, d1.p, r.p, xv.p, dinv.p, 0.3, 0.1);
        else spmv_dot(c, A, x.p, y.p, c.d_scal + Ctx::kScal + 4096);
    };
    for (int i = 0; i < 3; ++i) once();
    cudaEvent_t e0, e1;
    PORO_CUDA(cudaEventCreate(&e0));
    PORO_CUDA(cudaEventCreate(&e1));
    PORO_CUDA(cudaEventRecord(e0, c.stream));
    for (int i = 0; i < reps; ++i) once();
    PORO_CUDA(cudaEventRecord(e1, c.stream));
    PORO_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    PORO_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_per_launch = ms / reps;
    API_END
}

// ---------------------------------------------------------------------------------------------
// halo plan and index sets
// ---------------------------------------------------------------------------------------------
int poro_halo_set(poro_ctx* h, int64_t n_owned, int nneigh, const int32_t* neigh, const int64_t* send_ptr,
                  const int32_t* send_idx, const int64_t* recv_count) {
    API_BEGIN
    Ctx& c = h->c;
    c.n_owned_raw = nneigh > 0 ? n_owned : -1;       // no neighbours: back to the single-rank layout (everything is owned)
    c.neigh.assign(neigh, neigh + nneigh);
    c.raw_send_ptr.assign(send_ptr, send_ptr + nneigh + 1);
    c.raw_send_idx.assign(send_idx, send_idx + send_ptr[nneigh]);
    c.raw_recv_count.assign(recv_count, recv_count + nneigh);
    HaloField& hf = h->raw_halo;
    hf.send_ptr = c.raw_send_ptr;
    hf.recv_ptr.assign(nneigh + 1, 0);
    for (int k = 0; k < nneigh; ++k) hf.recv_ptr[k + 1] = hf.recv_ptr[k] + recv_count[k];
    hf.n_halo = hf.recv_ptr[nneigh];
    hf.send_idx.alloc(c.raw_send_idx.size());
    hf.send_buf.alloc(c.raw_send_idx.size());
    if (!c.raw_send_idx.empty())
        PORO_CUDA(cudaMemcpy(hf.send_idx.p, c.raw_send_idx.data(), c.raw_send_idx.size() * 4, cudaMemcpyHostToDevice));
    if (c.nranks > 1) p2p_slots_setup(c, c.neigh, hf.send_ptr, hf.recv_ptr, hf.p2p);
    API_END
}

int poro_fields_set(poro_ctx* h, const int64_t* is_s, int64_t ns, const int64_t* is_f, int64_t nf, const int64_t* is_p,
                    int64_t np, const int64_t* is_fp, int64_t nfp, int two_way_local_fp, int block_dim) {
    API_BEGIN
    Ctx& c = h->c;
    Fields& fl = h->fl;
    const int64_t n_ext = ns + nf + np;
    const int64_t n_owned = c.n_owned_raw >= 0 ? c.n_owned_raw : n_ext;
    std::vector<int64_t> lists[3];
    lists[0].assign(is_s, is_s + ns);
    if (two_way_local_fp) {
        PORO_REQUIRE(is_fp && nfp == nf + np, "two-way remap needs is_fp with nf + np entries");
        lists[1].resize(nf);
        lists[2].resize(np);
        for (int64_t i = 0; i < nf; ++i) { PORO_REQUIRE(is_f[i] >= 0 && is_f[i] < nfp, "is_f out of the fp range"); lists[1][i] = is_fp[is_f[i]]; }
        for (int64_t i = 0; i < np; ++i) { PORO_REQUIRE(is_p[i] >= 0 && is_p[i] < nfp, "is_p out of the fp range"); lists[2][i] = is_fp[is_p[i]]; }
    } else {
        lists[1].assign(is_f, is_f + nf);
        lists[2].assign(is_p, is_p + np);
    }
    std::vector<int> field_of((size_t)n_ext, -1), new_of_old((size_t)n_ext, -1);
    std::vector<int64_t> halo_lists[3];
    for (int t = 0; t < 3; ++t) {
        fl.n[t] = 0;
        for (int64_t g : lists[t]) {
            PORO_REQUIRE(g >= 0 && g < n_ext, "index set entry out of range");
            PORO_REQUIRE(field_of[g] < 0, "index sets overlap");
            field_of[g] = t;
            if (g < n_owned) fl.n[t]++; else halo_lists[t].push_back(g);
        }
    }
    fl.off[0] = 0; fl.off[1] = fl.n[0]; fl.off[2] = fl.n[0] + fl.n[1];
    fl.n_owned = n_owned;
    fl.n_ext = n_ext;
    PORO_REQUIRE(fl.n[0] + fl.n[1] + fl.n[2] == n_owned, "index sets do not cover the owned dofs");
    int64_t ho = 0;
    for (int t = 0; t < 3; ++t) {
        std::sort(halo_lists[t].begin(), halo_lists[t].end());
        fl.nh[t] = (int64_t)halo_lists[t].size();
        fl.hoff[t] = ho;
        ho += fl.nh[t];
    }
    for (int t = 0; t < 3; ++t) {
        int64_t k = 0;
        for (int64_t g : lists[t]) if (g < n_owned) new_of_old[g] = (int)(fl.off[t] + k++);
        k = 0;
        for (int64_t g : halo_lists[t]) new_of_old[g] = (int)(n_owned + fl.hoff[t] + k++);
    }
    fl.identity = fl.owned_identity = true;
    for (int64_t g = 0; g < n_ext; ++g)
        if (new_of_old[g] != (int)g) {
            fl.identity = false;
            if (g < n_owned) fl.owned_identity = false;
        }
    std::vector<int> old_of_new((size_t)n_owned);
    for (int64_t g = 0; g < n_owned; ++g) old_of_new[new_of_old[g]] = (int)g;
    fl.new_of_old.alloc((size_t)n_ext);
    fl.old_of_new.alloc((size_t)n_owned);
    PORO_CUDA(cudaMemcpy(fl.new_of_old.p, new_of_old.data(), (size_t)n_ext * 4, cudaMemcpyHostToDevice));
    PORO_CUDA(cudaMemcpy(fl.old_of_new.p, old_of_new.data(), (size_t)n_owned * 4, cudaMemcpyHostToDevice));
    fl.block_dim = block_dim;
    // per-field halo plans
    const int nneigh = (int)c.neigh.size();
    for (int t = 0; t < 3; ++t) {
        HaloField& hf = fl.halo[t];
        hf.send_ptr.assign(nneigh + 1, 0);
        hf.recv_ptr.assign(nneigh + 1, 0);
        std::vector<int> sidx;
        int64_t rbase = n_owned;
        for (int k = 0; k < nneigh; ++k) {
            for (int64_t q = c.raw_send_ptr[k]; q < c.raw_send_ptr[k + 1]; ++q) {
                int g = c.raw_send_idx[q];
                if (field_of[g] == t) sidx.push_back(new_of_old[g] - (int)fl.off[t]);
            }
            hf.send_ptr[k + 1] = (int64_t)sidx.size();
            int64_t cnt = 0;
            for (int64_t g = rbase; g < rbase + c.raw_recv_count[k]; ++g) if (field_of[g] == t) cnt++;
            hf.recv_ptr[k + 1] = hf.recv_ptr[k] + cnt;
            rbase += c.raw_recv_count[k];
        }
        hf.n_halo = hf.recv_ptr[nneigh];
        PORO_REQUIRE(hf.n_halo == fl.nh[t], "halo plan and index sets disagree");
        hf.send_idx.alloc(sidx.size());
        hf.send_buf.alloc(sidx.size());
        if (!sidx.empty()) PORO_CUDA(cudaMemcpy(hf.send_idx.p, sidx.data(), sidx.size() * 4, cudaMemcpyHostToDevice));
        if (c.nranks > 1) p2p_slots_setup(c, c.neigh, hf.send_ptr, hf.recv_ptr, hf.p2p);     // collective (same order on every rank)
    }
    fl.set = true;
    API_END
}

int poro_fields_set_coords(poro_ctx* h, int dim, const double* coords_s, const double* coords_p) {
    API_BEGIN
    Fields& fl = h->fl;
    PORO_REQUIRE(fl.set, "call poro_fields_set first");
    fl.coord_dim = dim;
    // coordinates are given in the order of the s index set (owned entries first in that order)
    if (coords_s) fl.coords_s.assign(coords_s, coords_s + (size_t)fl.n[0] * dim);
    if (coords_p) fl.coords_p.assign(coords_p, coords_p + (size_t)fl.n[2] * dim);
    API_END
}

// ---------------------------------------------------------------------------------------------
// block extraction helpers
// ---------------------------------------------------------------------------------------------
// the fields of the solver are the generator's fields in the generator's order, and nothing lives in a halo
static bool stencil_layout_matches(const Fields& fl, const StencilOp& s) {
    if (!fl.identity) return false;
    for (int t = 0; t < 3; ++t)
        if (fl.nh[t] || fl.off[t] != s.d->row0[t] || fl.n[t] != s.d->row0[t + 1] - s.d->row0[t]) return false;
    return true;
}

// the owned rows of the solver's fields are the generator's owned rows in the generator's order (halos may be reordered)
static bool slab_layout_matches(const Fields& fl, const StencilOp& s) {
    if (!fl.owned_identity || !s.d->slab) return false;
    for (int t = 0; t < 3; ++t)
        if (fl.off[t] != s.d->row0[t] || fl.n[t] != s.d->row0[t + 1] - s.d->row0[t]) return false;
    return true;
}

// columns: list of (field) pieces in order; rows: contiguous permuted range [r0, r1)
static std::unique_ptr<MatOp> extract_block(poro_ctx* h, const Csr& Mp, int64_t r0, int64_t r1, std::vector<int> col_fields) {
    Ctx& c = h->c;
    Fields& fl = h->fl;
    auto op = std::make_unique<MatOp>();
    op->ctx = &c;
    std::vector<int> cmap((size_t)fl.n_ext, -1), rmap((size_t)fl.n_owned, -1);
    for (int64_t i = r0; i < r1; ++i) rmap[i] = (int)(i - r0);
    int64_t pos = 0;
    std::vector<int64_t> owned_pos(3, 0);
    for (int t : col_fields) {
        owned_pos[t] = pos;
        for (int64_t i = 0; i < fl.n[t]; ++i) cmap[fl.off[t] + i] = (int)(pos + i);
        pos += fl.n[t];
    }
    op->n_owned_cols = pos;
    for (int t : col_fields) {
        // multi-rank: the exchange is collective, so a rank without ghosts of field t still takes part (it may have to send)
        if (fl.nh[t] || c.nranks > 1) {
            for (int64_t i = 0; i < fl.nh[t]; ++i) cmap[fl.n_owned + fl.hoff[t] + i] = (int)(pos + i);
            op->pieces.push_back({&fl.halo[t], owned_pos[t], pos});
            pos += fl.nh[t];
        }
    }
    DBuf<int> d_r(rmap.size()), d_c(cmap.size());
    PORO_CUDA(cudaMemcpy(d_r.p, rmap.data(), rmap.size() * 4, cudaMemcpyHostToDevice));
    PORO_CUDA(cudaMemcpy(d_c.p, cmap.data(), cmap.size() * 4, cudaMemcpyHostToDevice));
    csr_extract(c, Mp, d_r.p, d_c.p, (int)(r1 - r0), (int)pos, op->M);
    // a generated matrix cut along whole fields (one row field x one column field) keeps its tables: the block's products
    // run from them (stencil.cu).  Partial ranges, several column fields and permuted matrices stay assembled.
    if (Mp.stencil && Mp.stencil->fr < 0 && c.nranks == 1 && col_fields.size() == 1 && stencil_layout_matches(fl, *Mp.stencil)) {
        for (int fr = 0; fr < 3; ++fr)
            if (fl.n[fr] > 0 && r0 == fl.off[fr] && r1 == fl.off[fr] + fl.n[fr]) {
                op->M.stencil = std::make_shared<StencilOp>(StencilOp{Mp.stencil->d, fr, col_fields[0]});
                break;
            }
    }
    // a diagonal field block of a row-partitioned slab keeps its descriptor for `-<prefix>pc_type mg` (never applied from it)
    if (Mp.stencil && Mp.stencil->fr < 0 && c.nranks > 1 && col_fields.size() == 1 && slab_layout_matches(fl, *Mp.stencil)) {
        const int fr = col_fields[0];
        if (r0 == fl.off[fr] && r1 == fl.off[fr] + fl.n[fr]) op->M.stencil = std::make_shared<StencilOp>(StencilOp{Mp.stencil->d, fr, fr});
    }
    return op;
}

// square local part (owned columns only) of a block operator: what the inner PCs are built on
static void local_square(Ctx& c, const MatOp& op, Csr& out) {
    const Csr& M = op.mat();
    if (M.ncols == M.nrows) {
        csr_copy(c, M, out);
        out.stencil = M.stencil;        // the same operator
        PORO_CUDA(cudaStreamSynchronize(c.stream));
        return;
    }
    std::vector<int> rmap((size_t)M.nrows), cmap((size_t)M.ncols, -1);
    for (int i = 0; i < M.nrows; ++i) { rmap[i] = i; cmap[i] = i; }
    DBuf<int> d_r(rmap.size()), d_c(cmap.size());
    PORO_CUDA(cudaMemcpy(d_r.p, rmap.data(), rmap.size() * 4, cudaMemcpyHostToDevice));
    PORO_CUDA(cudaMemcpy(d_c.p, cmap.data(), cmap.size() * 4, cudaMemcpyHostToDevice));
    csr_extract(c, M, d_r.p, d_c.p, M.nrows, M.nrows, out);
}

static void permute_matrix(poro_ctx* h, const Csr& raw, Csr& out) {
    Fields& fl = h->fl;
    PORO_REQUIRE(raw.nrows == fl.n_owned && raw.ncols == fl.n_ext, "matrix shape does not match the index sets");
    csr_extract(h->c, raw, fl.new_of_old.p, fl.new_of_old.p, (int)fl.n_owned, (int)fl.n_ext, out);
}

// an elliptic inner solver: KSP(type) + PC(type) then options with `prefix` (lib/Preconditioner.py:94-100)
static std::unique_ptr<KSP> make_inner(poro_ctx* h, MatOp* op, const std::string& ksp_type, const std::string& pc_type,
                                       const std::string& prefix, int bs, const double* coords, int cdim) {
    Ctx& c = h->c;
    if (c.has_opt("-poro_verbose"))
        fprintf(stderr, "  [pc] inner solver %s: n=%d nnz=%lld bs=%d\n", prefix.c_str(), op->mat().nrows, (long long)op->mat().nnz, bs);
    auto k = std::make_unique<KSP>();
    k->ctx = &c;
    k->A = op;
    k->type = ksp_type;
    k->set_from_options(prefix);
    std::string pt = c.opt("-" + prefix + "pc_type", pc_type);
    if (pt == "fieldsplit") pt = "amg";
    const Csr* src = &op->mat();
    const bool amg_type = pt == "hypre" || pt == "amg" || pt == "gamg" || pt == "ml" || pt == "chebyshev" || pt == "mg";
    // row-partitioned runs: hierarchies are distributed (global Galerkin coarse levels, distamg.cu) whenever the block has
    // ONE halo plan; the decision uses global sizes so that every rank takes the same (collective) path
    DistPlan* plan = nullptr;
    if (c.nranks > 1 && (amg_type || pt == "lu") && c.opt_i("-poro_amg_distributed", 1)) plan = op->plan_for_amg();
    const int64_t rows_glob = plan ? plan->offsets.back() : src->nrows;
    if (c.nranks > 1 && (pt == "lu" || pt == "cholesky") && c.opt("-" + prefix + "pc_factor_mat_solver_type", "") == "poro")
        throw Error("-" + prefix + "pc_factor_mat_solver_type poro: the sparse LU factorises a block on one GPU, this block is "
                    "row-partitioned over " + std::to_string(c.nranks) + " ranks");
    // with -<prefix>pc_factor_mat_solver_type poro a block above the dense limit is factorised (PCSparseLU, via make_pc)
    const bool big_lu = pt == "lu" && rows_glob > c.opt_i("-poro_dense_lu_limit", 8192) && !use_sparse_lu(c, pt, prefix, rows_glob);
    if (amg_type || big_lu) {
        // the AMG keeps a pointer to its finest operator: it must live as long as the KSP.  A square block (single rank) or
        // a distributed block with its plan is used in place; otherwise the owned-column part is cut out and kept in owned_op.
        std::unique_ptr<MatOp> holder;
        if (!plan && src->ncols != src->nrows) {
            holder = std::make_unique<MatOp>();
            holder->ctx = &c;
            local_square(c, *op, holder->M);
            csr_choose_lanes(holder->M);
            holder->M.block_hint = bs;
            src = &holder->M;
        }
        k->owned_pc = make_pc(c, pt, *src, bs, coords, cdim, prefix, plan);
        if (pt == "lu") {
            // "exact" block too large for a dense factorisation: iterate to tight tolerance instead
            k->type = c.opt("-" + prefix + "poro_exact_ksp_type", "gmres");
            k->rtol = c.opt_d("-" + prefix + "poro_exact_rtol", 1e-12);
            k->atol = 1e-300;
            k->max_it = 500;
            k->restart = 100;
            k->right = true;
        }
        k->owned_op = std::move(holder);
    } else {
        Csr loc;
        if (src->ncols != src->nrows) { local_square(c, *op, loc); src = &loc; }
        k->owned_pc = make_pc(c, pt, *src, bs, coords, cdim, prefix);
    }
    k->pc = k->owned_pc.get();
    if (PCAmg* a = dynamic_cast<PCAmg*>(k->pc))
        a->amg.prof_base = prefix == "s_" ? 8 : (bs > 1 ? 16 : (prefix.find("fieldsplit") != std::string::npos ? 24 : -1));
    return k;
}

// ---------------------------------------------------------------------------------------------
// preconditioner
// ---------------------------------------------------------------------------------------------
int poro_pc_setup(poro_ctx* h, poro_mat* A, poro_mat* P, poro_mat* P_diff, const char* pc_type_c,
                  const char* inner_ksp_type_c, const char* inner_pc_type_c, const int64_t* bcs_sub_pressure, int64_t nbc,
                  int accel_order, double w1, double w2, poro_pc** out) {
    API_BEGIN
    Ctx& c = h->c;
    Fields& fl = h->fl;
    PORO_CUDA(cudaSetDevice(c.device));
    PORO_REQUIRE(fl.set, "call poro_fields_set before poro_pc_setup");
    std::string pc_type = pc_type_c ? pc_type_c : "diagonal";
    std::string iksp = inner_ksp_type_c ? inner_ksp_type_c : "gmres";
    std::string ipc = inner_pc_type_c ? inner_pc_type_c : "hypre";
    static const char* valid[] = {"undrained", "undrained 3-way", "diagonal", "diagonal 3-way", "diagonal 3-way-II", "lu"};
    bool ok = false;
    for (auto v : valid) ok = ok || pc_type == v;
    if (!ok) throw Error("pc type must be one of lu, undrained, diagonal, diagonal 3-way, diagonal 3-way-II.");   // Preconditioner.py:278-280
    auto pc = std::make_unique<poro_pc>();
    pc->ctx = h;
    PCBlockCC& cc = pc->cc;
    cc.ctx = &c;
    cc.fl = &fl;
    cc.three_way = pc_type == "diagonal 3-way" || pc_type == "undrained 3-way";   // Preconditioner.py:283
    cc.w1 = w1;
    cc.w2 = w2;
    cc.timing = c.has_opt("-poro_pc_timing");
    const Csr* Pp = &P->raw;
    if (!fl.identity) { permute_matrix(h, P->raw, pc->Pperm); Pp = &pc->Pperm; }
    else PORO_REQUIRE(P->raw.nrows == fl.n_owned && P->raw.ncols == fl.n_ext, "P shape does not match the index sets");
    const int64_t ns = fl.n[0], nf = fl.n[1], np = fl.n[2];
    const int64_t os = fl.off[0], of = fl.off[1], op_ = fl.off[2];
    const int bd = fl.block_dim;
    const int bs_v = (bd > 0 && ns % bd == 0 && nf % bd == 0) ? bd : 1;
    const double* cs = fl.coords_s.empty() ? nullptr : fl.coords_s.data();
    const int cdim = fl.coord_dim;
    cc.Ms_s = extract_block(h, *Pp, os, os + ns, {0});
    cc.Ms_s->M.block_hint = bs_v;          // also with halo columns: any grouping of columns in triples is valid
    cc.ksp_s = make_inner(h, cc.Ms_s.get(), iksp, ipc, "s_", bs_v, cs, cdim);
    cc.t_s.alloc(ns); cc.t_f.alloc(nf); cc.t_p.alloc(np); cc.t_fp.alloc(nf + np);
    if (cc.three_way) {
        PORO_REQUIRE(P_diff != nullptr, "3-way splittings need P_diff");
        cc.Ms_f = extract_block(h, *Pp, os, os + ns, {1});
        cc.Ms_p = extract_block(h, *Pp, os, os + ns, {2});
        cc.Mf_f = extract_block(h, *Pp, of, of + nf, {1});
        cc.Mf_f->M.block_hint = bs_v;
        cc.Mf_p = extract_block(h, *Pp, of, of + nf, {2});
        cc.Mp_p = extract_block(h, *Pp, op_, op_ + np, {2});
        {
            Csr Dp;
            const Csr* Dsrc = &P_diff->raw;
            if (!fl.identity) { permute_matrix(h, P_diff->raw, Dp); Dsrc = &Dp; }
            cc.Mp_diff = extract_block(h, *Dsrc, op_, op_ + np, {2});
        }
        cc.ksp_f = make_inner(h, cc.Mf_f.get(), iksp, ipc, "f_", bs_v, cs, cdim);
        cc.ksp_p = make_inner(h, cc.Mp_p.get(), iksp, ipc, "p_", 1, nullptr, 0);
        cc.ksp_diff = make_inner(h, cc.Mp_diff.get(), iksp, ipc, "diff_", 1, nullptr, 0);
        cc.y_sd.alloc(ns); cc.y_fd.alloc(nf); cc.y_pd.alloc(np);
        if (nbc > 0) {
            std::vector<int> b32((size_t)nbc);
            for (int64_t i = 0; i < nbc; ++i) { PORO_REQUIRE(bcs_sub_pressure[i] >= 0 && bcs_sub_pressure[i] < np, "pressure BC index out of range"); b32[i] = (int)bcs_sub_pressure[i]; }
            cc.bcs_sub_pressure.alloc((size_t)nbc);
            PORO_CUDA(cudaMemcpy(cc.bcs_sub_pressure.p, b32.data(), (size_t)nbc * 4, cudaMemcpyHostToDevice));
        }
    } else {
        cc.Mfp_s = extract_block(h, *Pp, of, of + nf + np, {0});
        // fp solver: lib/Preconditioner.py:135-138: LU on the whole block, or GMRES + fieldsplit then options
        std::string fp_pc = ipc == "lu" ? "lu" : c.opt("-fp_pc_type", "fieldsplit");
        // an "exact" fp block too large for the dense inverse: the fp block is a non-symmetric saddle-type matrix on
        // which AMG is meaningless, so iterate GMRES on it to 1e-12 with a full Schur factorisation whose sub-blocks
        // are themselves exact (dense) or tightly iterated
        const bool fp_exact_big = fp_pc == "lu" && (nf + np) > c.opt_i("poro_dense_lu_limit", 8192);
        // ... unless -fp_pc_factor_mat_solver_type poro asks for the sparse LU of the whole block
        if (fp_pc != "fieldsplit" && (!fp_exact_big || use_sparse_lu(c, fp_pc, "fp_", nf + np))) {
            cc.Mfp_fp = extract_block(h, *Pp, of, of + nf + np, {1, 2});
            cc.ksp_fp = make_inner(h, cc.Mfp_fp.get(), ipc == "lu" ? iksp : "gmres", fp_pc, "fp_", 1, nullptr, 0);
        } else {
            auto k = std::make_unique<KSP>();
            k->ctx = &c;
            k->type = "gmres";
            k->set_from_options("fp_");
            if (fp_exact_big) {
                k->type = "gmres"; k->rtol = 1e-12; k->atol = 1e-300; k->max_it = 400; k->restart = 200; k->right = true;
            }
            auto sch = std::make_unique<PCSchur>();
            sch->ctx = &c;
            // the exact big block always runs the full Schur factorisation
            const std::string fs_type = fp_exact_big ? "schur" : c.opt("-fp_pc_fieldsplit_type", "schur");
            if (fs_type == "additive") sch->type = FS_ADDITIVE;
            else if (fs_type == "multiplicative") sch->type = FS_MULTIPLICATIVE;
            else if (fs_type != "schur")
                throw Error("-fp_pc_fieldsplit_type " + fs_type + " is not supported (schur, additive or multiplicative; two splits)");
            std::string order = c.opt("-fp_pc_fieldsplit_order", fp_exact_big ? "fp" : "pf");   // "pf" = reference (Preconditioner.py:113-114)
            sch->p_first = order != "fp";
            std::string fact = c.opt("-fp_pc_fieldsplit_schur_fact_type", fp_exact_big ? "full" : "lower");
            sch->fact = fact == "lower" ? 0 : fact == "upper" ? 1 : fact == "full" ? 2 : fact == "diag" ? 3 : -1;
            PORO_REQUIRE(sch->fact >= 0, "unknown -fp_pc_fieldsplit_schur_fact_type");
            const int t0 = sch->p_first ? 2 : 1, t1 = sch->p_first ? 1 : 2;
            sch->n0 = fl.n[t0]; sch->n1 = fl.n[t1];
            sch->off0 = sch->p_first ? nf : 0;
            sch->off1 = sch->p_first ? 0 : nf;
            sch->A00 = extract_block(h, *Pp, fl.off[t0], fl.off[t0] + fl.n[t0], {t0});
            sch->A01 = extract_block(h, *Pp, fl.off[t0], fl.off[t0] + fl.n[t0], {t1});
            sch->A10 = extract_block(h, *Pp, fl.off[t1], fl.off[t1] + fl.n[t1], {t0});
            sch->A11 = extract_block(h, *Pp, fl.off[t1], fl.off[t1] + fl.n[t1], {t1});
            (t0 == 1 ? sch->A00 : sch->A11)->M.block_hint = bs_v;
            if (sch->type != FS_SCHUR) {
                // PETSc's defaults for the sub-solvers: preonly + ILU(0), block Jacobi + ILU(0) on a row-partitioned block
                const char* sub_pc = c.nranks > 1 ? "bjacobi" : "ilu";
                const int bs0 = t0 == 1 ? bs_v : 1, bs1 = t1 == 1 ? bs_v : 1;
                sch->k0 = make_inner(h, sch->A00.get(), "preonly", sub_pc, "fp_fieldsplit_0_", bs0, t0 == 1 ? cs : nullptr, t0 == 1 ? cdim : 0);
                sch->k1 = make_inner(h, sch->A11.get(), "preonly", sub_pc, "fp_fieldsplit_1_", bs1, t1 == 1 ? cs : nullptr, t1 == 1 ? cdim : 0);
                sch->t1.alloc((size_t)sch->n1);
            } else {
                // selfp: S = A11 - A10 diag(A00)^-1 A01
                // cc (extension): the diagonal is the lumped mass + drag part of the velocity block, mass_scale * |diag(A_fs)| of
                // the SYSTEM matrix (A_fs = -(phi^2 / (k_f dt)) M_v with the rows of fluid Dirichlet dofs zeroed, which then get 1),
                // and the viscous limit visc_scale * P_pp is added in the application (PCSchur::solve1); oracle: SchurLowerCC
                const std::string sprec = c.opt("-fp_pc_fieldsplit_schur_precondition", "selfp");
                PORO_REQUIRE(sprec == "selfp" || sprec == "cc", "-fp_pc_fieldsplit_schur_precondition must be selfp or cc");
                DBuf<double> d_mass;
                if (sprec == "cc") {
                    PORO_REQUIRE(!sch->p_first && pc_type == "diagonal", "schur_precondition cc needs pc type 'diagonal' and -fp_pc_fieldsplit_order fp");
                    PORO_REQUIRE(A != nullptr && c.has_opt("-fp_pc_fieldsplit_schur_cc_mass_scale") && c.has_opt("-fp_pc_fieldsplit_schur_cc_visc_scale"),
                                 "schur_precondition cc needs A and the -fp_pc_fieldsplit_schur_cc_mass_scale / _visc_scale options (lib/Preconditioner.py sets them)");
                    PORO_REQUIRE(ns == nf, "schur_precondition cc expects the displacement and velocity fields on the same nodes");
                    const double ms = c.opt_d("-fp_pc_fieldsplit_schur_cc_mass_scale", 0.0);
                    sch->visc_scale = c.opt_d("-fp_pc_fieldsplit_schur_cc_visc_scale", 0.0);
                    PORO_REQUIRE(ms > 0.0 && sch->visc_scale > 0.0, "schur_precondition cc: the two scales must be positive");
                    Csr Aperm;
                    const Csr* Ap = &A->raw;
                    if (!fl.identity) { permute_matrix(h, A->raw, Aperm); Ap = &Aperm; }
                    auto Afs = extract_block(h, *Ap, of, of + nf, {0});
                    d_mass.alloc((size_t)nf);
                    csr_diag(c, Afs->M, d_mass.p);
                    vec_abs_scale(c, d_mass.p, ms, nf);
                    PORO_CUDA(cudaStreamSynchronize(c.stream));
                }
                DistPlan* plan0 = nullptr;
                DistPlan* plan1 = nullptr;
                if (c.nranks > 1 && c.opt_i("-poro_amg_distributed", 1)) { plan0 = sch->A00->plan_for_amg(); plan1 = sch->A11->plan_for_amg(); }
                if (plan0 && plan1) {
                    // row-partitioned: exact complement of the owned rows -- the A01 rows and the diagonal of the ghost dofs of split 0
                    // arrive by one sparse-row and one vector exchange; S gets its own (wider) halo plan
                    sch->S = std::make_unique<MatOp>();
                    sch->S->ctx = &c;
                    sch->S->dplan = std::make_unique<DistPlan>();
                    dist_selfp_schur(c, *plan0, *plan1, sch->A00->mat(), sch->A01->mat(), sch->A10->mat(), sch->A11->mat(), sch->S->M,
                                     *sch->S->dplan, d_mass.p);
                    sch->S->n_owned_cols = sch->n1;
                } else
                // single rank (or -poro_amg_distributed 0): from the local (owned) parts
                {
                    Csr a00, a01, a10, a11;
                    local_square(c, *sch->A00, a00);
                    auto owned_cols = [&](const MatOp& m, int ncols_owned, Csr& o) {
                        if (m.M.ncols == ncols_owned) { csr_copy(c, m.M, o); PORO_CUDA(cudaStreamSynchronize(c.stream)); return; }
                        std::vector<int> rmap((size_t)m.M.nrows), cmap((size_t)m.M.ncols, -1);
                        for (int i = 0; i < m.M.nrows; ++i) rmap[i] = i;
                        for (int i = 0; i < ncols_owned; ++i) cmap[i] = i;
                        DBuf<int> d_r(rmap.size()), d_c(cmap.size());
                        PORO_CUDA(cudaMemcpy(d_r.p, rmap.data(), rmap.size() * 4, cudaMemcpyHostToDevice));
                        PORO_CUDA(cudaMemcpy(d_c.p, cmap.data(), cmap.size() * 4, cudaMemcpyHostToDevice));
                        csr_extract(c, m.M, d_r.p, d_c.p, m.M.nrows, ncols_owned, o);
                    };
                    owned_cols(*sch->A01, (int)sch->n1, a01);
                    owned_cols(*sch->A10, (int)sch->n0, a10);
                    owned_cols(*sch->A11, (int)sch->n1, a11);
                    DBuf<double> dinv((size_t)sch->n0);
                    if (d_mass.p) PORO_CUDA(cudaMemcpy(dinv.p, d_mass.p, (size_t)sch->n0 * 8, cudaMemcpyDeviceToDevice));
                    else csr_diag(c, a00, dinv.p);
                    std::vector<double> hd((size_t)sch->n0);
                    PORO_CUDA(cudaMemcpy(hd.data(), dinv.p, hd.size() * 8, cudaMemcpyDeviceToHost));
                    for (auto& v : hd) v = v != 0.0 ? 1.0 / v : 1.0;
                    PORO_CUDA(cudaMemcpy(dinv.p, hd.data(), hd.size() * 8, cudaMemcpyHostToDevice));
                    csr_scale_cols(c, a10, dinv.p);                      // A10 diag(A00)^-1
                    Csr prod;
                    csr_spgemm(c, a10, a01, prod);
                    sch->S = std::make_unique<MatOp>();
                    sch->S->ctx = &c;
                    csr_add_scaled(c, a11, prod, -1.0, nullptr, sch->S->M);
                }
                const int bs0 = t0 == 1 ? bs_v : 1, bs1 = t1 == 1 ? bs_v : 1;
                const char* sub_pc = fp_exact_big ? "lu" : "amg";
                sch->k0 = make_inner(h, sch->A00.get(), "preonly", sub_pc, "fp_fieldsplit_0_", bs0, t0 == 1 ? cs : nullptr, t0 == 1 ? cdim : 0);
                // K1: operator A11 (PETSc applies the Schur operator matrix-free for Krylov K1; with preonly only the PC matters),
                // preconditioner built from the assembled selfp matrix
                sch->k1 = make_inner(h, sch->S.get(), "preonly", sub_pc, "fp_fieldsplit_1_", bs1, t1 == 1 ? cs : nullptr, t1 == 1 ? cdim : 0);
                sch->t0.alloc((size_t)sch->n0); sch->t1.alloc((size_t)sch->n1); sch->u0.alloc((size_t)sch->n0);
                if (sprec == "cc") {
                    // Chebyshev(4) on the pressure mass matrix P_pp (scale-equivariant: the factor is applied to the result)
                    sch->kv = make_inner(h, sch->A11.get(), "preonly", "chebyshev", "fp_fieldsplit_1_visc_", 1, nullptr, 0);
                    sch->tv.alloc((size_t)sch->n1);
                }
            }
            cc.schur = sch.get();
            k->owned_pc = std::move(sch);
            k->pc = k->owned_pc.get();
            if (k->type != "preonly") {
                cc.Mfp_fp = extract_block(h, *Pp, of, of + nf + np, {1, 2});
                k->A = cc.Mfp_fp.get();
            }
            cc.ksp_fp = std::move(k);
        }
    }
    if (accel_order > 0) cc.anderson.init(&c, accel_order, fl.n_owned);
    {
        // CUDA graph of the application: only when it is a fixed launch sequence (no inner Krylov loop with host-side tests)
        bool fixed = true;
        for (KSP* k : {cc.ksp_s.get(), cc.ksp_f.get(), cc.ksp_p.get(), cc.ksp_fp.get(), cc.ksp_diff.get(),
                       cc.schur ? cc.schur->k0.get() : nullptr, cc.schur ? cc.schur->k1.get() : nullptr})
            if (k && k->type != "preonly") fixed = false;
        cc.graph_enabled = fixed && c.opt_i("-poro_pc_graph", 1) != 0;
        cc.overlap_blocks = cc.graph_enabled && !cc.three_way && c.opt_i("-poro_pc_overlap_blocks", 1) != 0;
    }
    // the permuted copy of P is no longer needed
    pc->Pperm = Csr();
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    *out = pc.release();
    API_END
}

int poro_pc_apply(poro_pc* pc, const double* x, double* y) {
    API_BEGIN
    Ctx& c = pc->ctx->c;
    Fields& fl = pc->ctx->fl;
    if (fl.identity) { pc->cc.apply(x, y); return 0; }
    const int64_t n = fl.n_owned;
    if ((int64_t)pc->xp.n < n) { pc->xp.alloc(n); pc->yp.alloc(n); }
    vec_gather(c, pc->xp.p, x, fl.old_of_new.p, n);
    pc->cc.apply(pc->xp.p, pc->yp.p);
    vec_scatter(c, y, pc->yp.p, fl.old_of_new.p, n);
    API_END
}

int poro_pc_destroy(poro_pc* pc) {
    API_BEGIN
    delete pc;
    API_END
}

int poro_pc_stats(poro_pc* pc, double* out, int n) {
    API_BEGIN
    PCBlockCC& cc = pc->cc;
    std::vector<double> v = {cc.t_total, cc.t_solid, cc.t_fluid, cc.t_press, cc.t_alloc};
    auto add = [&](KSP* k) { v.push_back(k ? (double)k->total_its : 0.0); v.push_back(k ? (double)k->calls : 0.0); };
    add(cc.ksp_s.get()); add(cc.ksp_f.get()); add(cc.ksp_p.get()); add(cc.ksp_fp.get()); add(cc.ksp_diff.get());
    add(cc.schur ? cc.schur->k0.get() : nullptr);
    add(cc.schur ? cc.schur->k1.get() : nullptr);
    v.push_back((double)cc.graph_replays);
    for (int i = 0; i < n; ++i) out[i] = i < (int)v.size() ? v[i] : 0.0;
    API_END
}

static MatOp* find_block(poro_pc* pc, const std::string& nm) {
    PCBlockCC& cc = pc->cc;
    if (nm == "ss") return cc.Ms_s.get();
    if (nm == "sf") return cc.Ms_f.get();
    if (nm == "sp") return cc.Ms_p.get();
    if (nm == "ff") return cc.Mf_f.get() ? cc.Mf_f.get() : (cc.schur ? (cc.schur->p_first ? cc.schur->A11.get() : cc.schur->A00.get()) : nullptr);
    if (nm == "fp") return cc.Mf_p.get();
    if (nm == "pp") return cc.Mp_p.get() ? cc.Mp_p.get() : (cc.schur ? (cc.schur->p_first ? cc.schur->A00.get() : cc.schur->A11.get()) : nullptr);
    if (nm == "fps") return cc.Mfp_s.get();
    if (nm == "fpfp") return cc.Mfp_fp.get();
    if (nm == "schur") return cc.schur ? cc.schur->S.get() : nullptr;
    if (nm == "diff") return cc.Mp_diff.get();
    return nullptr;
}

int poro_pc_block_info(poro_pc* pc, const char* name, int64_t* nrows, int64_t* ncols, int64_t* nnz) {
    API_BEGIN
    MatOp* m = find_block(pc, name);
    if (!m) throw Error(std::string("no such block: ") + name);
    if (nrows) *nrows = m->mat().nrows;
    if (ncols) *ncols = m->mat().ncols;
    if (nnz) *nnz = m->mat().nnz;
    API_END
}

// algorithmic bytes of ONE plain product y = B x with a block in the format it is launched in (0 CSR, 1 BSR, 2 diagonal BSR,
// 4 stencil: generated block applied from its class tables)
int poro_pc_block_bytes(poro_pc* pc, const char* name, int64_t* bytes, int* format) {
    API_BEGIN
    MatOp* m = find_block(pc, name);
    if (!m) throw Error(std::string("no such block: ") + name);
    const Csr& B = m->mat();
    if (stencil_runs(B)) {
        *bytes = stencil_bytes(*B.stencil);
        *format = 4;
        return 0;
    }
    csr_ensure_bsr(pc->ctx->c, B);
    if (B.bsr_state == 1) {
        const Bsr& b = *B.bsr;
        const int64_t ne = b.diag_only ? b.bs : b.bs * b.bs;
        *bytes = ((b.fp32 ? 4 : 8) * ne + 4) * b.nnzb + 4 * ((int64_t)b.nbrows + 1) + 8 * (int64_t)B.nrows + 8 * (int64_t)B.ncols;
        *format = b.diag_only ? 2 : 1;
    } else {
        *bytes = 12 * B.nnz + 4 * ((int64_t)B.nrows + 1) + 8 * (int64_t)B.nrows + 8 * (int64_t)B.ncols;
        *format = 0;
    }
    API_END
}

int poro_pc_block_mult(poro_pc* pc, const char* name, int mode, const double* x, double* y, const double* z, double* r, double* d_new,
                       double* xv, const double* dinv, double c1, double c2, double* dot) {
    API_BEGIN
    MatOp* m = find_block(pc, name);
    if (!m) throw Error(std::string("no such block: ") + name);
    mult_in_mode(pc->ctx->c, m->mat(), m, mode, x, y, z, r, d_new, xv, dinv, c1, c2, dot);
    API_END
}

int poro_pc_block_copy(poro_pc* pc, const char* name, int64_t* rowptr, int32_t* col, double* val) {
    API_BEGIN
    MatOp* m = find_block(pc, name);
    if (!m) throw Error(std::string("no such block: ") + name);
    std::vector<int> rp, ci;
    std::vector<double> v;
    csr_to_host(m->mat(), rp, ci, v);
    for (size_t i = 0; i < rp.size(); ++i) rowptr[i] = rp[i];
    for (size_t i = 0; i < ci.size(); ++i) { col[i] = ci[i]; val[i] = v[i]; }
    API_END
}

static KSP* find_ksp(poro_pc* pc, const std::string& nm) {
    PCBlockCC& cc = pc->cc;
    if (nm == "s") return cc.ksp_s.get();
    if (nm == "f") return cc.ksp_f.get();
    if (nm == "p") return cc.ksp_p.get();
    if (nm == "fp") return cc.ksp_fp.get();
    if (nm == "diff") return cc.ksp_diff.get();
    if (nm == "fp0") return cc.schur ? cc.schur->k0.get() : nullptr;
    if (nm == "fp1") return cc.schur ? cc.schur->k1.get() : nullptr;
    return nullptr;
}

int poro_pc_inner_solve(poro_pc* pc, const char* name, const double* r, double* z) {
    API_BEGIN
    KSP* k = find_ksp(pc, name);
    if (!k) throw Error(std::string("no such inner solver: ") + name);
    k->solve(r, z);
    API_END
}

int poro_pc_inner_result(poro_pc* pc, const char* name, int* its, int* reason, double* rnorm) {
    API_BEGIN
    KSP* k = find_ksp(pc, name);
    if (!k) throw Error(std::string("no such inner solver: ") + name);
    PORO_CUDA(cudaStreamSynchronize(pc->ctx->c.stream));
    if (its) *its = k->its;
    if (reason) *reason = k->reason;
    if (rnorm) *rnorm = k->rnorm;
    API_END
}

int poro_pc_amg_info(poro_pc* pc, const char* name, int64_t* rows, int64_t* nnz, int cap, int* nlevels) {
    API_BEGIN
    KSP* k = find_ksp(pc, name);
    if (!k) throw Error(std::string("no such inner solver: ") + name);
    PCAmg* a = dynamic_cast<PCAmg*>(k->pc);
    if (!a) { *nlevels = 0; return 0; }
    *nlevels = (int)a->amg.levels.size();
    for (int l = 0; l < *nlevels && l < cap; ++l) { rows[l] = a->amg.op(l).nrows; nnz[l] = a->amg.op(l).nnz; }
    API_END
}

static Amg& amg_level_of(poro_pc* pc, const char* name, int level, const char* who) {
    KSP* k = find_ksp(pc, name ? name : "");
    if (!k) throw Error(std::string(who) + ": no such inner solver: " + (name ? name : ""));
    PCAmg* a = dynamic_cast<PCAmg*>(k->pc);
    if (!a) throw Error(std::string(who) + ": inner solver '" + name + "' has no AMG hierarchy");
    PORO_REQUIRE(!a->amg.dist, std::string(who) + ": the hierarchy of '" + name + "' is row-partitioned");
    PORO_REQUIRE(level >= 0 && level < (int)a->amg.levels.size(), std::string(who) + ": level " + std::to_string(level) + " out of range (" +
                                                                   std::to_string(a->amg.levels.size()) + " levels)");
    return a->amg;
}

int poro_pc_amg_level_info(poro_pc* pc, const char* name, int level, int64_t* out, int n, double* lmax) {
    API_BEGIN
    Amg& a = amg_level_of(pc, name, level, "poro_pc_amg_level_info");
    const AmgLevel& L = *a.levels[level];
    const bool last = level + 1 == (int)a.levels.size();
    std::vector<int64_t> v;
    auto dims = [&](const Csr& M) { v.push_back(M.nrows); v.push_back(M.ncols); v.push_back(M.nnz); };
    dims(a.op(level));
    dims(L.P);
    dims(L.R);
    dims(L.keep_T);
    v.insert(v.end(), {L.bs, L.k, L.n_agg, L.mg ? 1 : 0, last ? 1 : 0, last && a.coarse_direct ? 1 : 0, L.kept ? 1 : 0,
                       L.spgemm_chunks[0], L.spgemm_chunks[1], L.spgemm_chunks[2]});
    for (int i = 0; i < n; ++i) out[i] = i < (int)v.size() ? v[i] : 0;
    if (lmax) *lmax = L.lmax;
    API_END
}

int poro_pc_amg_level_copy(poro_pc* pc, const char* name, int level, const char* what, int64_t* rowptr, int32_t* col, double* val) {
    API_BEGIN
    Amg& a = amg_level_of(pc, name, level, "poro_pc_amg_level_copy");
    const AmgLevel& L = *a.levels[level];
    const std::string w = what ? what : "";
    const std::string at = "poro_pc_amg_level_copy('" + w + "', level " + std::to_string(level) + "): ";
    const bool last = level + 1 == (int)a.levels.size();
    auto csr_out = [&](const Csr& M) {
        std::vector<int> rp, ci;
        std::vector<double> v;
        csr_to_host(M, rp, ci, v);
        for (size_t i = 0; i < rp.size(); ++i) rowptr[i] = rp[i];
        for (size_t i = 0; i < ci.size(); ++i) { col[i] = ci[i]; val[i] = v[i]; }
    };
    auto dev_out = [&](const void* src, size_t bytes, void* dst) {
        PORO_CUDA(cudaStreamSynchronize(a.ctx->stream));
        if (bytes) PORO_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    };
    if (w == "A") { csr_out(a.op(level)); return 0; }
    if (w == "dinv") { dev_out(L.dinv.p, (size_t)a.op(level).nrows * sizeof(double), val); return 0; }
    if (w == "inv") {
        PORO_REQUIRE(last && a.coarse_direct, at + "only the coarsest level of a hierarchy solved directly has an inverse");
        dev_out(a.coarse_inv.p, a.coarse_inv.bytes(), val);
        return 0;
    }
    const bool transfer = w == "P" || w == "R" || w == "T";
    PORO_REQUIRE(transfer || w == "agg" || w == "B", at + "unknown item (A P R T agg B dinv inv)");
    PORO_REQUIRE(!(L.mg && w != "B"), at + "the level is geometric: its transfer has no matrix and it has no aggregates");
    PORO_REQUIRE(!(last && w != "B"), at + "the coarsest level has no transfer and no aggregates");
    if (w == "P" || w == "R") { csr_out(w == "P" ? L.P : L.R); return 0; }
    PORO_REQUIRE(L.kept, at + "the set-up data was not kept (set -poro_amg_keep_setup 1 before the set-up)");
    if (w == "T") csr_out(L.keep_T);
    else if (w == "agg") dev_out(L.keep_agg.p, L.keep_agg.bytes(), col);
    else dev_out(L.keep_B.p, L.keep_B.bytes(), val);
    API_END
}

int poro_mat_setup_op(poro_mat* a, poro_mat* b, const char* op, double alpha, const double* s_dev, poro_mat** out, int* chunks) {
    API_BEGIN
    Ctx& c = a->ctx->c;
    const std::string o = op ? op : "";
    PORO_REQUIRE(o == "transpose" || (b && b->ctx == a->ctx), "poro_mat_setup_op: '" + o + "' needs a second matrix of the same context");
    Csr C;
    int ch = 0;
    if (o == "spgemm") csr_spgemm(c, a->raw, b->raw, C, &ch);
    else if (o == "transpose") csr_transpose(c, a->raw, C);
    else if (o == "add_scaled") csr_add_scaled(c, a->raw, b->raw, alpha, s_dev, C);
    else throw Error("poro_mat_setup_op: unknown operation '" + o + "' (spgemm transpose add_scaled)");
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    if (chunks) *chunks = ch;
    *out = poro_mat_adopt(a->ctx, std::move(C));
    API_END
}

int poro_dense_inverse(poro_ctx* h, int n, const double* a_host, double* inv_host) {
    API_BEGIN
    Ctx& c = h->c;
    PORO_REQUIRE(n > 0, "poro_dense_inverse: n must be positive");
    DBuf<double> A((size_t)n * n), inv;
    PORO_CUDA(cudaMemcpy(A.p, a_host, A.bytes(), cudaMemcpyHostToDevice));
    dense_inverse_full(c, A.p, n, inv);
    PORO_CUDA(cudaMemcpy(inv_host, inv.p, inv.bytes(), cudaMemcpyDeviceToHost));
    API_END
}

static Amg& mg_amg(poro_pc* pc, const char* name) {
    KSP* k = find_ksp(pc, name ? name : "");
    if (!k) throw Error(std::string("no such inner solver: ") + (name ? name : ""));
    PCAmg* a = dynamic_cast<PCAmg*>(k->pc);
    if (!a || a->amg.par.mg_levels < 1) throw Error(std::string("inner solver '") + name + "' is not a geometric multigrid (pc_type mg)");
    return a->amg;
}

int poro_pc_mg_info(poro_pc* pc, const char* name, int64_t* out, int n) {
    API_BEGIN
    Amg& a = mg_amg(pc, name);
    int geo = 1;
    while (geo < (int)a.levels.size() && a.levels[geo - 1]->mg) ++geo;
    std::vector<int64_t> v = {geo};
    for (int l = 0; l < geo; ++l) {
        const Csr& A = a.op(l);
        const bool st = A.stencil && A.stencil->fr >= 0;
        v.push_back(st ? A.stencil->d->N : -1);
        v.push_back(A.nrows);
        v.push_back(stencil_runs(A) ? 4 : 0);
    }
    v.push_back((int64_t)a.levels.size() - geo);
    for (int i = 0; i < n; ++i) out[i] = i < (int)v.size() ? v[i] : 0;
    API_END
}

int poro_pc_mg_transfer(poro_pc* pc, const char* name, int level, int dir, int mode, const double* x, double* y) {
    API_BEGIN
    Amg& a = mg_amg(pc, name);
    PORO_REQUIRE(level >= 0 && level < (int)a.levels.size() && a.levels[level]->mg, "poro_pc_mg_transfer: level " + std::to_string(level) +
                                                                                        " has no geometric transfer");
    PORO_REQUIRE(dir == 0 || dir == 1, "poro_pc_mg_transfer: dir is 0 (prolongation) or 1 (restriction)");
    PORO_REQUIRE(mode == 0 || mode == 1, "poro_pc_mg_transfer: mode is 0 (set) or 1 (add)");
    PORO_REQUIRE(dir == 0 || mode == 0, "poro_pc_mg_transfer: restriction has mode 0 only");
    Ctx& c = pc->ctx->c;
    if (dir == 0) mg_prolong(c, *a.levels[level]->mg, a.ext(level + 1, x), y, mode == 1);   // row-partitioned: coarse ghosts of x
    else mg_restrict(c, *a.levels[level]->mg, x, y);
    API_END
}

int poro_pc_mg_bytes(poro_pc* pc, const char* name, int level, int64_t* out) {
    API_BEGIN
    Amg& a = mg_amg(pc, name);
    PORO_REQUIRE(level >= 0 && level < (int)a.levels.size() && a.levels[level]->mg, "poro_pc_mg_bytes: level " + std::to_string(level) +
                                                                                     " has no geometric transfer");
    const MgTransfer& t = *a.levels[level]->mg;
    out[0] = mg_prolong_bytes(t, false);
    out[1] = mg_prolong_bytes(t, true);
    out[2] = mg_restrict_bytes(t);
    API_END
}

int poro_pc_factor_info(poro_pc* pc, const char* name, int64_t* out, int n) {
    API_BEGIN
    const std::string nm = name ? name : "";
    KSP* k = (nm == "s" || nm == "f" || nm == "p" || nm == "fp" || nm == "diff") ? find_ksp(pc, nm) : nullptr;
    if (!k) throw Error("no such inner solver: " + nm);
    const PCSparseLU* f = dynamic_cast<const PCSparseLU*>(k->pc);
    if (!f) throw Error("block '" + nm + "' is not factorised by the sparse LU (its inner PC is " + k->pc->kind() +
                        "; select it with -" + nm + "_pc_factor_mat_solver_type poro above -poro_dense_lu_limit rows)");
    const int64_t v[] = {f->n, f->nnz_l, f->nnz_u, f->amalg_zeros, f->nsuper, f->nlevels, f->max_front, f->npert,
                         f->device_bytes, (int64_t)f->flops, (int64_t)std::llround(f->factor_ms * 1e3), f->apply_bytes};
    for (int i = 0; i < n; ++i) out[i] = i < (int)(sizeof v / sizeof v[0]) ? v[i] : 0;
    API_END
}

int poro_pc_ilu_info(poro_pc* pc, const char* name, double* out, int n) {
    API_BEGIN
    const std::string nm = name ? name : "";
    KSP* k = find_ksp(pc, nm);
    if (!k) throw Error("no such inner solver: " + nm);
    const PCIlu* f = dynamic_cast<const PCIlu*>(k->pc);
    if (!f) throw Error("inner solver '" + nm + "' is not an incomplete factorisation (its inner PC is " + k->pc->kind() +
                        "; select it with -<prefix>pc_type ilu or bjacobi)");
    const double v[] = {(double)f->n, (double)f->L.nnz, (double)f->U.nnz, (double)f->lptr.size() - 1, (double)f->uptr.size() - 1,
                        f->min_pivot, (double)f->device_bytes, (double)f->apply_bytes};
    for (int i = 0; i < n; ++i) out[i] = i < (int)(sizeof v / sizeof v[0]) ? v[i] : 0.0;
    API_END
}

// ---------------------------------------------------------------------------------------------
// outer solvers
// ---------------------------------------------------------------------------------------------
static std::unique_ptr<MatOp> make_outer_op(poro_ctx* h, poro_mat* A) {
    Fields& fl = h->fl;
    Ctx& c = h->c;
    PORO_REQUIRE(fl.set, "call poro_fields_set first");
    auto op = std::make_unique<MatOp>();
    op->ctx = &c;
    if (fl.identity) {
        PORO_REQUIRE(A->raw.nrows == fl.n_owned && A->raw.ncols == fl.n_ext, "A shape does not match the index sets");
        op->ref = &A->raw;          // borrowed: the poro_mat must outlive the solver (documented in poro.h)
    } else permute_matrix(h, A->raw, op->M);
    op->n_owned_cols = fl.n_owned;
    for (int t = 0; t < 3; ++t)
        if (fl.nh[t] || c.nranks > 1) op->pieces.push_back({&fl.halo[t], fl.off[t], fl.n_owned + fl.hoff[t]});
    if (!op->ref) csr_choose_lanes(op->M);
    // generated matrix on one rank: one stencil launch per row field, each summing the row field's tables (stencil.cu)
    if (op->ref && A->raw.stencil && A->raw.stencil->fr < 0 && c.nranks == 1 && stencil_layout_matches(fl, *A->raw.stencil)) {
        for (int fr = 0; fr < 3; ++fr)
            if (fl.n[fr] > 0) op->stencil_rows.push_back(std::make_shared<StencilOp>(StencilOp{A->raw.stencil->d, fr, -1}));
        return op;
    }
    // node-blocked s and f diagonal blocks (owned columns) -> BSR parts; everything else stays in one CSR remainder
    const int bd = fl.block_dim;
    if (bd > 1 && fl.n[0] % bd == 0 && fl.n[1] % bd == 0 && c.opt_i("-poro_use_bsr", 1)) {
        // ss, ff (dense node blocks -> BSR) and sf, fs (mass couplings M (x) I -> diagonal-block BSR)
        Csr rem;
        bool have_rem = false;
        for (int tr = 0; tr < 2; ++tr)
            for (int tc = 0; tc < 2; ++tc) {
                const Csr& src = have_rem ? rem : op->mat();
                auto part = std::make_unique<MatOp::DiagPart>();
                const int r0 = (int)fl.off[tr], r1 = (int)(fl.off[tr] + fl.n[tr]);
                const int c0 = (int)fl.off[tc], c1 = (int)(fl.off[tc] + fl.n[tc]);
                csr_select(c, src, r0, r1, c0, c1, true, part->B);
                if (part->B.nnz == 0) continue;
                part->B.block_hint = bd;
                part->row_off = r0;
                part->col_off = c0;
                op->parts.push_back(std::move(part));
                Csr next;
                csr_select(c, src, r0, r1, c0, c1, false, next);
                rem = std::move(next);
                have_rem = true;
            }
        if (have_rem) { op->M = std::move(rem); op->ref = nullptr; }
        // the mass couplings A_sf, A_fs = c M (x) I (lib/Assembler.py:83,88) share the node pattern of A_ss, A_ff: let each ride
        // along its diagonal block as one scalar per block (one pass, one launch per field row instead of two)
        if (c.opt_i("-poro_fuse_couplings", 1)) {
            auto find = [&](int64_t r0, int64_t c0) -> int {
                for (size_t i = 0; i < op->parts.size(); ++i) if (op->parts[i]->row_off == r0 && op->parts[i]->col_off == c0) return (int)i;
                return -1;
            };
            for (int t = 0; t < 2; ++t) {
                const int im = find(fl.off[t], fl.off[t]), ic = find(fl.off[t], fl.off[1 - t]);
                if (im < 0 || ic < 0 || fl.n[0] != fl.n[1]) continue;
                if (csr_fuse_coupling(c, op->parts[im]->B, op->parts[ic]->B)) {
                    op->parts[im]->x2_off = op->parts[ic]->col_off;
                    op->parts.erase(op->parts.begin() + ic);
                }
            }
        }
    }
    return op;
}

int poro_ksp_create(poro_ctx* h, poro_mat* A, poro_pc* pc, const char* type, double rtol, double atol, double divtol,
                    int maxit, int restart, const char* prefix, poro_ksp** out) {
    API_BEGIN
    PORO_CUDA(cudaSetDevice(h->c.device));
    auto k = std::make_unique<poro_ksp>();
    k->ctx = h;
    k->pc = pc;
    k->A = make_outer_op(h, A);
    KSP& s = k->ksp;
    s.ctx = &h->c;
    s.A = k->A.get();
    s.pc = &pc->cc;
    s.type = type ? type : "gmres";
    s.rtol = rtol; s.atol = atol; s.dtol = divtol; s.max_it = maxit;
    if (restart > 0) s.restart = restart;
    s.fields = &h->fl;
    s.set_from_options(prefix ? prefix : "global_");
    *out = k.release();
    API_END
}

int poro_ksp_solve(poro_ksp* k, const double* b, double* x, int* its, int* reason, double* rnorm) {
    API_BEGIN
    Ctx& c = k->ctx->c;
    Fields& fl = k->ctx->fl;
    PORO_CUDA(cudaSetDevice(c.device));
    const int64_t n = fl.n_owned;
    if (fl.identity) k->ksp.solve(b, x);
    else {
        if ((int64_t)k->bp.n < n) { k->bp.alloc(n); k->xp.alloc(n); }
        vec_gather(c, k->bp.p, b, fl.old_of_new.p, n);
        if (k->ksp.guess_nonzero) vec_gather(c, k->xp.p, x, fl.old_of_new.p, n);
        k->ksp.solve(k->bp.p, k->xp.p);
        vec_scatter(c, x, k->xp.p, fl.old_of_new.p, n);
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    if (its) *its = k->ksp.its;
    if (reason) *reason = k->ksp.reason;
    if (rnorm) *rnorm = k->ksp.rnorm;
    API_END
}

int poro_ksp_solve_host(poro_ksp* k, const double* b_host, double* x_host, int* its, int* reason, double* rnorm) {
    Ctx& c = k->ctx->c;
    const int64_t n = k->ctx->fl.n_owned;
    try {
        PORO_CUDA(cudaSetDevice(c.device));
        if ((int64_t)k->bdev.n < n) { k->bdev.alloc(n); k->xdev.alloc(n); }
        PORO_CUDA(cudaMemcpyAsync(k->bdev.p, b_host, n * 8, cudaMemcpyHostToDevice, c.stream));
        if (k->ksp.guess_nonzero) PORO_CUDA(cudaMemcpyAsync(k->xdev.p, x_host, n * 8, cudaMemcpyHostToDevice, c.stream));
    } catch (const std::exception& e) { g_err = e.what(); return -1; }
    int rc = poro_ksp_solve(k, k->bdev.p, k->xdev.p, its, reason, rnorm);
    if (rc) return rc;
    API_BEGIN
    PORO_CUDA(cudaMemcpyAsync(x_host, k->xdev.p, n * 8, cudaMemcpyDeviceToHost, c.stream));
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    API_END
}

int poro_ksp_residual_history(poro_ksp* k, double* out, int cap, int* n) {
    API_BEGIN
    int m = (int)k->ksp.history.size();
    if (n) *n = m;
    for (int i = 0; i < m && i < cap; ++i) out[i] = k->ksp.history[i];
    API_END
}

int poro_ksp_set_initial_guess_nonzero(poro_ksp* k, int flag) {
    API_BEGIN
    k->ksp.guess_nonzero = flag != 0;
    API_END
}

int poro_ksp_field_history(poro_ksp* k, double* out, int cap, int* n) {
    API_BEGIN
    int m = (int)k->ksp.field_history.size();
    if (n) *n = m;
    for (int i = 0; i < m && i < cap; ++i) out[i] = k->ksp.field_history[i];
    API_END
}

int poro_ksp_profile(poro_ksp* k, int enable, double* op_ms, int64_t* op_calls, int64_t* op_bytes) {
    API_BEGIN
    KSP& s = k->ksp;
    s.profile_flush();
    if (op_ms) *op_ms = s.op_ms;
    if (op_calls) *op_calls = s.op_calls;
    if (op_bytes) {
        // algorithmic bytes of the formats actually launched: CSR remainder + BSR diagonal parts, or the stencil launches
        const Csr& A = k->A->mat();
        int64_t bytes = 0;
        for (auto& s : k->A->stencil_rows) bytes += stencil_bytes(*s);
        if (k->A->stencil_rows.empty()) bytes += 12 * A.nnz + 4 * ((int64_t)A.nrows + 1) + 8 * (int64_t)A.nrows + 8 * (int64_t)A.ncols;
        for (auto& p : k->A->parts) {
            const Csr& B = p->B;
            if (B.bsr_state == 1) {
                const Bsr& b = *B.bsr;
                const int64_t ne = (b.diag_only ? b.bs : b.bs * b.bs) + (p->x2_off >= 0 ? 1 : 0);
                bytes += (8 * ne + 4) * b.nnzb + 4 * ((int64_t)b.nbrows + 1) + 16 * (int64_t)B.nrows + 8 * (int64_t)B.ncols * (p->x2_off >= 0 ? 2 : 1);
            } else bytes += 12 * B.nnz + 4 * ((int64_t)B.nrows + 1) + 16 * (int64_t)B.nrows + 8 * (int64_t)B.ncols;
        }
        *op_bytes = bytes;
    }
    if (enable >= 0) { s.profile_op = enable != 0; if (enable) { s.op_ms = 0.0; s.op_calls = 0; } }
    API_END
}

// algorithmic bytes of each launch of the outer operator: [CSR remainder, part 0, part 1, ...], or one stencil launch per
// row field (format 4) for a generated matrix; returns count in *n
int poro_ksp_parts_info(poro_ksp* k, int64_t* bytes, int* is_bsr, int cap, int* n) {
    API_BEGIN
    std::vector<int64_t> b;
    std::vector<int> f;
    if (!k->A->stencil_rows.empty()) {
        for (auto& s : k->A->stencil_rows) { b.push_back(stencil_bytes(*s)); f.push_back(4); }
        *n = (int)b.size();
        for (int i = 0; i < *n && i < cap; ++i) { bytes[i] = b[i]; is_bsr[i] = f[i]; }
        return 0;
    }
    const Csr& A = k->A->mat();
    b.push_back(12 * A.nnz + 4 * ((int64_t)A.nrows + 1) + 8 * (int64_t)A.nrows + 8 * (int64_t)A.ncols);
    f.push_back(0);
    for (auto& p : k->A->parts) {
        const Csr& B = p->B;
        if (B.bsr_state == 1) {
            const Bsr& bb = *B.bsr;
            const bool fused = p->x2_off >= 0;
            const int64_t ne = (bb.diag_only ? bb.bs : bb.bs * bb.bs) + (fused ? 1 : 0);
            b.push_back((8 * ne + 4) * bb.nnzb + 4 * ((int64_t)bb.nbrows + 1) + 16 * (int64_t)B.nrows + 8 * (int64_t)B.ncols * (fused ? 2 : 1));
            f.push_back(fused ? 3 : (bb.diag_only ? 2 : 1));
        } else {
            b.push_back(12 * B.nnz + 4 * ((int64_t)B.nrows + 1) + 16 * (int64_t)B.nrows + 8 * (int64_t)B.ncols);
            f.push_back(0);
        }
    }
    *n = (int)b.size();
    for (int i = 0; i < *n && i < cap; ++i) { bytes[i] = b[i]; is_bsr[i] = f[i]; }
    API_END
}

int poro_profile(poro_ctx* h, int enable, double* ms, int64_t* calls, int n) {
    API_BEGIN
    Ctx& c = h->c;
    prof_flush(c);
    for (int i = 0; i < n && i < Ctx::Prof::kSlots; ++i) { if (ms) ms[i] = c.prof.ms[i]; if (calls) calls[i] = c.prof.calls[i]; }
    if (enable >= 0) {
        c.prof.on = enable != 0;
        if (enable) for (int i = 0; i < Ctx::Prof::kSlots; ++i) { c.prof.ms[i] = 0; c.prof.calls[i] = 0; }
    }
    API_END
}

int poro_ksp_mult(poro_ksp* k, const double* x, double* y) {
    API_BEGIN
    k->A->apply(x, y);
    API_END
}

int poro_ksp_destroy(poro_ksp* k) {
    API_BEGIN
    delete k;
    API_END
}

int poro_aar_create(poro_ctx* h, poro_mat* A, poro_pc* pc, int order, int p, double omega, double beta, double atol,
                    double rtol, int maxit, int monitor, poro_aar** out) {
    API_BEGIN
    PORO_CUDA(cudaSetDevice(h->c.device));
    PORO_REQUIRE(order >= 0 && order <= 32, "AAR order must be in [0, 32]");
    PORO_REQUIRE(p >= 1, "AAR p must be >= 1");
    auto a = std::make_unique<poro_aar>();
    a->ctx = h;
    a->pc = pc;
    a->A = make_outer_op(h, A);
    AAR& s = a->aar;
    s.ctx = &h->c; s.A = a->A.get(); s.pc = &pc->cc;
    s.order = order; s.p = p; s.omega = omega; s.beta = beta; s.atol = atol; s.rtol = rtol; s.maxit = maxit;
    s.monitor = monitor != 0;
    *out = a.release();
    API_END
}

int poro_aar_solve(poro_aar* a, const double* b, double* x, int* its) {
    API_BEGIN
    Ctx& c = a->ctx->c;
    Fields& fl = a->ctx->fl;
    PORO_CUDA(cudaSetDevice(c.device));
    const int64_t n = fl.n_owned;
    if (fl.identity) a->aar.solve(b, x);
    else {
        if ((int64_t)a->bp.n < n) { a->bp.alloc(n); a->xp.alloc(n); }
        vec_gather(c, a->bp.p, b, fl.old_of_new.p, n);
        a->aar.solve(a->bp.p, a->xp.p);
        vec_scatter(c, x, a->xp.p, fl.old_of_new.p, n);
    }
    PORO_CUDA(cudaStreamSynchronize(c.stream));
    if (its) *its = a->aar.it;
    API_END
}

int poro_aar_residual_history(poro_aar* a, double* out, int cap, int* n) {
    API_BEGIN
    int m = (int)a->aar.history.size();
    if (n) *n = m;
    for (int i = 0; i < m && i < cap; ++i) out[i] = a->aar.history[i];
    API_END
}

int poro_aar_destroy(poro_aar* a) {
    API_BEGIN
    delete a;
    API_END
}
