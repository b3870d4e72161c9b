// common.cuh -- context, device buffers, error handling shared by all translation units.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace poro {

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define PORO_CUDA(expr)                                                                          \
    do {                                                                                         \
        cudaError_t e__ = (expr);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            char buf__[512];                                                                     \
            snprintf(buf__, sizeof buf__, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e__),   \
                     __FILE__, __LINE__, cudaGetErrorString(e__));                               \
            throw poro::Error(buf__);                                                            \
        }                                                                                        \
    } while (0)

#define PORO_REQUIRE(cond, msg)                                                                  \
    do {                                                                                         \
        if (!(cond)) throw poro::Error(std::string(msg) + " [" #cond "]");                       \
    } while (0)

// ---- device buffer ---------------------------------------------------------------------
template <class T>
struct DBuf {
    T* p = nullptr;
    size_t n = 0;
    DBuf() = default;
    explicit DBuf(size_t n_) { alloc(n_); }
    DBuf(const DBuf&) = delete;
    DBuf& operator=(const DBuf&) = delete;
    DBuf(DBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DBuf& operator=(DBuf&& o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
        return *this;
    }
    ~DBuf() { release(); }
    void alloc(size_t n_) {
        release();
        n = n_;
        if (n) PORO_CUDA(cudaMalloc(&p, n * sizeof(T)));
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    void zero(cudaStream_t s) { if (n) PORO_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
    size_t bytes() const { return n * sizeof(T); }
};

// ---- NCCL through dlopen (no link-time dependency; single-GPU runs never touch it) -------
struct NcclApi;

// ---- peer-to-peer halo slots (dist.cu: p2p_*) --------------------------------------------------------------------
// Neighbour exchanges over NVLink without NCCL: a pack kernel STORES the boundary values straight into the neighbour's
// receive region (CUDA-IPC mapped peer memory) and releases a sequence flag there; the receiver's kernel spins on its own
// flags and copies the region behind its owned entries.  Regions are double-buffered by sequence parity; the sequence
// numbers live in device memory so that the exchanges can be captured in CUDA graphs.
struct P2PNeighDev {
    double* peer_data[2];        // where this rank writes (neighbour's arena), per parity
    uint32_t* peer_flag;         // neighbour's flag for messages from this rank
    const double* my_data[2];    // where the neighbour writes (this rank's arena)
    const uint32_t* my_flag;
    int send_begin, send_end, recv_begin, recv_end;
};
struct P2PArgs {
    P2PNeighDev nb[8];
    int nn;
};
struct P2PSlots {
    bool ready = false;
    P2PArgs args{};
    int nsend = 0, nrecv = 0;
    uint32_t* d_state = nullptr;  // [push_seq, wait_seq, push_ticket, wait_ticket] in device memory
};

// ---- halo plan (per field after permutation) -----------------------------------------------
struct HaloField {
    // for neighbour k: send owned entries send_idx[send_ptr[k]..send_ptr[k+1]) (field-local index),
    // receive recv_ptr[k+1]-recv_ptr[k] values into halo[recv_ptr[k]..)
    std::vector<int64_t> send_ptr, recv_ptr;
    DBuf<int> send_idx;
    DBuf<double> send_buf;
    int64_t n_halo = 0;
    P2PSlots p2p;
};

// ---- halo plan of one distributed matrix / AMG level (oracle/distamg_rank.py: Plan) -----------------------------
// Rows are numbered rank-contiguously per level (`offsets`), local columns are [owned | ghost]; ghosts are ordered
// neighbour-major and, inside one neighbour, in the order the owner sends them.
struct DistPlan {
    int64_t offset = 0;                   // global id of the first owned row
    int n_owned = 0, n_ghost = 0;
    std::vector<int64_t> offsets;         // nranks + 1
    DBuf<int> ghost_gid;                  // global ids of the ghost columns (n_ghost)
    std::vector<int> neigh;               // ranks we exchange with
    std::vector<int64_t> send_ptr, recv_ptr;   // per neighbour, neigh.size() + 1 entries
    DBuf<int> send_idx;                   // owned local indices to send, neighbour-major
    DBuf<double> send_buf;                // packing scratch of the vector exchanges
    P2PSlots p2p;                         // NVLink peer-store path of the width-1 exchanges (when available)
};

struct Ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    int rank = 0, nranks = 1;
    bool local_only = false;     // reductions stay on this rank (rank-local set-up such as the AMG power iteration)
    void* comm = nullptr;
    NcclApi* nccl = nullptr;
    struct P2PState* p2p = nullptr;   // receive arena + mapped peer arenas (dist.cu)
    bool p2p_fused = true;            // one kernel per exchange (push + wait + copy) instead of two
    std::map<std::string, std::string> opts;
    double* h_pin = nullptr;     // pinned host scratch for scalar read-back
    double* d_scal = nullptr;    // device scratch for reductions
    static constexpr int kScal = 1 << 18;   // partials; +8192 doubles of small slots behind it
    int64_t launches = 0;
    std::vector<void*>* capture_log = nullptr;   // while a CUDA graph is being captured: the preonly KSPs that were applied
    cudaEvent_t t0 = nullptr, t1 = nullptr;   // poro_timer_start / poro_timer_stop
    // phase profile: CUDA events on the launching stream, resolved lazily (no sync on the hot path)
    struct Prof {
        enum { kSlots = 40 };
        bool on = false;
        std::vector<cudaEvent_t> ev;
        std::vector<int> slot;
        size_t used = 0;
        double ms[kSlots] = {0};
        int64_t calls[kSlots] = {0};
    } prof;
    // distributed layout
    std::vector<int> neigh;
    int64_t n_owned_raw = -1;
    std::vector<int64_t> raw_send_ptr, raw_recv_count;
    std::vector<int32_t> raw_send_idx;

    // keys are stored with their leading '-' (poro_options_set); look-ups accept both spellings
    std::map<std::string, std::string>::const_iterator find_opt(const std::string& k) const {
        return (!k.empty() && k[0] == '-') ? opts.find(k) : opts.find("-" + k);
    }
    bool has_opt(const std::string& k) const { return find_opt(k) != opts.end(); }
    std::string opt(const std::string& k, const std::string& def) const {
        auto it = find_opt(k);
        return it == opts.end() ? def : it->second;
    }
    double opt_d(const std::string& k, double def) const {
        auto it = find_opt(k);
        return it == opts.end() ? def : atof(it->second.c_str());
    }
    int opt_i(const std::string& k, int def) const {
        auto it = find_opt(k);
        return it == opts.end() ? def : atoi(it->second.c_str());
    }
};

// slots: 0 outer operator, 1 preconditioner apply, 2 solid solve, 3 fp split 0, 4 fp split 1, 5 orthogonalisation,
//        6 fp coupling product, 8+l / 16+l / 24+l: AMG level l (inclusive) of the s / f / p hierarchy
struct ProfScope {
    Ctx& c; int idx = -1;
    ProfScope(Ctx& c_, int slot) : c(c_) {
        if (!c.prof.on || slot < 0 || slot >= Ctx::Prof::kSlots) return;
        auto& p = c.prof;
        if (p.used + 2 > p.ev.size()) for (int i = 0; i < 64; ++i) { cudaEvent_t e; cudaEventCreate(&e); p.ev.push_back(e); p.slot.push_back(0); }
        idx = (int)p.used;
        p.slot[idx] = slot;
        cudaEventRecord(p.ev[idx], c.stream);
        p.used += 2;
    }
    ~ProfScope() { if (idx >= 0) cudaEventRecord(c.prof.ev[idx + 1], c.stream); }
};
inline void prof_flush(Ctx& c) {
    auto& p = c.prof;
    if (!p.used) return;
    cudaStreamSynchronize(c.stream);
    for (size_t i = 0; i + 1 < p.used; i += 2) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.ev[i], p.ev[i + 1]) == cudaSuccess) { p.ms[p.slot[i]] += ms; p.calls[p.slot[i]]++; }
    }
    p.used = 0;
}

inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// grid for streaming kernels: a few CTAs per SM, never more than needed
inline int stream_grid(const Ctx& c, int64_t n, int block, int per_thread = 4, int ctas_per_sm = 8) {
    int64_t need = (n + (int64_t)block * per_thread - 1) / ((int64_t)block * per_thread);
    int64_t cap = (int64_t)c.sm_count * ctas_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

#define PORO_LAUNCH_CHECK(ctx) do { (ctx).launches++; PORO_CUDA(cudaGetLastError()); } while (0)

// ---- block-CSR companion of a Csr (bsr.cu): BS x BS blocks, values interleaved per 32 blocks ----------
struct Bsr {
    int bs = 0, nbrows = 0, nbcols = 0;
    int64_t nnzb = 0;
    int ntb = 1;                // blocks per thread of the stream kernel (chunk capacity = 256 * ntb)
    bool diag_only = false;     // blocks are diagonal (e.g. M (x) I couplings): BS values per block instead of BS^2
    DBuf<int> rowptr, col;
    DBuf<double> val;
    DBuf<float> val32;          // optional fp32 STORAGE of the values (arithmetic stays fp64), `-poro_pc_fp32_matrices`
    bool fp32 = false;
    DBuf<int> blk_row, blk_desc;    // chunk boundaries; per chunk {first block row, block rows, first block, blocks}
    int nblk = 0;
    bool pref = false;          // every chunk has <= 256 scalar rows: epilogue operands are prefetched (k_bsr_stream PREF)
    bool coop = false;          // cooperative (lane-contiguous) gathers of x, see k_bsr_stream COOP
    int pf_groups = 0;          // L2 prefetch distance of the stream kernel in groups of 32 blocks (0 = off), see bsr.cu
    int pf_rows = 0;            // the same distance in scalar rows (epilogue operands)
    bool fused = false;         // a mass coupling rides along (plain layout): one scalar per block + row mask in the column word
    DBuf<double> f_m;
    DBuf<int> f_col;
    // chunked layout of the TMA kernel (bsr_tma.cu); when present the plain val / col arrays above are released
    bool t_ok = false, t_fused = false;
    int t_nchunk = 0, t_cfg = 0;
    int64_t t_blocks_padded = 0;
    DBuf<int> t_desc, t_rp, t_col, t_colf;   // chunk descriptors (4 ints each), local row pointers, block columns (+ row mask)
    DBuf<double> t_val, t_m;                 // values (32-interleaved per chunk); one coupling scalar per block (fused)
};

struct StencilOp;   // stencil.cuh

// ---- sparse matrix (device CSR, local rows) ---------------------------------------------------
struct Csr {
    int nrows = 0, ncols = 0;
    int64_t nnz = 0;
    DBuf<int> rowptr;      // nrows+1 (nnz < 2^31 per local matrix, checked at creation)
    DBuf<int> col;
    DBuf<double> val;
    int lanes = 0;         // lanes per row of the fallback vector-CSR SpMV
    // row blocks of the CSR-stream SpMV, built lazily at the first product (-1 = not built, 0 = unusable)
    mutable int nblk = -1;
    mutable DBuf<int> blk_row;
    // node-block size hint (dofs per mesh node); > 1 makes the first product try a BSR conversion
    int block_hint = 0;
    mutable bool fp32_hint = false;             // store the BSR values in fp32 (preconditioner matrices only, opt-in)
    mutable int bsr_state = -1;                 // -1 not tried, 0 rejected (fill-in / shape), 1 in use
    mutable std::shared_ptr<Bsr> bsr;
    // generated structured-mesh matrix (stencil.cuh): products run from the class tables instead of the CSR (single rank)
    std::shared_ptr<StencilOp> stencil;
    double avg_row() const { return nrows ? (double)nnz / nrows : 0.0; }
};

// ---- vec.cu ---------------------------------------------------------------------------------
void vec_copy(Ctx& c, double* y, const double* x, int64_t n);
void vec_set(Ctx& c, double* y, double a, int64_t n);
void vec_scale(Ctx& c, double* y, double a, int64_t n);
void vec_abs_scale(Ctx& c, double* y, double a, int64_t n);                           // y = a |y|
void vec_axpy(Ctx& c, double* y, double a, const double* x, int64_t n);             // y += a x
void vec_aypx(Ctx& c, double* y, double a, const double* x, int64_t n);             // y = x + a y
void vec_axpby(Ctx& c, double* y, double a, const double* x, double b, int64_t n);  // y = a x + b y
void vec_waxpby(Ctx& c, double* w, double a, const double* x, double b, const double* y, int64_t n);
void vec_pmult(Ctx& c, double* w, const double* d, const double* x, int64_t n);     // w = d .* x
void vec_gather(Ctx& c, double* y, const double* x, const int* idx, int64_t n);     // y[i] = x[idx[i]]
void vec_scatter(Ctx& c, double* y, const double* x, const int* idx, int64_t n);    // y[idx[i]] = x[i]
void vec_set_idx(Ctx& c, double* y, const int* idx, double a, int64_t n);           // y[idx[i]] = a
// reductions: results land in device memory `d_out` (k doubles), local to this rank
void vec_dots(Ctx& c, int k, const double* const* xs, const double* const* ys, int64_t n, double* d_out);
// h[j] = V_j . w for j < ncol (V column-major with leading dimension ld), optional extra ww = w.w at h[ncol]
void vec_mdot(Ctx& c, const double* V, int64_t ld, int ncol, const double* w, int64_t n, double* d_h, bool with_ww);
// w -= V h (h device, ncol entries); d_nrm2 (device, 1 double) receives ||w_new||^2 (local)
void vec_maxpy_norm(Ctx& c, double* w, const double* V, int64_t ld, int ncol, const double* d_h, int64_t n, double* d_nrm2);
// w = scale * (w - V h): projection and normalisation in one pass (h device, ncol entries)
void vec_maxpy_scale(Ctx& c, double* w, const double* V, int64_t ld, int ncol, const double* d_h, int64_t n, double scale);
// y += V h with host coefficients (solution update)
void vec_maxpy_host(Ctx& c, double* y, const double* V, int64_t ld, int ncol, const double* h_host, int64_t n);
// sum over ranks in place (no-op on one rank), then copy to host and synchronise
void allreduce_sum(Ctx& c, double* d_vals, int k);
void allreduce_max(Ctx& c, double* d_vals, int k);
// out[j] = max_i |x_j[i]| over nseg segments (lengths len[j]) of one vector; local to this rank
void vec_amax_segments(Ctx& c, const double* x, const int64_t* off, const int64_t* len, int nseg, double* d_out);
void fetch(Ctx& c, const double* d_vals, int k, double* host);
double dot_host(Ctx& c, const double* x, const double* y, int64_t n);   // allreduced, synchronous
double norm2_host(Ctx& c, const double* x, int64_t n);

// ---- spmv.cu --------------------------------------------------------------------------------
enum SpmvMode { SPMV_SET = 0, SPMV_SUB = 1, SPMV_ADD = 2 };   // y = Ax | y = z - Ax | y = z + Ax
void csr_choose_lanes(Csr& A);
void spmv(Ctx& c, const Csr& A, const double* x, double* y, SpmvMode mode = SPMV_SET, const double* z = nullptr);
// converts a node-blocked matrix to BSR now (normally done lazily at the first product); true when BSR is in use
bool csr_ensure_bsr(Ctx& c, const Csr& A);
// tries to let the diagonal-block coupling C ride along the BSR form of A (same block rows / columns); on success
// spmv_fused(A, x, x2, ...) computes A x + C x2 in one pass over A's blocks
bool csr_fuse_coupling(Ctx& c, const Csr& A, const Csr& C);
void spmv_fused(Ctx& c, const Csr& A, const double* x, const double* x2, double* y, SpmvMode mode = SPMV_SET, const double* z = nullptr);
// what the next product with A launches, after the conversion it would do (fields: include/poro.h, poro_mat_kernel_info)
constexpr int kSpmvInfoFields = 11;
void spmv_kernel_info(Ctx& c, const Csr& A, int64_t* v);
// fused Chebyshev step: t = A d_old; r -= t; d_new = c1 d_old + c2 dinv.*r; x += d_new
void spmv_cheb_step(Ctx& c, const Csr& A, const double* x_in, const double* d_old, double* d_new, double* r, double* x,
                    const double* dinv, double c1, double c2);
// w = A p and *d_dot += p . w (local partial; d_dot must be zeroed by caller)
void spmv_dot(Ctx& c, const Csr& A, const double* p, double* w, double* d_dot);

// ---- setup.cu (device sparse set-up primitives) ----------------------------------------------------
enum CombineOp { COMBINE_SUM = 0, COMBINE_MAX = 1 };
// unsorted (key = row<<32 | col, val) with duplicates -> CSR with sorted unique columns. keys/vals are consumed.
void coo_to_csr(Ctx& c, int nrows, int ncols, int64_t nent, DBuf<uint64_t>& keys, DBuf<double>& vals, Csr& out,
                CombineOp op = COMBINE_SUM);
void csr_spgemm(Ctx& c, const Csr& A, const Csr& B, Csr& C, int* chunks = nullptr);   // C = A B; *chunks: row chunks used
void csr_transpose(Ctx& c, const Csr& A, Csr& At);
// C = A[rows, cols] with maps old index -> new index (or -1 to drop); new sizes given
void csr_extract(Ctx& c, const Csr& A, const int* row_map, const int* col_map, int new_rows, int new_cols, Csr& C);
void csr_diag(Ctx& c, const Csr& A, double* d);                          // missing diagonal -> 0
void csr_copy(Ctx& c, const Csr& A, Csr& B);
void csr_select(Ctx& c, const Csr& A, int r0, int r1, int c0, int c1, bool inside, Csr& C);
// C = A + alpha * diag(s) * B  (s may be null)
void csr_add_scaled(Ctx& c, const Csr& A, const Csr& B, double alpha, const double* s, Csr& C);
void csr_scale_cols(Ctx& c, Csr& A, const double* s);                    // A = A diag(s)
void csr_to_host(const Csr& A, std::vector<int>& rp, std::vector<int>& ci, std::vector<double>& v);
void csr_from_host(Ctx& c, int nrows, int ncols, const int64_t* rp, const int* ci, const double* v, Csr& out);
// dense n x n inverse of a CSR matrix by Gauss-Jordan with partial pivoting (row-major result)
void dense_inverse(Ctx& c, const Csr& A, DBuf<double>& inv);
void dense_inverse_full(Ctx& c, const double* A_dense, int n, DBuf<double>& inv);
void dense_gemv(Ctx& c, const double* M, int n, const double* x, double* y);
void dense_gemv_rect(Ctx& c, const double* M, int nrows, int ncols, const double* x, double* y);   // M row-major nrows x ncols

}  // namespace poro
