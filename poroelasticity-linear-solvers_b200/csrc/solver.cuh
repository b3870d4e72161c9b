// solver.cuh -- operators, preconditioners and Krylov solvers of the solve phase.
#pragma once
#include "amg.cuh"
#include "common.cuh"
#include "dist.cuh"
#include "distamg.cuh"
#include "stencil.cuh"

namespace poro {

// ---- field layout (IndexSet semantics, lib/IndexSet.py:29-67) -------------------------------
struct Fields {
    // owned sizes, owned offsets in the permuted vector [s | f | p], halo sizes per field
    int64_t n[3] = {0, 0, 0}, off[3] = {0, 0, 0}, nh[3] = {0, 0, 0}, hoff[3] = {0, 0, 0};
    int64_t n_owned = 0, n_ext = 0;
    DBuf<int> new_of_old;   // extended raw index -> extended permuted index
    DBuf<int> old_of_new;   // owned permuted index -> owned raw index
    bool identity = false;
    bool owned_identity = false;    // the owned entries keep their raw order (identity may still permute the halo)
    int block_dim = 0;
    int coord_dim = 0;
    std::vector<double> coords_s, coords_p;   // host copies, permuted order
    HaloField halo[3];
    bool set = false;
};

struct LinOp {
    virtual ~LinOp() {}
    virtual int64_t rows() const = 0;
    // y = A x | y = z - A x | y = z + A x
    virtual void apply(const double* x, double* y, SpmvMode mode = SPMV_SET, const double* z = nullptr) = 0;
};

// CSR block whose columns index [owned part of some fields | their halos]
struct MatOp : LinOp {
    Ctx* ctx = nullptr;
    Csr M;
    const Csr* ref = nullptr;      // borrowed matrix (caller-owned) instead of M
    const Csr& mat() const { return ref ? *ref : M; }
    // halo pieces to refresh before the product: (plan, offset of the owned field slice inside x, offset in xext)
    struct Piece { HaloField* hf; int64_t x_off; int64_t ext_off; };
    std::vector<Piece> pieces;
    // alternative to `pieces`: one plan for all ghost columns (assembled Schur complements, whose halo is wider than a field's)
    std::unique_ptr<DistPlan> dplan;
    // plan handed to a distributed AMG built on this block: dplan, or one derived from the single halo piece
    std::unique_ptr<DistPlan> amg_plan;
    DistPlan* plan_for_amg();
    int64_t n_owned_cols = 0;
    // node-blocked diagonal field blocks cut out of M and applied as BSR: y[row_off..] += B x[col_off..]
    // x2_off >= 0: a mass coupling rides along B (bsr_tma.cu, FUSE): y[row_off..] += B x[col_off..] + C x[x2_off..]
    struct DiagPart { Csr B; int64_t row_off, col_off; int64_t x2_off = -1; };
    std::vector<std::unique_ptr<DiagPart>> parts;
    // outer operator of a generated matrix on one rank: one stencil launch per row field (stencil.cu) instead of M / parts
    std::vector<std::shared_ptr<StencilOp>> stencil_rows;
    DBuf<double> xext;
    int64_t rows() const override { return mat().nrows; }
    void apply(const double* x, double* y, SpmvMode mode = SPMV_SET, const double* z = nullptr) override;
    const double* extended(const double* x);   // returns pointer usable as SpMV input
};

struct PC {
    virtual ~PC() {}
    virtual void apply(const double* x, double* y) = 0;   // y = M^-1 x, x != y
    virtual const char* kind() const = 0;
};

struct PCNone : PC {
    Ctx* ctx; int64_t n;
    PCNone(Ctx* c, int64_t n_) : ctx(c), n(n_) {}
    void apply(const double* x, double* y) override { vec_copy(*ctx, y, x, n); }
    const char* kind() const override { return "none"; }
};

struct PCJacobi : PC {
    Ctx* ctx; DBuf<double> dinv;
    PCJacobi(Ctx* c, const Csr& A);
    void apply(const double* x, double* y) override { vec_pmult(*ctx, y, dinv.p, x, (int64_t)dinv.n); }
    const char* kind() const override { return "jacobi"; }
};

struct PCDense : PC {   // exact block solve: explicit inverse (stands in for MUMPS `preonly + lu` on small blocks)
    Ctx* ctx; DBuf<double> inv; int n;
    // one step of iterative refinement with the sparse block (y += inv (x - A y)): the Gauss-Jordan inverse of the
    // ill-conditioned `undrained` blocks (k_s = 1e6) alone is only good to ~1e-6 against a sparse LU
    Csr A; DBuf<double> r, d; int refine = 1;
    PCDense(Ctx* c, const Csr& A);
    void apply(const double* x, double* y) override;
    const char* kind() const override { return "lu(dense)"; }
};

// one supernode of PCSparseLU: pivot rows [first, first + k) of the permuted block, a front of m rows
struct SluNode {
    int first, k, m, child_begin, child_end;
    int64_t rows, upd, front, fac;   // offsets: row list, update rows (relmap / update vectors), set-up front, stored factor
};

// exact block solve by a multifrontal sparse LU (sparse_lu.cu, symbolic analysis in lu_symbolic.h): selected for `lu` /
// `cholesky` blocks above -poro_dense_lu_limit rows by -<prefix>pc_factor_mat_solver_type poro (use_sparse_lu)
struct PCSparseLU : PC {
    Ctx* ctx; int n;
    DBuf<SluNode> sn;
    DBuf<int> relmap, child, row_idx, level_sn, perm;
    std::vector<int> level_ptr;
    int nlevels = 0;
    size_t smem = 0;                 // dynamic shared memory of the solve kernels: the largest front
    DBuf<double> fac, xw, wbuf;      // factors; permuted work vector; per-supernode update vectors
    // perturbed pivots: one step of iterative refinement with the block (y += LU^-1 (x - B y)), like PCDense
    Csr A; DBuf<double> r, d;
    // factor_info
    int64_t nnz_l = 0, nnz_u = 0, amalg_zeros = 0, npert = 0, device_bytes = 0, apply_bytes = 0;
    int nsuper = 0, max_front = 0;
    double flops = 0.0, factor_ms = 0.0;
    PCSparseLU(Ctx* c, const Csr& A, const std::string& prefix);
    void apply(const double* x, double* y) override;
    const char* kind() const override { return "lu(sparse)"; }
  private:
    void solve(const double* b, double* x);
};
// the block of `prefix` (pc type `pc_type`, `rows` rows) is factorised by PCSparseLU
bool use_sparse_lu(const Ctx& c, const std::string& pc_type, const std::string& prefix, int64_t rows);

struct PCAmg : PC {
    Amg amg;
    void apply(const double* x, double* y) override { amg.apply(x, y); }
    const char* kind() const override { return "amg"; }
};

struct KSP {
    Ctx* ctx = nullptr;
    LinOp* A = nullptr;
    PC* pc = nullptr;
    std::unique_ptr<PC> owned_pc;
    std::unique_ptr<LinOp> owned_op;
    std::string type = "gmres", prefix;
    double rtol = 1e-5, atol = 1e-50, dtol = 1e5;
    int max_it = 10000, restart = 30;
    bool right = false, unprec_norm = false, natural_norm = false, cgs2 = false;
    bool monitor = false;
    bool verify_true = false;           // -<prefix>ksp_gmres_verify_true_residual: confirm convergence with b - A x, restart if needed
    bool fused_gs = false;              // one-pass projection + normalisation with the Pythagorean norm: unsafe, see solve_gmres
    bool converged_reason = false;      // -<prefix>ksp_converged_reason
    bool guess_nonzero = false;         // KSPSetInitialGuessNonzero / -<prefix>ksp_initial_guess_nonzero (warm start over time steps)
    // per-field infinity-norm residual monitor / convergence test: the `converged` callback of lib/Solver.py:8-51
    // (dead code in the reference).  Needs the field layout; builds the true residual every iteration (GMRES only).
    const Fields* fields = nullptr;
    bool monitor_fields = false, test_fields = false;
    double b0_fields[3] = {0, 0, 0};
    std::vector<double> field_history;  // per iteration: abs_s, abs_f, abs_p
    // results
    int its = 0, reason = 0;
    double rnorm = 0.0;
    std::vector<double> history;
    int64_t total_its = 0, calls = 0;
    // work
    DBuf<double> V, Z, w1, w2, w3, xtmp;
    int v_cols = 0;
    // optional live profile of the operator product (CUDA events on the launching stream)
    bool profile_op = false;
    std::vector<cudaEvent_t> ev;
    size_t ev_used = 0;
    double op_ms = 0.0;
    int64_t op_calls = 0;
    void op_apply(const double* x, double* y, SpmvMode mode = SPMV_SET, const double* z = nullptr);
    void profile_flush();
    ~KSP();

    void set_from_options(const std::string& prefix);
    void solve(const double* b, double* x);     // zero initial guess
  private:
    void solve_gmres(const double* b, double* x, bool flexible);
    void solve_cg(const double* b, double* x);
    int converged(double rn, int it, double& rnorm0, double& ttol) const;
    int fields_test(const double* b, const double* xcur, int it);
};

// PCFIELDSPLIT on the fp block: schur (lib/Preconditioner.py:102-118, petsc-options-inexact:78-80), or PETSc's additive /
// multiplicative with K1 built on A11 (no S): additive y0 = K0 x0, y1 = K1 x1; multiplicative y1 = K1 (x1 - A10 y0)
enum FieldsplitType { FS_SCHUR = 0, FS_ADDITIVE = 1, FS_MULTIPLICATIVE = 2 };
struct PCSchur : PC {
    Ctx* ctx = nullptr;
    bool p_first = true;            // reference order: split 0 = pressure, split 1 = fluid velocity
    int type = FS_SCHUR;
    int fact = 0;                   // 0 lower, 1 upper, 2 full, 3 diag (schur only)
    int64_t n0 = 0, n1 = 0, off0 = 0, off1 = 0;   // offsets inside the fp vector [f | p]
    std::unique_ptr<MatOp> A00, A01, A10, A11, S;
    std::unique_ptr<KSP> k0, k1;
    // `cc` (additive Cahouet-Chabard form, the pressure treatment of the reference's 3-way variants, lib/Assembler.py:131-137,
    // inside the 2-way fieldsplit): y1 = K1(S_mass) r + (1 / visc_scale) Chebyshev(A11) r, S_visc = visc_scale * A11
    std::unique_ptr<KSP> kv;
    double visc_scale = 0.0;
    DBuf<double> t0, t1, u0, tv;
    void solve1(const double* r, double* y1);
    void apply(const double* x, double* y) override;
    const char* kind() const override { return "fieldsplit"; }
};

struct Anderson {   // lib/AndersonAcceleration.py:19-78
    Ctx* ctx = nullptr;
    int order = 0;
    int64_t n = 0;
    int64_t k = 0;
    DBuf<double> xk, fk, dxk, dfk, F, X;
    int nF = 0, nX = 0, headF = 0, headX = 0;
    void init(Ctx* c, int order_, int64_t n_);
    void get_next_vector(double* gk);
};

// least-squares coefficients alpha = argmin || f + F alpha || through the Gram matrix
void gram_alpha(Ctx& c, const double* F, int64_t ld, int order, int nF, int headF, const double* f, int64_t n,
                std::vector<double>& alpha);

// PreconditionerCC (lib/Preconditioner.py:8-260)
struct PCBlockCC : PC {
    Ctx* ctx = nullptr;
    Fields* fl = nullptr;
    bool three_way = false;
    double w1 = 1.0, w2 = 0.1;
    std::unique_ptr<MatOp> Ms_s, Ms_f, Ms_p, Mf_f, Mf_p, Mp_p, Mfp_s, Mfp_fp, Mp_diff;
    std::unique_ptr<KSP> ksp_s, ksp_f, ksp_p, ksp_fp, ksp_diff;
    PCSchur* schur = nullptr;       // when ksp_fp's PC is a fieldsplit
    DBuf<int> bcs_sub_pressure;
    DBuf<double> t_s, t_f, t_p, y_sd, y_fd, y_pd, t_fp;
    Anderson anderson;
    // timings (seconds) like lib/Preconditioner.py:35-39; measured only when `poro_pc_timing` is set
    double t_total = 0, t_solid = 0, t_fluid = 0, t_press = 0, t_alloc = 0;
    bool timing = false;
    // One application is a fixed sequence of kernels (and halo exchanges) whenever every inner solver is `preonly`: it is
    // captured once into a CUDA graph and replayed, which removes the launch latency of the ~60 small kernels of the coarse
    // AMG levels (the reference pays the same sequence as PETSc/hypre calls on the host, lib/Preconditioner.py:141-250).
    bool graph_enabled = false;
    int eager_calls = 0;
    cudaGraphExec_t gexec = nullptr;
    DBuf<double> g_in, g_out;
    int64_t g_launches = 0;
    int64_t graph_replays = 0;      // applications that ran as the captured graph (poro_pc_stats)
    std::vector<KSP*> g_ksps;
    // 2-way `diagonal` splitting: P_fp,s is structurally empty, so the solid solve and the fluid-pressure solve are independent.
    // Inside the captured graph they are forked onto two streams (two parallel branches of the graph): the latency-bound
    // coarse levels of one hierarchy run under the bandwidth-bound level-0 launches of the other.  Single rank only: the
    // distributed coarse solves share one peer-store all-reduce channel whose use must stay ordered across ranks.
    bool overlap_blocks = false;
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    void apply(const double* x, double* y) override;
    void apply_impl(const double* x, double* y);
    ~PCBlockCC() override {
        if (gexec) cudaGraphExecDestroy(gexec);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (side_stream) cudaStreamDestroy(side_stream);
    }
    const char* kind() const override { return "blockcc"; }
};

struct AAR {   // lib/AAR.py:7-137
    Ctx* ctx = nullptr;
    LinOp* A = nullptr;
    PC* pc = nullptr;
    int order = 10, p = 5, maxit = 1000;
    double omega = 1, beta = 1, atol = 1e-12, rtol = 1e-8;
    bool monitor = false;
    int64_t n = 0;
    DBuf<double> xk, fk, dfk, dxk, tmp, F, X;
    int nF = 0, nX = 0, headF = 0, headX = 0;
    int it = 0;
    std::vector<double> history;
    std::string types;
    void solve(const double* b, double* x);
};

// builds a PC of the requested PETSc-style type for a block
std::unique_ptr<PC> make_pc(Ctx& c, const std::string& pc_type, const Csr& A, int bs, const double* coords_host,
                            int coord_dim, const std::string& prefix, DistPlan* plan = nullptr);

}  // namespace poro
