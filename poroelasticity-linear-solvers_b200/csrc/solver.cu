// solver.cu -- Krylov solvers and preconditioner compositions, all device-resident.
//
//   KSP::solve_gmres   KSPSolve_GMRES/FGMRES behind Solver.solve (lib/Solver.py:92-102,148-152):
//                      zero guess, left/right PC, classical Gram-Schmidt (one fused multi-dot pass
//                      + one fused multi-axpy+norm pass over the basis; optional second pass =
//                      CGS2), Givens recurrence on the host from (j+2) scalars per step.
//   KSP::solve_cg      KSPSolve_CG for the inner s_/f_/p_/fp_fieldsplit_0_ solves
//                      (petsc-options-inexact:12-15,28-31,44-47,82-87).
//   PCSchur            PCFIELDSPLIT schur (lib/Preconditioner.py:102-118).
//   PCBlockCC::apply   PreconditionerCC.apply, 2-way and 3-way (lib/Preconditioner.py:141-250).
//   AAR::solve         AAR.solve (lib/AAR.py:46-128) including its quirks.
//   Anderson           AndersonAcceleration.get_next_vector (lib/AndersonAcceleration.py:19-78).
#include "solver.cuh"
#include <algorithm>
#include <chrono>
#include <cmath>

namespace poro {

// =============================================================================================
// operators
// =============================================================================================
DistPlan* MatOp::plan_for_amg() {
    Ctx& c = *ctx;
    if (c.nranks <= 1) return nullptr;
    if (dplan) return dplan.get();
    if (amg_plan) return amg_plan.get();
    if (pieces.size() != 1 || pieces[0].x_off != 0 || pieces[0].ext_off != mat().nrows) return nullptr;   // single-field square blocks only
    amg_plan = std::make_unique<DistPlan>();
    dist_plan_from_halo(c, *pieces[0].hf, mat().nrows, *amg_plan);
    return amg_plan.get();
}

const double* MatOp::extended(const double* x) {
    Ctx& c = *ctx;
    if (c.nranks > 1 && dplan) {
        const int64_t next = mat().ncols;
        if ((int64_t)xext.n < next) xext.alloc((size_t)next);
        vec_copy(c, xext.p, x, dplan->n_owned);
        dist_halo_vec(c, *dplan, xext.p, 1, xext.p + dplan->n_owned);
        return xext.p;
    }
    if (c.nranks <= 1 || pieces.empty()) return x;
    int64_t next = mat().ncols;
    if ((int64_t)xext.n < next) xext.alloc((size_t)next);
    vec_copy(c, xext.p, x, n_owned_cols);
    for (auto& p : pieces)
        dist_halo_exchange(c, *p.hf, x + p.x_off, xext.p + p.ext_off);    // collective: also with no ghosts of our own
    return xext.p;
}

void MatOp::apply(const double* x, double* y, SpmvMode mode, const double* z) {
    const Csr& A = mat();
    // the halo exchange is collective: every rank runs it, also one whose local block is empty
    const double* xe = extended(x);
    if (!stencil_rows.empty()) {
        int ip = 0;
        for (auto& s : stencil_rows) {
            ProfScope ps(*ctx, 33 + ip++);
            const int64_t o = s->d->row0[s->fr];
            stencil_spmv(*ctx, *s, xe, y + o, mode, z ? z + o : nullptr);
        }
        return;
    }
    const bool prof = !parts.empty();
    if (A.nnz == 0) {                               // structurally empty block (or everything lives in `parts`)
        if (mode == SPMV_SET) vec_set(*ctx, y, 0.0, A.nrows);
        else if (y != z) vec_copy(*ctx, y, z, A.nrows);
    } else { ProfScope ps(*ctx, prof ? 32 : -1); spmv(*ctx, A, xe, y, mode, z); }
    int ip = 0;
    for (auto& p : parts) {
        double* yp = y + p->row_off;
        ProfScope ps(*ctx, 33 + ip++);
        if (p->x2_off >= 0) spmv_fused(*ctx, p->B, xe + p->col_off, xe + p->x2_off, yp, mode == SPMV_SET ? SPMV_ADD : mode, yp);
        else spmv(*ctx, p->B, xe + p->col_off, yp, mode == SPMV_SET ? SPMV_ADD : mode, yp);
    }
}

__global__ void __launch_bounds__(256) k_invert_diag(double* __restrict__ d, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n) d[i] = d[i] != 0.0 ? 1.0 / d[i] : 1.0;
}

PCJacobi::PCJacobi(Ctx* c, const Csr& A) : ctx(c) {
    dinv.alloc((size_t)A.nrows);
    csr_diag(*c, A, dinv.p);
    if (A.nrows) k_invert_diag<<<ceil_div(A.nrows, 256), 256, 0, c->stream>>>(dinv.p, A.nrows);
    PORO_LAUNCH_CHECK(*c);
}

PCDense::PCDense(Ctx* c, const Csr& A_) : ctx(c), n(A_.nrows) {
    dense_inverse(*c, A_, inv);
    refine = c->opt_i("-poro_dense_refine", 1);
    if (refine > 0) {
        csr_copy(*c, A_, A);
        csr_choose_lanes(A);
        r.alloc((size_t)n);
        d.alloc((size_t)n);
        PORO_CUDA(cudaStreamSynchronize(c->stream));
    }
}

void PCDense::apply(const double* x, double* y) {
    dense_gemv(*ctx, inv.p, n, x, y);
    for (int it = 0; it < refine; ++it) {
        spmv(*ctx, A, y, r.p, SPMV_SUB, x);          // r = x - A y
        dense_gemv(*ctx, inv.p, n, r.p, d.p);
        vec_axpy(*ctx, y, 1.0, d.p, n);
    }
}

// rigid-body modes from dof coordinates (host), node-blocked dofs; mirrors oracle/amg.py
static void rigid_body_modes(const double* coords, int64_t ndof, int dim, std::vector<double>& B, int& k) {
    int64_t nn = ndof / dim;
    k = dim == 2 ? 3 : 6;
    B.assign((size_t)ndof * k, 0.0);
    std::vector<double> mean(dim, 0.0);
    for (int64_t a = 0; a < nn; ++a) for (int d = 0; d < dim; ++d) mean[d] += coords[(a * dim) * dim + d];
    for (int d = 0; d < dim; ++d) mean[d] /= (double)nn;
    double s = 0.0;
    for (int64_t a = 0; a < nn; ++a) for (int d = 0; d < dim; ++d) s = std::max(s, std::fabs(coords[(a * dim) * dim + d] - mean[d]));
    if (s == 0.0) s = 1.0;
    for (int64_t a = 0; a < nn; ++a) {
        double X[3] = {0, 0, 0};
        for (int d = 0; d < dim; ++d) X[d] = (coords[(a * dim) * dim + d] - mean[d]) / s;
        double* b = &B[(size_t)a * dim * k];
        for (int cpt = 0; cpt < dim; ++cpt) b[cpt * k + cpt] = 1.0;
        if (dim == 2) {
            b[0 * k + 2] = -X[1];
            b[1 * k + 2] = X[0];
        } else {
            b[1 * k + 3] = -X[2]; b[2 * k + 3] = X[1];
            b[0 * k + 4] = X[2];  b[2 * k + 4] = -X[0];
            b[0 * k + 5] = -X[1]; b[1 * k + 5] = X[0];
        }
    }
}

std::unique_ptr<PC> make_pc(Ctx& c, const std::string& pc_type, const Csr& A, int bs, const double* coords_host,
                            int coord_dim, const std::string& prefix, DistPlan* plan) {
    if (pc_type == "none") return std::make_unique<PCNone>(&c, A.nrows);
    if (pc_type == "jacobi") return std::make_unique<PCJacobi>(&c, A);
    bool want_lu = pc_type == "lu" || pc_type == "cholesky";
    if (!plan && use_sparse_lu(c, pc_type, prefix, A.nrows)) return std::make_unique<PCSparseLU>(&c, A, prefix);
    if (want_lu && !plan && A.nrows <=c.opt_i("-poro_dense_lu_limit", 8192)) return std::make_unique<PCDense>(&c, A);
    const bool cheb_only = pc_type == "chebyshev";      // Chebyshev(degree) on D^-1 A = a one-level hierarchy
    const bool mg = pc_type == "mg";                    // geometric levels on top of the SA-AMG (mg.cuh)
    int mg_levels = 0;
    if (mg) {
        const std::string key = "-" + prefix + "pc_type mg";
        if (!A.stencil || A.stencil->fr < 0 || A.stencil->fc != A.stencil->fr)
            throw Error(key + " needs a single generated field block; this block has no class-stencil descriptor (uploaded "
                        "through poro_mat_create_csr, permuted, cut across several fields, or a Schur complement)");
        if (c.nranks > 1 && !(plan && A.stencil->d->slab))
            throw Error(key + ": a row-partitioned block runs the distributed hierarchy on its generated slabs (-poro_amg_distributed 1)");
        const int attached = mg_attached_levels(*A.stencil);
        if (attached == 0)
            throw Error(key + ": the generated matrix has no coarse levels attached (poro_mat_set_coarse, or mg_levels > 1 in "
                        "the generator)");
        mg_levels = c.opt_i("-" + prefix + "pc_mg_levels", attached + 1);
        if (mg_levels < 1) throw Error("-" + prefix + "pc_mg_levels must be at least 1");
        mg_levels = std::min(mg_levels, attached + 1);
    }
    if (want_lu || cheb_only || mg || pc_type == "hypre" || pc_type == "amg" || pc_type == "gamg" || pc_type == "ml") {
        auto pc = std::make_unique<PCAmg>();
        AmgParams p;
        p.theta = c.opt_d("-" + prefix + "pc_amg_theta", c.opt_d("-pc_amg_theta", p.theta));
        p.cheby_degree = c.opt_i("-" + prefix + "pc_amg_cheby_degree", c.opt_i("-pc_amg_cheby_degree", p.cheby_degree));
        p.coarse_size = c.opt_i("-" + prefix + "pc_amg_coarse_size", c.opt_i("-pc_amg_coarse_size", p.coarse_size));
        p.max_levels = c.opt_i("-" + prefix + "pc_amg_max_levels", c.opt_i("-pc_amg_max_levels", p.max_levels));
        p.cheby_ratio = c.opt_d("-" + prefix + "pc_amg_cheby_ratio", c.opt_d("-pc_amg_cheby_ratio", p.cheby_ratio));
        p.post_smooth = c.opt_i("-" + prefix + "pc_amg_post_smooth", c.opt_i("-pc_amg_post_smooth", p.post_smooth));
        p.power_its = c.opt_i("-" + prefix + "pc_amg_power_its", c.opt_i("-pc_amg_power_its", p.power_its));
        if (cheb_only) {
            p.smoother_only = true;       // Chebyshev(degree) at every size: never the dense coarse inverse
            p.max_levels = 1;
            p.cheby_degree = c.opt_i("-" + prefix + "pc_amg_cheby_degree", 4);
        }
        p.mg_levels = mg_levels;
        bool use_rbm = c.opt_i("-" + prefix + "pc_amg_rigid_body_modes", c.opt_i("-pc_amg_rigid_body_modes", 1)) != 0;
        if (bs > 1 && coords_host && coord_dim == bs && use_rbm) {
            std::vector<double> B;
            int k;
            rigid_body_modes(coords_host, A.nrows, coord_dim, B, k);
            DBuf<double> Bd(B.size());
            PORO_CUDA(cudaMemcpy(Bd.p, B.data(), B.size() * 8, cudaMemcpyHostToDevice));
            pc->amg.setup(c, A, bs, Bd.p, k, p, plan);
        } else {
            pc->amg.setup(c, A, bs > 0 ? bs : 1, nullptr, bs > 0 ? bs : 1, p, plan);
        }
        return pc;
    }
    throw Error("unsupported pc type '" + pc_type + "' for prefix " + prefix);
}

// =============================================================================================
// KSP
// =============================================================================================
void KSP::set_from_options(const std::string& pre) {
    prefix = pre;
    Ctx& c = *ctx;
    auto key = [&](const char* k) { return "-" + pre + k; };
    type = c.opt(key("ksp_type"), type);
    rtol = c.opt_d(key("ksp_rtol"), rtol);
    atol = c.opt_d(key("ksp_atol"), atol);
    dtol = c.opt_d(key("ksp_divtol"), dtol);
    max_it = c.opt_i(key("ksp_max_it"), max_it);
    restart = c.opt_i(key("ksp_gmres_restart"), restart);
    if (c.has_opt(key("ksp_pc_side"))) right = c.opt(key("ksp_pc_side"), "left") == "right";
    if (c.has_opt(key("ksp_norm_type"))) {
        std::string nt = c.opt(key("ksp_norm_type"), "");
        unprec_norm = nt == "unpreconditioned";
        natural_norm = nt == "natural";
        if (unprec_norm && (type == "gmres")) right = true;   // PETSc: GMRES supports the true norm only with right PC
    }
    std::string ref = c.opt(key("ksp_gmres_cgs_refinement_type"), "");
    if (ref == "refine_always") cgs2 = true;
    if (ref == "refine_never") cgs2 = false;
    monitor = c.has_opt(key("ksp_monitor"));
    fused_gs = c.opt_i("-poro_gmres_fused_gs", 0) != 0;
    verify_true = c.has_opt(key("ksp_gmres_verify_true_residual")) && c.opt(key("ksp_gmres_verify_true_residual"), "1") != "0";
    converged_reason = c.has_opt(key("ksp_converged_reason"));
    if (c.has_opt(key("ksp_initial_guess_nonzero"))) {
        std::string v = c.opt(key("ksp_initial_guess_nonzero"), "");
        guess_nonzero = !(v == "0" || v == "false" || v == "no");
    }
    monitor_fields = c.has_opt(key("ksp_monitor_fields"));
    test_fields = c.has_opt(key("ksp_convergence_test_fields"));
    if (type == "fgmres") right = true;
}

int KSP::converged(double rn, int it, double& rnorm0, double& ttol) const {
    if (it == 0) { rnorm0 = rn; ttol = std::max(rtol * rn, atol); }
    if (rn != rn) return -9;
    if (rn <= ttol) return rn < atol ? 3 : 2;
    if (rn >= dtol * rnorm0) return -4;
    return 0;
}

KSP::~KSP() {
    for (auto e : ev) cudaEventDestroy(e);
}

void KSP::op_apply(const double* x, double* y, SpmvMode mode, const double* z) {
    ProfScope ps(*ctx, 0);
    if (!profile_op) { A->apply(x, y, mode, z); return; }
    if (ev_used + 2 > ev.size()) {
        for (int i = 0; i < 2; ++i) { cudaEvent_t e; PORO_CUDA(cudaEventCreate(&e)); ev.push_back(e); }
    }
    PORO_CUDA(cudaEventRecord(ev[ev_used], ctx->stream));
    A->apply(x, y, mode, z);
    PORO_CUDA(cudaEventRecord(ev[ev_used + 1], ctx->stream));
    ev_used += 2;
}

void KSP::profile_flush() {
    if (!ev_used) return;
    PORO_CUDA(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i + 1 < ev_used; i += 2) {
        float ms = 0.f;
        PORO_CUDA(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
        op_ms += ms;
        op_calls++;
    }
    ev_used = 0;
}

void KSP::solve(const double* b, double* x) {
    calls++;
    history.clear();
    its = 0;
    reason = 0;
    if (type == "preonly") {
        if (ctx->capture_log) ctx->capture_log->push_back(this);
        pc->apply(b, x);
        its = 1;
        reason = 4;
        total_its += 1;
        return;
    }
    if (type == "cg") solve_cg(b, x);
    else if (type == "gmres") solve_gmres(b, x, false);
    else if (type == "fgmres") solve_gmres(b, x, true);
    else throw Error("unsupported ksp type '" + type + "' (prefix " + prefix + ")");
    total_its += its;
    if (profile_op) profile_flush();
    if (converged_reason && ctx->rank == 0) {
        // PETSc's -ksp_converged_reason line (KSPConvergedReasonView)
        const char* nm = reason == 2 ? "CONVERGED_RTOL" : reason == 3 ? "CONVERGED_ATOL" : reason == 4 ? "CONVERGED_ITS" :
                         reason == -3 ? "DIVERGED_ITS" : reason == -4 ? "DIVERGED_DTOL" : reason == -5 ? "DIVERGED_BREAKDOWN" :
                         reason == -8 ? "DIVERGED_INDEFINITE_PC" : reason == -9 ? "DIVERGED_NANORINF" :
                         reason == -10 ? "DIVERGED_INDEFINITE_MAT" : "UNKNOWN";
        printf("Linear %s solve %s due to %s iterations %d\n", prefix.c_str(), reason > 0 ? "converged" : "did not converge", nm, its);
    }
}

// The revived `converged` callback of lib/Solver.py:8-51: per-field infinity norms of the TRUE residual b - A x_it,
// normalised by max(||b_s||_2, ||b_f||_2, ||b_p||_2) (lib/Solver.py:17-18,125-127).  Returns 1 / -1 / 0 like the reference.
int KSP::fields_test(const double* b, const double* xcur, int it) {
    Ctx& c = *ctx;
    const int64_t n = A->rows();
    if ((int64_t)w3.n < n) w3.alloc(n);
    double* ds = c.d_scal + Ctx::kScal + 4096 + 4096 - 32;
    double h[3];
    if (it == 0) {
        const double* xs[3] = {b + fields->off[0], b + fields->off[1], b + fields->off[2]};
        // three segment dots of different lengths: one launch each (set-up of the monitor, once per solve)
        for (int t = 0; t < 3; ++t) {
            if (fields->n[t] > 0) vec_dots(c, 1, &xs[t], &xs[t], fields->n[t], ds + t);
            else PORO_CUDA(cudaMemsetAsync(ds + t, 0, sizeof(double), c.stream));
        }
        allreduce_sum(c, ds, 3);
        fetch(c, ds, 3, h);
        for (int t = 0; t < 3; ++t) b0_fields[t] = std::sqrt(h[t]);
        field_history.clear();
    }
    if (xcur) A->apply(xcur, w3.p, SPMV_SUB, b); else vec_copy(c, w3.p, b, n);     // KSP.buildResidual (lib/Solver.py:19)
    vec_amax_segments(c, w3.p, fields->off, fields->n, 3, ds);
    allreduce_max(c, ds, 3);
    fetch(c, ds, 3, h);
    const double normalize = std::max(b0_fields[0], std::max(b0_fields[1], b0_fields[2]));
    const double rr[3] = {h[0] / normalize, h[1] / normalize, h[2] / normalize};
    for (int t = 0; t < 3; ++t) field_history.push_back(h[t]);
    if (monitor_fields && c.rank == 0) {
        if (it == 0) printf("KSP errors: %11s, %11s, %11s, %11s, %11s, %11s\n", "abs_s", "abs_f", "abs_p", "rel_s", "rel_f", "rel_p");
        printf("KSP it %d:   %.5e, %.5e, %.5e, %.5e, %.5e, %.5e\n", it, h[0], h[1], h[2], rr[0], rr[1], rr[2]);
    }
    const double error_abs = std::max(h[0], std::max(h[1], h[2])), error_rel = std::max(rr[0], std::max(rr[1], rr[2]));
    if (error_abs < atol || error_rel < rtol) return 1;
    if (it > max_it || error_abs > dtol) return -1;
    return 0;
}

void KSP::solve_gmres(const double* b, double* x, bool flexible) {
    Ctx& c = *ctx;
    const int64_t n = A->rows();
    const bool rpc = right || flexible;
    const int m = std::max(1, std::min(restart, max_it));
    const bool use_fields = fields && fields->set && (monitor_fields || test_fields);
    if (v_cols < m + 1 || (int64_t)V.n < (int64_t)(m + 1) * n) { V.alloc((size_t)(m + 1) * n); v_cols = m + 1; }
    if (flexible && (int64_t)Z.n < (int64_t)m * n) Z.alloc((size_t)m * n);
    if ((int64_t)w1.n < n) { w1.alloc(n); w2.alloc(n); }
    if ((use_fields || verify_true) && (int64_t)xtmp.n < n) xtmp.alloc(n);      // persistent: no allocation inside a solve
    bool refine = cgs2;          // second Gram-Schmidt pass; switched on for the rest of a solve when a verification fails
    double calib = 1.0;          // measured ratio (true residual) / (recurrence estimate), applied to the convergence test
    bool x_final = false;        // x already holds the verified solution of the current cycle
    std::vector<double> H((size_t)(m + 1) * m, 0.0), cs(m), sn(m), g(m + 1), hbuf(2 * (m + 1) + 2);
    auto Hm = [&](int i, int j) -> double& { return H[(size_t)i * m + j]; };
    double* d_h = c.d_scal + Ctx::kScal + 4096 + 16;   // [h (m+1) | h2 (m+1) | nrm2]; small-slot region
    PORO_REQUIRE(2 * (m + 1) + 2 <= 4096 - 16, "restart too large for the scalar scratch");
    if (!guess_nonzero) vec_set(c, x, 0.0, n);
    double rnorm0 = 0, ttol = 0;
    bool first = true;
    reason = 0;
    its = 0;
    // xt += (correction of the current cycle after j steps): the Hessenberg least squares, then V y (through the PC for right PC)
    auto add_correction = [&](double* xt, int j) {
        if (j <= 0) return;
        std::vector<double> y(j);
        for (int i = j - 1; i >= 0; --i) {
            double sum = g[i];
            for (int q = i + 1; q < j; ++q) sum -= Hm(i, q) * y[q];
            y[i] = sum / Hm(i, i);
        }
        if (flexible) vec_maxpy_host(c, xt, Z.p, n, j, y.data(), n);
        else if (rpc) {
            vec_set(c, w1.p, 0.0, n);
            vec_maxpy_host(c, w1.p, V.p, n, j, y.data(), n);
            pc->apply(w1.p, w2.p);
            vec_axpy(c, xt, 1.0, w2.p, n);
        } else vec_maxpy_host(c, xt, V.p, n, j, y.data(), n);
    };
    while (reason == 0) {
        double* r = V.p;   // column 0
        const bool zero_x = first && !guess_nonzero;
        if (zero_x) vec_copy(c, w1.p, b, n);
        else A->apply(x, w1.p, SPMV_SUB, b);
        if (!rpc) pc->apply(w1.p, r); else vec_copy(c, r, w1.p, n);
        double beta = norm2_host(c, r, n);
        if (first) {
            history.push_back(beta);
            double bnorm = beta;
            if (guess_nonzero) {
                // PETSc's default test measures against ||b|| (preconditioned for left PC) when the guess is non-zero
                if (!rpc) { pc->apply(b, w2.p); bnorm = norm2_host(c, w2.p, n); }
                else bnorm = norm2_host(c, b, n);
            }
            reason = converged(bnorm, 0, rnorm0, ttol);
            if (guess_nonzero) reason = beta != beta ? -9 : (beta <= ttol ? (beta < atol ? 3 : 2) : 0);
            first = false;
            if (monitor && c.rank == 0) printf("  %s KSP residual norm[%d] %.12e\n", prefix.c_str(), 0, beta);
            if (use_fields) {
                int t = fields_test(b, zero_x ? nullptr : x, 0);
                if (test_fields) reason = t > 0 ? 2 : (t < 0 ? -4 : 0);
            }
            if (reason) break;
        }
        if (beta == 0.0) { reason = 3; break; }
        vec_scale(c, r, 1.0 / beta, n);
        std::fill(g.begin(), g.end(), 0.0);
        g[0] = beta;
        int j = 0;
        while (reason == 0 && j < m && its < max_it) {
            double* vj = V.p + (size_t)j * n;
            double* w = V.p + (size_t)(j + 1) * n;
            if (flexible) { double* zj = Z.p + (size_t)j * n; pc->apply(vj, zj); op_apply(zj, w); }
            else if (rpc) { pc->apply(vj, w1.p); op_apply(w1.p, w); }
            else { op_apply(vj, w1.p); pc->apply(w1.p, w); }
            // classical Gram-Schmidt: one multi-dot pass, one multi-axpy(+norm) pass, one scaling pass.
            // (-poro_gmres_fused_gs 1 takes the norm from Pythagoras, ||w - V h||^2 = w.w - h.h, and fuses update and scaling
            // into one pass.  MEASURED TO BE UNSAFE with unrefined CGS: as orthogonality of V degrades the identity is off by
            // O(loss) * w.w, which is of the size of the norm itself late in a solve; the Arnoldi relation breaks and the
            // recurrence residual stalls while the true one keeps falling (100 instead of 36 iterations).  Off by default.)
            double hn = 0.0;
            bool scaled = false;
            {
                ProfScope ps_gs(c, 5);
                if (!refine && fused_gs) {
                    vec_mdot(c, V.p, n, j + 1, w, n, d_h, true);
                    allreduce_sum(c, d_h, j + 2);
                    fetch(c, d_h, j + 2, hbuf.data());
                    double hh = 0.0;
                    for (int i = 0; i <= j; ++i) hh += hbuf[i] * hbuf[i];
                    const double ww = hbuf[j + 1], hn2 = ww - hh;
                    if (hn2 > 1e-4 * ww) {
                        hn = std::sqrt(hn2);
                        vec_maxpy_scale(c, w, V.p, n, j + 1, d_h, n, 1.0 / hn);
                        scaled = true;
                    } else {
                        vec_maxpy_norm(c, w, V.p, n, j + 1, d_h, n, d_h + 2 * (m + 1));
                        allreduce_sum(c, d_h + 2 * (m + 1), 1);
                        double nn2;
                        fetch(c, d_h + 2 * (m + 1), 1, &nn2);
                        hn = std::sqrt(nn2);
                    }
                    for (int i = 0; i <= j; ++i) hbuf[(m + 1) + i] = 0.0;
                } else {
                    vec_mdot(c, V.p, n, j + 1, w, n, d_h, false);
                    allreduce_sum(c, d_h, j + 1);
                    vec_maxpy_norm(c, w, V.p, n, j + 1, d_h, n, d_h + 2 * (m + 1));
                    if (refine) {
                        double* d_h2 = d_h + (m + 1);
                        vec_mdot(c, V.p, n, j + 1, w, n, d_h2, false);
                        allreduce_sum(c, d_h2, j + 1);
                        vec_maxpy_norm(c, w, V.p, n, j + 1, d_h2, n, d_h + 2 * (m + 1));
                    }
                    allreduce_sum(c, d_h + 2 * (m + 1), 1);
                    fetch(c, d_h, 2 * (m + 1) + 1, hbuf.data());
                    hn = std::sqrt(hbuf[2 * (m + 1)]);
                }
            }
            for (int i = 0; i <= j; ++i) Hm(i, j) = hbuf[i] + (refine ? hbuf[(m + 1) + i] : 0.0);
            Hm(j + 1, j) = hn;
            if (hn > 0.0 && !scaled) vec_scale(c, w, 1.0 / hn, n);
            for (int i = 0; i < j; ++i) {
                double t = cs[i] * Hm(i, j) + sn[i] * Hm(i + 1, j);
                Hm(i + 1, j) = -sn[i] * Hm(i, j) + cs[i] * Hm(i + 1, j);
                Hm(i, j) = t;
            }
            double den = std::hypot(Hm(j, j), Hm(j + 1, j));
            if (den == 0.0 || den != den) { reason = den != den ? -9 : -5; break; }
            cs[j] = Hm(j, j) / den;
            sn[j] = Hm(j + 1, j) / den;
            Hm(j, j) = den;
            Hm(j + 1, j) = 0.0;
            g[j + 1] = -sn[j] * g[j];
            g[j] = cs[j] * g[j];
            ++its;
            ++j;
            double res = std::fabs(g[j]);
            history.push_back(res);
            if (monitor && c.rank == 0) printf("  %s KSP residual norm[%d] %.12e\n", prefix.c_str(), its, res);
            reason = converged(res * calib, its, rnorm0, ttol);
            if (reason > 0 && verify_true && rpc && !flexible) {
                // The recurrence says "converged".  Classical Gram-Schmidt loses orthogonality over long cycles and the
                // estimate then runs ahead of the true residual: form the candidate solution, check b - A x, and if it is not
                // there yet KEEP the Krylov space, calibrate the estimate, switch the second Gram-Schmidt pass on and go on.
                vec_copy(c, xtmp.p, x, n);
                add_correction(xtmp.p, j);
                A->apply(xtmp.p, w1.p, SPMV_SUB, b);
                const double tr = norm2_host(c, w1.p, n);
                if (tr <= ttol) {
                    vec_copy(c, x, xtmp.p, n);
                    history.back() = tr;
                    x_final = true;
                } else {
                    if (monitor && c.rank == 0)
                        printf("  %s true residual %.6e (estimate %.6e) above %.6e at iteration %d: continuing with refinement\n",
                               prefix.c_str(), tr, res, ttol, its);
                    calib = std::max(calib, 1.1 * tr / std::max(res, 1e-300));
                    refine = true;
                    reason = 0;
                }
            }
            if (use_fields) {
                vec_copy(c, xtmp.p, x, n);
                add_correction(xtmp.p, j);
                int t = fields_test(b, xtmp.p, its);
                if (test_fields) reason = t > 0 ? 2 : (t < 0 ? -4 : 0);
            }
            if (hn == 0.0 && reason == 0) reason = 2;
        }
        if (!x_final) add_correction(x, j);
        if (reason == 0 && its >= max_it) reason = -3;
    }
    rnorm = history.empty() ? 0.0 : history.back();
}

// x += a p ; r -= a w with a = beta / dpi read from device scalars
__global__ void __launch_bounds__(256) k_cg_update(double* __restrict__ x, double* __restrict__ r,
                                                   const double* __restrict__ p, const double* __restrict__ w,
                                                   const double* __restrict__ beta, const double* __restrict__ dpi,
                                                   int64_t n) {
    const double d = *dpi;
    if (!(d > 0.0)) return;      // indefinite operator (or NaN): leave x, r untouched; the host reports -10 / -9
    const double a = *beta / d;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        x[i] = fma(a, p[i], x[i]);
        r[i] = fma(-a, w[i], r[i]);
    }
}

void KSP::solve_cg(const double* b, double* x) {
    Ctx& c = *ctx;
    const int64_t n = A->rows();
    if ((int64_t)w1.n < n) { w1.alloc(n); w2.alloc(n); }
    if ((int64_t)w3.n < n) w3.alloc(n);
    if ((int64_t)V.n < n) V.alloc(n);
    double* r = w1.p; double* z = w2.p; double* p = w3.p; double* w = V.p;
    double* ds = c.d_scal + Ctx::kScal + 4096 + 4096 - 64;   // [beta, nrm, dpi]
    double hs[4];
    vec_set(c, x, 0.0, n);
    vec_copy(c, r, b, n);
    pc->apply(r, z);
    auto norms = [&]() {
        // beta = r.z ; second = z.z | r.r | (natural: beta)
        const double* xs[2] = {r, unprec_norm ? r : z};
        const double* ys[2] = {z, unprec_norm ? r : z};
        vec_dots(c, 2, xs, ys, n, ds);
        allreduce_sum(c, ds, 3);
        fetch(c, ds, 3, hs);
    };
    PORO_CUDA(cudaMemsetAsync(ds + 2, 0, sizeof(double), c.stream));
    norms();
    double beta = hs[0];
    double dp = natural_norm ? std::sqrt(std::fabs(beta)) : std::sqrt(hs[1]);
    double rnorm0 = 0, ttol = 0;
    history.push_back(dp);
    reason = converged(dp, 0, rnorm0, ttol);
    double betaold = 1.0;
    bool have_p = false;
    while (reason == 0) {
        if (beta == 0.0) { reason = 3; break; }
        if (!have_p) { vec_copy(c, p, z, n); have_p = true; }
        else vec_aypx(c, p, beta / betaold, z, n);
        // w = A p ; dpi = p.w (fused); a = beta/dpi stays on the device
        {
            MatOp* mo = dynamic_cast<MatOp*>(A);
            if (mo && c.nranks == 1 && mo->parts.empty() && mo->pieces.empty()) spmv_dot(c, mo->mat(), p, w, ds + 2);
            else {
                A->apply(p, w);
                const double* xs[1] = {p};
                const double* ys[1] = {w};
                vec_dots(c, 1, xs, ys, n, ds + 2);
            }
        }
        if (c.nranks > 1) allreduce_sum(c, ds + 2, 1);
        k_cg_update<<<stream_grid(c, n, 256, 2), 256, 0, c.stream>>>(x, r, p, w, ds, ds + 2, n);
        PORO_LAUNCH_CHECK(c);
        pc->apply(r, z);
        betaold = beta;
        {
            const double* xs[2] = {r, unprec_norm ? r : z};
            const double* ys[2] = {z, unprec_norm ? r : z};
            double* dn = ds + 4;   // new [beta, nrm]; copied over the old ones after the fetch
            vec_dots(c, 2, xs, ys, n, dn);
            if (c.nranks > 1) allreduce_sum(c, dn, 2);
            double h5[5];
            fetch(c, ds + 2, 4, h5);   // dpi, pad, beta_new, nrm_new
            double dpi = h5[0];
            beta = h5[2];
            dp = natural_norm ? std::sqrt(std::fabs(beta)) : std::sqrt(h5[3]);
            PORO_CUDA(cudaMemcpyAsync(ds, dn, 2 * sizeof(double), cudaMemcpyDeviceToDevice, c.stream));
            if (!(dpi > 0.0)) { reason = dpi != dpi ? -9 : -10; }   // KSP_DIVERGED_INDEFINITE_MAT
        }
        ++its;
        history.push_back(dp);
        if (monitor && c.rank == 0) printf("    %s KSP residual norm[%d] %.12e\n", prefix.c_str(), its, dp);
        if (reason == 0) reason = converged(dp, its, rnorm0, ttol);
        if (reason == 0 && its >= max_it) reason = -3;
    }
    rnorm = dp;
}

// =============================================================================================
// fieldsplit Schur on the fp block
// =============================================================================================
void PCSchur::solve1(const double* r, double* y1) {
    k1->solve(r, y1);
    if (kv) {
        kv->solve(r, tv.p);
        vec_axpy(*ctx, y1, 1.0 / visc_scale, tv.p, n1);
    }
}

void PCSchur::apply(const double* x, double* y) {
    Ctx& c = *ctx;
    const double* x0 = x + off0; const double* x1 = x + off1;
    double* y0 = y + off0; double* y1 = y + off1;
    if (fact == 0) {                       // lower: y0 = K0 x0 ; y1 = K1 (x1 - A10 y0)
        { ProfScope ps(c, 3); k0->solve(x0, y0); }
        { ProfScope ps(c, 6); A10->apply(y0, t1.p, SPMV_SUB, x1); }
        { ProfScope ps(c, 4); solve1(t1.p, y1); }
    } else if (fact == 1) {                // upper: y1 = K1 x1 ; y0 = K0 (x0 - A01 y1)
        solve1(x1, y1);
        A01->apply(y1, t0.p, SPMV_SUB, x0);
        k0->solve(t0.p, y0);
    } else if (fact == 2) {                // full: lower sweep then upper correction
        k0->solve(x0, u0.p);
        A10->apply(u0.p, t1.p, SPMV_SUB, x1);
        solve1(t1.p, y1);
        A01->apply(y1, t0.p, SPMV_SUB, x0);
        k0->solve(t0.p, y0);
    } else {                               // diag (PETSc flips the sign of the Schur block)
        k0->solve(x0, y0);
        solve1(x1, y1);
        vec_scale(c, y1, -1.0, n1);
    }
}

// =============================================================================================
// Gram least squares shared by AAR and Anderson
// =============================================================================================
// G = F^T F and g = F^T f in one pass over the window (tall-skinny Gram), m <= 10 columns
template <int MAXM>
__global__ void __launch_bounds__(256) k_gram(const double* __restrict__ F, int64_t ld, int m, const double* __restrict__ f,
                                              int64_t n, double* __restrict__ partial) {
    constexpr int NT = MAXM * (MAXM + 1) / 2 + MAXM;
    double acc[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) acc[t] = 0.0;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double v[MAXM];
#pragma unroll
        for (int a = 0; a < MAXM; ++a) v[a] = a < m ? F[(int64_t)a * ld + i] : 0.0;
        const double fi = f[i];
        int t = 0;
#pragma unroll
        for (int a = 0; a < MAXM; ++a) {
#pragma unroll
            for (int b = a; b < MAXM; ++b) { acc[t] = fma(v[a], v[b], acc[t]); ++t; }
        }
#pragma unroll
        for (int a = 0; a < MAXM; ++a) acc[t + a] = fma(v[a], fi, acc[t + a]);
    }
    __shared__ double sm[8][NT];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        double s = acc[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
        if (lane == 0) sm[warp][t] = s;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < NT; t += 256) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += sm[w][t];
        partial[(size_t)blockIdx.x * NT + t] = s;
    }
}

__global__ void k_sum_cols(const double* __restrict__ partial, int nparts, int k, double* __restrict__ out) {
    int j = blockIdx.x;
    __shared__ double sm[8];
    double s = 0.0;
    for (int p = threadIdx.x; p < nparts; p += 256) s += partial[(size_t)p * k + j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { double t = 0.0; for (int w = 0; w < 8; ++w) t += sm[w]; out[j] = t; }
}

// symmetric eigen-decomposition by cyclic Jacobi (m <= ~16)
static void jacobi_eig(int m, std::vector<double>& A, std::vector<double>& V, std::vector<double>& w) {
    V.assign((size_t)m * m, 0.0);
    for (int i = 0; i < m; ++i) V[(size_t)i * m + i] = 1.0;
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0;
        for (int i = 0; i < m; ++i) for (int j = i + 1; j < m; ++j) off += A[(size_t)i * m + j] * A[(size_t)i * m + j];
        if (off < 1e-300) break;
        for (int p = 0; p < m; ++p)
            for (int q = p + 1; q < m; ++q) {
                double apq = A[(size_t)p * m + q];
                if (std::fabs(apq) < 1e-300) continue;
                double app = A[(size_t)p * m + p], aqq = A[(size_t)q * m + q];
                double tau = (aqq - app) / (2.0 * apq);
                double t = (tau >= 0 ? 1.0 : -1.0) / (std::fabs(tau) + std::sqrt(1.0 + tau * tau));
                double cc = 1.0 / std::sqrt(1.0 + t * t), ss = t * cc;
                for (int k = 0; k < m; ++k) {
                    double akp = A[(size_t)k * m + p], akq = A[(size_t)k * m + q];
                    A[(size_t)k * m + p] = cc * akp - ss * akq;
                    A[(size_t)k * m + q] = ss * akp + cc * akq;
                }
                for (int k = 0; k < m; ++k) {
                    double apk = A[(size_t)p * m + k], aqk = A[(size_t)q * m + k];
                    A[(size_t)p * m + k] = cc * apk - ss * aqk;
                    A[(size_t)q * m + k] = ss * apk + cc * aqk;
                }
                for (int k = 0; k < m; ++k) {
                    double vkp = V[(size_t)k * m + p], vkq = V[(size_t)k * m + q];
                    V[(size_t)k * m + p] = cc * vkp - ss * vkq;
                    V[(size_t)k * m + q] = ss * vkp + cc * vkq;
                }
            }
    }
    w.resize(m);
    for (int i = 0; i < m; ++i) w[i] = A[(size_t)i * m + i];
}

void gram_alpha(Ctx& c, const double* F, int64_t ld, int order, int nF, int headF, const double* f, int64_t n,
                std::vector<double>& alpha) {
    // slot s holds logical column (s - headF) mod order; compute on slots, permute on the host
    const int m = nF;
    alpha.assign(m, 0.0);
    if (m == 0) return;
    std::vector<double> G((size_t)m * m), rhs(m);
    const int nslots = nF < order ? nF : order;   // slots 0..nslots-1 are populated
    if (nslots <= 10) {
        constexpr int MAXM = 10;
        constexpr int NT = MAXM * (MAXM + 1) / 2 + MAXM;
        int grid = stream_grid(c, n, 256, 2, 2);
        while ((int64_t)grid * NT > Ctx::kScal && grid > 1) grid /= 2;
        k_gram<MAXM><<<grid, 256, 0, c.stream>>>(F, ld, nslots, f, n, c.d_scal);
        PORO_LAUNCH_CHECK(c);
        double* d_out = c.d_scal + Ctx::kScal + 4096 + 16;
        k_sum_cols<<<NT, 256, 0, c.stream>>>(c.d_scal, grid, NT, d_out);
        PORO_LAUNCH_CHECK(c);
        allreduce_sum(c, d_out, NT);
        std::vector<double> h(NT);
        fetch(c, d_out, NT, h.data());
        std::vector<double> Gs((size_t)MAXM * MAXM, 0.0);
        int t = 0;
        for (int a = 0; a < MAXM; ++a) for (int b = a; b < MAXM; ++b) { Gs[(size_t)a * MAXM + b] = Gs[(size_t)b * MAXM + a] = h[t]; ++t; }
        for (int i = 0; i < m; ++i) {
            int si = (headF + i) % order;
            rhs[i] = -h[t + si];
            for (int j = 0; j < m; ++j) { int sj = (headF + j) % order; G[(size_t)i * m + j] = Gs[(size_t)si * MAXM + sj]; }
        }
    } else {
        double* d_out = c.d_scal + Ctx::kScal + 4096 + 16;
        std::vector<double> h(nslots + 1);
        std::vector<double> Gs((size_t)nslots * nslots), gs(nslots);
        for (int a = 0; a < nslots; ++a) {
            vec_mdot(c, F, ld, nslots, F + (int64_t)a * ld, n, d_out, false);
            allreduce_sum(c, d_out, nslots);
            fetch(c, d_out, nslots, h.data());
            for (int b = 0; b < nslots; ++b) Gs[(size_t)a * nslots + b] = h[b];
        }
        vec_mdot(c, F, ld, nslots, f, n, d_out, false);
        allreduce_sum(c, d_out, nslots);
        fetch(c, d_out, nslots, gs.data());
        for (int i = 0; i < m; ++i) {
            int si = (headF + i) % order;
            rhs[i] = -gs[si];
            for (int j = 0; j < m; ++j) { int sj = (headF + j) % order; G[(size_t)i * m + j] = Gs[(size_t)si * nslots + sj]; }
        }
    }
    // Jacobi-scaled eigen-solve with relative truncation (same as oracle/aar.py:gram_solve)
    std::vector<double> d(m);
    for (int i = 0; i < m; ++i) d[i] = std::sqrt(std::max(G[(size_t)i * m + i], 1e-300));
    for (int i = 0; i < m; ++i) for (int j = 0; j < m; ++j) G[(size_t)i * m + j] /= d[i] * d[j];
    std::vector<double> Vv, w;
    jacobi_eig(m, G, Vv, w);
    double wmax = 0.0;
    for (double v : w) wmax = std::max(wmax, v);
    std::vector<double> y(m, 0.0);
    for (int e = 0; e < m; ++e) {
        if (!(w[e] > 1e-14 * wmax)) continue;
        double proj = 0.0;
        for (int i = 0; i < m; ++i) proj += Vv[(size_t)i * m + e] * (rhs[i] / d[i]);
        proj /= w[e];
        for (int i = 0; i < m; ++i) y[i] += Vv[(size_t)i * m + e] * proj;
    }
    for (int i = 0; i < m; ++i) alpha[i] = y[i] / d[i];
}

// x += beta f + sum_i alpha_i (X_i + beta F_i), X/F given per logical index through slot maps
__global__ void __launch_bounds__(256) k_anderson_update(double* __restrict__ x, const double* __restrict__ f, double beta,
                                                         const double* __restrict__ X, const double* __restrict__ F,
                                                         int64_t ld, int mk, const double* __restrict__ coef,
                                                         const int* __restrict__ slotX, const int* __restrict__ slotF, int64_t n) {
    __shared__ double a[32];
    __shared__ int sx[32], sf[32];
    if (threadIdx.x < mk) { a[threadIdx.x] = coef[threadIdx.x]; sx[threadIdx.x] = slotX[threadIdx.x]; sf[threadIdx.x] = slotF[threadIdx.x]; }
    __syncthreads();
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double v = fma(beta, f[i], x[i]);
        for (int q = 0; q < mk; ++q) v = fma(a[q], X[(int64_t)sx[q] * ld + i] + beta * F[(int64_t)sf[q] * ld + i], v);
        x[i] = v;
    }
}

static void anderson_update(Ctx& c, double* x, const double* f, double beta, const double* X, const double* F, int64_t ld,
                            int mk, const std::vector<double>& alpha, int order, int headX, int headF, int64_t n) {
    PORO_REQUIRE(mk <= 32, "Anderson window larger than 32");
    double* hp = c.h_pin + 4096;
    int* hi = (int*)(hp + 64);
    for (int q = 0; q < mk; ++q) { hp[q] = alpha[q]; hi[q] = (headX + q) % order; hi[32 + q] = (headF + q) % order; }
    double* dcoef = c.d_scal + Ctx::kScal;
    PORO_CUDA(cudaMemcpyAsync(dcoef, hp, (64 + 32) * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    const int* dslot = (const int*)(dcoef + 64);
    k_anderson_update<<<stream_grid(c, n, 256, 2), 256, 0, c.stream>>>(x, f, beta, X, F, ld, mk, dcoef, dslot, dslot + 32, n);
    PORO_LAUNCH_CHECK(c);
    PORO_CUDA(cudaStreamSynchronize(c.stream));
}

// ring-buffer append: returns slot written
static int ring_push(int order, int& count, int& head) {
    if (count < order) return (head + count++) % order;
    int slot = head;
    head = (head + 1) % order;
    return slot;
}

// =============================================================================================
// AAR
// =============================================================================================
void AAR::solve(const double* b, double* sol) {
    Ctx& c = *ctx;
    n = A->rows();
    if ((int64_t)xk.n < n) {
        xk.alloc(n); fk.alloc(n); dfk.alloc(n); dxk.alloc(n); tmp.alloc(n);
        if (order > 0) { F.alloc((size_t)order * n); X.alloc((size_t)order * n); }
    }
    history.clear();
    types.clear();
    vec_set(c, xk.p, 0.0, n);                               // AAR.py:48-50
    vec_copy(c, fk.p, b, n);                                // AAR.py:55-56 (x0 = 0)
    double error0 = norm2_host(c, fk.p, n);                 // :67
    double err_abs = error0, err_rel = 1.0;
    it = 0;
    history.push_back(err_abs);
    while (err_abs > atol && err_rel > rtol && it < maxit) {  // :73
        vec_copy(c, dfk.p, fk.p, n);                        // :75
        vec_copy(c, dxk.p, xk.p, n);                        // :76
        A->apply(xk.p, tmp.p, SPMV_SUB, b);                 // :133-135
        pc->apply(tmp.p, fk.p);                             // :137
        vec_aypx(c, dfk.p, -1.0, fk.p, n);                  // :78  dfk = fk - dfk
        if (order > 0) {
            int slot = ring_push(order, nF, headF);         // :80-82
            vec_copy(c, F.p + (size_t)slot * n, dfk.p, n);
        }
        double nf = norm2_host(c, fk.p, n);
        char typ = ' ';
        bool natural = std::fmod((double)(it + 1) / (double)p, 1.0) > 0.0;
        if (nf < 1e-14) {                                   // :91
        } else if (it == 0 || order == 0 || natural) {      // :94
            typ = 'R';
            vec_axpy(c, xk.p, omega, fk.p, n);
        } else {
            typ = 'A';
            int mk = std::min(order, it);                   // :99
            std::vector<double> alpha;
            gram_alpha(c, F.p, n, order, nF, headF, fk.p, n, alpha);   // :102-105 via the Gram matrix
            mk = std::min(mk, nX);
            anderson_update(c, xk.p, fk.p, beta, X.p, F.p, n, mk, alpha, order, headX, headF, n);   // :109-111
        }
        vec_aypx(c, dxk.p, -1.0, xk.p, n);                  // :113
        if (order > 0) {
            int slot = ring_push(order, nX, headX);         // :114-116
            vec_copy(c, X.p + (size_t)slot * n, dxk.p, n);
        }
        err_abs = nf;                                       // :117
        err_rel = err_abs / error0;
        ++it;
        history.push_back(err_abs);
        types.push_back(typ);
        if (monitor && c.rank == 0)
            printf("---- Iteration [%c] %3d\tabs=%1.2e\trel=%1.2e\n", typ, it, err_abs, err_rel);
    }
    vec_copy(c, sol, xk.p, n);                              // :126
}

// =============================================================================================
// Anderson acceleration of the preconditioner output
// =============================================================================================
void Anderson::init(Ctx* c, int order_, int64_t n_) {
    ctx = c; order = order_; n = n_; k = 0;
    nF = nX = headF = headX = 0;
}

void Anderson::get_next_vector(double* gk) {
    Ctx& c = *ctx;
    if (k == 0 && (int64_t)xk.n < n) {
        xk.alloc(n); fk.alloc(n); dxk.alloc(n); dfk.alloc(n);
        F.alloc((size_t)order * n); X.alloc((size_t)order * n);
    }
    if (k == 0) { vec_set(c, xk.p, 0.0, n); vec_set(c, fk.p, 0.0, n); }
    vec_copy(c, dfk.p, fk.p, n);                           // :36
    vec_copy(c, dxk.p, xk.p, n);                           // :37
    vec_waxpby(c, fk.p, 1.0, gk, -1.0, xk.p, n);           // :39-40
    int mk = (int)std::min<int64_t>(k, order);             // :42
    if (mk > 0) {
        vec_aypx(c, dfk.p, -1.0, fk.p, n);                 // :44
        if (norm2_host(c, dfk.p, n) < 1e-12) {             // :45-47
            k -= 1;
            vec_copy(c, xk.p, gk, n);
        } else {
            int slot = ring_push(order, nF, headF);        // :49-51
            vec_copy(c, F.p + (size_t)slot * n, dfk.p, n);
            std::vector<double> alpha;
            gram_alpha(c, F.p, n, order, nF, headF, fk.p, n, alpha);   // :60-63
            mk = std::min(mk, std::min(nX, nF));
            anderson_update(c, xk.p, fk.p, 1.0, X.p, F.p, n, mk, alpha, order, headX, headF, n);   // :67-69
        }
    } else {
        vec_copy(c, xk.p, gk, n);                          // :71
    }
    vec_aypx(c, dxk.p, -1.0, xk.p, n);                     // :73
    int slot = ring_push(order, nX, headX);                // :74-76
    vec_copy(c, X.p + (size_t)slot * n, dxk.p, n);
    k += 1;
    vec_copy(c, gk, xk.p, n);                              // :78
}

// =============================================================================================
// PreconditionerCC.apply
// =============================================================================================
struct PhaseTimer {
    Ctx& c; bool on; double& acc;
    std::chrono::steady_clock::time_point t0;
    PhaseTimer(Ctx& c_, bool on_, double& acc_) : c(c_), on(on_), acc(acc_) {
        if (on) { cudaStreamSynchronize(c.stream); t0 = std::chrono::steady_clock::now(); }
    }
    ~PhaseTimer() {
        if (on) {
            cudaStreamSynchronize(c.stream);
            acc += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        }
    }
};

void PCBlockCC::apply(const double* x, double* y) {
    Ctx& c = *ctx;
    const bool can_graph = graph_enabled && !c.prof.on && !timing && anderson.order == 0 && c.capture_log == nullptr;
    if (!can_graph) { apply_impl(x, y); return; }
    // the first application runs eagerly: it performs every lazy allocation and format conversion of the blocks
    if (eager_calls < 1) { ++eager_calls; apply_impl(x, y); return; }
    const int64_t n = fl->n_owned;
    bool fresh = false;
    if (!gexec) {
        g_in.alloc((size_t)n);
        g_out.alloc((size_t)n);
        std::vector<void*> log;
        const int64_t l0 = c.launches;
        cudaGraph_t graph = nullptr;
        PORO_CUDA(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
        c.capture_log = &log;
        try {
            apply_impl(g_in.p, g_out.p);
        } catch (...) {
            c.capture_log = nullptr;
            cudaStreamEndCapture(c.stream, &graph);
            if (graph) cudaGraphDestroy(graph);
            throw;
        }
        c.capture_log = nullptr;
        PORO_CUDA(cudaStreamEndCapture(c.stream, &graph));
        g_launches = c.launches - l0;
        c.launches = l0;
        PORO_CUDA(cudaGraphInstantiate(&gexec, graph, 0));
        cudaGraphDestroy(graph);
        for (void* k : log) g_ksps.push_back(static_cast<KSP*>(k));
        fresh = true;
    }
    vec_copy(c, g_in.p, x, n);
    PORO_CUDA(cudaGraphLaunch(gexec, c.stream));
    ++graph_replays;
    vec_copy(c, y, g_out.p, n);
    c.launches += g_launches;
    if (!fresh)
        for (KSP* k : g_ksps) { k->calls++; k->total_its++; k->its = 1; k->reason = 4; }
}

void PCBlockCC::apply_impl(const double* x, double* y) {
    Ctx& c = *ctx;
    ProfScope ps_pc(c, 1);
    PhaseTimer tt(c, timing, t_total);
    const int64_t ns = fl->n[0], nf = fl->n[1], np = fl->n[2];
    const double* xs = x + fl->off[0]; const double* xf = x + fl->off[1]; const double* xp = x + fl->off[2];
    double* ys = y + fl->off[0]; double* yf = y + fl->off[1]; double* yp = y + fl->off[2];
    if (three_way) {
        {
            PhaseTimer t(c, timing, t_press);
            ksp_p->solve(xp, yp);                                           // :170
            vec_copy(c, t_p.p, xp, np);
            if (bcs_sub_pressure.n) vec_set_idx(c, t_p.p, bcs_sub_pressure.p, 0.0, (int64_t)bcs_sub_pressure.n);   // :172-173
            ksp_diff->solve(t_p.p, y_pd.p);                                 // :174
        }
        {
            PhaseTimer t(c, timing, t_fluid);
            Mf_p->apply(yp, t_f.p, SPMV_SUB, xf);                           // :180-181
            ksp_f->solve(t_f.p, yf);                                        // :182
            Mf_p->apply(y_pd.p, t_f.p, SPMV_SUB, xf);                       // :184-185
            ksp_f->solve(t_f.p, y_fd.p);                                    // :186
        }
        {
            PhaseTimer t(c, timing, t_solid);
            Ms_f->apply(yf, t_s.p, SPMV_SUB, xs);                           // :192-195 (x - Msf yf - Msp yp)
            Ms_p->apply(yp, t_s.p, SPMV_SUB, t_s.p);
            ksp_s->solve(t_s.p, ys);                                        // :196
            Ms_f->apply(y_fd.p, t_s.p, SPMV_SUB, xs);                       // :198-201
            Ms_p->apply(y_pd.p, t_s.p, SPMV_SUB, t_s.p);
            ksp_s->solve(t_s.p, y_sd.p);                                    // :202
        }
        vec_axpby(c, yp, w2, y_pd.p, w1, np);                               // :207-212
        vec_axpby(c, yf, w2, y_fd.p, w1, nf);
        vec_axpby(c, ys, w2, y_sd.p, w1, ns);
    } else if (overlap_blocks && c.capture_log != nullptr && c.nranks <= 1 && Mfp_s->mat().nnz == 0 && Mfp_s->parts.empty()) {
        // being captured: fork / join through events makes the two solves parallel branches of the graph
        if (!side_stream) {
            PORO_CUDA(cudaStreamCreateWithFlags(&side_stream, cudaStreamNonBlocking));
            PORO_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
            PORO_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
        }
        cudaStream_t main_stream = c.stream;
        struct Restore { Ctx& c; cudaStream_t s; ~Restore() { c.stream = s; } } restore{c, main_stream};
        PORO_CUDA(cudaEventRecord(ev_fork, main_stream));
        PORO_CUDA(cudaStreamWaitEvent(side_stream, ev_fork, 0));
        ksp_s->solve(xs, ys);                                               // :221
        c.stream = side_stream;
        ksp_fp->solve(xf, yf);                                              // :232-234 with P_fp,s = 0: t_fp = x_fp
        PORO_CUDA(cudaEventRecord(ev_join, side_stream));
        c.stream = main_stream;
        PORO_CUDA(cudaStreamWaitEvent(main_stream, ev_join, 0));
    } else {
        {
            PhaseTimer t(c, timing, t_solid);
            ProfScope ps(c, 2);
            ksp_s->solve(xs, ys);                                           // :221
        }
        {
            PhaseTimer t(c, timing, t_fluid);
            Mfp_s->apply(ys, t_fp.p, SPMV_SUB, xf);                         // :232-233 (x_fp contiguous from xf)
            ksp_fp->solve(t_fp.p, yf);                                      // :234 (y_fp contiguous from yf)
        }
        t_press = t_fluid;
    }
    if (anderson.order > 0) anderson.get_next_vector(y);                    // :248-249
}

}  // namespace poro
