/* poro.h -- C ABI of libporo.so: the B200 solve phase for three-field poromechanics.
 *
 * The reference (nabw/poroelasticity-linear-solvers) has no C ABI of its own: its solve
 * phase is Python over petsc4py.  Every entry point below names the reference call sites
 * (file:line under the reference root) whose work it takes over; INTEGRATION.md shows the
 * ctypes stubs a maintainer would put in lib/Solver.py / lib/Preconditioner.py.
 *
 * Conventions
 *  - every function returns 0 on success, <0 on error; poro_last_error() gives the message.
 *    Nothing throws across the ABI.  Non-convergence is NOT an error (PETSc semantics): read
 *    `reason` (PETSc KSPConvergedReason codes: 2 rtol, 3 atol, 4 its(preonly), -3 max_it,
 *    -4 dtol, -5 breakdown, -8 indefinite PC, -9 nan, -10 indefinite operator).
 *  - all arithmetic is fp64; column indices int32; row pointers int64 at the ABI.
 *  - pointers named *_dev are device pointers on the ctx's GPU (e.g. torch tensor
 *    data_ptr()); *_host are host pointers.  Vectors are caller-owned and borrowed for the
 *    duration of the call; matrices are copied at creation.
 *  - a ctx is single-threaded; one ctx per process per GPU.  There is no CPU fallback:
 *    poro_ctx_create fails when no CUDA device is present.
 */
#ifndef PORO_H
#define PORO_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct poro_ctx poro_ctx;
typedef struct poro_mat poro_mat;
typedef struct poro_pc poro_pc;
typedef struct poro_ksp poro_ksp;

const char* poro_last_error(void);
int poro_version(void);

/* ---- context -------------------------------------------------------------------------
 * Replaces the implicit PETSc/MPI world of the reference (mpi4py COMM_WORLD, lib/AAR.py:27;
 * PETSc.Options, lib/Parser.py:70-73). */
int poro_ctx_create(int device, poro_ctx** out);
int poro_ctx_destroy(poro_ctx* ctx);
/* one rank per GPU: `nccl_unique_id` = 128 bytes obtained from poro_nccl_unique_id on rank 0
 * and broadcast by the host layer (torch.distributed).  nranks == 1 needs no call. */
int poro_nccl_unique_id(unsigned char* id128);
int poro_ctx_init_dist(poro_ctx* ctx, int rank, int nranks, const unsigned char* id128);
/* PETSc.Options().setValue(key, val) -- lib/Parser.py:70-73; val may be NULL for bare flags */
int poro_options_set(poro_ctx* ctx, const char* key, const char* val);
int poro_options_clear(poro_ctx* ctx);
/* number of CUDA kernels this ctx has launched so far (bench.py's gpu_launches) */
int64_t poro_launch_count(poro_ctx* ctx);
int poro_sync(poro_ctx* ctx);
/* CUDA-event stopwatch on the library's own stream (torch.cuda.Event would only see torch's current stream) */
int poro_timer_start(poro_ctx* ctx);
int poro_timer_stop(poro_ctx* ctx, double* elapsed_ms);

/* ---- matrices ------------------------------------------------------------------------
 * A.mat(), P.mat(), P_diff.mat() handed to Solver / Preconditioner
 * (lib/Solver.py:95, lib/Preconditioner.py:284-289).  CSR of the LOCAL rows; columns index
 * the local extended vector [owned | halo] (single rank: the global vector).  on_device != 0
 * means the three arrays are device pointers. */
int poro_mat_create_csr(poro_ctx* ctx, int64_t nrows, int64_t ncols, const int64_t* rowptr,
                        const int32_t* col, const double* val, int on_device, poro_mat** out);
int poro_mat_destroy(poro_mat* m);
int poro_mat_info(poro_mat* m, int64_t* nrows, int64_t* ncols, int64_t* nnz);
/* y = A x on the raw (un-permuted) matrix: Mat.mult / `matA * x` (lib/AAR.py:56,135); also the
 * SpMV micro-benchmark entry point. */
int poro_mat_mult(poro_mat* m, const double* x_dev, double* y_dev);
/* SpMV micro-benchmark of one uploaded matrix in one of the fused epilogue modes the solver uses (the reference's
 * `mult` + `aypx(-1)` pairs, lib/Preconditioner.py:180-199): 0 y = A x, 1 y = z - A x, 2 y = z + A x, 3 Chebyshev step,
 * 4 w = A p with p.w.  Returns the device time per launch (CUDA events on the library's stream). */
int poro_mat_bench(poro_mat* m, int mode, int reps, double* ms_per_launch);
/* tests of the product kernels on a raw matrix (single rank).  `-poro_mat_block_hint BS` at creation makes the first product
 * try BSR, `-poro_mat_fp32_values 1` stores those BSR values in fp32; the `-poro_bsr_*` options are read at that conversion.
 * poro_mat_mult_mode: one product in the epilogue modes of poro_pc_block_mult.
 * poro_mat_kernel_info: what the next product launches (converting first, as a product would).  out[0..n) receives:
 * format (0 CSR stream, 1 BSR, 2 diagonal BSR, 4 stencil, 5 vector-CSR fallback), lanes per row or block row (G of the
 * stream kernels, L of the fallback), block size, PREF, cooperative gathers, fp32 values, TMA layout, TMA config (-1
 * none), fused coupling, chunks (row blocks of the CSR stream, chunks of the BSR kernels), L2 prefetch.
 * poro_mat_mult_fused: modes 0..2 of y = A x + C x2; the first call tries to let C ride along A's BSR (*fused = 1),
 * otherwise A and C are applied one after the other (*fused = 0). */
int poro_mat_mult_mode(poro_mat* m, int mode, const double* x, double* y, const double* z, double* r, double* d_new, double* xv,
                       const double* dinv, double c1, double c2, double* dot);
int poro_mat_kernel_info(poro_mat* m, int64_t* out, int n);
int poro_mat_mult_fused(poro_mat* a, poro_mat* c, int mode, const double* x, const double* x2, double* y, const double* z,
                        int* fused);

int poro_mat_copy(poro_mat* m, int64_t* rowptr, int32_t* col, double* val);
/* the set-up primitives on raw matrices (tests): op "spgemm" (a b), "transpose" (a^T) or "add_scaled"
 * (a + alpha diag(s) b, s a device vector or NULL for ones); *out is a new matrix, *chunks the SpGEMM's row chunks under
 * -poro_spgemm_chunk (0 for the other ops).  poro_dense_inverse: the Gauss-Jordan inverse of the coarsest AMG level of a
 * row-major n x n host matrix. */
int poro_mat_setup_op(poro_mat* a, poro_mat* b, const char* op, double alpha, const double* s_dev, poro_mat** out, int* chunks);
int poro_dense_inverse(poro_ctx* ctx, int n, const double* a_host, double* inv_host);

/* ---- device-side generator of the assembled system (SURVEY 8 f1) ------------------------------------
 * Replaces the host assembly + DirichletBC.apply of lib/Assembler.py:66-221, lib/Poromechanics.py:76-83 on dolfin's
 * UnitSquareMesh / UnitCubeMesh (lib/MeshCreation.py:11-19,169-178): every field block is one macro-cell matrix scattered
 * over the cells, so a node's block row is one of a few class stencils, shifted.  `tables`: 9 entries, row-major over the
 * field pairs (s, f, p) x (s, f, p); kr / kc: lattice of the row / column field (2 = P2 nodes, 1 = P1 nodes), br x bc
 * values per entry, cls_ptr (ncls + 1), off = column-node offsets, vals; an empty block has cls_ptr == NULL.
 * `layout` (22 int64): for the P1 then the P2 lattice [owned node range o0 o1 | lower-neighbour ghost range | upper-neighbour
 * ghost range]; local dof offsets of the owned / lower-ghost / upper-ghost part of each field (3 + 3 + 3); local column
 * count.  Rows are the owned nodes' dofs, field-major; `bc_flags_host`: one byte per local row (1 = Dirichlet) or NULL.
 * The result is an ordinary poro_mat (local rows x [owned | ghost] columns). */
typedef struct poro_gen_table {
    int kr, kc, br, bc, diag_block, ncls;
    const int32_t* cls_ptr;
    const int64_t* off;
    const double* vals;
} poro_gen_table;
int poro_gen_matrix(poro_ctx* ctx, int dim, int N, const poro_gen_table* tables, const int64_t* layout,
                    const uint8_t* bc_flags_host, poro_mat** out);
/* makes `coarse` the next geometric level of `fine` for `-<prefix>pc_type mg`.  Both come from poro_gen_matrix on one rank
 * with the same dim, the same present tables, the same lattice kinds and block sizes per field, and N_fine = 2 N_coarse;
 * anything else fails naming what differs.  `coarse` may have its own coarse level.  `fine` keeps its own reference to the
 * coarse matrix, so destroying the coarse handle afterwards is safe. */
int poro_mat_set_coarse(poro_mat* fine, poro_mat* coarse);

/* ---- halo plan for row-partitioned runs (MatMult_MPIAIJ's VecScatter in the reference) ---
 * neighbours k = 0..nneigh-1: this rank sends x[send_idx[send_ptr[k]..send_ptr[k+1])] (owned,
 * local numbering) to rank neigh[k] and receives recv_count[k] values which land, in the
 * sender's order, in the halo part of the extended vector (neighbour-major). */
int poro_halo_set(poro_ctx* ctx, int64_t n_owned, int nneigh, const int32_t* neigh,
                  const int64_t* send_ptr, const int32_t* send_idx, const int64_t* recv_count);

/* ---- index sets ----------------------------------------------------------------------
 * IndexSet.get_index_sets() / get_dimensions() (lib/IndexSet.py:29-67).  Entries are positions
 * in the local extended vector (owned first).  two_way_local_fp != 0 declares that is_f / is_p
 * are positions INSIDE the fp sub-vector (the 2-way remap of lib/IndexSet.py:43-54); is_fp is
 * then required.  block_dim = dofs per mesh node of the s and f fields when they are stored
 * node-blocked (0 = unknown / scalar treatment). */
int poro_fields_set(poro_ctx* ctx, const int64_t* is_s, int64_t ns, const int64_t* is_f, int64_t nf,
                    const int64_t* is_p, int64_t np, const int64_t* is_fp, int64_t nfp,
                    int two_way_local_fp, int block_dim);
/* optional: coordinates of the dofs of s (= f) and p, (n x dim) row-major host arrays; used
 * to build rigid-body near-nullspaces for the AMG (PETSc's MatSetNearNullSpace role). */
int poro_fields_set_coords(poro_ctx* ctx, int dim, const double* coords_s_host, const double* coords_p_host);

/* ---- preconditioner ------------------------------------------------------------------
 * Preconditioner.get_pc() + PreconditionerCC.setUp (lib/Preconditioner.py:60-139, 282-291):
 * sub-matrix extraction, inner KSP creation with prefixes s_ f_ p_ fp_ diff_, fieldsplit. */
int poro_pc_setup(poro_ctx* ctx, poro_mat* A, poro_mat* P, poro_mat* P_diff_or_null, const char* pc_type,
                  const char* inner_ksp_type, const char* inner_pc_type,
                  const int64_t* bcs_sub_pressure, int64_t nbc, int accel_order, double w1, double w2,
                  poro_pc** out);
/* PreconditionerCC.apply(pc, x, y) (lib/Preconditioner.py:141-250); x != y */
int poro_pc_apply(poro_pc* pc, const double* x_dev, double* y_dev);
int poro_pc_destroy(poro_pc* pc);
/* t_total, t_solid, t_fluid, t_press, t_alloc (lib/Preconditioner.py:252-260), then
 * per-block inner iteration totals and call counts: s, f, p, fp, diff, fp_split0, fp_split1, then the number of
 * applications replayed from the captured CUDA graph */
int poro_pc_stats(poro_pc* pc, double* out, int n);

/* ---- outer Krylov solver -------------------------------------------------------------
 * Solver.create_solver (lib/Solver.py:92-102): KSP().create(), setOptionsPrefix("global_"),
 * setOperators(A), setType, setTolerances(rtol, atol, divtol, maxit), setPC,
 * setGMRESRestart, setFromOptions. */
int poro_ksp_create(poro_ctx* ctx, poro_mat* A, poro_pc* pc, const char* type, double rtol, double atol,
                    double divtol, int maxit, int restart, const char* options_prefix, poro_ksp** out);
/* Solver.solve -> KSP.solve(b, x) (lib/Solver.py:148-152); zero initial guess. */
int poro_ksp_solve(poro_ksp* ksp, const double* b_dev, double* x_dev, int* its, int* reason, double* rnorm);
/* same with HOST vectors: copies b in and x out inside the call (the end-to-end path) */
int poro_ksp_solve_host(poro_ksp* ksp, const double* b_host, double* x_host, int* its, int* reason, double* rnorm);
int poro_ksp_residual_history(poro_ksp* ksp, double* out, int cap, int* n);
/* KSP.setInitialGuessNonzero -- commented out at lib/Solver.py:94; the time loop (lib/AbstractPhysics.py:73-81,
 * lib/Poromechanics.py:70-98) re-solves with the same operators every step, so the previous step's solution in x is a
 * useful start.  Also `-<prefix>ksp_initial_guess_nonzero`.  Convergence is then measured against ||b|| (PETSc default). */
int poro_ksp_set_initial_guess_nonzero(poro_ksp* ksp, int flag);
/* per-field infinity norms (abs_s, abs_f, abs_p per iteration) of the true residual recorded by the
 * `-<prefix>ksp_monitor_fields` monitor / `-<prefix>ksp_convergence_test_fields` test: the `converged` callback the
 * reference defines at lib/Solver.py:8-51 and never installs.  `-<prefix>ksp_converged_reason` prints PETSc's line. */
int poro_ksp_field_history(poro_ksp* ksp, double* out, int cap, int* n);
int poro_ksp_destroy(poro_ksp* ksp);

/* ---- AAR ------------------------------------------------------------------------------
 * AAR.solve (lib/AAR.py:46-128).  The window (F, X) lives in the handle and is never reset
 * between solves, like the reference's (lib/AAR.py:20-22). */
typedef struct poro_aar poro_aar;
int poro_aar_create(poro_ctx* ctx, poro_mat* A, poro_pc* pc, int order, int p, double omega, double beta,
                    double atol, double rtol, int maxit, int monitor, poro_aar** out);
int poro_aar_solve(poro_aar* aar, const double* b_dev, double* x_dev, int* its);
int poro_aar_residual_history(poro_aar* aar, double* out, int cap, int* n);
int poro_aar_destroy(poro_aar* aar);

/* ---- micro-benchmark / introspection entry points ----------------------------------------- */
/* block names: "A" (whole permuted operator), "ss","sf","sp","fs","ff","fp","ps","pf","pp" of P */
int poro_pc_block_info(poro_pc* pc, const char* name, int64_t* nrows, int64_t* ncols, int64_t* nnz);
/* algorithmic bytes of one product y = B x with a block in the format it is launched in (0 CSR, 1 BSR, 2 diagonal BSR,
 * 4 stencil): 12 nnz + 4 (nrows+1) + 8 nrows + 8 ncols, or (8 BS^2 + 4) nnzb + 4 (nbrows+1) + 8 nrows + 8 ncols, or for a
 * generated block applied from its class tables 8 ncols + table bytes + Dirichlet flags (1 B per row) + 8 nrows */
int poro_pc_block_bytes(poro_pc* pc, const char* name, int64_t* bytes, int* format);
/* one product with a block in the path its solvers use, on device vectors (tests of the product kernels):
 * mode 0 y = B x, 1 y = z - B x, 2 y = z + B x, 3 Chebyshev step (x = d_old; r -= B x; d_new = c1 x + c2 dinv.*r; xv += d_new),
 * 4 y = B x and *dot = x . y (dot: one device double).  Unused pointers may be null. */
int poro_pc_block_mult(poro_pc* pc, const char* name, int mode, const double* x, double* y, const double* z, double* r, double* d_new,
                       double* xv, const double* dinv, double c1, double c2, double* dot);
/* copy a block to host CSR arrays sized from poro_pc_block_info (tests: createSubMatrix parity) */
int poro_pc_block_copy(poro_pc* pc, const char* name, int64_t* rowptr, int32_t* col, double* val);
/* one application of the inner solver of a block: "s","f","p","fp","diff" (z = K \ r) */
int poro_pc_inner_solve(poro_pc* pc, const char* name, const double* r_dev, double* z_dev);
/* iterations / reason / residual norm of the last application of an inner solver ("s","f","p","fp","diff","fp0","fp1"):
 * what `ksp.getIterationNumber()` reports in the single-block drivers (solid.py:177-180, fluid-pressure.py:133-136) */
int poro_pc_inner_result(poro_pc* pc, const char* name, int* its, int* reason, double* rnorm);
/* AMG hierarchy of a block's inner PC: per level rows and nnz; returns number of levels */
int poro_pc_amg_info(poro_pc* pc, const char* name, int64_t* rows, int64_t* nnz, int cap, int* nlevels);
/* one level of a block's single-rank AMG hierarchy (tests of the set-up).  out[0..n) receives: rows, columns and nnz of
 * A_l, P_l, R_l and T_l (the tentative prolongator; zeros unless kept), block size, near-nullspace modes k, aggregates,
 * geometric level, coarsest level, coarsest level solved directly, set-up data kept, and the row chunks of the SpGEMMs
 * A T, A P and R (A P); *lmax receives the Chebyshev bound 1.1 lambda_max(D^-1 A_l).  `-poro_amg_keep_setup 1` before the
 * set-up keeps per level the aggregates, the near-nullspace as the level used it (after the Dirichlet zeroing; the
 * coarsest level's as received) and T_l.  Row-partitioned hierarchies and levels out of range are refused. */
int poro_pc_amg_level_info(poro_pc* pc, const char* name, int level, int64_t* out, int n, double* lmax);
/* copy of one item of that level to host arrays sized from poro_pc_amg_level_info: "A" "P" "R" "T" as CSR; "agg" (int32,
 * in col); "B" (n x k row-major), "dinv" (n) and "inv" (the coarsest dense inverse, n x n row-major) in val.  Refused
 * with the reason: set-up data not kept (agg B T), a geometric level (P R T agg), the coarsest level (P R T agg), no
 * direct coarsest solve (inv), a row-partitioned hierarchy, a level out of range. */
int poro_pc_amg_level_copy(poro_pc* pc, const char* name, int level, const char* what, int64_t* rowptr, int32_t* col, double* val);
/* sparse LU of a block's inner PC ("s","f","p","fp","diff"; -<prefix>pc_factor_mat_solver_type poro above
 * -poro_dense_lu_limit rows).  out[0..n) receives, in this order: rows, nnz(L) (strictly lower), nnz(U) (with the
 * diagonal), explicit zeros stored by supernode amalgamation, supernodes, levels of the supernodal tree, rows of the
 * largest front, perturbed pivots, device bytes held after set-up, flops of the numeric factorisation, its device time
 * in microseconds, algorithmic bytes of one application without refinement.  Fails for a block that is not a sparse LU. */
int poro_pc_factor_info(poro_pc* pc, const char* name, int64_t* out, int n);
/* geometric multigrid of a block's inner PC (`-<prefix>pc_type mg`).  out[0..n) receives the number G of geometric levels
 * (the finest included), then per geometric level N, rows and the launch format of its operator (4 = stencil), then the
 * number of algebraic levels below.  Fails for an inner PC that is not `mg`. */
int poro_pc_mg_info(poro_pc* pc, const char* name, int64_t* out, int n);
/* one geometric transfer between level `level` and `level + 1` on device vectors: dir 0 prolongation (x coarse, y fine;
 * mode 0 y = P~ x, mode 1 y += P~ x), dir 1 restriction (x fine, y coarse, y = P~^T x, mode 0) */
int poro_pc_mg_transfer(poro_pc* pc, const char* name, int level, int dir, int mode, const double* x_dev, double* y_dev);
/* algorithmic bytes of the transfers of `level`: out[0] prolongation (set), out[1] prolongation (add), out[2] restriction */
int poro_pc_mg_bytes(poro_pc* pc, const char* name, int level, int64_t* out);
/* live profile of the outer operator product (the dominant SpMV): CUDA events recorded on the
 * launching stream around every y = A x inside poro_ksp_solve.  enable = 1 resets and starts,
 * 0 stops, -1 only reads.  op_bytes = algorithmic bytes of one product
 * (12 nnz + 4 (nrows+1) + 8 nrows + 8 ncols). */
int poro_ksp_profile(poro_ksp* ksp, int enable, double* op_ms, int64_t* op_calls, int64_t* op_bytes);
/* algorithmic bytes of every launch of the outer operator product: [CSR remainder, node-blocked part 0, 1, ...]
 * (format flag 0 CSR, 1 BSR, 2 diagonal-block BSR); matches phase-profile slots 32, 33, ... */
int poro_ksp_parts_info(poro_ksp* ksp, int64_t* bytes, int* format, int cap, int* n);
/* phase profile (CUDA events on the launching stream): slots 0 outer operator, 1 preconditioner apply,
 * 2 solid solve, 3 fp split 0, 4 fp split 1, 5 orthogonalisation, 6 fp coupling product,
 * 8+l / 16+l / 24+l AMG level l (inclusive) of the s / f / p hierarchies, 32.. the launches of the outer operator,
 * 37 the level-0 Chebyshev-step launch of the solid hierarchy.  enable as in poro_ksp_profile. */
int poro_profile(poro_ctx* ctx, int enable, double* ms, int64_t* calls, int n);
/* operator y = A x in the solver's internal (field-major) ordering incl. halo exchange */
int poro_ksp_mult(poro_ksp* ksp, const double* x_dev, double* y_dev);

#ifdef __cplusplus
}
#endif
#endif
