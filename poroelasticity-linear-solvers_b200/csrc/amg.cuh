// amg.cuh -- smoothed-aggregation AMG hierarchy (device set-up + V-cycle).
#pragma once
#include "common.cuh"
#include "mg.cuh"
#include <functional>

namespace poro {

struct AmgParams {
    double theta = 0.08;
    int max_levels = 10;
    int coarse_size = 400;
    int cheby_degree = 2;
    double cheby_ratio = 10.0;
    int power_its = 15;
    int post_smooth = 1;        // 0: V(nu,0) cycle (non-symmetric: only under GMRES/FGMRES)
    bool smoother_only = false; // `-*_pc_type chebyshev`: one level, no coarse solve of any kind
    // `-*_pc_type mg`: levels 0 .. mg_levels - 1 are the generated block and its attached coarse levels (geometric transfer,
    // mg.cuh); the last of them is level 0 of the SA-AMG below, and max_levels counts from there
    int mg_levels = 0;
};

struct AmgLevel {
    Csr A, P, R;
    DBuf<double> dinv;
    double lmax = 1.0;
    int bs = 1;
    int n_agg = 0;
    // work vectors; in a distributed hierarchy x, r, d0, d1 have room for [owned | ghost] so that the halo lands in place
    DBuf<double> x, b, r, d0, d1;
    // distributed hierarchy: halo plan of this level's operator (level 0 borrows the plan of the block operator)
    DistPlan* plan = nullptr;
    std::unique_ptr<DistPlan> owned_plan;
    bool replicated = false;        // this level and everything below is gathered on every rank and cycled redundantly (Amg::tail)
    DBuf<double> ext;               // staging for vectors that are not stored extended (the caller's x on level 0)
    std::unique_ptr<MgTransfer> mg; // geometric level: the transfer to the next level replaces P and R
    int k = 0;                      // near-nullspace modes of this level
    int spgemm_chunks[3] = {0, 0, 0};   // row chunks of A T, A P and R (A P)
    // `-poro_amg_keep_setup 1` (tests of the set-up): the aggregates (-1 = not aggregated), the near-nullspace as this level
    // used it (after the Dirichlet zeroing; the coarsest level's as received) and the tentative prolongator
    bool kept = false;
    DBuf<int> keep_agg;
    DBuf<double> keep_B;
    Csr keep_T;
};

struct Amg {
    Ctx* ctx = nullptr;
    AmgParams par;
    std::vector<std::unique_ptr<AmgLevel>> levels;
    const Csr* A0 = nullptr;        // finest operator is borrowed
    DBuf<double> coarse_inv;
    bool coarse_direct = false;
    // row-partitioned runs (plan0 given): every level operator is distributed (local rows x [owned | ghost] columns),
    // aggregates stay inside a rank, prolongator smoothing and the Galerkin product use the distributed operator
    // (distamg.cu); the coarsest operator is gathered on every rank.  Without a plan the hierarchy is rank-local.
    bool dist = false;
    // small distributed levels are latency-bound (6 halo exchanges per level visit): below `-poro_amg_replicate_below` global
    // rows a level is gathered ONCE at set-up, the rest of the hierarchy is built and cycled redundantly on every rank, and a
    // cycle pays one all-gather of the level's right-hand side instead (oracle/distamg.py: replicate_below).  OFF by default:
    // measured on 8 GPUs (N = 68) the redundant 20k-row solid level costs more than its six exchanges (259 vs 253 ms per solve),
    // on 2 GPUs it gains 1.5 % (128.1 vs 130.3 ms); profiles/r2_scaling.md
    std::unique_ptr<Amg> tail;
    Csr tail_A;
    DBuf<double> tail_b, tail_x;
    int64_t coarse_n_global = 0;
    DBuf<double> coarse_full;       // gathered right-hand side of the coarsest level
    int prof_base = -1;             // phase-profile slot of level 0 (-1: not profiled)

    // B: device n x k row-major near-nullspace (may be null -> one constant per component)
    void setup(Ctx& c, const Csr& A, int bs, const double* B_dev, int k, const AmgParams& p, DistPlan* plan0 = nullptr);
    void apply(const double* b, double* x);     // x = V-cycle(b), zero initial guess
    const Csr& op(int l) const { return l == 0 ? *A0 : levels[l]->A; }
    double complexity() const;

    const double* ext(int l, const double* v);   // [owned | ghost] view of a level-l vector, ghosts refreshed (collective)
    int64_t rows_global(int l) const { return dist ? levels[l]->plan->offsets.back() : op(l).nrows; }
    void cheby(int l, const double* b, double* x, bool zero_guess);
    void cycle(int l, const double* b, double* x);
};

}  // namespace poro
