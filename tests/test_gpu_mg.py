"""Geometric multigrid (`-<prefix>pc_type mg`) on generated structured-mesh blocks: the matrix-free transfer kernels
(csrc/mg.cu) against the scipy P~ of hostfem/mg.py, the level structure, one application against the CPU twin
(hostfem.mg.GeometricMG), whole solves with options/petsc-options-mg, and the set-up refusals."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MG_OPTIONS = open(os.path.join(ROOT, "options", "petsc-options-mg")).read()
THREE_WAY_MG = """
-global_ksp_type gmres
-global_ksp_pc_side right
-s_ksp_type preonly
-s_pc_type mg
-f_ksp_type preonly
-f_pc_type mg
-p_ksp_type preonly
-p_pc_type mg
-diff_ksp_type preonly
-diff_pc_type mg
"""


def _generate(ctx, dim, N, pc_type, mg_levels):
    from poro_b200.generator import generate_swelling2d, generate_swelling3d
    return (generate_swelling2d if dim == 2 else generate_swelling3d)(ctx, N, pc_type, mg_levels=mg_levels)


def _setup(ctx, dim, N, pc_type, options, mg_levels):
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    ctx.clear_options()
    load_petsc_options(ctx, options, is_text=True)
    g = _generate(ctx, dim, N, pc_type, mg_levels)
    par = dict(g.par)
    par.update({"solver rtol": 1e-8, "solver atol": 0.0, "solver maxiter": 300})
    pc = Preconditioner(g.index_set(), g.A, g.P, g.P_diff, par, g.bcs_sub_pressure).get_pc()
    return g, pc, par


def _solve(ctx, g, pc, par):
    from poro_b200.lib.backend import DeviceVector
    from poro_b200.lib.Solver import Solver
    db, dx = DeviceVector(g.b, ctx=ctx), DeviceVector(n=len(g.b), ctx=ctx)
    s = Solver(g.A, db, pc, par, g.index_set())
    s.create_solver(g.A, db, pc)
    s.solve(db, dx)
    return s.solver.reason, s.getIterationNumber(), dx.numpy()


def _true_res(g, x):
    A = g.A.to_scipy()
    return np.linalg.norm(g.b - A @ x) / np.linalg.norm(g.b)


def _flags(dim, N):
    """Dirichlet flags per dof of the s, f, p (P, no pressure BCs) and diff (P_diff) blocks at N."""
    from hostfem.stencil import swelling_generator
    gen = swelling_generator(dim, N)[0]
    return {"s": gen.bc_s.ravel(), "f": gen.bc_f.ravel(), "p": None, "diff": gen.bc_p}


@pytest.mark.gpu
@pytest.mark.parametrize("N", [2, 4, 8, 16])
@pytest.mark.parametrize("dim", [2, 3])
def test_transfer_kernels_match_scipy(gpu_ctx, dim, N):
    import torch
    from hostfem.mg import masked_prolongation
    g, pc, par = _setup(gpu_ctx, dim, N, "diagonal 3-way", THREE_WAY_MG, 2)
    pcc = pc.getPythonContext()
    ff, fc = _flags(dim, N), _flags(dim, N // 2)
    rng = np.random.default_rng(N)
    for name in ("s", "f", "p", "diff"):
        kind, bs = (2, dim) if name in ("s", "f") else (1, 1)
        P = masked_prolongation(dim, N // 2, kind, bs, ff[name], fc[name])
        absP = abs(P)
        x = rng.standard_normal(P.shape[1])
        r = rng.standard_normal(P.shape[0])
        y0 = rng.standard_normal(P.shape[0])
        cases = [(0, 0, x, np.full(P.shape[0], np.nan), P @ x, absP @ np.abs(x)),
                 (0, 1, x, y0, y0 + P @ x, np.abs(y0) + absP @ np.abs(x)),
                 (1, 0, r, np.full(P.shape[1], np.nan), P.T @ r, absP.T @ np.abs(r))]
        for direction, mode, xin, yinit, want, scale in cases:
            outs = []
            for _ in range(2):
                xt = torch.tensor(xin, device="cuda")
                yt = torch.tensor(yinit, device="cuda")
                pcc.mg_transfer(name, 0, direction, mode, xt, yt)
                torch.cuda.synchronize()
                outs.append(yt.cpu().numpy())
            assert np.array_equal(outs[0], outs[1]), (name, direction, mode)
            y = outs[0]
            assert np.isfinite(y).all(), (name, direction, mode)
            bad = np.abs(y - want) > 1e-14 * scale + 1e-300
            assert not bad.any(), (name, direction, mode, int(bad.sum()))
        pb, pa, rb = pcc.mg_bytes(name, 0)
        assert pa - pb == 8 * P.shape[0] and rb > 0
    # the 3-way splitting with mg on every block converges
    reason, its, x = _solve(gpu_ctx, g, pc, par)
    assert reason > 0 and _true_res(g, x) <= 1e-7, (its, _true_res(g, x))


@pytest.mark.gpu
def test_level_structure(gpu_ctx):
    g, pc, par = _setup(gpu_ctx, 3, 16, "diagonal", MG_OPTIONS + "-s_pc_mg_levels 3\n", 4)
    levels, alg = pc.getPythonContext().mg_info("s")
    assert [(n, f) for n, _, f in levels] == [(16, 4), (8, 4), (4, 4)]
    assert [r for _, r, _ in levels] == [3 * (2 * n + 1) ** 3 for n in (16, 8, 4)]
    amg = pc.getPythonContext().amg_info("s")
    assert len(amg) == 3 + alg and [r for r, _ in amg[:3]] == [r for _, r, _ in levels]
    levels, alg = pc.getPythonContext().mg_info("fp0")          # all attached levels by default
    assert [n for n, _, _ in levels] == [16, 8, 4, 2]


def _twin(g, name, N, dim, options):
    """CPU twin of the inner PC `name` ("s" or "fp0": the velocity block) of a generated system."""
    from hostfem.mg import GeometricMG, injection, masked_prolongation
    from hostfem.stencil import swelling_generator
    from oracle.amg import rigid_body_modes
    blocks, flags = [], []
    n = N
    while True:
        gen, par, loads = swelling_generator(dim, n)
        s = gen.system("diagonal", par["t0"] + par["dt"], **loads)
        sl = slice(0, s.ns) if name == "s" else slice(s.ns, s.ns + s.nf)
        blocks.append(s.P[sl, sl].tocsr())
        flags.append((gen.bc_s if name == "s" else gen.bc_f).ravel())
        if n % 2:
            break
        n //= 2
    P = [masked_prolongation(dim, N >> (l + 1), 2, dim, flags[l], flags[l + 1]) for l in range(len(blocks) - 1)]
    inj = [injection(dim, N >> (l + 1), 2) for l in range(len(blocks) - 1)]
    B = rigid_body_modes(np.asarray(g.index_set().coords_s), dim)
    return GeometricMG(blocks, P, inj, bs=dim, B=B, theta=0.04, coarse_size=6000, dense_limit=8192), blocks[0]


@pytest.mark.gpu
@pytest.mark.parametrize("dim,N", [(3, 8), (2, 16)])
def test_one_application_matches_cpu_twin(gpu_ctx, dim, N):
    import torch
    mg_levels = 1
    while N % (1 << mg_levels) == 0:
        mg_levels += 1
    g, pc, par = _setup(gpu_ctx, dim, N, "diagonal", MG_OPTIONS, mg_levels)
    pcc = pc.getPythonContext()
    for name in ("s", "fp0"):
        twin, B0 = _twin(g, name, N, dim, MG_OPTIONS)
        r = np.random.default_rng(3).standard_normal(B0.shape[0])
        rt = torch.tensor(r, device="cuda")
        zt = torch.zeros_like(rt)
        pcc.inner_solve(name, rt, zt)
        torch.cuda.synchronize()
        z = zt.cpu().numpy()
        want = twin(r)
        assert np.abs(z - want).max() <= 1e-10 * np.abs(want).max(), name


@pytest.mark.gpu
def test_solid_block_cg_is_mesh_independent(gpu_ctx):
    import sys
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    from _single_block import DEFAULTS, build
    its = {}
    for N in (8, 32):
        opts = DEFAULTS["s"].replace("-s_pc_type hypre", "-s_pc_type mg") + "-s_pc_amg_coarse_size 6000\n-poro_amg_dense_limit 8192\n"
        ctx, cc, db, dx, host, rhs, keep = build("s", N, ctx=gpu_ctx, options_text=opts)
        cc.inner_solve("s", db, dx)
        ctx.sync()
        n_its, reason, rnorm = cc.inner_result("s")
        assert reason > 0, (N, n_its, reason)
        its[N] = n_its
    assert its[32] <= its[8] + 3, its


@pytest.mark.gpu
@pytest.mark.parametrize("dim,N", [(3, 16), (2, 32), (3, 34)])
def test_whole_solve_with_mg_options(gpu_ctx, dim, N):
    import bench
    from poro_b200.lib.Parser import load_petsc_options
    mg_levels = 1
    while N % (1 << mg_levels) == 0:
        mg_levels += 1
    g, pc, par = _setup(gpu_ctx, dim, N, "diagonal", MG_OPTIONS, mg_levels)
    if N == 34:
        levels, alg = pc.getPythonContext().mg_info("s")
        assert [n for n, _, _ in levels] == [34, 17] and alg >= 1
    reason, its, x = _solve(gpu_ctx, g, pc, par)
    assert reason > 0 and _true_res(g, x) <= 1e-8, (its, _true_res(g, x))
    reason2, its2, x2 = _solve(gpu_ctx, g, pc, par)
    assert its2 == its and np.array_equal(x, x2)
    # eager application (-poro_pc_timing switches the CUDA graph off) gives the same solve
    gpu_ctx.set_option("-poro_pc_timing")
    from poro_b200.lib.Preconditioner import Preconditioner
    pce = Preconditioner(g.index_set(), g.A, g.P, g.P_diff, par, g.bcs_sub_pressure).get_pc()
    reason_e, its_e, xe = _solve(gpu_ctx, g, pce, par)
    assert its_e == its and np.abs(xe - x).max() <= 1e-12 * np.abs(x).max()
    # to 1e-12 the solution is the benchmarked set's
    tight = dict(par, **{"solver rtol": 1e-12})
    gpu_ctx.clear_options()
    load_petsc_options(gpu_ctx, MG_OPTIONS, is_text=True)
    pcm = Preconditioner(g.index_set(), g.A, g.P, g.P_diff, tight, g.bcs_sub_pressure).get_pc()
    _, _, xm = _solve(gpu_ctx, g, pcm, tight)
    gpu_ctx.clear_options()
    load_petsc_options(gpu_ctx, bench.BENCH_OPTIONS, is_text=True)
    pcb = Preconditioner(g.index_set(), g.A, g.P, g.P_diff, tight, g.bcs_sub_pressure).get_pc()
    _, _, xb = _solve(gpu_ctx, g, pcb, tight)
    assert np.abs(xm - xb).max() <= 1e-8 * np.abs(xb).max()


def _expect_refusal(fn, *needles):
    with pytest.raises(Exception) as e:
        fn()
    msg = str(e.value)
    for s in needles:
        assert s in msg, msg


@pytest.mark.gpu
def test_refusals(gpu_ctx):
    from poro_b200 import _capi
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    from poro_b200.lib.backend import DeviceMatrix

    def setup(options, mg_levels=2, upload=False):
        gpu_ctx.clear_options()
        load_petsc_options(gpu_ctx, options, is_text=True)
        g = _generate(gpu_ctx, 3, 4, "diagonal", mg_levels)
        A, P = (DeviceMatrix(g.A.to_scipy(), ctx=gpu_ctx), DeviceMatrix(g.P.to_scipy(), ctx=gpu_ctx)) if upload else (g.A, g.P)
        return Preconditioner(g.index_set(), A, P, None, dict(g.par), g.bcs_sub_pressure).get_pc()

    _expect_refusal(lambda: setup(MG_OPTIONS, upload=True), "-s_pc_type mg", "descriptor")
    _expect_refusal(lambda: setup(MG_OPTIONS, mg_levels=1), "-s_pc_type mg", "no coarse levels")
    _expect_refusal(lambda: setup(MG_OPTIONS.replace("-fp_fieldsplit_1_pc_type hypre", "-fp_fieldsplit_1_pc_type mg")),
                    "-fp_fieldsplit_1_pc_type mg", "descriptor")
    from poro_b200.generator import WholeLayout, _swelling_operators
    A4, P4, _, _, _, _ = _swelling_operators(gpu_ctx, 3, 4, "diagonal", None, WholeLayout(3, 4))
    A3, _, _, _, _, _ = _swelling_operators(gpu_ctx, 3, 3, "diagonal", None, WholeLayout(3, 3))
    A2, P2, _, _, _, _ = _swelling_operators(gpu_ctx, 3, 2, "diagonal", None, WholeLayout(3, 2))
    A2d, _, _, _, _, _ = _swelling_operators(gpu_ctx, 2, 2, "diagonal", None, WholeLayout(2, 2))
    lib = gpu_ctx.lib
    _expect_refusal(lambda: _capi.check(lib.poro_mat_set_coarse(A4.handle, A3.handle)), "N_fine must be 2 N_coarse")
    _expect_refusal(lambda: _capi.check(lib.poro_mat_set_coarse(A4.handle, A2d.handle)), "dim differs")
    _expect_refusal(lambda: _capi.check(lib.poro_mat_set_coarse(A4.handle, P2.handle)), "present tables differ")
    _capi.check(lib.poro_mat_set_coarse(A4.handle, A2.handle))
