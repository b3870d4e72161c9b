"""GPU tests of the device ILU(0) (`-<prefix>pc_type ilu`, csrc/ilu.cu) and of PETSc's additive / multiplicative fieldsplit on
the fp block, against the numpy twins of tests/ilu_twin.py: one application per block, the split applications, whole solves
with options/petsc-options-fieldsplit, CUDA-graph replay, the refusals, the unchanged schur default, and block Jacobi on two
ranks (tests/ilu_multi_worker.py, skipped with fewer GPUs)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import AMG_OPTIONS, gpu_solve, rel
from ilu_twin import ILU0, FieldSplit, level_sets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
FIELDSPLIT_OPTIONS = open(os.path.join(ROOT, "options", "petsc-options-fieldsplit")).read()
ILU_3WAY = "".join("-%s_ksp_type preonly\n-%s_pc_type ilu\n" % (p, p) for p in ("s", "f", "p", "diff"))
ILU_2WAY = "-s_ksp_type preonly\n-s_pc_type ilu\n-fp_ksp_type preonly\n-fp_pc_type ilu\n"


def _setup(sys_, par, options_text, pc_type):
    """The preconditioner alone (no solve); returns (PreconditionerCC, objects to keep alive)."""
    from poro_b200.lib.backend import DeviceMatrix, get_context
    from poro_b200.lib.IndexSet import IndexSet
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    ctx = get_context(0)
    ctx.clear_options()
    load_petsc_options(ctx, options_text, is_text=True)
    par = dict(par)
    par["pc type"] = pc_type
    imap = IndexSet(sys_.is_s, sys_.is_f, sys_.is_p, two_way="3-way" not in pc_type, block_dim=sys_.dim,
                    coords_s=sys_.coords_s, coords_p=sys_.coords_p)
    dA, dP = DeviceMatrix(sys_.A, ctx), DeviceMatrix(sys_.P, ctx)
    dPd = DeviceMatrix(sys_.P_diff, ctx) if sys_.P_diff is not None else None
    pc = Preconditioner(imap, dA, dP, dPd, par, sys_.bcs_sub_pressure).get_pc()
    return pc.getPythonContext(), (pc, dA, dP, dPd, imap)


def _apply(ctx, cc, name, r):
    from poro_b200.lib.backend import DeviceVector
    dr, dz = DeviceVector(r, ctx=ctx), DeviceVector(n=len(r), ctx=ctx)
    cc.inner_solve(name, dr, dz)
    ctx.sync()
    return dz.numpy()


@pytest.mark.parametrize("dim,N", [(2, 8), (2, 16), (3, 4), (3, 8)])
def test_ilu_application_matches_twin(gpu_ctx, dim, N):
    from oracle.problems import swelling
    rng = np.random.default_rng(17)
    for pc_type, opts, names in (("diagonal 3-way", ILU_3WAY, (("s", "ss"), ("f", "ff"), ("p", "pp"))),
                                 ("diagonal", ILU_2WAY, (("fp", "fpfp"),))):
        sys_, par = swelling(dim, N, pc_type)
        cc, keep = _setup(sys_, par, opts, pc_type)
        for name, blk in names:
            B = cc.block(blk)
            info = cc.ilu_info(name)
            twin = ILU0(B)
            assert info["rows"] == B.shape[0]
            assert info["nnz_l"] == twin.L.nnz and info["nnz_u"] == twin.U.nnz, (name, info)
            assert info["lower_levels"] == len(level_sets(B)[0]) - 1, (name, info)
            assert info["upper_levels"] == len(level_sets(B, True)[0]) - 1, (name, info)
            assert info["min_pivot"] == pytest.approx(np.abs(twin.d).min(), rel=1e-10)
            r = rng.standard_normal(B.shape[0])
            z1, z2 = _apply(gpu_ctx, cc, name, r), _apply(gpu_ctx, cc, name, r)
            assert np.array_equal(z1, z2), name                       # bitwise reproducible
            assert rel(z1, twin(r)) <= 1e-12, (dim, N, name, rel(z1, twin(r)))
        cc.destroy()


@pytest.mark.parametrize("typ", ["additive", "multiplicative"])
@pytest.mark.parametrize("sub", ["ilu", "lu"])
@pytest.mark.parametrize("order", ["pf", "fp"])
def test_fieldsplit_application_matches_twin(gpu_ctx, typ, sub, order):
    from oracle.blockpc import LU
    from oracle.problems import swelling
    sys_, par = swelling(2, 8, "diagonal")
    opts = ("-s_ksp_type preonly\n-s_pc_type jacobi\n-fp_ksp_type preonly\n-fp_pc_fieldsplit_type %s\n-fp_pc_fieldsplit_order %s\n"
            "-fp_fieldsplit_0_ksp_type preonly\n-fp_fieldsplit_0_pc_type %s\n-fp_fieldsplit_1_ksp_type preonly\n"
            "-fp_fieldsplit_1_pc_type %s\n" % (typ, order, sub, sub))
    cc, keep = _setup(sys_, par, opts, "diagonal")
    first = "p" if order == "pf" else "f"
    i0, i1 = (sys_.is_p, sys_.is_f) if first == "p" else (sys_.is_f, sys_.is_p)
    b0, b1 = ("pp", "ff") if first == "p" else ("ff", "pp")
    make = ILU0 if sub == "ilu" else LU
    fs = FieldSplit.from_blocks(typ, cc.block(b0), sys_.P[i1][:, i0], cc.block(b1), sys_.nf, make, make, first)
    tol = 1e-12 if sub == "ilu" else 1e-10
    rng = np.random.default_rng(23)
    x0, x1 = rng.standard_normal(len(i0)), rng.standard_normal(len(i1))
    assert rel(_apply(gpu_ctx, cc, "fp0", x0), fs.split0(x0)) <= tol
    assert rel(_apply(gpu_ctx, cc, "fp1", x1), fs.split1(x1)) <= tol
    x = rng.standard_normal(sys_.nf + sys_.np_)
    assert rel(_apply(gpu_ctx, cc, "fp", x), fs(x)) <= tol
    if sub == "ilu":
        assert cc.ilu_info("fp0")["rows"] == len(i0) and cc.ilu_info("fp1")["rows"] == len(i1)
    cc.destroy()


def _twin_solve(sys_, par):
    """The petsc-options-fieldsplit solve on the CPU: FGMRES, one SA-AMG V-cycle on s, GMRES + multiplicative (pf) ILU(0)."""
    from oracle.amg import SAAMG, rigid_body_modes
    from oracle.blockpc import BlockPC, krylov_solver
    from oracle.krylov import gmres
    B = rigid_body_modes(sys_.coords_s, sys_.dim)
    fs = lambda M: FieldSplit("multiplicative", M, sys_.nf, sys_.np_, ILU0, ILU0, "p")
    pc = BlockPC(sys_, {"s": krylov_solver("preonly", lambda M: SAAMG(M, sys_.dim, B)), "fp": krylov_solver("gmres", fs)})
    m = par["solver maxiter"]
    return gmres(lambda v: sys_.A @ v, sys_.b, pc, rtol=par["solver rtol"], atol=par["solver atol"], dtol=1e20, max_it=m, restart=m,
                 flexible=True)


@pytest.mark.parametrize("dim,N", [(2, 16), (3, 8)])
def test_fieldsplit_solve_matches_twin(gpu_ctx, dim, N):
    from oracle.problems import swelling
    sys_, par = swelling(dim, N, "diagonal")
    g = gpu_solve(sys_, par, FIELDSPLIT_OPTIONS)
    ro = _twin_solve(sys_, par)
    assert g["reason"] > 0 and ro.reason > 0, (g["reason"], ro.reason)
    assert abs(g["its"] - ro.its) <= 1, (g["its"], ro.its)
    nb = np.linalg.norm(sys_.b)
    assert np.linalg.norm(sys_.b - sys_.A @ g["x"]) <= max(par["solver rtol"] * nb, par["solver atol"])
    assert g["stats"]["its_fp_split0"] > 0 and g["stats"]["graph_replays"] == 0     # fp GMRES: not a fixed launch sequence


@pytest.mark.parametrize("dim,N", [(2, 16), (3, 8)])
def test_fieldsplit_graph_bitwise(gpu_ctx, dim, N):
    """With every inner solve preonly the application is captured and replayed; the replays give the eager bits."""
    from oracle.problems import swelling
    sys_, par = swelling(dim, N, "diagonal")
    opts = FIELDSPLIT_OPTIONS.replace("-fp_ksp_type gmres", "-fp_ksp_type preonly").replace("fgmres", "gmres") + "-global_ksp_pc_side right\n"
    over = {"solver maxiter": 12}
    g1 = gpu_solve(sys_, par, opts, overrides=over)
    g0 = gpu_solve(sys_, par, opts + "-poro_pc_graph 0\n", overrides=over)
    assert g1["stats"]["graph_replays"] > 0 and g0["stats"]["graph_replays"] == 0
    assert np.array_equal(g1["x"], g0["x"]) and g1["its"] == g0["its"]


@pytest.mark.parametrize("extra,match", [
    ("-s_ksp_type preonly\n-s_pc_type ilu\n-s_pc_factor_levels 1\n", "s_pc_factor_levels"),
    ("-s_ksp_type preonly\n-s_pc_type ilu\n-s_pc_factor_mat_ordering_type rcm\n", "natural ordering"),
    ("-s_ksp_type preonly\n-s_pc_type ilu\n-s_pc_factor_shift_type nonzero\n", "shift"),
    ("-fp_pc_fieldsplit_type symmetric_multiplicative\n", "symmetric_multiplicative"),
    ("-s_ksp_type preonly\n-s_pc_type ilu\n-s_pc_factor_zeropivot 1e300\n", r"-s_pc_type ilu: zero pivot in row 0 "),
    ("-fp_pc_fieldsplit_type additive\n-fp_fieldsplit_1_pc_type ilu\n-fp_fieldsplit_1_pc_factor_zeropivot 1e300\n",
     r"-fp_fieldsplit_1_pc_type ilu: zero pivot in row 0 "),
])
def test_refusals(gpu_ctx, extra, match):
    from oracle.problems import swelling
    from poro_b200._capi import PoroError
    sys_, par = swelling(2, 4, "diagonal")
    with pytest.raises(PoroError, match=match):
        _setup(sys_, par, "-fp_ksp_type preonly\n" + extra, "diagonal")


def test_default_fieldsplit_is_schur(gpu_ctx):
    from oracle.problems import swelling
    sys_, par = swelling(2, 8, "diagonal")
    implicit = AMG_OPTIONS.replace("-fp_pc_fieldsplit_type schur\n", "")
    assert implicit != AMG_OPTIONS
    g1, g0 = gpu_solve(sys_, par, AMG_OPTIONS), gpu_solve(sys_, par, implicit)
    assert np.array_equal(g1["x"], g0["x"]) and g1["its"] == g0["its"]


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_ngpus() < 2, reason="needs 2 GPUs")
def test_two_rank_bjacobi():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(ROOT, "tests", "ilu_multi_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "ILU MULTI-GPU OK" in r.stdout
