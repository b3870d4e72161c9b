"""Geometric multigrid on row-partitioned generated slabs (tests/mg_multi_worker.py under torch.distributed.run; the
multi-rank tests skip on a box with fewer GPUs, which verifies nothing): the distributed transfers against the global
masked prolongation, one solid-block V-cycle, solid CG and a whole petsc-options-mg solve against one rank, the refusals.
The single-rank references are computed here, on one GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
MG_OPTIONS = open(os.path.join(ROOT, "options", "petsc-options-mg")).read()
# CG + mg on the solid block; the coarsest geometric level (N = 4) is solved densely on every rank count, so one and two
# ranks run the same hierarchy
SOLID_MG = {Ns: ("-s_ksp_type cg\n-s_ksp_rtol 1e-8\n-s_ksp_atol 0.0\n-s_ksp_max_it 500\n-s_pc_type mg\n-s_pc_mg_levels %d\n"
                 "-s_pc_amg_coarse_size 6000\n-poro_amg_dense_limit 8192\n" % lev) for Ns, lev in ((16, 3), (32, 4))}


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _run(nproc, port, env):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mg_multi_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=ROOT, env=dict(os.environ, **env))
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert "MG MULTI-GPU OK" in r.stdout


def _reference(gpu_ctx, path):
    """Single-rank references of the worker's checks 2-4 (npz at `path`); returns the preconditioner statistics."""
    from poro_b200.generator import generate_swelling3d
    from poro_b200.lib.backend import DeviceVector
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    from poro_b200.lib.Solver import Solver
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    from _single_block import build as build_block
    gpu_ctx.clear_options()
    load_petsc_options(gpu_ctx, MG_OPTIONS, is_text=True)
    g = generate_swelling3d(gpu_ctx, 16, "diagonal", mg_levels=3)
    par = dict(g.par)
    par.update({"solver rtol": 1e-8, "solver atol": 0.0, "solver maxiter": 300})
    pc = Preconditioner(g.index_set(), g.A, g.P, g.P_diff, par, g.bcs_sub_pressure).get_pc()
    ns = g.layout.n_field[0]
    r_s = np.random.default_rng(11).standard_normal(ns)
    dr, dz = DeviceVector(r_s, ctx=gpu_ctx), DeviceVector(n=ns, ctx=gpu_ctx)
    pc.getPythonContext().inner_solve("s", dr, dz)
    gpu_ctx.sync()
    z_s = dz.numpy()
    db, dx = DeviceVector(g.b, ctx=gpu_ctx), DeviceVector(n=len(g.b), ctx=gpu_ctx)
    s = Solver(g.A, db, pc, par, g.index_set())
    s.create_solver(g.A, db, pc)
    s.solve(db, dx)
    assert s.solver.reason > 0
    solid = {}
    for Ns in (16, 32):
        _, cc, dbs, dxs, _, _, keep = build_block("s", Ns, ctx=gpu_ctx, options_text=SOLID_MG[Ns])
        cc.inner_solve("s", dbs, dxs)
        gpu_ctx.sync()
        its, reason, _ = cc.inner_result("s")
        assert reason > 0
        solid["solid_its_%d" % Ns] = its
        cc.destroy()
    np.savez(path, x=dx.numpy(), its=s.getIterationNumber(), r_s=r_s, z_s=z_s, **solid)
    return pc.getPythonContext().stats(), solid


def test_single_rank_references(gpu_ctx, tmp_path):
    """The references on one rank: the whole solve replays the preconditioner's CUDA graph, solid CG + mg converges."""
    stats, solid = _reference(gpu_ctx, tmp_path / "mg_ref.npz")
    assert stats["graph_replays"] > 0, stats
    assert all(0 < its < 100 for its in solid.values()), solid


@pytest.mark.skipif(_ngpus() < 2, reason="needs 2 GPUs")
def test_two_rank_mg_matches_single(gpu_ctx, tmp_path):
    """2 ranks at N = 16: the slabs start at fine P2 planes 17 (level 0), 9 (level 1) and 5 (level 2), all odd, so the
    restriction reads 3 planes above rank 0 but never 3 below a slab; test_three_rank_transfers covers that case."""
    ref = tmp_path / "mg_ref.npz"
    _reference(gpu_ctx, ref)
    _run(2, 29623, {"PORO_MG_REF": str(ref)})


@pytest.mark.skipif(_ngpus() < 3, reason="needs 3 GPUs")
def test_three_rank_transfers():
    """3 ranks at N = 8 (2 levels): rank 2 starts at fine P2 plane 12, a multiple of 4, where the restriction reads 3 fine
    planes below the slab through the transfer halo."""
    _run(3, 29624, {"PORO_MG_N": "8", "PORO_MG_LEVELS": "2", "PORO_MG_TRANSFERS_ONLY": "1"})
