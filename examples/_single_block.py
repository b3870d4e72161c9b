"""Shared logic of the reference's single-block drivers on the GPU solve phase (SURVEY 8 f3).

    solid.py           (reference solid.py:111-180)          KSP with prefix `s_`  on the solid block
                       a_s = rho_s/dt^2 phi_s (u,v) + (hooke(eps u), eps v) + phi^2/(kf dt) (u,v)      = A_ss
    fluid-pressure.py  (reference fluid-pressure.py:85-136)  KSP with prefix `fp_` + PCFIELDSPLIT(f, p) on
                       a_f + a_p                                                                        = A[fp, fp]
Both forms are exactly the (s,s) and (fp,fp) blocks of the three-field operator A (lib/Assembler.py:80-97) with the boundary
conditions of swelling-3d.py, so the drivers build the 3D swelling system (ks = 1e6 as in the two scripts), hand A to the
library as the preconditioner matrix and apply the inner solver of the block: `poro_pc_inner_solve(pc, "s" | "fp", b, x)`.
Options come from --petsc-options like in the reference; without a file the defaults of options/petsc-options-b200 apply.
"""
from __future__ import annotations

import os
import sys
from time import perf_counter as time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

DEFAULTS = {
    "s": "-s_ksp_type cg\n-s_ksp_rtol 1e-8\n-s_ksp_atol 0.0\n-s_ksp_max_it 500\n-s_pc_type hypre\n",
    "fp": ("-fp_ksp_type gmres\n-fp_ksp_pc_side right\n-fp_ksp_rtol 1e-8\n-fp_ksp_atol 0.0\n-fp_ksp_max_it 500\n-fp_ksp_gmres_restart 500\n"
           "-fp_pc_fieldsplit_type schur\n-fp_pc_fieldsplit_schur_fact_type lower\n-fp_pc_fieldsplit_schur_precondition selfp\n"
           "-fp_pc_fieldsplit_order fp\n-fp_fieldsplit_0_ksp_type preonly\n-fp_fieldsplit_0_pc_type hypre\n"
           "-fp_fieldsplit_1_ksp_type preonly\n-fp_fieldsplit_1_pc_type hypre\n"),
}


def build(block: str, N: int, overrides=None, assemble="device", ctx=None, options_text=None):
    """Returns (ctx, preconditioner context, device rhs, device solution, host block, host rhs) for block 's' or 'fp'."""
    from poro_b200.lib.backend import DeviceMatrix, DeviceVector, get_context
    from poro_b200.lib.IndexSet import IndexSet
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    ctx = ctx or get_context()
    if options_text is not None:
        ctx.clear_options()
        load_petsc_options(ctx, options_text, is_text=True)
    ov = {"ks": 1e6}                                   # solid.py:50, fluid-pressure.py:44
    ov.update(overrides or {})
    host = None
    if assemble == "device":
        from poro_b200.generator import generate_swelling3d
        from poro_b200.generator import max_mg_levels
        # under torchrun every rank generates its z-slab (the process group is initialised by `run`)
        rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
        # `-<prefix>pc_type mg` on the block: attach every coarse level N and the slabs allow (halving while N stays even
        # and every rank keeps two P2 planes)
        prefixes = ("s_",) if block == "s" else ("fp_fieldsplit_0_",)
        mg_levels = 1
        if any(str(ctx.get_option("-" + p + "pc_type", "")) == "mg" for p in prefixes):
            mg_levels = max_mg_levels(N, world)
        g = generate_swelling3d(ctx, N, "diagonal", rank, world, overrides=ov, mg_levels=mg_levels,
                                init_dist=getattr(ctx, "nranks", 1) != world)
        A, b, imap, par, bcs_p = g.A, g.b, g.index_set(), g.par, g.bcs_sub_pressure
        ns, nf, npp = g.layout.n_field
    else:
        from hostfem.problems import swelling
        host, par = swelling(3, N, "diagonal", ov)
        A, b, bcs_p = DeviceMatrix(host.A, ctx), host.b, host.bcs_sub_pressure
        imap = IndexSet(host.is_s, host.is_f, host.is_p, two_way=True, block_dim=3, coords_s=host.coords_s, coords_p=host.coords_p)
        ns, nf, npp = host.ns, host.nf, host.np_
    par = dict(par)
    par.update({"pc type": "diagonal", "inner ksp type": "gmres", "inner pc type": "hypre"})
    pcw = Preconditioner(imap, A, A, None, par, bcs_p)       # P := A  =>  P_ss = A_ss, P_fpfp = A[fp, fp]
    cc = pcw.get_pc().getPythonContext()
    sl = slice(0, ns) if block == "s" else slice(ns, ns + nf + npp)
    rhs = np.ascontiguousarray(b[sl])
    db, dx = DeviceVector(rhs, ctx=ctx), DeviceVector(n=len(rhs), ctx=ctx)
    return ctx, cc, db, dx, host, rhs, (pcw, A, imap)


def run(block: str, default_N: int, argv=None):
    from poro_b200.lib.Parser import Parser, load_petsc_options
    from poro_b200.lib.Printing import parprint
    from poro_b200.lib.backend import get_context
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = get_context()
    load_petsc_options(ctx, DEFAULTS[block], is_text=True)
    parser = Parser(argv, ctx=ctx)                           # --petsc-options FILE overrides the defaults
    N = parser.options.N or default_N
    tt = time()
    ctx, cc, db, dx, host, rhs, keep = build(block, N, ctx=ctx)
    ctx.sync()
    parprint("Dofs = {}".format(len(rhs)))
    parprint("Assembled and set up in {}s".format(time() - tt))
    tt = time()
    cc.inner_solve(block, db, dx)
    ctx.sync()
    its, reason, rnorm = cc.inner_result(block)
    parprint("Solved in {} iterations in {}s".format(its, time() - tt))      # solid.py:180, fluid-pressure.py:136
    return dict(its=its, reason=reason, rnorm=rnorm, x=dx.numpy(), n=len(rhs))
