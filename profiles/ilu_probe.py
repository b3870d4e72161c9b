"""ILU(0) (`-<prefix>pc_type ilu`) and the reference's default fp block (options/petsc-options-fieldsplit) on swelling-3d, one GPU.

1. Per block (P_ss, P_ff, P_pp from the `diagonal 3-way` splitting, the whole fp block from `diagonal`) at N (default 34):
   the set-up time of the preconditioner that factors them (host clock around a set-up that ends in a device synchronise),
   rows, nnz(L) + nnz(U), lower / upper levels, and ms per application (CUDA events over `reps` applications after 3
   warm-up ones).
2. Whole solves, petsc-options-fieldsplit (as is, and with the sub-PCs' zero-pivot threshold at 0) against
   petsc-options-b200 at N = 16 and 34: a set-up refusal, or iterations, ms per solve (CUDA events
   around 2 solves after one warm-up solve) and the true relative residual.  The solver tolerances are the driver's.

The JSON object (with the card name and power limit read in the same run) is printed again after every result, so a run
cut short keeps what it measured; the last line is the complete one.

    python profiles/ilu_probe.py [N] [--reps R] [--solve-sizes 16,34]
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import bench
from poro_b200._capi import PoroError
from poro_b200.generator import generate_swelling3d
from poro_b200.lib.backend import DeviceVector, get_context
from poro_b200.lib.Parser import load_petsc_options
from poro_b200.lib.Preconditioner import Preconditioner
from poro_b200.lib.Solver import Solver

args = sys.argv[1:]
reps = int(args[args.index("--reps") + 1]) if "--reps" in args else 20
sizes = [int(v) for v in args[args.index("--solve-sizes") + 1].split(",")] if "--solve-sizes" in args else [16, 34]
pos = [a for i, a in enumerate(args) if a.isdigit() and (i == 0 or not args[i - 1].startswith("--"))]
N = int(pos[0]) if pos else 34
FIELDSPLIT = open(os.path.join(ROOT, "options", "petsc-options-fieldsplit")).read()
ILU_3WAY = "".join("-%s_ksp_type preonly\n-%s_pc_type ilu\n" % (p, p) for p in ("s", "f", "p", "diff"))
# the pressure pivots scale like h^3: at N >= 16 some fall below PETSc's absolute default threshold (2.22e-14)
ZP0 = "-fp_fieldsplit_0_pc_factor_zeropivot 0\n-fp_fieldsplit_1_pc_factor_zeropivot 0\n"
ILU_FP = "-s_ksp_type preonly\n-s_pc_type jacobi\n-fp_ksp_type preonly\n-fp_pc_type ilu\n"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0]


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


ctx = get_context(0)
out = {"card": card(), "N": N, "reps": reps, "blocks": {}, "solves": {}}
for pc_type, opts, names in (("diagonal 3-way", ILU_3WAY, (("P_ss", "s"), ("P_ff", "f"), ("P_pp", "p"))),
                             ("diagonal", ILU_FP, (("fp", "fp"),))):
    ctx.clear_options()
    load_petsc_options(ctx, opts, is_text=True)
    g = generate_swelling3d(ctx, N, pc_type)
    ctx.sync()
    t0 = time.perf_counter()
    pc = Preconditioner(g.index_set(), g.A, g.P, g.P_diff, dict(g.par), g.bcs_sub_pressure).get_pc()
    ctx.sync()
    setup_s = time.perf_counter() - t0
    cc = pc.getPythonContext()
    for label, name in names:
        info = cc.ilu_info(name)
        n = info["rows"]
        r = DeviceVector(np.random.default_rng(1).standard_normal(n), ctx=ctx)
        z = DeviceVector(n=n, ctx=ctx)
        apply = lambda: cc.inner_solve(name, r, z)
        timed(apply, 3)
        ms = timed(apply, reps)
        out["blocks"][label] = dict(info, pc_setup_s=setup_s, pc_type=pc_type, ms_per_apply=ms,
                                    apply_GBps=info["apply_bytes"] / (ms * 1e-3) / 1e9)
        print(json.dumps(out), flush=True)
    cc.destroy()
    del pc, g
for Ns in sizes:
    ctx.clear_options()
    g = generate_swelling3d(ctx, Ns, "diagonal")
    par = dict(g.par)
    imap = g.index_set()
    db, dx, dr = DeviceVector(g.b, ctx=ctx), DeviceVector(n=len(g.b), ctx=ctx), DeviceVector(n=len(g.b), ctx=ctx)
    for arm, opts in (("fieldsplit", FIELDSPLIT), ("fieldsplit_zeropivot0", FIELDSPLIT + ZP0), ("b200", bench.BENCH_OPTIONS)):
        ctx.clear_options()
        load_petsc_options(ctx, opts, is_text=True)
        t0 = time.perf_counter()
        try:
            pc = Preconditioner(imap, g.A, g.P, None, par, g.bcs_sub_pressure).get_pc()
        except PoroError as e:                 # e.g. a pivot below the absolute zero-pivot threshold
            out["solves"]["%s_N%d" % (arm, Ns)] = dict(refused=str(e), dofs=len(g.b))
            print(json.dumps(out), flush=True)
            continue
        ctx.sync()
        setup_s = time.perf_counter() - t0
        s = Solver(g.A, db, pc, par, imap)
        s.create_solver(g.A, db, pc)
        s.solve(db, dx)
        ms = timed(lambda: s.solve(db, dx), 2)
        g.A.mult(dx, dr)
        ctx.sync()
        res = float(np.linalg.norm(g.b - dr.numpy()) / np.linalg.norm(g.b))
        out["solves"]["%s_N%d" % (arm, Ns)] = dict(its=s.getIterationNumber(), reason=s.solver.reason, setup_s=setup_s,
                                                   ms_per_solve=ms, true_rel_res=res, dofs=len(g.b))
        pc.getPythonContext().destroy()
        print(json.dumps(out), flush=True)
