"""BASELINE config 3 on the GPU: the mesh-size robustness sweep of paper-scripts/robustness_2d.sh
(swelling.py -N {10,20,40,80[,160]} x {2-way 'diagonal', 3-way 'diagonal 3-way'} x {exact, AMG}),
one time step each, rtol 1e-6 / atol 1e-8 / maxiter 500 as in swelling.py:64-66.

exact        = petsc-options-exact semantics (dense inverse up to 8192 rows per block, GMRES+AMG to 1e-12 beyond)
exact-sparse = the same with -<prefix>pc_factor_mat_solver_type poro: blocks beyond 8192 rows get the device sparse LU
amg          = linear AMG preconditioner (one V-cycle per block, pressure Schur), right-preconditioned GMRES
    python profiles/robustness_2d.py [maxN] [option sets, comma-separated: exact,exact-sparse,amg]
"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
from helpers import AMG_OPTIONS, EXACT_OPTIONS, gpu_solve
from hostfem.problems import swelling

AMG3 = AMG_OPTIONS + """
-f_ksp_type preonly
-f_pc_type hypre
-p_ksp_type preonly
-p_pc_type hypre
-diff_ksp_type preonly
-diff_pc_type hypre
"""
EXACT_SPARSE = EXACT_OPTIONS + "".join("-%s_pc_factor_mat_solver_type poro\n" % p for p in ("s", "f", "p", "diff", "fp"))
maxN = int(sys.argv[1]) if len(sys.argv) > 1 else 160
SETS = (sys.argv[2] if len(sys.argv) > 2 else "exact,exact-sparse,amg").split(",")
from hostfem.problems import footing
from poro_b200.lib.backend import DeviceVector, get_context
print("%-9s %-4s %-16s %-12s %8s %5s %7s %10s %10s" % ("problem", "N", "pc type", "inner", "DoFs", "its", "reason", "solve ms", "true res"))
LEGS = [("swelling", n, pct) for n in (10, 20, 40, 80, 160) for pct in ("diagonal", "diagonal 3-way")] + \
       [("footing", n, pct) for n in (10, 20, 40, 80) for pct in ("undrained", "undrained 3-way")]      # paper-scripts/robustness_2d.sh:26-70
for prob, N, pct in LEGS:
    if N > maxN:
        continue
    s, par = swelling(2, N, pct) if prob == "swelling" else footing(N, pct)
    for name, opts in (("exact", EXACT_OPTIONS), ("exact-sparse", EXACT_SPARSE), ("amg", AMG3)):
        if name not in SETS:
            continue
        if name == "exact" and N > 40:
            continue            # blocks beyond 8 192 rows: the exact stand-in (GMRES + AMG to 1e-12) takes seconds per outer iteration
        g = gpu_solve(s, par, opts)
        ksp = g["solver"].solver
        ctx = get_context(0)
        db, dx = DeviceVector(s.b, ctx=ctx), DeviceVector(n=s.n, ctx=ctx)
        ctx.sync(); ctx.timer_start(); ksp.solve(db, dx); dt = ctx.timer_stop()        # second solve: the first includes lazy set-up
        res = np.linalg.norm(s.b - s.A @ dx.numpy()) / np.linalg.norm(s.b)
        print("%-9s %-4d %-16s %-12s %8d %5d %7d %10.2f %10.2e" % (prob, N, pct, name, s.n, ksp.its, ksp.reason, dt, res), flush=True)
        del g, ksp
