"""Sparse LU of the exact blocks on the GPU (-<prefix>pc_factor_mat_solver_type poro, csrc/sparse_lu.cu).

For the `s` and `fp` blocks of swelling 2D N = 40 / 80 / 160 and 3D N = 8 / 16 (`diagonal`, petsc-options-exact + poro):
factor time (device, numeric phase), achieved fp64 FLOP/s of the factorisation (flops counted from the symbolic structure),
nnz(L+U), device bytes, time per application (CUDA events over `reps` inner applications) and the application's achieved
bandwidth (algorithmic bytes: 8 B per stored factor entry + indices + vectors) against the measured 6 559 GB/s of
MEASURED_PEAKS.json; then the outer GMRES (iterations, device time of a second solve).  Last, the N = 20 rows through both
exact paths (sparse LU forced with -poro_dense_lu_limit 10, against the dense inverse), for the dense / sparse crossover.

    python profiles/sparse_lu_probe.py [reps] [cases]      cases: comma list of 2:40,2:80,2:160,3:8,3:16,x20
"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
from helpers import EXACT_OPTIONS, gpu_solve
from hostfem.problems import swelling

PEAK_GBS = 6559.4
SPARSE = EXACT_OPTIONS + "".join("-%s_pc_factor_mat_solver_type poro\n" % p for p in ("s", "f", "p", "diff", "fp"))
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
cases = (sys.argv[2] if len(sys.argv) > 2 else "2:40,2:80,2:160,3:8,3:16,x20").split(",")

from poro_b200.lib.backend import DeviceVector, get_context

ctx = get_context(0)
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as e:          # the card is named in the report either way
    card = "nvidia-smi unavailable (%s)" % e
print("card: %s" % card)


def second_solve_ms(g, s):
    ksp = g["solver"].solver
    db, dx = DeviceVector(s.b, ctx=ctx), DeviceVector(n=s.n, ctx=ctx)
    ctx.sync(); ctx.timer_start(); ksp.solve(db, dx); dt = ctx.timer_stop()
    res = np.linalg.norm(s.b - s.A @ dx.numpy()) / np.linalg.norm(s.b)
    return ksp.its, dt, res


print("%-4s %-6s %5s %8s %11s %9s %9s %8s %9s %7s %9s %9s %8s %5s %7s %9s" % (
    "dim", "N", "block", "rows", "nnz(L+U)", "zeros %", "dev MB", "levels", "max front", "pert", "factor ms",
    "GFLOP/s", "apply ms", "GB/s", "% peak", "outer"))
for case in cases:
    if case == "x20":
        continue
    dim, N = (int(v) for v in case.split(":"))
    t0 = time.time()
    s, par = swelling(dim, N, "diagonal")
    t_asm = time.time() - t0
    g = gpu_solve(s, par, SPARSE, return_objects=True)
    cc = g["pc"].pc.getPythonContext()
    its, ms, res = second_solve_ms(g, s)
    for name in ("s", "fp"):
        fi = cc.factor_info(name)
        n = fi["rows"]
        x = DeviceVector(np.random.default_rng(0).standard_normal(n), ctx=ctx)
        y = DeviceVector(n=n, ctx=ctx)
        for _ in range(3):
            cc.inner_solve(name, x, y)
        ctx.sync(); ctx.timer_start()
        for _ in range(reps):
            cc.inner_solve(name, x, y)
        t_apply = ctx.timer_stop() / reps
        gbs = fi["apply_bytes"] / (t_apply * 1e-3) / 1e9
        fms = fi["factor_us"] * 1e-3
        print("%-4d %-6d %5s %8d %11d %9.1f %9.1f %8d %9d %7d %9.2f %9.1f %8.3f %5.0f %7.1f %4d its %8.2f ms res %.1e" % (
            dim, N, name, n, fi["nnz_l"] + fi["nnz_u"], 100.0 * fi["amalgamation_zeros"] / (fi["nnz_l"] + fi["nnz_u"]),
            fi["device_bytes"] / 2 ** 20, fi["levels"], fi["max_front"], fi["perturbed_pivots"], fms,
            fi["factor_flops"] / (fms * 1e-3) / 1e9 if fms > 0 else 0.0, t_apply, gbs, 100.0 * gbs / PEAK_GBS, its, ms, res),
            flush=True)
    print("     (host assembly %.1f s, preconditioner set-up %.2f s incl. symbolic analysis)" % (t_asm, cc.t_setup), flush=True)
    del g, cc

if "x20" in cases:
    # dense inverse (default limit) against the sparse LU forced below it, swelling 2D N = 20, both pc types
    print("\ncrossover at N = 20 (blocks <= 8 192 rows): outer solve ms (device, second solve) and set-up s")
    for pct in ("diagonal", "diagonal 3-way"):
        s, par = swelling(2, 20, pct)
        for label, opts in (("dense", EXACT_OPTIONS), ("sparse", SPARSE + "-poro_dense_lu_limit 10\n")):
            g = gpu_solve(s, par, opts, return_objects=True)
            its, ms, res = second_solve_ms(g, s)
            print("  %-15s %-6s its %3d  solve %8.2f ms  set-up %6.2f s  true res %.2e" % (
                pct, label, its, ms, g["pc"].pc.getPythonContext().t_setup, res), flush=True)
            del g
