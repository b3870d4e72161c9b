"""Stencil products (csrc/stencil.cu) against the assembled kernels, in one process on the same values.

Generates swelling-3d at N cells per side (default 34, the benchmarked system) with the benchmarked options, then builds a
second copy of A and P through poro_mat_create_csr from poro_mat_copy of the generated matrices: the copies carry no
stencil tables and run the assembled path (fused BSR3 / CSR).  For both it times with CUDA events, over `reps` launches
after warm-up:
  - the outer operator y = A x (poro_ksp_mult);
  - one solid V-cycle (poro_pc_inner_solve "s") and one velocity V-cycle ("fp0");
  - the level-0 Chebyshev step of the solid V-cycle (phase slot 37, CUDA events around each launch);
and checks that both paths give the same products to the last bits.  Prints one JSON line.

    python profiles/stencil_probe.py [N] [reps]
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import bench
from poro_b200.generator import generate_swelling3d
from poro_b200.lib.backend import DeviceMatrix, get_context
from poro_b200.lib.Parser import load_petsc_options
from poro_b200.lib.Preconditioner import Preconditioner
from poro_b200.lib.Solver import Solver

N = int(sys.argv[1]) if len(sys.argv) > 1 else 34
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 50

ctx = get_context(0)
ctx.clear_options()
load_petsc_options(ctx, bench.BENCH_OPTIONS, is_text=True)
g = generate_swelling3d(ctx, N, "diagonal")
par = dict(g.par)
par.update({"solver rtol": 1e-8, "solver atol": 0.0, "solver maxiter": 200})
imap = g.index_set()
n = len(g.b)


def build(A, P):
    pc = Preconditioner(imap, A, P, None, par, g.bcs_sub_pressure).get_pc()
    s = Solver(A, None, pc, par, imap)
    s.create_solver(A, None, pc)
    return pc, s


def timed(fn):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


paths = {"stencil": build(g.A, g.P)}
paths["assembled"] = build(DeviceMatrix(g.A.to_scipy(), ctx=ctx), DeviceMatrix(g.P.to_scipy(), ctx=ctx))
rng = np.random.default_rng(0)
x = torch.tensor(rng.standard_normal(n), device="cuda")
ns = imap.ns
nf = imap.nf
rs = torch.tensor(rng.standard_normal(ns), device="cuda")
rf = torch.tensor(rng.standard_normal(nf), device="cuda")
out = {"N": N, "dofs": n, "reps": reps, "gpu": torch.cuda.get_device_name(0)}
res = {}
for name, (pc, s) in paths.items():
    pcc = pc.getPythonContext()
    y = torch.zeros(n, dtype=torch.float64, device="cuda")
    zs = torch.zeros(ns, dtype=torch.float64, device="cuda")
    zf = torch.zeros(nf, dtype=torch.float64, device="cuda")
    r = {"outer_mult_ms": timed(lambda: s.solver.mult(x, y)),
         "s_vcycle_ms": timed(lambda: pcc.inner_solve("s", rs, zs)),
         "f_vcycle_ms": timed(lambda: pcc.inner_solve("fp0", rf, zf)),
         "ss_format": pcc.block_bytes("ss")[1], "outer_parts": s.solver.parts_info()}
    ctx.profile(1)
    for _ in range(reps):
        pcc.inner_solve("s", rs, zs)
    ph = ctx.profile(0)
    ms37, n37 = ph.get(37, (0.0, 0))
    r["s_L0_cheby_step_ms"] = ms37 / max(n37, 1)
    r["s_L0_cheby_step_launches"] = n37
    res[name] = r
    r["_y"], r["_zs"], r["_zf"] = y.cpu().numpy(), zs.cpu().numpy(), zf.cpu().numpy()
for k in ("_y", "_zs", "_zf"):
    a, b = res["stencil"].pop(k), res["assembled"].pop(k)
    out["rel_diff" + k] = float(np.abs(a - b).max() / np.abs(b).max())
out.update(res)
out["speedup"] = {k: res["assembled"][k] / res["stencil"][k] for k in ("outer_mult_ms", "s_vcycle_ms", "f_vcycle_ms", "s_L0_cheby_step_ms")
                  if res["stencil"][k] > 0}
print(json.dumps(out))
