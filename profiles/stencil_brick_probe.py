"""Brick path of the class-stencil kernel (csrc/stencil.cu, `-poro_stencil_brick`) against the per-class warps, in one
process on the same values.

Generates swelling-3d at N cells per side (default 34, the benchmarked system) twice with the benchmarked options, once
with `-poro_stencil_brick 0` and once with 1, and times with CUDA events, the two settings alternated round by round:
  - the level-0 Chebyshev step of the solid V-cycle on P_ss (phase slot 37, events around each launch);
  - a plain product y = P_ss x (poro_pc_block_mult, mode 0);
  - the outer operator y = A x (poro_ksp_mult);
  - one solid V-cycle (poro_pc_inner_solve "s") and one velocity V-cycle ("fp0").
Prints the medians over the rounds and the largest relative difference (max norm) of each product between the settings
as one JSON line.

    python profiles/stencil_brick_probe.py [N] [reps] [rounds]
"""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import bench
from poro_b200.generator import generate_swelling3d
from poro_b200.lib.backend import get_context
from poro_b200.lib.Parser import load_petsc_options
from poro_b200.lib.Preconditioner import Preconditioner
from poro_b200.lib.Solver import Solver

N = int(sys.argv[1]) if len(sys.argv) > 1 else 34
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 50
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5

ctx = get_context(0)


def build(brick):
    ctx.clear_options()
    load_petsc_options(ctx, bench.BENCH_OPTIONS + "\n-poro_stencil_brick %d\n" % brick, is_text=True)
    g = generate_swelling3d(ctx, N, "diagonal")
    par = dict(g.par)
    par.update({"solver rtol": 1e-8, "solver atol": 0.0, "solver maxiter": 200})
    imap = g.index_set()
    pc = Preconditioner(imap, g.A, g.P, None, par, g.bcs_sub_pressure).get_pc()
    s = Solver(g.A, None, pc, par, imap)
    s.create_solver(g.A, None, pc)
    return g, imap, pc, s


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


paths = {b: build(b) for b in (0, 1)}
g, imap = paths[0][0], paths[0][1]
n, ns, nf = len(g.b), imap.ns, imap.nf
rng = np.random.default_rng(0)
x = torch.tensor(rng.standard_normal(n), device="cuda")
xs = torch.tensor(rng.standard_normal(ns), device="cuda")
rs = torch.tensor(rng.standard_normal(ns), device="cuda")
rf = torch.tensor(rng.standard_normal(nf), device="cuda")
bufs = {b: {"y": torch.zeros(n, dtype=torch.float64, device="cuda"), "yss": torch.zeros(ns, dtype=torch.float64, device="cuda"),
            "zs": torch.zeros(ns, dtype=torch.float64, device="cuda"), "zf": torch.zeros(nf, dtype=torch.float64, device="cuda")}
        for b in paths}


def ss_mult(pcc, y):
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    rc = pcc.ctx.lib.poro_pc_block_mult(pcc.h, b"ss", 0, p(xs), p(y), None, None, None, None, None, 0.0, 0.0, None)
    assert rc == 0, pcc.ctx.lib.poro_last_error()


keys = ("s_L0_cheby_step_ms", "ss_mult_ms", "outer_mult_ms", "s_vcycle_ms", "f_vcycle_ms")
times = {b: {k: [] for k in keys} for b in paths}
for _ in range(rounds):
    for b, (_, _, pc, s) in paths.items():
        pcc = pc.getPythonContext()
        v = bufs[b]
        t = times[b]
        ctx.profile(1)
        for _ in range(reps):
            pcc.inner_solve("s", rs, v["zs"])
        ph = ctx.profile(0)
        ms37, n37 = ph.get(37, (0.0, 0))
        t["s_L0_cheby_step_ms"].append(ms37 / max(n37, 1))
        t["ss_mult_ms"].append(timed(lambda: ss_mult(pcc, v["yss"])))
        t["outer_mult_ms"].append(timed(lambda: s.solver.mult(x, v["y"])))
        t["s_vcycle_ms"].append(timed(lambda: pcc.inner_solve("s", rs, v["zs"])))
        t["f_vcycle_ms"].append(timed(lambda: pcc.inner_solve("fp0", rf, v["zf"])))
torch.cuda.synchronize()
out = {"N": N, "dofs": n, "reps": reps, "rounds": rounds, "gpu": torch.cuda.get_device_name(0),
       "ss_bytes": paths[1][2].getPythonContext().block_bytes("ss")[0]}
for b in paths:
    out["brick%d" % b] = {k: float(np.median(v)) for k, v in times[b].items()}
    out["brick%d_spread" % b] = {k: float(np.max(v) - np.min(v)) for k, v in times[b].items()}
out["speedup"] = {k: out["brick0"][k] / out["brick1"][k] for k in keys if out["brick1"][k] > 0}
for k in ("y", "yss", "zs", "zf"):
    a, c = bufs[1][k].cpu().numpy(), bufs[0][k].cpu().numpy()
    out["rel_diff_" + k] = float(np.abs(a - c).max() / np.abs(c).max())
print(json.dumps(out))
