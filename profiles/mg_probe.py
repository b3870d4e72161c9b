"""The benchmarked option set against options/petsc-options-mg on swelling-3d, in one process and alternated.

For each N the system is generated once with every coarse level N allows attached (the SA-AMG arm ignores them).  The two
arms are set up and solved in turn, `rounds` times each.  Per arm it reports:
  - PC set-up time (host clock around the set-up, which ends in a device synchronise);
  - iterations and ms per solve (CUDA events on the library's stream around poro_ksp_solve);
  - per-level V-cycle time of the solid and velocity hierarchies from the phase-profile slots 8+l / 16+l;
  - for the mg arm, the time of each geometric transfer kernel of the solid hierarchy (CUDA events over `reps` launches)
    and its achieved bandwidth against the algorithmic bytes of poro_pc_mg_bytes.
Prints one JSON line per N, with the card name and power limit.

    python profiles/mg_probe.py [N ...] [--rounds R] [--reps K]
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
from poro_b200.generator import generate_swelling3d
from poro_b200.lib.backend import DeviceVector, get_context
from poro_b200.lib.Parser import load_petsc_options
from poro_b200.lib.Preconditioner import Preconditioner
from poro_b200.lib.Solver import Solver

args = [a for a in sys.argv[1:]]
rounds = int(args[args.index("--rounds") + 1]) if "--rounds" in args else 3
reps = int(args[args.index("--reps") + 1]) if "--reps" in args else 50
Ns = [int(a) for i, a in enumerate(args) if a.isdigit() and (i == 0 or not args[i - 1].startswith("--"))] or [32, 34, 48, 64]
MG_OPTIONS = open(os.path.join(ROOT, "options", "petsc-options-mg")).read()
ARMS = {"saamg": bench.BENCH_OPTIONS, "mg": MG_OPTIONS}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[0]
    except Exception:
        return torch.cuda.get_device_name(0)


def events(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


ctx = get_context(0)
for N in Ns:
    mg_levels = 1
    while N % (1 << mg_levels) == 0:
        mg_levels += 1
    ctx.clear_options()
    g = generate_swelling3d(ctx, N, "diagonal", mg_levels=mg_levels)
    par = dict(g.par)
    par.update({"solver rtol": 1e-8, "solver atol": 0.0, "solver maxiter": 300})
    imap = g.index_set()
    db, dx = DeviceVector(g.b, ctx=ctx), DeviceVector(n=len(g.b), ctx=ctx)
    res = {arm: {"setup_s": [], "its": [], "ms_per_solve": []} for arm in ARMS}
    for _ in range(rounds):
        for arm, opts in ARMS.items():
            ctx.clear_options()
            load_petsc_options(ctx, opts, is_text=True)
            ctx.sync()
            t0 = time.perf_counter()
            pc = Preconditioner(imap, g.A, g.P, None, par, g.bcs_sub_pressure).get_pc()
            ctx.sync()
            res[arm]["setup_s"].append(time.perf_counter() - t0)
            s = Solver(g.A, db, pc, par, imap)
            s.create_solver(g.A, db, pc)
            s.solve(db, dx)                                    # warm-up (graph capture)
            ms = events(lambda: s.solve(db, dx), 3)
            res[arm]["its"].append(s.getIterationNumber())
            res[arm]["ms_per_solve"].append(ms)
            res[arm]["true_rel_res"] = float(np.linalg.norm(g.b - g.A.to_scipy() @ dx.numpy()) / np.linalg.norm(g.b))
            ctx.profile(1)
            s.solve(db, dx)
            ph = ctx.profile(0)
            res[arm]["s_levels_ms"] = [ph[8 + l][0] for l in range(8) if ph.get(8 + l, (0, 0))[1]]
            res[arm]["f_levels_ms"] = [ph[16 + l][0] for l in range(8) if ph.get(16 + l, (0, 0))[1]]
            pcc = pc.getPythonContext()
            if arm == "mg":
                res[arm]["s_mg_info"] = pcc.mg_info("s")
                tr = []
                levels, _ = pcc.mg_info("s")
                for l in range(len(levels) - 1):
                    nf, nc = levels[l][1], levels[l + 1][1]
                    e = torch.ones(nc, dtype=torch.float64, device="cuda")
                    y = torch.zeros(nf, dtype=torch.float64, device="cuda")
                    yc = torch.zeros(nc, dtype=torch.float64, device="cuda")
                    bp, ba, br = pcc.mg_bytes("s", l)
                    t_p = events(lambda: pcc.mg_transfer("s", l, 0, 1, e, y), reps)
                    t_r = events(lambda: pcc.mg_transfer("s", l, 1, 0, y, yc), reps)
                    tr.append({"level": l, "prolong_add_ms": t_p, "prolong_add_TBps": ba / t_p * 1e-9,
                               "restrict_ms": t_r, "restrict_TBps": br / t_r * 1e-9, "bytes": [bp, ba, br]})
                res[arm]["s_transfers"] = tr
            pcc.destroy()
    out = {"N": N, "dofs": len(g.b), "card": card(), "rounds": rounds, "arms": res,
           "median_ms": {a: float(np.median(res[a]["ms_per_solve"])) for a in ARMS}}
    print(json.dumps(out), flush=True)
    del g, db, dx
    torch.cuda.empty_cache()
