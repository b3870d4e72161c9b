"""The benchmarked option set (petsc-options-b200) against options/petsc-options-mg on swelling-3d, on 1 GPU or
row-partitioned over several, alternated in one process per rank.

Weak-scaled meshes divisible by 8 (the bench's N = 43 and 101 are odd, so mg cannot run there): N = 32 on 1 GPU, 40 on 2
and 48 on 4 unless N is given.  The system is generated once with every coarse level the slabs allow attached
(generator.max_mg_levels; the SA-AMG arm ignores them).  Per arm and round it reports the PC set-up time (host clock around
a set-up that ends in a device synchronise, the slowest rank), iterations, ms per timed solve to rtol 1e-8 (CUDA events,
as bench.py) and the true relative residual (distributed product).  Rank 0 prints one JSON line with the card name and
power limit read in the same run.

    python profiles/mg_multi_probe.py [N] [--rounds R]
    python -m torch.distributed.run --nproc-per-node W profiles/mg_multi_probe.py [N] [--rounds R]
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
from poro_b200.generator import generate_swelling3d, max_mg_levels
from poro_b200.lib.backend import DeviceVector, get_context
from poro_b200.lib.Parser import load_petsc_options
from poro_b200.lib.Preconditioner import Preconditioner
from poro_b200.lib.Solver import Solver

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
args = sys.argv[1:]
rounds = int(args[args.index("--rounds") + 1]) if "--rounds" in args else 3
pos = [a for i, a in enumerate(args) if a.isdigit() and (i == 0 or not args[i - 1].startswith("--"))]
N = int(pos[0]) if pos else {1: 32, 2: 40, 4: 48}.get(world, 48)
ARMS = {"b200": bench.BENCH_OPTIONS, "mg": open(os.path.join(ROOT, "options", "petsc-options-mg")).read()}


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0]


def allreduce(vals, op="sum"):
    t = torch.tensor(vals, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return t.cpu().numpy()


ctx = get_context(local)
mg_levels = max_mg_levels(N, world)
ctx.clear_options()
g = generate_swelling3d(ctx, N, "diagonal", rank, world, mg_levels=mg_levels)
par = dict(g.par)
par.update({"solver rtol": 1e-8, "solver atol": 0.0, "solver maxiter": 300})
imap = g.index_set()
db, dx = DeviceVector(g.b, ctx=ctx), DeviceVector(n=len(g.b), ctx=ctx)
dr = DeviceVector(n=len(g.b), ctx=ctx)
res = {arm: {"setup_s": [], "its": [], "ms_per_solve": [], "true_rel_res": []} for arm in ARMS}
for _ in range(rounds):
    for arm, opts in ARMS.items():
        ctx.clear_options()
        load_petsc_options(ctx, opts, is_text=True)
        ctx.sync()
        allreduce([0.0])
        t0 = time.perf_counter()
        pc = Preconditioner(imap, g.A, g.P, None, par, g.bcs_sub_pressure).get_pc()
        ctx.sync()
        res[arm]["setup_s"].append(float(allreduce([time.perf_counter() - t0], "max")[0]))
        s = Solver(g.A, db, pc, par, imap)
        s.create_solver(g.A, db, pc)
        s.solve(db, dx)                                    # warm-up (graph capture)
        allreduce([0.0])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            s.solve(db, dx)
        e1.record()
        torch.cuda.synchronize()
        res[arm]["ms_per_solve"].append(float(allreduce([e0.elapsed_time(e1) / 3], "max")[0]))
        res[arm]["its"].append(s.getIterationNumber())
        g.A.mult(dx, dr)
        ctx.sync()
        r = g.b - dr.numpy()
        nr = allreduce([float(r @ r), float(g.b @ g.b)])
        res[arm]["true_rel_res"].append(float(np.sqrt(nr[0] / nr[1])))
        pc.getPythonContext().destroy()
if rank == 0:
    out = {"gpus": world, "N": N, "dofs": int(g.n_global), "mg_levels": mg_levels, "card": card(), "rounds": rounds, "arms": res,
           "median_ms": {a: float(np.median(res[a]["ms_per_solve"])) for a in ARMS},
           "median_setup_s": {a: float(np.median(res[a]["setup_s"])) for a in ARMS}}
    print(json.dumps(out), flush=True)
if world > 1:
    dist.destroy_process_group()
