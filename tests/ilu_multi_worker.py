"""Worker of tests/test_gpu_ilu_fieldsplit.py::test_two_rank_bjacobi, run under torch.distributed.run on 2 ranks:
block Jacobi + ILU(0) per rank against the twin's ILU(0) of that rank's owned diagonal block, the petsc-options-fieldsplit
solve with the default multi-rank sub-PC (bjacobi), and the refusal of `ilu` on a row-partitioned block."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torch.distributed as dist

from ilu_twin import ILU0

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))

from poro_b200._capi import PoroError
from poro_b200.lib.backend import DeviceMatrix, DeviceVector, get_context
from poro_b200.lib.Parser import load_petsc_options
from poro_b200.lib.Preconditioner import Preconditioner
from poro_b200.lib.Solver import Solver
from poro_b200.partition import distributed_problem

ctx = get_context(local)
OPTIONS = open(os.path.join(ROOT, "options", "petsc-options-fieldsplit")).read()
load_petsc_options(ctx, OPTIONS, is_text=True)
prob = distributed_problem(3, 8, "diagonal", rank, world, ctx)
s, par = prob.sys, dict(prob.par)
imap = prob.index_set()
dA, dP = DeviceMatrix(s.A, ctx), DeviceMatrix(s.P, ctx)
db, dx = DeviceVector(s.b, ctx=ctx), DeviceVector(n=len(s.b), ctx=ctx)
pc = Preconditioner(imap, dA, dP, None, par, s.bcs_sub_pressure).get_pc()
cc = pc.getPythonContext()
ok = True
# 1. bjacobi = ILU(0) of the owned diagonal block of each split (owned columns come first in the extracted block)
rng = np.random.default_rng(31 + rank)
for name, blk in (("fp0", "pp"), ("fp1", "ff")):
    B = cc.block(blk)
    Bl = B[:, : B.shape[0]].tocsr()
    info = cc.ilu_info(name)
    r = rng.standard_normal(B.shape[0])
    dr, dz = DeviceVector(r, ctx=ctx), DeviceVector(n=len(r), ctx=ctx)
    cc.inner_solve(name, dr, dz)
    ctx.sync()
    e = np.linalg.norm(dz.numpy() - ILU0(Bl)(r)) / np.linalg.norm(ILU0(Bl)(r))
    print("rank", rank, name, "rows", info["rows"], "levels", info["lower_levels"], "err %.2e" % e, flush=True)
    ok = ok and e <= 1e-12 and info["rows"] == B.shape[0]
# 2. the whole solve converges with the true residual below rtol
solver = Solver(dA, db, pc, par, imap)
solver.create_solver(dA, db, pc)
solver.solve(db, dx)
dr = DeviceVector(n=len(s.b), ctx=ctx)
dA.mult(dx, dr)
ctx.sync()
loc = torch.tensor([np.sum((s.b - dr.numpy()) ** 2), np.sum(s.b ** 2)], device="cuda", dtype=torch.float64)
dist.all_reduce(loc)
res, nb = float(torch.sqrt(loc[0])), float(torch.sqrt(loc[1]))
its, reason = solver.getIterationNumber(), solver.solver.reason
if rank == 0:
    print("its", its, "reason", reason, "true residual %.3e" % (res / nb), flush=True)
ok = ok and reason > 0 and res <= max(par["solver rtol"] * nb, par["solver atol"])
# 3. ilu on a row-partitioned block is refused
ctx.set_option("-fp_fieldsplit_0_pc_type", "ilu")
try:
    Preconditioner(imap, dA, dP, None, par, s.bcs_sub_pressure).get_pc()
    ok = False
except PoroError as err:
    ok = ok and "row-partitioned" in str(err)
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0 and int(flag) == 1:
    print("ILU MULTI-GPU OK", flush=True)
dist.destroy_process_group()
sys.exit(0 if int(flag) == 1 else 1)
