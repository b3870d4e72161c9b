"""Worker of tests/test_gpu_mg_multi.py (under torch.distributed.run): `-<prefix>pc_type mg` on row-partitioned generated
slabs.  Checks, on every rank's owned rows:
  1. the distributed transfer kernels against the global masked prolongation of hostfem/mg.py and its transpose, on every
     geometric level ($PORO_MG_N, default 16, with $PORO_MG_LEVELS, default 3, levels), for the s, f, p and diff blocks;
  2. one `-s_pc_type mg` application (N = 16, 3 levels: the coarsest level, N = 4, is solved by the gathered dense inverse)
     against the single-rank application in $PORO_MG_REF to 1e-12;
  3. CG on the solid block (examples/solid.py) with mg at N = 16 and 32: the single-rank iteration count +-1;
  4. a whole swelling-3d solve with options/petsc-options-mg against the single-rank solution: true residual <= 1e-8,
     solution within 1e-8, iterations within 10 %, the preconditioner replayed from its captured CUDA graph;
  5. the refusals: a host-assembled row-partitioned block, a non-nesting poro_mat_set_coarse pair, too many levels.
$PORO_MG_TRANSFERS_ONLY=1 runs check 1 alone (no reference needed: more ranks, other slab starts)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torch.distributed as dist

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))

from hostfem.mg import masked_prolongation
from hostfem.stencil import swelling_generator
from poro_b200 import _capi
from poro_b200.generator import SlabLayout, generate_matrix, generate_swelling3d
from poro_b200.lib.backend import DeviceVector, get_context
from poro_b200.lib.Parser import load_petsc_options
from poro_b200.lib.Preconditioner import Preconditioner
from poro_b200.lib.Solver import Solver
from test_gpu_mg_multi import SOLID_MG

MG_OPTIONS = open(os.path.join(ROOT, "options", "petsc-options-mg")).read()
THREE_WAY_MG = "".join("-%s_ksp_type preonly\n-%s_pc_type mg\n" % (b, b) for b in ("s", "f", "p", "diff"))
THREE_WAY_MG = "-global_ksp_type gmres\n-global_ksp_pc_side right\n" + THREE_WAY_MG
N, LEVELS = int(os.environ.get("PORO_MG_N", "16")), int(os.environ.get("PORO_MG_LEVELS", "3"))
TRANSFERS_ONLY = os.environ.get("PORO_MG_TRANSFERS_ONLY", "0") == "1"
ctx = get_context(local)
failures = []


def check(ok, what):
    if not ok:
        failures.append(what)
        print("rank %d FAILED: %s" % (rank, what), flush=True)


def setup(options, pc_type, init_dist):
    ctx.clear_options()
    load_petsc_options(ctx, options, is_text=True)
    g = generate_swelling3d(ctx, N, pc_type, rank, world, init_dist=init_dist, mg_levels=LEVELS)
    par = dict(g.par)
    par.update({"solver rtol": 1e-8, "solver atol": 0.0, "solver maxiter": 300})
    pc = Preconditioner(g.index_set(), g.A, g.P, g.P_diff, par, g.bcs_sub_pressure).get_pc()
    return g, pc, par


# ---- 1. transfers on every geometric level ---------------------------------------------------------------------------
g, pc, par = setup(THREE_WAY_MG, "diagonal 3-way", True)
pcc = pc.getPythonContext()
lays = [SlabLayout(3, N, rank, world)]
for _ in range(1, LEVELS):
    lays.append(lays[-1].coarsen())
gens = [swelling_generator(3, N >> l)[0] for l in range(LEVELS)]
flags = [{"s": q.bc_s.ravel(), "f": q.bc_f.ravel(), "p": None, "diff": q.bc_p} for q in gens]
rng = np.random.default_rng(7)                              # the same vectors on every rank
for lev in range(LEVELS - 1):
    Nc = N >> (lev + 1)
    for name in ("s", "f", "p", "diff"):
        kind, bs = (2, 3) if name in ("s", "f") else (1, 1)
        k = 1 if kind == 2 else 0
        P = masked_prolongation(3, Nc, kind, bs, flags[lev][name], flags[lev + 1][name])
        x, r = rng.standard_normal(P.shape[1]), rng.standard_normal(P.shape[0])
        fo, co = lays[lev].owned[k], lays[lev + 1].owned[k]
        fs, cs = slice(fo[0] * bs, fo[1] * bs), slice(co[0] * bs, co[1] * bs)
        for direction, xin, want, rows in ((0, x[cs], P @ x, fs), (1, r[fs], P.T @ r, cs)):
            scale = (abs(P) @ np.abs(x)) if direction == 0 else (abs(P).T @ np.abs(r))
            xt = torch.tensor(xin, device="cuda")
            yt = torch.full((rows.stop - rows.start,), float("nan"), dtype=torch.float64, device="cuda")
            pcc.mg_transfer(name, lev, direction, 0, xt, yt)
            torch.cuda.synchronize()
            y = yt.cpu().numpy()
            bad = ~(np.abs(y - want[rows]) <= 1e-14 * scale[rows] + 1e-300)
            check(not bad.any(), "transfer %s level %d dir %d: %d bad rows (slab %s)" % (name, lev, direction, int(bad.sum()),
                                                                                       lays[lev].planes2))


def finish():
    flag = torch.tensor([0 if failures else 1], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0 and int(flag) == 1:
        print("MG MULTI-GPU OK", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 1 else 1)


if TRANSFERS_ONLY:
    finish()
db, dx = DeviceVector(g.b, ctx=ctx), DeviceVector(n=len(g.b), ctx=ctx)
s = Solver(g.A, db, pc, par, g.index_set())
s.create_solver(g.A, db, pc)
s.solve(db, dx)
check(s.solver.reason > 0, "3-way mg solve did not converge (reason %d)" % s.solver.reason)

def rel_err(x, xr):
    num = torch.tensor([np.sum((x - xr) ** 2), np.sum(xr ** 2)], device="cuda")
    dist.all_reduce(num)
    return float(torch.sqrt(num[0] / num[1]))


ref = np.load(os.environ["PORO_MG_REF"])

# ---- 2. one application of the solid block's geometric V-cycle -------------------------------------------------------
g, pc, par = setup(MG_OPTIONS, "diagonal", False)
own_s = slice(lays[0].owned[1][0] * 3, lays[0].owned[1][1] * 3)
r_s = DeviceVector(np.ascontiguousarray(ref["r_s"][own_s]), ctx=ctx)
z_s = DeviceVector(n=own_s.stop - own_s.start, ctx=ctx)
pc.getPythonContext().inner_solve("s", r_s, z_s)
ctx.sync()
err = rel_err(z_s.numpy(), ref["z_s"][own_s])
if rank == 0:
    print("one s_ mg application on %d ranks: relative difference to one rank %.2e" % (world, err), flush=True)
check(err <= 1e-12, "one s_ mg application differs from the single-rank one by %.2e" % err)

# ---- 4. whole solve with petsc-options-mg against the single-rank solution -------------------------------------------
db, dx = DeviceVector(g.b, ctx=ctx), DeviceVector(n=len(g.b), ctx=ctx)
s = Solver(g.A, db, pc, par, g.index_set())
s.create_solver(g.A, db, pc)
s.solve(db, dx)
its = s.getIterationNumber()
x = dx.numpy()
replays = pc.getPythonContext().stats()["graph_replays"]
xr = ref["x"][g.owned_global]
# true residual of the distributed solution: A x with the global host matrix of the same problem
from oracle.problems import swelling
glob, _ = swelling(3, N, "diagonal")
xs = torch.zeros(glob.n, dtype=torch.float64, device="cuda")
xs[torch.tensor(g.owned_global, device="cuda")] = torch.tensor(x, device="cuda")
dist.all_reduce(xs)
xg = xs.cpu().numpy()
res = np.linalg.norm(glob.b - glob.A @ xg) / np.linalg.norm(glob.b)
err = rel_err(x, xr)
if rank == 0:
    print("mg on %d ranks: its %d (single rank %d) true residual %.2e, solution err %.2e" % (world, its, int(ref["its"]), res, err), flush=True)
check(s.solver.reason > 0 and res <= 1e-8, "solve: reason %d true residual %.2e" % (s.solver.reason, res))
check(err <= 1e-8, "solution differs from the single-rank one by %.2e" % err)
check(abs(its - int(ref["its"])) <= max(1, int(ref["its"]) // 10), "iterations %d vs %d" % (its, int(ref["its"])))
# the transfer halos are exchanged inside the preconditioner's CUDA graph: the solve replayed it
check(replays > 0, "the preconditioner never ran as its captured CUDA graph")

# ---- 3. CG on the solid block (examples/solid.py) -------------------------------------------------------------------
sys.path.insert(0, os.path.join(ROOT, "examples"))
from _single_block import build as build_block
for Ns in (16, 32):
    _, cc, dbs, dxs, _, _, keep = build_block("s", Ns, ctx=ctx, options_text=SOLID_MG[Ns])
    cc.inner_solve("s", dbs, dxs)
    ctx.sync()
    its_s, reason_s, _ = cc.inner_result("s")
    want = int(ref["solid_its_%d" % Ns])
    if rank == 0:
        print("solid CG + mg N = %d on %d ranks: %d iterations (single rank %d)" % (Ns, world, its_s, want), flush=True)
    check(reason_s > 0 and abs(its_s - want) <= 1, "solid CG N = %d: %d iterations (reason %d) vs %d" % (Ns, its_s, reason_s, want))
    cc.destroy()
    del keep

# ---- 5. refusals -------------------------------------------------------------------------------------------------------
try:
    generate_swelling3d(ctx, 8, "diagonal", rank, world, init_dist=False, mg_levels=4)
    check(False, "too many levels were accepted")
except ValueError as e:
    check("level" in str(e) and "rank" in str(e), "too-many-levels message: %s" % e)
gen, _, _ = swelling_generator(3, 16)
genc, _, _ = swelling_generator(3, 8)
fine = SlabLayout(3, 16, rank, world)
bad = SlabLayout(3, 8, rank, world, p2_planes=[(0, 7), (7, 17)][rank] if world == 2 else None)
Af = generate_matrix(ctx, gen, fine, "A", "diagonal", None)
Ac = generate_matrix(ctx, genc, bad, "A", "diagonal", None)
try:
    _capi.check(ctx.lib.poro_mat_set_coarse(Af.handle, Ac.handle))
    check(False, "a non-nesting coarse slab was accepted")
except Exception as e:
    check("do not nest" in str(e), "non-nesting message: %s" % e)
from poro_b200.lib.backend import DeviceMatrix
from poro_b200.partition import distributed_problem
ctx.clear_options()
load_petsc_options(ctx, MG_OPTIONS, is_text=True)
prob = distributed_problem(3, 8, "diagonal", rank, world, ctx)
par = dict(prob.par)
try:
    Preconditioner(prob.index_set(), DeviceMatrix(prob.sys.A, ctx), DeviceMatrix(prob.sys.P, ctx), None, par,
                   prob.sys.bcs_sub_pressure).get_pc()
    check(False, "a host-assembled row-partitioned block took pc_type mg")
except Exception as e:
    check("generated" in str(e), "host-assembled message: %s" % e)

finish()
