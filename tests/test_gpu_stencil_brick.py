"""Brick path of the class-stencil products (csrc/stencil.cu, `-poro_stencil_brick`, default 1).

The interior rows of the 3-D P2 row fields (s and f) are applied by CTAs that stage the column region of a box of rows in
shared memory; the boundary classes, the P1 rows and the lattices too small for a box stay on the per-class warps.  These
tests check every generated block in every epilogue mode and the outer operator against scipy products of the generated
CSR at sizes below, at and above one box (and not a multiple of it along any axis), that repeated launches give the same
bits, and that a whole solve with the path on matches one with it off."""
import ctypes as C

import numpy as np
import pytest

PC_TYPES = ["diagonal", "diagonal 3-way", "undrained", "undrained 3-way", "lu"]
TOL = 1e-13
BLOCKS = {"ss": ("s", "s"), "sf": ("s", "f"), "sp": ("s", "p"), "ff": ("f", "f"), "fp": ("f", "p"), "pp": ("p", "p"),
          "fps": ("fp", "s"), "fpfp": ("fp", "fp"), "diff": ("p", "p")}


def _setup(ctx, N, pc_type, options, brick):
    from poro_b200.generator import generate_swelling3d
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    ctx.clear_options()
    load_petsc_options(ctx, options + "\n-poro_stencil_brick %d\n" % brick, is_text=True)
    g = generate_swelling3d(ctx, N, pc_type)
    par = dict(g.par)
    par.update({"solver rtol": 1e-10, "solver atol": 0.0, "solver maxiter": 200})
    imap = g.index_set()
    pc = Preconditioner(imap, g.A, g.P, g.P_diff, par, g.bcs_sub_pressure).get_pc()
    return g, imap, pc, par


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _block_mult(pcc, name, mode, x, z=None, r=None, dinv=None, xv=None, c1=0.3, c2=0.7):
    import torch
    n = pcc.block_info(name)[0]
    y = torch.zeros(n, dtype=torch.float64, device="cuda")
    dn = torch.zeros(n, dtype=torch.float64, device="cuda")
    dot = torch.zeros(1, dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    torch.cuda.synchronize()
    rc = pcc.ctx.lib.poro_pc_block_mult(pcc.h, name.encode(), mode, p(x), p(y), p(z), p(r), p(dn), p(xv), p(dinv), c1, c2, p(dot))
    assert rc == 0, pcc.ctx.lib.poro_last_error()
    torch.cuda.synchronize()
    return y.cpu().numpy(), dn.cpu().numpy(), float(dot.cpu()[0])


@pytest.mark.gpu
@pytest.mark.parametrize("pc_type", PC_TYPES)
@pytest.mark.parametrize("N", [1, 2, 3, 5, 8, 17, 34])
def test_brick_products_match_generated_csr(gpu_ctx, N, pc_type):
    import torch
    from helpers import AMG_OPTIONS
    from poro_b200.lib.Solver import Solver
    g, imap, pc, par = _setup(gpu_ctx, N, pc_type, AMG_OPTIONS, 1)
    pcc = pc.getPythonContext()
    As, Ps = g.A.to_scipy(), g.P.to_scipy()
    Ds = g.P_diff.to_scipy() if g.P_diff is not None else None
    o = np.concatenate([[0], np.cumsum([imap.ns, imap.nf, imap.np])])
    rng = {"s": (o[0], o[1]), "f": (o[1], o[2]), "p": (o[2], o[3]), "fp": (o[1], o[3])}
    gen = np.random.default_rng(1000 + N)

    # outer operator: one launch per row field, twice (same bits)
    solver = Solver(g.A, None, pc, par, imap)
    solver.create_solver(g.A, None, pc)
    n = As.shape[0]
    x = gen.standard_normal(n)
    xt = torch.tensor(x, device="cuda")
    y1 = torch.zeros(n, dtype=torch.float64, device="cuda")
    y2 = torch.zeros(n, dtype=torch.float64, device="cuda")
    solver.solver.mult(xt, y1)
    solver.solver.mult(xt, y2)
    torch.cuda.synchronize()
    assert _rel(y1.cpu().numpy(), As @ x) <= TOL
    assert torch.equal(y1, y2)

    found = 0
    for name, (rf, cf) in BLOCKS.items():
        try:
            nr, nc, _ = pcc.block_info(name)
        except Exception:
            continue
        found += 1
        src = Ds if name == "diff" else Ps
        B = src[rng[rf][0]:rng[rf][1]][:, rng[cf][0]:rng[cf][1]].tocsr()
        xb, zb = gen.standard_normal(nc), gen.standard_normal(nr)
        xbt, zbt = torch.tensor(xb, device="cuda"), torch.tensor(zb, device="cuda")
        Bx = B @ xb
        y0, _, _ = _block_mult(pcc, name, 0, xbt)
        y0b, _, _ = _block_mult(pcc, name, 0, xbt)
        ys, _, _ = _block_mult(pcc, name, 1, xbt, z=zbt)
        ya, _, _ = _block_mult(pcc, name, 2, xbt, z=zbt)
        assert _rel(y0, Bx) <= TOL, name
        assert np.array_equal(y0, y0b), name
        assert np.abs(ys - (zb - Bx)).max() <= TOL * max(np.abs(zb - Bx).max(), np.abs(Bx).max()), name
        assert np.abs(ya - (zb + Bx)).max() <= TOL * max(np.abs(zb + Bx).max(), np.abs(Bx).max()), name
        if nr != nc:
            continue
        r0, dinv, xv0 = gen.standard_normal(nr), gen.uniform(0.5, 2.0, nr), gen.standard_normal(nr)
        rt, dt, xvt = (torch.tensor(v, device="cuda") for v in (r0, dinv, xv0))
        _, dn, _ = _block_mult(pcc, name, 3, xbt, r=rt, dinv=dt, xv=xvt)
        r_want = r0 - Bx
        d_want = 0.3 * xb + 0.7 * dinv * r_want
        assert np.abs(rt.cpu().numpy() - r_want).max() <= TOL * max(np.abs(r_want).max(), np.abs(Bx).max()), name
        assert np.abs(dn - d_want).max() <= TOL * max(np.abs(d_want).max(), np.abs(Bx).max()), name
        assert np.abs(xvt.cpu().numpy() - (xv0 + d_want)).max() <= TOL * np.abs(xv0 + d_want).max() * 10, name
        y4, _, dot = _block_mult(pcc, name, 4, xbt)
        _, _, dot2 = _block_mult(pcc, name, 4, xbt)
        assert _rel(y4, Bx) <= TOL, name
        assert abs(dot - xb @ Bx) <= TOL * np.abs(xb).max() * np.abs(Bx).sum() * 10, name
        assert dot == dot2, name
    assert found >= 3


@pytest.mark.gpu
def test_brick_solve_matches_per_class_warps(gpu_ctx):
    """N = 16, benchmarked options: the same iterations and a solution within 1e-12 with the brick path off and on."""
    import bench
    from poro_b200.lib.backend import DeviceVector
    from poro_b200.lib.Solver import Solver

    def solve(brick):
        g, imap, pc, par = _setup(gpu_ctx, 16, "diagonal", bench.BENCH_OPTIONS, brick)
        db, dx = DeviceVector(g.b, ctx=gpu_ctx), DeviceVector(n=len(g.b), ctx=gpu_ctx)
        s = Solver(g.A, db, pc, par, imap)
        s.create_solver(g.A, db, pc)
        s.solve(db, dx)
        assert s.solver.reason > 0
        return s.getIterationNumber(), dx.numpy()

    its0, x0 = solve(0)
    its1, x1 = solve(1)
    its1b, x1b = solve(1)
    assert its0 == its1
    assert _rel(x1, x0) <= 1e-12
    assert its1b == its1 and np.array_equal(x1, x1b)
