"""Generated structured-mesh operators applied from their class tables (csrc/stencil.cu).

A matrix generated on the device keeps its stencil tables; the blocks cut out of it along whole fields, and the outer
operator, are applied by k_stencil instead of streaming the assembled CSR.  These tests compare every such product --
the outer operator, each block in every epilogue mode (plain, z - Bx, z + Bx, the fused Chebyshev step, the product with
its dot) -- against scipy products of the generated CSR, for dim 2 and 3 and sizes at which every boundary class meets
every other; check where the tables must NOT travel (permuted P, multi-field blocks, the Schur complement); and compare
a whole solve against the same system uploaded as an assembled matrix."""
import ctypes as C

import numpy as np
import pytest

PC_TYPES = ["diagonal", "diagonal 3-way", "undrained", "undrained 3-way", "lu"]     # the pc types the generator builds
TOL = 1e-13


class _Layout2D:
    """Single-rank layout of the 2D unit square (the slab layout of generator.py covers the cube only)."""

    def __init__(self, N):
        d, L2, L1 = 2, 2 * N + 1, N + 1
        self.n2, self.n1 = L2 ** d, L1 ** d
        self.n_field = [d * self.n2, d * self.n2, self.n1]
        self.off_owned = [0, self.n_field[0], self.n_field[0] + self.n_field[1]]
        self.n_owned = self.n_ext = sum(self.n_field)

    def layout_array(self):
        o = self.n_owned
        return np.asarray([0, self.n1, 0, 0, 0, 0, 0, self.n2, 0, 0, 0, 0, *self.off_owned, o, o, o, o, o, o, o], np.int64)


def _generate(ctx, dim, N, pc_type):
    """(A, P, P_diff, b, index set, bcs_sub_pressure, par) of the swelling problem generated on the device, one rank."""
    from poro_b200.generator import generate_matrix, generate_swelling3d
    from poro_b200.lib.IndexSet import IndexSet
    if dim == 3:
        g = generate_swelling3d(ctx, N, pc_type)
        return g.A, g.P, g.P_diff, g.b, g.index_set(), g.bcs_sub_pressure, g.par
    from hostfem.stencil import swelling_generator
    gen, par, loads = swelling_generator(2, N)
    par = dict(par)
    par["pc type"] = pc_type
    lay = _Layout2D(N)
    ctx.set_halo(0, [], [0], [], [])
    flags = np.concatenate([gen.bc_s.ravel(), gen.bc_f.ravel(), np.zeros(lay.n1, bool)])
    A = generate_matrix(ctx, gen, lay, "A", pc_type, flags)
    P = generate_matrix(ctx, gen, lay, "P", pc_type, flags)
    Pd = None
    if "3-way" in pc_type:
        Pd = generate_matrix(ctx, gen, lay, "P_diff", pc_type, np.concatenate([gen.bc_s.ravel(), gen.bc_f.ravel(), gen.bc_p]))
    b = gen.rhs(par["t0"] + par["dt"], **loads)
    L2, L1 = 2 * N + 1, N + 1
    n2, n1 = np.arange(lay.n2), np.arange(lay.n1)
    c2 = np.stack([n2 % L2, n2 // L2], 1) / (2 * N)
    c1 = np.stack([n1 % L1, n1 // L1], 1) / N
    o = lay.off_owned
    imap = IndexSet(o[0] + np.arange(lay.n_field[0]), o[1] + np.arange(lay.n_field[1]), o[2] + np.arange(lay.n_field[2]),
                    two_way=True, block_dim=2, coords_s=np.repeat(c2, 2, axis=0), coords_p=c1)
    return A, P, Pd, b, imap, np.flatnonzero(gen.bc_p).astype(np.int64), par


def _setup(ctx, dim, N, pc_type, options, imap_override=None):
    from helpers import AMG_OPTIONS
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    ctx.clear_options()
    load_petsc_options(ctx, options or AMG_OPTIONS, is_text=True)
    A, P, Pd, b, imap, bcs, par = _generate(ctx, dim, N, pc_type)
    if imap_override is not None:
        imap = imap_override(imap)
    par = dict(par)
    par.update({"solver rtol": 1e-10, "solver atol": 0.0, "solver maxiter": 200})
    pc = Preconditioner(imap, A, P, Pd, par, bcs).get_pc()
    return A, P, Pd, b, imap, pc, par, bcs


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
    return y.cpu().numpy(), dn.cpu().numpy(), float(dot.cpu()[0])


def _field_ranges(imap_sizes):
    o = np.concatenate([[0], np.cumsum(imap_sizes)])
    return {"s": (o[0], o[1]), "f": (o[1], o[2]), "p": (o[2], o[3])}


# block name -> (row fields, column fields); the matrix it is cut from
BLOCKS = {"ss": ("s", "s"), "sf": ("s", "f"), "sp": ("s", "p"), "ff": ("f", "f"), "fp": ("f", "p"), "pp": ("p", "p"),
          "fps": ("fp", "s"), "fpfp": ("fp", "fp"), "diff": ("p", "p")}
STENCIL_FORMAT = 4


@pytest.mark.gpu
@pytest.mark.parametrize("pc_type", PC_TYPES)
@pytest.mark.parametrize("N", [1, 2, 5, 8])
@pytest.mark.parametrize("dim", [2, 3])
def test_stencil_products_match_assembled_csr(gpu_ctx, dim, N, pc_type):
    import torch
    from poro_b200.lib.Solver import Solver
    A, P, Pd, b, imap, pc, par, bcs = _setup(gpu_ctx, dim, N, pc_type, None)
    pcc = pc.getPythonContext()
    As, Ps = A.to_scipy(), P.to_scipy()
    Ds = Pd.to_scipy() if Pd is not None else None
    n = As.shape[0]
    rng = _field_ranges([imap.ns, imap.nf, imap.np])
    rng["fp"] = (rng["f"][0], rng["p"][1])
    gen = np.random.default_rng(dim * 100 + N)

    # outer operator (one stencil launch per row field) in its three modes
    solver = Solver(A, None, pc, par, imap)
    solver.create_solver(A, None, pc)
    x = gen.standard_normal(n)
    xt = torch.tensor(x, device="cuda")
    yt = torch.zeros(n, dtype=torch.float64, device="cuda")
    solver.solver.mult(xt, yt)
    torch.cuda.synchronize()
    assert _rel(yt.cpu().numpy(), As @ x) <= TOL
    assert all(f == STENCIL_FORMAT for _, f in solver.solver.parts_info())

    found = 0
    for name, (rf, cf) in BLOCKS.items():
        try:
            nr, nc, _ = pcc.block_info(name)
        except Exception:
            continue
        src = Ds if name == "diff" else Ps
        want_B = src[rng[rf][0]:rng[rf][1]][:, rng[cf][0]:rng[cf][1]].tocsr()
        assert want_B.shape == (nr, nc), name
        _, fmt = pcc.block_bytes(name)
        assert (fmt == STENCIL_FORMAT) == (name not in ("fps", "fpfp")), (name, fmt)
        found += 1
        xb = gen.standard_normal(nc)
        zb = gen.standard_normal(nr)
        xbt, zbt = torch.tensor(xb, device="cuda"), torch.tensor(zb, device="cuda")
        Bx = want_B @ xb
        y0, _, _ = _block_mult(pcc, name, 0, xbt)
        y1, _, _ = _block_mult(pcc, name, 1, xbt, z=zbt)
        y2, _, _ = _block_mult(pcc, name, 2, xbt, z=zbt)
        assert _rel(y0, Bx) <= TOL, name
        assert np.abs(y1 - (zb - Bx)).max() <= TOL * max(np.abs(zb - Bx).max(), np.abs(Bx).max()), name
        assert np.abs(y2 - (zb + Bx)).max() <= TOL * max(np.abs(zb + Bx).max(), np.abs(Bx).max()), name
        if nr != nc:
            continue
        r0 = gen.standard_normal(nr)
        dinv = gen.uniform(0.5, 2.0, nr)
        xv0 = gen.standard_normal(nr)
        rt, dt, xvt = (torch.tensor(v, device="cuda") for v in (r0, dinv, xv0))
        _, dn, _ = _block_mult(pcc, name, 3, xbt, r=rt, dinv=dt, xv=xvt, c1=0.3, c2=0.7)
        r_want = r0 - Bx
        d_want = 0.3 * xb + 0.7 * dinv * r_want
        assert np.abs(rt.cpu().numpy() - r_want).max() <= TOL * max(np.abs(r_want).max(), np.abs(Bx).max()), name
        assert np.abs(dn - d_want).max() <= TOL * max(np.abs(d_want).max(), np.abs(Bx).max()), name
        assert np.abs(xvt.cpu().numpy() - (xv0 + d_want)).max() <= TOL * np.abs(xv0 + d_want).max() * 10, name
        y4, _, dot = _block_mult(pcc, name, 4, xbt)
        assert _rel(y4, Bx) <= TOL, name
        assert abs(dot - xb @ Bx) <= TOL * np.abs(xb).max() * np.abs(Bx).sum() * 10, name
    assert found >= 3


@pytest.mark.gpu
def test_stencil_not_attached_to_permuted_or_product_blocks(gpu_ctx):
    """A permuted P, a multi-field block and the Schur complement stay assembled, and their products stay right."""
    import bench
    from poro_b200.lib.IndexSet import IndexSet

    def reverse_s(imap):
        return IndexSet(np.asarray(imap.is_s)[::-1].copy(), imap.is_fp[imap.is_f], imap.is_fp[imap.is_p], two_way=True, block_dim=3,
                        coords_s=np.asarray(imap.coords_s)[::-1].copy(), coords_p=imap.coords_p)

    A, P, Pd, b, imap, pc, par, bcs = _setup(gpu_ctx, 3, 4, "diagonal", bench.BENCH_OPTIONS)
    pcc = pc.getPythonContext()
    assert pcc.block_bytes("ss")[1] == STENCIL_FORMAT and pcc.block_bytes("ff")[1] == STENCIL_FORMAT
    assert pcc.block_bytes("schur")[1] != STENCIL_FORMAT
    assert pcc.block_bytes("fps")[1] != STENCIL_FORMAT
    A, P, Pd, b, imap, pc, par, bcs = _setup(gpu_ctx, 3, 4, "diagonal", bench.BENCH_OPTIONS, reverse_s)
    pcc = pc.getPythonContext()
    assert pcc.block_bytes("ss")[1] != STENCIL_FORMAT          # extracted from the permuted copy of P
    assert pcc.block_bytes("ff")[1] != STENCIL_FORMAT
    import torch
    Ps = P.to_scipy()
    is_s = np.asarray(imap.is_s)                                # the reversed order the block was extracted in
    want = Ps[is_s][:, is_s]
    x = np.random.default_rng(1).standard_normal(len(is_s))
    y, _, _ = _block_mult(pcc, "ss", 0, torch.tensor(x, device="cuda"))
    assert _rel(y, want @ x) <= TOL


@pytest.mark.gpu
def test_solve_on_stencil_path_matches_assembled_upload(gpu_ctx):
    """N = 16, benchmarked options: the same iterations and solution as the same matrices uploaded through
    poro_mat_create_csr (assembled path), and two solves on the stencil path give identical bits."""
    import bench
    from poro_b200.lib.backend import DeviceMatrix, DeviceVector
    from poro_b200.lib.Preconditioner import Preconditioner
    from poro_b200.lib.Solver import Solver
    A, P, Pd, b, imap, pc, par, bcs = _setup(gpu_ctx, 3, 16, "diagonal", bench.BENCH_OPTIONS)
    assert pc.getPythonContext().block_bytes("ss")[1] == STENCIL_FORMAT

    def solve(A_, pc_):
        db, dx = DeviceVector(b, ctx=gpu_ctx), DeviceVector(n=len(b), ctx=gpu_ctx)
        s = Solver(A_, db, pc_, par, imap)
        s.create_solver(A_, db, pc_)
        s.solve(db, dx)
        assert s.solver.reason > 0
        return s.getIterationNumber(), dx.numpy()

    its1, x1 = solve(A, pc)
    its2, x2 = solve(A, pc)
    assert its1 == its2 and np.array_equal(x1, x2)
    Aa, Pa = DeviceMatrix(A.to_scipy(), ctx=gpu_ctx), DeviceMatrix(P.to_scipy(), ctx=gpu_ctx)
    pca = Preconditioner(imap, Aa, Pa, None, par, bcs).get_pc()
    assert pca.getPythonContext().block_bytes("ss")[1] != STENCIL_FORMAT
    its_a, xa = solve(Aa, pca)
    assert its_a == its1
    assert _rel(x1, xa) <= 1e-9
