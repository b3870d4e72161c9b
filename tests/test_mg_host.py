"""Geometric transfer of `-<prefix>pc_type mg` on the CPU: the scipy prolongation of hostfem/mg.py (interpolation of
polynomials, Galerkin identity with the generated coarse blocks) and the class tables of csrc/mg_transfer.h expanded by a
g++ harness, which must give the same P~ and P~^T entry by entry."""
import ctypes as C
import functools
import itertools
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from hostfem.mg import GeometricMG, injection, masked_prolongation, prolongation

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "poroelasticity-linear-solvers_b200", "csrc")
PC_TYPES = ["diagonal", "diagonal 3-way", "undrained", "undrained 3-way", "lu"]


def _coords(dim, L):
    g = np.stack(np.meshgrid(*[np.arange(L)] * dim, indexing="ij"), -1).reshape(-1, dim)[:, ::-1]
    return g / (L - 1)


@pytest.mark.parametrize("kind", [2, 1])
@pytest.mark.parametrize("Nc", [1, 2, 3, 4])
@pytest.mark.parametrize("dim", [2, 3])
def test_prolongation_reproduces_polynomials(dim, Nc, kind):
    P = prolongation(dim, Nc, kind)
    Lc, Lf = (2 * Nc + 1, 4 * Nc + 1) if kind == 2 else (Nc + 1, 2 * Nc + 1)
    xc, xf = _coords(dim, Lc), _coords(dim, Lf)
    assert P.shape == (len(xf), len(xc))
    for a in itertools.product(range(kind + 1), repeat=dim):
        if sum(a) > kind:
            continue
        q = lambda x: np.prod([x[:, m] ** a[m] for m in range(dim)], axis=0)
        assert np.abs(P @ q(xc) - q(xf)).max() <= 1e-13, a
    # rows of coinciding nodes are unit rows: injection is a right inverse
    inj = injection(dim, Nc, kind)
    assert np.array_equal(P[inj].toarray(), np.eye(len(xc)))


@functools.lru_cache(maxsize=None)
def _system(dim, N, pc_type):
    from hostfem.stencil import swelling_generator
    gen, par, loads = swelling_generator(dim, N)
    s = gen.system(pc_type, par["t0"] + par["dt"], **loads)
    return gen, s


def _blocks(dim, N, pc_type):
    """name -> (BC'd block, kind, bs, Dirichlet flags per dof or None)."""
    gen, s = _system(dim, N, pc_type)
    ns, nf = s.ns, s.nf
    out = {"ss": (s.P[:ns, :ns], 2, dim, gen.bc_s.ravel()), "ff": (s.P[ns:ns + nf, ns:ns + nf], 2, dim, gen.bc_f.ravel()),
           "pp": (s.P[ns + nf:, ns + nf:], 1, 1, None)}
    if s.P_diff is not None:
        out["diff"] = (s.P_diff[ns + nf:, ns + nf:], 1, 1, gen.bc_p)
    return out


@pytest.mark.parametrize("pc_type", PC_TYPES)
@pytest.mark.parametrize("N", [4, 8])
@pytest.mark.parametrize("dim", [2, 3])
def test_rediscretisation_is_galerkin(dim, N, pc_type):
    fine, coarse = _blocks(dim, N, pc_type), _blocks(dim, N // 2, pc_type)
    for name, (B, kind, bs, bcf) in fine.items():
        Bc, _, _, bcc = coarse[name]
        P = masked_prolongation(dim, N // 2, kind, bs, bcf, bcc)
        G = (P.T @ sp.csr_matrix(B) @ P).toarray()
        Bc = Bc.toarray()
        free = np.ones(len(Bc), bool) if bcc is None else ~np.asarray(bcc, bool)
        ref = Bc[np.ix_(free, free)]
        assert np.abs(G[np.ix_(free, free)] - ref).max() <= 1e-12 * np.abs(ref).max(), name
        if bcc is not None:
            d = np.flatnonzero(~free)
            assert np.array_equal(Bc[d], np.eye(len(Bc))[d]), name          # the generator's unit rows


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("mgtab") / "mg_transfer_harness.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + CSRC, os.path.join(ROOT, "tests", "mg_transfer_harness.cpp"),
                    "-o", out], check=True)
    lib = C.CDLL(out)
    lib.mg_expand.restype = C.c_int64
    lib.mg_expand.argtypes = [C.c_int] * 4 + [C.c_void_p] * 2 + [C.c_int] + [C.c_void_p] * 3 + [C.c_int64]
    return lib


def _expand(lib, dim, kind, Nc, bs, bcf, bcc, direction, shape):
    p = lambda a: None if a is None else a.ctypes.data
    n = lib.mg_expand(dim, kind, Nc, bs, p(bcf), p(bcc), direction, None, None, None, 0)
    r, c, v = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n)
    lib.mg_expand(dim, kind, Nc, bs, p(bcf), p(bcc), direction, p(r), p(c), p(v), n)
    assert len(set(zip(r.tolist(), c.tolist()))) == n, "duplicate entries"
    return sp.csr_matrix((v, (r, c)), shape=shape)


@pytest.mark.parametrize("Nc", [1, 2, 3, 4])
@pytest.mark.parametrize("dim", [2, 3])
def test_class_tables_equal_scipy_transfer(harness, dim, Nc):
    from hostfem.stencil import swelling_generator
    gf, gc = swelling_generator(dim, 2 * Nc)[0], swelling_generator(dim, Nc)[0]
    cases = [(2, dim, gf.bc_s.ravel(), gc.bc_s.ravel()), (2, dim, gf.bc_f.ravel(), gc.bc_f.ravel()), (1, 1, gf.bc_p, gc.bc_p),
             (1, 1, None, None), (2, 1, None, None)]
    for kind, bs, bcf, bcc in cases:
        u8 = lambda a: None if a is None else np.ascontiguousarray(a, np.uint8)
        P = masked_prolongation(dim, Nc, kind, bs, bcf, bcc)
        Pt = _expand(harness, dim, kind, Nc, bs, u8(bcf), u8(bcc), 0, P.shape)
        Rt = _expand(harness, dim, kind, Nc, bs, u8(bcf), u8(bcc), 1, P.T.shape)
        assert (Pt != P).nnz == 0, (kind, bs)
        assert (Rt != P.T).nnz == 0, (kind, bs)


def test_twin_geometric_levels_stack_on_saamg():
    """The CPU twin: geometric levels above SA-AMG, the injected near-nullspace and a contracting V-cycle."""
    dim, N = 2, 8
    fine, mid, coarse = _blocks(dim, N, "diagonal"), _blocks(dim, N // 2, "diagonal"), _blocks(dim, N // 4, "diagonal")
    B0, kind, bs, bcf = fine["ss"]
    Pa = masked_prolongation(dim, N // 2, kind, bs, bcf, mid["ss"][3])
    Pb = masked_prolongation(dim, N // 4, kind, bs, mid["ss"][3], coarse["ss"][3])
    mg = GeometricMG([B0, mid["ss"][0], coarse["ss"][0]], [Pa, Pb], [injection(dim, N // 2, kind), injection(dim, N // 4, kind)],
                     bs=bs, coarse_size=10)
    assert [L.A.shape[0] for L in mg.levels[:3]] == [B0.shape[0], mid["ss"][0].shape[0], coarse["ss"][0].shape[0]]
    rng = np.random.default_rng(0)
    b = rng.standard_normal(B0.shape[0])
    A = sp.csr_matrix(B0)
    x = mg(b)
    r1 = np.linalg.norm(b - A @ x)
    for _ in range(9):
        x = x + mg(b - A @ x)
    # stationary V-cycles on the solid block (Dirichlet columns kept, so not symmetric): the residual contracts
    assert np.linalg.norm(b - A @ x) <= 1e-2 * r1
