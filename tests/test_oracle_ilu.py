"""CPU tests of the ILU(0) and fieldsplit twins (tests/ilu_twin.py) that the GPU tests of `-<prefix>pc_type ilu` and of
`-fp_pc_fieldsplit_type additive | multiplicative` compare against."""
import numpy as np
import pytest
import scipy.sparse as sp

from ilu_twin import ILU0, FieldSplit, level_sets


def _lu_nopivot(A):
    A = np.array(A, dtype=np.float64)
    n = A.shape[0]
    for k in range(n):
        A[k + 1:, k] /= A[k, k]
        A[k + 1:, k + 1:] -= np.outer(A[k + 1:, k], A[k, k + 1:])
    return np.tril(A, -1) + np.eye(n), np.triu(A)


def _closed_patterns():
    rng = np.random.default_rng(3)
    n = 40
    tri = sp.diags([rng.uniform(-1, 0, n - 1), rng.uniform(3, 4, n), rng.uniform(-1, 0, n - 1)], [-1, 0, 1], format="csr")
    blocks = [rng.standard_normal((5, 5)) + 6 * np.eye(5) for _ in range(6)]
    bd = sp.block_diag([sp.csr_matrix(b) for b in blocks], format="csr")
    return [tri, bd]


@pytest.mark.parametrize("k", [0, 1])
def test_closed_pattern_equals_lu(k):
    A = _closed_patterns()[k]
    L, U = ILU0(A).factors()
    Le, Ue = _lu_nopivot(A.toarray())
    assert np.abs(L.toarray() - Le).max() <= 1e-14 * np.abs(Le).max()
    assert np.abs(U.toarray() - Ue).max() <= 1e-14 * np.abs(Ue).max()
    x = np.random.default_rng(1).standard_normal(A.shape[0])
    assert np.linalg.norm(ILU0(A)(x) - np.linalg.solve(A.toarray(), x)) <= 1e-13 * np.linalg.norm(np.linalg.solve(A.toarray(), x))


def _blocks(dim, N):
    from hostfem.problems import swelling
    s, _ = swelling(dim, N, pc_type="diagonal")
    P = sp.csr_matrix(s.P)
    return {nm: P[idx][:, idx].tocsr() for nm, idx in (("ss", s.is_s), ("ff", s.is_f), ("pp", s.is_p), ("fp", s.is_fp))}


@pytest.mark.parametrize("dim,N", [(2, 8), (3, 4)])
def test_generated_blocks_factor_on_pattern(dim, N):
    for nm, B in _blocks(dim, N).items():
        L, U = ILU0(B).factors()
        LU = (L @ U).tocsr()
        rows, cols = np.repeat(np.arange(B.shape[0]), np.diff(B.indptr)), B.indices
        got = np.asarray(LU[rows, cols]).ravel()
        ref = B.data
        assert np.abs(got - ref).max() <= 1e-13 * np.abs(ref).max(), nm


def _check_topological(B, upper):
    ptr, rows = level_sets(B, upper)
    lev = np.empty(B.shape[0], np.int64)
    for l in range(len(ptr) - 1):
        lev[rows[ptr[l]:ptr[l + 1]]] = l
    assert sorted(rows.tolist()) == list(range(B.shape[0]))
    r = np.repeat(np.arange(B.shape[0]), np.diff(B.indptr))
    dep = B.indices > r if upper else B.indices < r
    assert np.all(lev[r[dep]] > lev[B.indices[dep]])
    return len(ptr) - 1


# lower level counts of the stored patterns, natural ordering (hostfem, `diagonal` splitting)
LEVELS = {(2, 16): dict(ss=159, ff=157, pp=33, fp=159), (3, 4): dict(ss=150, ff=132, pp=13, fp=135)}


@pytest.mark.parametrize("dim,N", sorted(LEVELS))
def test_level_sets(dim, N):
    for nm, B in _blocks(dim, N).items():
        assert _check_topological(B, False) == LEVELS[(dim, N)][nm], nm
        _check_topological(B, True)


def test_refusals():
    # a stored zero on the diagonal: the pattern keeps it, and the pivot is 0 - 1/2 * 1 = -0.5
    A = sp.csr_matrix((np.array([2.0, 1.0, 1.0, 0.0, 1.0, 1.0, 2.0]), np.array([0, 1, 0, 1, 2, 1, 2]), np.array([0, 2, 5, 7])),
                      shape=(3, 3))
    ILU0(A)
    with pytest.raises(ZeroDivisionError, match="row 0"):
        ILU0(A, zeropivot=1e300)
    B = sp.csr_matrix(np.array([[2.0, 1.0], [1.0, 0.0]]))
    B.eliminate_zeros()
    with pytest.raises(ValueError, match="row 1"):
        ILU0(B)


@pytest.mark.parametrize("first", ["p", "f"])
def test_fieldsplit_twin(first):
    rng = np.random.default_rng(5)
    nf, npp = 7, 4
    M = rng.standard_normal((nf + npp, nf + npp)) + 8 * np.eye(nf + npp)
    exact = lambda B: (lambda x, D=B.toarray(): np.linalg.solve(D, x))
    i0 = nf + np.arange(npp) if first == "p" else np.arange(nf)
    i1 = np.arange(nf) if first == "p" else nf + np.arange(npp)
    perm = np.concatenate([i0, i1])
    Mb = M[np.ix_(perm, perm)]
    n0 = len(i0)
    D = np.zeros_like(Mb); D[:n0, :n0] = Mb[:n0, :n0]; D[n0:, n0:] = Mb[n0:, n0:]
    T = D.copy(); T[n0:, :n0] = Mb[n0:, :n0]
    x = rng.standard_normal(nf + npp)
    for typ, ref in (("additive", D), ("multiplicative", T)):
        fs = FieldSplit(typ, sp.csr_matrix(M), nf, npp, exact, exact, first)
        y = fs(x)
        yr = np.empty_like(x)
        yr[perm] = np.linalg.solve(ref, x[perm])
        assert np.linalg.norm(y - yr) <= 1e-13 * np.linalg.norm(yr), typ
