"""The symbolic analysis of the device sparse LU (csrc/lu_symbolic.h, plain C++) run on the CPU through a g++ harness, on the
inner blocks of the oracle's problems: the ordering is a permutation, the supernodal structure holds the exact fill of the
factorisation (checked against a dense Cholesky of an SPD matrix with the pattern of B + B^T), amalgamation stays cheap, and
the ordering is a nested dissection (fill ~ n log n), not a band (fill ~ n N).  The numeric factorisation and the solves are
tested on the GPU in tests/test_gpu_sparse_lu.py."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "poroelasticity-linear-solvers_b200", "csrc")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("lusym") / "lusym_harness.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + CSRC,
                    os.path.join(ROOT, "tests", "lu_symbolic_harness.cpp"), "-o", out], check=True)
    lib = C.CDLL(out)
    lib.lusym_analyse.restype = C.c_void_p
    lib.lusym_analyse.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
    lib.lusym_sizes.argtypes = [C.c_void_p, C.c_void_p]
    lib.lusym_copy.argtypes = [C.c_void_p] + [C.c_void_p] * 6
    lib.lusym_free.argtypes = [C.c_void_p]
    return lib


def analyse(lib, B):
    B = sp.csr_matrix(B)
    n = B.shape[0]
    rp, ci = np.ascontiguousarray(B.indptr, np.int64), np.ascontiguousarray(B.indices, np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    h = lib.lusym_analyse(n, vp(rp), vp(ci))
    assert h, "analysis failed"
    try:
        sz = np.zeros(8, np.int64)
        lib.lusym_sizes(h, vp(sz))
        ns = int(sz[1])
        out = dict(n=int(sz[0]), nsuper=ns, nlevels=int(sz[2]), nnz_l=int(sz[4]), nnz_u=int(sz[5]), zeros=int(sz[6]),
                   max_front=int(sz[7]))
        out["perm"] = np.zeros(n, np.int32)
        out["first"] = np.zeros(ns + 1, np.int32)
        out["parent"] = np.zeros(ns, np.int32)
        out["row_ptr"] = np.zeros(ns + 1, np.int64)
        out["row_idx"] = np.zeros(int(sz[3]), np.int32)
        out["level"] = np.zeros(ns, np.int32)
        lib.lusym_copy(h, *(vp(out[k]) for k in ("perm", "first", "parent", "row_ptr", "row_idx", "level")))
    finally:
        lib.lusym_free(h)
    return out


def blocks(sys_, pc_type):
    P = sp.csr_matrix(sys_.P)
    sub = lambda M, idx: M[idx][:, idx].tocsr()
    if "3-way" in pc_type:
        return {"s": sub(P, sys_.is_s), "f": sub(P, sys_.is_f), "p": sub(P, sys_.is_p),
                "diff": sub(sp.csr_matrix(sys_.P_diff), sys_.is_p)}
    return {"s": sub(P, sys_.is_s), "fp": sub(P, np.concatenate([sys_.is_f, sys_.is_p]))}


def problem(name, dim, N, pc_type):
    from oracle import problems
    return problems.swelling(dim, N, pc_type)[0] if name == "swelling" else problems.footing(N, pc_type)[0]


CASES = [("swelling", 2, 6, "diagonal"), ("swelling", 2, 10, "diagonal"), ("swelling", 2, 8, "diagonal 3-way"),
         ("swelling", 2, 6, "undrained"), ("footing", 2, 6, "undrained"), ("swelling", 3, 3, "diagonal"),
         ("swelling", 3, 3, "diagonal 3-way")]


@pytest.mark.parametrize("name,dim,N,pc_type", CASES)
def test_structure_holds_the_exact_fill(harness, name, dim, N, pc_type):
    rng = np.random.default_rng(3)
    for blk, B in blocks(problem(name, dim, N, pc_type), pc_type).items():
        n = B.shape[0]
        s = analyse(harness, B)
        perm = s["perm"]
        assert np.array_equal(np.sort(perm), np.arange(n)), blk
        first, rows = s["first"], s["row_idx"]
        assert first[0] == 0 and first[-1] == n and np.all(np.diff(first) > 0)
        # an SPD matrix with the pattern of B + B^T: generic values, diagonally dominant
        pat = (abs(B) + abs(B).T).tocoo()
        off = pat.row != pat.col
        vals = rng.uniform(0.5, 1.5, off.sum())
        M = sp.coo_matrix((vals, (pat.row[off], pat.col[off])), shape=(n, n)).tocsr()
        M = M + M.T
        M = M + sp.diags(np.asarray(abs(M).sum(axis=1)).ravel() + 1.0)
        L = np.linalg.cholesky(M.toarray()[np.ix_(perm, perm)])
        fill = np.abs(L) > 1e-300
        allowed = np.zeros((n, n), bool)
        for t in range(s["nsuper"]):
            R = rows[s["row_ptr"][t]:s["row_ptr"][t + 1]]
            k = first[t + 1] - first[t]
            assert np.array_equal(R[:k], np.arange(first[t], first[t + 1]))
            assert np.all(np.diff(R[k:]) > 0) and (k == len(R) or R[k] >= first[t + 1])
            allowed[np.ix_(R, np.arange(first[t], first[t + 1]))] = True
            p = s["parent"][t]
            if p >= 0:
                assert s["level"][p] > s["level"][t]
                assert set(R[k:].tolist()) <= set(rows[s["row_ptr"][p]:s["row_ptr"][p + 1]].tolist())
            else:
                assert k == len(R)
        allowed = np.tril(allowed)
        assert not np.any(fill & ~allowed), (blk, int(np.sum(fill & ~allowed)))
        # the reported explicit zeros are exactly what the structure stores beyond the true fill
        true_lu = 2 * int(np.tril(fill, -1).sum()) + n
        assert s["nnz_l"] + s["nnz_u"] - s["zeros"] == true_lu, blk
        assert s["zeros"] <= 0.5 * true_lu, (blk, s["zeros"], true_lu)


def test_nested_dissection_not_a_band(harness):
    """2D s block: nnz(L+U) grows like n log n under refinement (x 4.5 from N = 40 to 80), a band would grow x 7.9."""
    from oracle import problems
    nnz = {}
    for N in (40, 80):
        sys_, _ = problems.swelling(2, N, "diagonal")
        s = analyse(harness, blocks(sys_, "diagonal")["s"])
        nnz[N] = s["nnz_l"] + s["nnz_u"]
        assert s["zeros"] <= 0.5 * (nnz[N] - s["zeros"])
    assert nnz[80] / nnz[40] <= 5.5, nnz
