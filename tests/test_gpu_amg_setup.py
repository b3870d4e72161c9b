"""The device SA-AMG set-up (csrc/amg.cu, csrc/setup.cu) level by level against an extended-precision reference.

`Amg::setup` builds every hierarchy of the iterative option sets as a chain of stages: the nodal strength graph, MIS(2)
aggregation, the tentative prolongator T from per-aggregate modified Gram-Schmidt (`k_mgs`), the Jacobi-smoothed
prolongator P = T - w D^-1 A T, its transpose R and the Galerkin product R (A P), with the Dirichlet zeroing of the
near-nullspace, the power-iteration bound and the dead-coarse-dof patch in between, and the Gauss-Jordan inverse of the
coarsest level.  Each stage is fed the DEVICE's own inputs of its level (exported with `-poro_amg_keep_setup 1`) and its
output is compared with a np.longdouble reference of that one stage, entry by entry, against a rounding bound that holds
for any summation order (u = 2^-53, m = terms in the entry).  Drift between the device and its CPU twin (oracle/amg.py)
compounds level by level; fed its own inputs, a kernel error cannot hide behind it.

Every hierarchy is also rebuilt with one SpGEMM row per chunk and with a budget that splits the largest products into a
few chunks (`-poro_spgemm_chunk`): every exported array must stay bit-identical.  The primitives (`poro_mat_setup_op`,
`poro_dense_inverse`) are tested alone at their edges, and one V-cycle on the device's own levels is compared with the
twin's.  The comparators themselves are shown, without a GPU, to reject planted defects that a norm-wise check accepts."""
import numpy as np
import pytest
import scipy.sparse as sp

U = 2.0 ** -53
LD = np.longdouble
MGS_TOL = 1e-8                    # amg.cu k_mgs: a column whose norm after projection is <= this is dead
DEFAULT_CHUNK = 300_000_000       # setup.cu: -poro_spgemm_chunk default


# ---------------------------------------------------------------------------------------------------------------------
# reference products and comparators (plain numpy / scipy: no GPU needed)
# ---------------------------------------------------------------------------------------------------------------------
def _ones(A):
    """the stored pattern of A with value 1 per stored entry (explicit zeros and duplicates count)"""
    return sp.csr_matrix((np.ones(A.nnz, np.int64), A.indices.copy(), A.indptr.copy()), shape=A.shape)


def _ld(A, absval=False):
    d = np.asarray(A.data, LD)
    return sp.csr_matrix((np.abs(d) if absval else d, A.indices.copy(), A.indptr.copy()), shape=A.shape)


def _canon(M):
    M = sp.csr_matrix(M, copy=True)
    M.sum_duplicates()
    M.sort_indices()
    return M


def _rows(M):
    return np.repeat(np.arange(M.shape[0]), np.diff(M.indptr))


def _at(M, pat):
    """values of M (summed duplicates) at the stored positions of the canonical pattern `pat`, zero where M has none"""
    M = _canon(M)
    km = _rows(M).astype(np.int64) * M.shape[1] + M.indices
    kp = _rows(pat).astype(np.int64) * pat.shape[1] + pat.indices
    out = np.zeros(len(kp), M.dtype)
    if len(km) == 0:
        return out
    pos = np.minimum(np.searchsorted(km, kp), len(km) - 1)
    hit = km[pos] == kp
    out[hit] = M.data[pos[hit]]
    return out


def symbolic(*mats):
    """term counts of the product of the stored patterns (a count per stored entry of the result: never cancels)"""
    C = _ones(mats[0])
    for M in mats[1:]:
        C = _canon(C @ _ones(M))
    return _canon(C)


def assert_pattern(got, want, what):
    """got (device CSR, canonical by construction) has exactly the stored pattern of want"""
    assert got.shape == want.shape, "%s: shape %s, want %s" % (what, got.shape, want.shape)
    rg, rw = np.diff(got.indptr), np.diff(want.indptr)
    bad = np.flatnonzero(rg != rw)
    if len(bad) == 0:
        d = np.flatnonzero(got.indices != want.indices)
        if len(d) == 0:
            return
        bad = [int(np.searchsorted(got.indptr, d[0], side="right") - 1)]
    i = int(bad[0])
    raise AssertionError("%s: pattern differs first in row %d: columns %s, want %s" % (
        what, i, got.indices[got.indptr[i]:got.indptr[i + 1]].tolist(), want.indices[want.indptr[i]:want.indptr[i + 1]].tolist()))


def assert_entries(got, want, bound, what):
    err = np.abs(np.asarray(got, LD) - want)
    bad = np.flatnonzero(~(err <= bound))
    if len(bad):
        j = bad[np.argmax(np.nan_to_num(err[bad] / np.maximum(bound[bad], 1e-300), nan=np.inf))]
        raise AssertionError("%s: %d of %d entries outside the rounding bound; entry %d: got %r, want %r, bound %.3e"
                             % (what, len(bad), len(want), j, got[j], float(want[j]), float(bound[j])))


def check_spgemm(A, B, C, what="spgemm"):
    """C = A B: exact symbolic pattern (cancellations kept), entries within (m + 2) u (|A| |B|)_ij"""
    cnt = symbolic(A, B)
    assert_pattern(C, cnt, what)
    want = _at(_ld(A) @ _ld(B), C)
    absv = _at(_ld(A, True) @ _ld(B, True), C)
    assert_entries(C.data, want, (cnt.data + 2) * U * absv, what)


def check_prolongator(T, A, dinv, lmax, P, what="P"):
    """P = T - w D^-1 A T with w = 4 / (3 lmax / 1.1) as amg.cu computes it; entries within (m + 3) u (|T| + |w D^-1| |A| |T|)"""
    omega = 4.0 / (3.0 * lmax / 1.1)
    cat = symbolic(A, T)
    pat = _canon(_ones(T) + cat)
    assert_pattern(P, pat, what)
    wd = sp.diags(np.asarray(-omega * dinv, LD))
    want = _at(_ld(T), P) + _at(wd @ (_ld(A) @ _ld(T)), P)
    absv = _at(_ld(T, True), P) + _at(abs(wd) @ (_ld(A, True) @ _ld(T, True)), P)
    m = _at(cat, P)
    assert_entries(P.data, want, (m + 3) * U * absv, what)


def check_transpose(P, R, what="R"):
    """R is P^T bit for bit: pattern and values"""
    want = P.T.tocsr()
    want.sort_indices()
    assert_pattern(R, want, what)
    bad = np.flatnonzero(R.data.view(np.int64) != want.data.view(np.int64))
    assert len(bad) == 0, "%s: %d values differ from P^T, first entry %d: %r, want %r" % (what, len(bad), bad[0], R.data[bad[0]],
                                                                                          want.data[bad[0]])


def check_galerkin(R, A, P, Ac, what="A_c"):
    """A_c = R (A P): the symbolic pattern of R A P, entries within (m1 + m2 + 4) u (|R| (|A| |P|))_ij, a dead coarse dof
    (zero column of P) has the unit diagonal; returns the number of dead dofs"""
    cap = symbolic(A, P)
    c2 = symbolic(R, cap)
    assert_pattern(Ac, c2, what)
    want = _at(_ld(R) @ (_ld(A) @ _ld(P)), Ac)
    absv = _at(_ld(R, True) @ (_ld(A, True) @ _ld(P, True)), Ac)
    m1 = int(cap.data.max()) if cap.nnz else 0
    rows = _rows(Ac)
    dead_rows = np.flatnonzero(np.asarray(abs(P).sum(0)).ravel() == 0)
    diag = (rows == Ac.indices) & np.isin(rows, dead_rows)
    want[diag] = 1.0
    assert_entries(Ac.data, want, (m1 + c2.data + 4) * U * absv, what)
    return len(dead_rows)


def dirichlet_rows(A):
    """amg.cu's rule: sum |offdiag| <= 1e-14 |diag|, off-diagonals and diagonal summed in stored order"""
    rows = _rows(A)
    on = rows == A.indices
    d = np.zeros(A.shape[0])
    off = np.zeros(A.shape[0])
    np.add.at(d, rows[on], A.data[on])
    np.add.at(off, rows[~on], np.abs(A.data[~on]))
    return off <= 1e-14 * np.abs(d)


def check_dinv(A, dinv, what="dinv"):
    d = np.zeros(A.shape[0])
    rows = _rows(A)
    on = rows == A.indices
    np.add.at(d, rows[on], A.data[on])
    want = np.where(d != 0, 1.0 / np.where(d != 0, d, 1.0), 1.0)
    bad = np.flatnonzero(want.view(np.int64) != np.asarray(dinv).view(np.int64))
    assert len(bad) == 0, "%s: %d rows differ, row %d: %r, want %r" % (what, len(bad), bad[0], dinv[bad[0]], want[bad[0]])


def check_aggregates(A, bs, theta, agg, what="agg"):
    """integer-equal to oracle aggregate_mis2(strength_graph(A, bs, theta))"""
    from oracle.amg import aggregate_mis2, strength_graph
    S = strength_graph(A, bs, theta)
    want, n_agg = aggregate_mis2(S)
    agg = np.asarray(agg, np.int64)
    bad = np.flatnonzero(agg != want)
    if len(bad):
        i = int(bad[0])
        nb = S.indices[S.indptr[i]:S.indptr[i + 1]]
        cand = ", ".join("node %d w=%r agg %d" % (j, w, want[j]) for j, w in zip(nb, S.data[S.indptr[i]:S.indptr[i + 1]]))
        raise AssertionError("%s: %d of %d nodes differ; first node %d: device %d, oracle %d; candidates: %s"
                             % (what, len(bad), len(agg), i, agg[i], want[i], cand))
    return n_agg


def check_tentative(T, agg, bs, k, B, Bnext_raw, what="T"):
    """T against the QR of each aggregate's near-nullspace B_agg = Q R, with R the next level's stacked factors (before its
    Dirichlet zeroing): the pattern is members x k with explicit zeros, live columns orthonormal, Q R = B_agg, R upper
    triangular with a non-negative diagonal, dead columns zero with a zero R row.  Returns the number of dead columns."""
    agg = np.asarray(agg, np.int64)
    n_agg = T.shape[1] // k
    rows_agg = np.repeat(agg, bs)
    want_cnt = np.where(rows_agg >= 0, k, 0)
    assert np.array_equal(np.diff(T.indptr), want_cnt), "%s: a row does not hold exactly k entries per member" % what
    mem = rows_agg >= 0
    cols = (rows_agg[mem][:, None] * k + np.arange(k)[None, :]).ravel()
    assert np.array_equal(T.indices, cols), "%s: columns are not the k modes of the row's aggregate" % what
    Tv = T.data.reshape(-1, k)
    Bm = B[mem]
    Rall = Bnext_raw.reshape(n_agg, k, k)
    am = rows_agg[mem]
    order = np.argsort(am, kind="stable")
    starts = np.searchsorted(am[order], np.arange(n_agg + 1))
    dead = 0
    from oracle.amg import tentative_prolongator
    Tref, _ = tentative_prolongator(agg, n_agg, bs, B)
    Tref_v = _at(Tref, T)
    for a in range(n_agg):
        idx = order[starts[a]:starts[a + 1]]
        Q, Ba, R = np.asarray(Tv[idx], LD), np.asarray(Bm[idx], LD), np.asarray(Rall[a], LD)
        nb = max(float(np.abs(Ba).max()), 1e-300)
        live = np.diag(Rall[a]) > 0
        assert np.all(np.tril(Rall[a], -1) == 0) and np.all(np.diag(Rall[a]) >= 0), "%s: aggregate %d: R not upper triangular with diagonal >= 0" % (what, a)
        assert np.all(Q[:, ~live] == 0) and np.all(Rall[a][~live] == 0), "%s: aggregate %d: a dead column is not zero" % (what, a)
        dead += int((~live).sum())
        G = Q[:, live].T @ Q[:, live]
        assert np.abs(G - np.eye(int(live.sum()))).max() <= 1e-13, "%s: aggregate %d: live columns not orthonormal" % (what, a)
        assert np.abs(Q @ R - Ba).max() <= 1e-13 * nb, "%s: aggregate %d: Q R != B_agg" % (what, a)
        # the norm each column has after projection on the live columns before it decides live or dead: near the
        # threshold both answers are right and the case proves nothing
        for j in range(k):
            prev = [i for i in range(j) if live[i]]
            res = Ba[:, j] - Q[:, prev] @ (Q[:, prev].T @ Ba[:, j])
            nr = float(np.sqrt(np.sum(res * res)))
            assert not MGS_TOL / 2 < nr < 2 * MGS_TOL, "%s: aggregate %d column %d: norm %.3e within a factor 2 of %g: ambiguous case" % (
                what, a, j, nr, MGS_TOL)
            assert live[j] == (nr > MGS_TOL), "%s: aggregate %d column %d: norm %.3e but %s" % (what, a, j, nr, "live" if live[j] else "dead")
        sv = np.linalg.svd(np.asarray(Bm[idx], float), compute_uv=False)
        if live.all() and sv[-1] > 0 and sv[0] / sv[-1] <= 1e3:
            e = np.abs(Tv[idx] - Tref_v.reshape(-1, k)[idx]).max()
            assert e <= 1e-11, "%s: aggregate %d: %.3e from the oracle's tentative prolongator" % (what, a, e)
    return dead


# ---------------------------------------------------------------------------------------------------------------------
# the chain of one hierarchy
# ---------------------------------------------------------------------------------------------------------------------
EXPORTS = ("A", "P", "R", "T", "agg", "B", "dinv", "inv")


def export(pcc, name):
    """every exported array of every level, {(level, item): array}, and the level infos"""
    out, infos = {}, []
    l = 0
    while True:
        info = pcc.amg_level_info(name, l)
        infos.append(info)
        for w in EXPORTS:
            if w == "inv" and not info["direct"]:
                continue
            if w in ("P", "R", "T", "agg") and (info["coarsest"] or info["geometric"]):
                continue
            if w in ("T", "agg", "B") and not info["kept"]:
                continue
            out[(l, w)] = pcc.amg_level(name, l, w)
        if info["coarsest"]:
            return out, infos
        l += 1


def check_chain(ex, infos, theta, B0=None, name=""):
    """every stage of every algebraic level fed the device's inputs; returns what the hierarchy reached"""
    from oracle.amg import power_lmax
    stats = dict(levels=len(infos), dead=0, coarsest_rows=infos[-1]["A_rows"], direct=bool(infos[-1]["direct"]),
                 chunks=[(i["chunks_AT"], i["chunks_AP"], i["chunks_RAP"]) for i in infos])
    for l, info in enumerate(infos):
        at = "%s level %d" % (name, l)
        A, dinv, lmax = ex[(l, "A")], ex[(l, "dinv")], info["lmax"]
        check_dinv(A, dinv, at + " dinv")
        want = 1.1 * power_lmax(A, dinv)
        assert abs(lmax - want) <= 1e-10 * want, "%s lmax: %r, want %r" % (at, lmax, want)
        B = ex[(l, "B")]
        zero = dirichlet_rows(A) if not info["coarsest"] else np.zeros(A.shape[0], bool)
        assert np.all(B[zero] == 0), at + ": a Dirichlet row of B is not zero"
        if l == 0 and B0 is not None:
            assert np.abs(B[~zero] - B0[~zero]).max() <= 1e-15, at + ": B differs from the oracle's near-nullspace"
        if info["geometric"] or info["coarsest"]:
            continue
        bs, k = info["bs"], info["k"]
        n_agg = check_aggregates(A, bs, theta, ex[(l, "agg")], at + " agg")
        assert n_agg == info["n_agg"], (at, n_agg, info["n_agg"])
        T, P, R, Ac = ex[(l, "T")], ex[(l, "P")], ex[(l, "R")], ex[(l + 1, "A")]
        Bn = ex[(l + 1, "B")]
        # B_{l+1} = stacked R factors with level l+1's Dirichlet rows zeroed: recover the factors from Q^T B_agg where zeroed
        zn = dirichlet_rows(Ac)
        Rf = Bn.copy()
        if zn.any():
            Qt = np.asarray(T.T @ B)
            Rf[zn] = np.where(np.abs(Qt[zn]) <= 1e-13 * max(np.abs(B).max(), 1e-300), 0.0, Qt[zn])
        stats["dead"] += check_tentative(T, ex[(l, "agg")], bs, k, B, Rf, at + " T")
        check_prolongator(T, A, dinv, lmax, P, at + " P")
        check_transpose(P, R, at + " R")
        check_galerkin(R, A, P, Ac, at + " A_%d" % (l + 1))
    if infos[-1]["direct"]:
        Ac, X = ex[(len(infos) - 1, "A")].toarray(), ex[(len(infos) - 1, "inv")]
        check_inverse(Ac, X, name + " coarsest inverse")
    return stats


def check_inverse(A, X, what, ref=None):
    """|| I - A X ||_max <= 4 n u ||A||_inf ||X||_inf and X within a kappa-scaled distance of the inverse"""
    n = A.shape[0]
    an, xn = np.abs(A).sum(1).max(), np.abs(X).sum(1).max()
    res = np.abs(np.eye(n) - A @ X).max()
    assert res <= 4 * n * U * an * xn, "%s: ||I - A X||_max = %.3e > %.3e" % (what, res, 4 * n * U * an * xn)
    Xr = np.linalg.inv(A) if ref is None else ref
    kappa = an * xn
    e = np.abs(X - Xr).max()
    assert e <= 4 * n * U * kappa * np.abs(Xr).max(), "%s: %.3e from the inverse (kappa %.2e)" % (what, e, kappa)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the comparators reject planted defects
# ---------------------------------------------------------------------------------------------------------------------
def _reference_level(A, bs, B, theta=0.08):
    """one level computed the way the device computes it (fp64 rounding of the longdouble stages, exact patterns)"""
    from oracle.amg import aggregate_mis2, power_lmax, strength_graph, tentative_prolongator
    d = A.diagonal()
    dinv = 1.0 / np.where(d != 0, d, 1.0)
    lmax = 1.1 * power_lmax(A, dinv)
    agg, n_agg = aggregate_mis2(strength_graph(A, bs, theta))
    T, _ = tentative_prolongator(agg, n_agg, bs, B)
    omega = 4.0 / (3.0 * lmax / 1.1)
    pat = _canon(_ones(T) + symbolic(A, T))
    Pv = _at(_ld(T), pat) + _at(sp.diags(np.asarray(-omega * dinv, LD)) @ (_ld(A) @ _ld(T)), pat)
    P = sp.csr_matrix((np.asarray(Pv, float), pat.indices, pat.indptr), shape=pat.shape)
    R = P.T.tocsr()
    R.sort_indices()
    cp = symbolic(R, symbolic(A, P))
    Acv = _at(_ld(R) @ (_ld(A) @ _ld(P)), cp)
    Ac = sp.csr_matrix((np.asarray(Acv, float), cp.indices, cp.indptr), shape=cp.shape)
    return dict(agg=agg, T=T, dinv=dinv, lmax=lmax, P=P, R=R, Ac=Ac)


def test_comparators_reject_planted_defects():
    from oracle.amg import aggregate_mis2, rigid_body_modes, strength_graph
    from oracle.problems import swelling
    s, _ = swelling(2, 6, "diagonal")
    A = sp.csr_matrix(s.P)[s.is_s][:, s.is_s].tocsr()
    A.sort_indices()
    B = rigid_body_modes(s.coords_s, 2)
    ref = _reference_level(A, 2, B)
    T, P, R, Ac, dinv, lmax = ref["T"], ref["P"], ref["R"], ref["Ac"], ref["dinv"], ref["lmax"]
    # the clean data passes every check
    check_aggregates(A, 2, 0.08, ref["agg"])
    check_prolongator(T, A, dinv, lmax, P)
    check_transpose(P, R)
    check_galerkin(R, A, P, Ac)

    def norm_wise_ok(got, want):
        return np.linalg.norm(got - want) <= 1e-12 * np.linalg.norm(want)

    # 1. one dropped term in one Galerkin entry: the entry of the row with the smallest scale
    AP = _ld(A) @ _ld(P)
    rows = _rows(Ac)
    scale = _at(_ld(R, True) @ (_ld(A, True) @ _ld(P, True)), Ac)
    j = int(np.argmin(np.where((rows == Ac.indices) | (scale == 0), np.inf, scale)))
    i, c = rows[j], Ac.indices[j]
    Rr = R.getrow(i)
    q = Rr.indices[np.argmax(np.abs(Rr.data) * np.abs(np.asarray(AP[Rr.indices, c].todense(), float).ravel()))]
    bad = Ac.copy()
    bad.data[j] = float(LD(Ac.data[j]) - LD(R[i, q]) * AP[q, c])
    with pytest.raises(AssertionError, match="outside the rounding bound"):
        check_galerkin(R, A, P, bad)
    accepted = ["dropped Galerkin term"] if norm_wise_ok(bad.toarray(), Ac.toarray()) else []
    # 2. a flipped tie-break in aggregate_mis2's joining round: the largest aggregate id wins a tie instead of the smallest
    S = strength_graph(A, 2, 0.08)
    good, _ = aggregate_mis2(S)
    flipped = _flipped_tiebreak(S)
    assert not np.array_equal(flipped, good), "no tie in the joining rounds of this mesh"
    with pytest.raises(AssertionError, match="nodes differ"):
        check_aggregates(A, 2, 0.08, flipped)
    # 3. the wrong sign of omega
    Pbad = _reference_level(A, 2, B)["P"]
    Pbad.data = np.asarray(_at(_ld(T), Pbad) - (_at(_ld(P), Pbad) - _at(_ld(T), Pbad)), float)
    with pytest.raises(AssertionError, match="outside the rounding bound"):
        check_prolongator(T, A, dinv, lmax, Pbad)
    # 4. a transposed R with one swapped value
    #    (the two neighbours in one row whose values differ least: invisible norm-wise)
    Rbad = R.copy()
    same_row = _rows(Rbad)[1:] == _rows(Rbad)[:-1]
    gap = np.where(same_row, np.abs(np.diff(Rbad.data)), np.inf)
    a = int(np.argmin(np.where(gap > 0, gap, np.inf)))
    Rbad.data[[a, a + 1]] = Rbad.data[[a + 1, a]]
    with pytest.raises(AssertionError, match="values differ"):
        check_transpose(P, Rbad)
    if norm_wise_ok(Rbad.toarray(), R.toarray()):
        accepted.append("swapped R value")
    assert accepted, "a 1e-12 norm-wise check rejects every planted defect: the case shows nothing"


def _flipped_tiebreak(S):
    """aggregate_mis2 with its joining rounds preferring the LARGEST aggregate id on a weight tie"""
    from oracle import amg
    orig = np.lexsort
    try:
        def lexsort(keys):
            a, w, r = keys
            return orig((-a, w, r))
        np.lexsort = lexsort
        return amg.aggregate_mis2(S)[0]
    finally:
        np.lexsort = orig


def test_strength_weights_are_summed_in_stored_order():
    """oracle strength_graph sums each block's squares one after the other in stored order, as the device does"""
    from oracle.amg import strength_graph
    v = np.array([1e16, 1.0, -1e16, 1.0])                    # squares 1e32, 1, 1e32, 1: order-dependent sums
    A = sp.csr_matrix((v, ([0, 0, 1, 1], [2, 3, 2, 3])), shape=(4, 4)) + sp.eye(4) * 1e17
    A = sp.csr_matrix(A)
    A.sort_indices()
    S = strength_graph(A, 2, 0.0)
    seq = 0.0
    for x in sp.csr_matrix(A)[0:2, 2:4].toarray().ravel():
        seq = seq + x * x if seq else x * x
    assert S[0, 1] == seq


# ---------------------------------------------------------------------------------------------------------------------
# GPU: hierarchies of the solver's blocks
# ---------------------------------------------------------------------------------------------------------------------
def _amg_options(theta, coarse, extra=""):
    from helpers import AMG_OPTIONS
    o = AMG_OPTIONS
    for p in ("s_", "fp_fieldsplit_0_", "fp_fieldsplit_1_"):
        o += "-%spc_amg_theta %g\n-%spc_amg_coarse_size %d\n" % (p, theta, p, coarse)
    return o + "-poro_amg_keep_setup 1\n" + extra


def _build(ctx, sys_, options):
    from poro_b200.lib.backend import DeviceMatrix
    from poro_b200.lib.IndexSet import IndexSet
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    ctx.clear_options()
    load_petsc_options(ctx, options, is_text=True)
    par = {"pc type": "diagonal", "inner ksp type": "preonly", "inner pc type": "hypre", "inner rtol": 1e-6, "inner atol": 1e-6,
           "inner maxiter": 100, "inner accel order": 0, "inner monitor": False}
    imap = IndexSet(sys_.is_s, sys_.is_f, sys_.is_p, two_way=True, block_dim=sys_.dim, coords_s=sys_.coords_s, coords_p=sys_.coords_p)
    keep = (DeviceMatrix(sys_.A, ctx), DeviceMatrix(sys_.P, ctx))
    pc = Preconditioner(imap, keep[0], keep[1], None, par, sys_.bcs_sub_pressure).get_pc()
    return pc.getPythonContext(), keep


def chunk_count(counts, budget):
    """setup.cu csr_spgemm's host split of the rows under a product budget"""
    hoff = np.concatenate([[0], np.cumsum(counts)])
    n, r0, parts = len(counts), 0, 0
    while r0 < n:
        r1 = int(np.searchsorted(hoff[r0 + 1:], hoff[r0] + budget, side="right")) + r0
        r1 = min(max(r1, r0 + 1), n)
        parts, r0 = parts + 1, r1
    return parts


def _product_rows(A, B):
    return np.asarray(_ones(A) @ np.diff(B.indptr)).ravel()


def _level_products(ex, infos):
    """per algebraic level the per-row product counts of A T, A P and R (A P)"""
    out = {}
    for l, info in enumerate(infos):
        if info["geometric"] or info["coarsest"]:
            continue
        A, T, P, R = ex[(l, "A")], ex[(l, "T")], ex[(l, "P")], ex[(l, "R")]
        AP = symbolic(A, P)
        out[l] = (_product_rows(A, T), _product_rows(A, P), _product_rows(R, AP))
    return out


def _assert_same(ex1, ex2, what):
    assert ex1.keys() == ex2.keys(), what
    for key, a in ex1.items():
        b = ex2[key]
        if sp.issparse(a):
            same = (a.shape == b.shape and np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
                    and np.array_equal(a.data.view(np.int64), b.data.view(np.int64)))
        else:
            same = np.array_equal(np.asarray(a).view(np.int64) if a.dtype == np.float64 else a,
                                  np.asarray(b).view(np.int64) if b.dtype == np.float64 else b)
        assert same, "%s: %s of level %d differs" % (what, key[1], key[0])


def _budget_for(products):
    """a budget under which A T, A P and R (A P) of level 0 each split into several chunks (replica of the host split): 2..5
    for all three where one budget allows it, otherwise (3D: R (A P) has over 5x the products of A T) A T in 2..5 and the
    others in as few as that leaves"""
    tot = [int(c.sum()) for c in products[0]]
    mx = max(int(c.max()) for c in products[0])
    cands = sorted({t // d + e for t in tot for d in (2, 3, 4, 5) for e in (0, 1)})
    ok = [b for b in cands if b >= mx and all(chunk_count(c, b) >= 2 for c in products[0]) and chunk_count(products[0][0], b) <= 5]
    assert ok, "no budget splits each of A T, A P and R (A P) of level 0: totals %s" % tot
    return min(ok, key=lambda b: max(chunk_count(c, b) for c in products[0]))


SWELLING_CASES = {
    # name: (dim, N, theta, coarse size, extra options, expected edge)
    "2d_theta008": (2, 24, 0.08, 16, "", "levels"),
    "2d_theta004_nondirect": (2, 24, 0.04, 16, "-poro_amg_dense_limit 0\n", "nondirect"),
    "3d_theta008_big_coarse": (3, 6, 0.08, 400, "", "coarse>256"),
    "3d_theta004": (3, 6, 0.04, 10, "", "levels"),
    "2d_max_levels": (2, 24, 0.08, 1, "-s_pc_amg_max_levels 3\n-fp_fieldsplit_0_pc_amg_max_levels 3\n-fp_fieldsplit_1_pc_amg_max_levels 3\n", "max_levels"),
    "2d_ratio_stop": (2, 12, 0.08, 1, "", "ratio"),
}
REACHED = {}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SWELLING_CASES))
def test_swelling_hierarchy_stages(gpu_ctx, case):
    from oracle.amg import rigid_body_modes
    from oracle.problems import swelling
    dim, N, theta, coarse, extra, edge = SWELLING_CASES[case]
    sys_, _ = swelling(dim, N, "diagonal")
    opts = _amg_options(theta, coarse, extra)
    pcc, keep = _build(gpu_ctx, sys_, opts)
    results = {}
    for name in ("s", "fp0", "fp1"):
        ex, infos = export(pcc, name)
        B0 = rigid_body_modes(np.asarray(sys_.coords_s), dim) if name == "s" else None
        if B0 is not None and infos[0]["k"] != B0.shape[1]:
            B0 = None
        results[name] = (ex, infos, check_chain(ex, infos, theta, B0, "%s %s" % (case, name)))
    st = {n: r[2] for n, r in results.items()}
    if edge == "levels":
        assert st["s"]["levels"] >= 4, st["s"]
    elif edge == "nondirect":
        assert st["s"]["levels"] >= 4 and not st["s"]["direct"], st["s"]
    elif edge == "coarse>256":
        assert any(v["direct"] and v["coarsest_rows"] > 256 for v in st.values()), st
    elif edge == "max_levels":
        assert st["s"]["levels"] == 3 and st["s"]["coarsest_rows"] > 1, st["s"]
    elif edge == "ratio":
        # stopped by the 0.8 coarsening ratio, above a coarse size of 1: the next level would keep >= 0.8 of the rows
        last = results["s"][1][-1]
        assert last["A_rows"] > 1 and st["s"]["levels"] < 10, st["s"]
    REACHED[case] = {n: dict(levels=v["levels"], dead=v["dead"], coarsest=v["coarsest_rows"], direct=v["direct"]) for n, v in st.items()}
    # rebuilt with one row per SpGEMM chunk and with a budget that splits level 0's products into 2..5 chunks: bit-identical
    products = _level_products(*results["s"][:2])
    budget = _budget_for(products)
    for opt, tag in (("1", "one row per chunk"), (str(budget), "budget %d" % budget), (None, "second default set-up")):
        pc2, keep2 = _build(gpu_ctx, sys_, opts + ("-poro_spgemm_chunk %s\n" % opt if opt else ""))
        for name in ("s", "fp0", "fp1"):
            ex2, infos2 = export(pc2, name)
            _assert_same(results[name][0], ex2, "%s %s, %s" % (case, name, tag))
            if name == "s":
                b = DEFAULT_CHUNK if opt is None else int(opt)
                for l, cnts in _level_products(ex2, infos2).items():
                    got = (infos2[l]["chunks_AT"], infos2[l]["chunks_AP"], infos2[l]["chunks_RAP"])
                    assert got == tuple(chunk_count(c, b) for c in cnts), (case, tag, l, got)
                    if l == 0 and opt == str(budget):
                        assert all(g >= 2 for g in got) and got[0] <= 5, got
                        REACHED[case]["chunks"] = got
        pc2.destroy()
    pcc.destroy()


@pytest.mark.gpu
def test_dead_dof_reached():
    """across the swelling cases at least one rank-deficient aggregate gave a dead coarse dof (runs after them)"""
    if not REACHED:
        pytest.skip("run with the hierarchy cases")
    print("levels, dead coarse dofs, coarsest rows, direct, level-0 chunks per case:", REACHED)
    assert any(v["dead"] > 0 for c in REACHED.values() for k, v in c.items() if k != "chunks"), REACHED


@pytest.mark.gpu
@pytest.mark.parametrize("mg_levels", [1, 2])
def test_generated_hierarchy_stages(gpu_ctx, mg_levels):
    """a generated 3D system (level 0 carries a stencil descriptor) with the benchmarked options and a low coarse size; with
    mg_levels 2 the solid and velocity blocks are `pc_type mg` and the algebraic levels below get the same checks"""
    import bench
    from hostfem.mg import injection
    from poro_b200.generator import generate_swelling3d
    from poro_b200.lib.Parser import load_petsc_options
    from poro_b200.lib.Preconditioner import Preconditioner
    N = 8
    opts = bench.BENCH_OPTIONS.replace("coarse_size 6000", "coarse_size 40") + "-poro_amg_keep_setup 1\n"
    if mg_levels > 1:
        opts = opts.replace("-s_pc_type hypre", "-s_pc_type mg").replace("-fp_fieldsplit_0_pc_type hypre", "-fp_fieldsplit_0_pc_type mg")
    gpu_ctx.clear_options()
    load_petsc_options(gpu_ctx, opts, is_text=True)
    g = generate_swelling3d(gpu_ctx, N, "diagonal", mg_levels=mg_levels)
    pcc = Preconditioner(g.index_set(), g.A, g.P, None, dict(g.par), g.bcs_sub_pressure).get_pc().getPythonContext()
    for name, theta in (("s", 0.04), ("fp0", 0.04), ("fp1", 0.08)):
        ex, infos = export(pcc, name)
        st = check_chain(ex, infos, theta, None, "generated %s" % name)
        assert st["levels"] >= 3, (name, st)
        if mg_levels > 1 and name in ("s", "fp0"):
            assert infos[0]["geometric"] and not infos[1]["geometric"]
            # the near-nullspace injected at the coinciding nodes, bit for bit, then zeroed on level 1's Dirichlet rows
            inj = injection(3, N // 2, 2)
            inj_dofs = (np.asarray(inj)[:, None] * 3 + np.arange(3)[None, :]).ravel()
            Bf, Bc = ex[(0, "B")], ex[(1, "B")]
            z = dirichlet_rows(ex[(1, "A")])
            want = Bf[inj_dofs]
            want[z] = 0.0
            assert np.array_equal(Bc.view(np.int64), want.view(np.int64)), name


def _twin_from_levels(ex, infos, deg, post_smooth):
    from oracle.amg import SAAMG, Level
    tw = SAAMG.__new__(SAAMG)
    tw.deg, tw.ratio, tw.post_smooth = deg, 10.0, bool(post_smooth)
    tw.levels = []
    for l, info in enumerate(infos):
        L = Level()
        L.A, L.dinv, L.lmax = ex[(l, "A")], ex[(l, "dinv")], info["lmax"]
        if not info["coarsest"]:
            L.P, L.R = ex[(l, "P")], ex[(l, "R")]
        tw.levels.append(L)
    tw.coarse_direct = bool(infos[-1]["direct"])
    if tw.coarse_direct:
        tw.levels[-1].inv = ex[(len(infos) - 1, "inv")]
    return tw


@pytest.mark.gpu
@pytest.mark.parametrize("direct", [True, False])
@pytest.mark.parametrize("post_smooth", [0, 1])
@pytest.mark.parametrize("deg", [1, 2, 4])
def test_vcycle_matches_twin_on_device_levels(gpu_ctx, deg, post_smooth, direct):
    """one V-cycle (restriction, prolongation with SPMV_ADD, coarse k_gemv or Chebyshev, multi-level Chebyshev) of s, fp0 and
    fp1 against SAAMG._cycle loaded with the device's own levels"""
    import torch
    from oracle.problems import swelling
    sys_, _ = swelling(2, 16, "diagonal")
    extra = "-pc_amg_cheby_degree %d\n-pc_amg_post_smooth %d\n" % (deg, post_smooth) + ("" if direct else "-poro_amg_dense_limit 0\n")
    pcc, keep = _build(gpu_ctx, sys_, _amg_options(0.08, 30, extra))
    for name in ("s", "fp0", "fp1"):
        ex, infos = export(pcc, name)
        assert len(infos) >= (3 if name == "s" else 2) and bool(infos[-1]["direct"]) == direct, (name, len(infos))
        tw = _twin_from_levels(ex, infos, deg, post_smooth)
        r = np.random.default_rng(deg).standard_normal(infos[0]["A_rows"])
        rt = torch.tensor(r, device="cuda")
        zt = torch.full_like(rt, float("nan"))
        pcc.inner_solve(name, rt, zt)
        torch.cuda.synchronize()
        z, want = zt.cpu().numpy(), tw(r)
        assert np.abs(z - want).max() <= 1e-12 * np.abs(want).max(), (name, np.abs(z - want).max() / np.abs(want).max())
    pcc.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the primitives alone
# ---------------------------------------------------------------------------------------------------------------------
def _upload(ctx, A):
    from poro_b200._capi import Mat
    A = sp.csr_matrix(A)
    return Mat(ctx, A.indptr, A.indices, A.data, A.shape)


def _noncanonical(A, seed):
    """each entry split into two copies, columns shuffled within rows (how FEM assembly hands a CSR over)"""
    rng = np.random.default_rng(seed)
    A = _canon(A)
    rows, cols, vals = _rows(A), A.indices, A.data
    f = rng.uniform(0.25, 0.75, len(vals))
    r2, c2, v2 = np.concatenate([rows, rows]), np.concatenate([cols, cols]), np.concatenate([vals * f, vals - vals * f])
    o = np.lexsort((rng.random(len(r2)), r2))
    return sp.csr_matrix((v2[o], c2[o], np.concatenate([[0], np.cumsum(np.bincount(r2, minlength=A.shape[0]))])), shape=A.shape)


def _rand(rng, m, n, density, empty_rows=()):
    A = sp.random(m, n, density=density, format="csr", random_state=rng, data_rvs=lambda k: rng.standard_normal(k))
    A = A.tolil()
    for i in empty_rows:
        A.rows[i], A.data[i] = [], []
    return _canon(A.tocsr())


def _spgemm_cases():
    rng = np.random.default_rng(11)
    cases = {}
    A = _rand(rng, 300, 200, 0.03, empty_rows=range(40, 90))
    cases["zero_rows"] = (A, _rand(rng, 200, 150, 0.05))
    cases["all_rows_empty"] = (sp.csr_matrix((50, 40)), _rand(rng, 40, 30, 0.2))
    B = _rand(rng, 200, 150, 0.05, empty_rows=range(0, 200, 3))
    cases["empty_b_rows_referenced"] = (_rand(rng, 120, 200, 0.05), B)
    a = sp.csr_matrix(np.array([[1.0, 1.0, 0.0], [0.0, 2.0, -2.0], [3.0, 0.0, 0.0]]))
    b = sp.csr_matrix(np.array([[1.0, 2.0], [-1.0, -2.0], [-1.0, -2.0]]))
    cases["cancel_to_zero"] = (a, b)
    cases["duplicates"] = (_noncanonical(_rand(rng, 150, 120, 0.06), 1), _noncanonical(_rand(rng, 120, 90, 0.06), 2))
    cases["rectangular_wide"] = (_rand(rng, 20, 500, 0.05), _rand(rng, 500, 900, 0.01))
    for m in (20,):
        for n in (1 << m, (1 << m) + 1):
            Ar = sp.csr_matrix((np.array([1.5, -2.0]), np.array([0, n - 1]), np.r_[np.zeros(n, np.int64), [2]]), shape=(n, n))
            Br = sp.csr_matrix((np.array([3.0, 0.5, 7.0]), np.array([n - 1, 0, n - 1]), np.r_[[0, 2], np.full(n - 1, 3)]), shape=(n, n))
            cases["last_row_only_%d" % n] = (Ar, Br)
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_spgemm_cases()))
def test_spgemm_edges(gpu_ctx, case):
    A, B = _spgemm_cases()[case]
    cnt = _product_rows(A, B)
    total = int(cnt.sum())
    prefix = np.cumsum(cnt)
    budgets = {DEFAULT_CHUNK}
    if total > 0:
        mid = int(prefix[np.searchsorted(prefix, total // 2)])
        budgets |= {mid, max(mid - 1, 1), mid + 1, 1, max(int(cnt.max()) - 1, 1)}
        empty = np.flatnonzero(cnt == 0)
        if len(empty):                                             # a boundary inside a run of empty rows
            budgets.add(max(int(prefix[empty[len(empty) // 2]]), 1))
    da, db = _upload(gpu_ctx, A), _upload(gpu_ctx, B)
    first = None
    for budget in sorted(budgets):
        gpu_ctx.clear_options()
        gpu_ctx.set_option("-poro_spgemm_chunk", budget)
        m, chunks = da.setup_op(db, "spgemm")
        C = m.to_scipy()
        m.destroy()
        assert chunks == chunk_count(cnt, budget), (case, budget, chunks, chunk_count(cnt, budget))
        if first is None:
            check_spgemm(A, B, C, "%s budget %d" % (case, budget))
            first = C
        else:
            _assert_same({(0, "C"): first}, {(0, "C"): C}, "%s budget %d" % (case, budget))
    gpu_ctx.clear_options()
    if total > 1 and cnt.max() > 1:
        gpu_ctx.set_option("-poro_spgemm_chunk", int(cnt.max()) - 1)       # a single row over the budget is its own chunk
        m, chunks = da.setup_op(db, "spgemm")
        assert chunks == chunk_count(cnt, int(cnt.max()) - 1) and chunks >= 2
        m.destroy()
        gpu_ctx.clear_options()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(300, 200), (1 << 20, 7), (7, 1 << 20), ((1 << 20) + 1, (1 << 20) + 1)])
def test_transpose_exact(gpu_ctx, shape):
    rng = np.random.default_rng(3)
    m, n = shape
    if m * n > 10 ** 6:
        rows = np.sort(rng.integers(0, m, 500))
        rows[-1] = m - 1
        A = _canon(sp.csr_matrix((rng.standard_normal(500), (rows, rng.integers(0, n, 500))), shape=shape))
    else:
        A = _noncanonical(_rand(rng, m, n, 0.05), 4)
    m_, _ = _upload(gpu_ctx, A).setup_op(None, "transpose")
    At = m_.to_scipy()
    want = _canon(A).T.tocsr()
    want.sort_indices()
    if A.nnz == _canon(A).nnz:
        check_transpose(_canon(A), At, "transpose %s" % (shape,))
    else:        # duplicates are summed by the transpose's combine
        assert_pattern(At, want, "transpose %s" % (shape,))
        assert_entries(At.data, np.asarray(want.data, LD), 2 * U * np.abs(np.asarray(want.data, LD)), "transpose %s" % (shape,))


@pytest.mark.gpu
def test_add_scaled(gpu_ctx):
    import torch
    rng = np.random.default_rng(5)
    A = _noncanonical(_rand(rng, 400, 300, 0.04), 6)
    B = _noncanonical(_rand(rng, 400, 300, 0.04), 7)
    s = rng.standard_normal(400)
    alpha = -0.37
    for sv in (s, None):
        st = torch.tensor(sv, device="cuda") if sv is not None else None
        m, chunks = _upload(gpu_ctx, A).setup_op(_upload(gpu_ctx, B), "add_scaled", alpha, st)
        C = m.to_scipy()
        sc = np.asarray(alpha * (sv if sv is not None else np.ones(400)), LD)
        pat = _canon(_ones(A) + _ones(B))
        assert_pattern(C, pat, "add_scaled")
        want = _at(_ld(A), C) + _at(sp.diags(sc) @ _ld(B), C)
        absv = _at(_ld(A, True), C) + _at(abs(sp.diags(sc)) @ _ld(B, True), C)
        m = _at(_canon(_ones(A) + _ones(B)), C)
        assert_entries(C.data, want, (m + 2) * U * absv, "add_scaled")


def _ld_inverse(A):
    """Gauss-Jordan with partial pivoting in np.longdouble"""
    n = A.shape[0]
    M = np.concatenate([np.asarray(A, LD), np.eye(n, dtype=LD)], 1)
    for k in range(n):
        p = k + int(np.argmax(np.abs(M[k:, k])))
        M[[k, p]] = M[[p, k]]
        M[k] /= M[k, k]
        f = M[:, k].copy()
        f[k] = 0
        M -= np.outer(f, M[k])
    return np.asarray(M[:, n:], float)


def _gj_cases():
    rng = np.random.default_rng(9)
    cases = {}
    for n in (1, 2, 31, 32, 33, 255, 256, 257, 1000):
        A = rng.standard_normal((n, n))
        A += np.diag(np.abs(A).sum(1) + 1.0)
        cases["dd_%d" % n] = A
    perm = np.roll(np.arange(300), 1)
    cases["permutation_300"] = np.eye(300)[perm] * rng.uniform(1, 2, 300)[:, None]
    H = np.array([[1.0]])
    while H.shape[0] < 256:
        H = np.block([[H, H], [H, -H]])
    cases["hadamard_256"] = H
    A = rng.standard_normal((100, 100)) + np.diag(np.full(100, 30.0))
    dead = [0, 17, 63, 99]
    A[dead] = 0
    A[:, dead] = 0
    A[dead, dead] = 1.0
    cases["identity_rows"] = A
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_gj_cases()))
def test_dense_inverse(gpu_ctx, case):
    A = _gj_cases()[case]
    X = gpu_ctx.dense_inverse(A)
    n = A.shape[0]
    if case == "hadamard_256":
        assert np.array_equal(X, A.T / 256), "Hadamard: every pivot candidate ties; the inverse must be H^T / 256 exactly"
    ref = _ld_inverse(A) if n <= 400 else None
    check_inverse(A, X, case, ref)
    if case == "identity_rows":
        for d in (0, 17, 63, 99):
            assert X[d, d] == 1.0 and np.count_nonzero(X[d]) == 1 and np.count_nonzero(X[:, d]) == 1
