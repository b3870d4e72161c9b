"""CPU restatement of OUR smoothed-aggregation AMG (TEST INFRASTRUCTURE).

This is NOT hypre BoomerAMG (the reference's `-*_pc_type hypre`, petsc-options-inexact:16-24
and lib/Preconditioner.py:94-100): hypre's source is not in the reference tree and cannot
run here.  It is the numpy/scipy twin of the device AMG in
poroelasticity-linear-solvers_b200/csrc/amg.cu, written with the same deterministic
choices (hash priorities, synchronous Luby rounds, modified Gram-Schmidt per aggregate) so
that both build the same hierarchy and the GPU iteration counts can be compared with it.

Algorithm (per level)
  1. nodal strength graph from Frobenius norms of the bs x bs blocks, threshold theta,
     symmetrised;
  2. MIS(2) roots by synchronous Luby rounds with hashed priorities; distance-1 then
     distance-2 nodes join the aggregate they are most strongly connected to;
  3. tentative prolongator from the near-nullspace B by per-aggregate modified Gram-Schmidt;
  4. P = (I - 4/(3 rho) D^-1 A) T with rho from a deterministic power iteration;
  5. A_c = P^T A P, B_c = stacked R factors; coarse block size = number of modes.
V-cycle: Chebyshev(degree) on D^-1 A over [lmax/ratio, 1.1 lmax], dense solve on the coarsest.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp


def hash32(i: np.ndarray) -> np.ndarray:
    """Deterministic 32-bit mix (same constants in amg.cu)."""
    x = (i.astype(np.uint64) + np.uint64(0x9E3779B9)) & np.uint64(0xFFFFFFFF)
    x = ((x ^ (x >> np.uint64(16))) * np.uint64(0x85EBCA6B)) & np.uint64(0xFFFFFFFF)
    x = ((x ^ (x >> np.uint64(13))) * np.uint64(0xC2B2AE35)) & np.uint64(0xFFFFFFFF)
    x = x ^ (x >> np.uint64(16))
    return x.astype(np.int64)


def rigid_body_modes(coords: np.ndarray, dim: int) -> np.ndarray:
    """Near-nullspace of elasticity for node-blocked dofs; coords (n_dofs, dim) per dof."""
    n = coords.shape[0]
    nn = n // dim
    X = coords[::dim] - coords[::dim].mean(0)
    s = np.abs(X).max() or 1.0
    X = X / s
    if dim == 2:
        B = np.zeros((nn, 2, 3))
        B[:, 0, 0] = 1
        B[:, 1, 1] = 1
        B[:, 0, 2], B[:, 1, 2] = -X[:, 1], X[:, 0]
    else:
        B = np.zeros((nn, 3, 6))
        for c in range(3):
            B[:, c, c] = 1
        B[:, 1, 3], B[:, 2, 3] = -X[:, 2], X[:, 1]      # rotation about x
        B[:, 0, 4], B[:, 2, 4] = X[:, 2], -X[:, 0]      # about y
        B[:, 0, 5], B[:, 1, 5] = -X[:, 1], X[:, 0]      # about z
    return B.reshape(n, -1)


def strength_graph(A: sp.csr_matrix, bs: int, theta: float):
    """Symmetrised nodal strength graph (CSR pattern + weights = block Frobenius norms^2)."""
    nn = A.shape[0] // bs
    C = sp.csr_matrix(A).tocoo()
    # each block's squares summed one after the other in stored order, as amg.cu's segmented combine does: the weights are
    # then bit-equal to the device's, so a tie between neighbours is broken the same way on both sides
    key = (C.row // bs).astype(np.int64) * nn + C.col // bs
    order = np.argsort(key, kind="stable")
    key, sq = key[order], C.data[order] ** 2
    head = np.ones(len(key), bool)
    head[1:] = key[1:] != key[:-1]
    seg = np.cumsum(head) - 1
    start = np.flatnonzero(head)
    w = np.zeros(len(start))
    pos = np.arange(len(key)) - start[seg]
    for t in range(int(pos.max()) + 1 if len(pos) else 0):
        sel = pos == t
        w[seg[sel]] += sq[sel]
    N2 = sp.csr_matrix((w, (key[head] // nn, key[head] % nn)), shape=(nn, nn))
    d = N2.diagonal()
    G = N2.tocoo()
    strong = (G.row != G.col) & (G.data >= theta * theta * np.sqrt(d[G.row] * d[G.col])) & (G.data > 0)
    S = sp.coo_matrix((G.data[strong], (G.row[strong], G.col[strong])), shape=(nn, nn)).tocsr()
    S = S.maximum(S.T).tocsr()
    S.sort_indices()
    return S


def _nbr_max(S, key):
    """max over {i} U N(i) of key (int64), vectorised."""
    out = key.copy()
    rows = np.repeat(np.arange(S.shape[0]), np.diff(S.indptr))
    np.maximum.at(out, rows, key[S.indices])
    return out


def aggregate_mis2(S: sp.csr_matrix):
    """Deterministic MIS(2) aggregation.  Returns (agg (nn,) int, -1 = isolated; n_agg)."""
    nn = S.shape[0]
    deg = np.diff(S.indptr)
    prio = ((hash32(np.arange(nn)) >> 1) << 32) | (np.arange(nn) + 1)   # unique 63-bit key per node, > 0
    UNDEC, IN, OUT = 0, 1, 2
    state = np.where(deg == 0, OUT, UNDEC)
    while (state == UNDEC).any():
        key = np.where(state == UNDEC, prio, 0)
        m1 = _nbr_max(S, key)
        m2 = _nbr_max(S, m1)
        sel = (state == UNDEC) & (m2 == prio)
        state[sel] = IN
        # knock out everything within distance 2 of a selected node
        flag = sel.astype(np.int64)
        f1 = _nbr_max(S, flag)
        f2 = _nbr_max(S, f1)
        state[(state == UNDEC) & (f2 > 0)] = OUT
    roots = np.flatnonzero(state == IN)
    agg = np.full(nn, -1, np.int64)
    agg[roots] = np.arange(len(roots))
    # two joining rounds: pick the neighbour (already aggregated at round start) with the
    # strongest connection; ties -> smallest aggregate id
    for _ in range(2):
        rows = np.repeat(np.arange(nn), deg)
        cols = S.indices
        cand = (agg[rows] < 0) & (agg[cols] >= 0)
        r, w, a = rows[cand], S.data[cand], agg[cols[cand]]
        if len(r) == 0:
            break
        order = np.lexsort((a, -w, r))
        r, a = r[order], a[order]
        first = np.ones(len(r), bool)
        first[1:] = r[1:] != r[:-1]
        new = agg.copy()
        new[r[first]] = a[first]
        agg = new
    return agg, len(roots)


def tentative_prolongator(agg, n_agg, bs, B):
    """Per-aggregate modified Gram-Schmidt of B.  Returns (T csr n x n_agg*k, Bc (n_agg*k, k))."""
    n, k = B.shape
    nn = n // bs
    node_rows = np.arange(n).reshape(nn, bs)
    mem = np.flatnonzero(agg >= 0)
    order = mem[np.argsort(agg[mem], kind="stable")]          # members grouped by aggregate, ascending node id
    a_sorted = agg[order]
    counts = np.bincount(a_sorted, minlength=n_agg)
    start = np.concatenate([[0], np.cumsum(counts)])
    mmax = int(counts.max()) * bs
    pos_in_agg = np.arange(len(order)) - start[a_sorted]
    Q = np.zeros((n_agg, mmax, k))
    rows_of = node_rows[order]                                 # (nmem, bs)
    slot = pos_in_agg[:, None] * bs + np.arange(bs)[None, :]
    Q[a_sorted[:, None], slot, :] = B[rows_of]
    R = np.zeros((n_agg, k, k))
    for j in range(k):
        for i in range(j):
            R[:, i, j] = np.einsum("am,am->a", Q[:, :, i], Q[:, :, j])
            Q[:, :, j] -= R[:, i, j][:, None] * Q[:, :, i]
        # column norm before/after decides rank deficiency
        nrm = np.sqrt(np.einsum("am,am->a", Q[:, :, j], Q[:, :, j]))
        ok = nrm > 1e-8
        R[:, j, j] = np.where(ok, nrm, 0.0)
        Q[:, :, j] = np.where(ok[:, None], Q[:, :, j] / np.where(ok, nrm, 1.0)[:, None], 0.0)
    vals = Q[a_sorted[:, None], slot, :]                       # (nmem, bs, k)
    rr = np.repeat(rows_of.ravel(), k)
    cc = (np.repeat(a_sorted, bs)[:, None] * k + np.arange(k)[None, :]).ravel()
    T = sp.csr_matrix((vals.reshape(-1), (rr, cc)), shape=(n, n_agg * k))
    return T, R.reshape(n_agg * k, k)


def power_lmax(A: sp.csr_matrix, dinv: np.ndarray, its: int = 15) -> float:
    n = A.shape[0]
    v = (hash32(np.arange(n)) % 2048).astype(float) / 1024.0 - 1.0
    v /= np.linalg.norm(v)
    lam = 1.0
    for _ in range(its):
        w = dinv * (A @ v)
        lam = np.linalg.norm(w)
        if lam == 0:
            return 1.0
        v = w / lam
    return lam


class Level:
    pass


class SAAMG:
    post_smooth = True              # False: V(nu, 0) cycle (amg.cu: -*_pc_amg_post_smooth 0)

    def __init__(self, A: sp.csr_matrix, bs: int = 1, B: np.ndarray | None = None, theta: float = 0.08,
                 max_levels: int = 10, coarse_size: int = 400, cheby_degree: int = 2, cheby_ratio: float = 10.0,
                 power_its: int = 15, dense_limit: int = 4096, node_labels: np.ndarray | None = None,
                 local_smoothing: bool = False, post_smooth: bool = True):
        """node_labels (one int per node): aggregates never cross a label boundary ("uncoupled" aggregation
        of a row-partitioned matrix: each rank aggregates its own nodes) while smoothing of P and the Galerkin
        product stay global.  The coarse nodes inherit the label of their aggregate."""
        A = sp.csr_matrix(A)
        labels = None if node_labels is None else np.asarray(node_labels)
        self.level_labels = []
        n = A.shape[0]
        if B is None:
            B = np.zeros((n, bs))
            for c in range(bs):
                B[c::bs, c] = 1.0
        B = B.copy()
        self.levels = []
        self.deg, self.ratio, self.post_smooth = cheby_degree, cheby_ratio, post_smooth
        while True:
            L = Level()
            L.A = A
            d = A.diagonal()
            L.dinv = 1.0 / np.where(d != 0, d, 1.0)
            L.lmax = 1.1 * power_lmax(A, L.dinv, power_its)
            self.levels.append(L)
            n = A.shape[0]
            if n <= coarse_size or len(self.levels) >= max_levels:
                break
            # Dirichlet rows (diagonal only) carry no near-nullspace
            offdiag = np.diff(A.indptr) - (A.diagonal() != 0)
            rowabs = np.abs(A).sum(1).A1 if hasattr(np.abs(A).sum(1), "A1") else np.asarray(np.abs(A).sum(1)).ravel()
            dir_rows = (rowabs - np.abs(d)) <= 1e-14 * np.abs(d)
            B[dir_rows] = 0.0
            S = strength_graph(A, bs, theta)
            if labels is not None:
                G = S.tocoo()
                keep = labels[G.row] == labels[G.col]
                S = sp.coo_matrix((G.data[keep], (G.row[keep], G.col[keep])), shape=S.shape).tocsr()
                S.sort_indices()
            agg, n_agg = aggregate_mis2(S)
            if n_agg == 0 or n_agg * B.shape[1] >= 0.8 * n:
                break
            T, Bc = tentative_prolongator(agg, n_agg, bs, B)
            omega = 4.0 / (3.0 * L.lmax / 1.1)
            if labels is not None and local_smoothing:
                # block-diagonal prolongator (csrc/amg.cu, distributed set-up): rows of the nodes that touch another
                # rank (either direction of the pattern) keep their tentative row, every other row sees only owned
                # columns anyway -> P never leaves its rank; the Galerkin product still uses the full operator
                C = A.tocoo()
                cross = labels[C.row // bs] != labels[C.col // bs]
                bnd = np.zeros(n // bs, bool)
                bnd[C.row[cross] // bs] = True
                bnd[C.col[cross] // bs] = True
                keep_row = np.repeat(~bnd, bs).astype(float)
                P = (T - sp.diags(omega * L.dinv * keep_row) @ (A @ T)).tocsr()
            else:
                P = (T - sp.diags(omega * L.dinv) @ (A @ T)).tocsr()
            Ac = (P.T @ A @ P).tocsr()
            dc = Ac.diagonal()
            dead = dc == 0
            if dead.any():
                Ac = (Ac + sp.diags(dead.astype(float))).tocsr()
            L.P, L.R = P, P.T.tocsr()
            L.agg, L.n_agg = agg, n_agg
            if labels is not None:
                self.level_labels.append(labels)
                mem = agg >= 0
                cl = np.zeros(n_agg, labels.dtype)
                cl[agg[mem]] = labels[mem]
                labels = cl
            A, B, bs = Ac, Bc, B.shape[1]
        if labels is not None:
            self.level_labels.append(labels)
        Lc = self.levels[-1]
        # coarsest level: dense inverse when small (amg.cu: poro_amg_dense_limit), else smoothing only
        self.coarse_direct = Lc.A.shape[0] <= dense_limit
        if self.coarse_direct:
            Lc.inv = np.linalg.inv(Lc.A.toarray())

    def complexity(self):
        return sum(L.A.nnz for L in self.levels) / self.levels[0].A.nnz

    def _cheby(self, L, b, x, zero_guess):
        lmax = L.lmax
        lmin = lmax / self.ratio
        theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
        sigma = theta / delta
        rho = 1.0 / sigma
        r = b.copy() if zero_guess else b - L.A @ x
        dvec = (L.dinv * r) / theta
        for k in range(self.deg):
            x = x + dvec
            if k == self.deg - 1:
                break
            r = r - L.A @ dvec
            rho_new = 1.0 / (2.0 * sigma - rho)
            dvec = rho_new * rho * dvec + (2.0 * rho_new / delta) * (L.dinv * r)
            rho = rho_new
        return x

    def _cycle(self, l, b):
        L = self.levels[l]
        if l == len(self.levels) - 1:
            if self.coarse_direct:
                return L.inv @ b
            x = self._cheby(L, b, np.zeros_like(b), True)
            return x if len(self.levels) == 1 else self._cheby(L, b, x, False)
        x = self._cheby(L, b, np.zeros_like(b), True)
        r = b - L.A @ x
        xc = self._cycle(l + 1, L.R @ r)
        x = x + L.P @ xc
        return self._cheby(L, b, x, False) if self.post_smooth else x

    def __call__(self, b):
        return self._cycle(0, b)
