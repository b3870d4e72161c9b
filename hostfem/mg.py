"""Geometric transfer between the structured meshes at N/2 and N, and a CPU twin of `-<prefix>pc_type mg`.

The prolongation of one field is its coarse basis (P2 or P1 Lagrange) evaluated at the fine nodes, on the coarse simplex
that contains each node.  The simplices are taken from `unit_square_mesh` / `unit_cube_mesh` themselves, so no orientation
is assumed here; csrc/mg_transfer.h states the same operator as class tables and is checked against this one.

With P~ = diag(1 - bc_fine) P diag(1 - bc_coarse) (per-dof Dirichlet flags) and R~ = P~^T, the block the generator builds at
N/2 equals R~ B_N P~ on the free rows and columns: the meshes are nested, the coefficients constant, and a free coarse basis
function vanishes on every Dirichlet face.  `GeometricMG` is the V-cycle of csrc/amg.cu on such levels with the SA-AMG of
oracle.amg below the coarsest one.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from .fem import local_edges, unit_cube_mesh, unit_square_mesh


def _lattice(dim: int, L: int) -> np.ndarray:
    """(L^dim, dim) integer lattice coordinates, axis 0 fastest (the node numbering of hostfem.stencil)."""
    return np.stack(np.meshgrid(*[np.arange(L)] * dim, indexing="ij"), -1).reshape(-1, dim)[:, ::-1]


def _node_id(X: np.ndarray, L: int) -> np.ndarray:
    return sum(X[:, m].astype(np.int64) * L ** m for m in range(X.shape[1]))


def prolongation(dim: int, Nc: int, kind: int) -> sp.csr_matrix:
    """Scalar prolongation from the level with Nc cells per side to 2 Nc: kind 2 = P2 lattice, kind 1 = P1 lattice."""
    mesh = (unit_square_mesh if dim == 2 else unit_cube_mesh)(Nc, 1.0)
    M = 4 if kind == 2 else 2                                # fine lattice steps per coarse cell
    Lf, Lc = M * Nc + 1, (2 * Nc + 1) if kind == 2 else (Nc + 1)
    Xf = _lattice(dim, Lf)
    cube = np.minimum(Xf // M, Nc - 1)                       # a coarse cell containing the node
    cube_id = _node_id(cube, Nc)
    ntypes = len(mesh.cells) // Nc ** dim                    # simplices per cell, stored type-major
    best, best_lam, best_cell = np.full(len(Xf), -np.inf), None, None
    for t in range(ntypes):
        cells = mesh.cells[t * Nc ** dim + cube_id]          # (n, dim + 1) vertex ids
        V = mesh.vlat[cells].astype(float) * M               # vertex positions in fine lattice units
        T = np.transpose(V[:, 1:] - V[:, :1], (0, 2, 1))
        lam_rest = np.linalg.solve(T, (Xf - V[:, 0])[..., None])[..., 0]
        lam = np.concatenate([1.0 - lam_rest.sum(1, keepdims=True), lam_rest], 1)
        lam = np.round(lam * M) / M                          # barycentric coordinates of lattice nodes are multiples of 1/M
        score = lam.min(1)
        take = score > best
        best = np.where(take, score, best)
        best_lam = lam if best_lam is None else np.where(take[:, None], lam, best_lam)
        best_cell = cells if best_cell is None else np.where(take[:, None], cells, best_cell)
    assert (best >= 0).all(), "a fine node lies in no coarse simplex"
    vl = mesh.vlat[best_cell]                                # (n, dim + 1, dim) coarse vertex lattice coordinates
    rows, cols, vals = [], [], []
    fine = np.arange(len(Xf))
    if kind == 1:
        for i in range(dim + 1):
            rows.append(fine); cols.append(_node_id(vl[:, i], Lc)); vals.append(best_lam[:, i])
    else:
        for i in range(dim + 1):
            rows.append(fine); cols.append(_node_id(2 * vl[:, i], Lc)); vals.append(best_lam[:, i] * (2 * best_lam[:, i] - 1))
        for i, j in local_edges(dim):
            rows.append(fine); cols.append(_node_id(vl[:, i] + vl[:, j], Lc)); vals.append(4 * best_lam[:, i] * best_lam[:, j])
    r, c, v = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    keep = v != 0.0
    return sp.csr_matrix((v[keep], (r[keep], c[keep])), shape=(len(Xf), Lc ** dim))


def masked_prolongation(dim: int, Nc: int, kind: int, bs: int, bc_fine, bc_coarse) -> sp.csr_matrix:
    """P~ = diag(1 - bc_fine) (P (x) I_bs) diag(1 - bc_coarse) for node-blocked dofs (dof = bs * node + component)."""
    P = sp.kron(prolongation(dim, Nc, kind), sp.identity(bs), format="csr")
    keep_f = 1.0 - np.asarray(bc_fine, float).ravel() if bc_fine is not None else np.ones(P.shape[0])
    keep_c = 1.0 - np.asarray(bc_coarse, float).ravel() if bc_coarse is not None else np.ones(P.shape[1])
    P = (sp.diags(keep_f) @ P @ sp.diags(keep_c)).tocsr()
    P.eliminate_zeros()
    return P


def injection(dim: int, Nc: int, kind: int) -> np.ndarray:
    """Fine node of every coarse node (fine lattice index = 2 x coarse)."""
    Lc = (2 * Nc + 1) if kind == 2 else (Nc + 1)
    Lf = (4 * Nc + 1) if kind == 2 else (2 * Nc + 1)
    return _node_id(2 * _lattice(dim, Lc), Lf)


class GeometricMG:
    """CPU twin of `-<prefix>pc_type mg` (csrc/amg.cu): geometric levels (operators `blocks`, finest first, transfers
    P~_l between blocks[l] and blocks[l + 1]) on top of oracle.amg.SAAMG built on the coarsest block with the fine
    near-nullspace injected at the coinciding nodes.  The same Chebyshev smoother, hashed power iteration and V-cycle."""

    def __init__(self, blocks, transfers, inject, bs: int = 1, B=None, theta: float = 0.08, max_levels: int = 10,
                 coarse_size: int = 400, cheby_degree: int = 2, cheby_ratio: float = 10.0, power_its: int = 15,
                 dense_limit: int = 4096):
        from oracle.amg import SAAMG, Level, power_lmax
        n = blocks[0].shape[0]
        if B is None:
            B = np.zeros((n, bs))
            for c in range(bs):
                B[c::bs, c] = 1.0
        B = np.array(B, float)
        geo = []
        for l, P in enumerate(transfers):
            A = sp.csr_matrix(blocks[l])
            L = Level()
            L.A = A
            d = A.diagonal()
            L.dinv = 1.0 / np.where(d != 0, d, 1.0)
            L.lmax = 1.1 * power_lmax(A, L.dinv, power_its)
            L.P, L.R = P, P.T.tocsr()
            geo.append(L)
            rowabs = np.asarray(np.abs(A).sum(1)).ravel()
            B[(rowabs - np.abs(d)) <= 1e-14 * np.abs(d)] = 0.0
            rows = (bs * inject[l][:, None] + np.arange(bs)[None, :]).ravel()
            B = B[rows]
        self.tail = SAAMG(blocks[-1], bs, B, theta=theta, max_levels=max_levels, coarse_size=coarse_size, cheby_degree=cheby_degree,
                          cheby_ratio=cheby_ratio, power_its=power_its, dense_limit=dense_limit)
        self.tail.levels = geo + self.tail.levels
        self.levels = self.tail.levels

    def __call__(self, b):
        return self.tail(b)
