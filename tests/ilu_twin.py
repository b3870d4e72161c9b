"""Numpy twins of the device ILU(0) (csrc/ilu.cu) and of PETSc's additive / multiplicative fieldsplit on the fp block
(PCSchur with type additive / multiplicative), for the tests of those features.

The ILU twin factors exactly the stored pattern of the CSR it is given, explicit zeros included: build it from
`PreconditionerCC.block(name)`, which keeps them (scipy arithmetic on blocks can drop stored zeros)."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

ZEROPIVOT = 2.220446049250313e-14      # the device default of -<prefix>pc_factor_zeropivot


def level_sets(M, upper=False):
    """(ptr, rows): level(i) = 1 + max level(j) over the stored j < i (j > i for upper), 0 without such j; rows grouped
    contiguously per level, ascending inside a level."""
    M = sp.csr_matrix(M)
    n = M.shape[0]
    ip, ix = M.indptr, M.indices
    lev = np.zeros(n, np.int64)
    order = range(n - 1, -1, -1) if upper else range(n)
    for i in order:
        c = ix[ip[i]:ip[i + 1]]
        c = c[c > i] if upper else c[c < i]
        lev[i] = lev[c].max() + 1 if len(c) else 0
    nlev = int(lev.max()) + 1 if n else 0
    ptr = np.zeros(nlev + 1, np.int64)
    np.add.at(ptr, lev + 1, 1)
    return np.cumsum(ptr), np.argsort(lev, kind="stable")


class ILU0:
    """ILU(0) in natural order (IKJ) on the stored pattern; y = U^-1 L^-1 x with unit-diagonal L.  Refuses a missing
    diagonal and a pivot with |u_ii| <= zeropivot, naming the row."""

    def __init__(self, M, zeropivot=ZEROPIVOT):
        M = sp.csr_matrix(M)
        M.sort_indices()
        n = M.shape[0]
        ip, ix = M.indptr, M.indices
        F = M.data.astype(np.float64).copy()
        diag = np.full(n, -1, np.int64)
        for i in range(n):
            hit = np.nonzero(ix[ip[i]:ip[i + 1]] == i)[0]
            if not len(hit):
                raise ValueError("row %d of the block has no stored diagonal entry" % i)
            diag[i] = ip[i] + hit[0]
        for i in range(n):
            cols = ix[ip[i]:ip[i + 1]]
            for q in range(ip[i], diag[i]):
                k = ix[q]
                F[q] = F[q] / F[diag[k]]
                ks = slice(diag[k] + 1, ip[k + 1])
                kc, kv = ix[ks], F[ks]
                pos = np.searchsorted(cols, kc)
                ok = (pos < len(cols)) & (cols[np.minimum(pos, len(cols) - 1)] == kc)
                F[ip[i] + pos[ok]] -= F[q] * kv[ok]
            if not abs(F[diag[i]]) > zeropivot:
                raise ZeroDivisionError("zero pivot in row %d (|u_ii| = %.6e)" % (i, abs(F[diag[i]])))
        self.n = n
        rows = np.repeat(np.arange(n), np.diff(ip))
        lower, upper = ix < rows, ix > rows
        self.L = sp.csr_matrix((F[lower], ix[lower], np.concatenate([[0], np.cumsum(np.bincount(rows[lower], minlength=n))])),
                               shape=(n, n))
        self.U = sp.csr_matrix((F[upper], ix[upper], np.concatenate([[0], np.cumsum(np.bincount(rows[upper], minlength=n))])),
                               shape=(n, n))
        self.d = F[diag]

    def factors(self):
        """(unit-lower L, upper U with its diagonal) as CSR."""
        n = self.n
        return (self.L + sp.identity(n, format="csr")).tocsr(), (self.U + sp.diags(self.d)).tocsr()

    def __call__(self, x):
        if not hasattr(self, "_LU"):
            L, U = self.factors()
            self._LU = (L.tocsr(), U.tocsr())
        L, U = self._LU
        y = spla.spsolve_triangular(L, np.asarray(x, np.float64), lower=True, unit_diagonal=True)
        return spla.spsolve_triangular(U, y, lower=False)


class FieldSplit:
    """PETSc's 2-split PCFIELDSPLIT on the fp block [f | p] with K1 built on A11 (no Schur complement):
        additive:        y0 = K0 x0 ;  y1 = K1 x1
        multiplicative:  y0 = K0 x0 ;  y1 = K1 (x1 - A10 y0)
    first = 'p' (the reference's order pf) or 'f'.  make_k0 / make_k1: CSR block -> callable."""

    def __init__(self, type, Mfp_fp, nf, npp, make_k0, make_k1, first="p"):
        if type not in ("additive", "multiplicative"):
            raise ValueError("fieldsplit type %r" % type)
        Mfp_fp = sp.csr_matrix(Mfp_fp)
        f, p = np.arange(nf), nf + np.arange(npp)
        i0, i1 = (p, f) if first == "p" else (f, p)
        self.type, self.nf, self.first = type, nf, first
        self.A00 = Mfp_fp[i0][:, i0].tocsr()
        self.A10 = Mfp_fp[i1][:, i0].tocsr()
        self.A11 = Mfp_fp[i1][:, i1].tocsr()
        self.k0, self.k1 = make_k0(self.A00), make_k1(self.A11)

    @classmethod
    def from_blocks(cls, type, A00, A10, A11, nf, make_k0, make_k1, first="p"):
        """The same from the split blocks (e.g. the device's, which keep their explicit zeros)."""
        fs = cls.__new__(cls)
        fs.type, fs.nf, fs.first = type, nf, first
        fs.A00, fs.A10, fs.A11 = sp.csr_matrix(A00), sp.csr_matrix(A10), sp.csr_matrix(A11)
        fs.k0, fs.k1 = make_k0(fs.A00), make_k1(fs.A11)
        return fs

    def split0(self, x0):
        return self.k0(x0)

    def split1(self, x1):
        return self.k1(x1)

    def __call__(self, x):
        xf, xp = x[: self.nf], x[self.nf:]
        x0, x1 = (xp, xf) if self.first == "p" else (xf, xp)
        y0 = self.k0(x0)
        y1 = self.k1(x1 if self.type == "additive" else x1 - self.A10 @ y0)
        yf, yp = (y1, y0) if self.first == "p" else (y0, y1)
        return np.concatenate([yf, yp])
