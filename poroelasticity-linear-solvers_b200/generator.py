"""Device-side generation of a rank's z-slab of the structured-mesh systems (SURVEY 8 f1).

The reference assembles A, P, P_diff on the host with FEniCS (lib/Assembler.py:66-221), partitions with ParMETIS
(swelling-3d.py:7) and applies the Dirichlet conditions each step (lib/Poromechanics.py:76-83).  For dolfin's
UnitCubeMesh the assembled blocks are class stencils of ONE macro-cell matrix (hostfem/stencil.py), so each rank can
generate the rows of its slab of nodes directly in HBM (csrc/gen.cu: poro_gen_matrix) -- the host never holds a matrix,
which is what the >= 50 M-DoF configuration needs.  This module holds the host logic around the kernel:

  * `SlabLayout`: the analytic row partition (contiguous planes of the P2 / P1 lattices per rank), the local numbering
    [s | f | p | ghosts of rank-1: s f p | ghosts of rank+1: s f p], index sets and the halo plan -- the same contract as
    `partition.distributed_problem` (which assembles on the host and is kept as the cross-check);
  * `generate_system`: macro-cell tables from the element matrices (host, one cell), matrices on the device, right-hand
    side, boundary flags, coordinates.

The element matrices of the single macro cell come from hostfem (the stand-in for FEniCS); everything of size O(n) that
touches a matrix runs on the GPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _capi
from .partition import HaloPlan, slab_ranges


class _GenTable(C.Structure):
    _fields_ = [("kr", C.c_int), ("kc", C.c_int), ("br", C.c_int), ("bc", C.c_int), ("diag_block", C.c_int), ("ncls", C.c_int),
                ("cls_ptr", C.c_void_p), ("off", C.c_void_p), ("vals", C.c_void_p)]


@dataclass
class SlabLayout:
    dim: int
    N: int
    rank: int
    world: int
    # node ranges per lattice (index 0: P1, 1: P2): owned, lower ghost, upper ghost
    owned: list = field(default_factory=list)
    ghost_lo: list = field(default_factory=list)
    ghost_up: list = field(default_factory=list)
    # owned P2 planes [a, b); default: the even split of slab_ranges (a coarse level takes them from its fine level)
    p2_planes: tuple | None = None

    def __post_init__(self):
        d, N = self.dim, self.N
        assert d == 3, "slab layout is implemented for the structured cube"
        L2, L1 = 2 * N + 1, N + 1
        a, b = self.p2_planes if self.p2_planes is not None else slab_ranges(L2, self.world)[self.rank]
        assert b - a >= 2, "a z-slab needs at least two P2 planes"
        pa, pb = (a + 1) // 2, (b + 1) // 2                       # owned P1 planes: 2 zp in [a, b)
        lo, up = self.rank > 0, self.rank < self.world - 1
        s2, s1 = L2 * L2, L1 * L1
        self.planes2, self.planes1 = (a, b), (pa, pb)
        self.owned = [(pa * s1, pb * s1), (a * s2, b * s2)]
        self.ghost_lo = [((pa - 1) * s1, pa * s1) if lo else (0, 0), ((a - 2) * s2, a * s2) if lo else (0, 0)]
        self.ghost_up = [(pb * s1, (pb + 1) * s1) if up else (0, 0), (b * s2, min(L2, b + 2) * s2) if up else (0, 0)]
        # what the neighbours read from this rank (their ghost ranges, by the same rule)
        self.send_lo = [(pa * s1, (pa + 1) * s1) if lo else (0, 0), (a * s2, (a + 2) * s2) if lo else (0, 0)]
        self.send_up = [((pb - 1) * s1, pb * s1) if up else (0, 0), ((b - 2) * s2, b * s2) if up else (0, 0)]
        if up:
            # the upper neighbour's lower ghost range starts two planes below ITS first plane (= b)
            assert self.send_up[1][0] >= self.owned[1][0], "slab thinner than the halo"
        kind = [1, 1, 0]                                         # lattice index of s, f, p
        bdim = [d, d, 1]
        n = lambda r: r[1] - r[0]
        self.n_field = [n(self.owned[kind[f]]) * bdim[f] for f in range(3)]
        self.off_owned = [0, self.n_field[0], self.n_field[0] + self.n_field[1]]
        self.n_owned = sum(self.n_field)
        self.ngl = [n(self.ghost_lo[kind[f]]) * bdim[f] for f in range(3)]
        self.ngu = [n(self.ghost_up[kind[f]]) * bdim[f] for f in range(3)]
        o = self.n_owned
        self.off_gl = [o, o + self.ngl[0], o + self.ngl[0] + self.ngl[1]]
        o += sum(self.ngl)
        self.off_gu = [o, o + self.ngu[0], o + self.ngu[0] + self.ngu[1]]
        self.n_ext = o + sum(self.ngu)
        self.kind, self.bdim = kind, bdim
        self.n2, self.n1 = L2 ** d, L1 ** d
        self.n_global = 2 * d * self.n2 + self.n1

    def coarsen(self) -> "SlabLayout":
        """This rank's slab of the mesh at N/2 nested in this one: coarse P2 plane k is fine P2 plane 2k, so the coarse slab
        owns the coarse planes [ceil(a/2), ceil(b/2)).  Ghosts, index sets and halo plan follow by the usual rules."""
        assert self.N % 2 == 0, "the mesh at N/2 needs an even N"
        a, b = self.planes2
        return SlabLayout(self.dim, self.N // 2, self.rank, self.world, p2_planes=((a + 1) // 2, (b + 1) // 2))

    # ---- the arrays the C ABI wants ---------------------------------------------------------------------
    def layout_array(self) -> np.ndarray:
        v = []
        for k in (0, 1):
            v += [*self.owned[k], *self.ghost_lo[k], *self.ghost_up[k]]
        v += self.off_owned + self.off_gl + self.off_gu + [self.n_ext]
        return np.asarray(v, dtype=np.int64)

    def index_sets(self):
        """Positions of the s, f, p dofs in the local extended vector (owned first)."""
        out = []
        for f in range(3):
            out.append(np.concatenate([self.off_owned[f] + np.arange(self.n_field[f], dtype=np.int64),
                                       self.off_gl[f] + np.arange(self.ngl[f], dtype=np.int64),
                                       self.off_gu[f] + np.arange(self.ngu[f], dtype=np.int64)]))
        return out

    def _local_of_range(self, f: int, node_range) -> np.ndarray:
        """Local indices of the dofs of field f on the OWNED nodes node_range (ascending)."""
        k, bd = self.kind[f], self.bdim[f]
        o0 = self.owned[k][0]
        a, b = node_range
        return self.off_owned[f] + np.arange((a - o0) * bd, (b - o0) * bd, dtype=np.int64)

    def halo_plan(self) -> HaloPlan:
        neigh, send_ptr, send_idx, recv = [], [0], [], []
        for nb, send, ng in ((self.rank - 1, self.send_lo, self.ngl), (self.rank + 1, self.send_up, self.ngu)):
            if nb < 0 or nb >= self.world:
                continue
            idx = np.concatenate([self._local_of_range(f, send[self.kind[f]]) for f in range(3)])
            neigh.append(nb)
            send_idx.append(idx)
            send_ptr.append(send_ptr[-1] + len(idx))
            recv.append(sum(ng))
        return HaloPlan(self.n_owned, np.asarray(neigh, np.int32), np.asarray(send_ptr, np.int64),
                        np.concatenate(send_idx).astype(np.int32) if send_idx else np.zeros(0, np.int32),
                        np.asarray(recv, np.int64), self.ext_global()[self.n_owned:])

    def owned_global(self) -> np.ndarray:
        """Global (field-major, hostfem) ids of the owned dofs in local order."""
        d = self.dim
        base = [0, d * self.n2, 2 * d * self.n2]
        return np.concatenate([base[f] + np.arange(self.owned[self.kind[f]][0] * self.bdim[f], self.owned[self.kind[f]][1] * self.bdim[f],
                                                   dtype=np.int64) for f in range(3)])

    def ext_global(self) -> np.ndarray:
        d = self.dim
        base = [0, d * self.n2, 2 * d * self.n2]
        parts = [self.owned_global()]
        for gh in (self.ghost_lo, self.ghost_up):
            for f in range(3):
                r = gh[self.kind[f]]
                parts.append(base[f] + np.arange(r[0] * self.bdim[f], r[1] * self.bdim[f], dtype=np.int64))
        return np.concatenate(parts)


def _tables(gen, which: str, pc_type: str):
    """The 9 class-stencil tables (row-major over s, f, p) of one operator; keeps the arrays alive."""
    d = gen.dim
    shape = {"22": (2, 2, d, d), "21": (2, 1, d, 1), "12": (1, 2, 1, d), "11": (1, 1, 1, 1)}
    local = gen.cell.field_blocks(which, pc_type)
    arr = (_GenTable * 9)()
    keep = []
    for i, fr in enumerate("sfp"):
        for j, fc in enumerate("sfp"):
            kind, data = local[fr + fc]
            K = gen.cell._to_csr(kind, data).toarray()
            kr, kc, br, bc = shape[kind]
            t = arr[3 * i + j]
            t.kr, t.kc, t.br, t.bc, t.diag_block = kr, kc, br, bc, int(fr == fc)
            if not K.any():
                t.ncls, t.cls_ptr, t.off, t.vals = 0, None, None, None
                continue
            cls_ptr, off, vals = gen.table_arrays(K, kr, kc, br, bc)
            cls_ptr = np.ascontiguousarray(cls_ptr, np.int32)
            off = np.ascontiguousarray(off, np.int64)
            vals = np.ascontiguousarray(vals, np.float64)
            keep += [cls_ptr, off, vals]
            t.ncls = len(cls_ptr) - 1
            t.cls_ptr, t.off, t.vals = cls_ptr.ctypes.data, off.ctypes.data, vals.ctypes.data
    return arr, keep


class GeneratedMatrix:
    """A poro_mat produced on the device; quacks like backend.DeviceMatrix for Solver / Preconditioner."""

    def __init__(self, ctx, handle, shape):
        self.ctx, self._h, self.shape = ctx, handle, shape
        r, c, z = C.c_int64(), C.c_int64(), C.c_int64()
        _capi.check(ctx.lib.poro_mat_info(handle, C.byref(r), C.byref(c), C.byref(z)))
        self.nnz = z.value

    def mat(self):
        return self

    @property
    def handle(self):
        return self._h

    def mult(self, x, y):
        from .lib.backend import _tensor
        _capi.check(self.ctx.lib.poro_mat_mult(self._h, _capi._ptr(_tensor(x)), _capi._ptr(_tensor(y))))

    def to_scipy(self):
        import scipy.sparse as sp
        rp, ci, v = np.zeros(self.shape[0] + 1, np.int64), np.zeros(self.nnz, np.int32), np.zeros(self.nnz, np.float64)
        _capi.check(self.ctx.lib.poro_mat_copy(self._h, _capi._ptr(rp), _capi._ptr(ci), _capi._ptr(v)))
        return sp.csr_matrix((v, ci, rp), shape=self.shape)

    def destroy(self):
        if self._h:
            self.ctx.lib.poro_mat_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def generate_matrix(ctx, gen, layout: SlabLayout, which: str, pc_type: str, bc_flags: np.ndarray | None) -> GeneratedMatrix:
    tables, keep = _tables(gen, which, pc_type)
    lay = layout.layout_array()
    flags = None if bc_flags is None else np.ascontiguousarray(bc_flags, dtype=np.uint8)
    h = C.c_void_p()
    _capi.check(ctx.lib.poro_gen_matrix(ctx.h, gen.dim, gen.N, tables, _capi._ptr(lay), _capi._ptr(flags), C.byref(h)))
    del keep
    return GeneratedMatrix(ctx, h, (layout.n_owned, layout.n_ext))


@dataclass
class GeneratedSystem:
    dim: int
    A: GeneratedMatrix
    P: GeneratedMatrix
    P_diff: GeneratedMatrix | None
    b: np.ndarray
    is_s: np.ndarray
    is_f: np.ndarray
    is_p: np.ndarray
    bcs_sub_pressure: np.ndarray
    coords_s: np.ndarray
    coords_p: np.ndarray
    owned_global: np.ndarray
    plan: HaloPlan
    layout: SlabLayout
    n_global: int
    par: dict

    def index_set(self):
        from .lib.IndexSet import IndexSet
        return IndexSet(self.is_s, self.is_f, self.is_p, two_way=True, block_dim=self.dim, coords_s=self.coords_s,
                        coords_p=self.coords_p)


class WholeLayout:
    """Single-rank layout of the whole unit square or cube: every node owned, no ghosts, fields [s | f | p]."""

    def __init__(self, dim: int, N: int):
        L2, L1 = 2 * N + 1, N + 1
        self.dim, self.N = dim, N
        self.n2, self.n1 = L2 ** dim, L1 ** dim
        self.n_field = [dim * self.n2, dim * self.n2, self.n1]
        self.off_owned = [0, self.n_field[0], self.n_field[0] + self.n_field[1]]
        self.n_owned = self.n_ext = sum(self.n_field)

    def layout_array(self) -> np.ndarray:
        o = self.n_owned
        return np.asarray([0, self.n1, 0, 0, 0, 0, 0, self.n2, 0, 0, 0, 0, *self.off_owned, o, o, o, o, o, o, o], np.int64)


def _check_mg_levels(N: int, mg_levels: int, world: int = 1):
    if mg_levels < 1:
        raise ValueError("mg_levels must be at least 1, got %d" % mg_levels)
    if N % (1 << (mg_levels - 1)):
        raise ValueError("N = %d is not divisible by 2^(mg_levels - 1) = %d" % (N, 1 << (mg_levels - 1)))
    if world > 1 and mg_levels > 1:
        # every rank's slab must keep the two P2 planes a slab needs on every level
        L2 = 2 * N + 1
        for rank, (a, b) in enumerate(slab_ranges(L2, world)):
            if b - a < 2:
                raise ValueError("rank %d owns %d P2 plane(s) of the mesh at N = %d: a slab needs at least 2" % (rank, b - a, N))
            for lev in range(1, mg_levels):
                a, b = (a + 1) // 2, (b + 1) // 2
                if b - a < 2:
                    raise ValueError("mg_levels = %d: on level %d (N = %d) rank %d would own %d P2 plane(s) of %d ranks' slabs; a "
                                     "slab needs at least 2 (use fewer levels or fewer ranks)" % (mg_levels, lev, N >> lev, rank, b - a, world))


def max_mg_levels(N: int, world: int = 1) -> int:
    """The most geometric levels N allows: halving while N stays even and, on `world` ranks, every slab keeps 2 P2 planes."""
    lev = 1
    while N % (1 << lev) == 0:
        try:
            _check_mg_levels(N, lev + 1, world)
        except ValueError:
            break
        lev += 1
    return lev


def _swelling_operators(ctx, dim: int, N: int, pc_type: str, overrides, layout, p2_range=None, p1_range=None):
    """A, P, P_diff of the swelling problem on `layout` (the node ranges select the owned flags; default: all nodes)."""
    from hostfem.stencil import swelling_generator
    gen, par, loads = swelling_generator(dim, N, overrides)
    bc_s = gen.bc_s[slice(*p2_range) if p2_range else slice(None)].ravel()
    bc_f = gen.bc_f[slice(*p2_range) if p2_range else slice(None)].ravel()
    bc_p = gen.bc_p[slice(*p1_range) if p1_range else slice(None)]
    flags = np.concatenate([bc_s, bc_f, np.zeros(len(bc_p), bool)])   # pressure BCs only go to P_diff (lib/Poromechanics.py:76-83)
    A = generate_matrix(ctx, gen, layout, "A", pc_type, flags)
    P = generate_matrix(ctx, gen, layout, "P", pc_type, flags)
    Pd = None
    if "3-way" in pc_type:
        Pd = generate_matrix(ctx, gen, layout, "P_diff", pc_type, np.concatenate([bc_s, bc_f, bc_p]))
    return A, P, Pd, gen, par, loads


def _attach_coarse_levels(ctx, dim: int, N: int, pc_type: str, overrides, mg_levels: int, ops, layout=None):
    """Generates A, P, P_diff at N/2, N/4, ... (mg_levels - 1 levels) and links each fine matrix of `ops` to its coarse
    chain (poro_mat_set_coarse).  With a SlabLayout every level is this rank's slab nested in the one above
    (SlabLayout.coarsen).  The fine matrices keep the coarse ones alive; the coarse handles are released."""
    chains = [[m] for m in ops]
    for lev in range(1, mg_levels):
        Nc = N >> lev
        if isinstance(layout, SlabLayout):
            layout = layout.coarsen()
            A, P, Pd, _, _, _ = _swelling_operators(ctx, dim, Nc, pc_type, overrides, layout, p2_range=layout.owned[1],
                                                    p1_range=layout.owned[0])
        else:
            A, P, Pd, _, _, _ = _swelling_operators(ctx, dim, Nc, pc_type, overrides, WholeLayout(dim, Nc))
        for ch, m in zip(chains, (A, P, Pd)):
            ch.append(m)
    for ch in chains:
        if ch[0] is None:
            continue
        for i in range(len(ch) - 2, -1, -1):                       # bottom up: every coarse level already has its chain
            _capi.check(ctx.lib.poro_mat_set_coarse(ch[i].handle, ch[i + 1].handle))
        for m in ch[1:]:
            m.destroy()


def generate_swelling2d(ctx, N: int, pc_type: str = "diagonal", overrides: dict | None = None, mg_levels: int = 1) -> GeneratedSystem:
    """swelling.py on the unit square (x 1e-2) with N cells per side, generated on the device on one rank.  mg_levels > 1
    also generates the operators at N/2, N/4, ... and links them as geometric levels (`-<prefix>pc_type mg`)."""
    _check_mg_levels(N, mg_levels)
    lay = WholeLayout(2, N)
    ctx.set_halo(0, [], [0], [], [])
    A, P, Pd, gen, par, loads = _swelling_operators(ctx, 2, N, pc_type, overrides, lay)
    _attach_coarse_levels(ctx, 2, N, pc_type, overrides, mg_levels, (A, P, Pd))
    par = dict(par)
    par["pc type"] = pc_type
    b = gen.rhs(par["t0"] + par["dt"], **loads)
    o = lay.off_owned
    is_s, is_f, is_p = (o[f] + np.arange(lay.n_field[f], dtype=np.int64) for f in range(3))
    c2, c1 = gen.coords(2), gen.coords(1)
    plan = HaloPlan(lay.n_owned, np.zeros(0, np.int32), np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int64),
                    np.zeros(0, np.int64))
    return GeneratedSystem(2, A, P, Pd, b, is_s, is_f, is_p, np.flatnonzero(gen.bc_p).astype(np.int64), np.repeat(c2, 2, axis=0), c1,
                           np.arange(lay.n_owned, dtype=np.int64), plan, lay, lay.n_owned, par)


def generate_swelling3d(ctx, N: int, pc_type: str = "diagonal", rank: int = 0, world: int = 1, overrides: dict | None = None,
                        init_dist: bool = True, mg_levels: int = 1) -> GeneratedSystem:
    """swelling-3d.py on the unit cube (x 1e-2) with N cells per side: this rank's slab, generated on the device.
    mg_levels > 1 also generates the operators at N/2, N/4, ... (this rank's nested slab of each) and links them as
    geometric levels."""
    from hostfem.stencil import swelling_generator      # element matrices of ONE macro cell + loads (FEniCS stand-in)
    _check_mg_levels(N, mg_levels, world)
    gen, par, loads = swelling_generator(3, N, overrides)
    par = dict(par)
    par["pc type"] = pc_type
    lay = SlabLayout(3, N, rank, world)
    d = 3
    o1, o2 = lay.owned[0], lay.owned[1]
    bc_s = gen.bc_s[o2[0]:o2[1]].ravel()
    bc_f = gen.bc_f[o2[0]:o2[1]].ravel()
    bc_p = gen.bc_p[o1[0]:o1[1]]
    no_p = np.zeros(lay.n_field[2], bool)
    flags = np.concatenate([bc_s, bc_f, no_p])                    # pressure BCs only go to P_diff (lib/Poromechanics.py:76-83)
    if world > 1 and init_dist:
        import torch.distributed as dist
        uid = [_capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.init_dist(rank, world, uid[0])
    A = generate_matrix(ctx, gen, lay, "A", pc_type, flags)
    P = generate_matrix(ctx, gen, lay, "P", pc_type, flags)
    Pd = None
    if "3-way" in pc_type:
        Pd = generate_matrix(ctx, gen, lay, "P_diff", pc_type, np.concatenate([bc_s, bc_f, bc_p]))
    _attach_coarse_levels(ctx, 3, N, pc_type, overrides, mg_levels, (A, P, Pd), lay)
    t = par["t0"] + par["dt"]
    b = gen.rhs(t, **loads)[lay.owned_global()]
    is_s, is_f, is_p = lay.index_sets()
    h2, h1 = 1e-2 / (2 * N), 1e-2 / N
    L2, L1 = 2 * N + 1, N + 1
    n2 = np.arange(o2[0], o2[1])
    c2 = np.stack([n2 % L2, (n2 // L2) % L2, n2 // (L2 * L2)], 1) * h2
    n1 = np.arange(o1[0], o1[1])
    c1 = np.stack([n1 % L1, (n1 // L1) % L1, n1 // (L1 * L1)], 1) * h1
    plan = lay.halo_plan()
    ctx.set_halo(lay.n_owned, plan.neigh, plan.send_ptr, plan.send_idx, plan.recv_count)
    return GeneratedSystem(3, A, P, Pd, b, is_s, is_f, is_p, np.flatnonzero(bc_p).astype(np.int64), np.repeat(c2, d, axis=0), c1,
                           lay.owned_global(), plan, lay, lay.n_global, par)
