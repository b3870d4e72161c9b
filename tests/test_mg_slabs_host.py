"""Nested coarse slabs of `-<prefix>pc_type mg` on row-partitioned runs (generator.SlabLayout.coarsen) on the CPU: the
coarse slabs partition the coarse lattices, every coarse owned node coincides with a fine owned node, and the rows of the
masked prolongation (hostfem/mg.py) and of its transpose that a rank computes read only what its halos hold: the coarse
halo of the generated slab and the transfer halo that csrc/mg.cu builds from the class tables (poromg::plane_reach,
expanded here by a g++ harness)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hostfem.mg import masked_prolongation                       # noqa: E402
from poro_b200.generator import SlabLayout, _check_mg_levels, max_mg_levels   # noqa: E402


CSRC = os.path.join(ROOT, "poroelasticity-linear-solvers_b200", "csrc")


@pytest.fixture(scope="module")
def reach(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("mgreach") / "mg_reach_harness.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + CSRC, os.path.join(ROOT, "tests", "mg_reach_harness.cpp"),
                    "-o", out], check=True)
    lib = C.CDLL(out)
    lib.mg_reach.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]

    def planes(kind, prolong, a, b, L_to):
        lo, hi = C.c_int64(), C.c_int64()
        lib.mg_reach(kind, prolong, a, b, L_to, C.byref(lo), C.byref(hi))
        return lo.value, hi.value
    return planes


def _transfer_halo(reach, f, kind):
    """Fine planes [lo, hi) held for the restriction of slab `f`: owned + the transfer halo of mg_transfer_init."""
    c = f.coarsen()
    a, b = f.planes2 if kind == 2 else f.planes1
    ca, cb = c.planes2 if kind == 2 else c.planes1
    lo, hi = reach(kind, 0, ca, cb, (2 * f.N + 1) if kind == 2 else (f.N + 1))
    return min(lo, a), max(hi, b)


def _chain(N, world, levels):
    """Per rank the layouts of `levels` levels, finest first."""
    out = []
    for r in range(world):
        lays = [SlabLayout(3, N, r, world)]
        for _ in range(1, levels):
            lays.append(lays[-1].coarsen())
        out.append(lays)
    return out


def _cases():
    for world in range(2, 9):
        for N in (8, 16, 24, 32, 40, 48):
            lev = max_mg_levels(N, world)
            if lev > 1:
                yield world, N, lev


CASES = list(_cases())


@pytest.mark.parametrize("world,N,levels", CASES)
def test_coarse_slabs_partition_and_nest(world, N, levels):
    chain = _chain(N, world, levels)
    for lev in range(levels):
        Nl = N >> lev
        for k, n in ((0, (Nl + 1) ** 3), (1, (2 * Nl + 1) ** 3)):
            ranges = [chain[r][lev].owned[k] for r in range(world)]
            assert ranges[0][0] == 0 and ranges[-1][1] == n
            assert all(ranges[r][1] == ranges[r + 1][0] for r in range(world - 1))
        if lev == 0:
            continue
        for r in range(world):
            f, c = chain[r][lev - 1], chain[r][lev]
            Lc, Lf = 2 * c.N + 1, 2 * f.N + 1
            nodes = np.arange(*c.owned[1])
            X = np.stack([nodes % Lc, (nodes // Lc) % Lc, nodes // (Lc * Lc)], 1)
            fine = 2 * X[:, 0] + 2 * X[:, 1] * Lf + 2 * X[:, 2] * Lf * Lf
            assert ((fine >= f.owned[1][0]) & (fine < f.owned[1][1])).all()
            # the halo plan of the coarse slab follows the usual rules: what a rank sends is what its neighbour holds
            if r + 1 < world:
                assert c.send_up == chain[r + 1][lev].ghost_lo


def _bc(n, bs, seed):
    return np.random.default_rng(seed).random(n * bs) < 0.2


@pytest.mark.parametrize("world,N", [(2, 8), (3, 16), (4, 16), (5, 16), (2, 16), (6, 32)])
@pytest.mark.parametrize("kind,bs", [(2, 3), (1, 1)])
def test_transfer_rows_stay_inside_the_halos(reach, world, N, kind, bs):
    """Prolongation rows of owned fine nodes read coarse owned + ghost nodes, and the reach mg_transfer_init checks covers
    them; restriction rows (the transpose) of owned coarse nodes read fine owned + transfer-halo nodes, and the transfer
    halo is no wider than they need.  Both slab parities occur."""
    Nc = N // 2
    k = 1 if kind == 2 else 0
    Lf, Lc = (2 * N + 1, 2 * Nc + 1) if kind == 2 else (N + 1, Nc + 1)
    P = masked_prolongation(3, Nc, kind, bs, _bc(Lf ** 3, bs, 1), _bc(Lc ** 3, bs, 2))
    R = P.T.tocsr()
    parities = set()
    for r in range(world):
        f = SlabLayout(3, N, r, world)
        c = f.coarsen()
        parities.add(f.planes2[0] % 4)
        held_c = np.zeros(Lc ** 3, bool)
        for rng in (c.owned[k], c.ghost_lo[k], c.ghost_up[k]):
            held_c[rng[0]:rng[1]] = True
        rows = np.arange(f.owned[k][0] * bs, f.owned[k][1] * bs)
        cols = P[rows].indices // bs
        assert held_c[cols].all(), (r, np.setdiff1d(cols[~held_c[cols]], []))
        a, b = f.planes2 if kind == 2 else f.planes1
        plo, phi = reach(kind, 1, a, b, Lc)
        cplane = cols // (Lc * Lc)
        assert cplane.min() == plo and cplane.max() == phi - 1
        lo, hi = _transfer_halo(reach, f, kind)
        rows = np.arange(c.owned[k][0] * bs, c.owned[k][1] * bs)
        cols = R[rows].indices // bs
        plane = cols // (Lf * Lf)
        assert ((plane >= lo) & (plane < hi)).all(), (r, plane.min(), plane.max(), lo, hi)
        # and the halo is no wider than what the rows read
        if len(cols):
            assert plane.min() == lo and plane.max() == hi - 1
    if world >= 3 and kind == 2:
        assert len(parities) > 1


@pytest.mark.parametrize("planes,below", [((12, 33), 3), ((22, 33), 1), ((7, 33), 2), ((5, 33), 0)])
def test_p2_restriction_halo_width_follows_the_slab_start(reach, planes, below):
    """A coarse vertex plane gathers fine planes 2Y-3 .. 2Y+3: 3 planes below a slab starting at a multiple of 4."""
    lay = SlabLayout(3, 16, 1, 2, p2_planes=planes)
    assert lay.planes2[0] - _transfer_halo(reach, lay, 2)[0] == below


@pytest.mark.parametrize("world,N,levels,rank,level", [(8, 8, 2, 1, 1), (4, 8, 3, 1, 2), (6, 16, 3, 1, 2)])
def test_too_many_levels_names_rank_and_level(world, N, levels, rank, level):
    with pytest.raises(ValueError) as e:
        _check_mg_levels(N, levels, world)
    msg = str(e.value)
    assert "level %d" % level in msg and "rank %d" % rank in msg


def test_single_rank_and_refusals_unchanged():
    _check_mg_levels(16, 5, 1)
    with pytest.raises(ValueError, match="not divisible"):
        _check_mg_levels(12, 4, 2)
    assert max_mg_levels(16) == 5 and max_mg_levels(12) == 3
    assert max_mg_levels(32, 2) >= 3
