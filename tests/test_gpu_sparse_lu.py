"""GPU tests of the device sparse LU of the exact inner blocks (-<prefix>pc_factor_mat_solver_type poro, csrc/sparse_lu.cu):
one inner application against scipy's spsolve, outer GMRES / AAR against the oracle's exact (splu) configuration at forced
small sizes and at natural sizes above the dense limit, the golden systems, factor_info, determinism, CUDA-graph replay,
and that the selection is opt-in."""
import numpy as np
import pytest
import scipy.sparse.linalg as spla

from helpers import AMG_OPTIONS, EXACT_OPTIONS, gpu_solve, rel
from test_golden import FILES, _load

pytestmark = pytest.mark.gpu

PREFIXES = ("s", "f", "p", "diff", "fp")
SPARSE_OPTIONS = EXACT_OPTIONS + "".join("-%s_pc_factor_mat_solver_type poro\n" % p for p in PREFIXES)
FORCE = "-poro_dense_lu_limit 10\n"
BLOCK = {"s": "ss", "f": "ff", "p": "pp", "diff": "diff", "fp": "fpfp"}


def _names(pc_type):
    return ("s", "f", "p", "diff") if "3-way" in pc_type else ("s", "fp")


def _oracle_exact(sys_, par, solver_type="gmres"):
    from test_gpu_parity import _oracle_exact as oe
    return oe(sys_, par, solver_type)


@pytest.mark.parametrize("dim,N,pc_type", [(2, 8, "diagonal"), (2, 8, "diagonal 3-way"), (2, 8, "undrained"),
                                           (2, 8, "undrained 3-way"), (3, 3, "diagonal")])
def test_inner_application_equals_spsolve(gpu_ctx, dim, N, pc_type):
    from oracle.problems import swelling
    from poro_b200.lib.backend import DeviceVector
    sys_, par = swelling(dim, N, pc_type)
    g = gpu_solve(sys_, par, SPARSE_OPTIONS + FORCE, return_objects=True)
    cc = g["pc"].pc.getPythonContext()
    rng = np.random.default_rng(7)
    for name in _names(pc_type):
        B = cc.block(BLOCK[name])
        info = cc.factor_info(name)
        assert info["rows"] == B.shape[0] and info["perturbed_pivots"] == 0, (name, info)
        assert cc.amg_info(name) == []                      # the AMG stand-in was not built
        r = rng.standard_normal(B.shape[0])
        dr, dz = DeviceVector(r, ctx=gpu_ctx), DeviceVector(n=B.shape[0], ctx=gpu_ctx)
        cc.inner_solve(name, dr, dz)
        gpu_ctx.sync()
        assert rel(dz.numpy(), spla.spsolve(B.tocsc(), r)) <= 1e-10, name


@pytest.mark.parametrize("dim,N,pc_type", [(2, 10, "diagonal"), (2, 10, "diagonal 3-way"), (2, 10, "undrained"),
                                           (3, 3, "diagonal"), (3, 3, "diagonal 3-way")])
def test_gmres_forced_sparse_matches_oracle(gpu_ctx, dim, N, pc_type):
    from oracle.problems import swelling
    sys_, par = swelling(dim, N, pc_type)
    xo, its_o, _ = _oracle_exact(sys_, par)
    g = gpu_solve(sys_, par, SPARSE_OPTIONS + FORCE)
    assert g["its"] == its_o and g["reason"] in (2, 3)
    assert rel(g["x"], xo) <= 1e-8


@pytest.mark.parametrize("dim,N,pc_type", [(2, 40, "diagonal"), (2, 40, "diagonal 3-way"), (3, 8, "diagonal")])
def test_gmres_natural_size_matches_oracle(gpu_ctx, dim, N, pc_type):
    """Blocks above the default dense limit (8 192 rows): factorised, not iterated."""
    from oracle.problems import swelling
    sys_, par = swelling(dim, N, pc_type)
    xo, its_o, _ = _oracle_exact(sys_, par)
    g = gpu_solve(sys_, par, SPARSE_OPTIONS, return_objects=True)
    cc = g["pc"].pc.getPythonContext()
    info = cc.factor_info("s")
    assert info["rows"] > 8192 and info["perturbed_pivots"] == 0
    assert g["its"] == its_o
    assert rel(g["x"], xo) <= 1e-8


def test_aar_forced_sparse_matches_oracle(gpu_ctx):
    from oracle.problems import swelling
    sys_, par = swelling(2, 10, "diagonal")
    _, its_o, hist_o = _oracle_exact(sys_, par, "aar")
    g = gpu_solve(sys_, par, SPARSE_OPTIONS + FORCE, solver_type="aar")
    # the tolerances of the dense-block AAR test (tests/test_gpu_parity.py)
    assert abs(g["its"] - its_o) <= max(2, its_o // 10)
    assert rel(g["x"], spla.spsolve(sys_.A.tocsc(), sys_.b)) <= 1e-6
    np.testing.assert_allclose(g["history"][:4], hist_o[:4], rtol=1e-8)


@pytest.mark.parametrize("path", FILES, ids=[p.rsplit("/", 1)[-1][:-4] for p in FILES])
def test_golden_systems_through_sparse_path(gpu_ctx, path):
    gd, s, par = _load(path)
    out = gpu_solve(s, par, SPARSE_OPTIONS + FORCE, return_objects=True)
    assert out["pc"].pc.getPythonContext().factor_info("s")["perturbed_pivots"] == 0
    assert out["its"] == int(gd["gmres_its"])
    assert rel(out["x"], gd["gmres_x"]) <= 1e-8


def test_factor_info_raises_for_dense_and_amg_blocks(gpu_ctx):
    from oracle.problems import swelling
    from poro_b200._capi import PoroError
    sys_, par = swelling(2, 6, "diagonal")
    g = gpu_solve(sys_, par, EXACT_OPTIONS, return_objects=True)          # dense inverse
    with pytest.raises(PoroError, match="not factorised by the sparse LU"):
        g["pc"].pc.getPythonContext().factor_info("s")
    g = gpu_solve(sys_, par, AMG_OPTIONS, return_objects=True)            # AMG
    with pytest.raises(PoroError, match="not factorised by the sparse LU"):
        g["pc"].pc.getPythonContext().factor_info("s")


@pytest.mark.parametrize("key", [None, "mumps"])
def test_selection_is_opt_in(gpu_ctx, key):
    """Without the key (or with another solver type) a block above the limit is still the iterated AMG stand-in."""
    from oracle.problems import swelling
    from poro_b200._capi import PoroError
    sys_, par = swelling(2, 6, "diagonal")
    opts = EXACT_OPTIONS + FORCE + ("" if key is None else "-s_pc_factor_mat_solver_type %s\n" % key)
    g = gpu_solve(sys_, par, opts, return_objects=True)
    cc = g["pc"].pc.getPythonContext()
    assert len(cc.amg_info("s")) >= 1
    with pytest.raises(PoroError):
        cc.factor_info("s")


def test_two_setups_are_bitwise_identical(gpu_ctx):
    from oracle.problems import swelling
    sys_, par = swelling(2, 12, "diagonal 3-way")
    g1 = gpu_solve(sys_, par, SPARSE_OPTIONS + FORCE)
    g2 = gpu_solve(sys_, par, SPARSE_OPTIONS + FORCE)
    assert g1["its"] == g2["its"]
    assert np.array_equal(g1["x"], g2["x"])


@pytest.mark.parametrize("pc_type", ["diagonal", "diagonal 3-way"])
def test_graph_replay_equals_eager_application(gpu_ctx, pc_type):
    """PCBlockCC runs its first application eagerly and captures later ones in a CUDA graph: same bits."""
    from oracle.problems import swelling
    from poro_b200.lib.backend import DeviceVector
    sys_, par = swelling(2, 12, pc_type)
    g = gpu_solve(sys_, par, SPARSE_OPTIONS + FORCE, return_objects=True)
    # a fresh preconditioner: its applications start eager again
    from poro_b200.lib.Preconditioner import PreconditionerCC
    cc_old = g["pc"].pc.getPythonContext()
    cc = PreconditionerCC(cc_old.M, cc_old.M_diff, cc_old.index_map, cc_old.flag_3_way, cc_old.inner_ksp_type,
                          cc_old.inner_pc_type, bcs_sub_pressure=cc_old.bcs_sub_pressure, pc_type=cc_old.pc_type,
                          A=cc_old.A, ctx=gpu_ctx)
    cc.setUp()
    x = DeviceVector(np.random.default_rng(11).standard_normal(sys_.n), ctx=gpu_ctx)
    outs = []
    for _ in range(3):                    # eager, captured, replayed
        y = DeviceVector(n=sys_.n, ctx=gpu_ctx)
        cc.apply(None, x, y)
        gpu_ctx.sync()
        outs.append(y.numpy())
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    assert np.all(np.isfinite(outs[0])) and np.linalg.norm(outs[0]) > 0
