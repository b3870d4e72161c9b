"""Preconditioner / PreconditionerCC with the reference's surface (lib/Preconditioner.py).

`Preconditioner(index_map, A, P, P_diff, parameters, bcs_sub_pressure).get_pc()` returns a PC
object exposing `apply(x, y)`, `getPythonContext()` and `setUp()` like petsc4py's python-type
PC.  The block extraction, inner-solver creation (prefixes s_ f_ p_ fp_ diff_) and the
2-way / 3-way sweeps run inside libporo.so on the GPU; Python is not re-entered per outer
iteration (the reference re-enters through PCApply_Python, lib/Preconditioner.py:141).
"""
from __future__ import annotations

import ctypes as C
from time import perf_counter as time

import numpy as np

from .. import _capi
from .AndersonAcceleration import AndersonAcceleration
from .backend import _tensor, get_context
from .Printing import parprint


class PreconditionerCC(object):
    def __init__(self, M, M_diff, index_map, flag_3_way, inner_ksp_type="gmres", inner_pc_type="lu", inner_rtol=1e-6,
                 inner_atol=1e-6, inner_maxiter=1000, inner_monitor=True, w1=1.0, w2=0.1, accel_order=0,
                 bcs_sub_pressure=None, pc_type=None, A=None, ctx=None):
        self.M, self.M_diff, self.A = M, M_diff, A
        self.flag_3_way = flag_3_way
        self.w1, self.w2 = w1, w2
        self.index_map = index_map
        self.ns, self.nf, self.np = index_map.get_dimensions()
        self.is_s, self.is_f, self.is_p, self.is_fp = index_map.get_index_sets()
        self.inner_ksp_type, self.inner_pc_type = inner_ksp_type, inner_pc_type
        # stored but never applied to any KSP, exactly like the reference (lib/Preconditioner.py:24-27)
        self.inner_maxiter, self.inner_rtol, self.inner_atol, self.inner_monitor = inner_maxiter, inner_rtol, inner_atol, inner_monitor
        self.anderson = AndersonAcceleration(accel_order)
        self.bcs_sub_pressure = np.asarray(bcs_sub_pressure if bcs_sub_pressure is not None else [], dtype=np.int64)
        self.pc_type = pc_type or ("diagonal 3-way" if flag_3_way else "diagonal")
        self.ctx = ctx or get_context()
        self.h = None
        self.t_setup = 0.0

    def setUp(self, pc=None):
        t0_setup = time()
        lib = self.ctx.lib
        self.index_map.install(self.ctx)
        h = C.c_void_p()
        pd = self.M_diff.mat().handle if (self.M_diff is not None and self.flag_3_way) else None
        _capi.check(lib.poro_pc_setup(self.ctx.h, self.A.mat().handle if self.A is not None else None,
                                      self.M.mat().handle, pd, self.pc_type.encode(), self.inner_ksp_type.encode(),
                                      self.inner_pc_type.encode(), _capi._ptr(self.bcs_sub_pressure),
                                      len(self.bcs_sub_pressure), int(self.anderson.order), float(self.w1),
                                      float(self.w2), C.byref(h)))
        self.h = h
        self.t_setup = time() - t0_setup
        parprint("---- [Preconditioner] Set up in {}s".format(self.t_setup))

    def apply(self, pc, x, y):
        """y = M^-1 x (lib/Preconditioner.py:141-250); x, y device vectors in the caller's ordering."""
        _capi.check(self.ctx.lib.poro_pc_apply(self.h, _capi._ptr(_tensor(x)), _capi._ptr(_tensor(y))))

    def stats(self):
        out = (C.c_double * 20)()
        _capi.check(self.ctx.lib.poro_pc_stats(self.h, out, 20))
        v = list(out)
        keys = ["s", "f", "p", "fp", "diff", "fp_split0", "fp_split1"]
        d = dict(t_total=v[0], t_solid=v[1], t_fluid=v[2], t_press=v[3], t_alloc=v[4])
        for i, k in enumerate(keys):
            d["its_" + k], d["calls_" + k] = int(v[5 + 2 * i]), int(v[6 + 2 * i])
        d["graph_replays"] = int(v[19])
        return d

    def block_info(self, name):
        r, c, z = C.c_int64(), C.c_int64(), C.c_int64()
        _capi.check(self.ctx.lib.poro_pc_block_info(self.h, name.encode(), C.byref(r), C.byref(c), C.byref(z)))
        return r.value, c.value, z.value

    def block_bytes(self, name):
        """(algorithmic bytes of one product with the block, format 0 CSR / 1 BSR / 2 diagonal BSR / 4 stencil)."""
        b, f = C.c_int64(), C.c_int()
        _capi.check(self.ctx.lib.poro_pc_block_bytes(self.h, name.encode(), C.byref(b), C.byref(f)))
        return b.value, f.value

    def block(self, name):
        """Copy of a device block as scipy CSR (blocks: ss sf sp ff fp pp fps fpfp schur diff)."""
        import scipy.sparse as sp
        r, c, z = self.block_info(name)
        rp, ci, v = np.zeros(r + 1, np.int64), np.zeros(z, np.int32), np.zeros(z, np.float64)
        _capi.check(self.ctx.lib.poro_pc_block_copy(self.h, name.encode(), _capi._ptr(rp), _capi._ptr(ci), _capi._ptr(v)))
        return sp.csr_matrix((v, ci, rp), shape=(r, c))

    def amg_info(self, name):
        rows, nnz, nl = (C.c_int64 * 32)(), (C.c_int64 * 32)(), C.c_int()
        _capi.check(self.ctx.lib.poro_pc_amg_info(self.h, name.encode(), rows, nnz, 32, C.byref(nl)))
        return [(rows[i], nnz[i]) for i in range(nl.value)]

    AMG_LEVEL_KEYS = ("A_rows", "A_cols", "A_nnz", "P_rows", "P_cols", "P_nnz", "R_rows", "R_cols", "R_nnz", "T_rows", "T_cols",
                      "T_nnz", "bs", "k", "n_agg", "geometric", "coarsest", "direct", "kept", "chunks_AT", "chunks_AP", "chunks_RAP")

    def amg_level_info(self, name, level):
        """One level of a block's AMG hierarchy (poro_pc_amg_level_info) as a dict (keys: AMG_LEVEL_KEYS and "lmax")."""
        out, lmax = (C.c_int64 * len(self.AMG_LEVEL_KEYS))(), C.c_double()
        _capi.check(self.ctx.lib.poro_pc_amg_level_info(self.h, name.encode(), int(level), out, len(out), C.byref(lmax)))
        d = dict(zip(self.AMG_LEVEL_KEYS, (int(v) for v in out)))
        d["lmax"] = lmax.value
        return d

    def amg_level(self, name, level, what):
        """Host copy of one item of an AMG level (poro_pc_amg_level_copy): "A" "P" "R" "T" as scipy CSR (explicit zeros
        kept), "agg" int32 (n / bs), "B" (n, k), "dinv" (n), "inv" (n, n).  "agg", "B" and "T" need -poro_amg_keep_setup 1."""
        import scipy.sparse as sp
        info = self.amg_level_info(name, level)
        n = info["A_rows"]
        rp = ci = v = None
        if what in ("A", "P", "R", "T"):
            r, c, z = info[what + "_rows"], info[what + "_cols"], info[what + "_nnz"]
            rp, ci, v = np.zeros(r + 1, np.int64), np.zeros(z, np.int32), np.zeros(z, np.float64)
        elif what == "agg":
            ci = np.zeros(n // max(info["bs"], 1), np.int32)
        else:
            v = np.zeros({"B": n * info["k"], "dinv": n, "inv": n * n}.get(what, 0), np.float64)
        _capi.check(self.ctx.lib.poro_pc_amg_level_copy(self.h, name.encode(), int(level), what.encode(), _capi._ptr(rp),
                                                        _capi._ptr(ci), _capi._ptr(v)))
        if rp is not None:
            return sp.csr_matrix((v, ci, rp), shape=(r, c))
        if what == "agg":
            return ci
        return v.reshape(n, -1) if what in ("B", "inv") else v

    FACTOR_INFO_KEYS = ("rows", "nnz_l", "nnz_u", "amalgamation_zeros", "supernodes", "levels", "max_front",
                        "perturbed_pivots", "device_bytes", "factor_flops", "factor_us", "apply_bytes")

    def factor_info(self, name):
        """Sparse LU of a block's inner PC ("s","f","p","fp","diff") as a dict (keys: FACTOR_INFO_KEYS, see
        poro_pc_factor_info in include/poro.h); raises for a block that is not factorised by the sparse LU."""
        out = (C.c_int64 * len(self.FACTOR_INFO_KEYS))()
        _capi.check(self.ctx.lib.poro_pc_factor_info(self.h, name.encode(), out, len(out)))
        return dict(zip(self.FACTOR_INFO_KEYS, (int(v) for v in out)))

    ILU_INFO_KEYS = ("rows", "nnz_l", "nnz_u", "lower_levels", "upper_levels", "min_pivot", "device_bytes", "apply_bytes")

    def ilu_info(self, name):
        """ILU(0) of an inner PC ("s","f","p","fp","diff","fp0","fp1"; -<prefix>pc_type ilu or bjacobi) as a dict (keys:
        ILU_INFO_KEYS, see poro_pc_ilu_info in include/poro.h); raises for an inner PC that is not ILU / bjacobi."""
        out = (C.c_double * len(self.ILU_INFO_KEYS))()
        _capi.check(self.ctx.lib.poro_pc_ilu_info(self.h, name.encode(), out, len(out)))
        return {k: (float(v) if k == "min_pivot" else int(v)) for k, v in zip(self.ILU_INFO_KEYS, out)}

    def mg_info(self, name):
        """Geometric multigrid of an inner PC (`-<prefix>pc_type mg`): ([(N, rows, format) per geometric level, finest
        first], number of algebraic levels below); raises for an inner PC that is not `mg`."""
        out = (C.c_int64 * 64)()
        _capi.check(self.ctx.lib.poro_pc_mg_info(self.h, name.encode(), out, len(out)))
        g = int(out[0])
        return [tuple(int(v) for v in out[1 + 3 * l: 4 + 3 * l]) for l in range(g)], int(out[1 + 3 * g])

    def mg_transfer(self, name, level, direction, mode, x, y):
        """One geometric transfer between `level` and `level + 1` (direction 0: y = / += P~ x, 1: y = P~^T x)."""
        _capi.check(self.ctx.lib.poro_pc_mg_transfer(self.h, name.encode(), level, direction, mode, _capi._ptr(_tensor(x)),
                                                     _capi._ptr(_tensor(y))))

    def mg_bytes(self, name, level):
        """Algorithmic bytes of the transfers of `level`: (prolongation set, prolongation add, restriction)."""
        out = (C.c_int64 * 3)()
        _capi.check(self.ctx.lib.poro_pc_mg_bytes(self.h, name.encode(), level, out))
        return tuple(int(v) for v in out)

    def inner_solve(self, name, r, z):
        _capi.check(self.ctx.lib.poro_pc_inner_solve(self.h, name.encode(), _capi._ptr(_tensor(r)), _capi._ptr(_tensor(z))))

    def inner_result(self, name):
        """(iterations, reason, residual norm) of the last application of an inner solver."""
        its, reason, rnorm = C.c_int(), C.c_int(), C.c_double()
        _capi.check(self.ctx.lib.poro_pc_inner_result(self.h, name.encode(), C.byref(its), C.byref(reason), C.byref(rnorm)))
        return its.value, reason.value, rnorm.value

    def print_timings(self):
        s = self.stats()
        parprint("\n===== Timing preconditioner: {:.3f}s".format(s["t_total"]))
        if self.flag_3_way:
            parprint("\tSolid solver: {:.3f}s\n\tFluid solver: {:.3f}s\n\tPressure solver: {:.3f}s".format(
                s["t_solid"], s["t_fluid"], s["t_press"]))
        else:
            parprint("\tSolid solver: {:.3f}s\n\tFluid-pressure solver: {:.3f}s".format(s["t_solid"], s["t_fluid"]))
        parprint("\n\tAllocation time: {:.3f}".format(s["t_alloc"]))

    def destroy(self):
        if self.h:
            self.ctx.lib.poro_pc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class _PC:
    """The petsc4py `PC` of type 'python' the reference builds at lib/Preconditioner.py:286-290."""

    def __init__(self, ctx_obj):
        self._ctx_obj = ctx_obj
        self.type = "python"

    def getPythonContext(self):
        return self._ctx_obj

    def setUp(self):
        self._ctx_obj.setUp(self)

    def apply(self, x, y):
        self._ctx_obj.apply(self, x, y)

    def getType(self):
        return self.type

    @property
    def handle(self):
        return self._ctx_obj.h


def cc_scales(parameters, dim):
    """The two scalars of `-fp_pc_fieldsplit_schur_precondition cc` from the reference's parameter dict
    (the coefficients of lib/Assembler.py:127-160, `diagonal` splitting):

        mass_scale * |diag(A_fs)| = diag(c M_v),  A_fs = -(phi0^2 / (k_f dt)) M_v,  c = rho_f phi0 / dt + (1 + beta_f) phi0^2 / k_f
        visc_scale * P_pp = (phi0 d / (2 mu_f)) M_p  (beta_CC1, lib/Assembler.py:131),  P_pp = (phi_s^2 / (k_s dt) + beta_p) M_p"""
    phi0, dt, kf = float(parameters["phi0"]), float(parameters["dt"]), float(parameters["kf"])
    phis = 1.0 - phi0
    drag = phi0 ** 2 / kf
    c = float(parameters["rhof"]) * phi0 / dt + (1.0 + float(parameters["betaf"])) * drag
    beta_p = float(parameters["betap"]) * phis ** 2 / (dt * (2.0 * float(parameters["mu_s"]) / dim + float(parameters["lmbda"])))
    mass_scale = c * dt / drag
    visc_scale = (phi0 * dim / (2.0 * float(parameters["mu_f"]))) / (phis ** 2 / (float(parameters["ks"]) * dt) + beta_p)
    return mass_scale, visc_scale


class Preconditioner:
    def __init__(self, index_map, A, P, P_diff, parameters, bcs_sub_pressure):
        self.index_map = index_map
        self.parameters = parameters
        self.A, self.P, self.P_diff = A, P, P_diff
        self.pc_type = parameters["pc type"]
        self.inner_ksp_type = parameters["inner ksp type"]
        self.inner_pc_type = parameters["inner pc type"]
        self.inner_rtol = parameters["inner rtol"]
        self.inner_atol = parameters["inner atol"]
        self.inner_maxiter = parameters["inner maxiter"]
        self.inner_accel_order = parameters["inner accel order"]
        self.inner_monitor = parameters["inner monitor"]
        self.bcs_sub_pressure = bcs_sub_pressure
        if self.pc_type not in ("undrained", "undrained 3-way", "diagonal", "diagonal 3-way", "diagonal 3-way-II", "lu"):
            import sys
            sys.exit("pc type must be one of lu, undrained, diagonal, diagonal 3-way, diagonal 3-way-II.")

    def get_pc(self):
        flag_3_way = self.pc_type in ("diagonal 3-way", "undrained 3-way")
        lib_ctx = get_context()
        if (self.pc_type == "diagonal" and lib_ctx.get_option("fp_pc_fieldsplit_schur_precondition") == "cc"
                and lib_ctx.get_option("fp_pc_fieldsplit_schur_cc_mass_scale") is None):
            dim = int(getattr(self.index_map, "block_dim", 0) or self.parameters.get("dim", 0))
            if dim <= 0 and getattr(self.index_map, "coords_s", None) is not None:
                dim = int(np.asarray(self.index_map.coords_s).shape[1])
            try:
                ms, vs = cc_scales(self.parameters, dim)
            except (KeyError, ZeroDivisionError) as e:
                raise ValueError("-fp_pc_fieldsplit_schur_precondition cc needs the physical parameters of the reference's "
                                 "parameter dict (phi0, dt, kf, ks, rhof, mu_f, mu_s, lmbda, betaf, betap) and the space "
                                 "dimension, or explicit -fp_pc_fieldsplit_schur_cc_mass_scale / _visc_scale options: %r" % (e,))
            lib_ctx.set_option("-fp_pc_fieldsplit_schur_cc_mass_scale", repr(ms))
            lib_ctx.set_option("-fp_pc_fieldsplit_schur_cc_visc_scale", repr(vs))
        ctx = PreconditionerCC(self.P.mat(), self.P_diff.mat() if self.P_diff is not None else None, self.index_map,
                               flag_3_way, self.inner_ksp_type, self.inner_pc_type, self.inner_rtol, self.inner_atol,
                               self.inner_maxiter, self.inner_monitor, 1.0, 0.1, self.inner_accel_order,
                               self.bcs_sub_pressure, pc_type=self.pc_type, A=self.A.mat())
        self.pc = _PC(ctx)
        self.pc.setUp()
        return self.pc

    def print_timings(self):
        self.pc.getPythonContext().print_timings()
