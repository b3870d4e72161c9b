"""Solver with the reference's surface (lib/Solver.py:54-155).

create_solver builds either the AAR object (lib/Solver.py:84-90) or a KSP with prefix
`global_`, tolerances (rtol, atol, 1e20, maxiter), GMRES restart = maxiter and
setFromOptions (lib/Solver.py:92-102) -- here a device KSP in libporo.so.  `set_up`
reproduces the reference's (unused) per-field norm computation only as a no-op timing
line: the `converged` test it prepares is never installed (lib/Solver.py:105-143).
"""
from __future__ import annotations

import ctypes as C
from time import perf_counter as time

from .. import _capi
from .AAR import AAR
from .backend import _tensor, get_context
from .Printing import parprint


class _KSP:
    """Device Krylov solver handle (the PETSc.KSP of lib/Solver.py:92)."""

    def __init__(self, ctx, A, pc, ksp_type, rtol, atol, divtol, maxit, restart, prefix="global_"):
        self.ctx = ctx
        h = C.c_void_p()
        _capi.check(ctx.lib.poro_ksp_create(ctx.h, A.mat().handle, pc.handle, ksp_type.encode(), float(rtol), float(atol),
                                            float(divtol), int(maxit), int(restart), prefix.encode(), C.byref(h)))
        self.h = h
        self._keep = (A, pc)      # the library borrows A when the numbering is already field-major: keep it alive
        self.its, self.reason, self.rnorm = 0, 0, 0.0
        self.max_it = maxit

    def solve(self, b, x):
        its, reason, rnorm = C.c_int(), C.c_int(), C.c_double()
        _capi.check(self.ctx.lib.poro_ksp_solve(self.h, _capi._ptr(_tensor(b)), _capi._ptr(_tensor(x)), C.byref(its),
                                                C.byref(reason), C.byref(rnorm)))
        self.its, self.reason, self.rnorm = its.value, reason.value, rnorm.value

    def solve_host(self, b_host, x_host):
        """b, x: host numpy / pinned torch buffers; copies happen inside the call (end-to-end path)."""
        its, reason, rnorm = C.c_int(), C.c_int(), C.c_double()
        _capi.check(self.ctx.lib.poro_ksp_solve_host(self.h, _capi._ptr(b_host), _capi._ptr(x_host), C.byref(its),
                                                     C.byref(reason), C.byref(rnorm)))
        self.its, self.reason, self.rnorm = its.value, reason.value, rnorm.value

    def mult(self, x, y):
        _capi.check(self.ctx.lib.poro_ksp_mult(self.h, _capi._ptr(_tensor(x)), _capi._ptr(_tensor(y))))

    def profile(self, enable=-1):
        """(ms, calls, algorithmic bytes per product) of the outer SpMV measured by CUDA events."""
        ms, calls, nbytes = C.c_double(), C.c_int64(), C.c_int64()
        _capi.check(self.ctx.lib.poro_ksp_profile(self.h, int(enable), C.byref(ms), C.byref(calls), C.byref(nbytes)))
        return ms.value, calls.value, nbytes.value

    def parts_info(self):
        """[(algorithmic bytes, format)] of each launch of the outer operator (format 0 CSR, 1 BSR, 2 diagonal BSR, 3 fused BSR, 4 stencil)."""
        b, f, n = (C.c_int64 * 16)(), (C.c_int * 16)(), C.c_int()
        _capi.check(self.ctx.lib.poro_ksp_parts_info(self.h, b, f, 16, C.byref(n)))
        return [(b[i], f[i]) for i in range(n.value)]

    def setInitialGuessNonzero(self, flag=True):
        """petsc4py KSP.setInitialGuessNonzero (lib/Solver.py:94, commented out there): warm start over time steps."""
        _capi.check(self.ctx.lib.poro_ksp_set_initial_guess_nonzero(self.h, int(bool(flag))))

    def getFieldHistory(self):
        """[(abs_s, abs_f, abs_p)] per iteration from the per-field monitor (lib/Solver.py:8-51)."""
        n = C.c_int()
        cap = 3 * (self.max_it + 2)
        buf = (C.c_double * cap)()
        _capi.check(self.ctx.lib.poro_ksp_field_history(self.h, buf, cap, C.byref(n)))
        v = list(buf)[: min(n.value, cap)]
        return [tuple(v[i:i + 3]) for i in range(0, len(v) - 2, 3)]

    def getIterationNumber(self):
        return self.its

    def getConvergedReason(self):
        return self.reason

    def getResidualNorm(self):
        return self.rnorm

    def getConvergenceHistory(self):
        n = C.c_int()
        cap = self.max_it + 2
        buf = (C.c_double * cap)()
        _capi.check(self.ctx.lib.poro_ksp_residual_history(self.h, buf, cap, C.byref(n)))
        return list(buf)[: min(n.value, cap)]

    def __del__(self):
        try:
            if self.h:
                self.ctx.lib.poro_ksp_destroy(self.h)
                self.h = None
        except Exception:
            pass


class Solver:
    def __init__(self, A, b, PC, parameters, index_map):
        self.A, self.b, self.PC = A, b, PC
        self.solver = None
        self.parameters = parameters
        self.index_map = index_map
        self.t_total = 0

    def create_solver(self, A=None, b=None, PC=None):
        t0_create = time()
        ctx = get_context()
        solver_type = self.parameters["solver type"]
        atol = self.parameters["solver atol"]
        rtol = self.parameters["solver rtol"]
        maxiter = self.parameters["solver maxiter"]
        monitor_convergence = self.parameters["solver monitor"]
        if solver_type == "aar":
            self.solver = AAR(self.parameters["AAR order"], self.parameters["AAR p"], self.parameters["AAR omega"],
                              self.parameters["AAR beta"], self.A.mat(), x0=None, pc=self.PC, atol=atol, rtol=rtol,
                              maxiter=maxiter, monitor_convergence=monitor_convergence)
        else:
            if monitor_convergence:
                ctx.set_option("-global_ksp_monitor")
            restart = maxiter if solver_type in ("gmres", "fgmres") else 30      # lib/Solver.py:99-100
            self.solver = _KSP(ctx, self.A.mat(), self.PC, solver_type, rtol, atol, 1e20, maxiter, restart, "global_")
        parprint("---- [Solver] Solver created in {}s".format(time() - t0_create))

    def set_up(self):
        t0_setup = time()
        parprint("---- [Solver] Solver set up in {}s".format(time() - t0_setup))

    def getIterationNumber(self):
        return self.solver.getIterationNumber()

    def solve(self, b, x):
        t0 = time()
        self.solver.solve(b, x)
        self.t_total += time() - t0

    def print_timings(self):
        parprint("\n===== Timing Solver: {:.3f}s".format(self.t_total))
