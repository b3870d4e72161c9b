"""ctypes binding of libporo.so (the C ABI declared in include/poro.h).

There is no CPU fallback: if the library is missing or no CUDA device is present the calls
raise.  PyTorch is used by the callers only to own device buffers; this module passes raw
device pointers (`tensor.data_ptr()`).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libporo.so")
_lib = None

c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)
vp = C.c_void_p

# name -> (argtypes); every function returns int except where noted
SIGNATURES = {
    "poro_ctx_create": [C.c_int, C.POINTER(vp)],
    "poro_ctx_destroy": [vp],
    "poro_nccl_unique_id": [C.c_char_p],
    "poro_ctx_init_dist": [vp, C.c_int, C.c_int, C.c_char_p],
    "poro_options_set": [vp, C.c_char_p, C.c_char_p],
    "poro_options_clear": [vp],
    "poro_sync": [vp],
    "poro_timer_start": [vp],
    "poro_timer_stop": [vp, c_f64p],
    "poro_mat_create_csr": [vp, C.c_int64, C.c_int64, vp, vp, vp, C.c_int, C.POINTER(vp)],
    "poro_mat_destroy": [vp],
    "poro_mat_info": [vp, c_i64p, c_i64p, c_i64p],
    "poro_mat_mult": [vp, vp, vp],
    "poro_mat_bench": [vp, C.c_int, C.c_int, c_f64p],
    "poro_mat_copy": [vp, vp, vp, vp],
    "poro_mat_setup_op": [vp, vp, C.c_char_p, C.c_double, vp, C.POINTER(vp), C.POINTER(C.c_int)],
    "poro_dense_inverse": [vp, C.c_int, vp, vp],
    "poro_mat_mult_mode": [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_double, vp],
    "poro_mat_kernel_info": [vp, c_i64p, C.c_int],
    "poro_mat_mult_fused": [vp, vp, C.c_int, vp, vp, vp, vp, C.POINTER(C.c_int)],
    "poro_gen_matrix": [vp, C.c_int, C.c_int, vp, vp, vp, C.POINTER(vp)],
    "poro_mat_set_coarse": [vp, vp],
    "poro_halo_set": [vp, C.c_int64, C.c_int, vp, vp, vp, vp],
    "poro_fields_set": [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, C.c_int, C.c_int],
    "poro_fields_set_coords": [vp, C.c_int, vp, vp],
    "poro_pc_setup": [vp, vp, vp, vp, C.c_char_p, C.c_char_p, C.c_char_p, vp, C.c_int64, C.c_int, C.c_double,
                      C.c_double, C.POINTER(vp)],
    "poro_pc_apply": [vp, vp, vp],
    "poro_pc_destroy": [vp],
    "poro_pc_stats": [vp, c_f64p, C.c_int],
    "poro_ksp_create": [vp, vp, vp, C.c_char_p, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_char_p,
                        C.POINTER(vp)],
    "poro_ksp_solve": [vp, vp, vp, C.POINTER(C.c_int), C.POINTER(C.c_int), c_f64p],
    "poro_ksp_solve_host": [vp, vp, vp, C.POINTER(C.c_int), C.POINTER(C.c_int), c_f64p],
    "poro_ksp_residual_history": [vp, c_f64p, C.c_int, C.POINTER(C.c_int)],
    "poro_ksp_set_initial_guess_nonzero": [vp, C.c_int],
    "poro_ksp_field_history": [vp, c_f64p, C.c_int, C.POINTER(C.c_int)],
    "poro_pc_inner_result": [vp, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), c_f64p],
    "poro_ksp_destroy": [vp],
    "poro_aar_create": [vp, vp, vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                        C.POINTER(vp)],
    "poro_aar_solve": [vp, vp, vp, C.POINTER(C.c_int)],
    "poro_aar_residual_history": [vp, c_f64p, C.c_int, C.POINTER(C.c_int)],
    "poro_aar_destroy": [vp],
    "poro_pc_block_info": [vp, C.c_char_p, c_i64p, c_i64p, c_i64p],
    "poro_pc_block_copy": [vp, C.c_char_p, vp, vp, vp],
    "poro_pc_block_bytes": [vp, C.c_char_p, c_i64p, C.POINTER(C.c_int)],
    "poro_pc_block_mult": [vp, C.c_char_p, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_double, vp],
    "poro_pc_inner_solve": [vp, C.c_char_p, vp, vp],
    "poro_pc_amg_info": [vp, C.c_char_p, c_i64p, c_i64p, C.c_int, C.POINTER(C.c_int)],
    "poro_pc_amg_level_info": [vp, C.c_char_p, C.c_int, c_i64p, C.c_int, c_f64p],
    "poro_pc_amg_level_copy": [vp, C.c_char_p, C.c_int, C.c_char_p, vp, vp, vp],
    "poro_pc_factor_info": [vp, C.c_char_p, c_i64p, C.c_int],
    "poro_pc_mg_info": [vp, C.c_char_p, c_i64p, C.c_int],
    "poro_pc_mg_transfer": [vp, C.c_char_p, C.c_int, C.c_int, C.c_int, vp, vp],
    "poro_pc_mg_bytes": [vp, C.c_char_p, C.c_int, c_i64p],
    "poro_ksp_mult": [vp, vp, vp],
    "poro_ksp_profile": [vp, C.c_int, c_f64p, c_i64p, c_i64p],
    "poro_profile": [vp, C.c_int, c_f64p, c_i64p, C.c_int],
    "poro_ksp_parts_info": [vp, c_i64p, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)],
}


class PoroError(RuntimeError):
    pass


def library_path() -> str:
    return _LIB_PATH


def load():
    """dlopen libporo.so and declare every prototype; raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise PoroError("libporo.so not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    lib = C.CDLL(_LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.poro_last_error.restype = C.c_char_p
    lib.poro_last_error.argtypes = []
    lib.poro_version.restype = C.c_int
    lib.poro_launch_count.restype = C.c_int64
    lib.poro_launch_count.argtypes = [vp]
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise PoroError(load().poro_last_error().decode())


def _ptr(a):
    """Raw pointer of a numpy array, torch tensor, int or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return int(a)


def _np(a, dtype):
    return np.ascontiguousarray(np.asarray(a), dtype=dtype)


class Context:
    """One per process per GPU: stream, scratch, options database, field layout."""

    def __init__(self, device: int = 0):
        lib = load()
        h = vp()
        check(lib.poro_ctx_create(device, C.byref(h)))
        self.h, self.lib, self.device = h, lib, device
        self.rank, self.nranks = 0, 1
        self._keep = []

    def close(self):
        if self.h:
            self.lib.poro_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- options (PETSc.Options().setValue, lib/Parser.py:70-73)
    def set_option(self, key: str, val=None):
        check(self.lib.poro_options_set(self.h, key.encode(), None if val is None else str(val).encode()))
        self.__dict__.setdefault("_options", {})[key.lstrip("-")] = val

    def get_option(self, key: str, default=None):
        """Host-side mirror of the options database (what set_option stored since the last clear_options)."""
        return self.__dict__.get("_options", {}).get(key.lstrip("-"), default)

    def clear_options(self):
        check(self.lib.poro_options_clear(self.h))
        self.__dict__["_options"] = {}

    def profile(self, enable=-1):
        """Phase profile {slot: (ms, calls)} from CUDA events (slots: see include/poro.h)."""
        ms, calls = (C.c_double * 40)(), (C.c_int64 * 40)()
        check(self.lib.poro_profile(self.h, int(enable), ms, calls, 40))
        return {i: (ms[i], calls[i]) for i in range(40) if calls[i]}

    def launch_count(self) -> int:
        return int(self.lib.poro_launch_count(self.h))

    def sync(self):
        check(self.lib.poro_sync(self.h))

    def timer_start(self):
        check(self.lib.poro_timer_start(self.h))

    def timer_stop(self) -> float:
        """Milliseconds between timer_start and now, measured by CUDA events on the library's stream."""
        ms = C.c_double()
        check(self.lib.poro_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def dense_inverse(self, A):
        """Gauss-Jordan inverse of a dense host matrix on the device (the coarsest AMG level's solver)."""
        A = np.ascontiguousarray(A, dtype=np.float64)
        inv = np.empty_like(A)
        check(self.lib.poro_dense_inverse(self.h, A.shape[0], _ptr(A), _ptr(inv)))
        return inv

    def init_dist(self, rank: int, nranks: int, unique_id: bytes):
        check(self.lib.poro_ctx_init_dist(self.h, rank, nranks, unique_id))
        self.rank, self.nranks = rank, nranks

    def set_halo(self, n_owned, neigh, send_ptr, send_idx, recv_count):
        neigh, send_ptr = _np(neigh, np.int32), _np(send_ptr, np.int64)
        send_idx, recv_count = _np(send_idx, np.int32), _np(recv_count, np.int64)
        check(self.lib.poro_halo_set(self.h, int(n_owned), len(neigh), _ptr(neigh), _ptr(send_ptr), _ptr(send_idx),
                                     _ptr(recv_count)))

    def set_fields(self, is_s, is_f, is_p, is_fp=None, two_way_local_fp=False, block_dim=0):
        a = [_np(v, np.int64) for v in (is_s, is_f, is_p)]
        fp = _np(is_fp, np.int64) if is_fp is not None else np.zeros(0, np.int64)
        check(self.lib.poro_fields_set(self.h, _ptr(a[0]), len(a[0]), _ptr(a[1]), len(a[1]), _ptr(a[2]), len(a[2]),
                                       _ptr(fp), len(fp), int(bool(two_way_local_fp)), int(block_dim)))

    def set_coords(self, dim, coords_s=None, coords_p=None):
        cs = _np(coords_s, np.float64) if coords_s is not None else None
        cp = _np(coords_p, np.float64) if coords_p is not None else None
        check(self.lib.poro_fields_set_coords(self.h, int(dim), _ptr(cs), _ptr(cp)))


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    check(load().poro_nccl_unique_id(buf))
    return buf.raw


class Mat:
    """Device CSR matrix (copied at creation)."""

    def __init__(self, ctx: Context, indptr, indices, data, shape, on_device=False):
        self.ctx = ctx
        if not on_device:
            indptr, indices, data = _np(indptr, np.int64), _np(indices, np.int32), _np(data, np.float64)
        h = vp()
        check(ctx.lib.poro_mat_create_csr(ctx.h, int(shape[0]), int(shape[1]), _ptr(indptr), _ptr(indices), _ptr(data),
                                          int(on_device), C.byref(h)))
        self.h, self.shape = h, tuple(shape)

    @classmethod
    def from_scipy(cls, ctx, A):
        A = A.tocsr()
        return cls(ctx, A.indptr, A.indices, A.data, A.shape)

    def info(self):
        r, c, z = C.c_int64(), C.c_int64(), C.c_int64()
        check(self.ctx.lib.poro_mat_info(self.h, C.byref(r), C.byref(c), C.byref(z)))
        return r.value, c.value, z.value

    def mult(self, x, y):
        check(self.ctx.lib.poro_mat_mult(self.h, _ptr(x), _ptr(y)))

    def to_scipy(self):
        """Host copy of the device CSR as it is stored (explicit zeros kept)."""
        import scipy.sparse as sp
        r, c, z = self.info()
        rp, ci, v = np.zeros(r + 1, np.int64), np.zeros(z, np.int32), np.zeros(z, np.float64)
        check(self.ctx.lib.poro_mat_copy(self.h, _ptr(rp), _ptr(ci), _ptr(v)))
        return sp.csr_matrix((v, ci, rp), shape=(r, c))

    def setup_op(self, other, op: str, alpha: float = 0.0, s=None):
        """One set-up primitive (poro_mat_setup_op): ("spgemm", B) self B, ("transpose", None) self^T, ("add_scaled", B)
        self + alpha diag(s) B with s a device vector or None.  Returns (new Mat, SpGEMM row chunks)."""
        h, chunks = vp(), C.c_int()
        check(self.ctx.lib.poro_mat_setup_op(self.h, other.h if other is not None else None, op.encode(), float(alpha), _ptr(s),
                                             C.byref(h), C.byref(chunks)))
        m = Mat.__new__(Mat)
        r, c, _ = (C.c_int64(), C.c_int64(), C.c_int64())
        check(self.ctx.lib.poro_mat_info(h, C.byref(r), C.byref(c), None))
        m.ctx, m.h, m.shape = self.ctx, h, (r.value, c.value)
        return m, chunks.value

    def bench(self, mode: int, reps: int = 20) -> float:
        """Device milliseconds per launch of the SpMV in epilogue mode 0..4 (see include/poro.h)."""
        ms = C.c_double()
        check(self.ctx.lib.poro_mat_bench(self.h, int(mode), int(reps), C.byref(ms)))
        return ms.value

    def destroy(self):
        if self.h:
            self.ctx.lib.poro_mat_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass
