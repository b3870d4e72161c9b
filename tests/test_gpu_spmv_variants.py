"""Every SpMV kernel variant and epilogue against an extended-precision reference, at the edges of its chunking.

`launch_spmv` (csrc/spmv.cu) streams a raw matrix through one of: the CSR stream kernel (lanes G per row from the average
row length), the vector-CSR fallback (a row longer than a row block; L lanes per row), the plain block-CSR kernel (csrc/bsr.cu:
BS 2 / 3, dense or diagonal blocks, PREF, cooperative gathers, L2 prefetch, fp32 values, a fused mass coupling) or the
persistent TMA block-CSR kernel (csrc/bsr_tma.cu, three pipeline configs).  Each packs whole rows into chunks under a
nonzero and a row limit.  The cases below sit on those limits, derived from the constants of the kernels, and every case
asserts through `poro_mat_kernel_info` the kernel, the configuration and the chunk count it meant to hit.

Each product is compared ROW BY ROW with scipy in np.longdouble against a rounding bound that holds for any summation
order, so a dropped or doubled entry in a row at 1e-12 of the largest row scale is still seen.  Every case also runs on
the same matrix uploaded non-canonically (each entry split into two copies, columns shuffled within rows), which is how
FEM assembly hands a scipy CSR over."""
import ctypes as C
import math
import zlib

import numpy as np
import pytest
import scipy.sparse as sp

U = 2.0 ** -53
LD = np.longdouble
C1, C2 = 0.3, -0.7          # Chebyshev-step coefficients

# kernel constants the shapes are derived from
CSR_CAP, CSR_MAX_ROWS = 2048, 1024                  # spmv.cu: kCap nonzeros, kMaxRows rows per row block
BSR_CAP, BSR_MAX_BROWS, BSR_THREADS = 512, 256, 256  # bsr.cu: 256 threads x 2 blocks, kMaxBRows block rows per chunk
TMA_CAP, TMA_STAGES, TMA_MIN_CTAS = {0: 512, 1: 256, 2: 256}, {0: 2, 1: 2, 2: 3}, {0: 2, 1: 4, 2: 3}
TMA_MAX_BROWS = 64                                   # bsr_tma.cu: kMaxR
PREF_MIN_AVG = 6                                     # bsr.cu: PREF when nnzb >= 6 nbrows
DEFAULT_MAX_FILL = 1.42
CSR_STREAM, BSR, DIAG_BSR, VECTOR_CSR = 0, 1, 2, 5
INFO = ("format", "lanes", "bs", "pref", "coop", "fp32", "tma", "tma_cfg", "fused", "chunks", "l2_prefetch")


# ---------------------------------------------------------------------------------------------------------------------
# reference and comparison
# ---------------------------------------------------------------------------------------------------------------------
def _ld(A, data=None):
    """longdouble copy keeping the stored entries as they are (astype and abs would sum duplicates first)"""
    d = A.data if data is None else data
    return sp.csr_matrix((np.asarray(d, LD), A.indices.copy(), A.indptr.copy()), shape=A.shape)


class _Ref:
    """sum_t A_t x_t in longdouble, with the row sums of |A_t| |x_t| and the stored entries per row"""

    def __init__(self, terms):
        n = terms[0][0].shape[0]
        self.ax, self.abs, self.k = np.zeros(n, LD), np.zeros(n, LD), np.full(n, 2.0)
        for A, x in terms:
            xl = np.asarray(x, LD)
            self.ax += _ld(A) @ xl
            self.abs += _ld(A, np.abs(A.data)) @ np.abs(xl)
            self.k += np.diff(A.indptr)

    def bound(self, extra=0.0):
        """|y_i - yref_i| <= (entries_i + 2) u (sum_j |a_ij x_j| + |extra_i|)"""
        return self.k * U * (self.abs + np.abs(np.asarray(extra, LD)))


def _outside(got, want, bound):
    """rows where got is not within bound of want (NaN counts as outside)"""
    err = np.abs(np.asarray(got, LD) - want)
    return np.flatnonzero(~(err <= bound))


def _assert_rows(got, want, bound, what):
    bad = _outside(got, want, bound)
    if len(bad):
        i = bad[np.argmax(np.nan_to_num(np.abs(np.asarray(got, LD)[bad] - want[bad]) / bound[bad], nan=np.inf))]
        raise AssertionError("%s: %d of %d rows outside the rounding bound; row %d: got %r, want %r, bound %.3e"
                             % (what, len(bad), len(want), i, got[i], float(want[i]), float(bound[i])))


def _epilogue_refs(ref, x, z, r, dinv, xv, d_old):
    """reference values and bounds of every epilogue mode (modes 3 and 4 only for square matrices)"""
    out = {"y": (ref.ax, ref.bound()), "sub": (np.asarray(z, LD) - ref.ax, ref.bound(z)),
           "add": (np.asarray(z, LD) + ref.ax, ref.bound(z))}
    if d_old is not None:
        rn = np.asarray(r, LD) - ref.ax
        br = ref.bound(r)
        c2d = LD(C2) * np.asarray(dinv, LD)
        dn = LD(C1) * np.asarray(d_old, LD) + c2d * rn
        bd = np.abs(c2d) * br + 4 * U * (np.abs(LD(C1) * np.asarray(d_old, LD)) + np.abs(c2d * rn))
        xn = np.asarray(xv, LD) + dn
        bx = bd + 2 * U * (np.abs(np.asarray(xv, LD)) + np.abs(dn))
        out.update({"r": (rn, br), "d_new": (dn, bd), "xv": (xn, bx)})
        xl = np.asarray(x, LD)
        dot = np.sum(xl * ref.ax)
        out["dot"] = (np.array([dot]), np.array([np.sum(np.abs(xl) * ref.bound()) + len(x) * U * np.sum(np.abs(xl * ref.ax))]))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# matrices
# ---------------------------------------------------------------------------------------------------------------------
def _pattern(rowlens, ncols, rng):
    """(rows, cols) with rowlens[i] distinct columns in row i: an arithmetic progression modulo ncols"""
    rowlens = np.asarray(rowlens, np.int64)
    assert rowlens.max(initial=0) <= ncols
    n = len(rowlens)
    rows = np.repeat(np.arange(n), rowlens)
    j = np.arange(rowlens.sum()) - np.repeat(np.cumsum(rowlens) - rowlens, rowlens)
    strides = np.array([s for s in (1, 3, 7, 11, 13, 101) if math.gcd(s, ncols) == 1])
    st, off = rng.choice(strides, n), rng.integers(0, max(ncols, 1), n)
    return rows, (off[rows] + j * st[rows]) % max(ncols, 1)


def _csr(rows, cols, shape, rng):
    """canonical CSR with values scaled by random row and column factors 10^U(-6, 6), signs and 5 % explicit zeros"""
    rs, cs = 10.0 ** rng.uniform(-6, 6, shape[0]), 10.0 ** rng.uniform(-6, 6, shape[1])
    v = rng.standard_normal(len(rows)) * rs[rows] * cs[cols]
    v[rng.random(len(rows)) < 0.05] = 0.0
    A = sp.csr_matrix((v, (rows, cols)), shape=shape)
    A.sort_indices()
    assert A.nnz == len(rows)
    return A


def _scalar(rng, rowlens, ncols=None):
    ncols = len(rowlens) if ncols is None else ncols
    r, c = _pattern(rowlens, ncols, rng)
    return _csr(r, c, (len(rowlens), ncols), rng)


def _block(rng, browlens, bs, nbcols=None, diag=False):
    """node-blocked matrix: block row I has browlens[I] dense (or diagonal) bs x bs blocks"""
    nbcols = len(browlens) if nbcols is None else nbcols
    R, J = _pattern(browlens, nbcols, rng)
    q = np.arange(bs)
    if diag:
        rows, cols = (R[:, None] * bs + q).ravel(), (J[:, None] * bs + q).ravel()
    else:
        rows = (R[:, None, None] * bs + q[:, None] + 0 * q).ravel()
        cols = (J[:, None, None] * bs + 0 * q[:, None] + q).ravel()
    return _csr(rows, cols, (len(browlens) * bs, nbcols * bs), rng)


def _avg_lens(rng, n, total):
    return rng.multinomial(total, np.full(n, 1.0 / n))


def _noncanonical(A, rng):
    """the same operator with every stored entry split into two copies and the columns shuffled within each row"""
    cnt = np.diff(A.indptr)
    rows = np.repeat(np.arange(A.shape[0]), cnt)
    a1 = A.data * rng.uniform(0.1, 0.9, A.nnz)
    r2, c2, v2 = np.concatenate([rows, rows]), np.concatenate([A.indices, A.indices]), np.concatenate([a1, A.data - a1])
    order = np.argsort(r2 + rng.random(len(r2)), kind="stable")
    B = sp.csr_matrix((v2[order], c2[order], np.concatenate([[0], np.cumsum(2 * cnt)])), shape=A.shape)
    assert B.nnz == 2 * A.nnz
    return B


def _fp32_values(A):
    """the canonical matrix (duplicates summed in fp64, as the BSR conversion does) with values rounded to float32"""
    B = sp.csr_matrix((A.data.copy(), A.indices.copy(), A.indptr.copy()), shape=A.shape)
    B.sum_duplicates()
    B.data = B.data.astype(np.float32).astype(np.float64)
    return B


def _vec(rng, n, zeros=0.1):
    v = rng.standard_normal(n)
    v[rng.random(n) < zeros] = 0.0
    return v


# ---------------------------------------------------------------------------------------------------------------------
# what the next product launches: a replica of the dispatch and chunking of spmv.cu / bsr.cu / bsr_tma.cu
# ---------------------------------------------------------------------------------------------------------------------
def _group_lanes(avg):
    return next((g for g, t in ((1, 1.5), (2, 4), (4, 12), (8, 48), (16, 160)) if avg <= t), 32)


def _vector_lanes(avg):
    return next((l for l, t in ((2, 3), (4, 6), (8, 12), (16, 24)) if avg <= t), 32)


def _pack(rp, cap, max_rows):
    """chunks [r0, r1) of whole rows with at most cap entries and max_rows rows; None if one row exceeds cap"""
    out, r, n = [], 0, len(rp) - 1
    while r < n:
        hi = min(int(np.searchsorted(rp, rp[r] + cap, side="right")) - 1, r + max_rows)
        if hi <= r:
            return None
        out.append((r, hi))
        r = hi
    return out


def _pack_tma(rp, cap):
    out, r, n = [], 0, len(rp) - 1
    while r < n:
        hi = min(int(np.searchsorted(rp, rp[r] + cap, side="right")) - 1, r + TMA_MAX_BROWS)
        if hi <= r:
            return None
        best, best_w = hi, 1e300
        for h in range(hi, max(r, hi - 4), -1):       # among the last admissible boundaries, the least padding per block
            cnt = int(rp[h] - rp[r])
            if cnt <= 0:
                continue
            w = (((cnt + 31) & ~31) - cnt) / cnt + (0.0 if h == hi else 0.004 * (hi - h))
            if w < best_w:
                best_w, best = w, h
        out.append((r, best))
        r = best
    return out


def _block_pattern(A, bs):
    rows = np.repeat(np.arange(A.shape[0]), np.diff(A.indptr))
    P = sp.csr_matrix((np.ones(A.nnz), (rows // bs, A.indices // bs)), shape=(A.shape[0] // bs, A.shape[1] // bs))
    P.sum_duplicates()
    return P, bool(np.all(rows % bs == A.indices % bs))


def _predict(A, hint, opts, fp32):
    nr, nc = A.shape
    info = dict.fromkeys(INFO, 0)
    info["tma_cfg"] = -1
    bs = 0 if hint <= 1 else 3 if hint % 3 == 0 else 2 if hint % 2 == 0 else 0
    if bs and nr > 0 and nr % bs == 0 and nc % bs == 0 and A.nnz > 0:
        P, diag = _block_pattern(A, bs)
        nbr, nnzb = P.shape[0], P.nnz
        ne = bs if diag else bs * bs
        pref = nnzb >= PREF_MIN_AVG * nbr and int(opts.get("-poro_bsr_prefetch", 1)) != 0
        chunks = _pack(P.indptr, BSR_CAP, BSR_THREADS // bs if pref else BSR_MAX_BROWS)
        if nnzb * (8.0 * ne + 4.0) <= float(opts.get("-poro_bsr_max_fill", DEFAULT_MAX_FILL)) * 8.44 * A.nnz and chunks:
            cfg = int(opts.get("-poro_bsr_tma_cfg", 1))
            tma = None if fp32 or not int(opts.get("-poro_bsr_tma", 0)) else _pack_tma(P.indptr, TMA_CAP[cfg])
            l2 = int(opts.get("-poro_bsr_l2_prefetch_chunks", 0))
            info.update(format=DIAG_BSR if diag else BSR, lanes=_group_lanes(nnzb / nbr), bs=bs, fp32=int(fp32))
            if tma:
                info.update(tma=1, tma_cfg=cfg, chunks=len(tma))
            else:
                info.update(pref=int(pref), coop=int(int(opts.get("-poro_bsr_coop_gather", 0)) != 0 and not fp32),
                            chunks=len(chunks), l2_prefetch=int(0 < l2 and -(-nnzb // BSR_CAP) > 2 * l2))
            return info
    blocks = _pack(A.indptr, CSR_CAP, CSR_MAX_ROWS)
    avg = A.nnz / nr if nr else 0.0
    if blocks is None:
        info.update(format=VECTOR_CSR, lanes=_vector_lanes(avg))
    else:
        info.update(format=CSR_STREAM, lanes=_group_lanes(avg), chunks=len(blocks))
    return info


# ---------------------------------------------------------------------------------------------------------------------
# device side
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def ctx(gpu_ctx):
    """the session context with a clean option set before and after (the -poro_bsr_* options stick to a context)"""
    gpu_ctx.clear_options()
    yield gpu_ctx
    gpu_ctx.clear_options()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _info(ctx, m):
    from poro_b200 import _capi
    out = (C.c_int64 * len(INFO))()
    _capi.check(ctx.lib.poro_mat_kernel_info(m.h, out, len(INFO)))
    return dict(zip(INFO, list(out)))


def _upload(ctx, A, hint=0, opts=None, fp32=False):
    """uploads A with the conversion options in force and converts it as its first product would; the -poro_bsr_* options
    are read at that conversion, so they are cleared only afterwards"""
    from poro_b200 import _capi
    ctx.clear_options()
    opts = {k: (v(A) if callable(v) else v) for k, v in (opts or {}).items()}
    for k, v in opts.items():
        ctx.set_option(k, v)
    if hint:
        ctx.set_option("-poro_mat_block_hint", hint)
    if fp32:
        ctx.set_option("-poro_mat_fp32_values", 1)
    m = _capi.Mat(ctx, A.indptr, A.indices, A.data, A.shape)
    info = _info(ctx, m)
    ctx.clear_options()
    return m, info, opts


def _dev(v):
    import torch
    return None if v is None else torch.tensor(np.asarray(v, np.float64), device="cuda")


def _nan(n):
    import torch
    return torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")


def _mult_mode(ctx, m, mode, x, z=None, r=None, dinv=None, xv=None, alias=False):
    """one product through poro_mat_mult_mode on fresh device copies; unwritten outputs stay NaN"""
    import torch
    from poro_b200 import _capi
    nr = m.shape[0]
    t = {k: _dev(v) for k, v in dict(x=x, z=z, r=r, dinv=dinv, xv=xv).items()}
    y = t["z"] if alias else _nan(nr)
    dn, dot = _nan(nr), _nan(1)
    torch.cuda.synchronize()
    _capi.check(ctx.lib.poro_mat_mult_mode(m.h, mode, _ptr(t["x"]), _ptr(y), _ptr(t["z"]), _ptr(t["r"]), _ptr(dn),
                                           _ptr(t["xv"]), _ptr(t["dinv"]), C1, C2, _ptr(dot)))
    out = {"y": y, "x": t["x"], "d_new": dn, "dot": dot, "r": t["r"], "xv": t["xv"]}
    return {k: v.cpu().numpy() for k, v in out.items() if v is not None}


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def _check_modes(ctx, m, terms, rng, label):
    """every epilogue mode (3 and 4 for square matrices) within its bound, modes 1 / 2 also with z aliasing y; x untouched
    by the Chebyshev step; a second call gives identical bits.  Returns the mode-0 output."""
    nr, nc = terms[0][0].shape
    square = nr == nc
    x = terms[0][1]
    z, r, xv = _vec(rng, nr, 0.0), _vec(rng, nr, 0.0), _vec(rng, nr, 0.0)
    dinv = rng.uniform(0.5, 2.0, nr) * 10.0 ** rng.uniform(-3, 3, nr)
    want = _epilogue_refs(_Ref(terms), x, z, r, dinv, xv, x if square else None)
    run = (lambda mode, alias: _mult_mode(ctx, m, mode, x, z=z if mode in (1, 2) else None, alias=alias,
                                                 **(dict(r=r, dinv=dinv, xv=xv) if mode == 3 else {})))
    plan = [(0, False, {"y": "y"}), (1, False, {"y": "sub"}), (1, True, {"y": "sub"}), (2, False, {"y": "add"}),
            (2, True, {"y": "add"})]
    if square:
        plan += [(3, False, {"r": "r", "d_new": "d_new", "xv": "xv"}), (4, False, {"y": "y", "dot": "dot"})]
    y0 = None
    for mode, alias, checks in plan:
        a, b = run(mode, alias), run(mode, alias)
        for key, name in checks.items():
            _assert_rows(a[key], *want[name], "%s mode %d%s %s" % (label, mode, " (z = y)" if alias else "", key))
            assert _same_bits(a[key], b[key]), "%s mode %d %s differs between two calls" % (label, mode, key)
        if mode == 3:
            assert _same_bits(a["x"], np.asarray(x, np.float64)), "%s: the Chebyshev step wrote its input" % label
        if mode == 0:
            y0 = a["y"]
    return y0, want["y"]


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------
# cases: name -> builder(rng, sm) -> dict(A, hint, opts, fp32, expect); `expect` holds what the case is about
# ---------------------------------------------------------------------------------------------------------------------
CASES = {}


def _case(name, scalar=False):
    def reg(f):
        CASES[name] = (f, scalar)
        return f
    return reg


# CSR stream: the average row length at each G threshold and just above it
for _avg, _g in ((1.5, 1), (4, 2), (12, 4), (48, 8), (160, 16)):
    def _at(rng, sm, avg=_avg, g=_g):
        n = 2000 if avg < 20 else 400
        return dict(A=_scalar(rng, _avg_lens(rng, n, int(avg * n)), n), expect=dict(format=CSR_STREAM, lanes=g))

    def _above(rng, sm, avg=_avg, g=_g):
        n = 2000 if avg < 20 else 400
        return dict(A=_scalar(rng, _avg_lens(rng, n, int(avg * n) + 1), n), expect=dict(format=CSR_STREAM, lanes=2 * g))
    _case("csr_avg_%g" % _avg, True)(_at)
    _case("csr_avg_above_%g" % _avg, True)(_above)


@_case("csr_block_ends_at_cap", True)
def _(rng, sm):
    return dict(A=_scalar(rng, np.full(64, CSR_CAP // 8), 512), expect=dict(format=CSR_STREAM, chunks=8))


@_case("csr_row_of_cap", True)
def _(rng, sm):
    lens = _avg_lens(rng, 2100, 6000)
    lens[700] = CSR_CAP
    return dict(A=_scalar(rng, lens), expect=dict(format=CSR_STREAM))


@_case("csr_empty_run_over_row_cap", True)
def _(rng, sm):
    lens = _avg_lens(rng, 3000, 15000)
    lens[500:500 + CSR_MAX_ROWS + 476] = 0
    return dict(A=_scalar(rng, lens), expect=dict(format=CSR_STREAM))


@_case("csr_all_rows_empty", True)
def _(rng, sm):
    return dict(A=sp.csr_matrix((3000, 3000)), expect=dict(format=CSR_STREAM, chunks=3))


@_case("csr_1x1", True)
def _(rng, sm):
    return dict(A=_scalar(rng, [1], 1), expect=dict(format=CSR_STREAM, chunks=1))


@_case("csr_tall", True)
def _(rng, sm):
    return dict(A=_scalar(rng, rng.integers(0, 8, 5000), 7), expect=dict(format=CSR_STREAM))


@_case("csr_wide", True)
def _(rng, sm):
    return dict(A=_scalar(rng, np.full(20, 1500), 30000), expect=dict(format=CSR_STREAM, lanes=32, chunks=20))


# vector-CSR fallback: one row longer than a row block, averages giving each L
for _avg, _l in ((2.5, 2), (5, 4), (10, 8), (20, 16), (40, 32)):
    def _vec_case(rng, sm, avg=_avg, l=_l):
        n = 2200
        lens = np.concatenate([[CSR_CAP + 1], _avg_lens(rng, n - 1, int(avg * n) - CSR_CAP - 1)])
        return dict(A=_scalar(rng, rng.permutation(lens)), expect=dict(format=VECTOR_CSR, lanes=l))
    _case("vector_csr_L%d" % _l, True)(_vec_case)


def _fill_ratio(A, bs):
    P, diag = _block_pattern(A, bs)
    return P.nnz * (8.0 * (bs if diag else bs * bs) + 4.0) / (8.44 * A.nnz)


# plain block-CSR, BS 2 and 3
for _bs in (2, 3):
    def _reg(name, bs=_bs):
        return _case("bsr%d_%s" % (bs, name))

    _reg("dense_pref")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 300, 6 * 300), bs), hint=bs,
                                                    expect=dict(format=BSR, bs=bs, pref=1)))
    _reg("dense_nopref")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 300, 6 * 300 - 1), bs), hint=bs,
                                                      expect=dict(format=BSR, bs=bs, pref=0)))
    _reg("diag")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 300, 6 * 300), bs, diag=True), hint=bs,
                                              expect=dict(format=DIAG_BSR, bs=bs, pref=1)))

    def _one_offdiag(rng, sm, bs=_bs):
        A = _block(rng, _avg_lens(rng, 300, 6 * 300), bs, diag=True).tolil()
        A[4 * bs, 7 * bs + 1] = 2.5
        return dict(A=A.tocsr(), hint=bs, opts={"-poro_bsr_max_fill": 10}, expect=dict(format=BSR, bs=bs))
    _reg("diag_plus_one_offdiag")(_one_offdiag)

    def _long_row(rng, sm, bs=_bs, nb=BSR_CAP, fmt=BSR):
        lens = _avg_lens(rng, 8, 40)
        lens[3] = nb
        return dict(A=_block(rng, lens, bs, nbcols=600), hint=bs, expect=dict(format=fmt))
    _reg("row_of_cap")(_long_row)
    _case("bsr%d_row_over_cap_falls_back_to_csr" % _bs, True)(lambda rng, sm, bs=_bs: _long_row(rng, sm, bs, BSR_CAP + 1, CSR_STREAM))

    def _row_cap_pref(rng, sm, bs=_bs):
        short, long_ = (5, 7) if bs == 3 else (3, 9)         # average 6: PREF on; the short rows hit the row cap first
        cap = BSR_THREADS // bs
        n = 4 * cap
        lens = np.concatenate([np.full(n, short), np.full(n, long_)])
        return dict(A=_block(rng, lens, bs), hint=bs,
                    expect=dict(format=BSR, pref=1, chunks=4 + len(_pack(np.arange(n + 1) * long_, BSR_CAP, cap))))
    _reg("row_cap_pref")(_row_cap_pref)
    _reg("row_cap_nopref")(lambda rng, sm, bs=_bs: dict(A=_block(rng, np.ones(1000, int), bs), hint=bs,
                                                        expect=dict(format=BSR, pref=0, chunks=-(-1000 // BSR_MAX_BROWS))))
    _reg("rectangular")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 200, 1200), bs, nbcols=350), hint=bs,
                                                     expect=dict(format=BSR)))

    def _ragged(rng, sm, bs=_bs):
        A = _block(rng, _avg_lens(rng, 200, 1200), bs)
        extra = _scalar(rng, [5], A.shape[1])
        return dict(A=sp.vstack([A, extra], format="csr"), hint=bs, expect=dict(format=CSR_STREAM))
    _reg("rows_not_multiple_of_bs_refused")(_ragged)
    for _side, _f in (("accepted", 1 + 1e-6), ("refused", 1 - 1e-6)):
        _reg("fill_just_%s" % _side)(lambda rng, sm, bs=_bs, f=_f, side=_side: dict(
            A=_block(rng, _avg_lens(rng, 300, 1800), bs), hint=bs,
            opts={"-poro_bsr_max_fill": lambda A, bs=bs, f=f: repr(_fill_ratio(A, bs) * f)},
            expect=dict(format=BSR if side == "accepted" else CSR_STREAM)))
    _reg("prefetch_off")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 300, 1800), bs), hint=bs,
                                                      opts={"-poro_bsr_prefetch": 0}, expect=dict(format=BSR, pref=0)))
    _reg("coop_gather")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 300, 1800), bs), hint=bs,
                                                     opts={"-poro_bsr_coop_gather": 1}, expect=dict(format=BSR, coop=1)))
    _reg("l2_prefetch")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 1000, 6000), bs), hint=bs,
                                                     opts={"-poro_bsr_l2_prefetch_chunks": 4},
                                                     expect=dict(format=BSR, l2_prefetch=1)))
    _reg("fp32_values")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 300, 1800), bs), hint=bs, fp32=True,
                                                     expect=dict(format=BSR, fp32=1)))
    _reg("coop_with_fp32_values")(lambda rng, sm, bs=_bs: dict(A=_block(rng, _avg_lens(rng, 300, 1800), bs), hint=bs,
                                                               fp32=True, opts={"-poro_bsr_coop_gather": 1},
                                                               expect=dict(format=BSR, fp32=1, coop=0)))


# persistent TMA block-CSR, the three pipeline configs
for _cfg, _bs in ((0, 3), (1, 2), (2, 3)):
    def _treg(name, cfg=_cfg):
        return _case("tma%d_%s" % (cfg, name))

    def _topts(cfg):
        return {"-poro_bsr_tma": 1, "-poro_bsr_tma_cfg": cfg}

    _treg("one_row_chunks")(lambda rng, sm, cfg=_cfg, bs=_bs: dict(
        A=_block(rng, np.full(10, TMA_CAP[cfg] // 2 + 20), bs, nbcols=TMA_CAP[cfg]), hint=bs, opts=_topts(cfg),
        expect=dict(tma=1, tma_cfg=cfg, chunks=10)))
    _treg("row_cap")(lambda rng, sm, cfg=_cfg, bs=_bs: dict(
        A=_block(rng, np.ones(64 * 5, int), bs), hint=bs, opts=_topts(cfg), expect=dict(tma=1, tma_cfg=cfg, chunks=5)))
    if TMA_CAP[_cfg] < BSR_CAP:
        def _over(rng, sm, cfg=_cfg, bs=_bs):
            lens = _avg_lens(rng, 40, 200)
            lens[17] = TMA_CAP[cfg] + 1
            return dict(A=_block(rng, lens, bs, nbcols=400), hint=bs, opts=_topts(cfg), expect=dict(format=BSR, tma=0))
        _treg("row_over_chunk_cap_plain")(_over)

    def _wrap(rng, sm, cfg=_cfg):
        grid = TMA_MIN_CTAS[cfg] * sm
        nchunk = (2 * TMA_STAGES[cfg] + 1) * grid + 3          # every CTA walks its ring more than twice
        return dict(A=_block(rng, np.ones(TMA_MAX_BROWS * nchunk, int), 2, diag=True), hint=2, opts=_topts(cfg),
                    expect=dict(format=DIAG_BSR, tma=1, tma_cfg=cfg, chunks=nchunk))
    _treg("parity_wraps")(_wrap)

    def _empty_runs(rng, sm, cfg=_cfg, bs=_bs):
        lens = np.concatenate([_avg_lens(rng, 100, 600), np.zeros(150, int), _avg_lens(rng, 100, 600), np.zeros(130, int)])
        return dict(A=_block(rng, lens, bs), hint=bs, opts=_topts(cfg), expect=dict(tma=1, tma_cfg=cfg))
    _treg("empty_block_row_runs")(_empty_runs)


@pytest.mark.gpu
@pytest.mark.parametrize("canonical", [True, False], ids=["canonical", "duplicates"])
@pytest.mark.parametrize("name", list(CASES))
def test_spmv_variant_matches_longdouble(ctx, name, canonical):
    build, scalar = CASES[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    case = build(rng, _sm_count())
    A = case["A"] if canonical else _noncanonical(case["A"], rng)
    m, info, opts = _upload(ctx, A, case.get("hint", 0), case.get("opts"), case.get("fp32", False))
    assert info == _predict(A, case.get("hint", 0), opts, case.get("fp32", False)), (name, info)
    if canonical or not scalar:         # a CSR case changes its row lengths with the duplicates; block cases do not
        for k, v in case["expect"].items():
            assert info[k] == v, (name, k, info)
    if name.endswith("empty_block_row_runs"):
        P, _ = _block_pattern(A, case["hint"])
        assert any(P.indptr[b] == P.indptr[a] for a, b in _pack_tma(P.indptr, TMA_CAP[info["tma_cfg"]]))
    x = _vec(rng, A.shape[1])
    terms = [(_fp32_values(A) if info["fp32"] else A, x)]
    y0, (want64, bound64) = _check_modes(ctx, m, terms, rng, name)
    if info["fp32"]:                    # the values really were stored in fp32
        assert len(_outside(y0, _Ref([(A, x)]).ax, _Ref([(A, x)]).bound())) > 0


# ---------------------------------------------------------------------------------------------------------------------
# fused mass coupling y = A x + C x2
# ---------------------------------------------------------------------------------------------------------------------
def _coupling(A, bs, rng, defect=None):
    """C = c M (x) I on A's block pattern: one scalar per block on its diagonal; per block row a component mask (Dirichlet
    rows of the coupling: absent or explicit zeros).  `defect` adds one thing fusion must refuse."""
    P, _ = _block_pattern(A, bs)
    I = np.repeat(np.arange(P.shape[0]), np.diff(P.indptr))
    J = P.indices
    full = (1 << bs) - 1
    masks = rng.choice([full, full, 0b101 if bs == 3 else 0b01, 0b010 if bs == 3 else 0b10, 0], P.shape[0])
    m = rng.standard_normal(len(I)) * 10.0 ** rng.uniform(-3, 3, len(I))
    rows, cols, vals = [], [], []
    for q in range(bs):
        on = (masks[I] >> q) & 1 == 1
        zero = ~on & (rng.random(len(I)) < 0.5)
        keep = on | zero
        rows.append(I[keep] * bs + q)
        cols.append(J[keep] * bs + q)
        vals.append(np.where(on[keep], m[keep], 0.0))
    rows, cols, vals = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    Cm = sp.csr_matrix((vals, (rows, cols)), shape=A.shape)
    Cm.sort_indices()
    if defect == "unequal":              # two different values on the diagonal of one block
        Cm = Cm.tolil()
        I0 = int(np.flatnonzero(masks[I] == full)[0])
        Cm[I[I0] * bs + 1, J[I0] * bs + 1] = 1.5 * m[I0]
    elif defect == "off_block_diagonal":
        Cm = Cm.tolil()
        Cm[I[0] * bs, J[0] * bs + 1] = 0.75
    elif defect == "outside_pattern":
        Cm = Cm.tolil()
        free = np.setdiff1d(np.arange(P.shape[1]), P.indices[P.indptr[5]:P.indptr[6]])
        Cm[5 * bs, free[0] * bs] = 0.5
    Cm = Cm.tocsr()
    Cm.sort_indices()
    if defect == "duplicate":            # one entry stored twice (adjacent, so the row stays sorted)
        k = int(np.flatnonzero(Cm.data != 0)[0])
        row = int(np.searchsorted(Cm.indptr, k, side="right") - 1)
        data = np.insert(Cm.data, k, 0.25 * Cm.data[k])
        data[k + 1] *= 0.75
        indptr = Cm.indptr.copy()
        indptr[row + 1:] += 1
        Cm = sp.csr_matrix((data, np.insert(Cm.indices, k, Cm.indices[k]), indptr), shape=Cm.shape)
    return Cm


FUSED = [(bs, tma, defect) for bs in (2, 3) for tma in (None, 1 if bs == 2 else 2)
         for defect in (None, "unequal", "off_block_diagonal", "outside_pattern", "duplicate", "fp32")]


@pytest.mark.gpu
@pytest.mark.parametrize("canonical", [True, False], ids=["canonical", "duplicates"])
@pytest.mark.parametrize("bs,tma,defect", FUSED, ids=["bsr%d_%s_%s" % (b, "tma%d" % t if t is not None else "plain", d or "fused")
                                                      for b, t, d in FUSED])
def test_fused_coupling_matches_longdouble(ctx, bs, tma, defect, canonical):
    import torch
    from poro_b200 import _capi
    rng = np.random.default_rng(zlib.crc32(("fused%d%s%s" % (bs, tma, defect)).encode()))
    A0 = _block(rng, _avg_lens(rng, 240, 240 * 7), bs)
    Cm = _coupling(A0, bs, rng, None if defect == "fp32" else defect)
    A = A0 if canonical else _noncanonical(A0, rng)
    opts = {"-poro_bsr_tma": 1, "-poro_bsr_tma_cfg": tma} if tma is not None else {}
    m, info, _ = _upload(ctx, A, bs, opts, fp32=defect == "fp32")
    mc, _, _ = _upload(ctx, Cm)
    # fp32 value storage keeps the plain layout (bsr_from_csr builds no TMA chunks for it), so its fusion is tried there
    tma_layout = tma is not None and defect != "fp32"
    assert info["format"] == BSR and info["tma"] == int(tma_layout) and info["fp32"] == int(defect == "fp32"), info
    x, x2 = _vec(rng, A.shape[1]), _vec(rng, A.shape[1])
    fused = C.c_int(-1)

    def run(mode, alias):
        z = _vec(np.random.default_rng(mode), A.shape[0], 0.0)
        t = {k: _dev(v) for k, v in dict(x=x, x2=x2, z=z).items()}
        y = t["z"] if alias else _nan(A.shape[0])
        torch.cuda.synchronize()
        _capi.check(ctx.lib.poro_mat_mult_fused(m.h, mc.h, mode, _ptr(t["x"]), _ptr(t["x2"]), _ptr(y),
                                                _ptr(t["z"]) if mode else None, C.byref(fused)))
        return {"y": y.cpu().numpy()}

    # the reference's z is the one `run` draws for each mode
    Av = _fp32_values(A) if defect == "fp32" else A
    ref = _Ref([(Av, x), (Cm, x2)])
    for mode, alias in ((0, False), (1, False), (1, True), (2, False), (2, True)):
        z = _vec(np.random.default_rng(mode), A.shape[0], 0.0)
        want = (ref.ax, ref.bound()) if mode == 0 else ((z - ref.ax if mode == 1 else z + ref.ax), ref.bound(z))
        a, b = run(mode, alias), run(mode, alias)
        _assert_rows(a["y"], *want, "fused bs=%d tma=%s %s mode %d" % (bs, tma, defect, mode))
        assert _same_bits(a["y"], b["y"])
    assert fused.value == int(defect is None), (defect, fused.value)
    assert _info(ctx, m)["fused"] == int(defect is None)


# ---------------------------------------------------------------------------------------------------------------------
# all variants of one matrix are the same operator
# ---------------------------------------------------------------------------------------------------------------------
VARIANTS = {"csr": ({"-poro_use_bsr": 0}, dict(format=CSR_STREAM)),
            "plain": ({}, dict(format=BSR, pref=1, tma=0)),
            "prefetch_off": ({"-poro_bsr_prefetch": 0}, dict(pref=0)),
            "coop": ({"-poro_bsr_coop_gather": 1}, dict(coop=1)),
            "l2_prefetch": ({"-poro_bsr_l2_prefetch_chunks": 4}, dict(l2_prefetch=1)),
            **{"tma%d" % k: ({"-poro_bsr_tma": 1, "-poro_bsr_tma_cfg": k}, dict(tma=1, tma_cfg=k)) for k in range(3)}}


@pytest.mark.gpu
@pytest.mark.parametrize("bs", [2, 3])
def test_variants_of_one_matrix_agree(ctx, bs):
    rng = np.random.default_rng(bs)
    A = _block(rng, _avg_lens(rng, 1500, 1500 * 7), bs)
    x = _vec(rng, A.shape[1])
    ref = _Ref([(A, x)])
    ys = {}
    for name, (opts, expect) in VARIANTS.items():
        m, info, _ = _upload(ctx, A, bs, opts)
        assert all(info[k] == v for k, v in expect.items()), (name, info)
        y = _mult_mode(ctx, m, 0, x)["y"]
        _assert_rows(y, ref.ax, ref.bound(), name)
        ys[name] = y
    names = list(ys)
    for i, a in enumerate(names):
        for b in names[i + 1:]:
            assert np.all(np.abs(ys[a].astype(LD) - ys[b]) <= 2 * ref.bound()), (a, b)


# ---------------------------------------------------------------------------------------------------------------------
# the outer operator of a solve built from a non-canonical upload
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dim,N", [(2, 8), (3, 4)])
def test_outer_operator_from_noncanonical_upload(ctx, dim, N):
    """Identity field order cuts the BSR parts of the outer operator out of the raw CSR as it was uploaded, duplicates
    included: its products and a solve with it must be those of the canonical system."""
    import bench
    import torch
    from test_gpu_stencil_apply import _setup
    from poro_b200.lib.backend import DeviceMatrix, DeviceVector
    from poro_b200.lib.Solver import Solver
    A, P, Pd, b, imap, pc, par, bcs = _setup(ctx, dim, N, "diagonal", bench.BENCH_OPTIONS)
    rng = np.random.default_rng(dim)
    As = A.to_scipy().tocsr()
    An = _noncanonical(As, rng)
    Ad = DeviceMatrix(An, ctx=ctx)
    solver = Solver(Ad, None, pc, par, imap)
    solver.create_solver(Ad, None, pc)
    assert any(f in (BSR, DIAG_BSR, 3) for _, f in solver.solver.parts_info()), solver.solver.parts_info()
    x = _vec(rng, As.shape[0])
    y = torch.full((As.shape[0],), float("nan"), dtype=torch.float64, device="cuda")
    solver.solver.mult(torch.tensor(x, device="cuda"), y)
    torch.cuda.synchronize()
    ref = _Ref([(An, x)])
    _assert_rows(y.cpu().numpy(), ref.ax, ref.bound(), "outer operator dim %d" % dim)
    db, dx = DeviceVector(b, ctx=ctx), DeviceVector(n=len(b), ctx=ctx)
    s = Solver(Ad, db, pc, par, imap)
    s.create_solver(Ad, db, pc)
    s.solve(db, dx)
    assert s.solver.reason > 0
    res = np.linalg.norm(b - As @ dx.numpy()) / np.linalg.norm(b)
    assert res <= 1e-9, res


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the comparator sees what a norm-wise check cannot
# ---------------------------------------------------------------------------------------------------------------------
def test_rowwise_bound_sees_a_dropped_entry_that_a_normwise_check_accepts():
    rng = np.random.default_rng(7)
    A = _scalar(rng, _avg_lens(rng, 400, 400 * 9))
    x = _vec(rng, A.shape[1])
    ref = _Ref([(A, x)])
    assert ref.ax.dtype == LD and LD(1) + LD(2.0 ** -60) != LD(1)         # the reference really carries extra bits
    rowscale = np.array([np.abs(A.data[A.indptr[i]:A.indptr[i + 1]]).max(initial=0.0) for i in range(A.shape[0])])
    i = int(np.argmin(np.where(rowscale > 0, rowscale, np.inf)))          # the smallest-scaled non-empty row
    lo, hi = A.indptr[i], A.indptr[i + 1]
    contrib = np.abs(A.data[lo:hi] * x[A.indices[lo:hi]])
    tol = 1e-13 * float(np.linalg.norm(ref.ax.astype(np.float64)))
    k = lo + int(np.argmax(np.where(contrib <= tol, contrib, -1.0)))
    assert 0 < abs(A.data[k] * x[A.indices[k]]) <= tol
    dropped = A.copy()
    dropped.data[k] = 0.0
    y = (_ld(dropped) @ np.asarray(x, LD)).astype(np.float64)
    assert np.linalg.norm(y - ref.ax.astype(np.float64)) <= 1e-13 * np.linalg.norm(ref.ax.astype(np.float64))
    assert list(_outside(y, ref.ax, ref.bound())) == [i]
    assert len(_outside(ref.ax.astype(np.float64), ref.ax, ref.bound())) == 0   # the rounded reference itself passes
