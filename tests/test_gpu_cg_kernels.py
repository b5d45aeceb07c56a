"""The kernels of the fused CG iteration, called through the C ABI (ctypes, raw device pointers):

  b2s_spmv_csr_dot       q = A p and p.q in one pass, on every consumer of the SpMV kernels
  b2s_cg_update          x += alpha p ; r -= alpha q ; rr = r.r
  b2s_cg_pupdate         p = r + beta p   (rho1 == 0: p = r)
  b2s_axpby, b2s_dot, b2s_nrm2 and the reuse of one reduction workspace
  peer stores            b2s_spmv_csr_bcast, b2s_cg_pupdate_bcast / _halo, local buffers standing in for peers
  b2s_allreduce_board    with one rank

Two kinds of reference.

EXACT: small integers for every matrix value and vector entry, and scalar ratios whose divisor is a power of
two with a zero imaginary part, so every product and every partial sum is an integer.  Each test asserts
that the sum of the magnitudes of the terms stays below 2^24 (f32 / c64) or 2^53 (f64 / c128); then every
summation order gives the same bits, and the kernels must match an int64 reference BIT FOR BIT.  A
dropped, duplicated or misassigned term fails, whatever its size.

ROUNDING: random data against a reference in a wider type (f64 for f32 / c64, long double for f64 / c128),
element by element against a rounding bound (C_ROUND below).  This catches accumulation in too narrow a
type, which integer data cannot.
"""
import contextlib
import ctypes
from ctypes import byref, c_int64, c_void_p

import numpy as np
import pytest
import torch

from legate_sparse import _native as N

pytestmark = pytest.mark.gpu

NULL = c_void_p(0)
B2S_ERR_ARG = 1   # include/b200sparse.h
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]
VT = {np.float32: N.B2S_F32, np.float64: N.B2S_F64, np.complex64: N.B2S_C64, np.complex128: N.B2S_C128}
MANT = {np.float32: 24, np.float64: 53, np.complex64: 24, np.complex128: 53}   # significand bits
EXT = {np.float32: np.float64, np.float64: np.longdouble, np.complex64: np.complex128,
       np.complex128: np.clongdouble}                                          # reference type of the ROUNDING tests
REAL = {np.float32: np.float32, np.float64: np.float64, np.complex64: np.float32, np.complex128: np.float64}
# The rounding bounds are C_ROUND * (number of terms) * u * (sum of the magnitudes of the terms), u = 2^-MANT.
# A complex product alone is off by up to 2*sqrt(2) u |a||x|; every addition adds at most u times the
# running magnitude.
C_ROUND = 4
# the vector kernels run at most 1184 CTAs (8 per SM) of 256 threads x 4 packs of 16 bytes; past this many
# packs every thread strides over more packs
GRID_CAP_PACKS = 1184 * 256 * 4


def _name(dt):
    return np.dtype(dt).name


def _cplx(dt):
    return np.dtype(dt).kind == "c"


def _pack(dt):
    """elements per 16-byte pack (the vector path of the vector kernels)"""
    return 16 // np.dtype(dt).itemsize


def _misalign(dt):
    """byte offset that breaks 16-byte alignment but keeps the element type's own alignment
    (c128 is 8-byte aligned in numpy)"""
    return min(np.dtype(dt).itemsize, 8)


class _Dev:
    """device copy of a numpy array, placed `off` bytes past the start of a fresh allocation"""

    def __init__(self, a, off=0):
        a = np.ascontiguousarray(a)
        self.dtype, self.n, self.off = a.dtype, a.size, off
        self.buf = torch.empty(off + max(a.nbytes, 16), dtype=torch.uint8, device="cuda")
        assert self.buf.data_ptr() % 256 == 0
        if a.nbytes:
            self.buf[off:off + a.nbytes].copy_(torch.from_numpy(a.reshape(-1).view(np.uint8)))

    @property
    def ptr(self):
        return c_void_p(self.buf.data_ptr() + self.off)

    def get(self):
        return self.buf[self.off:self.off + self.n * self.dtype.itemsize].cpu().numpy().view(self.dtype)


def _peer_array(ptrs):
    arr = (c_void_p * len(ptrs))(*ptrs)
    return arr, ctypes.cast(arr, c_void_p)


def _assert_bits(got, want, what):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, want.dtype, got.shape, want.shape)
    if got.size == 0:
        return
    g = got.reshape(-1).view(np.uint8).reshape(got.size, -1)
    w = want.reshape(-1).view(np.uint8).reshape(want.size, -1)
    bad = np.flatnonzero((g != w).any(axis=1))
    assert bad.size == 0, (f"{what}: {bad.size} of {got.size} elements differ, first at {bad[0]}: "
                           f"{got.reshape(-1)[bad[0]]!r} != {want.reshape(-1)[bad[0]]!r}")


# ------------------------------------------------------------------ exact integer arithmetic
# An integer-valued real or complex array is carried as a pair (re, im) of int64 arrays.
def _ip(a):
    a = np.asarray(a)
    re, im = a.real.astype(np.int64), np.imag(a).astype(np.int64)
    assert np.array_equal(re, a.real) and np.array_equal(im, np.imag(a)), "not integer valued"
    return re, im


def _imul(a, b):
    return a[0] * b[0] - a[1] * b[1], a[0] * b[1] + a[1] * b[0]


def _iadd(a, b):
    return a[0] + b[0], a[1] + b[1]


def _iconj(a):
    return a[0], -a[1]


def _isum(a):
    return np.int64(a[0].sum()), np.int64(a[1].sum())


def _mag(a):
    """|re| + |im|: bounds both components of anything multiplied by it"""
    return np.abs(a[0]) + np.abs(a[1])


def _ito(a, dt):
    out = np.empty(np.shape(a[0]), dt)
    if _cplx(dt):
        out.real, out.imag = a[0], a[1]
    else:
        assert not np.any(a[1])
        out[...] = a[0]
    return out


def _scalar(dt, re, im=0):
    """a device-scalar value: the imaginary part is dropped for real types"""
    return (re, im if _cplx(dt) else 0)


def _peak(a):
    return int(np.max(a, initial=0))


def _assert_exact(bound, dt, what):
    assert int(bound) < 2 ** MANT[dt], f"{what}: integer data too large to stay exact ({int(bound)} >= 2^{MANT[dt]})"


def _ints(rng, n, dt, hi, nonzero=False, density=1.0):
    """integer-valued array, components uniform in [-hi, hi] (nonzero: in +-{1..hi}); `density`: the
    fraction of entries left non-zero"""
    def comp():
        if nonzero:
            return rng.integers(1, hi + 1, size=n) * rng.choice(np.array([-1, 1]), size=n)
        return rng.integers(-hi, hi + 1, size=n)

    a = np.empty(n, dt)
    if _cplx(dt):
        a.real, a.imag = comp(), comp()
    else:
        a[:] = comp()
    if density < 1.0:
        a[rng.random(n) >= density] = 0
    return a


def _rand(rng, n, dt):
    a = rng.standard_normal(n)
    if _cplx(dt):
        a = a + 1j * rng.standard_normal(n)
    return a.astype(dt)


def _nan(n, dt):
    return np.full(n, complex(np.nan, np.nan) if _cplx(dt) else np.nan, dt)


def _segsum(v, indptr):
    """per-row sums of v (rows given by indptr), in v's dtype, summed left to right; empty rows give 0"""
    out = np.zeros(len(indptr) - 1, v.dtype)
    nonempty = np.flatnonzero(np.diff(indptr) > 0)
    if nonempty.size:
        out[nonempty] = np.add.reduceat(v, indptr[:-1][nonempty])
    return out


def _isegsum(a, indptr):
    cs = [np.concatenate([[0], np.cumsum(c)]) for c in a]
    return tuple(c[indptr[1:]] - c[indptr[:-1]] for c in cs)


# ------------------------------------------------------------------ SpMV cases
# b2s_spmv_csr_dot always runs with variant AUTO; the consumer is steered by the plan (tile size, x
# windows) and the alignment of the arrays.  Each case: (consumer, tile nnz, banded matrix, 16-byte
# misaligned index / value views).
#   rowwalk  : pipe kernel, every tile stages its x window (banded matrix) -> row-walk consumer, 2-stage ring
#   products : pipe kernel, B2S_SPMV_NO_WINDOW=1 -> two ping-pong products groups; 3-stage ring for
#              1024-nnz tiles, 2-stage for 2048
#   tile     : register-staged tile kernel, 256 threads x IPT = tile/256 non-zeros: misaligned views
#              (scalar loads) or a 4096-nnz plan, which the pipe kernel does not take (128-bit loads)
SPMV_CASES = {
    "rowwalk-1024": ("rowwalk", 1024, True, False),
    "rowwalk-2048": ("rowwalk", 2048, True, False),
    "products-1024": ("products", 1024, False, False),
    "products-2048": ("products", 2048, False, False),
    "tile-ipt4-window": ("tile", 1024, True, True),
    "tile-ipt8-gather": ("tile", 2048, False, True),
    "tile-ipt16-window": ("tile", 4096, True, True),
    "tile-ipt16-vec": ("tile", 4096, False, False),
}
# the plain b2s_spmv_csr of these cases may run another kernel than the fused one: for skewed row lengths
# and 1024-nnz tiles it takes the async-gather kernel (4- and 8-byte values) or the long-row pass
PLAIN_MAY_DIFFER = {"products-1024"}
ITYPES = {"i32": (N.B2S_I32, np.int32), "i64": (N.B2S_I64, np.int64)}
BAND = 40   # banded matrices: columns within +-BAND of the diagonal


def _pattern(rng, T, banded, ncols_mod4, seg_rows=800):
    """CSR pattern with the rows where tile ownership goes wrong: empty rows first, in the middle, on a
    tile boundary and last; a row of exactly one tile starting on a tile boundary and one straddling two
    tiles; a row spanning 4 or 5 tiles (the tiles inside it hold no row start).  Banded: ncols is
    ncols_mod4 (mod 4) and the last rows reach the last column, so the x window of the last tile runs
    into the tail of x."""
    def seg():
        return list(rng.integers(0, 15, size=seg_rows))

    deg = [0, 0, 0] + seg() + [0] * 7 + seg()
    deg.append(-sum(deg) % T)                # pad up to a tile boundary (0: one more empty row)
    deg += [T, 0, 0, 0] + seg()              # a whole tile, then three empty rows on the next boundary
    if sum(deg) % T == 0:
        deg.append(1)
    deg += [T] + seg() + [3 * T + T // 3] + seg() + [0] * 4
    deg = np.array(deg, dtype=np.int64)
    nrows = len(deg)
    ncols = nrows + (ncols_mod4 - nrows) % 4 + (0 if banded else 997 * 4)
    indptr = np.zeros(nrows + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    rows = np.repeat(np.arange(nrows), deg)
    if banded:
        center = rows * (ncols - 1) // (nrows - 1)
        cols = np.clip(center + rng.integers(-BAND, BAND + 1, size=rows.size), 0, ncols - 1)
    else:
        cols = rng.integers(0, ncols, size=rows.size)
    return indptr, cols, ncols


class _Csr:
    """one SpMV case on the device: matrix, x, w, plan"""

    def __init__(self, lib, case, dt, itype, rng, exact, seg_rows=800):
        consumer, T, banded, misaligned = SPMV_CASES[case]
        self.lib, self.case, self.dt, self.consumer = lib, case, dt, consumer
        self.it, idt = ITYPES[itype]
        self.indptr, cols, self.ncols = _pattern(rng, T, banded, 1 + list(SPMV_CASES).index(case) % 3, seg_rows)
        self.cols = cols.astype(idt)
        self.nrows, self.nnz = len(self.indptr) - 1, int(self.indptr[-1])
        if exact:   # 24-bit types get smaller integers so that the sums stay below 2^24
            ha, hx = (2, 4) if MANT[dt] == 24 else (4, 8)
            self.data = _ints(rng, self.nnz, dt, ha, nonzero=True)
            self.x, self.w = _ints(rng, self.ncols, dt, hx), _ints(rng, self.nrows, dt, hx)
        else:
            self.data, self.x, self.w = _rand(rng, self.nnz, dt), _rand(rng, self.ncols, dt), _rand(rng, self.nrows, dt)
        self.ip = _Dev(self.indptr)
        self.ix = _Dev(self.cols, off=self.cols.itemsize if misaligned else 0)
        self.dv = _Dev(self.data, off=self.data.itemsize if misaligned else 0)
        if misaligned:
            assert self.ix.buf.data_ptr() % 16 == 0 and (self.ix.buf.data_ptr() + self.ix.off) % 16 != 0
        self.xd, self.wd = _Dev(self.x), _Dev(self.w)
        nbytes = lib.b2s_spmv_plan_workspace_bytes(self.nrows, self.nnz)
        self.ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        self.plan = c_void_p(0)
        assert lib.b2s_spmv_plan_create(self.it, self.nrows, self.ncols, self.nnz, self.ip.ptr, self.ix.ptr,
                                        c_void_p(self.ws.data_ptr()), nbytes, NULL, byref(self.plan)) == 0, N.last_error()
        nt, tn, wt = c_int64(0), c_int64(0), c_int64(0)
        assert lib.b2s_spmv_plan_info(self.plan, byref(nt), byref(tn), byref(wt)) == 0
        self.ntiles, self.window_tiles = nt.value, wt.value
        assert tn.value == T, (case, tn.value)
        if consumer == "rowwalk" or (consumer == "tile" and banded):
            assert self.window_tiles == self.ntiles, (case, self.window_tiles, self.ntiles)

    def args(self):
        return (VT[self.dt], self.it, self.nrows, self.ncols, self.nnz, self.ip.ptr, self.ix.ptr, self.dv.ptr)

    def dot(self):
        y, d = _Dev(_nan(self.nrows, self.dt)), _Dev(_nan(1, self.dt))
        assert self.lib.b2s_spmv_csr_dot(*self.args(), self.xd.ptr, y.ptr, self.wd.ptr, self.plan, d.ptr,
                                         NULL) == 0, N.last_error()
        return y.get(), d.get()

    def plain(self):
        y = _Dev(_nan(self.nrows, self.dt))
        assert self.lib.b2s_spmv_csr(*self.args(), self.xd.ptr, y.ptr, self.plan, N.B2S_SPMV_AUTO, NULL) == 0, N.last_error()
        return y.get()

    def exact_reference(self):
        """y = A x and w.y in int64, after checking that every partial sum of the kernels stays exact"""
        a, x, w = _ip(self.data), _ip(self.x), _ip(self.w)
        xc = (x[0][self.cols], x[1][self.cols])
        y = _isegsum(_imul(a, xc), self.indptr)
        # row pieces and dot terms (w[r] * piece of row r) are all bounded by |w_r| * sum_j |a_rj||x_j|
        row_mag = _isegsum((_mag(a) * _mag(xc), np.zeros(self.nnz, np.int64)), self.indptr)[0]
        _assert_exact((np.maximum(_mag(w), 1) * row_mag).sum(), self.dt, self.case)
        return _ito(y, self.dt), _ito(_isum(_imul(w, y)), self.dt).reshape(1)


@contextlib.contextmanager
def _csr(monkeypatch, case, dt, itype, rng, exact, seg_rows=800, ctas=None):
    consumer, T, _, _ = SPMV_CASES[case]
    monkeypatch.setenv("B2S_SPMV_TILE_NNZ", str(T))
    for var in ("B2S_SPMV_NO_WINDOW", "B2S_SPMV_CTAS"):
        monkeypatch.delenv(var, raising=False)
    if consumer == "products":
        monkeypatch.setenv("B2S_SPMV_NO_WINDOW", "1")
    if ctas is not None:
        monkeypatch.setenv("B2S_SPMV_CTAS", str(ctas))
    m = _Csr(N.load(), case, dt, itype, rng, exact, seg_rows)
    try:
        yield m
    finally:
        m.lib.b2s_spmv_plan_destroy(m.plan)


@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
@pytest.mark.parametrize("case", list(SPMV_CASES))
def test_spmv_dot_exact(monkeypatch, case, dtype, itype):
    """integer data: y and w.y bit-exact on every consumer, the same bits on a second call, and the
    plain SpMV gives the same y"""
    rng = np.random.default_rng([list(SPMV_CASES).index(case), DTYPES.index(dtype), list(ITYPES).index(itype)])
    with _csr(monkeypatch, case, dtype, itype, rng, exact=True) as m:
        y_ref, d_ref = m.exact_reference()
        y, d = m.dot()
        _assert_bits(y, y_ref, "y")
        _assert_bits(d, d_ref, "w.y")
        y2, d2 = m.dot()
        _assert_bits(y2, y, "y, second call")
        _assert_bits(d2, d, "w.y, second call")
        _assert_bits(m.plain(), y_ref, "y of b2s_spmv_csr")


@pytest.mark.parametrize("case,ctas", [("rowwalk-1024", 1), ("products-1024", 1), ("tile-ipt4-window", None)])
def test_spmv_dot_exact_many_tiles(monkeypatch, case, ctas):
    """~1400 tiles.  One resident CTA per SM on the pipe kernel: each CTA (each products group) carries its
    dot partial across several tiles.  The tile kernel writes one partial per tile: more than 1024 of
    them, so the final reduction loops over its partials."""
    rng = np.random.default_rng(77 + list(SPMV_CASES).index(case))
    with _csr(monkeypatch, case, np.float64, "i32", rng, exact=True, seg_rows=40000, ctas=ctas) as m:
        assert m.ntiles > 1024
        y_ref, d_ref = m.exact_reference()
        y, d = m.dot()
        _assert_bits(y, y_ref, "y")
        _assert_bits(d, d_ref, "w.y")


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
@pytest.mark.parametrize("case", list(SPMV_CASES))
def test_spmv_dot_rounding_bound(monkeypatch, case, dtype):
    """random data: every y[r] and w.y within a rounding bound of a wider-type reference"""
    rng = np.random.default_rng([100 + list(SPMV_CASES).index(case), DTYPES.index(dtype)])
    with _csr(monkeypatch, case, dtype, "i32", rng, exact=False) as m:
        ext, u = EXT[dtype], 2.0 ** -MANT[dtype]
        xc = m.x[m.cols]
        y_ref = _segsum(m.data.astype(ext) * xc.astype(ext), m.indptr)
        row_mag = _segsum(np.abs(m.data).astype(np.float64) * np.abs(xc), m.indptr)   # sum_j |a_rj||x_j|
        lens = np.diff(m.indptr)
        y, d = m.dot()

        def check_y(got, what):
            err = np.abs(got.astype(ext) - y_ref)
            bound = C_ROUND * lens * u * row_mag
            bad = np.flatnonzero(err > bound)
            assert bad.size == 0, f"{what}: row {bad[0]} (len {lens[bad[0]]}) off by {err[bad[0]]}, bound {bound[bad[0]]}"

        check_y(y, "y")
        # dot: the kernels add w[r] * (piece of row r in a tile); the pieces of a row that straddles tiles may
        # cancel, so the magnitude is sum_r |w_r| sum_j |a_rj||x_j|, not sum_r |w_r y_r|
        mag = float((np.abs(m.w).astype(np.float64) * row_mag).sum())
        terms = m.nrows + m.ntiles
        d_ref = (m.w.astype(ext) * y_ref).sum()
        assert abs(d[0].astype(ext) - d_ref) <= C_ROUND * (terms + lens.max()) * u * mag, (d[0], d_ref)
        # the reduction alone, against the y the kernel returned
        d_ret = (m.w.astype(ext) * y.astype(ext)).sum()
        assert abs(d[0].astype(ext) - d_ret) <= C_ROUND * terms * u * mag, (d[0], d_ret)
        y2, d2 = m.dot()
        _assert_bits(y2, y, "y, second call")
        _assert_bits(d2, d, "w.y, second call")
        if case in PLAIN_MAY_DIFFER:
            check_y(m.plain(), "y of b2s_spmv_csr")
        else:
            _assert_bits(m.plain(), y, "y of b2s_spmv_csr")


def _kernel_template_args(names, kernel):
    hits = [n for n in names if kernel + "<" in n]
    assert len(hits) == 1, (kernel, names)
    return [a.strip() for a in hits[0].split(kernel + "<", 1)[1].split(">", 1)[0].split(",")]


@pytest.mark.parametrize("case", list(SPMV_CASES))
def test_spmv_dot_runs_the_named_consumer(monkeypatch, case):
    """the kernel each case of the tests above steers b2s_spmv_csr_dot to, read from a kernel trace"""
    from torch.profiler import ProfilerActivity, profile

    consumer, T, banded, misaligned = SPMV_CASES[case]
    with _csr(monkeypatch, case, np.float64, "i32", np.random.default_rng(5), exact=True) as m:
        m.dot()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
            m.dot()
            torch.cuda.synchronize()
        names = sorted({e.key for e in prof.key_averages()})
    b = lambda v: "true" if v else "false"   # noqa: E731
    if consumer == "tile":
        # spmv_tile_kernel<V, I, IPT, VEC, WINDOW, DOT>
        assert not any("spmv_pipe_kernel<" in n for n in names), names
        assert _kernel_template_args(names, "spmv_tile_kernel")[2:] == [str(T // 256), b(not misaligned), b(banded), "true"]
    else:
        # spmv_pipe_kernel<V, I, TILE, STAGES, WINDOW, DOT, BCAST, NG, LONGROWS>
        want = [str(T), "2", "true", "true", "false", "1", "false"] if consumer == "rowwalk" else \
               [str(T), "3" if T == 1024 else "2", "false", "true", "false", "2", "false"]
        assert _kernel_template_args(names, "spmv_pipe_kernel")[2:] == want


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_spmv_dot_edge_calls(dtype):
    lib = N.load()
    vt = VT[dtype]
    # no rows: dot_out = 0
    ip0 = _Dev(np.zeros(1, np.int64))
    ws = torch.zeros(lib.b2s_spmv_plan_workspace_bytes(0, 0), dtype=torch.uint8, device="cuda")
    plan = c_void_p(0)
    assert lib.b2s_spmv_plan_create(N.B2S_I32, 0, 5, 0, ip0.ptr, NULL, c_void_p(ws.data_ptr()), ws.numel(), NULL, byref(plan)) == 0
    d = _Dev(_nan(1, dtype))
    assert lib.b2s_spmv_csr_dot(vt, N.B2S_I32, 0, 5, 0, ip0.ptr, NULL, NULL, NULL, NULL, NULL, plan, d.ptr, NULL) == 0
    _assert_bits(d.get(), np.zeros(1, dtype), "dot of 0 rows")
    lib.b2s_spmv_plan_destroy(plan)
    # rows but no non-zeros: y = 0 and dot_out = 0 (y and dot_out start as NaN)
    ip = _Dev(np.zeros(8, np.int64))
    x, w, y, d = _Dev(np.ones(5, dtype)), _Dev(np.ones(7, dtype)), _Dev(_nan(7, dtype)), _Dev(_nan(1, dtype))
    plan = c_void_p(0)
    assert lib.b2s_spmv_plan_create(N.B2S_I32, 7, 5, 0, ip.ptr, NULL, c_void_p(ws.data_ptr()), ws.numel(), NULL, byref(plan)) == 0
    assert lib.b2s_spmv_csr_dot(vt, N.B2S_I32, 7, 5, 0, ip.ptr, NULL, NULL, x.ptr, y.ptr, w.ptr, plan, d.ptr, NULL) == 0
    _assert_bits(y.get(), np.zeros(7, dtype), "y of an empty matrix")
    _assert_bits(d.get(), np.zeros(1, dtype), "dot of an empty matrix")
    # refused: w missing while there are rows, no plan, no dot_out
    assert lib.b2s_spmv_csr_dot(vt, N.B2S_I32, 7, 5, 0, ip.ptr, NULL, NULL, x.ptr, y.ptr, NULL, plan, d.ptr, NULL) == B2S_ERR_ARG
    assert lib.b2s_spmv_csr_dot(vt, N.B2S_I32, 7, 5, 0, ip.ptr, NULL, NULL, x.ptr, y.ptr, w.ptr, NULL, d.ptr, NULL) == B2S_ERR_ARG
    assert lib.b2s_spmv_csr_dot(vt, N.B2S_I32, 7, 5, 0, ip.ptr, NULL, NULL, x.ptr, y.ptr, w.ptr, plan, NULL, NULL) == B2S_ERR_ARG
    lib.b2s_spmv_plan_destroy(plan)


# ------------------------------------------------------------------ vector kernels
def _vec_sizes(dt):
    n = _pack(dt)
    return sorted({0, 1, n - 1, n, n + 1, 1023, n * (GRID_CAP_PACKS + 4099) + n - 1})


VEC_CASES = [pytest.param(dt, n, id=f"{_name(dt)}-{n}") for dt in DTYPES for n in _vec_sizes(dt)]
# every array 16-byte aligned (vector path); the LAST array of a call shifted by a few bytes (scalar
# path); every array shifted by one 16-byte pack (vector path on views)
VIEWS = ("aligned", "last-unaligned", "pack-offset")


def _offsets(view, k, dt):
    if view == "aligned":
        return [0] * k
    if view == "pack-offset":
        return [16] * k
    return [0] * (k - 1) + [_misalign(dt)]


def _sparse_density(n, dt, budget):
    """24-bit types at the large sizes: keep roughly `budget` non-zeros so the sums stay exact"""
    return 1.0 if MANT[dt] == 53 or n <= budget else budget / n


@pytest.mark.parametrize("dtype,n", VEC_CASES)
def test_cg_update_exact(dtype, n):
    """x += alpha p ; r -= alpha q ; rr = sum r*r (no conjugation), alpha = rho/pq with pq = 4"""
    lib = N.load()
    rng = np.random.default_rng([1, DTYPES.index(dtype), n])
    alpha = _scalar(dtype, -2, 1)
    rho, pq = _ito((np.int64(4 * alpha[0]), np.int64(4 * alpha[1])), dtype), _ito(_scalar(dtype, 4), dtype)
    x = _ints(rng, n, dtype, 8)
    p, q = _ints(rng, n, dtype, 4, nonzero=True), _ints(rng, n, dtype, 4, nonzero=True)   # every x, r changes
    r_new = _ip(_ints(rng, n, dtype, 3, density=0.2))
    r = _iadd(r_new, _imul(alpha, _ip(q)))          # r - alpha q == r_new
    x_new = _iadd(_ip(x), _imul(alpha, _ip(p)))
    rr = _isum(_imul(r_new, r_new))
    _assert_exact(max(_peak(_mag(_ip(x)) + 3 * _mag(_ip(p))), _peak(_mag(r) + 3 * _mag(_ip(q)))), dtype, "x, r")
    _assert_exact(_mag(r_new).astype(np.int64) @ _mag(r_new), dtype, "r.r")
    ws = torch.zeros(lib.b2s_reduce_workspace_bytes(), dtype=torch.uint8, device="cuda")
    for view in VIEWS:
        o = _offsets(view, 4, dtype)
        X, R, Pd, Q = _Dev(x, o[0]), _Dev(_ito(r, dtype), o[1]), _Dev(p, o[2]), _Dev(q, o[3])
        out = _Dev(_nan(1, dtype))
        assert lib.b2s_cg_update(VT[dtype], n, X.ptr, R.ptr, Pd.ptr, Q.ptr, _Dev(rho).ptr, _Dev(pq).ptr, out.ptr,
                                 c_void_p(ws.data_ptr()), NULL) == 0, N.last_error()
        _assert_bits(X.get(), _ito(x_new, dtype), f"x ({view})")
        _assert_bits(R.get(), _ito(r_new, dtype), f"r ({view})")
        _assert_bits(out.get(), _ito(rr, dtype).reshape(1), f"rr ({view})")


def _zeros_of(dt):
    """rho1 values that mean 'first step'"""
    return [complex(0.0, 0.0), complex(-0.0, -0.0), complex(-0.0, 0.0)] if _cplx(dt) else [0.0, -0.0]


@pytest.mark.parametrize("dtype,n", VEC_CASES)
def test_cg_pupdate_exact(dtype, n):
    """first step (rho1 == 0, p full of NaN: p must not be read) gives p = r; then p = r + (rho/rho1) p"""
    lib = N.load()
    rng = np.random.default_rng([2, DTYPES.index(dtype), n])
    beta = _scalar(dtype, -2, 3)
    rho, rho1 = _ito((np.int64(-2 * beta[0]), np.int64(-2 * beta[1])), dtype), _ito(_scalar(dtype, -2), dtype)
    r, p = _ints(rng, n, dtype, 8), _ints(rng, n, dtype, 8, nonzero=True)
    p_new = _iadd(_ip(r), _imul(beta, _ip(p)))
    _assert_exact(_peak(_mag(_ip(r)) + 5 * _mag(_ip(p))), dtype, "p")
    for view in VIEWS:
        o = _offsets(view, 2, dtype)
        R = _Dev(r, o[1])
        for z in _zeros_of(dtype):
            Pd = _Dev(_nan(n, dtype), o[0])
            assert lib.b2s_cg_pupdate(VT[dtype], n, Pd.ptr, R.ptr, _Dev(rho).ptr, _Dev(np.array([z], dtype)).ptr, NULL) == 0
            _assert_bits(Pd.get(), r, f"first step, rho1 = {z} ({view})")
        Pd = _Dev(p, o[0])
        assert lib.b2s_cg_pupdate(VT[dtype], n, Pd.ptr, R.ptr, _Dev(rho).ptr, _Dev(rho1).ptr, NULL) == 0
        _assert_bits(Pd.get(), _ito(p_new, dtype), f"p ({view})")


@pytest.mark.parametrize("dtype,n", VEC_CASES)
def test_axpby_exact(dtype, n):
    """val = a/b (b = 4), negated if asked; isalpha: y = val x + y, else y = x + val y"""
    lib = N.load()
    rng = np.random.default_rng([3, DTYPES.index(dtype), n])
    val = _scalar(dtype, 2, 1)
    a, b = _ito((np.int64(4 * val[0]), np.int64(4 * val[1])), dtype), _ito(_scalar(dtype, 4), dtype)
    x, y = _ints(rng, n, dtype, 8), _ints(rng, n, dtype, 8)
    _assert_exact(_peak(3 * _mag(_ip(x)) + 3 * _mag(_ip(y))), dtype, "axpby")
    for isalpha in (0, 1):
        for negate in (0, 1):
            v = (-val[0], -val[1]) if negate else val
            want = _iadd(_imul(v, _ip(x)), _ip(y)) if isalpha else _iadd(_ip(x), _imul(v, _ip(y)))
            for view in VIEWS:
                o = _offsets(view, 2, dtype)
                Y, X = _Dev(y, o[0]), _Dev(x, o[1])
                assert lib.b2s_axpby(VT[dtype], n, Y.ptr, X.ptr, _Dev(a).ptr, _Dev(b).ptr, isalpha, negate, NULL) == 0
                _assert_bits(Y.get(), _ito(want, dtype), f"isalpha={isalpha} negate={negate} ({view})")


def _dot_data(rng, n, dt):
    """x, y and their exact dot / vdot"""
    x, y = _ints(rng, n, dt, 8), _ints(rng, n, dt, 8)
    zero = rng.random(n) >= _sparse_density(n, dt, 50000)
    x[zero], y[zero] = 0, 0
    k = min(n, _pack(dt) + 1)                       # the pack tail is never empty
    if k:
        x[n - k:], y[n - k:] = _ints(rng, k, dt, 8, nonzero=True), _ints(rng, k, dt, 8, nonzero=True)
    _assert_exact(_mag(_ip(x)) @ _mag(_ip(y)), dt, "dot")
    return x, y, _ito(_isum(_imul(_ip(x), _ip(y))), dt), _ito(_isum(_imul(_iconj(_ip(x)), _ip(y))), dt)


def _square_norm_data(rng, n, dt):
    """integer vector whose sum of squares is a perfect square k^2: with S = sum_{i>0} |z_i|^2,
    z_0^2 + S = k^2 has the integer solution k - z_0 = 1 (S odd) or 2 (S = 0 mod 4)"""
    z = _ints(rng, n, dt, 2, density=_sparse_density(n, dt, 500))
    if n == 0:
        return z, 0

    def sq(a):
        re, im = _ip(a)
        return int((re * re + im * im).sum())

    s = sq(z[1:])
    if s % 4 == 2:               # no solution: replace the last entry by 1 or 2, whichever makes S odd
        s -= sq(z[n - 1:])
        z[n - 1] = 1 if (s + 1) % 2 else 2
        s += sq(z[n - 1:])
    k, z0 = ((s + 1) // 2, (s - 1) // 2) if s % 2 else (s // 4 + 1, s // 4 - 1)
    z[0] = z0
    _assert_exact(k * k, dt, "nrm2")
    return z, k


@pytest.mark.parametrize("dtype,n", VEC_CASES)
def test_dot_nrm2_exact(dtype, n):
    lib = N.load()
    rng = np.random.default_rng([4, DTYPES.index(dtype), n])
    x, y, d_ref, v_ref = _dot_data(rng, n, dtype)
    z, k = _square_norm_data(rng, n, dtype)
    ws = torch.zeros(lib.b2s_reduce_workspace_bytes(), dtype=torch.uint8, device="cuda")
    for view in VIEWS:
        o = _offsets(view, 2, dtype)
        X, Y = _Dev(x, o[0]), _Dev(y, o[1])
        for conj, want in ((0, d_ref), (1, v_ref)):
            out = _Dev(_nan(1, dtype))
            assert lib.b2s_dot(VT[dtype], n, X.ptr, Y.ptr, conj, out.ptr, c_void_p(ws.data_ptr()), NULL) == 0
            _assert_bits(out.get(), want.reshape(1), f"dot conj={conj} ({view})")
        Z, out = _Dev(z, o[1]), _Dev(_nan(1, REAL[dtype]))
        assert lib.b2s_nrm2(VT[dtype], n, Z.ptr, out.ptr, c_void_p(ws.data_ptr()), NULL) == 0
        _assert_bits(out.get(), np.array([k], REAL[dtype]), f"nrm2 ({view})")


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_reduce_workspace_reuse(dtype):
    """dot, nrm2 and cg_update on ONE workspace with grids of 1184, 1 and 1184 CTAs in turn: the last CTA
    is found by an atomicInc that must leave the counter at 0 for the next call, whatever its grid"""
    lib = N.load()
    rng = np.random.default_rng([5, DTYPES.index(dtype)])
    big, small = _vec_sizes(dtype)[-1], 5
    wsb = torch.zeros(lib.b2s_reduce_workspace_bytes(), dtype=torch.uint8, device="cuda")   # zeroed once
    ws = c_void_p(wsb.data_ptr())

    def dot(n):
        x, y, d_ref, _ = _dot_data(rng, n, dtype)
        out = _Dev(_nan(1, dtype))
        assert lib.b2s_dot(VT[dtype], n, _Dev(x).ptr, _Dev(y).ptr, 0, out.ptr, ws, NULL) == 0
        _assert_bits(out.get(), d_ref.reshape(1), f"dot n={n}")

    def nrm2(n):
        z, k = _square_norm_data(rng, n, dtype)
        out = _Dev(_nan(1, REAL[dtype]))
        assert lib.b2s_nrm2(VT[dtype], n, _Dev(z).ptr, out.ptr, ws, NULL) == 0
        _assert_bits(out.get(), np.array([k], REAL[dtype]), f"nrm2 n={n}")

    def cg_update(n):   # alpha = 1: x += p, r -= q, rr = r.r
        x, p, r, q = (_ints(rng, n, dtype, 3, density=_sparse_density(n, dtype, 50000)) for _ in range(4))
        one = _ito(_scalar(dtype, 1), dtype)
        r_new = _iadd(_ip(r), (-_ip(q)[0], -_ip(q)[1]))
        X, R, out = _Dev(x), _Dev(r), _Dev(_nan(1, dtype))
        assert lib.b2s_cg_update(VT[dtype], n, X.ptr, R.ptr, _Dev(p).ptr, _Dev(q).ptr, _Dev(one).ptr, _Dev(one).ptr,
                                 out.ptr, ws, NULL) == 0
        _assert_exact(_mag(r_new) @ _mag(r_new), dtype, "r.r")
        _assert_bits(X.get(), _ito(_iadd(_ip(x), _ip(p)), dtype), f"x n={n}")
        _assert_bits(R.get(), _ito(r_new, dtype), f"r n={n}")
        _assert_bits(out.get(), _ito(_isum(_imul(r_new, r_new)), dtype).reshape(1), f"rr n={n}")

    for step in (lambda: dot(big), lambda: nrm2(small), lambda: cg_update(big), lambda: dot(small),
                 lambda: nrm2(big), lambda: cg_update(small), lambda: dot(big)):
        step()


# ------------------------------------------------------------------ peer stores (local buffers as peers)
def _sentinel(dt):
    return np.array([complex(-12345.25, 777.5) if _cplx(dt) else -12345.25], dt)[0]


class _Peers:
    """one buffer per peer; peer g's block of n elements starts 256 + offs[g] bytes into its buffer (as a
    rank's block sits inside the replicated vector of another rank) and holds sentinels, the bytes around
    it a filler pattern"""

    def __init__(self, n, dt, offs, margin=256):
        self.n, self.dt, self.isz = n, dt, np.dtype(dt).itemsize
        self.lo = [margin + o for o in offs]                             # byte offset of the block
        self.init = []
        for lo in self.lo:
            init = np.full(lo + n * self.isz + margin, 0xA5, np.uint8)
            init[lo:lo + n * self.isz] = np.full(n, _sentinel(dt), dt).view(np.uint8)
            self.init.append(init)
        self.bufs = [_Dev(init) for init in self.init]
        self.arr, self.ptr = _peer_array([c_void_p(b.buf.data_ptr() + lo) for b, lo in zip(self.bufs, self.lo)])

    def check(self, g, want, written, maybe=None, what=""):
        """peer g: the block holds `want` where `written` and the sentinel elsewhere (where `maybe`: either);
        the bytes around the block are untouched"""
        raw, init = self.bufs[g].get(), self.init[g]
        a, b = self.lo[g], self.lo[g] + self.n * self.isz
        assert np.array_equal(raw[:a], init[:a]) and np.array_equal(raw[b:], init[b:]), \
            f"peer {g}: stores outside the block {what}"
        blk = raw[a:b].copy().view(self.dt)
        exp = np.where(written, want, np.full(self.n, _sentinel(self.dt), self.dt))
        if maybe is not None:
            same = (blk.view(np.uint8).reshape(self.n, -1) == want.view(np.uint8).reshape(self.n, -1)).all(axis=1)
            exp = np.where(maybe & same, want, exp)
        _assert_bits(blk, exp, f"peer {g} {what}")


@pytest.mark.parametrize("npeers", [1, 3, 7])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
@pytest.mark.parametrize("case", ["rowwalk-2048", "products-1024"])
def test_spmv_bcast_peers_hold_final_y(monkeypatch, case, dtype, npeers):
    """every peer receives the FINAL y (rows straddling tiles are completed by the fix-up kernel, which
    stores to the peers as well), and nothing outside the block"""
    rng = np.random.default_rng([200 + npeers, DTYPES.index(dtype), len(case)])
    with _csr(monkeypatch, case, dtype, "i32", rng, exact=True) as m:
        y_ref, _ = m.exact_reference()
        isz = np.dtype(dtype).itemsize
        peers = _Peers(m.nrows, dtype, [isz * (3 * g + 1) for g in range(npeers)])
        y = _Dev(_nan(m.nrows, dtype))
        assert m.lib.b2s_spmv_csr_bcast(*m.args(), m.xd.ptr, y.ptr, peers.ptr, npeers, m.plan, NULL) == 0, N.last_error()
        _assert_bits(y.get(), y_ref, "local y")
        everywhere = np.ones(m.nrows, bool)
        for g in range(npeers):
            peers.check(g, y_ref, everywhere)


@pytest.mark.parametrize("peer_view", ["pack-offset", "unaligned"])
@pytest.mark.parametrize("npeers", [1, 3, 7])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_cg_pupdate_bcast_peers(dtype, npeers, peer_view):
    """p = r + beta p stored to every peer as well; first step with p full of NaN.  Peers offset by whole
    16-byte packs keep the vector path, one unaligned peer sends the whole call down the scalar path."""
    lib = N.load()
    rng = np.random.default_rng([300 + npeers, DTYPES.index(dtype)])
    n = 1000 * _pack(dtype) + _pack(dtype) - 1
    beta = _scalar(dtype, 3, -1)
    rho, rho1 = _ito((np.int64(4 * beta[0]), np.int64(4 * beta[1])), dtype), _ito(_scalar(dtype, 4), dtype)
    r, p = _ints(rng, n, dtype, 8), _ints(rng, n, dtype, 8)
    p_new = _ito(_iadd(_ip(r), _imul(beta, _ip(p))), dtype)
    offs = [16 * (g + 1) for g in range(npeers)]
    if peer_view == "unaligned":
        offs[-1] += _misalign(dtype)
    everywhere = np.ones(n, bool)
    for first in (True, False):
        peers = _Peers(n, dtype, offs)
        Pd, R = _Dev(_nan(n, dtype) if first else p), _Dev(r)
        d = _Dev(np.zeros(1, dtype) if first else rho1)
        assert lib.b2s_cg_pupdate_bcast(VT[dtype], n, Pd.ptr, R.ptr, _Dev(rho).ptr, d.ptr, peers.ptr, npeers, NULL) == 0
        want = r if first else p_new
        _assert_bits(Pd.get(), want, "local p")
        for g in range(npeers):
            peers.check(g, want, everywhere, what="first step" if first else "")


def _halo_ranges(n, pk):
    m = n // pk
    return [
        (5, 5),                                 # empty (hi == lo)
        (1, 0),                                 # empty (hi < lo): a peer that never reads this block
        (0, n),                                 # everything
        (10 * pk, 20 * pk),                     # middle, on pack boundaries
        (pk * (m - 3) + 1, n - 1),              # ends inside the scalar tail
        (5 * pk + pk - 1, 9 * pk + 1),          # starts on the last element of a pack, ends mid-pack
        (2 * pk + 1, 2 * pk + 2),               # one element
    ]


@pytest.mark.parametrize("path", ["vector", "scalar"])
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_cg_pupdate_halo_ranges(dtype, path):
    """peer g receives exactly [lo[g], hi[g]) of p, widened to whole 16-byte packs on the vector path (but
    never beyond the packs, and element by element on the scalar tail); an empty range receives nothing"""
    lib = N.load()
    rng = np.random.default_rng([400, DTYPES.index(dtype), len(path)])
    pk = _pack(dtype)
    n = 40 * pk + pk - 1
    ranges = _halo_ranges(n, pk)
    npeers = len(ranges)
    beta = _scalar(dtype, -1, 2)
    rho, rho1 = _ito((np.int64(2 * beta[0]), np.int64(2 * beta[1])), dtype), _ito(_scalar(dtype, 2), dtype)
    r, p = _ints(rng, n, dtype, 8), _ints(rng, n, dtype, 8)
    p_new = _ito(_iadd(_ip(r), _imul(beta, _ip(p))), dtype)
    offs = [16 * (g + 1) for g in range(npeers)]
    if path == "scalar":
        offs[0] += _misalign(dtype)              # one unaligned peer: the whole call takes the scalar path
    lo = (c_int64 * npeers)(*[a for a, _ in ranges])
    hi = (c_int64 * npeers)(*[b for _, b in ranges])
    idx = np.arange(n)
    packed = idx < (n // pk) * pk
    for first in (True, False):
        peers = _Peers(n, dtype, offs)
        Pd = _Dev(_nan(n, dtype) if first else p)
        d = _Dev(np.zeros(1, dtype) if first else rho1)
        assert lib.b2s_cg_pupdate_halo(VT[dtype], n, Pd.ptr, _Dev(r).ptr, _Dev(rho).ptr, d.ptr, peers.ptr, npeers,
                                       ctypes.cast(lo, c_void_p), ctypes.cast(hi, c_void_p), NULL) == 0, N.last_error()
        want = r if first else p_new
        _assert_bits(Pd.get(), want, "local p")
        for g, (a, b) in enumerate(ranges):
            inside = (idx >= a) & (idx < b)
            widened = inside.copy()
            if path == "vector" and b > a:
                widened |= packed & (idx // pk >= a // pk) & (idx // pk <= (b - 1) // pk)
            peers.check(g, want, inside, maybe=widened & ~inside, what=f"range [{a}, {b}) {path} first={first}")


# ------------------------------------------------------------------ scalar exchange board, one rank
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_allreduce_board_one_rank(dtype):
    """a rank exchanging with itself returns its value unchanged on every channel and both parities of the
    double buffer; prev_out <- cur_out, cur_out <- sum"""
    lib = N.load()
    rng = np.random.default_rng([500, DTYPES.index(dtype)])
    board = torch.zeros(lib.b2s_board_bytes(), dtype=torch.uint8, device="cuda")
    seq = torch.zeros(4, dtype=torch.int64, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    arr, boards = _peer_array([c_void_p(board.data_ptr())])
    cur, prev = _Dev(_rand(rng, 1, dtype)), _Dev(_nan(1, dtype))
    last = cur.get().copy()
    for rep in range(3):
        for ch in range(4):
            v = _rand(rng, 1, dtype)
            io = _Dev(v)
            with_outs = (rep + ch) % 2 == 0
            assert lib.b2s_allreduce_board(VT[dtype], io.ptr, boards, 0, 1, ch, c_void_p(seq.data_ptr()),
                                           cur.ptr if with_outs else NULL, prev.ptr if with_outs else NULL,
                                           c_void_p(err.data_ptr()), NULL) == 0, N.last_error()
            _assert_bits(io.get(), v, f"inout, channel {ch}, call {rep}")
            if with_outs:
                _assert_bits(prev.get(), last, "prev_out")
                _assert_bits(cur.get(), v, "cur_out")
                last = v
    assert seq.cpu().tolist() == [3, 3, 3, 3]
    assert err.item() == 0
    io = _Dev(_rand(rng, 1, dtype))
    for rank, nranks, ch in ((1, 1, 0), (-1, 1, 0), (0, 0, 0), (0, 9, 0), (0, 1, -1), (0, 1, 4)):
        assert lib.b2s_allreduce_board(VT[dtype], io.ptr, boards, rank, nranks, ch, c_void_p(seq.data_ptr()),
                                       NULL, NULL, NULL, NULL) == B2S_ERR_ARG, (rank, nranks, ch)
