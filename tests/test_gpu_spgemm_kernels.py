"""The SpGEMM kernels, called through the C ABI (ctypes, raw device pointers):

  b2s_spgemm_symbolic   per-row products -> row classes -> hash / dense symbolic kernels -> scan -> c_indptr
  b2s_spgemm_numeric    exact nnz per row -> row classes -> hash / dense numeric kernels -> sorted rows of C

Each row of A is routed to one of four kernel families (b2s_spgemm.cu): a warp hash table (<= 128 entries,
lane groups of 8 / 16 / 32), a CTA hash table (<= 1024), a CTA hash table (<= 4096) and a persistent dense
accumulator above that.  The symbolic pass bins rows by product count, the numeric pass by exact nnz, so one
row can take a different family in each pass.  The fixtures below hit every class boundary, every lane
group, hash chains that wrap past the last slot, more dense rows than dense CTAs, and c_indptr scans long
enough to carry across chunks of the block-sum scan.

The reference is an expand -> sort -> reduce Gustavson in numpy (_Gustavson): every product (i, j, a.b) is
expanded, sorted by (i, j) and each run reduced.  Like the kernels (and cuSPARSE) it keeps structural zeros
and gives sorted columns; it also gives each entry's term count and sum of |a||b| (for the rounding bound)
and each row's exact product count.  A CPU test pins it to oracle.spgemm.

Two kinds of check.

EXACT: small integers, both parts non-zero for complex data.  Each check asserts that the sum of the
magnitudes of an entry's terms stays below 2^24 (f32 / c64) or 2^53 (f64 / c128); then every summation order
gives the same bits, and c_indptr, c_indices and c_data must match an int64 reference BIT FOR BIT.  The
kernels add with floating-point atomics, so the order is arbitrary: bit-exact checks need integer data.

ROUNDING: random data against a reference in a wider type (f64 for f32 / c64, long double for f64 / c128),
entry by entry against C_ROUND * terms * u * sum |a||b|.

Run order: c_indptr, nnz(C) and the product count are checked before the numeric call, so a wrong structure
fails before the numeric kernel could write out of bounds.  c_indices and c_data are sized from the reference
nnz plus a guard tail and filled with sentinels: a skipped slot shows up as a sentinel, and the tail must
come back untouched.  The workspace carries guard bytes on both sides as well.
"""
import functools
import re
from ctypes import byref, c_int64, c_void_p

import numpy as np
import pytest
import torch

from legate_sparse import _native as N

gpu = pytest.mark.gpu

NULL = c_void_p(0)
B2S_ERR_WORKSPACE = 3   # include/b200sparse.h
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]
VT = {np.float32: N.B2S_F32, np.float64: N.B2S_F64, np.complex64: N.B2S_C64, np.complex128: N.B2S_C128}
MANT = {np.float32: 24, np.float64: 53, np.complex64: 24, np.complex128: 53}   # significand bits
EXT = {np.float32: np.float64, np.float64: np.longdouble, np.complex64: np.complex128,
       np.complex128: np.clongdouble}                                          # reference type of the ROUNDING tests
ITYPES = {"i32": (N.B2S_I32, np.int32), "i64": (N.B2S_I64, np.int64)}
# Rounding bound: C_ROUND * (terms of the entry) * u * (sum of |a||b| over its terms), u = 2^-MANT.  A complex
# product alone is off by up to 2*sqrt(2) u |a||b|; every addition adds at most u times the running magnitude.
C_ROUND = 4

# Mirrored from b2s_spgemm.cu.
# class_of(): work <= 0 -> no kernel, <= kCap1 -> warp hash, <= kCap2 -> CTA hash, <= kCap3 -> CTA hash,
# above -> dense accumulator.  Work is the product count in the symbolic pass and the exact nnz in the numeric.
CAP1, CAP2, CAP3 = 128, 1024, 4096
# hash tables of the three hash classes (kT1, kT2, kT3 slots)
TABLES = (256, 2048, 8192)
# hash_slot(): the key folded to 32 bits (low word ^ high word), times this constant mod 2^32, top log2(TABLE) bits
HASH_MUL = 0x9E3779B1
# alloc_dense(): at most kNumSMs * 2 persistent dense CTAs; past that many dense rows a CTA takes a second row
DENSE_CTAS = 148 * 2
# dense_row_kernel scans the bitmap 1024 words (32768 columns) per pass
DENSE_PASS_COLS = 1024 * 32

PTR_SENTINEL = -3
IDX_SENTINEL = -7   # not EMPTY (-1), the hash tables' empty key
GUARD = 64          # sentinel elements after c_indices / c_data, bytes after the workspace
WS_HEAD = 256       # bytes before the workspace: it starts on a 256-byte boundary plus ws_off
WS_FILL = 0x5A


def _name(dt):
    return np.dtype(dt).name


def _cplx(dt):
    return np.dtype(dt).kind == "c"


def class_of(w):
    w = np.asarray(w)
    return np.where(w <= 0, 0, np.where(w <= CAP1, 1, np.where(w <= CAP2, 2, np.where(w <= CAP3, 3, 4))))


def lane_group_size(nnzB, nrowsB):
    """lanes per A entry in the warp-class kernels (lane_group_size() in b2s_spgemm.cu)"""
    avg = nnzB / nrowsB if nrowsB > 0 else 32.0
    return 8 if avg <= 12.0 else (16 if avg <= 24.0 else 32)


def hash_slot(key, table):
    k = np.asarray(key, np.int64).astype(np.uint64)
    k = (k & np.uint64(0xFFFFFFFF)) ^ (k >> np.uint64(32))
    return ((k * np.uint64(HASH_MUL)) & np.uint64(0xFFFFFFFF)) >> np.uint64(32 - int(np.log2(table)))


# ------------------------------------------------------------------ helpers
class _Dev:
    """device copy of a numpy array"""

    def __init__(self, a):
        a = np.ascontiguousarray(a)
        self.dtype, self.n = a.dtype, a.size
        self.buf = torch.empty(max(a.nbytes, 16), dtype=torch.uint8, device="cuda")
        if a.nbytes:
            self.buf[:a.nbytes].copy_(torch.from_numpy(a.reshape(-1).view(np.uint8)))

    def at(self, i):
        """pointer to element i"""
        return c_void_p(self.buf.data_ptr() + i * self.dtype.itemsize)

    @property
    def ptr(self):
        return self.at(0)

    def get(self):
        return self.buf[:self.n * self.dtype.itemsize].cpu().numpy().view(self.dtype)


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


def _sentinel(dt):
    return np.array([complex(-12345.25, 777.5) if _cplx(dt) else -12345.25], dt)[0]


# integer-valued real or complex arrays are carried as pairs (re, im) of int64 arrays
def _ip(a):
    a = np.asarray(a)
    re, im = a.real.astype(np.int64), np.imag(a).astype(np.int64)
    assert np.array_equal(re, a.real) and np.array_equal(im, np.imag(a)), "not integer valued"
    return re, im


def _imul(a, b):
    return a[0] * b[0] - a[1] * b[1], a[0] * b[1] + a[1] * b[0]


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


def _ints(rng, n, dt, hi):
    """integer-valued array, every component in +-{1..hi}"""
    def comp():
        return rng.integers(1, hi + 1, size=n) * rng.choice(np.array([-1, 1]), size=n)

    a = np.empty(n, dt)
    if _cplx(dt):
        a.real, a.imag = comp(), comp()
    else:
        a[:] = comp()
    return a


def _exact_values(rng, n, dt):
    """24-bit types get smaller integers so that the sums stay exact"""
    return _ints(rng, n, dt, 2 if MANT[dt] == 24 else 4)


def _rand(rng, n, dt):
    a = rng.standard_normal(n)
    if _cplx(dt):
        a = a + 1j * rng.standard_normal(n)
    return a.astype(dt)


def _segsum(v, indptr):
    out = np.zeros(len(indptr) - 1, v.dtype)
    nonempty = np.flatnonzero(np.diff(indptr) > 0)
    if nonempty.size:
        out[nonempty] = np.add.reduceat(v, indptr[:-1][nonempty])
    return out


# ------------------------------------------------------------------ reference
class _Gustavson:
    """C = A B by expand -> sort -> reduce.  The structure (and the order of the products) depends on the
    patterns only; exact() and rounded() reduce the values of one pair of operands."""

    def __init__(self, a_ptr, a_col, b_ptr, b_col, ncolsB):
        a_ptr, b_ptr = np.asarray(a_ptr, np.int64), np.asarray(b_ptr, np.int64)
        a_col, b_col = np.asarray(a_col, np.int64), np.asarray(b_col, np.int64)
        nrows, nnzA = len(a_ptr) - 1, int(a_ptr[-1])
        per_a = (b_ptr[1:] - b_ptr[:-1])[a_col[:nnzA]]            # products of each A entry
        self.row_products = _segsum(per_a, a_ptr)
        self.products = int(per_a.sum())
        a_of = np.repeat(np.arange(nnzA), per_a)                   # A entry of each product
        first = np.cumsum(per_a) - per_a
        b_of = b_ptr[a_col[a_of]] + (np.arange(self.products) - first[a_of])   # B entry of each product
        rows = np.repeat(np.arange(nrows), np.diff(a_ptr))[a_of]
        cols = b_col[b_of]
        if nrows * max(ncolsB, 1) < 2 ** 62:
            order = np.argsort(rows * ncolsB + cols, kind="stable")
        else:
            order = np.lexsort((cols, rows))
        rows, cols = rows[order], cols[order]
        self.a_of, self.b_of = a_of[order], b_of[order]
        new = np.ones(self.products, bool)
        new[1:] = (rows[1:] != rows[:-1]) | (cols[1:] != cols[:-1])
        self.starts = np.flatnonzero(new)                           # first product of each entry of C
        self.indices = cols[self.starts]
        self.nnz = int(self.starts.size)
        self.indptr = np.zeros(nrows + 1, np.int64)
        np.cumsum(np.bincount(rows[self.starts], minlength=nrows), out=self.indptr[1:])
        self.row_nnz = np.diff(self.indptr)
        self.terms = np.diff(np.append(self.starts, self.products))

    def _reduce(self, v):
        return np.add.reduceat(v, self.starts) if self.nnz else v[:0]

    def exact(self, a_val, b_val, dt):
        """c_data of integer operands, summed in int64, after checking that every order of the float sum is exact"""
        a, b = _ip(a_val[self.a_of]), _ip(b_val[self.b_of])
        c = tuple(self._reduce(t) for t in _imul(a, b))
        mag = self._reduce(_mag(a) * _mag(b))
        assert int(mag.max(initial=0)) < 2 ** MANT[dt], f"integer data too large to stay exact in {_name(dt)}"
        return _ito(c, dt)

    def rounded(self, a_val, b_val, dt):
        """c_data in the wider type EXT[dt] and, per entry, sum |a||b|"""
        ext = EXT[dt]
        a, b = a_val[self.a_of], b_val[self.b_of]
        c = self._reduce(a.astype(ext) * b.astype(ext))
        mag = self._reduce(np.abs(a).astype(np.float64) * np.abs(b).astype(np.float64))
        return c, mag


class _Fx:
    """the patterns of A (nrows x ncolsA) and B (ncolsA x ncolsB), in CSR with int64 arrays"""

    def __init__(self, a_ptr, a_col, b_ptr, b_col, ncolsB):
        self.a_ptr, self.a_col = np.asarray(a_ptr, np.int64), np.asarray(a_col, np.int64)
        self.b_ptr, self.b_col = np.asarray(b_ptr, np.int64), np.asarray(b_col, np.int64)
        self.nrows, self.ncolsA, self.ncolsB = len(self.a_ptr) - 1, len(self.b_ptr) - 1, int(ncolsB)
        self.nnzA, self.nnzB = int(self.a_ptr[-1]), int(self.b_ptr[-1])

    @functools.cached_property
    def ref(self):
        return _Gustavson(self.a_ptr, self.a_col, self.b_ptr, self.b_col, self.ncolsB)


class _Builder:
    """A rows as lists of B rows"""

    def __init__(self, rng, ncolsB):
        self.rng, self.ncolsB = rng, ncolsB
        self.b_rows, self.a_rows = [], []

    def b(self, cols):
        self.b_rows.append(np.asarray(cols, np.int64).reshape(-1))
        return len(self.b_rows) - 1

    def a(self, ks):
        self.a_rows.append(np.asarray(ks, np.int64).reshape(-1))

    def disjoint(self, v, m):
        """an A row with exactly v products and v entries: v distinct columns over m B rows"""
        cols = self.rng.choice(self.ncolsB, v, replace=False)
        cuts = np.sort(self.rng.choice(np.arange(1, v), m - 1, replace=False)) if m > 1 else []
        self.a([self.b(p) for p in np.split(cols, cuts)])

    def overlapping(self, nnz, nsub, lo, hi):
        """an A row with exactly nnz entries and many more products: one B row holding all nnz columns and nsub
        B rows holding random subsets of lo..hi of them"""
        s = self.rng.choice(self.ncolsB, nnz, replace=False)
        ks = [self.b(s)] + [self.b(self.rng.choice(s, self.rng.integers(lo, hi + 1), replace=False))
                            for _ in range(nsub)]
        self.a(self.rng.permutation(ks))

    def build(self, shuffle=True):
        rows = [self.a_rows[i] for i in (self.rng.permutation(len(self.a_rows)) if shuffle else range(len(self.a_rows)))]

        def csr(rs):
            ptr = np.zeros(len(rs) + 1, np.int64)
            np.cumsum([len(r) for r in rs], out=ptr[1:])
            return ptr, (np.concatenate(rs) if rs else np.zeros(0, np.int64))

        a_ptr, a_col = csr(rows)
        b_ptr, b_col = csr(self.b_rows)
        return _Fx(a_ptr, a_col, b_ptr, b_col, self.ncolsB)


# ------------------------------------------------------------------ fixtures
BOUNDARY_VALUES = (0, 1, 32, 33, 64, 65, 128, 129, 1024, 1025, 4096, 4097)
# (symbolic class, numeric class, nnz range) of the rows whose two passes take different kernel families
CROSS_CLASSES = [(2, 1, (1, 32)), (3, 1, (65, 128)), (4, 1, (1, 32)), (4, 3, (1025, 4096))]


@functools.lru_cache(maxsize=None)
def _boundary_fx():
    """rows with products == nnz == every class boundary (each three times, over a few B rows), an A row with
    no entries, warp rows across the shared-memory sort, and rows whose two passes take different classes"""
    rng = np.random.default_rng(11)
    bld = _Builder(rng, 9001)           # 9001 % 32 != 0
    for v in BOUNDARY_VALUES:
        for _ in range(3):
            if v == 0:
                bld.a([bld.b([]), bld.b([])])          # an A row pointing only at empty B rows
            else:
                bld.disjoint(v, 1 + int(np.log2(v)))
    bld.a([])
    for v in rng.integers(CAP1 // 4 + 1, CAP1 + 1, size=40):   # nnz in (32, 128]: padded shared-memory bitonic
        bld.disjoint(int(v), 4)
    for _ in range(2):
        bld.overlapping(20, 30, 5, 20)          # products in (128, 1024], nnz <= 32
        bld.overlapping(100, 20, 60, 100)       # products in (1024, 4096], nnz in (64, 128]
        bld.overlapping(32, 200, 20, 32)        # products > 4096, nnz <= 32
        bld.overlapping(3000, 3, 800, 1200)     # products > 4096, nnz in (1024, 4096]
    return bld.build()


# the lane-group bands of lane_group_size() and, for each, the lengths of the B rows the A rows point at
LANE_B_LENGTHS = {8: (1, 12), 16: (13, 24), 32: (25, 64)}


@functools.lru_cache(maxsize=None)
def _lane_fx(gs):
    """warp-class rows (products <= 128) of 2 to 9 A entries each, over B rows whose mean length falls in the
    band of lane_group_size() that picks `gs` lanes per A entry"""
    rng = np.random.default_rng(13 + gs)
    bld = _Builder(rng, 3001)
    lo, hi = LANE_B_LENGTHS[gs]
    pool = [bld.b(rng.choice(bld.ncolsB, rng.integers(lo, hi + 1), replace=False)) for _ in range(200)]
    for _ in range(300):
        ks = list(rng.choice(pool, rng.integers(2, 10), replace=False))
        while len(ks) > 2 and sum(len(bld.b_rows[k]) for k in ks) > CAP1:
            ks.pop()
        bld.a(ks)
    return bld.build()


@functools.lru_cache(maxsize=None)
def _dense_fx():
    """more dense-class rows than dense CTAs, so every CTA resets its accumulator and bitmap between rows:
    300 rows of six B rows of 800 random columns (rows overlap), a row from column 0 to ncolsB - 1, a row in a
    narrow window at a high offset, and another row touching the last column"""
    rng = np.random.default_rng(12)
    ncolsB = 100_003                    # % 32 != 0; four 1024-word passes of the bitmap scan
    bld = _Builder(rng, ncolsB)
    pool = [bld.b(rng.choice(ncolsB, 800, replace=False)) for _ in range(600)]
    for _ in range(300):
        bld.a(rng.choice(pool, 6, replace=False))
    wide = rng.choice(np.arange(1, ncolsB - 1), 4400, replace=False)
    bld.a([bld.b(np.r_[wide[:2200], ncolsB - 1]), bld.b(np.r_[0, wide[2200:]])])
    lo = 70_001                         # 4600 consecutive columns, words 2187..2331
    bld.a([bld.b(np.arange(lo + 920 * i, lo + 920 * (i + 1))) for i in range(5)])
    bld.a(list(rng.choice(pool, 6, replace=False)) + [bld.b([ncolsB - 1, ncolsB - 2])])
    return bld.build()


@functools.lru_cache(maxsize=None)
def _colliding_ids(n=CAP3):
    """the first n int32 column ids that hash to slot 8191 of the 8192-slot table, hence also to the last
    slot of the 2048- and 256-slot tables (the top 13 bits include the top 11 and 8)"""
    out, found, lo, chunk = [], 0, 0, 1 << 22
    while found < n:
        assert lo < 1 << 26
        k = np.arange(lo, lo + chunk, dtype=np.int64)
        hit = k[hash_slot(k, TABLES[-1]) == TABLES[-1] - 1]
        out.append(hit)
        found += hit.size
        lo += chunk
    return np.concatenate(out)[:n]


@functools.lru_cache(maxsize=None)
def _collision_fx(itype):
    """one row per hash class (128, 1024 and 4096 entries) whose columns all hash to the table's LAST slot,
    so the probe chain wraps to slot 0 at once.  int32: searched ids; int64: (t << 32) | (t ^ c), which all
    fold to the 32-bit key c, with ncolsB just above the largest"""
    ids = _colliding_ids()
    if itype == "i64":
        t = np.arange(CAP3, dtype=np.int64)
        cols = (t << 32) | (t ^ int(ids[0]))
    else:
        cols = ids
    rng = np.random.default_rng(14 + len(itype))
    bld = _Builder(rng, int(cols.max()) + 2)
    for n, m in ((CAP1, 4), (CAP2, 8), (CAP3, 16)):
        bld.a([bld.b(p) for p in np.array_split(rng.permutation(cols[:n]), m)])
    bld.disjoint(40, 3)                 # and an ordinary row
    return bld.build(), cols


# c_indptr is scanned in blocks of 1024 rows; scan_sums_kernel scans the block sums in chunks of 1024 and
# carries each chunk's total into the next.  scan_add_kernel reads block sums 0 .. nblocks-2 only, so the
# carry first reaches c_indptr at 1026 blocks: 1025 * 1024 + 1 rows.
SCAN_ROWS = (1024, 1025, 1 << 20, (1 << 20) + 1, 1025 * 1024 + 1, 3 * (1 << 20) + 5)


@functools.lru_cache(maxsize=None)
def _scan_fx(nrows):
    """nrows rows of 0, 1 or 2 products (B rows of one column each): c_indptr is a long scan of small counts"""
    rng = np.random.default_rng(nrows)
    ncolsA, ncolsB = 64, 50
    a_ptr = np.zeros(nrows + 1, np.int64)
    np.cumsum(rng.integers(0, 3, size=nrows), out=a_ptr[1:])
    return _Fx(a_ptr, rng.integers(0, ncolsA, size=int(a_ptr[-1])), np.arange(ncolsA + 1),
               rng.integers(0, ncolsB, size=ncolsA), ncolsB)


def _zeros_fx():
    """a small product with room for explicit zeros and cancellation (values: _zeros_values)

    B rows (column: B entry):  0: {2: b0, 5: b1}   1: {5: b2, 6: b3}   2: {1: b4}   3: {0: b5, 6: b6}
    A rows (A entry -> B row): 0: a0 -> 0, a1 -> 1   1: a2 -> 3   2: a3 -> 2, a4 -> 0   3: a5 -> 1, a6 -> 3   4: empty
    """
    return _Fx([0, 2, 3, 5, 7, 7], [0, 1, 3, 2, 0, 1, 3], [0, 2, 4, 5, 7], [2, 5, 5, 6, 1, 0, 6], 7)


# (row, column) of the entries of C that _zeros_values makes exactly zero
ZERO_ENTRIES = [(0, 5), (1, 0), (1, 6), (2, 1), (3, 6)]


def _zeros_values(a, b, dt):
    """integer values of _zeros_fx, set so that the ZERO_ENTRIES of C are 0"""
    one = 1 + 2j if _cplx(dt) else 1
    a[0], a[1], b[1], b[2] = 2 * one, -3 * one, 3, 2    # (0, 5) = a0 b1 + a1 b2 = 6 one - 6 one
    a[2] = 0                                            # (1, 0) and (1, 6): a zero in A
    b[4] = 0                                            # (2, 1): a zero in B
    a[5], a[6], b[6] = one, -one, b[3]                  # (3, 6) = a5 b3 + a6 b6
    return a, b


def _bands():
    return {gs: lane_group_size(_lane_fx(gs).nnzB, _lane_fx(gs).ncolsA) for gs in LANE_B_LENGTHS}


# ------------------------------------------------------------------ CPU tests: the reference and the fixtures
def _small_case(seed):
    """random small integer operands with repeated columns in A rows and B rows, unsorted A columns,
    explicit zeros, an empty A row, an A row pointing at an empty B row, and a row whose two products cancel"""
    rng = np.random.default_rng(seed)
    nrows, ncolsA, ncolsB = 30, 20, 25
    deg_a = rng.integers(0, 7, size=nrows)
    deg_a[:5] = [3, 2, 4, 0, 1]
    deg_b = rng.integers(0, 6, size=ncolsA)
    deg_b[:2], deg_b[7] = 3, 0
    # the last A row points at two extra B rows of one entry each, in column 5
    a_ptr = np.r_[0, np.cumsum(deg_a), int(deg_a.sum()) + 2]
    a_col = np.r_[rng.integers(0, ncolsA, size=int(deg_a.sum())), ncolsA, ncolsA + 1]
    a_col[:3] = [5, 2, 5]               # row 0: a repeated column, unsorted
    a_col[a_ptr[4]] = 7                 # row 4 points at the empty B row 7
    b_ptr = np.r_[0, np.cumsum(deg_b), int(deg_b.sum()) + 1, int(deg_b.sum()) + 2]
    b_col = np.r_[rng.integers(0, ncolsB, size=int(deg_b.sum())), 5, 5]
    b_col[:3] = [4, 9, 4]               # B row 0: a repeated column
    a_val = rng.integers(-3, 4, size=a_col.size).astype(np.float64)   # explicit zeros among them
    b_val = rng.integers(-3, 4, size=b_col.size).astype(np.float64)
    a_val[-2:], b_val[-2:] = [2, -3], [3, 2]   # last row: 2*3 - 3*2 at column 5
    return a_ptr, a_col, b_ptr, b_col, ncolsB, a_val, b_val


def _sort_rows(ptr, col, val):
    order = np.lexsort((col, np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))))
    return col[order], val[order]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_reference_matches_oracle(seed):
    """_Gustavson against the reference's two-pass CPU Gustavson (oracle.spgemm, first-touch column order)
    after sorting each row; product counts against a plain loop; complex values against a dense product"""
    from oracle import oracle

    a_ptr, a_col, b_ptr, b_col, ncolsB, a_val, b_val = _small_case(seed)
    ref = _Gustavson(a_ptr, a_col, b_ptr, b_col, ncolsB)
    op, oi, ov = oracle.spgemm(a_ptr, a_col, a_val, b_ptr, b_col, b_val, ncolsB)
    assert np.array_equal(ref.indptr, op)
    oi, ov = _sort_rows(op, oi, ov)
    assert np.array_equal(ref.indices, oi)
    _assert_bits(ref.exact(a_val, b_val, np.float64), ov, "exact values vs oracle")
    last = ref.indptr[-2]
    assert ref.indices[last] == 5 and ref.exact(a_val, b_val, np.float64)[last] == 0 and ref.terms[last] == 2

    loop = [sum(int(b_ptr[k + 1] - b_ptr[k]) for k in a_col[a_ptr[i]:a_ptr[i + 1]]) for i in range(len(a_ptr) - 1)]
    assert ref.row_products.tolist() == loop and ref.products == sum(loop)
    assert ref.terms.sum() == ref.products

    rng = np.random.default_rng(100 + seed)
    ra, rb = rng.standard_normal(a_col.size), rng.standard_normal(b_col.size)
    c, mag = ref.rounded(ra, rb, np.float64)
    _, rv = _sort_rows(op, *oracle.spgemm(a_ptr, a_col, ra, b_ptr, b_col, rb, ncolsB)[1:])
    assert np.all(np.abs(c - rv) <= C_ROUND * ref.terms * 2.0 ** -53 * mag)

    def dense(ptr, col, val, shape):
        d = np.zeros(shape, np.complex128)
        np.add.at(d, (np.repeat(np.arange(len(ptr) - 1), np.diff(ptr)), col), val)
        return d

    ca = a_val + 1j * rng.integers(-3, 4, size=a_val.size)
    cb = b_val + 1j * rng.integers(-3, 4, size=b_val.size)
    got = dense(ref.indptr, ref.indices, ref.exact(ca, cb, np.complex128), (len(a_ptr) - 1, ncolsB))
    want = dense(a_ptr, a_col, ca, (len(a_ptr) - 1, len(b_ptr) - 1)) @ dense(b_ptr, b_col, cb, (len(b_ptr) - 1, ncolsB))
    assert np.array_equal(got, want)


def test_fixtures_reach_every_class():
    """the fixtures contain what the GPU tests below rely on"""
    ref = _boundary_fx().ref
    pairs = set(zip(ref.row_products.tolist(), ref.row_nnz.tolist()))
    for v in BOUNDARY_VALUES:
        assert (v, v) in pairs, v
    sym, num = class_of(ref.row_products), class_of(ref.row_nnz)
    for cs, cn, (lo, hi) in CROSS_CLASSES:
        assert np.any((sym == cs) & (num == cn) & (ref.row_nnz >= lo) & (ref.row_nnz <= hi)), (cs, cn)
    assert np.any(_boundary_fx().a_ptr[1:] == _boundary_fx().a_ptr[:-1])          # an A row with no entries

    assert _bands() == {8: 8, 16: 16, 32: 32}
    for gs in LANE_B_LENGTHS:
        r = _lane_fx(gs).ref
        assert np.all(class_of(r.row_products) == 1) and np.all(np.diff(_lane_fx(gs).a_ptr) >= 2)

    fx = _dense_fx()
    r = fx.ref
    dense = (class_of(r.row_products) == 4) & (class_of(r.row_nnz) == 4)
    assert dense.all() and dense.sum() > DENSE_CTAS
    assert fx.ncolsB % 32 != 0 and fx.ncolsB > 3 * DENSE_PASS_COLS
    first, last = r.indices[r.indptr[:-1]], r.indices[r.indptr[1:] - 1]             # columns sorted in a row
    assert np.any((first == 0) & (last == fx.ncolsB - 1))                           # spans every pass
    assert np.any((first > DENSE_PASS_COLS * 2) & (last - first < 5000))            # narrow window, high offset
    assert np.sum(last == fx.ncolsB - 1) >= 2

    for itype in ITYPES:
        fx, cols = _collision_fx(itype)
        for n, table in zip((CAP1, CAP2, CAP3), TABLES):
            assert np.all(hash_slot(cols[:n], table) == table - 1), (itype, table)
        assert cols.max() < fx.ncolsB and np.unique(cols).size == cols.size
        assert sorted(class_of(fx.ref.row_products).tolist()) == [1, 1, 2, 3]
        if itype == "i32":
            assert cols.max() < 2 ** 31
        else:
            assert cols.max() >= 2 ** 32 and np.unique((cols & 0xFFFFFFFF) ^ (cols >> 32)).size == 1


# ------------------------------------------------------------------ the product on the device
class _Product:
    """A @ B through b2s_spgemm_symbolic / b2s_spgemm_numeric, on rows [r0, r1) of A (a rebased indptr, the
    index and value pointers into the full arrays) and a workspace `ws_off` bytes past a 256-byte boundary,
    with guard bytes on both sides"""

    def __init__(self, fx, itype, rows=None, ws_off=0, ws_bytes=None):
        self.lib, self.fx = N.load(), fx
        self.it, self.idt = ITYPES[itype]
        self.r0, self.r1 = rows if rows is not None else (0, fx.nrows)
        self.lo, hi = int(fx.a_ptr[self.r0]), int(fx.a_ptr[self.r1])
        self.nrows, self.nnzA = self.r1 - self.r0, hi - self.lo
        self.a_ptr = _Dev(fx.a_ptr[self.r0:self.r1 + 1] - self.lo)
        self.a_col, self.b_ptr, self.b_col = _Dev(fx.a_col.astype(self.idt)), _Dev(fx.b_ptr), _Dev(fx.b_col.astype(self.idt))
        need = self.lib.b2s_spgemm_workspace_bytes(self.nrows, self.nnzA, fx.ncolsB)
        self.ws_bytes = need if ws_bytes is None else ws_bytes
        self.ws_pre = WS_HEAD + ws_off
        self.ws_buf = torch.full((self.ws_pre + self.ws_bytes + GUARD,), WS_FILL, dtype=torch.uint8, device="cuda")
        assert self.ws_buf.data_ptr() % 256 == 0
        self.ws = c_void_p(self.ws_buf.data_ptr() + self.ws_pre)

    def symbolic_rc(self, c_ptr):
        nnz, prod = c_int64(-1), c_int64(-1)
        rc = self.lib.b2s_spgemm_symbolic(self.it, self.nrows, self.fx.ncolsA, self.fx.ncolsB, self.a_ptr.ptr,
                                          self.a_col.at(self.lo), self.nnzA, self.b_ptr.ptr, self.b_col.ptr,
                                          self.fx.nnzB, c_ptr.ptr, self.ws, self.ws_bytes, byref(nnz), byref(prod), NULL)
        return rc, nnz.value, prod.value

    def symbolic(self):
        """c_indptr (filled with sentinels first), checked against the reference with nnz(C) and the product
        count before anything else runs"""
        ref = self.fx.ref
        c_ptr = _Dev(np.full(self.nrows + 1, PTR_SENTINEL, np.int64))
        rc, nnz, prod = self.symbolic_rc(c_ptr)
        assert rc == 0, N.last_error()
        e0 = ref.indptr[self.r0]
        _assert_bits(c_ptr.get(), ref.indptr[self.r0:self.r1 + 1] - e0, "c_indptr")
        assert nnz == ref.indptr[self.r1] - e0, ("nnz(C)", nnz)
        assert prod == int(ref.row_products[self.r0:self.r1].sum()), ("products", prod)
        self.check_ws_guards()
        return c_ptr, nnz

    def numeric(self, c_ptr, nnz, a_val, b_val, dt):
        """c_indices and c_data of the numeric phase; the guard tails must come back untouched"""
        av, bv = _Dev(np.asarray(a_val, dt)), _Dev(np.asarray(b_val, dt))
        c_col = _Dev(np.full(nnz + GUARD, IDX_SENTINEL, self.idt))
        c_val = _Dev(np.full(nnz + GUARD, _sentinel(dt), dt))
        rc = self.lib.b2s_spgemm_numeric(VT[dt], self.it, self.nrows, self.fx.ncolsA, self.fx.ncolsB, self.a_ptr.ptr,
                                         self.a_col.at(self.lo), av.at(self.lo), self.nnzA, self.b_ptr.ptr,
                                         self.b_col.ptr, bv.ptr, self.fx.nnzB, c_ptr.ptr, c_col.ptr, c_val.ptr,
                                         self.ws, self.ws_bytes, NULL)
        assert rc == 0, N.last_error()
        cols, vals = c_col.get(), c_val.get()
        _assert_bits(cols[nnz:], np.full(GUARD, IDX_SENTINEL, self.idt), "c_indices guard tail")
        _assert_bits(vals[nnz:], np.full(GUARD, _sentinel(dt), dt), "c_data guard tail")
        self.check_ws_guards()
        return cols[:nnz], vals[:nnz]

    def check_ws_guards(self):
        head = self.ws_buf[:self.ws_pre].cpu().numpy()
        tail = self.ws_buf[self.ws_pre + self.ws_bytes:].cpu().numpy()
        assert np.all(head == WS_FILL) and np.all(tail == WS_FILL), "stores outside the workspace"

    def exact(self, dt, seed, values=None):
        """symbolic, then numeric on integer data, all bit for bit; returns (indices, data)"""
        ref = self.fx.ref
        c_ptr, nnz = self.symbolic()
        if values is None:
            rng = np.random.default_rng(seed)
            values = _exact_values(rng, self.fx.nnzA, dt), _exact_values(rng, self.fx.nnzB, dt)
        a_val, b_val = values
        e0, e1 = ref.indptr[self.r0], ref.indptr[self.r1]
        want = ref.exact(a_val, b_val, dt)[e0:e1]
        cols, vals = self.numeric(c_ptr, nnz, a_val, b_val, dt)
        _assert_bits(cols, ref.indices[e0:e1].astype(self.idt), "c_indices")
        _assert_bits(vals, want, "c_data")
        return cols, vals


def _dseed(dt, itype, k):
    return [k, DTYPES.index(dt), list(ITYPES).index(itype)]


# ------------------------------------------------------------------ exact tests
@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_class_boundaries_exact(dtype, itype):
    """products == nnz at 0, 1, 32/33, 64/65, 128/129, 1024/1025, 4096/4097, and rows that take one class in
    the symbolic pass and another in the numeric pass"""
    _Product(_boundary_fx(), itype).exact(dtype, _dseed(dtype, itype, 1))


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
@pytest.mark.parametrize("gs", list(LANE_B_LENGTHS))
def test_lane_groups_exact(gs, dtype, itype):
    """warp-class rows of several A entries with 8, 16 and 32 lanes per A entry"""
    fx = _lane_fx(gs)
    assert lane_group_size(fx.nnzB, fx.ncolsA) == gs
    _Product(fx, itype).exact(dtype, _dseed(dtype, itype, 2 + gs))


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_dense_accumulator_exact(dtype, itype):
    """more dense rows than dense CTAs: each CTA must clear its accumulator and bitmap between rows"""
    _Product(_dense_fx(), itype).exact(dtype, _dseed(dtype, itype, 3))


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_hash_collisions_exact(dtype, itype):
    """every column of a row hashes to the table's last slot: probe chains of 128, 1024 and 4096 keys wrap
    to slot 0; for int64 the keys differ only in their high words"""
    fx, _ = _collision_fx(itype)
    _Product(fx, itype).exact(dtype, _dseed(dtype, itype, 4))


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("nrows", SCAN_ROWS)
def test_scan_carry(nrows, itype):
    """c_indptr of 1 scan block, 2, 1024 (one chunk of block sums), 1025 (two chunks, the carry unread),
    1026 (the first carry that reaches c_indptr) and 3073 blocks.  Numeric once, at the largest size."""
    fx = _scan_fx(nrows)
    P = _Product(fx, itype)
    if nrows == SCAN_ROWS[-1]:
        P.exact(np.float64 if itype == "i32" else np.complex64, [5, nrows])
    else:
        P.symbolic()


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
def test_empty_row_block_writes_indptr(itype):
    """nrowsA == 0: c_indptr[0] = nnz(C) = 0 over whatever the buffer held; the numeric phase does nothing"""
    lib = N.load()
    it, idt = ITYPES[itype]
    ws = torch.zeros(lib.b2s_spgemm_workspace_bytes(0, 0, 7), dtype=torch.uint8, device="cuda")
    b_ptr, b_col = _Dev(np.array([0, 2, 3], np.int64)), _Dev(np.array([1, 6, 3], idt))
    c_ptr = _Dev(np.full(1, PTR_SENTINEL, np.int64))
    nnz, prod = c_int64(-1), c_int64(-1)
    assert lib.b2s_spgemm_symbolic(it, 0, 2, 7, _Dev(np.zeros(1, np.int64)).ptr, NULL, 0, b_ptr.ptr, b_col.ptr, 3,
                                   c_ptr.ptr, c_void_p(ws.data_ptr()), ws.numel(), byref(nnz), byref(prod), NULL) == 0
    _assert_bits(c_ptr.get(), np.zeros(1, np.int64), "c_indptr of an empty row block")
    assert nnz.value == 0 and prod.value == 0
    assert lib.b2s_spgemm_numeric(N.B2S_F64, it, 0, 2, 7, _Dev(np.zeros(1, np.int64)).ptr, NULL, NULL, 0, b_ptr.ptr,
                                  b_col.ptr, _Dev(np.ones(3)).ptr, 3, c_ptr.ptr, NULL, NULL, c_void_p(ws.data_ptr()),
                                  ws.numel(), NULL) == 0
    _assert_bits(c_ptr.get(), np.zeros(1, np.int64), "c_indptr after the numeric phase")


EMPTY_OPERANDS = {
    # ncolsA = 0: A has rows but no entries, B has no rows
    "ncolsA=0": lambda: _Fx(np.zeros(6, np.int64), [], [0], [], 7),
    # ncolsB = 0: A has entries, B's rows are all empty
    "ncolsB=0": lambda: _Fx([0, 2, 2, 5], [0, 2, 1, 1, 0], [0, 0, 0, 0], [], 0),
    # nnzB = 0 with ncolsB > 0
    "nnzB=0": lambda: _Fx([0, 2, 2, 5], [0, 2, 1, 1, 0], [0, 0, 0, 0], [], 9),
}


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("case", list(EMPTY_OPERANDS))
def test_empty_operands(case, itype):
    fx = EMPTY_OPERANDS[case]()
    assert fx.ref.nnz == 0 and fx.ref.products == 0
    _Product(fx, itype).exact(np.complex128, [6])


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_explicit_and_cancelled_zeros(dtype, itype):
    """zeros in A or B and products that cancel to exactly 0 keep their entries in C, with value +0"""
    fx = _zeros_fx()
    rng = np.random.default_rng(_dseed(dtype, itype, 7))
    a, b = _zeros_values(_exact_values(rng, fx.nnzA, dtype), _exact_values(rng, fx.nnzB, dtype), dtype)
    ref = fx.ref
    c = ref.exact(a, b, dtype)
    rows = np.repeat(np.arange(fx.nrows), ref.row_nnz)
    for r, j in ZERO_ENTRIES:
        k = np.flatnonzero((rows == r) & (ref.indices == j))
        assert k.size == 1 and c[k[0]] == 0, (r, j)
    _, vals = _Product(fx, itype).exact(dtype, None, values=(a, b))
    assert np.sum(vals == 0) == len(ZERO_ENTRIES)


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_row_block_exact(dtype, itype):
    """rows [r0, r1) of A (rebased indptr, index and value pointers into the full arrays) give rows [r0, r1)
    of C"""
    fx = _boundary_fx()
    r0, r1 = fx.nrows // 3, fx.nrows - 5
    _Product(fx, itype, rows=(r0, r1)).exact(dtype, _dseed(dtype, itype, 8))


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
def test_misaligned_workspace(itype):
    """one workspace of exactly b2s_spgemm_workspace_bytes at 8 bytes past a 256-byte boundary, shared by
    both phases (guard bytes on both sides); one byte less is refused by both phases"""
    fx = _boundary_fx()
    P = _Product(fx, itype, ws_off=8)
    P.exact(np.complex128, [9])
    small = _Product(fx, itype, ws_bytes=P.ws_bytes - 1)
    rc, _, _ = small.symbolic_rc(_Dev(np.zeros(fx.nrows + 1, np.int64)))
    assert rc == B2S_ERR_WORKSPACE and "workspace too small" in N.last_error()
    c_ptr, nnz = P.symbolic()
    assert small.lib.b2s_spgemm_numeric(N.B2S_F64, small.it, fx.nrows, fx.ncolsA, fx.ncolsB, small.a_ptr.ptr,
                                        small.a_col.ptr, _Dev(np.ones(fx.nnzA)).ptr, fx.nnzA, small.b_ptr.ptr,
                                        small.b_col.ptr, _Dev(np.ones(fx.nnzB)).ptr, fx.nnzB, c_ptr.ptr,
                                        _Dev(np.zeros(nnz, small.idt)).ptr, _Dev(np.zeros(nnz)).ptr, small.ws,
                                        small.ws_bytes, NULL) == B2S_ERR_WORKSPACE


# ------------------------------------------------------------------ rounding and repeatability
ROUNDING_FIXTURES = {"boundary": _boundary_fx, "dense": _dense_fx}


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
@pytest.mark.parametrize("fixture", list(ROUNDING_FIXTURES))
def test_rounding_and_repeatability(fixture, dtype, itype):
    """random data: every entry within the rounding bound of a wider-type reference, and a second run gives
    the same c_indptr and c_indices bits (c_data may differ in the last bits: atomics)"""
    fx = ROUNDING_FIXTURES[fixture]()
    ref = fx.ref
    rng = np.random.default_rng(_dseed(dtype, itype, 10 + len(fixture)))
    a_val, b_val = _rand(rng, fx.nnzA, dtype), _rand(rng, fx.nnzB, dtype)
    c_ref, mag = ref.rounded(a_val, b_val, dtype)
    bound = C_ROUND * ref.terms * 2.0 ** -MANT[dtype] * mag
    P = _Product(fx, itype)
    runs = []
    for _ in range(2):
        c_ptr, nnz = P.symbolic()
        cols, vals = P.numeric(c_ptr, nnz, a_val, b_val, dtype)
        _assert_bits(cols, ref.indices.astype(P.idt), "c_indices")
        err = np.abs(vals.astype(EXT[dtype]) - c_ref)
        bad = np.flatnonzero(~(err <= bound))
        assert bad.size == 0, f"entry {bad[0]} ({ref.terms[bad[0]]} terms) off by {err[bad[0]]}, bound {bound[bad[0]]}"
        runs.append((c_ptr.get(), cols))
    _assert_bits(runs[1][0], runs[0][0], "c_indptr, second run")
    _assert_bits(runs[1][1], runs[0][1], "c_indices, second run")


# ------------------------------------------------------------------ routing
def _instantiations(names, kernel):
    """template arguments of every launched instantiation of `kernel`: casts and the namespace dropped,
    booleans spelled true / false"""
    out = set()
    for n in names:
        if kernel + "<" not in n:
            continue
        args = n.split(kernel + "<", 1)[1].split(">", 1)[0]
        args = [re.sub(r"\((?:int|bool)\)|b2s::", "", a).strip() for a in args.split(",")]
        args[-1] = {"0": "false", "1": "true"}.get(args[-1], args[-1])
        out.add(tuple(args))
    return out


CPP_V = {np.float32: "float", np.float64: "double", np.complex64: "c64", np.complex128: "c128"}
CPP_I = {"i32": "int", "i64": "long"}
# (TABLE, THREADS, WARP_PER_ROW) of the three hash classes
HASH_CONFIGS = [("256", "256", "true"), ("2048", "128", "false"), ("8192", "512", "false")]


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages()})


@gpu
@pytest.mark.parametrize("itype", list(ITYPES))
def test_boundary_fixture_launches_every_kernel(itype):
    """the class-boundary fixture runs every hash and dense instantiation of both phases, for every value type"""
    fx = _boundary_fx()
    names = _kernel_names(lambda: [_Product(fx, itype).exact(dt, [11]) for dt in DTYPES])
    I = CPP_I[itype]
    assert _instantiations(names, "sym_hash_kernel") == {(I, *c) for c in HASH_CONFIGS}, names
    assert _instantiations(names, "num_hash_kernel") == {(CPP_V[dt], I, *c) for dt in DTYPES for c in HASH_CONFIGS}, names
    assert _instantiations(names, "dense_row_kernel") == {("double", I, "false")} | \
        {(CPP_V[dt], I, "true") for dt in DTYPES}, names


@gpu
def test_scan_launches_the_block_sum_kernel():
    """scan_sums_kernel runs once c_indptr spans more than one scan block, and not for 1024 rows"""
    names = _kernel_names(lambda: _Product(_scan_fx(1024), "i32").symbolic())
    assert any("scan_block_kernel" in n for n in names) and not any("scan_sums_kernel" in n for n in names), names
    names = _kernel_names(lambda: _Product(_scan_fx((1 << 20) + 1), "i32").symbolic())
    assert any("scan_sums_kernel" in n for n in names), names


# ------------------------------------------------------------------ error path
@gpu
def test_too_wide_dense_accumulator_is_refused():
    """a dense-class row with ncolsB = 2^44 would need a 2 TB bitmap: B2S_ERR_WORKSPACE with a message, and
    the library keeps working"""
    rng = np.random.default_rng(15)
    ncolsB = 1 << 44
    cols = rng.choice(ncolsB, 2 * (CAP3 // 2 + 50), replace=False)
    fx = _Fx([0, 2], [0, 1], [0, cols.size // 2, cols.size], cols, ncolsB)
    P = _Product(fx, "i64")
    rc, _, _ = P.symbolic_rc(_Dev(np.zeros(2, np.int64)))
    assert rc == B2S_ERR_WORKSPACE and "dense accumulators" in N.last_error(), (rc, N.last_error())
    _Product(_zeros_fx(), "i64").exact(np.float64, [15])


# ------------------------------------------------------------------ public API
@gpu
def test_public_api_empty_row_block():
    import scipy.sparse as sp

    import legate_sparse as sparse

    B = sparse.csr_array(sp.random(7, 5, density=0.5, format="csr", random_state=1))
    E = sparse.csr_array((0, 7)) @ B
    assert E.shape == (0, 5) and E.nnz == 0
    assert np.array_equal(np.asarray(E.indptr), [0])


def _public(fx, a_val, b_val):
    import legate_sparse as sparse

    A = sparse.csr_array((a_val, fx.a_col, fx.a_ptr), shape=(fx.nrows, fx.ncolsA))
    B = sparse.csr_array((b_val, fx.b_col, fx.b_ptr), shape=(fx.ncolsA, fx.ncolsB))
    return A @ B


@gpu
def test_public_api_products_and_structure():
    """C._last_products is the exact product count; A @ B keeps the reference's structure and values"""
    fx = _boundary_fx()
    rng = np.random.default_rng(16)
    a_val, b_val = _exact_values(rng, fx.nnzA, np.float64), _exact_values(rng, fx.nnzB, np.float64)
    C = _public(fx, a_val, b_val)
    assert C._last_products == fx.ref.products
    assert np.array_equal(C.indptr, fx.ref.indptr) and np.array_equal(C.indices, fx.ref.indices)
    _assert_bits(np.asarray(C.data), fx.ref.exact(a_val, b_val, np.float64), "data")


@gpu
def test_public_api_keeps_cancelled_zero():
    """zeros in the operands and a cancellation keep their entries through A @ B"""
    fx = _zeros_fx()
    a, b = _zeros_values(np.arange(1.0, 8.0), np.arange(1.0, 8.0), np.float64)
    C = _public(fx, a, b)
    assert np.array_equal(C.indptr, fx.ref.indptr) and np.array_equal(C.indices, fx.ref.indices)
    _assert_bits(np.asarray(C.data), fx.ref.exact(a, b, np.float64), "data")
    assert np.sum(np.asarray(C.data) == 0) == len(ZERO_ENTRIES)
