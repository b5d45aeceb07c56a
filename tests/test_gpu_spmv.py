"""GPU parity: CSR SpMV through the public API / C ABI vs the oracle and scipy.
Mirrors reference tests/integration/test_spmv.py:25-38 (+ larger and ragged cases).
Tolerance: fp64 1e-10 relative (BASELINE.json north_star); f32 1e-5 (the reference's isclose)."""
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp

import legate_sparse as sparse
from oracle import oracle
from tests import gen

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def relerr(a, b):
    a, b = np.asarray(a), np.asarray(b)
    d = np.linalg.norm((a - b).ravel())
    n = np.linalg.norm(b.ravel())
    return d / n if n > 0 else d


@pytest.mark.parametrize("N", [5, 29])
@pytest.mark.parametrize("M", [7, 17])
@pytest.mark.parametrize("inline", [True, False])
def test_csr_spmv_reference_shapes(N, M, inline):
    a, x = gen.simple_system(N, M, seed=0)
    A = sparse.csr_array(a)
    if inline:
        y = np.ndarray((N,))
        A.dot(x, out=y)
    else:
        y = A @ x
    assert np.all(np.isclose(y, a @ x))
    yo = oracle.spmv(A.indptr, A.indices, A.data, x)
    assert relerr(y, yo) < 1e-13


def test_spmv_golden_fixture():
    z = np.load(os.path.join(G, "spmv_spgemm_scipy.npz"))
    A = sparse.csr_array((z["A_data"], z["A_indices"], z["A_indptr"]), shape=tuple(z["A_shape"]))
    y = A @ z["x"]
    assert relerr(y, z["y"]) < 1e-13
    with open(os.path.join(G, "reference_known_answers.json")) as f:
        k = json.load(f)["readme_tridiagonal"]
    T = sparse.diags([1] * 3, [-1, 0, 1], shape=(5, 5), format="csr", dtype=np.float64)
    assert np.array_equal(T @ np.ones(5), np.array(k["A_ones"], dtype=float))


@pytest.mark.parametrize("variant", ["rowvec", "tile", "pipe"])
@pytest.mark.parametrize("index64", ["0", "1"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.complex64, np.complex128])
def test_spmv_variants_types(monkeypatch, variant, index64, dtype):
    monkeypatch.setenv("B2S_SPMV_VARIANT", variant)
    monkeypatch.setenv("B2S_INDEX64", index64)
    rng = np.random.default_rng(5)
    S = sp.random(533, 407, density=0.05, format="csr", random_state=3, dtype=np.float64)
    S = S.astype(dtype)
    if np.dtype(dtype).kind == "c":
        S.data = S.data + 1j * rng.standard_normal(S.nnz).astype(S.data.real.dtype)
    x = rng.standard_normal(407).astype(dtype)
    if np.dtype(dtype).kind == "c":
        x = x + 1j * rng.standard_normal(407).astype(x.real.dtype)
    A = sparse.csr_array(S)
    y = A @ x
    assert y.dtype == np.dtype(dtype)
    tol = 1e-10 if np.dtype(dtype) in (np.float64, np.complex128) else 2e-5
    assert relerr(y, S @ x) < tol


@pytest.mark.parametrize("longrows,tile", [("0", "1024"), ("1", "1024"), ("0", "2048")])
@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.complex128])
def test_spmv_pipe_products_irregular_rows(monkeypatch, dtype, longrows, tile):
    """products consumer of the TMA pipe kernel (two ping-pong groups), both tile sizes, with and
    without the long-row pass: irregular rows, empty rows, rows longer than a tile"""
    monkeypatch.setenv("B2S_SPMV_VARIANT", "pipe")
    monkeypatch.setenv("B2S_SPMV_LONGROWS", longrows)
    monkeypatch.setenv("B2S_SPMV_TILE_NNZ", tile)
    monkeypatch.setenv("B2S_SPMV_NO_WINDOW", "1")
    rng = np.random.default_rng(12)
    n, m = 4000, 3500
    deg = rng.integers(0, 12, size=n)
    deg[:30] = 0
    deg[2000:2100] = 0
    deg[-7:] = 0
    deg[1234] = 3000
    deg[77] = 128
    deg[78] = 1024
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    cols = np.concatenate([np.sort(rng.choice(m, size=k, replace=False)) for k in deg]).astype(np.int64)
    data = rng.standard_normal(int(indptr[-1])).astype(dtype)
    x = rng.standard_normal(m).astype(dtype)
    if np.dtype(dtype).kind == "c":
        data = data + 1j * rng.standard_normal(data.shape[0])
        x = x + 1j * rng.standard_normal(m)
    S = sp.csr_array((data, cols, indptr), shape=(n, m))
    A = sparse.csr_array(S)
    y = A @ x
    tol = 1e-10 if np.dtype(dtype) != np.float32 else 3e-5
    assert relerr(y, S @ x) < tol
    assert A._block().plan.info()["tile_nnz"] == int(tile)


def _check(A_sp, seed=1, tol=1e-10):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal(A_sp.shape[1])
    A = sparse.csr_array(A_sp)
    y = A @ x
    assert relerr(y, A_sp @ x) < tol
    return A, x, y


def test_spmv_poisson_config1_full():
    # BASELINE config 1: 5-point Poisson, 1000x1000 grid, vs scipy AND the oracle's C loop
    N = 1000
    d, o = gen.poisson2d_diagonals(N)
    A = sparse.diags(d, o, dtype=np.float64).tocsr()
    S = gen.poisson2d_scipy(N)
    assert np.array_equal(A.indptr, S.indptr) and np.array_equal(A.indices, S.indices)
    for x in (np.ones(N * N), np.random.default_rng(0).random(N * N)):
        y = A @ x
        assert relerr(y, S @ x) < 1e-10
        assert relerr(y, oracle.spmv(S.indptr, S.indices, S.data, x)) < 1e-10
    info = A._block().plan.info()
    assert info["ntiles"] == -(-A.nnz // info["tile_nnz"])


def test_spmv_ragged_and_empty_rows():
    rng = np.random.default_rng(9)
    # empty rows at the start, in the middle (at tile boundaries) and at the end; one huge row
    n, m = 3000, 2500
    deg = rng.integers(0, 8, size=n)
    deg[:40] = 0
    deg[1000:1200] = 0
    deg[-25:] = 0
    deg[1500] = 2400  # spans several 1024/2048-nnz tiles
    deg[77] = 2048
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(deg, out=indptr[1:])
    cols = np.concatenate([np.sort(rng.choice(m, size=k, replace=False)) for k in deg]).astype(np.int64)
    data = rng.standard_normal(int(indptr[-1]))
    S = sp.csr_array((data, cols, indptr), shape=(n, m))
    _check(S)
    # unsorted columns + duplicates (COO ctor keeps both)
    r = rng.integers(0, 50, size=4000)
    c = rng.integers(0, 60, size=4000)
    v = rng.standard_normal(4000)
    A = sparse.csr_array((v, (r, c)), shape=(50, 60))
    x = rng.standard_normal(60)
    D = np.zeros((50, 60))
    np.add.at(D, (r, c), v)
    assert relerr(A @ x, D @ x) < 1e-10
    # all-empty matrix and zero-row / zero-col shapes
    E = sparse.csr_array((7, 9))
    assert np.array_equal(E @ np.ones(9), np.zeros(7))
    assert (sparse.csr_array((0, 5)) @ np.ones(5)).shape == (0,)


@pytest.mark.parametrize("tile", ["1024", "2048", "4096"])
def test_spmv_tile_sizes_banded_and_random(monkeypatch, tile):
    # 1024 / 2048: pipe kernel; 4096: tile kernel (IPT 16).  The plan's window statistic is the same for
    # every tile size: a tile of the banded matrix spans ~4096/51 rows, far inside the 1024-element window
    monkeypatch.setenv("B2S_SPMV_TILE_NNZ", tile)
    d, c, p = gen.banded_csr_arrays(20011, 51)
    S = sp.csr_array((d, c, p), shape=(20011, 20011))
    A, x, y = _check(S)
    info = A._block().plan.info()
    assert info["tile_nnz"] == int(tile)
    assert info["window_tiles"] == info["ntiles"]  # banded → every tile stages its x window
    d, c, p = gen.random_csr_fixed(30000, 40000, 50, seed=11)
    S = sp.csr_array((d, c, p), shape=(30000, 40000))
    A, x, y = _check(S)
    info = A._block().plan.info()
    assert info["tile_nnz"] == int(tile)
    assert info["window_tiles"] == 0


def test_spmv_2d_x_and_out_rules():
    a, x = gen.simple_system(29, 17, seed=4)
    A = sparse.csr_array(a)
    y2 = A @ x.reshape(-1, 1)
    assert y2.shape == (29, 1) and np.allclose(y2[:, 0], a @ x)
    out = np.zeros((29, 1))
    r = A.dot(x.reshape(-1, 1), out=out)
    assert r is out and np.allclose(out[:, 0], a @ x)
    with pytest.raises(ValueError):
        A.dot(x, out=np.zeros(29, dtype=np.float32))  # out dtype must equal the promoted dtype
    with pytest.raises(AssertionError):
        A.dot(x, out=np.zeros(28))
    # dtype promotion: f32 matrix x f64 vector → f64
    A32 = sparse.csr_array(a.astype(np.float32))
    assert (A32 @ x).dtype == np.float64
    # strided x → RuntimeWarning + implicit copy (reference csr.py:444-452)
    xs = np.zeros(34)
    xs[::2] = x
    with pytest.warns(RuntimeWarning):
        ys = A @ xs[::2]
    assert np.allclose(ys, a @ x)
    assert np.allclose(A.sum(axis=1).ravel(), a.sum(axis=1))


def test_spmv_device_tensor_io():
    import torch

    d, c, p = gen.random_csr_fixed(5000, 5000, 20, seed=2)
    S = sp.csr_array((d, c, p), shape=(5000, 5000))
    A = sparse.csr_array((torch.from_numpy(d).cuda(), torch.from_numpy(c).cuda(), torch.from_numpy(p).cuda()),
                         shape=(5000, 5000))
    x = np.random.default_rng(3).standard_normal(5000)
    xd = torch.from_numpy(x).cuda()
    yd = A @ xd
    assert isinstance(yd, torch.Tensor) and yd.is_cuda
    assert relerr(yd.cpu().numpy(), S @ x) < 1e-10
    out = torch.empty(5000, dtype=torch.float64, device="cuda")
    assert A.dot(xd, out=out) is out and relerr(out.cpu().numpy(), S @ x) < 1e-10
    # linearity property (size-independent check used at full size in bench)
    y2 = A @ (2.0 * xd)
    assert relerr(y2.cpu().numpy(), 2 * (S @ x)) < 1e-12


def test_spmv_powerlaw_small():
    d, c, p = gen.powerlaw_csr(20000, 20000, max_row=10000, seed=7)
    S = sp.csr_array((d, c, p), shape=(20000, 20000))
    _check(S)


def test_diagonal_and_transpose_device():
    a, _ = gen.simple_system(13, 13, seed=8, tol=0.2)
    for add_eye in (False, True):
        m = a + (np.eye(13) if add_eye else 0)
        A = sparse.csr_array(m)
        assert np.all(np.isclose(np.diagonal(m), A.diagonal()))
        assert np.allclose(A.diagonal(), oracle.diagonal(A.indptr, A.indices, A.data))
    with pytest.raises(NotImplementedError):
        A.diagonal(k=1)
    import torch

    S = sp.random(60, 45, density=0.2, format="csr", random_state=2)
    Ad = sparse.csr_array((torch.from_numpy(S.data).cuda(), torch.from_numpy(S.indices.astype(np.int64)).cuda(),
                           torch.from_numpy(S.indptr.astype(np.int64)).cuda()), shape=S.shape)
    assert np.array_equal(Ad.T.todense(), np.asarray(S.todense()).T)
def test_longrows_pass_on_skewed_rows(monkeypatch):
    """power-law row lengths: rows much longer than the tile average are summed by a full warp in a
    second pass of the products consumer (selected from the plan's max row; forced here as well)."""
    import scipy.sparse as sp
    import legate_sparse as sparse
    from tests import gen

    d, c, p = gen.powerlaw_csr(60000, 60000, max_row=5000, seed=11)
    S = sp.csr_array((d, c, p), shape=(60000, 60000))
    x = np.random.default_rng(4).standard_normal(60000)
    want = S @ x
    for force in (None, "1", "0"):
        if force is None:
            monkeypatch.delenv("B2S_SPMV_LONGROWS", raising=False)
        else:
            monkeypatch.setenv("B2S_SPMV_LONGROWS", force)
        A = sparse.csr_array(S)
        y = A @ x
        assert np.allclose(y, want, rtol=1e-11, atol=1e-11), force
