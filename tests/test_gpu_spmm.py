"""Multi-vector product A * X / transpose(A) * X (dsa_matrix_spmm_dense[_d], DynamicSparseMatrix.mul_dense with a 2-D x) on
the device: every column bit-identical to the single-vector product of that column, within 1e-12 of the oracle, strided
buffers, the torch path and its stream ordering, argument checks."""
import ctypes as C

import numpy as np
import pytest

import dsa_b200 as D
from dsa_b200 import _lib, api
from oracle import oracle as O

pytestmark = pytest.mark.gpu

SPMV_RTOL = 1e-12
KS = [1, 2, 3, 4, 5, 8, 13, 16, 33]     # remainder groups of 4, and more than one pass of 32 columns


def _rel_close(a, b, rtol=SPMV_RTOL):
    return np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b)))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _rand_coo(rng, m, n, nnz, integer_vals=False):
    I, J = rng.integers(1, m + 1, nnz), rng.integers(1, n + 1, nnz)
    V = rng.integers(1, 100, nnz).astype(float) if integer_vals else rng.random(nnz) + 0.5
    return I, J, V


def _state(name, integer_vals=False):
    """(device matrix, oracle matrix) in one of the states the product has to handle"""
    rng = np.random.default_rng(["bulk", "batches", "deleted", "tile"].index(name) + (10 if integer_vals else 0))
    m, n = 3000, 2000
    I, J, V = _rand_coo(rng, m, n, 120_000, integer_vals)
    gm, om = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    if name in ("batches", "tile"):
        prev = _lib.set_tile_mode(2) if name == "tile" else None
        try:
            for _ in range(2):   # inserts (some in new rows / columns), overwrites and deletes (value 0.0)
                nb = 20_000
                bi, bj = rng.integers(1, m + 40, nb), rng.integers(1, n + 40, nb)
                if name == "tile":   # the tile-streamed pipeline takes batches that create no row or column
                    bi, bj = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
                bv = np.where(rng.random(nb) < 0.4, 0.0, rng.integers(1, 50, nb).astype(float) if integer_vals else rng.random(nb) + 0.5)
                gm.set_batch(bi, bj, bv)
                om.set_batch_policy(bi, bj, bv)
        finally:
            if prev is not None:
                _lib.set_tile_mode(prev)
    if name == "deleted":   # tombstoned slots in both orientations, and live rows whose entries are all gone
        cols = np.unique(rng.integers(1, n + 1, 300))
        rows = np.unique(rng.integers(1, m + 1, 200))
        D.deletecolumn(gm, cols)
        om.delete_columns_policy(cols)
        D.deleterow(gm, rows)
        om.delete_rows_policy(rows)
        r = int(np.setdiff1d(np.arange(1, m + 1), rows)[0])   # empty one live row through deletes of all its entries
        js = np.unique(J[I == r])
        gm.set_batch(np.full(len(js), r), js, np.zeros(len(js)))
        om.set_batch_policy(np.full(len(js), r), js, np.zeros(len(js)))
    return gm, om


@pytest.mark.parametrize("state", ["bulk", "batches", "deleted", "tile"])
def test_columns_bit_identical_to_single_products(state):
    gm, om = _state(state)
    rng = np.random.default_rng(3)
    m, n = gm.size
    for trans in (False, True):
        nx, ny = (m, n) if trans else (n, m)
        for k in KS:
            X = rng.random((nx, k))
            Y = gm.mul_dense(X, trans=trans)
            assert Y.shape == (ny, k)
            for c in range(k):
                assert np.array_equal(Y[:, c], gm.mul_dense(X[:, c], trans=trans)), (state, trans, k, c)
            for c in (0, k - 1):
                assert _rel_close(Y[:, c], om.mul_dense(X[:, c], ny, trans=trans)), (state, trans, k, c)


@pytest.mark.parametrize("state", ["bulk", "deleted"])
def test_integer_values_match_the_oracle_exactly(state):
    gm, om = _state(state, integer_vals=True)
    rng = np.random.default_rng(4)
    m, n = gm.size
    for trans in (False, True):
        nx, ny = (m, n) if trans else (n, m)
        X = rng.integers(-3, 4, (nx, 13)).astype(float)
        Y = gm.mul_dense(X, trans=trans)
        for c in range(13):
            assert np.array_equal(Y[:, c], om.mul_dense(X[:, c], ny, trans=trans))


def test_empty_matrix_gives_zeros():
    gm = D.dynamicsparse(fill_mode=False)
    assert gm.mul_dense(np.ones((4, 3))).shape == (0, 3)
    L = D.lib()
    for trans in (0, 1):
        Y = np.full((7, 5), np.nan)
        _lib.check(L.dsa_matrix_spmm_dense(gm._h, C.c_int(trans), _p(np.ones((4, 5))), C.c_int64(4), C.c_int64(5), C.c_int64(5),
                                           _p(Y), C.c_int64(7), C.c_int64(5)))
        assert np.array_equal(Y, np.zeros((7, 5)))


def _spmm_host(gm, X, nx, k, ldx, Y, ny, ldy, trans=0):
    _lib.check(D.lib().dsa_matrix_spmm_dense(gm._h, C.c_int(trans), _p(X), C.c_int64(nx), C.c_int64(k), C.c_int64(ldx), _p(Y),
                                             C.c_int64(ny), C.c_int64(ldy)))


def _spmv_host(gm, x, ny, trans=0):
    x = np.ascontiguousarray(x)
    y = np.zeros(max(ny, 1))
    _lib.check(D.lib().dsa_matrix_spmv_dense(gm._h, C.c_int(trans), _p(x), C.c_int64(len(x)), _p(y), C.c_int64(ny)))
    return y[:ny]


def test_shape_edges_nx_and_ny():
    gm, _ = _state("bulk")
    m, n = gm.size
    rng = np.random.default_rng(5)
    for trans, (mx, my) in ((0, (n, m)), (1, (m, n))):
        for nx in (mx // 2, mx, mx + 37):            # keys above nx contribute nothing; x rows above the largest key are unused
            for ny in (my // 3, my):                 # partitions whose key is above ny are not written
                k = 6
                X = rng.random((nx, k))
                Y = np.full((ny, k), np.nan)
                _spmm_host(gm, X, nx, k, k, Y, ny, k, trans)
                for c in range(k):
                    assert np.array_equal(Y[:, c], _spmv_host(gm, X[:, c], ny, trans)), (trans, nx, ny, c)


def test_strided_host_buffers_keep_the_padding():
    gm, _ = _state("batches")
    m, n = gm.size
    rng = np.random.default_rng(6)
    for k, ldx, ldy in ((3, 5, 7), (8, 11, 9), (1, 4, 3), (33, 40, 35)):
        Xw = rng.random((n, ldx))
        Y = np.full((m, ldy), np.nan)
        _spmm_host(gm, Xw, n, k, ldx, Y, m, ldy)
        assert np.all(np.isnan(Y[:, k:]))
        for c in range(k):
            assert np.array_equal(Y[:, c], gm.mul_dense(Xw[:, c])), (k, ldx, ldy, c)


class _Recorder:
    """lib() proxy that records the arguments of the device entry points"""

    def __init__(self, L):
        self._L, self.calls = L, []

    def __getattr__(self, name):
        fn = getattr(self._L, name)
        if name.startswith("dsa_matrix_sp"):
            def rec(*args):
                self.calls.append((name, args))
                return fn(*args)
            return rec
        return fn


def test_torch_device_path(monkeypatch):
    torch = pytest.importorskip("torch")
    gm, _ = _state("batches")
    m, n = gm.size
    rng = np.random.default_rng(7)
    W = torch.from_numpy(rng.random((n, 24))).cuda()
    rec = _Recorder(D.lib())
    monkeypatch.setattr(api, "lib", lambda: rec)
    for k in (1, 5, 8, 16):
        view = W[:, :k]
        Y = gm.mul_dense(view)
        assert isinstance(Y, torch.Tensor) and Y.is_cuda and Y.dtype == torch.float64 and tuple(Y.shape) == (m, k)
        name, args = rec.calls[-1]
        assert name == "dsa_matrix_spmm_dense_d"
        assert args[2].value == view.data_ptr() and args[5].value == 24        # the strided view goes in without a copy
        Yh = gm.mul_dense(view.cpu().numpy())
        assert np.array_equal(Y.cpu().numpy(), Yh)                              # host and device paths: same bits
        Yt = gm.mul_dense(torch.from_numpy(rng.random((m, k))).cuda().t().contiguous().t(), trans=True)   # column-major: copied
        assert tuple(Yt.shape) == (n, k)
    x = W[:, 3]                                                                 # 1-D (strided) -> the single-vector entry point
    y = gm.mul_dense(x)
    assert rec.calls[-1][0] == "dsa_matrix_spmv_dense_d" and tuple(y.shape) == (m,)
    assert np.array_equal(y.cpu().numpy(), gm.mul_dense(x.cpu().numpy()))
    with pytest.raises(D.ArgumentError):
        gm.mul_dense(W.reshape(n, 4, 6))


def test_torch_path_is_ordered_against_the_current_stream():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(8)
    m, n = 20_000, 20_000
    I, J, V = _rand_coo(rng, m, n, 2_000_000)
    gm = D.dynamicsparse(I, J, V, m=m, n=n)
    Xh = rng.random((n, 8))
    want = gm.mul_dense(Xh)
    src = torch.from_numpy(Xh).cuda()
    for _ in range(3):
        X = torch.zeros_like(src)
        torch.cuda._sleep(50_000_000)      # a long op queued on the current stream ahead of the input's last write
        X.copy_(src)
        Y = gm.mul_dense(X)
        Z = Y * 1.0                        # read on the current stream right after the call, no synchronise
        assert np.array_equal(Z.cpu().numpy(), want)


def test_full_size_config2_vs_oracle():
    """config 2 at full size (bench.make_workload's COO, 1e5 x 1e5, 1e7 nnz, then two bench batches): k = 8 columns, both
    orientations, against the reference's sequential semantics within 1e-12, and against the single products bit for bit."""
    import bench as B
    _, coo, batches, _ = B.make_workload(3)
    m, n = B.M_ROWS, B.N_COLS
    gm = D.dynamicsparse(coo[0], coo[1], coo[2], m=m, n=n)
    seq = O.Matrix(coo[0], coo[1], coo[2], m=m, n=n)
    for bi, bj, bv in batches[:2]:
        gm.set_batch(bi, bj, bv)
        seq.set_many(bi, bj, bv)
    rng = np.random.default_rng(9)
    for trans in (False, True):
        X = rng.random((n, 8))
        Y = gm.mul_dense(X, trans=trans)
        for c in range(8):
            assert _rel_close(Y[:, c], seq.mul_dense(X[:, c], m, trans=trans)), (trans, c)
            assert np.array_equal(Y[:, c], gm.mul_dense(X[:, c], trans=trans))


def test_invalid_arguments_write_nothing():
    gm, _ = _state("bulk")
    m, n = gm.size
    L = D.lib()
    X = np.ones((n, 8))
    for nx, k, ldx, ny, ldy in ((n, -1, 8, m, 8), (n, 8, 7, m, 8), (n, 8, 8, m, 7), (-1, 8, 8, m, 8), (n, 8, 8, -1, 8)):
        Y = np.full((m, 8), np.nan)
        with pytest.raises(D.ArgumentError):
            _spmm_host(gm, X, nx, k, ldx, Y, ny, ldy)
        assert np.all(np.isnan(Y))
    torch = pytest.importorskip("torch")
    dX = torch.ones((n, 8), dtype=torch.float64, device="cuda")
    dY = torch.full((m, 8), float("nan"), dtype=torch.float64, device="cuda")
    for nx, k, ldx, ny, ldy in ((n, -1, 8, m, 8), (n, 8, 7, m, 8), (n, 8, 8, m, 7)):
        with pytest.raises(D.ArgumentError):
            _lib.check(L.dsa_matrix_spmm_dense_d(gm._h, C.c_int(0), C.c_void_p(dX.data_ptr()), C.c_int64(nx), C.c_int64(k),
                                                 C.c_int64(ldx), C.c_void_p(dY.data_ptr()), C.c_int64(ny), C.c_int64(ldy)))
    torch.cuda.synchronize()
    assert bool(torch.isnan(dY).all())
    Y = np.full((m, 8), np.nan)                      # k == 0: nothing is written either
    _spmm_host(gm, X, n, 0, 8, Y, m, 8)
    assert np.all(np.isnan(Y))

