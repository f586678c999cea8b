"""Host glue of the sparse multi-vector product (DynamicSparseMatrix.mul_sparse with a matrix X), on the CPU: the test double of
tests/fakelib.py (with the compaction of test_compress_glue, for DynamicSparseMatrix operands), extended with dsa_matrix_spmspm
answered column by column by the oracle's own loop (mpcsc_mul), with the library's argument checks."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import dsa_b200 as D  # noqa: E402
from dsa_b200 import _lib, api  # noqa: E402
from fakelib import _arr, _set, _val  # noqa: E402
from test_compress_glue import CompressFakeLib  # noqa: E402


class SpmspmFakeLib(CompressFakeLib):
    def dsa_matrix_spmspm(self, h, trans, xp, xk, xv, k, nnz_x, yp, yk, yv, cap, count_out):
        k, nnz_x, cap = int(_val(k)), int(_val(nnz_x)), int(_val(cap))
        _set(count_out, 0)
        self.calls.append(("dsa_matrix_spmspm", int(_val(trans)), k, nnz_x, bool(_val(yk))))
        if k < 0 or nnz_x < 0:
            self._err = b"spmspm: k and nnz_x must be >= 0"
            return _lib.DSA_ERR_ARGUMENT
        ptr = _arr(xp, k + 1, np.int64).copy()
        ok = ptr[0] == 0 and np.all(np.diff(ptr) >= 0) and ptr[k] == nnz_x
        keys, vals = (_arr(xk, nnz_x, np.int64).copy(), _arr(xv, nnz_x, np.float64).copy()) if ok else (None, None)
        if not ok or any(np.any(np.diff(keys[ptr[c]:ptr[c + 1]]) <= 0) for c in range(k)):
            self._err = b"x_ptr must start at 0, never decrease and end at nnz_x, and x keys must be strictly ascending"
            return _lib.DSA_ERR_ARGUMENT
        cols = [self._get(h).mul(keys[ptr[c]:ptr[c + 1]], vals[ptr[c]:ptr[c + 1]], trans=bool(_val(trans))) for c in range(k)]
        out_p = np.concatenate([[0], np.cumsum([len(c[0]) for c in cols])]).astype(np.int64)
        n = int(out_p[-1])
        _set(count_out, n)
        if n <= cap:
            if _val(yp):
                _arr(yp, k + 1, np.int64)[:] = out_p
            if n and _val(yk) and _val(yv):
                _arr(yk, n, np.int64)[:] = np.concatenate([c[0] for c in cols])
                _arr(yv, n, np.float64)[:] = np.concatenate([c[1] for c in cols])
        return 0


@pytest.fixture
def fake(monkeypatch):
    lib = SpmspmFakeLib()
    monkeypatch.setattr(_lib, "lib", lambda: lib)
    monkeypatch.setattr(api, "lib", lambda: lib)
    return lib


def _matrix(m=40, n=30, seed=11):
    rng = np.random.default_rng(seed)
    I, J = rng.integers(1, m + 1, 300), rng.integers(1, n + 1, 300)
    V = rng.integers(1, 9, 300).astype(float)
    a = np.zeros((m, n))
    np.add.at(a, (I - 1, J - 1), V)
    return D.dynamicsparse(I, J, V, m=m, n=n), a


def _spmspm_calls(fake):
    return [c for c in fake.calls if c[0] == "dsa_matrix_spmspm"]


def _expect(a, X):
    """integer-valued data: exact in any order; a column's touched keys are the rows with a stored entry in a selected column"""
    X = sp.csc_matrix(X)
    X.sum_duplicates()
    cols = []
    for c in range(X.shape[1]):
        sel = X.indices[X.indptr[c]:X.indptr[c + 1]]
        touched = np.nonzero((a[:, sel] != 0).any(axis=1))[0]
        cols.append((touched, (a @ X[:, c].toarray().ravel())[touched]))
    return cols


def _assert_csc(Y, a, X):
    assert isinstance(Y, sp.csc_matrix) and Y.shape == (a.shape[0], X.shape[1])
    for c, (rows, vals) in enumerate(_expect(a, X)):
        got = slice(Y.indptr[c], Y.indptr[c + 1])
        assert np.array_equal(Y.indices[got], rows) and np.array_equal(Y.data[got], vals), c


def test_scipy_formats_with_unsorted_indices_and_duplicates(fake):
    A, a = _matrix()
    # column 1 holds row 4 twice (summed to 3.0) and its rows out of order; column 2 is empty
    rows, cols, vals = np.array([4, 0, 4, 17, 29, 2]), np.array([1, 1, 1, 0, 3, 3]), np.array([1.0, -2.0, 2.0, 5.0, 1.0, -1.0])
    coo = sp.coo_matrix((vals, (rows, cols)), shape=(30, 4))
    csc = sp.csc_matrix((np.array([5.0, 1.0, -2.0, 2.0, -1.0, 1.0]), np.array([17, 4, 0, 4, 2, 29]), np.array([0, 1, 4, 4, 6])),
                        shape=(30, 4))
    assert not csc.has_canonical_format
    for X in (coo, coo.tocsr(), csc, sp.csr_array(coo), sp.lil_matrix(coo)):
        _assert_csc(A.mul_sparse(X), a, coo)
    assert all(c[1:4] == (0, 4, 5) for c in _spmspm_calls(fake))          # 5 entries: the duplicates summed
    names = [c[0] for c in fake.calls]
    assert "dsa_matrix_spmv" not in names and "dsa_matrix_spmspv" not in names


def test_transposed_product_and_result_shapes(fake):
    A, a = _matrix()
    X = sp.random(40, 6, density=0.2, random_state=3, format="csc")
    X.data[:] = np.arange(1, X.nnz + 1)
    Y = A.mul_sparse(X, trans=True)
    assert Y.shape == (30, 6)
    _assert_csc(Y, a.T, X)
    Z = A.mul_sparse(sp.csc_matrix((30, 0)))                                # k = 0
    assert Z.shape == (40, 0) and Z.nnz == 0 and Z.indptr.tolist() == [0]
    E = A.mul_sparse(sp.csc_matrix((30, 3)))                                # empty columns
    assert E.shape == (40, 3) and E.nnz == 0 and E.indptr.tolist() == [0, 0, 0, 0]
    W = A.mul_sparse(sp.csc_matrix(([1.0], ([0], [0])), shape=(1000, 2)))   # more rows than A has columns: not checked
    assert W.shape == (40, 2)


def test_size_query_then_fill(fake):
    A, _ = _matrix()
    A.mul_sparse(sp.eye(30, 5, format="csc"))
    calls = _spmspm_calls(fake)
    assert [c[4] for c in calls] == [False, True]


def test_dynamic_matrix_operand_is_its_column_major_compaction(fake):
    A, a = _matrix()
    B, b = _matrix(m=30, n=7, seed=12)
    Y, Yc = A.mul_sparse(B), A.mul_sparse(B.to_csc())
    assert (Y != Yc).nnz == 0 and np.array_equal(Y.indptr, Yc.indptr) and np.array_equal(Y.indices, Yc.indices)
    _assert_csc(Y, a, sp.csc_matrix(b))


def test_result_key_above_the_dimension_is_bounds_error(fake):
    A = D.dynamicsparse([1, 9], [1, 2], [1.0, 2.0], m=5, n=2)              # row 9 stored outside m = 5
    with pytest.raises(D.BoundsError):
        A.mul_sparse(sp.csc_matrix(([1.0], ([1], [0])), shape=(2, 1)))
    Y = A.mul_sparse(sp.csc_matrix(([1.0], ([0], [0])), shape=(2, 1)))     # column 1 stays inside
    assert Y.shape == (5, 1) and Y.indices.tolist() == [0] and Y.data.tolist() == [1.0]


def test_key_codec_is_refused_for_matrix_operands(fake):
    A = D.dynamicsparse([1, 2, 2], ['a', 'c', 'e'], [1.0, 2.0, 3.0], col_codec=D.CharCodec())
    B, _ = _matrix(m=3, n=2)
    for X in (sp.eye(3, 2, format="csc"), B):
        with pytest.raises(D.ArgumentError, match="codec"):
            A.mul_sparse(X)
    assert not _spmspm_calls(fake)


def test_argument_errors(fake):
    import ctypes as C
    A, _ = _matrix()
    L = api.lib()
    P = lambda a: np.asarray(a, np.int64).ctypes.data_as(C.c_void_p)  # noqa: E731

    def call(ptr, keys, k, nnz_x):
        ptr, keys = np.asarray(ptr, np.int64), np.asarray(keys, np.int64)
        vals = np.ones(max(len(keys), 1))
        cnt = C.c_int64(-1)
        yp = np.full(max(k, 0) + 1, -7, np.int64)
        code = L.dsa_matrix_spmspm(A._h, C.c_int(0), P(ptr), P(keys), vals.ctypes.data_as(C.c_void_p), C.c_int64(k), C.c_int64(nnz_x),
                                   yp.ctypes.data_as(C.c_void_p), None, None, C.c_int64(100), C.byref(cnt))
        return code, yp
    for ptr, keys, k, nnz_x in (([0, 1], [1], -1, 1), ([0, 1], [1], 1, -1), ([1, 2], [1, 2], 1, 2), ([0, 2, 1], [1, 2], 2, 2),
                                ([0, 2], [1, 2], 1, 3), ([0, 2], [3, 3], 1, 2), ([0, 2], [4, 3], 1, 2)):
        code, yp = call(ptr, keys, k, nnz_x)
        assert code == _lib.DSA_ERR_ARGUMENT and np.all(yp == -7), (ptr, keys, k, nnz_x)
    code, yp = call([0, 2, 3], [5, 9, 2], 2, 3)                          # descending across a column boundary is legal
    assert code == 0 and yp[0] == 0
    code, _ = call([0, 2], [2, 2], 1, 2)
    with pytest.raises(D.ArgumentError, match="ascending"):
        _lib.check(code)
