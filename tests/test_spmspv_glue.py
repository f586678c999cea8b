"""Host glue of the sparse-x product in the reference's order (DynamicSparseMatrix.mul_sparse), on the CPU: the test double of
tests/fakelib.py, extended with dsa_matrix_spmspv answered by the oracle's own loop (mpcsc_mul) on the same orientation."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import dsa_b200 as D  # noqa: E402
from dsa_b200 import _lib, api  # noqa: E402
from fakelib import FakeLib, _arr, _val  # noqa: E402


class SpmspvFakeLib(FakeLib):
    def dsa_matrix_spmspv(self, h, trans, xk, xv, nx, yk, yv, cap, count_out):
        keys, vals = _arr(xk, nx, np.int64).copy(), _arr(xv, nx, np.float64).copy()
        self.calls.append(("dsa_matrix_spmspv", int(_val(trans)), len(keys)))
        if np.any(np.diff(keys) <= 0):
            self._err = b"x keys must be strictly ascending"
            return _lib.DSA_ERR_ARGUMENT

        def run():
            k, v = self._get(h).mul(keys, vals, trans=bool(_val(trans)))
            self._span(k, v, yk, yv, cap, count_out)
        return self._guard(run)


@pytest.fixture
def fake(monkeypatch):
    lib = SpmspvFakeLib()
    monkeypatch.setattr(_lib, "lib", lambda: lib)
    monkeypatch.setattr(api, "lib", lambda: lib)
    return lib


def _matrix():
    rng = np.random.default_rng(11)
    I, J = rng.integers(1, 41, 300), rng.integers(1, 31, 300)
    V = rng.integers(1, 9, 300).astype(float)
    return D.dynamicsparse(I, J, V, m=40, n=30), (I, J, V)


def _dense(I, J, V, m, n):
    a = np.zeros((m, n))
    np.add.at(a, (I - 1, J - 1), V)
    return a


def _spmspv_calls(fake):
    return [c for c in fake.calls if c[0] == "dsa_matrix_spmspv"]


def _expect(a, xk, xv):
    """integer-valued data: exact in any order; the touched keys are the rows with a stored entry in a selected column"""
    xd = np.zeros(a.shape[1])
    xd[np.asarray(xk) - 1] = xv
    touched = np.nonzero((a[:, np.asarray(xk) - 1] != 0).any(axis=1))[0] + 1
    return touched, (a @ xd)[touched - 1]


def test_every_x_form_and_both_orientations(fake):
    A, (I, J, V) = _matrix()
    a = _dense(I, J, V, 40, 30)
    xk, xv = np.array([2, 5, 17, 30]), np.array([1.0, -2.0, 3.0, 0.0])
    want_k, want_v = _expect(a, xk, xv)
    forms = [(xk, xv), D.SparseVector(30, xk, xv), D.dynamicsparsevec(xk, xv, n=30)]
    for x in forms:
        y = A.mul_sparse(x)
        assert isinstance(y, D.SparseVector) and len(y) == 40
        assert np.array_equal(y.nzind, want_k) and np.array_equal(y.nzval, want_v)
    tk, tv = np.array([1, 9, 40]), np.array([2.0, 1.0, -1.0])
    want_k, want_v = _expect(a.T, tk, tv)
    y = A.mul_sparse((tk, tv), trans=True)
    assert len(y) == 30 and np.array_equal(y.nzind, want_k) and np.array_equal(y.nzval, want_v)
    assert _spmspv_calls(fake) == [("dsa_matrix_spmspv", 0, 4)] * 3 + [("dsa_matrix_spmspv", 1, 3)]
    assert not any(c[0] == "dsa_matrix_spmv" for c in fake.calls)


def test_same_result_as_the_streaming_product(fake):
    A, _ = _matrix()
    x = (np.array([3, 4, 8, 21]), np.array([0.5, 1.0, 2.0, -4.0]))
    for trans in (False, True):
        y, ys = A.mul_sparse(x, trans=trans), (A.T @ x if trans else A @ x)
        assert np.array_equal(y.nzind, ys.nzind) and np.array_equal(y.nzval, ys.nzval)


def test_codec_keys_give_a_dict(fake):
    A = D.dynamicsparse([1, 2, 2], ['a', 'c', 'e'], [1.0, 2.0, 3.0], col_codec=D.CharCodec())
    y = A.mul_sparse({'e': 2.0, 'a': 1.0})          # x over the column keys; integer row keys: a SparseVector
    assert isinstance(y, D.SparseVector) and y.nzind.tolist() == [1, 2] and y.nzval.tolist() == [1.0, 6.0]
    assert A.mul_sparse({2: 1.0}, trans=True) == {'c': 2.0, 'e': 3.0}   # output over the column keys: the Dict


def test_non_ascending_x_is_refused(fake):
    A, _ = _matrix()
    for keys in ([5, 5], [7, 3]):
        with pytest.raises(D.ArgumentError, match="ascending"):
            A.mul_sparse((np.array(keys), np.ones(2)))


def test_pending_writes_are_flushed_first(fake):
    A, (I, J, V) = _matrix()
    A[3, 4] = 100.0
    y = A.mul_sparse((np.array([4]), np.array([1.0])))
    names = [c[0] for c in fake.calls]
    assert names[-2:] == ["dsa_matrix_set_batch", "dsa_matrix_spmspv"]
    a = _dense(I, J, V, 40, 30)
    a[2, 3] = 100.0
    want_k, want_v = _expect(a, [4], [1.0])
    assert np.array_equal(y.nzind, want_k) and np.array_equal(y.nzval, want_v)


def test_fill_mode_is_refused(fake):
    A = D.dynamicsparse(fill_mode=True)
    A[1, 1] = 1.0
    with pytest.raises(D.ErrorException, match="Matrix is in fill mode"):
        A.mul_sparse((np.array([1]), np.array([1.0])))
    assert not _spmspv_calls(fake)
