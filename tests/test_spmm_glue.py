"""Host glue of the multi-vector product (DynamicSparseMatrix.mul_dense with a 2-D x), on the CPU: the test double of
tests/fakelib.py, extended with dsa_matrix_spmm_dense computed column by column by the oracle's dense product."""
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


class SpmmFakeLib(FakeLib):
    def dsa_matrix_spmm_dense(self, h, trans, X, nx, k, ldx, Y, ny, ldy):
        nx, k, ldx, ny, ldy = (int(_val(a)) for a in (nx, k, ldx, ny, ldy))
        self.calls.append(("dsa_matrix_spmm_dense", k))
        if nx < 0 or ny < 0 or k < 0 or ldx < k or ldy < k:
            self._err = b"spmm_dense: need nx >= 0, ny >= 0, k >= 0, ldx >= k and ldy >= k"
            return _lib.DSA_ERR_ARGUMENT
        if k == 0 or ny == 0:
            return 0
        xs = _arr(X, (nx - 1) * ldx + k, np.float64) if nx else np.zeros(0)
        ys = _arr(Y, (ny - 1) * ldy + k, np.float64)

        def run():
            for c in range(k):
                ys[c::ldy][:ny] = self._get(h).mul_dense(xs[c::ldx][:nx].copy(), ny, trans=bool(_val(trans)))
        return self._guard(run)

    def dsa_matrix_spmv_dense(self, h, trans, x, nx, y, ny):
        self.calls.append(("dsa_matrix_spmv_dense", int(_val(nx))))
        return super().dsa_matrix_spmv_dense(h, trans, x, nx, y, ny)


@pytest.fixture
def fake(monkeypatch):
    lib = SpmmFakeLib()
    monkeypatch.setattr(_lib, "lib", lambda: lib)
    monkeypatch.setattr(api, "lib", lambda: lib)
    return lib


def _matrix():
    rng = np.random.default_rng(5)
    I, J = rng.integers(1, 41, 300), rng.integers(1, 31, 300)
    V = rng.integers(1, 9, 300).astype(float)
    return D.dynamicsparse(I, J, V, m=40, n=30), (I, J, V)


def _dense(I, J, V, m, n):
    a = np.zeros((m, n))
    np.add.at(a, (I - 1, J - 1), V)
    return a


def _spmm_calls(fake):
    return [c for c in fake.calls if c[0] == "dsa_matrix_spmm_dense"]


@pytest.mark.parametrize("order", ["C", "F"])
def test_2d_numpy_input_both_orders(fake, order):
    A, (I, J, V) = _matrix()
    X = np.asarray(np.random.default_rng(1).integers(0, 5, (30, 6)), dtype=float, order=order)
    Y = A.mul_dense(X)
    assert isinstance(Y, np.ndarray) and Y.dtype == np.float64 and Y.shape == (40, 6)
    assert np.array_equal(Y, _dense(I, J, V, 40, 30) @ X)        # integer-valued data: exact in any order
    assert _spmm_calls(fake) == [("dsa_matrix_spmm_dense", 6)]
    assert not any(c[0] == "dsa_matrix_spmv_dense" for c in fake.calls)


def test_trans_takes_the_column_count(fake):
    A, (I, J, V) = _matrix()
    X = np.random.default_rng(2).integers(0, 5, (40, 3)).astype(float)
    Y = A.mul_dense(X, trans=True)
    assert Y.shape == (30, 3)                                       # size[1]
    assert np.array_equal(Y, _dense(I, J, V, 40, 30).T @ X)


def test_1d_input_keeps_the_single_vector_entry_point(fake):
    A, (I, J, V) = _matrix()
    x = np.arange(30, dtype=float)
    y = A.mul_dense(x)
    assert y.shape == (40,) and np.array_equal(y, _dense(I, J, V, 40, 30) @ x)
    assert [c for c in fake.calls if c[0] == "dsa_matrix_spmv_dense"] == [("dsa_matrix_spmv_dense", 30)]
    assert not _spmm_calls(fake)


def test_pending_writes_and_staged_batches_are_flushed_first(fake):
    A, (I, J, V) = _matrix()
    A[3, 4] = 100.0                                                 # queued single write
    rows, cols, vals = np.array([5, 6]), np.array([7, 8]), np.array([50.0, 60.0])
    A.stage_batch(rows, cols, vals)                                 # staged batch
    A[6, 8] = 0.0                                                   # later single write deletes a staged entry
    Y = A.mul_dense(np.ones((30, 2)))
    names = [c[0] for c in fake.calls]
    assert names[-3:] == ["dsa_matrix_apply_staged", "dsa_matrix_set_batch", "dsa_matrix_spmm_dense"]
    assert not A._staged and not len(A._pending)
    want = _dense(I, J, V, 40, 30)
    want[2, 3], want[4, 6], want[5, 7] = 100.0, 50.0, 0.0
    assert np.array_equal(Y[:, 0], want.sum(axis=1)) and np.array_equal(Y[:, 1], want.sum(axis=1))


def test_fill_mode_is_refused(fake):
    A = D.dynamicsparse(fill_mode=True)
    A[1, 1] = 1.0
    with pytest.raises(D.ErrorException, match="Matrix is in fill mode"):
        A.mul_dense(np.ones((1, 2)))
    assert not _spmm_calls(fake)


def test_3d_input_is_rejected(fake):
    A, _ = _matrix()
    with pytest.raises(D.ArgumentError):
        A.mul_dense(np.ones((30, 2, 2)))
    assert not _spmm_calls(fake)
