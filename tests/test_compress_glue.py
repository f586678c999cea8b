"""Host glue of the compressed snapshot (DynamicSparseMatrix.compressed / to_csr / to_csc), on the CPU: the test double of
tests/fakelib.py, extended with dsa_matrix_compress and dsa_matrix_compress_dense computed by a numpy compaction of the
oracle's export (same argument conventions: two-call size query, DSA_ERR_BOUNDS with nothing written)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import dsa_b200 as D  # noqa: E402
from dsa_b200 import _lib, api  # noqa: E402
from compress_ref import compact, dense, in_bounds  # noqa: E402
from fakelib import FakeLib, _arr, _set, _val  # noqa: E402


class CompressFakeLib(FakeLib):
    def dsa_matrix_compress(self, h, which, part_keys, ptr, keys, vals, cap_parts, cap_nnz, counts_out2):
        pk, p, k, v = compact(self._get(h).export(_val(which)))
        npart, nnz = len(pk), len(k)
        self.calls.append(("dsa_matrix_compress", nnz))
        _arr(counts_out2, 2, np.int64)[:] = [npart, nnz]
        if not _val(ptr) or _val(cap_parts) < npart or _val(cap_nnz) < nnz or (npart and not _val(part_keys)) or \
                (nnz and not (_val(keys) and _val(vals))):
            return 0
        _arr(part_keys, npart, np.int64)[:] = pk
        _arr(ptr, npart + 1, np.int64)[:] = p
        _arr(keys, nnz, np.int64)[:] = k
        _arr(vals, nnz, np.float64)[:] = v
        return 0

    def dsa_matrix_compress_dense(self, h, which, dim, idim, base, ptr, ind, vals, cap_nnz, nnz_out):
        dim, idim, base = int(_val(dim)), int(_val(idim)), int(_val(base))
        if base not in (0, 1) or dim < 0 or idim < 0:
            self._err = b"compress_dense: bad argument"
            return _lib.DSA_ERR_ARGUMENT
        pk, p, k, v = compact(self._get(h).export(_val(which)))
        self.calls.append(("dsa_matrix_compress_dense", len(k)))
        _set(nnz_out, len(k))
        if not _val(ptr) or _val(cap_nnz) < len(k) or (len(k) and not (_val(ind) and _val(vals))):
            return 0
        if not in_bounds(pk, p, k, dim, idim):
            self._err = b"compress_dense: an entry lies outside dim x idim"
            return _lib.DSA_ERR_BOUNDS
        pd, i = dense(pk, p, k, dim, base)
        _arr(ptr, dim + 1, np.int64)[:] = pd
        _arr(ind, len(k), np.int64)[:] = i
        _arr(vals, len(k), np.float64)[:] = v
        return 0


@pytest.fixture
def fake(monkeypatch):
    lib = CompressFakeLib()
    monkeypatch.setattr(_lib, "lib", lambda: lib)
    monkeypatch.setattr(api, "lib", lambda: lib)
    return lib


def _coo(seed=5, m=40, n=30, nnz=300):
    rng = np.random.default_rng(seed)
    I, J = rng.integers(1, m + 1, nnz), rng.integers(1, n + 1, nnz)
    V = rng.integers(-4, 9, nnz).astype(float)   # explicit zeros among them
    return I, J, V


def _dense(I, J, V, m, n):
    a = np.zeros((m, n))
    np.add.at(a, (I - 1, J - 1), V)
    return a


def _compress_calls(fake):
    return [c[0] for c in fake.calls if c[0].startswith("dsa_matrix_compress")]


@pytest.mark.parametrize("form", ["csr", "csc"])
def test_scipy_output_is_canonical_with_the_matrix_shape(fake, form):
    I, J, V = _coo()
    A = D.dynamicsparse(I, J, V, m=45, n=33)      # trailing empty rows and columns
    S = A.to_csr() if form == "csr" else A.to_csc()
    assert S.format == form and S.shape == A.size == (45, 33)
    assert S.has_canonical_format
    assert np.array_equal(S.toarray(), _dense(I, J, V, 45, 33))
    stored = len({(i, j) for i, j in zip(I.tolist(), J.tolist())})
    assert S.nnz == stored                         # sums that came out 0.0 stay stored entries
    assert _compress_calls(fake) == ["dsa_matrix_compress_dense"] * 2   # size query, then the fill


def test_compressed_is_the_partition_order_of_each_orientation(fake):
    I, J, V = _coo(seed=6)
    A = D.dynamicsparse(I, J, V)
    for which, (pkeys, ikeys) in ((_lib.COLMAJOR, (J, I)), (_lib.ROWMAJOR, (I, J))):
        pk, ptr, k, v = A.compressed(which)
        assert np.array_equal(pk, np.unique(pkeys)) and ptr[0] == 0 and ptr[-1] == len(k) == len(v)
        for t, key in enumerate(pk):
            want = np.unique(ikeys[pkeys == key])
            assert np.array_equal(k[ptr[t]:ptr[t + 1]], want)


def test_compressed_decodes_keys_through_the_codecs(fake):
    A = D.dynamicsparse(["a", "c", "b", "c"], [2, 1, 1, 2], [1.0, 2.0, 3.0, 4.0])
    assert isinstance(A._rc, api.CharCodec)
    pk, ptr, k, v = A.compressed(_lib.COLMAJOR)   # columns are integers, rows are characters
    assert pk.tolist() == [1, 2] and ptr.tolist() == [0, 2, 4]
    assert k.tolist() == ["b", "c", "a", "c"] and v.tolist() == [3.0, 2.0, 1.0, 4.0]
    pk, ptr, k, v = A.compressed(_lib.ROWMAJOR)
    assert pk.tolist() == ["a", "b", "c"] and ptr.tolist() == [0, 1, 2, 4] and k.tolist() == [2, 1, 1, 2]


@pytest.mark.parametrize("conv", ["to_csr", "to_csc"])
def test_codecs_are_refused_by_the_index_conversions(fake, conv):
    A = D.dynamicsparse(["a", "b"], [1, 2], [1.0, 2.0])
    with pytest.raises(D.ArgumentError, match="codec"):
        getattr(A, conv)()
    assert not _compress_calls(fake)


def test_entries_outside_the_size_raise_bounds_error(fake):
    A = D.dynamicsparse([1, 7], [1, 2], [1.0, 2.0], 5, 3)   # m = 5 < max(I): the entry in row 7 is stored
    with pytest.raises(D.BoundsError):
        A.to_csc()
    with pytest.raises(D.BoundsError):
        A.to_csr()
    pk, ptr, k, v = A.compressed(_lib.COLMAJOR)               # the key-space form has no bounds
    assert k.tolist() == [1, 7]


def test_empty_partition_above_the_size_is_accepted(fake):
    A = D.dynamicsparse([1, 2], [1, 2], [1.0, 2.0], 2, 2)
    A[1, 9] = 0.0                                              # creates column 9 without growing n
    assert A.size == (2, 2)
    assert np.array_equal(A.to_csc().toarray(), np.diag([1.0, 2.0]))


def test_pending_writes_and_staged_batches_are_flushed_first(fake):
    I, J, V = _coo(seed=7)
    A = D.dynamicsparse(I, J, V, m=40, n=30)
    A[3, 4] = 100.0
    A.stage_batch(np.array([5, 6]), np.array([7, 8]), np.array([50.0, 60.0]))
    A[6, 8] = 0.0
    S = A.to_csr()
    names = [c[0] for c in fake.calls]
    assert names[-4:] == ["dsa_matrix_apply_staged", "dsa_matrix_set_batch", "dsa_matrix_compress_dense", "dsa_matrix_compress_dense"]
    want = _dense(I, J, V, 40, 30)
    want[2, 3], want[4, 6], want[5, 7] = 100.0, 50.0, 0.0
    assert np.array_equal(S.toarray(), want)
    A[1, 1] = 42.0
    assert A.compressed(_lib.ROWMAJOR)[3][0] == 42.0          # row 1's first entry is column 1
    assert not len(A._pending)


@pytest.mark.parametrize("method", ["compressed", "to_csr", "to_csc"])
def test_fill_mode_is_refused(fake, method):
    A = D.dynamicsparse(fill_mode=True)
    A[1, 1] = 1.0
    with pytest.raises(D.ErrorException, match="fill mode"):
        getattr(A, method)()
    assert not _compress_calls(fake)
