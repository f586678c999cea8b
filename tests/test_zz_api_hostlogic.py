"""The host glue of the drop-in (dynamicsparsearrays.jl_b200/api.py): pending-write queue, fill-mode buffer, key codecs,
operand-order wrappers, sparse-vector arithmetic, exception mapping.

Every test runs twice: on CPU against tests/fakelib.py (a test double of libdsa.so executing on the oracle — host logic only,
no parity claim) and, under `-m gpu`, against the real library through the C ABI.  The expected values are the reference's
own known answers (file:line in each test)."""
import copy
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import dsa_b200 as D  # noqa: E402
from dsa_b200 import _lib, api  # noqa: E402


@pytest.fixture(params=["fake", pytest.param("libdsa", marks=pytest.mark.gpu)])
def backend(request, monkeypatch):
    if request.param == "fake":
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from fakelib import FakeLib
        fake = FakeLib()
        monkeypatch.setattr(_lib, "lib", lambda: fake)
        monkeypatch.setattr(api, "lib", lambda: fake)
        return fake
    _lib.require_gpu()
    return None


# ---------------------------------------------------------------------------------------------------------------------
def test_readme_sequence_and_write_queue(backend):   # README.md:19-40
    I = [1, 1, 2, 4, 3, 5, 1, 4, 1, 5, 1, 5, 4]
    J = [4, 3, 3, 7, 18, 9, 3, 18, 4, 2, 3, 1, 7]
    V = [1, 8, 10, 2, -5, 3, 2, 1, 1, 1, 5, 3, 2]
    A = D.dynamicsparse(I, J, V)
    assert A[1, 3] == 15.0 and A[4, 7] == 4.0 and A[1, 4] == 2.0 and A[2, 2] == 0.0
    A[4, 1] = 1
    A[2, 2] = 0
    A[4, 1] = 7          # same cell twice in the queue: the later write wins (a loop of setindex! would end the same)
    if backend is not None:
        assert not any(c[0] == "dsa_matrix_set_batch" for c in backend.calls)       # still queued on the host
    assert A[4, 1] == 7.0                                                            # the read flushes the queue ...
    if backend is not None:
        assert [c for c in backend.calls if c[0] == "dsa_matrix_set_batch"] == [("dsa_matrix_set_batch", 3)]   # ... as ONE batch
    D.deletecolumn(A, 2)
    assert A[5, 2] == 0.0
    assert A.size == (5, 18)
    with pytest.raises(D.ArgumentError):   # pcsr.jl:208: column does not exist
        D.deletecolumn(A, 999)
    ck = A.export(_lib.COLMAJOR)
    assert ck["col_keys"][ck["col_live"] == 1].tolist() == [1, 3, 4, 7, 9, 18]


def test_flush_threshold_bounds_the_queue(backend):
    A = D.dynamicsparse([1], [1], [1.0])
    A.flush_threshold = 4
    for k in range(2, 12):
        A[k, k] = float(k)
    assert len(A._pending) == 10 - 8      # two automatic flushes of 4
    assert D.nnz(A) == 11
    v = D.dynamicsparsevec([1], [1.0])
    v.flush_threshold = 3
    for k in range(2, 9):
        v[k] = float(k)
    assert len(v._pending) == 1 and D.nnz(v) == 8 and len(v) == 8


def test_char_column_keys(backend):   # test/functional/sparsematrix.jl:302-336 (Test C)
    I = [1, 1, 2, 4, 1, 2, 4, 5, 5, 2]
    J = ['a', 'c', 'c', 'a', 'd', 'a', 'e', 'e', 'c', 'd']
    V = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10]
    A = D.dynamicsparse(I, J, V)
    for i, j, v in zip(I, J, V):
        assert A[i, j] == v
    assert A.size == (5, 'e')
    A[2, 'b'] = 11
    assert A[2, 'b'] == 11
    assert D.nbpartitions(A.rowmajor) == 4 and D.nbpartitions(A.colmajor) == 5
    D.deletecolumn(A, 'a')
    assert A[1, 'a'] == 0 and A[2, 'a'] == 0
    D.deleterow(A, 5)
    assert A[5, 'c'] == 0 and A[5, 'e'] == 0
    assert D.nbpartitions(A.rowmajor) == 3 and D.nbpartitions(A.colmajor) == 4
    keys, vals = A.row(2)               # view(matrix, 2, :) yields the caller's key type
    assert keys == ['b', 'c', 'd'] and vals.tolist() == [11.0, 3.0, 10.0]
    assert list(A.view(2, slice(None))) == [('b', 11.0), ('c', 3.0), ('d', 10.0)]
    keys, vals = A.col('c')
    assert list(keys) == [1, 2] and vals.tolist() == [2.0, 3.0]
    B = copy.deepcopy(A)                # the codecs travel with the copy
    assert B[2, 'd'] == 10 and B.size == (5, 'e')   # deleting row 5 does not shrink the dimensions


def test_spmv_char_rows(backend):   # test/unit/spmv.jl:5-27 (test_spmv_1) and :29-58 (test_spmv_2)
    I = ['a', 'a', 'a', 'b', 'b', 'c', 'd', 'd', 'd']
    J = [1, 3, 5, 2, 4, 4, 1, 4, 5]
    V = [1, 2, 1, 2, 1, 3, 3, 2, 2]
    A = D.dynamicsparse(I, J, V)
    x = D.dynamicsparsevec([1, 3, 5], [1, 1, 1])
    y = A @ x                              # "The multiplication returns a Dict." (spmv.jl:18)
    assert isinstance(y, dict)
    assert y['a'] == 4 and y.get('b', 0.0) == 0.0 and y.get('c', 0.0) == 0.0 and y['d'] == 5 and y.get('e', 0.0) == 0.0
    xt = D.dynamicsparsevec(['a', 'c', 'e'], [1, 1, 1])
    At = A.T
    for i, j, v in zip(I, J, V):
        assert At[j, i] == A[i, j] == v
    yt = At @ xt
    assert yt[1] == 1 and yt[2] == 0.0 and yt[3] == 2 and yt[4] == 3 and yt[5] == 1
    At[2, 'e'] = 5
    assert At[2, 'e'] == A['e', 2] == 5
    assert (At @ {'e': 2.0})[2] == 10.0    # a plain dict is accepted as a vector over non-integer keys
    assert list(xt) == [('a', 1.0), ('c', 1.0), ('e', 1.0)] and xt['c'] == 1.0 and xt['b'] == 0.0


def test_custom_codec(backend):
    # Int32-like keys with negative values: shift by 2^31 (order-preserving, >= 1)
    codec = D.KeyCodec(lambda k: int(k) + (1 << 31) + 1, lambda c: c - (1 << 31) - 1)
    A = D.dynamicsparse([-5, -5, 7], [1, 2, 1], [1.0, 2.0, 3.0], row_codec=codec)
    assert A[-5, 2] == 2.0 and A[7, 1] == 3.0 and A[0, 1] == 0.0
    keys, vals = A.col(1)
    assert keys == [-5, 7] and vals.tolist() == [1.0, 3.0]
    with pytest.raises(D.ArgumentError):
        D.KeyCodec(lambda k: int(k), lambda c: c).encode([0])   # 0 is the semaphore key (pcsr.jl:23)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_vector_addition_subtraction(backend, seed):   # test/functional/math.jl:53-93
    rng = np.random.default_rng(seed)
    r1, v1 = rng.integers(1, 101, 25), rng.integers(1, 11, 25).astype(float)
    r2, v2 = rng.integers(1, 101, 25), rng.integers(1, 11, 25).astype(float)
    d1, d2 = np.zeros(100), np.zeros(100)
    np.add.at(d1, r1 - 1, v1)     # sparsevec(I, V, 100) combines duplicates with +
    np.add.at(d2, r2 - 1, v2)
    a, b = D.dynamicsparsevec(r1, v1, n=100), D.dynamicsparsevec(r2, v2, n=100)
    sa = D.SparseVector(100, np.nonzero(d1)[0] + 1, d1[d1 != 0])
    sb = D.SparseVector(100, np.nonzero(d2)[0] + 1, d2[d2 != 0])
    for s in (a + b, sa + b, a + sb):
        assert isinstance(s, D.SparseVector) and len(s) == 100 and np.array_equal(s.todense(), d1 + d2)
    for s in (a - b, sa - b, a - sb):
        assert np.array_equal(s.todense(), d1 - d2)
        assert not np.any(s.nzval == 0.0)            # cancelled entries are not stored
    assert np.array_equal((-a).todense(), -d1) and (-a) == -sa and (-b) == -sb
    assert a + b == sa + sb and a == sa              # AbstractSparseVector `==`
    with pytest.raises(D.ArgumentError):
        a + D.dynamicsparsevec([1], [1.0], n=7)


def test_fill_mode_buffer_and_views(backend):   # test/unit/views.jl:46-67; matrix.jl:43-51,113-134; buffer.jl:10-31
    A = D.dynamicsparse()                 # dynamicsparse(Int, Int, Int): fill mode
    for (i, j, v) in [(1, 2, 1), (2, 1, 2), (2, 2, 3), (3, 1, 4), (3, 2, 5), (1, 7, 3)]:
        A[i, j] = v
    ids, vals = A.buffer.row(1)
    assert ids.tolist() == [2, 7] and vals.tolist() == [1.0, 3.0]
    with pytest.raises(D.ErrorException):
        A.col(1)                          # matrix.jl:84
    with pytest.raises(D.ErrorException):
        D.deletecolumn(A, 1)              # matrix.jl:96
    with pytest.raises(D.ErrorException):
        A.buffer.addrow(1, [1], [1.0])    # buffer.jl:13: row already written
    D.addrow(A, 9, [5, 3], [1.0, 2.0])    # colids are sorted on entry (buffer.jl:14-16); dims untouched (matrix.jl:116-117)
    assert A.size == (3, 7)
    A[2, 2] = 4                           # duplicates are summed at close (sparsematrix.jl:436-441)
    assert D.closefillmode(A)
    with pytest.raises(D.ErrorException):
        D.closefillmode(A)                # matrix.jl:127
    assert A[2, 2] == 7.0 and A[9, 3] == 2.0 and A[1, 7] == 3.0
    k, v = A.row(9)
    assert list(k) == [3, 5] and v.tolist() == [2.0, 1.0]


def test_staged_flush_bookkeeping(backend):
    A = D.dynamicsparse([1, 2], [1, 2], [1.0, 2.0])
    r1, c1, v1 = np.array([3, 1]), np.array([3, 1]), np.array([3.0, 0.0])
    r2, c2, v2 = np.array([4]), np.array([4]), np.array([4.0])
    A.stage_batch(r1, c1, v1)
    A.stage_batch(r2, c2, v2)
    assert len(A._staged) == 2
    with pytest.raises(D.ErrorException):
        A.stage_batch(r2, c2, v2)         # both slots busy
    assert len(A._staged) == 2            # the failed call left the bookkeeping alone
    A.apply_staged()
    assert len(A._staged) == 1
    A.apply_staged()
    assert A[1, 1] == 0.0 and A[3, 3] == 3.0 and A[4, 4] == 4.0 and D.nnz(A) == 3
    with pytest.raises(D.ErrorException):
        A.apply_staged()                  # nothing staged


def test_vector_misc(backend):   # vector.jl:64,85-90; pma.jl:224-234
    v = D.dynamicsparsevec([1, 10, 3, 5, 3], [1.0, 2.4, 7.1, 1.1, 1.0])
    assert list(v) == [(1, 1.0), (3, 8.1), (5, 1.1), (10, 2.4)]
    w = copy.deepcopy(v)
    assert w == v
    w[10] = 0.0
    assert not (w == v) and D.shrink_size(w) == 5
    with pytest.raises(D.ErrorException):
        copy.copy(v)
    f = v.filter(lambda e: e[1] > 1.05)
    assert list(f) == [(3, 8.1), (5, 1.1), (10, 2.4)]
    with pytest.raises(D.ArgumentError):
        D.dynamicsparsevec([1, 2], [1.0])
    assert D.dynamicsparsevec([1, 2, 1], [2.0, 3.0, 4.0], combine="*")[1] == 8.0


def test_checkpoint_roundtrip(backend, tmp_path):   # SURVEY.md §8f-4
    rng = np.random.default_rng(5)
    I, J = rng.integers(1, 40, 300), rng.integers(1, 30, 300)
    V = rng.integers(-3, 4, 300).astype(float)          # includes explicit zeros at build time (stored, vector.jl:10-36)
    A = D.dynamicsparse(I, J, V, m=50, n=45)
    A.set_batch(rng.integers(1, 40, 60), rng.integers(1, 30, 60), np.where(rng.random(60) < 0.5, 0.0, 2.5))
    D.deletecolumn(A, int(J[0]))
    r, c, v = D.to_coo(A)
    assert len(r) == D.nnz(A) and np.all(np.diff(c) >= 0)            # column by column ...
    same = np.diff(c) == 0
    assert np.all(np.diff(r)[same] > 0)                              # ... ascending rows inside a column
    assert np.array_equal(A.get_batch(r, c), v)
    A[7, 44] = 0.0                                                   # a zero write creates column 44 and keeps it empty
    A[49, 3] = 0.0                                                   # ... and row 49
    D.save_checkpoint(A, tmp_path / "a")                             # np.savez appends ".npz"
    B = D.load_checkpoint(tmp_path / "a")
    assert B.size == A.size == (50, 45) and D.nnz(B) == D.nnz(A)
    for o in ("colmajor", "rowmajor"):                               # live partitions, empty ones included
        assert D.nbpartitions(getattr(B, o)) == D.nbpartitions(getattr(A, o))
    D.deletecolumn(B, 44)                                            # the empty column is there to be deleted
    rb, cb, vb = D.to_coo(B)
    assert np.array_equal(r, rb) and np.array_equal(c, cb) and np.array_equal(v.view(np.int64), vb.view(np.int64))
    x = rng.integers(0, 8, 45).astype(float)     # exact arithmetic: the two layouts may sum a row in different orders
    assert np.array_equal(A.mul_dense(x), B.mul_dense(x))
    w = D.dynamicsparsevec([5, 900, 17], [1.5, -2.0, 0.0], n=1000)
    D.save_checkpoint(w, tmp_path / "w.npz")
    w2 = D.load_checkpoint(tmp_path / "w.npz")
    assert w2 == w and len(w2) == 1000 and list(w2) == [(5, 1.5), (17, 0.0), (900, -2.0)]


def test_packedcsc_simple_use(backend):   # test/functional/sparsematrix.jl:1-121 (pcsc_simple_use)
    keys = [[1, 2, 3], [2, 6, 7], [1, 6, 8]]
    values = [[2, 3, 4], [2, 4, 5], [3, 5, 7]]
    p1 = D.PackedCSC(keys, values)
    assert D.nbpartitions(p1) == 3 and p1.ndim == 2 and D.nnz(p1) == 9
    M = np.array([[2, 0, 3], [3, 2, 0], [4, 0, 0], [0, 0, 0], [0, 0, 0], [0, 4, 5], [0, 5, 0], [0, 0, 7]], float)
    nr, nc = M.shape

    def same(p, M):
        for i in range(nr):
            for j in range(nc):
                assert p[i + 1, j + 1] == M[i, j], (i, j)

    same(p1, M)
    M[0, 0] = 4; p1[1, 1] = 4                       # set
    M[0, 1] += 3; p1[1, 2] = p1[1, 2] + 3           # new element
    M[2, 0] = 0; p1[3, 1] = 0                       # rm
    M[3, 1] = 1; p1[4, 2] = 1                       # new element
    assert D.nnz(p1) == 10 and D.nbpartitions(p1) == 3
    same(p1, M)
    p3 = copy.deepcopy(p1)                          # PackedCSC(pcsc1)
    row = p1[2, :]
    assert D.nnz(row) == 2 and [row[j + 1] for j in range(nc)] == M[1].tolist()
    col = p1[:, 2]
    assert D.nnz(col) == 5 and [col[i + 1] for i in range(nr)] == M[:, 1].tolist()
    for j in (1, 2, 3):
        p3[2, j] = 0
    assert D.nnz(p3[2, :]) == 0
    for i in range(1, 9):
        p3[i, 2] = 0
    assert D.nnz(p3[:, 2]) == 0
    p1[10, 5] = 9                                   # new element and new column: partitions 4 and 5 are created
    assert D.nnz(p1) == 11 and D.nbpartitions(p1) == 5
    p1[1, 4] = 2
    assert D.nnz(p1) == 12
    nb, nb2 = D.nnz(p1), D.nnz(p1[:, 2])
    D.deletepartition(p1, 2)
    assert D.nbpartitions(p1) == 4 and D.nnz(p1) == nb - nb2
    with pytest.raises(D.ErrorException):
        p1[1, 2] = 1                                # column 2 has been deleted (irreversible)
    assert D.nbpartitions(p3) == 3                  # the copy is independent
    # Test B: empty partition, duplicates combined with +
    keys = [[1, 2, 3, 1, 2], [], [2, 6, 7, 7, 5], [1, 6, 8, 2, 1]]
    values = [[2, 3, 4, 1, 1], [], [2, 4, 5, 1, 1], [3, 5, 7, 1, 1]]
    p2 = D.PackedCSC(keys, values)
    assert D.nbpartitions(p2) == 4 and D.nnz(p2) == 11
    M2 = np.array([[3, 0, 0, 4], [4, 0, 2, 1], [4, 0, 0, 0], [0, 0, 0, 0], [0, 0, 1, 0], [0, 0, 4, 5], [0, 0, 6, 0], [0, 0, 0, 7]], float)
    for i in range(8):
        for j in range(4):
            assert p2[i + 1, j + 1] == M2[i, j], (i, j)


# ---------------------------------------------------------------------------------------------------------------------
# round-1 advisor findings
def test_bad_queued_write_raises_at_the_write_site_and_loses_nothing(backend):
    """A[0, 3] = 1 must throw where it is written (the reference throws at the offending setindex!), and the valid writes
    queued around it must survive."""
    A = D.dynamicsparse([1], [1], [1.0])
    A[2, 2] = 5
    with pytest.raises(D.ArgumentError):
        A[0, 3] = 1
    A[3, 3] = 7
    assert A[2, 2] == 5.0 and A[3, 3] == 7.0 and A[1, 1] == 1.0
    v = D.dynamicsparsevec([1], [1.0])
    v[4] = 2.0
    with pytest.raises(D.ArgumentError):
        v[-(1 << 63)] = 1.0
    assert v[4] == 2.0


def test_staged_batch_keeps_arrival_order(backend):
    """stage_batch / apply_staged are last-writer-wins in ARRIVAL order whatever the caller interleaves: a write issued after
    a staged batch wins over it; reads, deletes and copies see the staged batch."""
    E = D.dynamicsparse([1], [1], [1.0])
    E.stage_batch([1], [1], [2.0])
    E[1, 1] = 3.0                          # later than the staged batch
    assert E[1, 1] == 3.0                  # the read drains the staged batch first, then the queue
    assert not E._staged
    E.stage_batch([2, 2], [2, 3], [4.0, 5.0])
    assert E[2, 3] == 5.0                  # reads see a staged batch
    E.stage_batch([3], [3], [6.0])
    c = copy.deepcopy(E)                   # so do copies ...
    assert c[3, 3] == 6.0
    E.stage_batch([4], [3], [8.0])
    D.deletecolumn(E, 3)                   # ... and deletes (the staged entry of column 3 is applied, then deleted)
    assert E[4, 3] == 0.0 and E[3, 3] == 0.0 and E[2, 2] == 4.0
    E.stage_batch([1], [1], [9.0])
    E.stage_batch([1], [1], [10.0])
    E.apply_staged()
    assert len(E._staged) == 1
    assert E[1, 1] == 10.0 and not E._staged


def test_missing_dimension_is_guessed_on_its_own(backend):   # matrix.jl:15: m = _guess_length(I), n = _guess_length(J)
    A = D.dynamicsparse([1, 3], [2, 7], [1.0, 2.0], m=5)
    assert A.size == (5, 7)
    B = D.dynamicsparse([1, 3], [2, 7], [1.0, 2.0], n=9)
    assert B.size == (3, 9)
    y = A.mul_dense(np.ones(5), trans=True)
    assert len(y) == 7 and y[1] == 1.0 and y[6] == 2.0


def test_bench_dump_outputs(backend, tmp_path, monkeypatch):
    """bench.py --dump-outputs at a reduced size: the last batch's values read back last-writer-wins, the entry sample is a
    seeded subset of to_coo, and every file is float64."""
    import bench as B
    monkeypatch.setattr(B, "N_OVER", 200)
    monkeypatch.setattr(B, "DUMP_SAMPLE", 3000)
    x, coo, batches, _ = B.make_workload(3, m=3000, n=3000, nnz0=20_000, nb=4000, seed=11)
    A = D.dynamicsparse(coo[0], coo[1], coo[2], m=3000, n=3000)
    for b in batches:
        A.set_batch(*b)
    y = A.mul_dense(x)
    B.dump_outputs(str(tmp_path), B.outputs_of_last_step(A, y, batches[-1]))
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(got) == ["batch_vals", "entries_cols", "entries_rows", "entries_vals", "y"]
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["y"], y)
    bi, bj, bv = batches[-1]
    lin = bi * 3001 + bj
    last = len(lin) - 1 - np.unique(lin[::-1], return_index=True)[1]   # the last write of every (i, j) in the batch
    assert np.array_equal(got["batch_vals"][last], bv[last])
    r, c, v = D.to_coo(A)
    pick = np.sort(np.random.default_rng(B.SEED).choice(len(r), 3000, replace=False))
    assert np.array_equal(got["entries_rows"], r[pick]) and np.array_equal(got["entries_cols"], c[pick])
    assert np.array_equal(got["entries_vals"], v[pick])
