"""Compressed snapshot (dsa_matrix_compress[_dense][_d], DynamicSparseMatrix.compressed / to_csr / to_csc / to_torch) on the
device: both orientations and both forms against a numpy compaction of the device's and of the oracle's export, in every state
an update can leave; bounds, size queries, edge values, the torch path and config 2 at full size."""
import ctypes as C
import time

import numpy as np
import pytest

import dsa_b200 as D
from dsa_b200 import _lib
from compress_ref import compact, dense
from oracle import oracle as O

pytestmark = pytest.mark.gpu

SENT = -7                     # sentinel of the int64 outputs: a call that must write nothing leaves it everywhere
STATES = ["bulk", "batches", "tile", "deleted", "zero_writes"]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _bits(v):
    return np.ascontiguousarray(v, np.float64).view(np.uint64)


def _same(got, want):
    (pk, ptr, k, v), (wpk, wptr, wk, wv) = got, want
    return (np.array_equal(pk, wpk) and np.array_equal(ptr, wptr) and np.array_equal(k, wk)
            and np.array_equal(_bits(v), _bits(wv)))


def _state(name):
    """(device matrix, oracle matrix) after the updates of one state"""
    rng = np.random.default_rng(STATES.index(name) + 40)
    m, n = 3000, 2000
    I, J = rng.integers(1, m + 1, 120_000), rng.integers(1, n + 1, 120_000)
    V = np.where(rng.random(120_000) < 0.02, 0.0, rng.random(120_000) + 0.5)     # explicit zeros from the builder are kept
    gm, om = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)

    def batch(bi, bj, bv):
        gm.set_batch(bi, bj, bv)
        om.set_batch_policy(bi, bj, bv)

    if name in ("batches", "tile"):
        prev = _lib.set_tile_mode(2 if name == "tile" else 0)
        try:
            for _ in range(2):   # inserts (new rows / columns on the random-access pipeline), overwrites, deletes (0.0)
                hi = (m, n) if name == "tile" else (m + 40, n + 40)
                bi, bj = rng.integers(1, hi[0] + 1, 20_000), rng.integers(1, hi[1] + 1, 20_000)
                batch(bi, bj, np.where(rng.random(20_000) < 0.4, 0.0, rng.random(20_000) + 0.5))
        finally:
            _lib.set_tile_mode(prev)
    if name == "deleted":     # tombstones in both orientations; a live column emptied entry by entry
        cols, rows = np.unique(rng.integers(1, n + 1, 300)), np.unique(rng.integers(1, m + 1, 200))
        D.deletecolumn(gm, cols)
        om.delete_columns_policy(cols)
        D.deleterow(gm, rows)
        om.delete_rows_policy(rows)
        c = int(np.setdiff1d(np.arange(1, n + 1), cols)[0])
        rs = np.setdiff1d(I[J == c], rows)                          # a zero write to a deleted row would create it again
        batch(rs, np.full(len(rs), c), np.zeros(len(rs)))
    if name == "zero_writes":  # partitions created by zero writes: empty, above the dimensions that do not grow
        batch(np.array([m + 3, m + 9, 5]), np.array([7, n + 4, n + 11]), np.zeros(3))
        assert gm.size == (m, n)
    return gm, om


def _dims(gm, which):
    m, n = gm.size
    return (n, m) if which == _lib.COLMAJOR else (m, n)


# ---- the four entry points, with sentinel-filled outputs ----------------------------------------------------------------
def _sparse(gm, which, cap=None):
    cnt = np.zeros(2, np.int64)
    _lib.check(D.lib().dsa_matrix_compress(gm._h, C.c_int(which), None, None, None, None, C.c_int64(0), C.c_int64(0), _p(cnt)))
    npart, nnz = (int(c) for c in cnt)
    cp, cn = cap or (npart, nnz)
    pk, ptr = np.full(max(cp, 1), SENT, np.int64), np.full(cp + 1, SENT, np.int64)
    k, v = np.full(max(cn, 1), SENT, np.int64), np.full(max(cn, 1), np.nan)
    _lib.check(D.lib().dsa_matrix_compress(gm._h, C.c_int(which), _p(pk), _p(ptr), _p(k), _p(v), C.c_int64(cp), C.c_int64(cn), _p(cnt)))
    assert cnt.tolist() == [npart, nnz]
    return pk[:npart], ptr[:npart + 1], k[:nnz], v[:nnz], (pk, ptr, k, v)


def _sparse_d(gm, which):
    import torch
    cnt = np.zeros(2, np.int64)
    _lib.check(D.lib().dsa_matrix_compress_d(gm._h, C.c_int(which), None, None, None, None, C.c_int64(0), C.c_int64(0), _p(cnt)))
    npart, nnz = (int(c) for c in cnt)
    t = [torch.full((npart,), SENT, dtype=torch.int64, device="cuda"), torch.full((npart + 1,), SENT, dtype=torch.int64, device="cuda"),
         torch.full((nnz,), SENT, dtype=torch.int64, device="cuda"), torch.full((nnz,), float("nan"), dtype=torch.float64, device="cuda")]
    torch.cuda.synchronize()
    _lib.check(D.lib().dsa_matrix_compress_d(gm._h, C.c_int(which), *(C.c_void_p(x.data_ptr()) for x in t), C.c_int64(npart),
                                             C.c_int64(nnz), _p(cnt)))
    torch.cuda.synchronize()
    return tuple(x.cpu().numpy() for x in t)


def _dense_h(gm, which, dim, idim, base, cap_nnz=None):
    """(return code, ptr, ind, vals) of dsa_matrix_compress_dense; outputs sentinel-filled beforehand"""
    nnz = C.c_int64()
    _lib.check(D.lib().dsa_matrix_compress_dense(gm._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(base), None, None,
                                                 None, C.c_int64(0), C.byref(nnz)))
    cap = nnz.value if cap_nnz is None else cap_nnz
    ptr, ind, v = np.full(dim + 1, SENT, np.int64), np.full(max(cap, 1), SENT, np.int64), np.full(max(cap, 1), np.nan)
    code = D.lib().dsa_matrix_compress_dense(gm._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(base), _p(ptr), _p(ind),
                                             _p(v), C.c_int64(cap), C.byref(nnz))
    return code, ptr, ind[:nnz.value], v[:nnz.value], (ptr, ind, v)


def _dense_d(gm, which, dim, idim, base):
    import torch
    nnz = C.c_int64()
    _lib.check(D.lib().dsa_matrix_compress_dense_d(gm._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(base), None, None,
                                                   None, C.c_int64(0), C.byref(nnz)))
    t = [torch.full((dim + 1,), SENT, dtype=torch.int64, device="cuda"), torch.full((nnz.value,), SENT, dtype=torch.int64, device="cuda"),
         torch.full((nnz.value,), float("nan"), dtype=torch.float64, device="cuda")]
    torch.cuda.synchronize()
    code = D.lib().dsa_matrix_compress_dense_d(gm._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(base),
                                               *(C.c_void_p(x.data_ptr()) for x in t), C.c_int64(nnz.value), C.byref(nnz))
    torch.cuda.synchronize()
    return (code,) + tuple(x.cpu().numpy() for x in t)


# ---- tests --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", [_lib.COLMAJOR, _lib.ROWMAJOR])
@pytest.mark.parametrize("state", STATES)
def test_both_forms_equal_the_compaction_of_both_exports(state, which):
    gm, om = _state(state)
    want = compact(gm.export(which))
    assert _same(compact(om.export(which)), want)                  # the device's layout holds the oracle's contents
    got = _sparse(gm, which)[:4]
    assert _same(got, want), state
    assert _same(_sparse_d(gm, which), want)
    pk, ptr, k, v = want
    assert len(pk) == gm.info(which)["nb_partitions"] and len(k) == gm.info(which)["nnz"]
    dim, idim = _dims(gm, which)
    for base in (0, 1):
        wptr, wind = dense(pk, ptr, k, dim, base)
        code, dptr, ind, dv, _ = _dense_h(gm, which, dim, idim, base)
        assert code == 0 and np.array_equal(dptr, wptr) and np.array_equal(ind, wind) and np.array_equal(_bits(dv), _bits(v))
        code, dptr, ind, dv = _dense_d(gm, which, dim, idim, base)
        assert code == 0 and np.array_equal(dptr, wptr) and np.array_equal(ind, wind) and np.array_equal(_bits(dv), _bits(v))


@pytest.mark.parametrize("which", [_lib.COLMAJOR, _lib.ROWMAJOR])
def test_dense_bounds_write_nothing(which):
    gm, _ = _state("zero_writes")
    dim, idim = _dims(gm, which)
    pk, ptr, k, _ = compact(gm.export(which))
    assert pk.max() > dim                                           # an empty partition above dim: accepted (previous test)
    held = pk[np.diff(ptr) > 0]
    for d, i in ((int(held.max()) - 1, idim), (dim, int(k.max()) - 1), (0, 0)):
        code, _, _, _, bufs = _dense_h(gm, which, d, i, 1)
        assert code == _lib.DSA_ERR_BOUNDS
        assert all((b == SENT).all() for b in bufs[:2]) and np.isnan(bufs[2]).all()
        code, *outs = _dense_d(gm, which, d, i, 0)
        assert code == _lib.DSA_ERR_BOUNDS
        assert all((o == SENT).all() for o in outs[:2]) and np.isnan(outs[2]).all()
    nnz = C.c_int64()
    for d, i, base in ((dim, idim, 2), (-1, idim, 0), (dim, -1, 0)):
        assert D.lib().dsa_matrix_compress_dense(gm._h, C.c_int(which), C.c_int64(d), C.c_int64(i), C.c_int(base), None, None, None,
                                                 C.c_int64(0), C.byref(nnz)) == _lib.DSA_ERR_ARGUMENT
    assert D.lib().dsa_matrix_compress(gm._h, C.c_int(2), None, None, None, None, C.c_int64(0), C.c_int64(0),
                                       _p(np.zeros(2, np.int64))) == _lib.DSA_ERR_ARGUMENT


def test_entries_outside_the_size_raise_bounds_error_in_the_conversions():
    gm = D.dynamicsparse(np.array([1, 7, 2]), np.array([1, 2, 5]), np.array([1.0, 2.0, 3.0]), 5, 3)   # row 7 > m, column 5 > n
    for conv in (gm.to_csr, gm.to_csc, gm.to_torch):
        with pytest.raises(D.BoundsError):
            conv()
    assert compact(gm.export(0))[2].tolist() == [1, 7, 2]


def test_edge_values_bit_for_bit_and_extreme_keys():
    vals = np.array([np.nan, -np.nan, np.inf, -np.inf, -0.0, 0.0, 5e-324, -2.2250738585072014e-309, 1.0], np.float64)
    vals[0] = np.frombuffer(np.uint64(0x7FF800000000BEEF).tobytes(), np.float64)[0]   # a NaN payload
    rows, cols = np.arange(1, 10), np.array([3, 1, 2, 3, 1, 2, 3, 1, 2])
    gm = D.dynamicsparse(rows, cols, vals)
    for which in (_lib.COLMAJOR, _lib.ROWMAJOR):
        want = compact(gm.export(which))
        assert _same(_sparse(gm, which)[:4], want) and _same(_sparse_d(gm, which), want)
        assert sorted(_bits(want[3]).tolist()) == sorted(_bits(vals).tolist())       # stored zeros and -0.0 are entries
    S = gm.to_csc()
    assert np.array_equal(_bits(S.data), _bits(compact(gm.export(0))[3]))
    big = 1 << 62
    gk = D.dynamicsparse(np.array([big - 1, big - 2, 5]), np.array([1, 2, 3]), np.array([1.0, 2.0, 3.0]))
    pk, ptr, k, v = _sparse(gk, _lib.COLMAJOR)[:4]
    assert pk.tolist() == [1, 2, 3] and k.tolist() == [big - 1, big - 2, 5] and ptr.tolist() == [0, 1, 2, 3]
    pk, ptr, k, v = _sparse(gk, _lib.ROWMAJOR)[:4]
    assert pk.tolist() == [5, big - 2, big - 1] and k.tolist() == [3, 2, 1] and v.tolist() == [3.0, 2.0, 1.0]


@pytest.mark.parametrize("which", [_lib.COLMAJOR, _lib.ROWMAJOR])
def test_size_query_and_short_caps_write_nothing(which):
    gm, _ = _state("bulk")
    pk, ptr, k, v = compact(gm.export(which))
    npart, nnz = len(pk), len(k)
    for cap in ((npart - 1, nnz), (npart, nnz - 1)):
        bufs = _sparse(gm, which, cap=cap)[4]
        assert all((b == SENT).all() for b in bufs[:3]) and np.isnan(bufs[3]).all()
    dim, idim = _dims(gm, which)
    code, _, _, _, bufs = _dense_h(gm, which, dim, idim, 0, cap_nnz=nnz - 1)
    assert code == 0 and all((b == SENT).all() for b in bufs[:2]) and np.isnan(bufs[2]).all()
    cnt = np.zeros(2, np.int64)                                     # NULL ptr with every other output present: size query
    _lib.check(D.lib().dsa_matrix_compress(gm._h, C.c_int(which), _p(np.zeros(npart, np.int64)), None, _p(np.zeros(nnz, np.int64)),
                                           _p(np.zeros(nnz)), C.c_int64(npart), C.c_int64(nnz), _p(cnt)))
    assert cnt.tolist() == [npart, nnz]


def test_small_cases():
    ge = D.dynamicsparse(fill_mode=False)                           # empty matrix
    for which in (0, 1):
        pk, ptr, k, v = _sparse(ge, which)[:4]
        assert len(pk) == 0 and ptr.tolist() == [0] and len(k) == 0
        for base in (0, 1):
            code, dptr, ind, _, _ = _dense_h(ge, which, 0, 0, base)
            assert code == 0 and dptr.tolist() == [base] and len(ind) == 0
            assert _dense_d(ge, which, 0, 0, base)[1].tolist() == [base]
    assert ge.to_csr().shape == (0, 0) and ge.to_csc().nnz == 0
    gz, oz = D.dynamicsparse(fill_mode=False), O.Matrix(fill_mode=False)   # live partitions, nnz = 0
    gz.set_batch(np.array([1, 2, 3]), np.array([4, 5, 6]), np.zeros(3))
    oz.set_batch_policy(np.array([1, 2, 3]), np.array([4, 5, 6]), np.zeros(3))
    for which in (0, 1):
        pk, ptr, k, v = _sparse(gz, which)[:4]
        assert pk.tolist() == ([4, 5, 6] if which == 0 else [1, 2, 3]) and ptr.tolist() == [0, 0, 0, 0] and len(k) == 0
        assert _same((pk, ptr, k, v), compact(oz.export(which)))
        assert _dense_h(gz, which, 0, 0, 1)[1].tolist() == [1]      # empty partitions above dim = 0
        assert _dense_h(gz, which, 7, 7, 0)[1].tolist() == [0] * 8


def test_torch_csr_and_csc():
    torch = pytest.importorskip("torch")
    gm, _ = _state("batches")
    m, n = gm.size
    for layout, S in ((torch.sparse_csr, gm.to_csr()), (torch.sparse_csc, gm.to_csc())):
        T = gm.to_torch(layout)
        assert T.layout == layout and T.is_cuda and T.dtype == torch.float64 and tuple(T.shape) == (m, n)
        ptr, ind = (T.crow_indices(), T.col_indices()) if layout == torch.sparse_csr else (T.ccol_indices(), T.row_indices())
        assert ptr.dtype == ind.dtype == torch.int64
        assert np.array_equal(ptr.cpu().numpy(), S.indptr) and np.array_equal(ind.cpu().numpy(), S.indices)
        assert np.array_equal(_bits(T.values().cpu().numpy()), _bits(S.data))
    rng = np.random.default_rng(11)
    x, y = rng.random(n), rng.random(m)
    Tr, Tc = gm.to_torch(torch.sparse_csr), gm.to_torch(torch.sparse_csc)
    for got, want in (((Tr @ torch.from_numpy(x).cuda()).cpu().numpy(), gm.mul_dense(x)),
                      ((Tc.t() @ torch.from_numpy(y).cuda()).cpu().numpy(), gm.mul_dense(y, trans=True))):
        assert np.all(np.abs(got - want) <= 1e-12 * np.maximum(np.abs(got), np.abs(want)))


def test_torch_path_needs_no_host_synchronise():
    torch = pytest.importorskip("torch")
    gm, _ = _state("bulk")
    S = gm.to_csr()
    gm.to_torch()                                                   # warm-up: module load, allocations
    torch.cuda.synchronize()
    for _ in range(3):
        torch.cuda._sleep(400_000_000)                              # ~0.2 s queued on the current stream ahead of the call
        t0 = time.perf_counter()
        T = gm.to_torch()
        host_s = time.perf_counter() - t0
        vals, crow = T.values() * 1.0, T.crow_indices() + 0         # read on the current stream right after the call
        assert np.array_equal(_bits(vals.cpu().numpy()), _bits(S.data)) and np.array_equal(crow.cpu().numpy(), S.indptr)
        assert host_s < 0.1, host_s                                 # the call returned while the sleep was still running


def test_full_size_config2_bit_for_bit():
    """config 2 (bench.make_workload's COO, 1e5 x 1e5, 1e7 nnz, then two bench batches), both orientations, both forms"""
    import bench as B
    _, coo, batches, _ = B.make_workload(3)
    gm = D.dynamicsparse(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    for b in batches[:2]:
        gm.set_batch(*b)
    for which in (_lib.COLMAJOR, _lib.ROWMAJOR):
        want = compact(gm.export(which))
        assert _same(_sparse(gm, which)[:4], want)
        assert _same(_sparse_d(gm, which), want)
        dim, idim = _dims(gm, which)
        wptr, wind = dense(want[0], want[1], want[2], dim, 0)
        code, dptr, ind, dv = _dense_d(gm, which, dim, idim, 0)
        assert code == 0 and np.array_equal(dptr, wptr) and np.array_equal(ind, wind) and np.array_equal(_bits(dv), _bits(want[3]))
