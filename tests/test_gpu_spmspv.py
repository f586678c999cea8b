"""Sparse-x product in the reference's order (dsa_matrix_spmspv[_d], DynamicSparseMatrix.mul_sparse) on the device.

Every result is compared with the oracle's `mul` (mpcsc_mul: a literal restatement of _mul_dyn_mat_col_loop!,
operations.jl:62-105) on the same orientation: keys exactly, values as their 64-bit patterns (NaN compared as NaN: the payload
a NaN propagates is the hardware's).  The streaming product (`A @ x`) must touch the same keys and stay within the error bound
of test_gpu_edge_values.check_rows, and the new call must never stream the matrix."""
import ctypes as C

import numpy as np
import pytest

import dsa_b200 as D
from oracle import oracle as O
from test_gpu_edge_values import GAP, bits, cancel_coo, check_rows, exact_products, paired, spread, _layout
from test_gpu_parity import _kernels_of

pytestmark = pytest.mark.gpu

STREAMING_KERNELS = ("spmv_blocked", "scatter_x")


def assert_like_oracle(y, om, xk, xv, trans, what=""):
    """y = (keys, values) or a SparseVector; equal to om.mul bit for bit (NaN by class)"""
    yk, yv = (y.nzind, y.nzval) if isinstance(y, D.SparseVector) else y
    ok, ov = om.mul(xk, xv, trans=trans)
    assert np.array_equal(np.asarray(yk), ok), (what, "keys differ from the oracle's", len(yk), len(ok))
    gv = np.asarray(yv, np.float64)
    gn, on = np.isnan(gv), np.isnan(ov)
    assert np.array_equal(gn, on), (what, "NaN rows differ", ok[gn != on][:5])
    diff = np.nonzero(bits(gv)[~gn] != bits(ov)[~on])[0]
    assert len(diff) == 0, (what, "value bits differ", ok[~on][diff[:5]], gv[~gn][diff[:5]], ov[~on][diff[:5]])


def check(gm, om, xk, xv, trans, what=""):
    xk, xv = np.asarray(xk, np.int64), np.asarray(xv, np.float64)
    y = gm.mul_sparse((xk, xv), trans=trans)
    assert len(y) == gm.size[1 if trans else 0]
    assert_like_oracle(y, om, xk, xv, trans, what)
    return y


def cross_check_streaming(gm, om, xk, xv, trans, what=""):
    """same touched keys as the streaming product, values within its error bound against the exact sums"""
    y = check(gm, om, xk, xv, trans, what)
    ys = (gm.T if trans else gm) @ (xk, xv)
    assert np.array_equal(y.nzind, ys.nzind), (what, "touched keys differ from A @ x")
    ref = exact_products(om, (xk, xv), trans)
    assert np.array_equal(ref["keys"], y.nzind)
    check_rows(np.asarray(y.nzval), ref, what)


def x_cases(rng, om, trans, dim):
    """(name, keys, values): ascending keys over the partition axis of the product (columns for A·x, rows for Aᵀ·x)"""
    e = om.export(1 if trans else 0)
    live = e["col_keys"][e["col_live"].astype(bool)]
    dead = np.setdiff1d(np.arange(1, dim + 1), live)           # deleted (tombstoned) or never created partitions
    sub = np.sort(rng.choice(live, max(1, len(live) // 3), replace=False)) if len(live) else np.zeros(0, np.int64)
    extra = np.array([-(2 ** 63) + 1, -7, 0, dim + 1, dim + 1000, 2 ** 62, 2 ** 63 - 1], np.int64)
    absent = np.unique(np.concatenate([sub, dead[:20], extra]))
    special = np.sort(rng.choice(live, min(len(live), 8), replace=False)) if len(live) else np.zeros(0, np.int64)
    sv = np.array([0.0, np.nan, np.inf, -np.inf, -0.0, 5e-324, 1e-310, -2.5])[:len(special)]
    allk = np.arange(1, dim + 1)
    return [
        ("subset", sub, spread(rng, len(sub))),
        ("absent_deleted_negative", absent, spread(rng, len(absent))),
        ("specials", special, sv),
        ("empty", np.zeros(0, np.int64), np.zeros(0)),
        ("single", live[:1], np.array([3.0])[:min(1, len(live))]),
        ("all", allk, paired(rng, dim)),
    ]


def run_cases(gm, om, rng, what):
    m, n = gm.size
    for trans in (False, True):
        dim = m if trans else n
        for name, xk, xv in x_cases(rng, om, trans, dim):
            if name == "specials":
                check(gm, om, xk, xv, trans, (what, trans, name))
            else:
                cross_check_streaming(gm, om, xk, xv, trans, (what, trans, name))


@pytest.mark.parametrize("name", ["bulk", "random_access", "tile", "deleted", "long", "short"])
def test_layouts_bit_for_bit(name):
    gm, om, _ = _layout(name)
    rng = np.random.default_rng(["bulk", "random_access", "tile", "deleted", "long", "short"].index(name) + 4900)
    run_cases(gm, om, rng, name)
    xk = np.arange(1, gm.size[1] + 1)
    names = _kernels_of(lambda: gm.mul_sparse((xk, np.ones(len(xk)))))
    assert "spmspv_emit" in names and not any(k in names for k in STREAMING_KERNELS), sorted(names)


def test_long_partition_is_cut_into_pieces():
    """column 5 and row 7 of the "long" layout hold 60 000 cells each: one x entry, many warps"""
    gm, om, _ = _layout("long")
    for trans, key in ((False, 5), (True, 7)):
        y = check(gm, om, [key], [1.5], trans, ("long", trans))
        assert len(y.nzind) >= 60_000


@pytest.mark.parametrize("shape", [(3, 3, 4), (5, 7, 12), (9, 6, 30), (12, 12, 60)])
def test_tiny_matrices(shape):
    m, n, nnz = shape
    rng = np.random.default_rng(nnz + 50)
    I, J, V = cancel_coo(rng, m, n, nnz)
    gm, om = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    run_cases(gm, om, rng, shape)


def test_empty_matrix():
    gm, om = D.dynamicsparse(fill_mode=False), O.Matrix(fill_mode=False)
    for trans in (False, True):
        for xk in ([], [1, 2, 3]):
            y = check(gm, om, xk, np.ones(len(xk)), trans, ("empty", trans))
            assert len(y.nzind) == 0


def test_negative_zero_products_fold_from_positive_zero():
    """a row whose only products are -0.0 comes out +0.0 (0.0 + -0.0), as the reference's get(result, row, 0.0) + p"""
    rng = np.random.default_rng(4950)
    gm = D.dynamicsparse([1, 2, 2, 3], [1, 1, 2, 2], [1.0, 2.0, -3.0, 4.0], m=3, n=2)
    om = O.Matrix([1, 2, 2, 3], [1, 1, 2, 2], [1.0, 2.0, -3.0, 4.0], m=3, n=2)
    y = check(gm, om, [1], [-0.0], False, "-0")
    assert y.nzind.tolist() == [1, 2] and np.all(bits(y.nzval) == 0)
    y = check(gm, om, [1, 2], [-0.0, 0.0], False, "-0 then +0")   # row 2: fl(fl(0 + -0) + fl(0 * -3)) = 0 + -0 = +0
    assert np.all(bits(y.nzval) == 0)
    check(gm, om, [1, 2], spread(rng, 2), True, "trans")


@pytest.mark.parametrize("base", [1 << 27, (1 << 62) - 10_000])
def test_keys_above_2_26_and_near_2_62(base):
    rng = np.random.default_rng(5000 + (base > 1 << 40))
    I, J, V = cancel_coo(rng, 800, 600, 12_000)
    I, J = I + base, J + base
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    for trans, keys in ((False, np.unique(J)), (True, np.unique(I))):
        xk = np.unique(np.concatenate([keys[rng.random(len(keys)) < 0.4], base + rng.integers(2000, 3000, 20), [-3, 5, 2 ** 63 - 1]]))
        xv = spread(rng, len(xk))
        names = _kernels_of(lambda: check(gm, om, xk, xv, trans, (base, trans)))
        assert not any(k in names for k in STREAMING_KERNELS), sorted(names)
        check(gm, om, keys, spread(rng, len(keys)), trans, (base, trans, "all"))


def test_full_size_config2_nx_1000():
    """bench.py's matrix at full size (1e5 x 1e5, 1e7 nnz): 1000 random present columns (rows), both orientations"""
    import bench as B
    _, coo, _, _ = B.make_workload(3)
    gm = D.dynamicsparse(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    om = O.Matrix(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    rng = np.random.default_rng(5100)
    for trans in (False, True):
        dim = B.M_ROWS if trans else B.N_COLS
        xk = np.sort(rng.choice(np.arange(1, dim + 1), 1000, replace=False))
        check(gm, om, xk, spread(rng, 1000), trans, ("config2", trans))


# ------------------------------------------------------------------------------------------- C ABI conventions
def _raw(gm, trans, xk, xv, cap, yk, yv):
    xk, xv = np.ascontiguousarray(xk, np.int64), np.ascontiguousarray(xv, np.float64)
    cnt = C.c_int64(-1)
    code = D.lib().dsa_matrix_spmspv(gm._h, C.c_int(trans), xk.ctypes.data_as(C.c_void_p), xv.ctypes.data_as(C.c_void_p),
                                     C.c_int64(len(xk)), None if yk is None else yk.ctypes.data_as(C.c_void_p),
                                     None if yv is None else yv.ctypes.data_as(C.c_void_p), C.c_int64(cap), C.byref(cnt))
    return code, cnt.value


def test_non_ascending_x_is_refused_and_nothing_is_written():
    gm, om, _ = _layout("bulk")
    SENT = -12345
    for keys in ([3, 3], [5, 9, 7], [2, 1]):
        yk, yv = np.full(1000, SENT, np.int64), np.full(1000, np.pi)
        with pytest.raises(D.ArgumentError, match="ascending"):
            gm.mul_sparse((np.array(keys), np.ones(len(keys))))
        code, _ = _raw(gm, 0, keys, np.ones(len(keys)), 1000, yk, yv)
        assert code == D._lib.DSA_ERR_ARGUMENT
        assert np.all(yk == SENT) and np.all(yv == np.pi)
    check(gm, om, [1, 2, 3], [1.0, 2.0, 3.0], False, "after a refusal")


def test_size_query_returns_the_count_and_writes_nothing():
    gm, om, _ = _layout("bulk")
    xk, xv = np.array([4, 9, 100]), np.array([1.0, -1.0, 2.0])
    want, _ = om.mul(xk, xv)
    assert len(want) > 1
    code, cnt = _raw(gm, 0, xk, xv, 0, None, None)
    assert code == 0 and cnt == len(want)
    yk, yv = np.full(len(want), GAP, np.int64), np.full(len(want), np.e)
    code, cnt = _raw(gm, 0, xk, xv, len(want) - 1, yk, yv)
    assert code == 0 and cnt == len(want) and np.all(yk == GAP) and np.all(yv == np.e)
    code, cnt = _raw(gm, 0, xk, xv, len(want), yk, yv)
    assert code == 0 and cnt == len(want) and np.array_equal(yk, want)


def test_device_pointers_on_a_torch_side_stream():
    import torch
    gm, om, _ = _layout("tile")
    rng = np.random.default_rng(5200)
    m, n = gm.size
    side = torch.cuda.Stream()
    for trans in (False, True):
        dim = m if trans else n
        xk = np.sort(rng.choice(np.arange(1, dim + 1), dim // 4, replace=False))
        xv = spread(rng, len(xk))
        with torch.cuda.stream(side):
            tk = torch.from_numpy(xk).cuda(non_blocking=True)
            tv = torch.from_numpy(xv).cuda(non_blocking=True) * 2.0     # queued on the side stream, not synchronised
            yk, yv = gm.mul_sparse((tk, tv), trans=trans)
            assert yk.is_cuda and yv.is_cuda and yk.dtype == torch.int64 and yv.dtype == torch.float64
            yk2, yv2 = yk + 0, yv * 1.0                                   # consumed on the same stream
        side.synchronize()
        assert_like_oracle((yk2.cpu().numpy(), yv2.cpu().numpy()), om, xk, xv * 2.0, trans, ("torch", trans))
    with pytest.raises(D.ArgumentError):
        gm.mul_sparse((torch.tensor([2, 1], device="cuda"), torch.ones(2, dtype=torch.float64, device="cuda")))


def test_device_entry_point_writes_nothing_on_refusal_or_small_cap():
    """dsa_matrix_spmspv_d: its fold writes straight into the caller's buffers, only when both are set and the count fits"""
    import torch
    gm, om, _ = _layout("bulk")
    L = D.lib()
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    xk, xv = np.array([4, 9, 100]), np.array([1.0, -1.0, 2.0])
    want_k, want_v = om.mul(xk, xv)
    n = len(want_k)
    assert n > 1

    def call(keys, vals, yk, yv, cap):
        tk, tv = torch.tensor(keys, dtype=torch.int64, device="cuda"), torch.tensor(vals, dtype=torch.float64, device="cuda")
        cnt = C.c_int64(-1)
        code = L.dsa_matrix_spmspv_d(gm._h, C.c_int(0), p(tk), p(tv), C.c_int64(len(keys)), p(yk), p(yv), C.c_int64(cap), C.byref(cnt))
        torch.cuda.synchronize()
        return code, cnt.value

    def sentinel():
        return torch.full((n + 8,), GAP, dtype=torch.int64, device="cuda"), torch.full((n + 8,), np.e, dtype=torch.float64, device="cuda")

    def untouched(yk, yv):
        return bool(torch.all(yk == GAP)) and bool(torch.all(yv == np.e))

    for keys in ([3, 3], [9, 4]):                                       # refused: nothing written
        yk, yv = sentinel()
        code, _ = call(keys, [1.0] * len(keys), yk, yv, n + 8)
        assert code == D._lib.DSA_ERR_ARGUMENT and untouched(yk, yv)
    yk, yv = sentinel()
    assert call(xk, xv, yk, yv, n - 1) == (0, n) and untouched(yk, yv)   # cap < count: the count only
    assert call(xk, xv, None, yv, n + 8) == (0, n) and untouched(yk, yv)  # a NULL output: nothing written
    assert call(xk, xv, yk, None, n + 8) == (0, n) and untouched(yk, yv)
    assert call(xk, xv, None, None, 0) == (0, n)                          # size query
    assert call(xk, xv, yk, yv, n) == (0, n)
    assert np.array_equal(yk[:n].cpu().numpy(), want_k) and np.array_equal(bits(yv[:n].cpu().numpy()), bits(want_v))
    assert bool(torch.all(yk[n:] == GAP)) and bool(torch.all(yv[n:] == np.e))


def test_torch_path_refuses_key_codecs():
    import torch
    gm = D.dynamicsparse([1, 2, 2], ['a', 'c', 'e'], [1.0, 2.0, 3.0], col_codec=D.CharCodec())
    with pytest.raises(D.ArgumentError, match="codec"):
        gm.mul_sparse((torch.tensor([97], device="cuda"), torch.ones(1, dtype=torch.float64, device="cuda")))
    y = gm.mul_sparse({'e': 2.0, 'a': 1.0})                               # the host forms encode and decode
    assert y.nzind.tolist() == [1, 2] and y.nzval.tolist() == [1.0, 6.0]
