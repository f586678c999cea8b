"""Sparse multi-vector product (dsa_matrix_spmspm[_d], DynamicSparseMatrix.mul_sparse with a matrix X) on the device.

Every column of every result is compared with the oracle's `mul` (mpcsc_mul, the reference's loop) on that column of X, keys
exactly and values as their 64-bit patterns (NaN by class), and with mul_sparse of that column (dsa_matrix_spmspv): the
product of k columns must be the k one-vector products, bit for bit."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import dsa_b200 as D
from oracle import oracle as O
from test_gpu_edge_values import GAP, bits, cancel_coo, paired, spread, _layout
from test_gpu_spmspv import STREAMING_KERNELS, assert_like_oracle

pytestmark = pytest.mark.gpu


def launches(fn):
    """kernel name -> launches of fn() (per-kernel event profile of the library)"""
    L = D.lib()
    L.dsa_prof_reset()
    L.dsa_prof_enable(C.c_int(1))
    try:
        fn()
    finally:
        L.dsa_prof_enable(C.c_int(0))
    L.dsa_prof_dump.restype = C.c_int64
    buf = C.create_string_buffer(int(L.dsa_prof_dump(None, C.c_int64(0))) + 16)
    L.dsa_prof_dump(buf, C.c_int64(len(buf)))
    L.dsa_prof_reset()
    return {ln.split(",")[0]: int(ln.split(",")[1]) for ln in buf.value.decode().strip().splitlines() if ln}


def raw(gm, trans, ptr, keys, vals, yp=None, yk=None, yv=None, cap=0):
    """dsa_matrix_spmspm with host buffers: (code, count)"""
    ptr, keys, vals = (np.ascontiguousarray(a, t) for a, t in ((ptr, np.int64), (keys, np.int64), (vals, np.float64)))
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    cnt = C.c_int64(-1)
    code = D.lib().dsa_matrix_spmspm(gm._h, C.c_int(trans), p(ptr), p(keys), p(vals), C.c_int64(len(ptr) - 1), C.c_int64(len(keys)),
                                     p(yp), p(yk), p(yv), C.c_int64(cap), C.byref(cnt))
    return code, cnt.value


def product(gm, trans, ptr, keys, vals):
    """(y_ptr, y_keys, y_vals) of the host entry point: size query, then the fill"""
    code, n = raw(gm, trans, ptr, keys, vals)
    assert code == 0, D.lib().dsa_last_error()
    yp, yk, yv = np.full(len(ptr), -1, np.int64), np.zeros(max(n, 1), np.int64), np.zeros(max(n, 1))
    code, n2 = raw(gm, trans, ptr, keys, vals, yp, yk, yv, n)
    assert code == 0 and n2 == n
    return yp, yk[:n], yv[:n]


def check_columns(gm, om, trans, ptr, keys, vals, what="", against_spmspv=True):
    """every column against the oracle's mul and against mul_sparse of that column, bit for bit"""
    yp, yk, yv = product(gm, trans, ptr, keys, vals)
    assert yp[0] == 0 and np.all(np.diff(yp) >= 0) and yp[-1] == len(yk), (what, "y_ptr")
    for c in range(len(ptr) - 1):
        xk, xv = np.asarray(keys[ptr[c]:ptr[c + 1]], np.int64), np.asarray(vals[ptr[c]:ptr[c + 1]], np.float64)
        col = (yk[yp[c]:yp[c + 1]], yv[yp[c]:yp[c + 1]])
        assert_like_oracle(col, om, xk, xv, trans, (what, trans, c))
        if against_spmspv:
            y1 = gm.mul_sparse((xk, xv), trans=trans)
            assert np.array_equal(col[0], y1.nzind) and np.array_equal(bits(col[1]), bits(np.asarray(y1.nzval))), (what, trans, c)
    return yp, yk, yv


def x_columns(rng, om, trans, dim, k=6):
    """CSC columns over the partition axis: subsets of the live partitions, an empty column, absent / deleted / negative /
    2^62-sized keys, IEEE specials, one column of everything"""
    e = om.export(1 if trans else 0)
    live = e["col_keys"][e["col_live"].astype(bool)]
    dead = np.setdiff1d(np.arange(1, dim + 1), live)
    extra = np.array([-(2 ** 63) + 1, -7, 0, dim + 1, 2 ** 62, 2 ** 63 - 1], np.int64)
    cols = []
    for _ in range(k):
        sub = np.sort(rng.choice(live, max(1, len(live) // 4), replace=False)) if len(live) else np.zeros(0, np.int64)
        cols.append((sub, spread(rng, len(sub))))
    cols.append((np.zeros(0, np.int64), np.zeros(0)))
    absent = np.unique(np.concatenate([live[:5], dead[:20], extra]))
    cols.append((absent, spread(rng, len(absent))))
    special = np.sort(rng.choice(live, min(len(live), 8), replace=False)) if len(live) else np.zeros(0, np.int64)
    cols.append((special, np.array([0.0, np.nan, np.inf, -np.inf, -0.0, 5e-324, 1e-310, -2.5])[:len(special)]))
    allk = np.arange(1, dim + 1)
    cols.append((allk, paired(rng, dim)))
    cols.append((np.zeros(0, np.int64), np.zeros(0)))                  # an empty last column
    ptr = np.concatenate([[0], np.cumsum([len(c[0]) for c in cols])]).astype(np.int64)
    return ptr, np.concatenate([c[0] for c in cols]).astype(np.int64), np.concatenate([c[1] for c in cols])


@pytest.mark.parametrize("name", ["bulk", "random_access", "tile", "deleted", "long", "short"])
def test_layouts_every_column_bit_for_bit(name):
    gm, om, _ = _layout(name)
    rng = np.random.default_rng(["bulk", "random_access", "tile", "deleted", "long", "short"].index(name) + 7100)
    m, n = gm.size
    for trans in (False, True):
        ptr, keys, vals = x_columns(rng, om, trans, m if trans else n)
        check_columns(gm, om, trans, ptr, keys, vals, name)
    ptr, keys, vals = x_columns(rng, om, False, n)
    counts = launches(lambda: product(gm, 0, ptr, keys, vals))
    assert "spmspv_emit" in counts and not any(k in counts for k in STREAMING_KERNELS), counts


@pytest.mark.parametrize("shape", [(3, 3, 4), (5, 7, 12), (12, 12, 60)])
def test_tiny_matrices(shape):
    m, n, nnz = shape
    rng = np.random.default_rng(nnz + 7200)
    I, J, V = cancel_coo(rng, m, n, nnz)
    gm, om = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    for trans in (False, True):
        ptr, keys, vals = x_columns(rng, om, trans, m if trans else n, k=3)
        check_columns(gm, om, trans, ptr, keys, vals, shape)


def test_empty_matrix_and_k_0_and_k_1():
    gm, om = D.dynamicsparse(fill_mode=False), O.Matrix(fill_mode=False)
    for trans in (False, True):
        yp, yk, _ = check_columns(gm, om, trans, np.array([0, 0, 3, 3]), np.array([1, 2, 3]), np.ones(3), "empty")
        assert yp.tolist() == [0, 0, 0, 0] and len(yk) == 0
    gm, om, _ = _layout("bulk")
    yp = np.full(1, -1, np.int64)
    assert raw(gm, 0, [0], [], [], yp, np.zeros(1, np.int64), np.zeros(1), 1) == (0, 0) and yp.tolist() == [0]   # k = 0
    for trans in (False, True):
        check_columns(gm, om, trans, np.array([0, 3]), np.array([2, 5, 9]), np.array([1.0, -2.0, 0.5]), "k = 1")


def test_keys_near_2_62_take_many_rounds():
    """in-array keys just below 2^62 take 62 bits of the 64-bit sort key: rounds of at most four columns"""
    base = (1 << 62) - 10_000
    rng = np.random.default_rng(7300)
    I, J, V = cancel_coo(rng, 800, 600, 12_000)
    I, J = I + base, J + base
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    for trans, keys in ((False, np.unique(J)), (True, np.unique(I))):
        cols = [np.sort(rng.choice(keys, 40, replace=False)) for _ in range(9)]
        cols[4:8] = [np.zeros(0, np.int64), np.array([-3, 5, 2 ** 63 - 1]), np.zeros(0, np.int64), np.array([7])]
        ptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int64)
        xk = np.concatenate(cols).astype(np.int64)
        xv = spread(rng, len(xk))
        counts = launches(lambda: check_columns(gm, om, trans, ptr, xk, xv, ("2^62", trans), against_spmspv=False))
        assert not any(k in counts for k in STREAMING_KERNELS), counts
        counts = launches(lambda: product(gm, int(trans), ptr, xk, xv))
        # two calls (query, fill) of three rounds: columns 0-3 and 8 fold, 4-7 (no products) only set their pointers
        assert counts["spmspv_fold"] == 2 * 2 and counts["spmspv_ptr_fill"] == 2, counts
        check_columns(gm, om, trans, ptr, xk, xv, ("2^62", trans))


def test_config2_above_the_round_budget():
    """bench.py's matrix at full size: a product of more than 2^27 products is cut into rounds by the budget"""
    import bench as B
    _, coo, _, _ = B.make_workload(3)
    gm = D.dynamicsparse(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    om = O.Matrix(coo[0], coo[1], coo[2], m=B.M_ROWS, n=B.N_COLS)
    rng = np.random.default_rng(7400)
    k, per = 64, 24_000                      # ~100 cells per column: 64 x 24 000 x 100 ~ 1.5e8 products
    cols = [np.sort(rng.choice(np.arange(1, B.N_COLS + 1), per, replace=False)) for _ in range(k)]
    ptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int64)
    xk, xv = np.concatenate(cols).astype(np.int64), spread(rng, k * per)
    yp, yk, yv = product(gm, 0, ptr, xk, xv)
    counts = launches(lambda: raw(gm, 0, ptr, xk, xv))
    assert counts["spmspv_fold"] >= 2, counts
    for c in rng.choice(k, 6, replace=False).tolist() + [0, k - 1]:       # a sample of columns, both ends of the rounds
        assert_like_oracle((yk[yp[c]:yp[c + 1]], yv[yp[c]:yp[c + 1]]), om, cols[c], xv[ptr[c]:ptr[c + 1]], False, ("config2", c))
    small = np.concatenate([[0], np.cumsum([200] * 8)]).astype(np.int64)
    check_columns(gm, om, True, small, np.concatenate([np.sort(rng.choice(B.M_ROWS, 200, replace=False)) + 1 for _ in range(8)]),
                  spread(rng, 1600), "config2 trans")


# ------------------------------------------------------------------------------------------- C ABI conventions
REFUSED = [  # (x_ptr, keys, k, nnz_x)
    ([0, 1], [1], -1, 1), ([0, 1], [1], 1, -1), ([1, 2], [1, 2], 1, 2), ([0, 2, 1], [1, 2], 2, 2), ([0, 2], [1, 2], 1, 3),
    ([0, 1, 2], [1, 2], 2, 1), ([0, 2], [3, 3], 1, 2), ([0, 3, 5], [1, 2, 2, 4, 6], 2, 5), ([0, 2, 4], [1, 2, 7, 5], 2, 4),
]


def test_refusals_write_nothing_host():
    gm, om, _ = _layout("bulk")
    for ptr, keys, k, nnz_x in REFUSED:
        yp, yk, yv = np.full(8, GAP, np.int64), np.full(100, GAP, np.int64), np.full(100, np.pi)
        pa, ka = np.asarray(ptr, np.int64), np.asarray(keys + [0] * 4, np.int64)
        cnt = C.c_int64(-1)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        code = D.lib().dsa_matrix_spmspm(gm._h, C.c_int(0), p(pa), p(ka), p(np.ones(len(ka))), C.c_int64(k), C.c_int64(nnz_x), p(yp),
                                         p(yk), p(yv), C.c_int64(100), C.byref(cnt))
        assert code == D._lib.DSA_ERR_ARGUMENT, (ptr, keys, k, nnz_x)
        assert np.all(yp == GAP) and np.all(yk == GAP) and np.all(yv == np.pi)
    check_columns(gm, om, False, np.array([0, 2, 3]), np.array([4, 9, 2]), np.ones(3), "after refusals")


def test_size_query_convention_host():
    gm, om, _ = _layout("bulk")
    ptr, keys, vals = np.array([0, 2, 3]), np.array([4, 9, 100]), np.array([1.0, -1.0, 2.0])
    code, n = raw(gm, 0, ptr, keys, vals)
    assert code == 0 and n > 1
    yp, yk, yv = np.full(3, GAP, np.int64), np.full(n, GAP, np.int64), np.full(n, np.e)
    assert raw(gm, 0, ptr, keys, vals, yp, yk, yv, n - 1) == (0, n)          # cap < count: the count only
    assert np.all(yp == GAP) and np.all(yk == GAP) and np.all(yv == np.e)
    assert raw(gm, 0, ptr, keys, vals, yp, None, None, n) == (0, n)          # y_ptr alone
    assert yp[-1] == n and np.all(yk == GAP)
    assert raw(gm, 0, ptr, keys, vals, yp, yk, yv, n) == (0, n)
    check_columns(gm, om, False, ptr, keys, vals, "size query")


def test_device_entry_point_refusals_and_size_query():
    """dsa_matrix_spmspm_d over sentinel-filled device buffers: a refusal writes nothing; cap < count writes only y_ptr"""
    import torch
    gm, om, _ = _layout("bulk")
    L = D.lib()
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731

    def call(ptr, keys, k, nnz_x, yp, yk, yv, cap):
        tp = torch.tensor(ptr, dtype=torch.int64, device="cuda")
        tk = torch.tensor(keys + [0], dtype=torch.int64, device="cuda")
        tv = torch.ones(len(keys) + 1, dtype=torch.float64, device="cuda")
        cnt = C.c_int64(-1)
        code = L.dsa_matrix_spmspm_d(gm._h, C.c_int(0), p(tp), p(tk), p(tv), C.c_int64(k), C.c_int64(nnz_x), p(yp), p(yk), p(yv),
                                     C.c_int64(cap), C.byref(cnt))
        torch.cuda.synchronize()
        return code, cnt.value

    def sentinel(n):
        return (torch.full((8,), GAP, dtype=torch.int64, device="cuda"), torch.full((n,), GAP, dtype=torch.int64, device="cuda"),
                torch.full((n,), np.e, dtype=torch.float64, device="cuda"))

    def untouched(*ts):
        return all(bool(torch.all(t == GAP)) if t.dtype == torch.int64 else bool(torch.all(t == np.e)) for t in ts)

    for ptr, keys, k, nnz_x in REFUSED:
        yp, yk, yv = sentinel(100)
        code, _ = call(ptr, keys, k, nnz_x, yp, yk, yv, 100)
        assert code == D._lib.DSA_ERR_ARGUMENT and untouched(yp, yk, yv), (ptr, keys, k, nnz_x)
    ptr, keys, vals = [0, 2, 3], [4, 9, 100], np.ones(3)
    yp_h, yk_h, yv_h = product(gm, 0, np.array(ptr), np.array(keys), vals)
    n = len(yk_h)
    yp, yk, yv = sentinel(n + 8)
    assert call(ptr, keys, 2, 3, None, None, None, 0) == (0, n)             # size query
    assert call(ptr, keys, 2, 3, yp, yk, yv, n - 1) == (0, n)               # one round: it does not fit, y_ptr is written
    assert untouched(yk, yv) and yp[:3].cpu().tolist() == yp_h.tolist() and untouched(yp[3:])
    assert call(ptr, keys, 2, 3, yp, None, yv, n + 8) == (0, n) and untouched(yk, yv)   # a NULL output: no keys, no values
    assert call(ptr, keys, 2, 3, yp, yk, yv, n) == (0, n)
    assert np.array_equal(yk[:n].cpu().numpy(), yk_h) and np.array_equal(bits(yv[:n].cpu().numpy()), bits(yv_h))
    assert untouched(yk[n:], yv[n:])
    yp1 = torch.full((1,), GAP, dtype=torch.int64, device="cuda")
    assert call([0], [], 0, 0, yp1, None, None, 0) == (0, 0) and yp1.item() == 0   # k = 0: y_ptr[0] = 0


def test_torch_csc_on_a_side_stream():
    import torch
    gm, om, _ = _layout("tile")
    rng = np.random.default_rng(7500)
    m, n = gm.size
    side = torch.cuda.Stream()
    for trans in (False, True):
        dim = m if trans else n
        X = sp.random(dim, 5, density=0.2, random_state=int(rng.integers(1 << 30)), format="csc")
        X.data[:] = spread(rng, X.nnz)
        X.sort_indices()
        with torch.cuda.stream(side):
            Xt = torch.sparse_csc_tensor(torch.from_numpy(X.indptr.astype(np.int64)), torch.from_numpy(X.indices.astype(np.int64)),
                                         torch.from_numpy(X.data), size=X.shape).cuda(non_blocking=True)
            Y = gm.mul_sparse(Xt, trans=trans)
            assert Y.layout == torch.sparse_csc and Y.shape == (n if trans else m, 5) and Y.values().dtype == torch.float64
            yp, yk, yv = (t.clone() for t in (Y.ccol_indices(), Y.row_indices(), Y.values()))
        side.synchronize()
        assert yp.dtype == torch.int64 and yk.dtype == torch.int64
        yp, yk, yv = yp.cpu().numpy(), yk.cpu().numpy() + 1, yv.cpu().numpy()
        for c in range(5):
            s = slice(X.indptr[c], X.indptr[c + 1])
            assert_like_oracle((yk[yp[c]:yp[c + 1]], yv[yp[c]:yp[c + 1]]), om, X.indices[s] + 1, X.data[s], trans, ("torch", trans, c))
    with pytest.raises(D.ArgumentError):      # rows out of order in a column
        gm.mul_sparse(torch.sparse_csc_tensor(torch.tensor([0, 2]), torch.tensor([3, 1]), torch.ones(2, dtype=torch.float64),
                                              size=(n, 1)).cuda())


def test_scipy_and_dynamic_matrix_operands():
    gm, om, _ = _layout("bulk")
    m, n = gm.size
    rng = np.random.default_rng(7600)
    I, J, V = cancel_coo(rng, n, 9, 400)
    B = D.dynamicsparse(I, J, V, m=n, n=9)
    Y, Yc = gm.mul_sparse(B), gm.mul_sparse(B.to_csc())
    assert Y.shape == (m, 9) and np.array_equal(Y.indptr, Yc.indptr) and np.array_equal(Y.indices, Yc.indices)
    assert np.array_equal(bits(Y.data), bits(Yc.data))
    X = B.to_csc()
    for c in range(9):
        s = slice(X.indptr[c], X.indptr[c + 1])
        assert_like_oracle((Y.indices[Y.indptr[c]:Y.indptr[c + 1]] + 1, Y.data[Y.indptr[c]:Y.indptr[c + 1]]), om, X.indices[s] + 1,
                           X.data[s], False, ("B", c))
    Yt = gm.mul_sparse(X.tocoo())
    assert np.array_equal(Yt.indptr, Y.indptr) and np.array_equal(bits(Yt.data), bits(Y.data))
    Z = gm.mul_sparse(sp.random(m, 4, density=0.05, random_state=1, format="csr"), trans=True)
    assert Z.shape == (n, 4)


def test_codec_refused_on_every_matrix_path():
    import torch
    gm = D.dynamicsparse([1, 2, 2], ['a', 'c', 'e'], [1.0, 2.0, 3.0], col_codec=D.CharCodec())
    B = D.dynamicsparse([1, 2], [1, 2], [1.0, 2.0], m=3, n=2)
    Xt = torch.sparse_csc_tensor(torch.tensor([0, 1]), torch.tensor([0]), torch.ones(1, dtype=torch.float64), size=(3, 1)).cuda()
    for X in (sp.eye(3, 2, format="csc"), B, Xt):
        with pytest.raises(D.ArgumentError, match="codec"):
            gm.mul_sparse(X)
