"""Edge values on the device, against the CPU oracle.

- Products (A·x, Aᵀ·x; dense x on the host and on the device, sparse x as a mask or by sorted-key lookup, k right-hand sides)
  against the exactly rounded sum of the oracle's own products: rows of one or two products must equal fl(p1 + p2), longer
  rows must meet the error bound of any summation order.  A fused multiply-add, a dropped or doubled term or a lost carry
  between 256-cell chunks fails these checks; a relative tolerance does not see them.
- NaN (with a payload too), ±Inf, -0.0, the smallest subnormal and DBL_MAX through every update pipeline: layouts and
  contents compared bit for bit (values as their 64-bit patterns, so NaN payloads and the sign of zero count).
- All six combine operators of the builders, with heavy duplication, NaN and ±0 among the duplicates.
- Keys at the ends of the Int64 range."""
import math

import numpy as np
import pytest

import dsa_b200 as D
from oracle import oracle as O
from test_gpu_parity import BIG_WINDOW_KERNELS, RESIZE_KERNELS, _kernels_of

pytestmark = pytest.mark.gpu

U = 2.0 ** -53                       # unit roundoff of Float64
CHUNK, LANE = 256, 8                 # cells per warp chunk and per lane of the SpMV kernels (pcsr.cuh SPMV_*)
GAP = -(1 << 63)                     # typemin(Int64): the gap sentinel of the device arrays (common.cuh GAP_KEY)
DBL_MAX = float(np.finfo(np.float64).max)
NAN_PAYLOAD = float(np.array([0x7FF8000000001234], np.int64).view(np.float64)[0])
SPECIALS = np.array([np.nan, NAN_PAYLOAD, np.inf, -np.inf, -0.0, 5e-324, DBL_MAX, -DBL_MAX])
# Base.min / Base.max on Float64 (known answers, both argument orders): NaN wins on either side, -0.0 orders below 0.0
MIN_MAX_KNOWN = [
    (O.COMB_MIN, 1.0, np.nan, np.nan), (O.COMB_MIN, np.nan, 1.0, np.nan),
    (O.COMB_MIN, 0.0, -0.0, -0.0), (O.COMB_MIN, -0.0, 0.0, -0.0),
    (O.COMB_MAX, -0.0, 0.0, 0.0), (O.COMB_MAX, 0.0, -0.0, 0.0),
    (O.COMB_MAX, 1.0, np.nan, np.nan), (O.COMB_MAX, np.nan, 1.0, np.nan),
    (O.COMB_MIN, -np.inf, NAN_PAYLOAD, NAN_PAYLOAD), (O.COMB_MAX, NAN_PAYLOAD, np.inf, NAN_PAYLOAD),
    (O.COMB_MIN, 2.0, -3.0, -3.0), (O.COMB_MAX, 2.0, -3.0, 2.0), (O.COMB_MIN, -np.inf, 5e-324, -np.inf),
    (O.COMB_MAX, -np.inf, 5e-324, 5e-324),
]
COMBINES = {"+": O.COMB_ADD, "*": O.COMB_MUL, "last": O.COMB_LAST, "first": O.COMB_FIRST, "min": O.COMB_MIN, "max": O.COMB_MAX}


# ------------------------------------------------------------------------------------------- bitwise comparisons
def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def assert_cells_bits(g_occ, g_key, g_val, o_tag, o_key, o_val):
    assert len(g_occ) == len(o_tag), "capacity differs"
    assert np.array_equal(g_occ, o_tag), "gap pattern differs"
    m = o_tag.astype(bool)
    assert np.array_equal(g_key[m], o_key[m]), "keys differ"
    assert np.array_equal(bits(g_val)[m], bits(o_val)[m]), "value bits differ"


def assert_vec_bits(gv, ov, layout=True):
    gi, oi = gv.info(), ov.info()
    for f in (("capacity", "segment_capacity", "nb_segments", "height") if layout else ()) + ("nnz", "n"):
        assert gi[f] == oi[f], (f, gi[f], oi[f])
    if layout:
        assert_cells_bits(*gv.export(), *ov.export())
    gk, gvals = gv.nonzeros()
    ok, ovals = ov.items()
    assert np.array_equal(gk, ok) and np.array_equal(bits(gvals), bits(ovals)), "nonzeros differ"


def assert_matrix_bits(gm, om, layout=True):
    """like test_gpu_parity.assert_matrix_equal, with values compared as bit patterns"""
    for which in (0, 1):
        ge, oe = gm.export(which), om.export(which)
        for f in ("nb_partitions", "nb_semaphores", "nnz", "m", "n"):
            assert ge[f] == oe[f], (which, f, ge[f], oe[f])
        assert ge["col_live"].tolist() == oe["col_live"].tolist()
        lv = oe["col_live"].astype(bool)
        assert np.array_equal(ge["col_keys"][lv], oe["col_keys"][lv])
        if layout:
            for f in ("capacity", "segment_capacity", "nb_segments", "nb_elements", "height"):
                assert ge[f] == oe[f], (which, f, ge[f], oe[f])
            assert_cells_bits(ge["tag"], ge["key"], ge["val"], oe["tag"], oe["key"], oe["val"])
            assert np.array_equal(ge["semaphores"][lv], oe["semaphores"][lv])
        else:
            mg, mo = ge["tag"].astype(bool), oe["tag"].astype(bool)
            assert np.array_equal(ge["key"][mg], oe["key"][mo])
            assert np.array_equal(bits(ge["val"][mg]), bits(oe["val"][mo])), (which, "value bits differ")


# ------------------------------------------------------------------------------------------- exact product reference
def stored_cells(om, which):
    """(partition key, cell key, value) of every stored cell of one orientation of the oracle, in layout order"""
    e = om.export(which)
    occ = np.nonzero(e["tag"])[0]
    key, val = e["key"][occ], e["val"][occ]
    sem = key == 0
    last = np.maximum.accumulate(np.where(sem, np.arange(len(occ)), -1))
    cell = ~sem & (last >= 0)
    part = val[last[cell]].astype(np.int64) - 1          # a semaphore's value is its partition id (pcsr.jl:40)
    live = e["col_live"][part].astype(bool)
    return e["col_keys"][part][live], key[cell][live], val[cell][live]


def exact_products(om, x, trans):
    """Per output key of mat * x (trans=False) or transpose(mat) * x, from the ORACLE's cells of the orientation the product
    reduces (row-major for A·x, column-major for Aᵀ·x): the products p = a * x (numpy rounds each multiply on its own) and
      S   = the correctly rounded exact sum (math.fsum), NaN for rows that are not `finite`,
      L   = the number of products, A = the sum of |p|,
      two = fl(p1 + p2) for L <= 2 (the value every summation order gives), NaN otherwise,
      finite = every product finite and no summation order can overflow,
      ambiguous = two or more huge finite products (|p| summing to >= 2^900 without the largest): whether a partial sum
                  overflows, and so which of NaN / ±Inf / finite the row comes out as, depends on the summation order.
    x is dense (x[key - 1]) or a pair (ascending keys, values): only the cells whose key x holds take part."""
    out, xkey, a = stored_cells(om, 0 if trans else 1)
    if isinstance(x, tuple):
        xk, xv = np.asarray(x[0], np.int64), np.asarray(x[1], np.float64)
        if len(xk) == 0:
            xk, xv = np.array([GAP], np.int64), np.zeros(1)
        pos = np.minimum(np.searchsorted(xk, xkey), len(xk) - 1)
        present, xval = xk[pos] == xkey, xv[pos]
    else:
        x = np.asarray(x, np.float64)
        present = (xkey >= 1) & (xkey <= len(x))
        xval = x[np.clip(xkey - 1, 0, max(len(x) - 1, 0))] if len(x) else np.zeros(len(xkey))
    with np.errstate(all="ignore"):
        p = a[present] * xval[present]
    out = out[present]
    order = np.argsort(out, kind="stable")
    out, p = out[order], p[order]
    keys, start, L = np.unique(out, return_index=True, return_counts=True)
    n = len(keys)
    S, two = np.full(n, np.nan), np.full(n, np.nan)
    with np.errstate(all="ignore"):
        A = np.add.reduceat(np.abs(p), start) if n else np.zeros(0)
        allfin = np.logical_and.reduceat(np.isfinite(p), start) if n else np.zeros(0, bool)
        one, pair = L == 1, L == 2
        two[one] = 0.0 + p[start[one]]
        two[pair] = p[start[pair]] + p[start[pair] + 1]
    finite = allfin & (L <= 2) & np.isfinite(two)          # one addition at most: no order to depend on
    S[finite] = two[finite]
    ambiguous = np.zeros(n, bool)
    for i in np.nonzero(L >= 3)[0]:
        g = p[start[i]:start[i] + L[i]]
        f = np.sort(np.abs(g[np.isfinite(g)]))
        try:
            if math.fsum(f[:-1]) >= 2.0 ** 900:            # two huge terms: a partial sum may overflow in some orders only
                ambiguous[i] = True
                continue
            if allfin[i]:
                A[i] = math.fsum(f)
                S[i] = math.fsum(g)
                finite[i] = True
        except OverflowError:
            ambiguous[i] = True
    return dict(keys=keys, S=S, L=L, A=A, two=two, finite=finite, ambiguous=ambiguous)


def check_rows(yv, ref, what=""):
    """yv aligned with ref["keys"]; the finite rows: L <= 2 exact (sign of a zero ignored), L >= 3 within the bound"""
    L, fin = ref["L"], ref["finite"]
    small = fin & (L <= 2)
    bad = np.nonzero(small & ~(yv == ref["two"]))[0]
    assert len(bad) == 0, (what, "rows of <= 2 products differ from fl(p1 + p2)", ref["keys"][bad[:5]], yv[bad[:5]], ref["two"][bad[:5]])
    big = fin & (L >= 3)
    err = np.abs(yv[big] - ref["S"][big])
    bound = 1.01 * L[big] * U * ref["A"][big]
    bad = np.nonzero(~(err <= bound))[0]
    assert len(bad) == 0, (what, "error bound exceeded", ref["keys"][big][bad[:5]], err[bad[:5]], bound[bad[:5]])


def assert_product(y, ref, what=""):
    """dense y (index key - 1): rows without a product exactly 0, the others as check_rows"""
    keys = ref["keys"]
    rest = np.ones(len(y), bool)
    rest[keys - 1] = False
    assert np.all(bits(y[rest]) == 0), (what, "a row without products is not +0.0", np.nonzero(bits(y) != 0)[0][:5])
    check_rows(y[keys - 1], ref, what)


def assert_classified_like(y, yo, ref, what=""):
    """y, yo aligned with ref["keys"]; rows whose products are not all finite: NaN / +Inf / -Inf exactly where the oracle's
    sequential sum has them.  Rows whose class depends on the summation order (`ambiguous`) are left out."""
    nf = ~ref["finite"] & ~ref["ambiguous"] & (ref["L"] > 0)
    for cls in (np.isnan, lambda v: v == np.inf, lambda v: v == -np.inf):
        assert np.array_equal(cls(y[nf]), cls(yo[nf])), (what, ref["keys"][nf][cls(y[nf]) != cls(yo[nf])][:5])


def chunk_coverage(e):
    """what the SpMV chunking meets in one orientation's layout (chunks of CHUNK cells, lanes of LANE cells)"""
    cap = len(e["tag"])
    occ = e["tag"].astype(bool)
    sem = np.nonzero(occ & (e["key"] == 0))[0]
    ends = np.append(sem[1:], cap) - 1
    used = np.cumsum(occ)
    cells = used[ends] - used[sem]                       # stored cells after each semaphore, up to the next one
    nchunks = (cap + CHUNK - 1) // CHUNK
    return dict(sem_at_chunk_start=int(np.sum(sem % CHUNK == 0)), sem_at_chunk_end=int(np.sum(sem % CHUNK == CHUNK - 1)),
                sem_at_lane_end=int(np.sum(sem % LANE == LANE - 1)),
                partition_over_3_chunks=int(np.sum(ends // CHUNK - sem // CHUNK + 1 >= 3)),
                chunk_without_sem=int(nchunks - len(np.unique(sem // CHUNK))), empty_partition=int(np.sum(cells == 0)),
                partial_single_chunk=int(cap < CHUNK))


def assert_chunk_coverage(exports, claims):
    tot = {}
    for e in exports:
        for k, v in chunk_coverage(e).items():
            tot[k] = tot.get(k, 0) + v
    missing = [c for c in claims if tot[c] == 0]
    assert not missing, (missing, tot)


# ------------------------------------------------------------------------------------------- data
def spread(rng, n):
    """random signs, magnitudes log-uniform over 1e-6 .. 1e6"""
    return rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-6, 6, n)


def paired(rng, n):
    """entries 2t and 2t+1 equal: the ±a pairs of cancel_coo cancel exactly in the products"""
    return np.repeat(spread(rng, (n + 1) // 2), 2)[:n]


def cancel_coo(rng, m, n, nnz):
    """spread values, plus rows (and columns) built to cancel: a and -a on two keys that x gives the same value, and a small
    remainder next to them"""
    I, J, V = [rng.integers(1, m + 1, nnz)], [rng.integers(1, n + 1, nnz)], [spread(rng, nnz)]
    k = max(nnz // 8, 2)
    r, c, a = rng.integers(1, m + 1, k), 2 * rng.integers(0, max(n // 2, 1), k) + 1, spread(rng, k)
    I += [r, r, r]
    J += [np.minimum(c, n), np.minimum(c + 1, n), rng.integers(1, n + 1, k)]
    V += [a, -a, a * 1e-7]
    c, r, b = rng.integers(1, n + 1, k), 2 * rng.integers(0, max(m // 2, 1), k) + 1, spread(rng, k)
    I += [np.minimum(r, m), np.minimum(r + 1, m), rng.integers(1, m + 1, k)]
    J += [c, c, c]
    V += [b, -b, b * 1e-7]
    return np.concatenate(I), np.concatenate(J), np.concatenate(V)


# ------------------------------------------------------------------------------------------- products
def _layout(name):
    """(device matrix, oracle matrix with the same layout, chunking cases the layout claims)"""
    rng = np.random.default_rng(["bulk", "random_access", "tile", "deleted", "long", "short"].index(name) + 4100)
    common = ("sem_at_chunk_start", "sem_at_chunk_end", "sem_at_lane_end")
    if name == "long":   # row 7 and column 5 hold 60 000 cells each: one partition over hundreds of chunks
        k = 60_000
        I0, J0, V0 = cancel_coo(rng, k, k, 4000)
        I = np.concatenate([I0, np.full(k, 7), np.arange(1, k + 1)])
        J = np.concatenate([J0, np.arange(1, k + 1), np.full(k, 5)])
        V = np.concatenate([V0, spread(rng, 2 * k)])
        gm, om = D.dynamicsparse(I, J, V, m=k, n=k), O.Matrix(I, J, V, m=k, n=k)
        return gm, om, ("partition_over_3_chunks", "chunk_without_sem") + common
    m, n, nnz = {"bulk": (700, 600, 25_000), "random_access": (400, 300, 8000), "tile": (400, 300, 12_000),
                 "deleted": (500, 400, 10_000), "short": (5000, 400, 6000)}[name]
    I, J, V = cancel_coo(rng, m, n, nnz)
    gm, om = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    if name in ("random_access", "tile"):
        prev = D.set_tile_mode(2 if name == "tile" else 0)
        try:
            for _ in range(3):
                nb = 3000
                grow = 0 if name == "tile" else 30       # the tile-streamed pipeline takes batches that create no row or column
                bi, bj = rng.integers(1, m + 1 + grow, nb), rng.integers(1, n + 1 + grow, nb)
                bv = np.where(rng.random(nb) < 0.3, 0.0, spread(rng, nb))
                names = _kernels_of(lambda: gm.set_batch(bi, bj, bv))
                om.set_batch_policy(bi, bj, bv)
                assert ("tile_merge" in names) == (name == "tile"), sorted(names)
        finally:
            D.set_tile_mode(prev)
        return gm, om, ("sem_at_chunk_start", "sem_at_lane_end")
    if name == "deleted":   # tombstoned slots in both orientations, and a live row and a live column left without entries
        cols, rows = np.unique(rng.integers(1, n + 1, 40)), np.unique(rng.integers(1, m + 1, 30))
        D.deletecolumn(gm, cols)
        om.delete_columns_policy(cols)
        D.deleterow(gm, rows)
        om.delete_rows_policy(rows)
        r = int(np.setdiff1d(np.arange(1, m + 1), rows)[0])
        c = int(np.setdiff1d(np.arange(1, n + 1), cols)[0])
        ks, _ = om.row(r)
        gm.set_batch(np.full(len(ks), r), ks, np.zeros(len(ks)))
        om.set_batch_policy(np.full(len(ks), r), ks, np.zeros(len(ks)))
        ks, _ = om.column(c)
        gm.set_batch(ks, np.full(len(ks), c), np.zeros(len(ks)))
        om.set_batch_policy(ks, np.full(len(ks), c), np.zeros(len(ks)))
        return gm, om, ("empty_partition",) + common
    return gm, om, common


def _sparse_x(rng, x, frac):
    keys = np.nonzero(rng.random(len(x)) < frac)[0] + 1
    return keys, x[keys - 1]


def _check_sparse(gm, om, xk, xv, trans, what):
    y = (gm.T if trans else gm) @ (xk, xv)
    yk, _ = om.mul(xk, xv, trans=trans)
    ref = exact_products(om, (xk, xv), trans)
    assert np.array_equal(y.nzind, yk), (what, "touched rows differ from the oracle's")
    assert np.array_equal(ref["keys"], yk)
    check_rows(np.asarray(y.nzval), ref, what)
    return ref


def _check_all_entry_points(gm, om, rng):
    import torch
    m, n = gm.size
    for trans in (False, True):
        nx = m if trans else n
        x = paired(rng, nx)
        ref = exact_products(om, x, trans)
        assert_product(gm.mul_dense(x, trans=trans), ref, ("host x", trans))
        yd = gm.mul_dense(torch.from_numpy(x).cuda(), trans=trans)
        torch.cuda.synchronize()
        assert_product(yd.cpu().numpy(), ref, ("device x", trans))
        for frac in (0.3, 0.9):   # sparse x, as a mask over a dense buffer (small key space); x may come out empty
            xk, xv = _sparse_x(rng, x, frac)
            names = _kernels_of(lambda: _check_sparse(gm, om, xk, xv, trans, ("sparse x", trans, frac)))
            assert ("scatter_x" in names) == (len(xk) > 0), sorted(names)
        for k in (1, 4, 33):
            X = np.stack([paired(rng, nx) for _ in range(k)], axis=1)
            Y = gm.mul_dense(X, trans=trans)
            for c in range(k):
                assert_product(Y[:, c], exact_products(om, X[:, c], trans), ("X", trans, k, c))


@pytest.mark.parametrize("name", ["bulk", "random_access", "tile", "deleted", "long", "short"])
def test_products_against_exact_sums(name):
    gm, om, claims = _layout(name)
    assert_matrix_bits(gm, om)       # the reference products are formed from the oracle's layout: it must be the device's
    assert_chunk_coverage([om.export(0), om.export(1)], claims)
    rng = np.random.default_rng(7)
    if name == "short":              # rows of one and two products are common: the exact check carries most of the weight
        ref = exact_products(om, paired(rng, gm.size[1]), False)
        assert np.sum(ref["L"] <= 2) >= 2000, np.bincount(ref["L"])[:4]
    _check_all_entry_points(gm, om, rng)


@pytest.mark.parametrize("shape", [(3, 3, 4), (5, 7, 12), (9, 6, 30), (12, 12, 60)])
def test_products_on_tiny_matrices(shape):
    m, n, nnz = shape
    rng = np.random.default_rng(nnz)
    I, J, V = cancel_coo(rng, m, n, nnz)
    gm, om = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    assert_matrix_bits(gm, om)
    caps = [om.info(w)["capacity"] for w in (0, 1)]
    assert all(16 <= c <= 128 for c in caps), caps
    assert_chunk_coverage([om.export(0), om.export(1)], ("partial_single_chunk",))
    _check_all_entry_points(gm, om, rng)


def test_sparse_products_by_sorted_key_lookup():
    """keys above 2^26 on both axes: x stays a sorted list and every cell looks its key up (libdsa.cu dsa_matrix_spmv)"""
    rng = np.random.default_rng(4200)
    base = 1 << 27
    I, J, V = cancel_coo(rng, 800, 600, 12_000)
    I, J = I + base, J + base
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    assert_matrix_bits(gm, om)
    pairs = spread(rng, 1500)
    for trans, keys in ((False, np.unique(J)), (True, np.unique(I))):
        for frac in (0.3, 1.0):
            xk = np.unique(np.concatenate([keys[rng.random(len(keys)) < frac], base + rng.integers(2000, 3000, 20)]))
            xv = pairs[(xk - base - 1) // 2]             # keys base + 2t + 1 and base + 2t + 2 share a value: the ±a pairs cancel
            names = _kernels_of(lambda: _check_sparse(gm, om, xk, xv, trans, ("lookup", trans, frac)))
            assert "scatter_x" not in names and "spmv_blocked" in names, sorted(names)


# ------------------------------------------------------------------------------------------- IEEE special values
def _special_products(gm, om, rng, what):
    """dense x (finite, magnitudes up to 1e6), and sparse x with an Inf on the key of a stored 0 that leaves out the keys of
    the stored Infs"""
    m, n = gm.size
    for trans in (False, True):
        nx, ny = (m, n) if trans else (n, m)
        x = spread(rng, nx)
        ref = exact_products(om, x, trans)
        y, yo = gm.mul_dense(x, trans=trans), om.mul_dense(x, ny, trans=trans)
        assert_classified_like(y[ref["keys"] - 1], yo[ref["keys"] - 1], ref, (what, "dense", trans))
        assert_product(y, ref, (what, "dense", trans))
        part, key, val = stored_cells(om, 0 if trans else 1)
        zero_key = int(key[val == 0.0][0])
        inf_keys = np.unique(key[np.isinf(val)])
        xk, xv = _sparse_x(rng, x, 0.5)
        xk = np.union1d(xk[~np.isin(xk, inf_keys)], [zero_key])
        xv = np.where(xk == zero_key, np.inf, spread(rng, len(xk)))
        y = (gm.T if trans else gm) @ (xk, xv)
        yk, yo = om.mul(xk, xv, trans=trans)
        assert np.array_equal(y.nzind, yk), (what, "sparse", trans)
        ref = exact_products(om, (xk, xv), trans)
        yv = np.asarray(y.nzval)
        assert_classified_like(yv, yo, ref, (what, "sparse", trans))
        check_rows(yv, ref, (what, "sparse", trans))
        nan_rows = np.unique(part[(key == zero_key) & (val == 0.0)])      # Inf * stored 0 = NaN on the row that holds the 0
        assert np.all(np.isin(nan_rows, y.nzind)) and np.all(np.isnan(yv[np.searchsorted(y.nzind, nan_rows)])), (what, trans)
        inf_rows = np.unique(part[np.isin(key, inf_keys)])               # a stored Inf that x leaves out touches nothing:
        i = np.searchsorted(ref["keys"], inf_rows)                       # rows whose present products are finite come out finite
        quiet = (i >= len(ref["keys"])) | ~np.isin(inf_rows, ref["keys"]) | ref["finite"][np.minimum(i, len(ref["keys"]) - 1)]
        # this only asserts that the data holds the case; what the device made of it is checked by the nzind equality and
        # check_rows above (a touched row whose present products are finite must meet the bound, so it is finite)
        assert quiet.any(), (what, trans, "no row shows the case")


def _check_matrix_step(gm, pol, seq, rng, what, cells=None):
    assert_matrix_bits(gm, pol)                      # layout: the batch policy
    assert_matrix_bits(gm, seq, layout=False)        # contents: the sequential setindex! loop
    assert gm.size == seq.size, (what, gm.size, seq.size)
    m, n = gm.size
    rq, cq = rng.integers(1, m + 2, 2000), rng.integers(1, n + 2, 2000)
    if cells is not None:
        rq, cq = np.concatenate([rq, cells[0]]), np.concatenate([cq, cells[1]])
    for which in (0, 1):
        assert np.array_equal(bits(gm.get_batch(rq, cq, which=which)), bits(seq.get_many(rq, cq, which=which))), (what, which)
        # typemin(Int64) is the gap key: a lookup of it finds nothing, never a gap cell
        g = gm.get_batch([GAP, int(rq[0]), GAP], [int(cq[0]), GAP, GAP], which=which)
        assert np.all(bits(g) == 0), (what, which, g)
    ec = seq.export(0)
    live_c = ec["col_keys"][ec["col_live"].astype(bool)]
    er = seq.export(1)
    live_r = er["col_keys"][er["col_live"].astype(bool)]
    for c in rng.choice(live_c, min(8, len(live_c)), replace=False):
        gk, gv = gm.col(int(c))
        ok, ov = seq.column(int(c))
        assert np.array_equal(gk, ok) and np.array_equal(bits(gv), bits(ov)), (what, "col", c)
    for r in rng.choice(live_r, min(8, len(live_r)), replace=False):
        gk, gv = gm.row(int(r))
        ok, ov = seq.row(int(r))
        assert np.array_equal(gk, ok) and np.array_equal(bits(gv), bits(ov)), (what, "row", r)
    _special_products(gm, pol, rng, what)


def _with_specials(rng, nb, p=0.15):
    v = spread(rng, nb)
    pick = rng.random(nb) < p
    v[pick] = rng.choice(SPECIALS, int(pick.sum()))
    return v


def test_vector_special_values():
    rng = np.random.default_rng(4300)
    keys = np.unique(rng.integers(1, 30_000, 3000))
    vals = spread(rng, len(keys))
    vals[:: len(keys) // len(SPECIALS)][: len(SPECIALS)] = SPECIALS
    neg0 = int(keys[np.nonzero(bits(vals) == bits(-0.0))[0][0]])
    gv, pol, seq = D.dynamicsparsevec(keys, vals), O.Vec(keys, vals), O.Vec(keys, vals)
    assert_vec_bits(gv, pol)
    assert bits(gv.get_batch([neg0]))[0] == bits(-0.0), "a -0.0 in a build is stored with its sign"
    for rnd in range(5):
        nb = int(rng.integers(200, 4000))
        k = np.concatenate([rng.integers(1, 30_000, nb), rng.choice(keys, 300)])
        v = _with_specials(rng, len(k))
        v[-300::3] = -0.0                                   # -0.0 writes on stored keys: deletes, like 0.0
        k = np.append(k, [30_000 + 1000 * rnd + 7, 30_000 + 1000 * rnd + 9])   # NaN and Inf writes grow n
        v = np.append(v, [np.nan, -np.inf])
        n_before = len(gv)
        gv.set_batch(k, v)
        pol.set_batch_policy(k, v)
        seq.set_many(k, v)
        assert_vec_bits(gv, pol)
        assert_vec_bits(gv, seq, layout=False)
        assert len(gv) == len(seq) and len(gv) >= max(n_before, int(k[-1]))
        last = dict(zip(k.tolist(), v.tolist()))
        deleted = [kk for kk, vv in last.items() if vv == 0.0]
        assert not np.isin(deleted, gv.nonzeros()[0]).any(), "a -0.0 write must delete"
        q = np.concatenate([k, rng.integers(1, 40_000, 500)])
        assert np.array_equal(bits(gv.get_batch(q)), bits(seq.get_many(q)))
        assert bits(gv.get_batch([GAP]))[0] == 0
    for t in range(60):   # single writes: a batch of one is the reference's own setindex!
        kk, vv = int(rng.integers(1, 31_000)), float(rng.choice(np.append(SPECIALS, [1.5, 0.0])))
        gv.set_batch([kk], [vv])
        seq[kk] = vv
        pol.set_batch_policy([kk], [vv])
        if t % 10 == 9:
            assert_vec_bits(gv, pol)
            assert_vec_bits(gv, seq, layout=False)


def test_matrix_special_values_through_every_pipeline():
    rng = np.random.default_rng(4400)
    m, n, nnz = 300, 200, 6000
    lin = rng.choice(m * n, nnz, replace=False)     # no duplicates: the build only moves the special values
    I, J, V = lin // n + 1, lin % n + 1, spread(rng, nnz)
    # at most one special value per row and per column: whether a product's partial sums overflow cannot depend on the order
    sp = rng.permutation(nnz)[:40]
    sp = sp[np.unique(I[sp], return_index=True)[1]]
    sp = sp[np.unique(J[sp], return_index=True)[1]]
    V[sp] = np.resize(SPECIALS, len(sp))
    z = rng.permutation(np.setdiff1d(np.arange(nnz), sp))[:20]
    V[z] = np.where(np.arange(20) % 2, 0.0, -0.0)   # stored zeros of both signs
    gm, pol, seq = D.dynamicsparse(I, J, V), O.Matrix(I, J, V), O.Matrix(I, J, V)
    _check_matrix_step(gm, pol, seq, rng, "build")
    nz = z[np.arange(20) % 2 == 0][0]
    assert bits(gm.get_batch([I[nz]], [J[nz]]))[0] == bits(-0.0), "a -0.0 in a build is stored with its sign"

    def step(what, bi, bj, bv, mode=0, expect=(), single=False):
        prev = D.set_tile_mode(mode)
        try:
            if single:
                names = set()
                for a, b, c in zip(bi.tolist(), bj.tolist(), bv.tolist()):
                    names |= _kernels_of(lambda: gm.set_batch([a], [b], [c]))
            else:
                names = _kernels_of(lambda: gm.set_batch(bi, bj, bv))
        finally:
            D.set_tile_mode(prev)
        if single:
            for a, b, c in zip(bi.tolist(), bj.tolist(), bv.tolist()):
                pol.set_batch_policy([a], [b], [c])
        else:
            pol.set_batch_policy(bi, bj, bv)
        seq.set_many(bi, bj, bv)
        for e in expect:
            assert e <= names if isinstance(e, set) else e in names, (what, sorted(names))
        _check_matrix_step(gm, pol, seq, rng, what, (bi, bj))

    # bucket path: every column exists and receives few ops; -0.0 on stored cells deletes them
    bi, bj = rng.integers(1, m + 1, 1500), rng.integers(1, n + 1, 1500)
    ec, er, _ = stored_cells(seq, 0)
    pick = rng.choice(len(er), 200, replace=False)
    er, ec = er[pick], ec[pick]
    bi, bj = np.concatenate([bi, er]), np.concatenate([bj, ec])
    bv = _with_specials(rng, len(bi))
    bv[-200:] = -0.0
    step("bucket", bi, bj, bv, expect=("bucket_rank_locate",))
    assert np.all(bits(gm.get_batch(er, ec)) == 0), "-0.0 writes delete"
    # radix path: a new column and a hot column of more than 256 ops; NaN / Inf writes on new keys grow m and n
    bi = np.concatenate([rng.integers(1, m + 1, 600), rng.integers(1, m + 1, 50), [m + 3, 2]])
    bj = np.concatenate([np.full(600, 7), np.full(50, n + 5), [3, n + 9]])
    bv = np.concatenate([_with_specials(rng, 650), [np.nan, -np.inf]])
    step("radix", bi, bj, bv, expect=("make_sortkeys",))
    assert gm.size == (m + 3, n + 9), gm.size
    newcol = n + 5
    m, n = gm.size
    # tile-streamed: existing rows and columns only
    bi, bj = rng.integers(1, 300, 2500), rng.integers(1, 200, 2500)
    step("tile", bi, bj, _with_specials(rng, 2500), mode=2, expect=("tile_merge",))
    # single writes
    bi, bj = rng.integers(1, m + 1, 40), rng.integers(1, n + 1, 40)
    step("single", bi, bj, _with_specials(rng, 40, p=0.6), single=True)
    # enough new cells to resize both orientations
    nb = 60_000
    step("resize", rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb), _with_specials(rng, nb, p=0.01), expect=(RESIZE_KERNELS,))
    # a run of consecutive row keys in one column that no window of SMALL_CELLS cells holds (the column-major orientation
    # keeps its capacity; the new rows resize the row-major one)
    cap = gm.info(0)["capacity"]
    step("big window", 20 + np.arange(3000), np.full(3000, 11), _with_specials(rng, 3000), expect=(BIG_WINDOW_KERNELS,))
    assert gm.info(0)["capacity"] == cap
    # deletecolumn! of columns that hold special values
    part, _, val = stored_cells(seq, 0)
    cols = np.unique(np.concatenate([part[np.isnan(val)][:1], part[np.isinf(val)][:1], [7, 11, newcol]]))
    D.deletecolumn(gm, cols)
    pol.delete_columns_policy(cols)
    for c in cols:
        seq.deletecolumn(int(c))
    _check_matrix_step(gm, pol, seq, rng, "deletecolumn")


# ------------------------------------------------------------------------------------------- combine operators
def _dup_values(rng, keys):
    """keys 1..20 draw among the special values too, 21..40 mostly ±0 among spread values, 41..45 only ±0, 46..50 ±0 among
    positive values (min ends on a zero), 51..55 ±0 among negative values (max ends on a zero), the rest finite"""
    v = spread(rng, len(keys))
    a = keys <= 20
    pick = a & (rng.random(len(keys)) < 0.004)
    v[pick] = rng.choice(SPECIALS, int(pick.sum()))
    v[(keys > 45) & (keys <= 50)] = np.abs(v[(keys > 45) & (keys <= 50)])
    v[(keys > 50) & (keys <= 55)] = -np.abs(v[(keys > 50) & (keys <= 55)])
    mixed = ((keys > 20) & (keys <= 40)) | ((keys > 45) & (keys <= 55))
    zb = (mixed & (rng.random(len(keys)) < 0.8)) | ((keys > 40) & (keys <= 45))
    v[zb] = np.where(rng.random(int(zb.sum())) < 0.5, 0.0, -0.0)
    return v


def _assert_zero_sign_decided(comb, cells, vals, got):
    """min / max: cells whose duplicates hold both +0.0 and -0.0 and whose result is a zero must hold -0.0 (min) or +0.0
    (max), Base.min / Base.max's order of the zeros; at least one such cell must exist.  cells: one int64 key per input
    entry; got(unique cells) -> the stored values."""
    u, inv = np.unique(cells, return_inverse=True)
    pos = np.bincount(inv, bits(vals) == bits(0.0), len(u)) > 0
    neg = np.bincount(inv, bits(vals) == bits(-0.0), len(u)) > 0
    cand = u[pos & neg]
    y = got(cand)
    decided = y == 0.0
    assert decided.sum() >= 1, (comb, "no cell where the sign of a zero result is decided")
    want = bits(-0.0 if comb == "min" else 0.0)[0]
    assert np.all(bits(y[decided]) == want), (comb, cand[decided][bits(y[decided]) != want][:5])


@pytest.mark.parametrize("comb", list(COMBINES))
def test_all_combine_operators_bit_exact(comb):
    """heavy duplication spread over the whole input (over many radix tiles): the left fold in input order depends on the sort
    being stable"""
    rng = np.random.default_rng(4500 + list(COMBINES).index(comb))
    nb = 40_000
    keys = rng.integers(1, 61, nb)
    vals = _dup_values(rng, keys)
    gv, ov = D.dynamicsparsevec(keys, vals, combine=comb), O.Vec(keys, vals, combine=COMBINES[comb])
    assert_vec_bits(gv, ov)
    part = rng.integers(1, 11, nb)                 # 10 columns; row keys 1..60 carry the value classes above
    gm, om = D.dynamicsparse(keys, part, vals, combine=comb), O.Matrix(keys, part, vals, combine=COMBINES[comb])
    assert_matrix_bits(gm, om)
    gm2, om2 = D.dynamicsparse(part, keys, vals, combine=comb), O.Matrix(part, keys, vals, combine=COMBINES[comb])
    assert_matrix_bits(gm2, om2)
    if comb in ("min", "max"):
        _assert_zero_sign_decided(comb, keys, vals, gv.get_batch)
        _assert_zero_sign_decided(comb, keys * 16 + part, vals, lambda c: gm.get_batch(c // 16, c % 16))
        _assert_zero_sign_decided(comb, part * 64 + keys, vals, lambda c: gm2.get_batch(c // 64, c % 64, which=1))


def test_min_max_known_answers_on_the_device():
    """Base.min / Base.max of two duplicates, in both orders: NaN wins on either side (the NaN argument itself), -0.0 orders
    below 0.0 — the vector builder and both orientations of the matrix builder"""
    for comb, a, b, expect in MIN_MAX_KNOWN:
        name = "min" if comb == O.COMB_MIN else "max"
        v = D.dynamicsparsevec([3, 3], [a, b], combine=name)
        assert bits(v.get_batch([3]))[0] == bits(expect)[0], (name, a, b, expect)
        m = D.dynamicsparse([3, 3], [2, 2], [a, b], combine=name)
        for which in (0, 1):
            assert bits(m.get_batch([3], [2], which=which))[0] == bits(expect)[0], (name, a, b, expect, which)


# ------------------------------------------------------------------------------------------- extreme keys
EXTREME = np.array([-(2 ** 63) + 1, -5, 0, 1, 2 ** 63 - 1], np.int64)


def _full_span(rng, n):
    return rng.integers(-(2 ** 63) + 1, 2 ** 63 - 1, n, dtype=np.int64)


def test_vector_keys_over_the_whole_int64_range():
    rng = np.random.default_rng(4600)
    keys = np.concatenate([EXTREME, _full_span(rng, 3000)])
    vals = spread(rng, len(keys))
    gv, pol, seq = D.dynamicsparsevec(keys, vals), O.Vec(keys, vals), O.Vec(keys, vals)
    assert_vec_bits(gv, pol)
    assert len(gv) == len(seq)
    live = keys.copy()
    for rnd in range(5):
        nb = int(rng.integers(100, 3000))
        k = np.concatenate([EXTREME, _full_span(rng, nb), rng.choice(live, 200)])
        v = np.where(rng.random(len(k)) < 0.3, 0.0, spread(rng, len(k)))
        gv.set_batch(k, v)
        pol.set_batch_policy(k, v)
        seq.set_many(k, v)
        live = np.concatenate([live, k])
        assert_vec_bits(gv, pol)
        assert_vec_bits(gv, seq, layout=False)
        assert len(gv) == len(seq)
        q = np.concatenate([EXTREME, k, _full_span(rng, 300)])
        assert np.array_equal(bits(gv.get_batch(q)), bits(seq.get_many(q)))
        assert bits(gv.get_batch([GAP]))[0] == 0
    neg = -np.unique(rng.integers(1, 1 << 62, 500))      # every key negative: shrink_size! (vector.jl:64)
    v = spread(rng, len(neg))
    gv, seq = D.dynamicsparsevec(neg, v), O.Vec(neg, v)
    assert len(gv) == len(seq)
    assert D.shrink_size(gv) == seq.shrink_size()
    assert len(gv) == len(seq)
    assert_vec_bits(gv, seq)


def _near_2_62(rng, nnz, high):
    base = 1 << 62
    hi, lo = base + rng.integers(0, 5001, nnz), rng.integers(1, 3001, nnz)
    return (hi, lo) if high == "rows" else (lo, hi)


@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("high", ["rows", "cols"])
def test_matrix_keys_near_2_62(high, mode):
    """row (or column) keys in [2^62, 2^62 + 5000], 3000 partitions on the other axis: the batch radix path packs the key
    range, not the largest key, next to the partition bits"""
    rng = np.random.default_rng(4700 + 2 * mode + (high == "cols"))
    I, J = _near_2_62(rng, 20_000, high)
    V = spread(rng, len(I))
    gm, pol, seq = D.dynamicsparse(I, J, V), O.Matrix(I, J, V), O.Matrix(I, J, V)
    assert_matrix_bits(gm, pol)
    hot_axis = J if high == "rows" else I

    def step(what, bi, bj, bv, expect):
        prev = D.set_tile_mode(mode)
        try:
            names = _kernels_of(lambda: gm.set_batch(bi, bj, bv))
        finally:
            D.set_tile_mode(prev)
        pol.set_batch_policy(bi, bj, bv)
        seq.set_many(bi, bj, bv)
        assert expect & names, (what, sorted(names))
        assert_matrix_bits(gm, pol)
        assert_matrix_bits(gm, seq, layout=False)
        q = rng.integers(0, len(I), 1000)
        rq, cq = np.concatenate([I[q], bi]), np.concatenate([J[q], bj])
        assert np.array_equal(bits(gm.get_batch(rq, cq)), bits(seq.get_many(rq, cq)))

    pick = rng.integers(0, len(I), 1500)          # spread over existing cells: few ops per partition
    step("spread", I[pick], J[pick], spread(rng, 1500), {"bucket_rank_locate", "tile_merge"})
    hot = int(hot_axis[0])
    pick = rng.integers(0, len(I), 700)
    bi, bj = (I[pick], np.full(700, hot)) if high == "rows" else (np.full(700, hot), J[pick])
    step("hot", bi, bj, spread(rng, 700), {"make_sortkeys", "tile_merge"})
    new = (1 << 62) + 6000 + np.arange(40)          # new partitions on the high axis, and new cells of existing ones
    pick = rng.integers(0, len(I), 400)
    if high == "rows":
        bi, bj = np.concatenate([new, I[pick]]), np.concatenate([J[:40], 3001 + np.arange(400) % 17])
    else:
        bi, bj = np.concatenate([I[:40], 3001 + np.arange(400) % 17]), np.concatenate([new, J[pick]])
    step("creating", bi, bj, spread(rng, 440), {"make_sortkeys"})


def test_documented_refusals_leave_the_structure_unchanged():
    rng = np.random.default_rng(4800)
    with pytest.raises(D.ArgumentError):
        D.dynamicsparse([1, 0], [1, 1], [1.0, 2.0])                   # key 0 is the semaphore key
    with pytest.raises(D.ArgumentError):
        D.dynamicsparse([1, 1 << 62], [1, 1 << 62], [1.0, 2.0])       # 62 + 62 bits of key ranges do not fit one sort key
    I, J = np.array([1, 1 << 62, 5, 9]), np.array([1, 2, 3, 2])
    V = spread(rng, 4)
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    before = [gm.export(w) for w in (0, 1)]

    def unchanged():
        for w in (0, 1):
            after = gm.export(w)
            for f in ("tag", "key", "val", "semaphores", "col_keys", "col_live"):
                assert np.array_equal(bits(after[f]) if f == "val" else after[f], bits(before[w][f]) if f == "val" else before[w][f]), f
        assert gm.size == om.size

    for bi, bj in (([3, 0], [1, 2]), ([3, 4], [1, 0])):
        with pytest.raises(D.ArgumentError):
            gm.set_batch(bi, bj, [1.0, 2.0])
        unchanged()
    # a new column whose rows span [1, 2^62]: 63 bits of key range + 3 bits of partitions (3 slots + 2 ops counted as absent)
    with pytest.raises(D.ArgumentError):
        gm.set_batch([1, 1 << 62], [10, 10], [1.0, 2.0])
    unchanged()
    gm.set_batch([2, 3], [10, 10], [1.0, 2.0])                        # a narrow one goes through
    om.set_batch_policy([2, 3], [10, 10], [1.0, 2.0])
    assert_matrix_bits(gm, om)
