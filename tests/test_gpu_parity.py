"""GPU parity tests: the CUDA path (through the C ABI, via the Python mirror of the reference API) against the CPU oracle
on the same seeded inputs.  Bit-exact for keys / values / layout / column structure; SpMV within 1e-12 relative."""
import copy

import numpy as np
import pytest

import dsa_b200 as D
from oracle import oracle as O

pytestmark = pytest.mark.gpu

SPMV_RTOL = 1e-12   # BASELINE.json north_star: "floating-point SpMV outputs within 1e-12 relative (Float64)"
# launch names of the rebalance tiers that ordinary batches rarely reach: windows above SMALL_CELLS cells, and a resize
BIG_WINDOW_KERNELS = {"merge_scatter_big", "scatter_inserts_big", "copyback_big"}
RESIZE_KERNELS = {"merge_scatter_root", "scatter_inserts_root"}


def _kernels_of(fn):
    """names of the kernels fn() launches (per-kernel event profile of the library)"""
    import ctypes as C
    L = D.lib()
    L.dsa_prof_reset()
    L.dsa_prof_enable(C.c_int(1))
    try:
        fn()
    finally:
        L.dsa_prof_enable(C.c_int(0))
    L.dsa_prof_dump.restype = C.c_int64
    need = L.dsa_prof_dump(None, C.c_int64(0))
    buf = C.create_string_buffer(int(need) + 16)
    L.dsa_prof_dump(buf, C.c_int64(len(buf)))
    L.dsa_prof_reset()
    return {ln.split(",")[0] for ln in buf.value.decode().strip().splitlines() if ln}


def assert_layout_equal(g_occ, g_key, g_val, o_tag, o_key, o_val):
    assert len(g_occ) == len(o_tag), "capacity differs"
    assert np.array_equal(g_occ, o_tag), "gap pattern differs"
    m = o_tag.astype(bool)
    assert np.array_equal(g_key[m], o_key[m])
    assert np.array_equal(g_val[m], o_val[m])


def assert_vec_equal(gv, ov, layout=True):
    gi, oi = gv.info(), ov.info()
    for f in ("capacity", "segment_capacity", "nb_segments", "nnz", "height", "n"):
        assert gi[f] == oi[f], (f, gi[f], oi[f])
    if layout:
        assert_layout_equal(*gv.export(), *ov.export())


def assert_matrix_equal(gm, om, layout=True):
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
            assert_layout_equal(ge["tag"], ge["key"], ge["val"], oe["tag"], oe["key"], oe["val"])
            assert np.array_equal(ge["semaphores"][lv], oe["semaphores"][lv])
        else:
            mg, mo = ge["tag"].astype(bool), oe["tag"].astype(bool)
            assert np.array_equal(ge["key"][mg], oe["key"][mo])
            assert np.array_equal(ge["val"][mg], oe["val"][mo])


# ------------------------------------------------------------------------------------------- vector
@pytest.mark.parametrize("n", [0, 1, 2, 5, 11, 100, 1000, 4097, 100_000])
def test_vec_build_layout_bit_exact(n):
    rng = np.random.default_rng(n)
    keys = rng.integers(1, max(10 * n, 10), n)          # duplicates on purpose
    vals = rng.integers(1, 1000, n) / 8.0
    gv = D.dynamicsparsevec(keys, vals)
    ov = O.Vec(keys, vals)
    assert_vec_equal(gv, ov)
    gk, gvv = gv.nonzeros()
    ok, ovv = ov.items()
    assert np.array_equal(gk, ok) and np.array_equal(gvv, ovv)


def test_vec_build_combine_fold_order():   # sparsevector.jl:6-30 pins the left-to-right fold
    I = [1, 2, 5, 5, 3, 10, 1, 8, 1, 5]
    V = [1.0, 3.5, 2.1, 8.5, 2.1, 1.1, 5.0, 7.8, 1.1, 2.0]
    v = D.dynamicsparsevec(I, V)
    assert v[1] == 1.0 + 1.1 + 5.0 and v[5] == 2.1 + 8.5 + 2.0 and v[4] == 0.0
    v2 = D.dynamicsparsevec(I, V, combine="*")
    assert v2[1] == 1.0 * 1.1 * 5.0 and v2[5] == 2.1 * 8.5 * 2.0
    assert len(v) == 10 and v.info()["capacity"] == 16 and D.nnz(v) == 6
    # Float64 fold order with many duplicates
    rng = np.random.default_rng(0)
    keys = rng.integers(1, 50, 5000)
    vals = rng.random(5000) * 1e6
    assert_vec_equal(D.dynamicsparsevec(keys, vals), O.Vec(keys, vals))
    assert_vec_equal(D.dynamicsparsevec(keys, vals, combine="*", n=77), O.Vec(keys, vals, combine=O.COMB_MUL, n=77))


def test_vec_simple_use_reference_sequence():   # sparsevector.jl:36-79
    I = [1, 2, 5, 5, 3, 10, 1, 8, 1, 5]
    V = [1.0, 3.5, 2.1, 8.5, 2.1, 1.1, 5.0, 7.8, 1.1, 2.0]
    vec = D.dynamicsparsevec(I, V)
    vec[1] = 0
    vec[2] = 0
    vec[3] = 0
    vec[22] = 0
    vec[1001] = 1.8
    vec[987] = 4.7
    vec[2] = 15 / 3
    vec[4] = 42
    assert vec[1] == 0 and vec[2] == 15 / 3 and vec[3] == 0 and vec[4] == 42 and vec[1001] == 1.8 and vec[987] == 4.7
    assert list(vec) == [(2, 5), (4, 42), (5, 12.6), (8, 7.8), (10, 1.1), (987, 4.7), (1001, 1.8)]
    assert len(vec) == 1001
    assert vec[:] is vec
    vec1 = D.dynamicsparsevec([1, 2, 3, 5, 6, 8, 9], [1.0, 1.0, 1.0, 2.0, 1.0, 1.0, 3.0])
    vec2 = D.dynamicsparsevec([1, 2, 3, 5, 6, 8, 9, 10, 11], [1.0, 1.0, 1.0, 2.0, 1.0, 1.0, 3.0, 2.0, 3.0])
    assert not (vec1 == vec2)
    vec2[10] = 0
    vec2[11] = 0
    D.shrink_size(vec1)
    D.shrink_size(vec2)
    assert vec1 == vec2
    with pytest.raises(D.ErrorException):
        copy.copy(vec1)
    c = copy.deepcopy(vec1)
    assert c == vec1
    assert D.dynamicsparsevec([1, 2, 3], [2.0, 3.0, 4.0]).filter(lambda e: e[0] % 2 == 0) == D.dynamicsparsevec([2], [3.0])


@pytest.mark.parametrize("seed", range(6))
def test_vec_batches_layout_equals_policy_and_contents_equal_reference(seed):
    rng = np.random.default_rng(seed)
    n0 = [0, 5, 100, 3000, 20000, 1000][seed]
    keys = np.unique(rng.integers(1, 50_000, n0)) if n0 else np.array([], np.int64)
    vals = rng.random(len(keys)) + 0.5
    gv, pol, seq = D.dynamicsparsevec(keys, vals), O.Vec(keys, vals), O.Vec(keys, vals)
    live = set(keys.tolist())
    names = set()
    for rnd in range(8):
        nb = int(rng.integers(1, 4000))
        mode = rnd % 4
        if mode == 0:
            k = rng.integers(1, 50_000, nb)
            v = np.where(rng.random(nb) < 0.4, 0.0, rng.random(nb) + 0.5)
        elif mode == 1:
            base = int(rng.integers(1, 40_000))
            k = base + np.arange(nb)
            v = rng.random(nb) + 0.5
        elif mode == 2:
            arr = np.array(sorted(live)) if live else np.array([1])
            k = rng.choice(arr, size=min(len(arr), nb * 4), replace=False)
            v = np.zeros(len(k))
        else:
            k = rng.integers(1, 200, nb)
            v = np.where(rng.random(nb) < 0.3, 0.0, rng.random(nb) + 0.5)
        names |= _kernels_of(lambda: gv.set_batch(k, v))
        pol.set_batch_policy(k, v)
        seq.set_many(k, v)
        for kk, vv in zip(k.tolist(), v.tolist()):
            (live.add if vv != 0 else live.discard)(kk)
        assert_vec_equal(gv, pol)                       # layout: bit-exact against the CPU statement of the batch policy
        gk, gvals = gv.nonzeros()
        sk, svals = seq.items()
        assert np.array_equal(gk, sk) and np.array_equal(gvals, svals)   # contents: bit-exact against the reference semantics
        assert gv.info()["n"] == seq.info()["n"]
        q = rng.integers(1, 50_000, 500)
        assert np.array_equal(gv.get_batch(q), seq.get_many(q))
    if seed in (0, 2, 4, 5):   # runs of consecutive keys that no window of SMALL_CELLS cells can hold
        assert BIG_WINDOW_KERNELS <= names, sorted(names)


def test_vec_grow_and_shrink():
    gv, pol = D.dynamicsparsevec([], []), O.Vec([], [])
    k = np.arange(1, 100_001)
    names = _kernels_of(lambda: gv.set_batch(k, np.full(len(k), 2.0)))
    assert RESIZE_KERNELS <= names, sorted(names)
    pol.set_batch_policy(k, np.full(len(k), 2.0))
    assert_vec_equal(gv, pol)
    assert gv.info()["segment_capacity"] == 8
    names = _kernels_of(lambda: gv.set_batch(k, np.zeros(len(k))))
    assert "merge_scatter_root" in names, sorted(names)
    pol.set_batch_policy(k, np.zeros(len(k)))
    assert_vec_equal(gv, pol)
    assert gv.info()["nnz"] == 0 and gv.info()["capacity"] == 16


def test_vec_single_writes_queue_flushes_in_order():
    gv, seq = D.dynamicsparsevec([3, 9], [1.0, 2.0]), O.Vec([3, 9], [1.0, 2.0])
    rng = np.random.default_rng(5)
    for _ in range(3000):
        k, v = int(rng.integers(1, 300)), float(rng.integers(0, 4))
        gv[k] = v
        seq[k] = v
    gk, gvals = gv.nonzeros()
    sk, svals = seq.items()
    assert np.array_equal(gk, sk) and np.array_equal(gvals, svals)
    assert len(gv) == len(seq)


# ------------------------------------------------------------------------------------------- matrix
def _rand_coo(rng, m, n, nnz, integer_vals=False):
    I, J = rng.integers(1, m + 1, nnz), rng.integers(1, n + 1, nnz)
    V = rng.integers(1, 100, nnz).astype(float) if integer_vals else rng.random(nnz) + 0.5
    return I, J, V


@pytest.mark.parametrize("m,n,nnz", [(8, 3, 9), (5, 5, 1), (30, 40, 200), (300, 200, 5000), (1000, 1000, 60_000), (50, 20_000, 30_000)])
def test_matrix_build_layout_bit_exact(m, n, nnz):
    rng = np.random.default_rng(nnz)
    I, J, V = _rand_coo(rng, m, n, nnz)
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    assert_matrix_equal(gm, om)
    assert gm.size == om.size
    q = 2000
    rq, cq = rng.integers(1, m + 2, q), rng.integers(1, n + 2, q)
    assert np.array_equal(gm.get_batch(rq, cq), om.get_many(rq, cq))
    assert np.array_equal(gm.get_batch(rq, cq, which=1), om.get_many(rq, cq, which=1))


def test_matrix_build_known_answers():   # sparsematrix.jl:174-195, 288-299; SURVEY §8c derived layouts
    J = [1, 1, 1, 2, 2, 2, 3, 3, 3]
    I = [1, 2, 3, 2, 6, 7, 1, 6, 8]
    V = [2, 3, 4, 2, 4, 5, 3, 5, 7]
    M = D.dynamicsparse(I, J, V)
    assert D.nnz(M.colmajor) == D.nnz(M.rowmajor) == D.nnz(M) == 9 and M.size == (8, 3)
    e0, e1 = M.export(0), M.export(1)
    _ = None
    exp = [_, (0, 1), _, _, (1, 2), _, (2, 3), _, _, (3, 4), _, _, (0, 2), _, (2, 2), _, _, (6, 4), _, _, (7, 5), _, (0, 3), _, _,
           (1, 3), _, _, (6, 5), _, (8, 7), _]
    got = [None if not t else (int(k), float(v)) for t, k, v in zip(e0["tag"], e0["key"], e0["val"])]
    assert got == exp and e0["semaphores"].tolist() == [2, 13, 23]
    assert e1["semaphores"].tolist() == [2, 8, 14, 19, 25, 29] and e1["col_keys"].tolist() == [1, 2, 3, 6, 7, 8]
    m2 = np.array([[2, 0, 3], [3, 2, 0], [4, 0, 0], [0, 0, 0], [0, 0, 0], [0, 4, 5], [0, 5, 0], [0, 0, 7]], float)
    for i in range(8):
        for j in range(3):
            assert M[i + 1, j + 1] == m2[i, j]
    I = [1, 1, 2, 4, 3, 5, 1, 3, 1, 5, 1, 5, 4]
    J = [4, 3, 3, 7, 18, 9, 3, 18, 4, 2, 3, 1, 7]
    V = [1, 8, 10, 2, -5, 3, 2, 1, 1, 1, 5, 3, 2]
    M = D.dynamicsparse(I, J, V)
    assert M[1, 4] == 2 and M[1, 3] == 15 and M[4, 7] == 4 and M[3, 18] == -4 and M[5, 9] == 3 and M[2, 3] == 10
    with pytest.raises(D.ArgumentError):
        D.dynamicsparse([1, 2], [1], [1.0, 2.0])
    with pytest.raises(D.ArgumentError):
        D.dynamicsparse([1, 0], [1, 1], [1.0, 2.0])   # device contract: in-array keys >= 1


def test_matrix_reference_sequence():   # sparsematrix.jl:197-285 (README.md:31-40 included)
    M = D.dynamicsparse([1, 2, 3, 2, 6, 7, 1, 6, 8], [1, 1, 1, 2, 2, 2, 3, 3, 3], [2, 3, 4, 2, 4, 5, 3, 5, 7])
    om = O.Matrix([1, 2, 3, 2, 6, 7, 1, 6, 8], [1, 1, 1, 2, 2, 2, 3, 3, 3], [2, 3, 4, 2, 4, 5, 3, 5, 7])
    M[1, 1] = 4
    M[1, 2] = M[1, 2] + 3
    M[3, 1] = 0
    M[4, 2] = 1
    for args in ((1, 1, 4.0), (1, 2, 3.0), (3, 1, 0.0), (4, 2, 1.0)):
        om[args[0], args[1]] = args[2]
    assert D.nnz(M.rowmajor) == D.nnz(M.colmajor) == 10 and M.size == (8, 3)
    k, v = M.row(2)
    assert len(k) == 2 and k.tolist() == [1, 2]
    k, v = M.col(2)
    assert len(k) == 5
    M[10, 5] = 9
    om[10, 5] = 9.0
    assert D.nnz(M) == 11 and D.nbpartitions(M.colmajor) == 4
    M[1, 4] = 2
    M[3, 4] = 5
    om[1, 4] = 2.0
    om[3, 4] = 5.0
    assert M[1, 4] == 2 and M[3, 4] == 5
    assert D.nbpartitions(M.colmajor) == 5
    assert_matrix_equal(M, om, layout=False)
    D.deletecolumn(M, 2)
    om.deletecolumn(2)
    assert D.nbpartitions(M.rowmajor) == om.info(1)["nb_partitions"] and D.nbpartitions(M.colmajor) == 4
    assert_matrix_equal(M, om, layout=False)
    M[1, 2] = 1
    om[1, 2] = 1.0
    assert M[1, 2] == 1
    assert_matrix_equal(M, om, layout=False)
    with pytest.raises(D.ArgumentError):
        D.deletecolumn(M, 77)


@pytest.mark.parametrize("seed", range(5))
def test_matrix_batches(seed):
    rng = np.random.default_rng(100 + seed)
    m, n = [30, 200, 1000, 50, 400][seed], [30, 300, 1000, 2000, 40][seed]
    nnz0 = [0, 2000, 20000, 5000, 3000][seed]
    if nnz0:
        I, J, V = _rand_coo(rng, m, n, nnz0)
        gm, pol, seq = D.dynamicsparse(I, J, V), O.Matrix(I, J, V), O.Matrix(I, J, V)
    else:
        gm, pol, seq = D.dynamicsparse(fill_mode=False), O.Matrix(fill_mode=False), O.Matrix(fill_mode=False)
    for rnd in range(6):
        nb = int(rng.integers(1, 3000))
        if rnd % 3 == 2:
            J2 = n + 1 + rnd * 1000 + np.sort(rng.integers(0, 500, nb))
            I2 = rng.integers(1, m + 1, nb)
        else:
            I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
        V2 = np.where(rng.random(nb) < 0.35, 0.0, rng.random(nb) + 0.5)
        gm.set_batch(I2, J2, V2)
        pol.set_batch_policy(I2, J2, V2)
        seq.set_many(I2, J2, V2)
        assert_matrix_equal(gm, pol)                  # layout + semaphores + column structure: bit-exact vs the batch policy
        assert_matrix_equal(gm, seq, layout=False)    # contents + column structure: bit-exact vs the reference semantics
        q = 1000
        rq, cq = rng.integers(1, m + 2, q), rng.integers(1, n + 600, q)
        assert np.array_equal(gm.get_batch(rq, cq), seq.get_many(rq, cq))


def test_matrix_batch_duplicates_last_writer_wins():
    """many writes to the same (i, j) inside one batch, on both sort paths: per-partition buckets (all columns exist, small
    buckets) and radix sort (a hot column overflows the bucket limit / new columns appear)"""
    rng = np.random.default_rng(31)
    m, n = 60, 50
    I, J, V = _rand_coo(rng, m, n, 1500)
    for hot in (False, True):
        gm, pol, seq = D.dynamicsparse(I, J, V), O.Matrix(I, J, V), O.Matrix(I, J, V)
        for rnd in range(3):
            nb = 6000
            I2 = rng.integers(1, m + 1, nb)
            J2 = rng.integers(1, n + 1, nb) if not hot else np.where(rng.random(nb) < 0.5, 7, rng.integers(1, n + 1, nb))
            V2 = np.where(rng.random(nb) < 0.4, 0.0, rng.integers(1, 9, nb).astype(float))
            gm.set_batch(I2, J2, V2)
            pol.set_batch_policy(I2, J2, V2)
            seq.set_many(I2, J2, V2)
            assert_matrix_equal(gm, pol)
            assert_matrix_equal(gm, seq, layout=False)


def test_staged_flush_equals_synchronous_flush():
    """dsa_matrix_stage_batch / dsa_matrix_apply_staged (double-buffered H2D) must be indistinguishable from set_batch"""
    rng = np.random.default_rng(41)
    I, J, V = _rand_coo(rng, 400, 300, 9000)
    a, b = D.dynamicsparse(I, J, V), D.dynamicsparse(I, J, V)
    batches = []
    for _ in range(4):
        nb = 5000
        batches.append((rng.integers(1, 450, nb), rng.integers(1, 350, nb), np.where(rng.random(nb) < 0.3, 0.0, rng.random(nb) + 0.5)))
    def same(a, b):
        for which in (0, 1):
            ea, eb = a.export(which), b.export(which)   # a read: drains whatever is still staged, in arrival order
            assert np.array_equal(ea["tag"], eb["tag"]) and np.array_equal(ea["key"], eb["key"]) and np.array_equal(ea["val"], eb["val"])
            assert np.array_equal(ea["semaphores"], eb["semaphores"])

    a.stage_batch(*batches[0])
    for s in range(4):
        if s + 1 < 4:
            a.stage_batch(*batches[s + 1])       # copy of the next batch overlaps the kernels of this one
        a.apply_staged()
        b.set_batch(*batches[s])
        if s == 1:                               # reading in the middle applies the staged batch 2 first: b must have it too
            b.set_batch(*batches[2])
            same(a, b)
            a.stage_batch(*batches[2])           # re-stage so that the loop's apply_staged has its batch (idempotent rewrite)
            b.set_batch(*batches[2])
    same(a, b)
    with pytest.raises(D.ErrorException):
        a.apply_staged()
    a.stage_batch(*batches[0])
    a.stage_batch(*batches[1])
    with pytest.raises(D.ErrorException):
        a.stage_batch(*batches[2])


def test_matrix_delete_columns_and_rows_bulk():
    rng = np.random.default_rng(11)
    I, J, V = _rand_coo(rng, 300, 400, 8000)
    gm, pol, seq = D.dynamicsparse(I, J, V), O.Matrix(I, J, V), O.Matrix(I, J, V)
    dc = rng.choice(np.unique(J)[:-1], 40, replace=False)
    D.deletecolumn(gm, dc)
    pol.delete_columns_policy(dc)
    for c in dc:
        seq.deletecolumn(int(c))
    assert_matrix_equal(gm, pol)
    assert_matrix_equal(gm, seq, layout=False)
    dr = rng.choice(np.unique(I)[:-1], 25, replace=False)
    D.deleterow(gm, dr)
    pol.delete_rows_policy(dr)
    for r in dr:
        seq.deleterow(int(r))
    assert_matrix_equal(gm, pol)
    assert_matrix_equal(gm, seq, layout=False)
    with pytest.raises(D.ArgumentError):
        D.deletecolumn(gm, int(dc[0]))
    before = gm.export(0)
    with pytest.raises(D.ArgumentError):       # a failed batch leaves the structure unchanged
        D.deletecolumn(gm, [int(np.unique(J)[-1]), int(dc[0])])
    after = gm.export(0)
    assert np.array_equal(before["key"], after["key"]) and np.array_equal(before["tag"], after["tag"])
    J2 = 1000 + np.arange(50)
    I2 = rng.integers(1, 300, 50)
    V2 = rng.random(50) + 1
    gm.set_batch(I2, J2, V2)
    pol.set_batch_policy(I2, J2, V2)
    assert_matrix_equal(gm, pol)
    # views after deletions
    for c in (int(np.unique(J)[0]), int(np.unique(J)[5]), 1003):
        gk, gv = gm.col(c)
        ok, ov = pol.column(c)
        assert np.array_equal(gk, ok) and np.array_equal(gv, ov)
    for r in (int(np.unique(I)[-1]), 7):
        gk, gv = gm.row(r)
        ok, ov = pol.row(r)
        assert np.array_equal(gk, ok) and np.array_equal(gv, ov)


def test_matrix_tombstone_reuse_follows_arrival_order():
    for order, expect in (([3, 5], [1, 3, 5, 9]), ([5, 3], [1, 3, 5, None, 9])):
        gm = D.dynamicsparse([1, 1, 1, 1], [1, 4, 6, 9], [1.0, 1.0, 1.0, 1.0])
        D.deletecolumn(gm, [4, 6])
        gm.set_batch([1, 1], order, [2.0, 2.0])
        e = gm.export(0)
        assert [int(k) if l else None for k, l in zip(e["col_keys"], e["col_live"])] == expect
        assert gm[1, 3] == 2.0 and gm[1, 5] == 2.0 and gm[1, 4] == 0.0


def test_fill_mode():   # sparsematrix.jl:412-519
    M, om = D.dynamicsparse(), O.Matrix()
    values = np.array([[1, 0, 0, 2, 0, 7, 0, 0, 0, 9, 1, 2], [0, 3, 0, 0, 1, 1, 0, 0, 0, 1, 0, 2], [0, 0, 0, 1, 1, 2, 0, 0, 1, 2, 0, 0],
                       [0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 1], [1, 2, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0]], float)
    for i in range(5):
        colids = np.nonzero(values[i])[0] + 1
        D.addrow(M, i + 1, colids, values[i, colids - 1])
        om.addrow(i + 1, colids, values[i, colids - 1])
    row = M[1, :]
    for j in range(12):
        assert row[j + 1] == values[0, j]
    M[1, 2] = 2
    M[1, 1] = 1
    om[1, 2] = 2.0
    om[1, 1] = 1.0
    with pytest.raises(D.ErrorException):
        M.col(1)
    with pytest.raises(D.ErrorException):
        D.deletecolumn(M, 1)
    D.closefillmode(M)
    om.closefillmode()
    assert_matrix_equal(M, om)
    values[0, 1] = 2
    values[0, 0] += 1
    for i in range(5):
        for j in range(12):
            assert M[i + 1, j + 1] == values[i, j]
            assert M.rowmajor[j + 1, i + 1] == values[i, j]
    D.addrow(M, 7, [1, 3, 4, 5], [2, 3, 6, 7])
    for j, v in zip([1, 3, 4, 5], [2, 3, 6, 7]):
        assert M[7, j] == v
    M4 = D.dynamicsparse()
    D.closefillmode(M4)
    assert D.nnz(M4) == 0 and M4[1, 1] == 0
    with pytest.raises(D.ErrorException):
        D.closefillmode(D.dynamicsparse(fill_mode=False))
    # sums duplicates like SparseArrays.sparse; without fill mode the last writer wins
    rng = np.random.default_rng(6)
    row, col = rng.integers(1, 101, 3000), rng.integers(1, 101, 3000)
    vals = rng.integers(1, 100001, 3000).astype(float)
    M, M2 = D.dynamicsparse(), D.dynamicsparse(fill_mode=False)
    dense, dense2 = np.zeros((100, 100)), np.zeros((100, 100))
    for r, c, v in zip(row, col, vals):
        M[int(r), int(c)] = float(v)
        M2[int(r), int(c)] = float(v)
        dense[r - 1, c - 1] += v
        dense2[r - 1, c - 1] = v
    D.closefillmode(M)
    rr, cc = np.meshgrid(np.arange(1, 101), np.arange(1, 101), indexing="ij")
    assert np.array_equal(M.get_batch(rr.ravel(), cc.ravel()), dense.ravel())
    assert np.array_equal(M2.get_batch(rr.ravel(), cc.ravel(), which=1), dense2.ravel())


# ------------------------------------------------------------------------------------------- SpMV
def _rel_close(a, b, rtol=SPMV_RTOL):
    return np.all(np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b)))


def test_spmv_known_answers():   # test/unit/spmv.jl:61-127
    M = D.dynamicsparse([1, 1, 3, 3, 4, 4, 4, 6, 6, 6], [2, 4, 1, 3, 1, 3, 6, 1, 3, 6], [1, 2, 1, 1, 1, 1, 1, 1, 1, 1])
    x = D.dynamicsparsevec([2, 3, 5, 6], [1, 1, 1, 1])
    r = M @ x
    assert [r[i] for i in range(1, 7)] == [1, 0, 1, 2, 0, 2]
    D.deletecolumn(M, 3)
    r = M @ x
    assert [r[i] for i in range(1, 7)] == [1, 0, 0, 1, 0, 1]
    D.deleterow(M, 4)
    r = M @ x
    assert [r[i] for i in range(1, 7)] == [1, 0, 0, 0, 0, 1]
    M = D.dynamicsparse([1, 1, 1, 2, 2, 3, 4, 4, 4], [1, 3, 5, 2, 4, 4, 1, 4, 5], [1, 2, 1, 2, 1, 3, 3, 2, 2])
    r = M.T @ D.dynamicsparsevec([1, 3, 5], [1, 1, 1])       # spmv.jl:29-58 with rows a..e -> 1..5
    assert [r[i] for i in range(1, 6)] == [1, 0, 2, 3, 1]


@pytest.mark.parametrize("m,n,nnz,nx", [(110, 100, 50, 25), (1000, 800, 30_000, 300), (5000, 7000, 400_000, 7000), (20, 100_000, 300_000, 50_000)])
def test_spmv_all_operand_orders_vs_oracle(m, n, nnz, nx):   # math.jl:1-51
    rng = np.random.default_rng(nnz)
    I, J, V = _rand_coo(rng, m, n, nnz)
    gm, om = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    xk = np.unique(rng.integers(1, n + 1, nx))
    xv = rng.random(len(xk)) * 2 - 1
    x = D.dynamicsparsevec(xk, xv, n=n)
    yk, yv = om.mul(xk, xv)
    a = gm @ x
    assert len(a) == m
    assert np.array_equal(a.nzind, yk)          # same touched rows (structure of the sparse result)
    assert _rel_close(a.nzval, yv)
    b = gm @ D.SparseVector(n, xk, xv)
    g = x @ gm.T
    assert np.array_equal(a.nzval, b.nzval) and np.array_equal(a.nzval, g.nzval)
    xk2 = np.unique(rng.integers(1, m + 1, max(nx // 4, 3)))
    xv2 = rng.random(len(xk2)) * 2 - 1
    x2 = D.dynamicsparsevec(xk2, xv2, n=m)
    yk, yv = om.mul(xk2, xv2, trans=True)
    d = gm.T @ x2
    assert len(d) == n and np.array_equal(d.nzind, yk) and _rel_close(d.nzval, yv)
    i_ = x2 @ gm
    assert np.array_equal(d.nzval, i_.nzval)
    # dense x
    xd = rng.random(n)
    yd = gm.mul_dense(xd)
    yo = om.mul_dense(xd, m)
    assert _rel_close(yd, yo)
    yd = gm.mul_dense(rng.random(m) * 0 + 1.0, trans=True)
    yo = om.mul_dense(np.ones(m), n, trans=True)
    assert _rel_close(yd, yo)


def test_spmv_integer_values_bit_exact_and_after_updates():
    rng = np.random.default_rng(21)
    m, n = 3000, 2000
    I, J, V = _rand_coo(rng, m, n, 100_000, integer_vals=True)
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    for rnd in range(3):
        nb = 20_000
        I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
        V2 = np.where(rng.random(nb) < 0.4, 0.0, rng.integers(1, 50, nb).astype(float))
        gm.set_batch(I2, J2, V2)
        om.set_batch_policy(I2, J2, V2)
        xd = rng.integers(0, 5, gm.size[1]).astype(float)
        assert np.array_equal(gm.mul_dense(xd), om.mul_dense(xd, gm.size[0]))        # integers: exact in any summation order
        xt = rng.integers(0, 5, gm.size[0]).astype(float)
        assert np.array_equal(gm.mul_dense(xt, trans=True), om.mul_dense(xt, gm.size[1], trans=True))
    # one very long row (spans many chunks) and many empty partitions
    I = np.concatenate([np.full(50_000, 7), np.arange(1, 2001)])
    J = np.concatenate([np.arange(1, 50_001), np.full(2000, 3)])
    V = np.ones(len(I))
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    xd = rng.integers(1, 4, 50_000).astype(float)
    assert np.array_equal(gm.mul_dense(xd), om.mul_dense(xd, gm.size[0]))
    assert np.array_equal(gm.mul_dense(np.ones(2000), trans=True), om.mul_dense(np.ones(2000), 50_000, trans=True))


# ------------------------------------------------------------------------------------------- golden fixtures + full-size properties
def test_golden_fixtures():
    import glob
    import os
    files = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))
    assert files, "tests/golden/*.npz missing (python tests/golden/make_golden.py)"
    for f in files:
        z = np.load(f)
        kind = str(z["kind"])
        if kind == "vec":
            gv = D.dynamicsparsevec(z["I"], z["V"])
            for b in range(int(z["nbatches"])):
                gv.set_batch(z[f"bk{b}"], z[f"bv{b}"])
            occ, k, v = gv.export()
            assert_layout_equal(occ, k, v, z["tag"], z["key"], z["val"])
        else:
            gm = D.dynamicsparse(z["I"], z["J"], z["V"])
            for b in range(int(z["nbatches"])):
                gm.set_batch(z[f"bi{b}"], z[f"bj{b}"], z[f"bv{b}"])
            if len(z["delcols"]):
                D.deletecolumn(gm, z["delcols"])
            for which in (0, 1):
                e = gm.export(which)
                assert_layout_equal(e["tag"], e["key"], e["val"], z[f"tag{which}"], z[f"key{which}"], z[f"val{which}"])
                assert np.array_equal(e["semaphores"], z[f"sem{which}"])
                assert np.array_equal(e["col_live"], z[f"live{which}"])
            y = gm.mul_dense(z["x"])
            assert _rel_close(y, z["y"])


def test_full_size_config2_properties():
    """BASELINE.json configs[1] at full size: PCSR 1e5 x 1e5, 1e7 nnz, one batch of 1M entries, SpMV.  Checked through
    size-independent properties (the sequential oracle would need minutes): geometry, counts, sortedness, semaphore
    bijection, point reads of the batch, SpMV linearity and row/column sums."""
    rng = np.random.default_rng(0xD5A00002)
    m = n = 100_000
    nnz = 10_000_000
    I, J = rng.integers(1, m + 1, nnz), rng.integers(1, n + 1, nnz)
    V = rng.random(nnz)
    gm = D.dynamicsparse(I, J, V, m=m, n=n)
    lin = (I - 1) * n + (J - 1)
    nuniq = len(np.unique(lin))
    for which in (0, 1):
        inf = gm.info(which)
        assert inf["nnz"] == nuniq and inf["nb_partitions"] == 100_000
        assert (inf["capacity"], inf["segment_capacity"], inf["height"]) == (1 << 24, 16, 20)   # SURVEY §8 table
    nb = 1_000_000
    I2, J2, V2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb), rng.random(nb) + 1.0
    gm.set_batch(I2, J2, V2)
    lin2 = (I2 - 1) * n + (J2 - 1)
    total = len(np.unique(np.concatenate([lin, lin2])))
    # last writer per (i, j) in the batch
    order = np.argsort(lin2, kind="stable")
    last = np.ones(nb, bool)
    last[:-1] = lin2[order][1:] != lin2[order][:-1]
    sel = order[last]
    for which in (0, 1):
        inf = gm.info(which)
        assert inf["nnz"] == total
        assert np.array_equal(gm.get_batch(I2[sel], J2[sel], which=which), V2[sel])
    e = gm.export(0)
    tag = e["tag"].astype(bool)
    keys = e["key"][tag]
    pos = np.nonzero(tag)[0] + 1
    semmask = keys == 0
    assert semmask.sum() == 100_000
    ids = e["val"][tag][semmask].astype(np.int64)
    assert np.array_equal(ids, np.arange(1, 100_001))                 # semaphores appear in partition order
    assert np.array_equal(e["semaphores"], pos[semmask])              # semaphores[] <-> array bijection (test/utils.jl:68-92)
    d = np.diff(keys)
    assert np.all((d > 0) | semmask[1:])                              # strictly increasing inside a partition (utils.jl:94-113)
    cnt = e["tag"].reshape(-1, 16).sum(axis=1)
    assert cnt.max() <= 16
    x1, x2 = rng.random(n), rng.random(n)
    y1, y2, y12 = gm.mul_dense(x1), gm.mul_dense(x2), gm.mul_dense(x1 + 2.0 * x2)
    assert np.allclose(y12, y1 + 2.0 * y2, rtol=1e-10, atol=0)        # linearity
    ones = gm.mul_dense(np.ones(n))
    vals = e["val"][tag][~semmask]
    assert abs(ones.sum() - vals.sum()) <= 1e-9 * vals.sum()          # checksum of checksums
    t = gm.mul_dense(np.ones(m), trans=True)
    assert abs(t.sum() - vals.sum()) <= 1e-9 * vals.sum()


def test_single_writes_keep_the_reference_layout():
    """A batch of ONE op is the reference's own setindex!: shift to the next gap (writes.jl:26-43, moves.jl:7-85) — across leaf
    and partition boundaries, to the left when the tail is full — one leaf->root walk, at most one _extend!/_shrink!.  The
    layout after every single write is compared BIT FOR BIT with the sequential oracle (= the reference), not with the batch
    policy: vectors, and matrix writes on existing rows / columns."""
    rng = np.random.default_rng(2024)
    # vector: random mix of new keys, overwrites and deletes
    keys = np.unique(rng.integers(1, 20_000, 3000))
    vals = rng.random(len(keys)) + 0.5
    gv, seq = D.dynamicsparsevec(keys, vals), O.Vec(keys, vals)
    live = keys.tolist()
    for t in range(600):
        r = rng.random()
        if r < 0.6:
            k, v = int(rng.integers(1, 20_000)), float(rng.random() + 0.5)
        elif r < 0.8:
            k, v = int(live[rng.integers(0, len(live))]), float(rng.random() + 0.5)   # overwrite (or re-insert)
        else:
            k, v = int(live[rng.integers(0, len(live))]), 0.0                          # delete (maybe already gone)
        gv.set_batch([k], [v])
        seq[k] = v
        live.append(k)
        if t % 25 == 24:
            assert_vec_equal(gv, seq)
    assert_vec_equal(gv, seq)
    # a tiny vector filled from the right end: no gap to the right -> shifts to the LEFT, and _extend! one step at a time
    gv, seq = D.dynamicsparsevec([5, 9], [1.0, 2.0]), O.Vec([5, 9], [1.0, 2.0])
    for t in range(120):
        k, v = 10 + 3 * t, float(t + 1)
        gv.set_batch([k], [v])
        seq[k] = v
        assert_vec_equal(gv, seq)
    for t in range(119, -1, -1):      # and emptied again: _shrink! one step per delete
        gv.set_batch([10 + 3 * t], [0.0])
        seq[10 + 3 * t] = 0.0
        assert_vec_equal(gv, seq)
    # matrix: single writes on existing rows and columns (both orientations shift independently, semaphores follow)
    m, n = 60, 50
    I, J = rng.integers(1, m + 1, 900), rng.integers(1, n + 1, 900)
    V = rng.random(900) + 0.5
    gm, sq = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    rows, cols = np.unique(I), np.unique(J)
    for t in range(500):
        i, j = int(rows[rng.integers(0, len(rows))]), int(cols[rng.integers(0, len(cols))])
        v = 0.0 if rng.random() < 0.3 else float(rng.random() + 0.5)
        gm.set_batch([i], [j], [v])
        sq[i, j] = v
        if t % 20 == 19:
            assert_matrix_equal(gm, sq)      # layout, semaphores, column map: bit-exact with the reference
    assert_matrix_equal(gm, sq)
    x = rng.random(n)
    assert _rel_close(gm.mul_dense(x), sq.mul_dense(x, m))


def test_spmv_sparse_x_over_a_huge_key_space():
    """ids around 1e10 (what a key codec for dates / UInt32 hashes produces): a dense x indexed by key would need tens of GB, the
    reference's Dict accumulator does not care.  The library switches to a sorted-x lookup (binary search per cell); same result."""
    rng = np.random.default_rng(77)
    nnz = 6000
    I, J = rng.integers(1, 100_000_000, nnz), rng.integers(1, 50_000_000_000, nnz)    # 27 + 36 key bits (the builder packs both in 64)
    J[: nnz // 2] = rng.choice(J[nnz // 2:], nnz // 2)        # columns with several entries
    I[: nnz // 3] = rng.choice(I[nnz // 3:], nnz // 3)        # rows with several entries
    V = rng.integers(1, 9, nnz).astype(float) / 4.0
    gm, om = D.dynamicsparse(I, J, V), O.Matrix(I, J, V)
    for trans, keys in ((False, J), (True, I)):
        xk = np.unique(np.concatenate([rng.choice(keys, 1500), rng.integers(1, int(keys.max()), 300)]))   # present and absent keys
        xv = rng.integers(1, 5, len(xk)).astype(float)
        y = (gm.T if trans else gm) @ (xk, xv)
        yk, yv = om.mul(xk, xv, trans=trans)
        assert np.array_equal(y.nzind, yk) and np.array_equal(y.nzval, yv)     # integer-valued data: exact
    gm.set_batch(I[:50], J[:50], np.zeros(50))                                  # and after a dynamic batch
    om.set_many(I[:50], J[:50], np.zeros(50))
    xk = np.unique(rng.choice(J, 2000))
    xv = rng.random(len(xk))
    y = gm @ (xk, xv)
    yk, yv = om.mul(xk, xv)
    assert np.array_equal(y.nzind, yk) and _rel_close(y.nzval, yv)
