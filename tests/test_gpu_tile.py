"""GPU parity of the tile-streamed batch pipeline (csrc/tile.cuh): forced on (dsa_set_tile_mode(2)) it must leave, bit for
bit, the layout of the oracle's batch policy, the contents of the reference's sequential setindex! loop (pcsr.jl:341-347), and
the layout the random-access pipeline (mode 0) leaves on a twin matrix fed the same batches."""
import numpy as np
import pytest

import dsa_b200 as D
from oracle import oracle as O
from test_gpu_parity import _kernels_of, assert_matrix_equal

pytestmark = pytest.mark.gpu


@pytest.fixture
def tile_mode():
    prev = D.set_tile_mode(2)
    yield D.set_tile_mode
    D.set_tile_mode(prev)


def _coo(rng, m, n, nnz):
    return rng.integers(1, m + 1, nnz), rng.integers(1, n + 1, nnz), rng.random(nnz) + 0.5


def _same_layout(a, b):
    for which in (0, 1):
        ea, eb = a.export(which), b.export(which)
        for f in ("tag", "key", "val", "semaphores"):
            assert np.array_equal(ea[f], eb[f]), (which, f)


def _mixed_batch(rng, m, n, nb, known, p_del=0.3, p_known=0.5, dup=0.02):
    """inserts of random cells, overwrites / deletes of cells known to exist, deletes of absent cells, repeated keys"""
    I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
    if known is not None and len(known[0]):
        pick = rng.random(nb) < p_known
        src = rng.integers(0, len(known[0]), nb)
        I2 = np.where(pick, known[0][src], I2)
        J2 = np.where(pick, known[1][src], J2)
    V2 = np.where(rng.random(nb) < p_del, 0.0, rng.integers(1, 1000, nb).astype(float))
    nd = int(nb * dup)
    if nd:   # the same (i, j) written several times inside the batch: last writer wins
        src, dst = rng.integers(0, nb, nd), rng.integers(0, nb, nd)
        I2[dst], J2[dst] = I2[src], J2[src]
    return I2, J2, V2


CASES = [
    # m, n, nnz0, batch sizes — capacity 2^13 (S = 8), 2^17 / 2^19 (S = 16); columns of 3 .. 15 000 cells (spans inside a tile / over 8 tiles)
    (300, 200, 5000, [300, 1500, 900, 2000]),
    (3000, 3000, 60_000, [4000, 12_000, 7000, 12_000, 2500]),
    (20, 100_000, 300_000, [30_000, 50_000, 20_000]),
    (100_000, 20, 300_000, [30_000, 50_000]),
    (2000, 40, 70_000, [9000, 5000]),
]


@pytest.mark.parametrize("case", range(len(CASES)))
def test_tile_streamed_batches_vs_oracle_and_vs_random_access_pipeline(case, tile_mode):
    m, n, nnz0, sizes = CASES[case]
    rng = np.random.default_rng(900 + case)
    I, J, V = _coo(rng, m, n, nnz0)
    gt, gr = D.dynamicsparse(I, J, V, m=m, n=n), D.dynamicsparse(I, J, V, m=m, n=n)
    pol, seq = O.Matrix(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    known = (I, J)
    launches = D.lib().dsa_launch_count
    for nb in sizes:
        I2, J2, V2 = _mixed_batch(rng, m, n, nb, known)
        tile_mode(2)
        gt.set_batch(I2, J2, V2)
        tile_mode(0)
        gr.set_batch(I2, J2, V2)
        pol.set_batch_policy(I2, J2, V2)
        seq.set_many(I2, J2, V2)
        assert_matrix_equal(gt, pol)
        assert_matrix_equal(gt, seq, layout=False)
        _same_layout(gt, gr)
        known = (np.concatenate([known[0], I2]), np.concatenate([known[1], J2]))
        q = 2000
        rq, cq = rng.integers(1, m + 2, q), rng.integers(1, n + 2, q)
        assert np.array_equal(gt.get_batch(rq, cq), seq.get_many(rq, cq))
    assert launches() > 0


def test_tile_streamed_growth_and_shrink(tile_mode):
    """insert-only batches until the root window fails (resize through the hand-over arrays), then delete-heavy batches until
    leaves fall under their lower bound (windows above leaf level, shrink)"""
    rng = np.random.default_rng(77)
    m, n = 4000, 4000
    I, J, V = _coo(rng, m, n, 40_000)
    gt, pol, seq = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    allI, allJ = [I], [J]
    caps = [gt.info(0)["capacity"]]
    for rnd in range(5):
        nb = 12_000
        I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
        V2 = rng.random(nb) + 0.5
        gt.set_batch(I2, J2, V2)
        pol.set_batch_policy(I2, J2, V2)
        seq.set_many(I2, J2, V2)
        assert_matrix_equal(gt, pol)
        assert_matrix_equal(gt, seq, layout=False)
        allI.append(I2)
        allJ.append(J2)
        caps.append(gt.info(0)["capacity"])
    assert caps[-1] > caps[0], "the test is meant to cross a resize"
    aI, aJ = np.concatenate(allI), np.concatenate(allJ)
    for rnd in range(6):
        pick = rng.permutation(len(aI))[: 14_000]
        I2, J2, V2 = aI[pick], aJ[pick], np.zeros(len(pick))
        gt.set_batch(I2, J2, V2)
        pol.set_batch_policy(I2, J2, V2)
        seq.set_many(I2, J2, V2)
        assert_matrix_equal(gt, pol)
        assert_matrix_equal(gt, seq, layout=False)
        caps.append(gt.info(0)["capacity"])
    x = rng.random(n)
    y, yo = gt.mul_dense(x), seq.mul_dense(x, m)
    assert np.all(np.abs(y - yo) <= 1e-12 * np.maximum(np.abs(y), np.abs(yo)))


def test_tile_streamed_hot_leaves_and_refusals(tile_mode):
    """many inserts between two neighbouring cells (one leaf receives far more than it can hold), many writes of one key, and a
    batch that overflows a tile's bucket or creates columns (refused: the general path applies it)"""
    rng = np.random.default_rng(5)
    m, n = 50_000, 300
    I, J, V = _coo(rng, m, n, 90_000)
    gt, pol, seq = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)

    def step(I2, J2, V2):
        gt.set_batch(I2, J2, V2)
        pol.set_batch_policy(I2, J2, V2)
        seq.set_many(I2, J2, V2)
        assert_matrix_equal(gt, pol)
        assert_matrix_equal(gt, seq, layout=False)

    # 300 inserts into a narrow row range of one column + background traffic
    nb = 4000
    I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
    I2[:300], J2[:300] = rng.integers(20_000, 20_400, 300), 17
    step(I2, J2, rng.random(nb) + 0.5)
    # one key written 200 times (set / delete alternating), last writer wins
    I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
    V2 = rng.random(nb) + 0.5
    I2[100:300], J2[100:300] = 31_337, 42
    V2[100:300:2] = 0.0
    step(I2, J2, V2)
    # a tile bucket overflows (3000 ops on one column's narrow range): refused, applied by the general path
    I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 1, nb)
    I2[:3000], J2[:3000] = rng.integers(10_000, 10_300, 3000), 99
    step(I2, J2, np.where(rng.random(nb) < 0.3, 0.0, rng.random(nb) + 0.5))
    # new columns: refused as well
    I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 40, nb)
    step(I2, J2, rng.random(nb) + 0.5)
    # and the next eligible batch is tile-streamed again (forced mode ignores the back-off)
    I2, J2 = rng.integers(1, m + 1, nb), rng.integers(1, n + 40, nb)
    step(I2, J2, np.where(rng.random(nb) < 0.5, 0.0, rng.random(nb) + 0.5))
    # keys < 1 are refused before anything changes
    before = gt.export(0)
    with pytest.raises(D.ArgumentError):
        gt.set_batch(np.array([5, 0, 7]), np.array([1, 2, 3]), np.array([1.0, 2.0, 3.0]))
    after = gt.export(0)
    assert np.array_equal(before["tag"], after["tag"]) and np.array_equal(before["key"], after["key"])


def test_tile_streamed_with_tombstones_and_empty_partitions(tile_mode):
    """deleted columns / rows leave tombstones in the column map (the span of a partition then ends at the next LIVE semaphore),
    a zero write to an absent column leaves an empty partition (semaphore only): batches over such a structure, tile-streamed and
    through the random-access pipeline, against the oracle"""
    rng = np.random.default_rng(321)
    m, n = 3000, 2500
    I, J, V = _coo(rng, m, n, 70_000)
    mats = [D.dynamicsparse(I, J, V, m=m, n=n), D.dynamicsparse(I, J, V, m=m, n=n)]
    pol, seq = O.Matrix(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    # empty partitions: zero writes to columns / rows that do not exist yet (pcsr.jl:341-347 creates the column)
    r0, c0 = 7, 11   # an existing row and column that stay alive
    ei, ej, ev = np.array([m + 5, r0, m + 9]), np.array([c0, n + 3, n + 8]), np.zeros(3)
    for g in mats:
        g.set_batch(ei, ej, ev)
    pol.set_batch_policy(ei, ej, ev)
    seq.set_many(ei, ej, ev)
    dead_cols = [int(c) for c in rng.choice(np.setdiff1d(np.arange(1, n + 1), [c0]), 120, replace=False)]
    dead_rows = [int(r) for r in rng.choice(np.setdiff1d(np.arange(1, m + 1), [r0]), 150, replace=False)]
    for g in mats:
        D.deletecolumn(g, dead_cols)
        D.deleterow(g, dead_rows)
    pol.delete_columns_policy(dead_cols)
    pol.delete_rows_policy(dead_rows)
    for c in dead_cols:
        seq.deletecolumn(c)
    for r in dead_rows:
        seq.deleterow(r)
    assert_matrix_equal(mats[0], pol)
    assert_matrix_equal(mats[0], seq, layout=False)
    live_c = np.setdiff1d(np.arange(1, n + 1), dead_cols)
    live_r = np.setdiff1d(np.arange(1, m + 1), dead_rows)
    for nb in (9000, 14_000, 6000):
        I2, J2 = rng.choice(live_r, nb), rng.choice(live_c, nb)   # existing rows and columns only: no partition is created
        V2 = np.where(rng.random(nb) < 0.35, 0.0, rng.integers(1, 50, nb).astype(float))
        I2[:3], J2[:3] = [m + 5, r0, m + 9], [c0, n + 3, n + 8]     # writes into the empty partitions (third one: a delete)
        V2[:3] = [4.0, 5.0, 0.0]
        tile_mode(2)
        mats[0].set_batch(I2, J2, V2)
        tile_mode(0)
        mats[1].set_batch(I2, J2, V2)
        pol.set_batch_policy(I2, J2, V2)
        seq.set_many(I2, J2, V2)
        assert_matrix_equal(mats[0], pol)
        assert_matrix_equal(mats[0], seq, layout=False)
        _same_layout(mats[0], mats[1])
    x = rng.random(n + 8)
    y, yo = mats[0].mul_dense(x), seq.mul_dense(x, mats[0].size[0])
    assert np.all(np.abs(y - yo) <= 1e-12 * np.maximum(np.abs(y), np.abs(yo)))


@pytest.mark.parametrize("seed", range(24))
def test_tile_streamed_equals_random_access_pipeline_randomized(seed, tile_mode):
    """many small random shapes and batch mixes: both pipelines must leave the same arrays (the random-access pipeline is the
    one the other tests tie to the oracle); every 4th seed is also checked against the oracle"""
    rng = np.random.default_rng(5000 + seed)
    m, n = int(rng.integers(20, 4000)), int(rng.integers(20, 4000))
    nnz0 = int(rng.integers(1500, 120_000))
    I, J, V = _coo(rng, m, n, nnz0)
    gt, gr = D.dynamicsparse(I, J, V, m=m, n=n), D.dynamicsparse(I, J, V, m=m, n=n)
    pol = O.Matrix(I, J, V, m=m, n=n) if seed % 4 == 0 else None
    known = (I, J)
    cap = gt.info(0)["capacity"]
    streamed = total = 0
    for rnd in range(4):
        nb = int(rng.integers(max(2, cap // 200), max(3, cap // 5)))
        p_del, p_known, dup = rng.random() * 0.9, rng.random(), rng.random() * 0.2
        I2, J2, V2 = _mixed_batch(rng, m, n, nb, known, p_del=p_del, p_known=p_known, dup=dup)
        # only existing rows / columns, so that the tile-streamed attempt is not refused for creating a partition
        ok = np.isin(I2, known[0]) & np.isin(J2, known[1])
        I2, J2, V2 = I2[ok], J2[ok], V2[ok]
        if len(I2) < 2:
            continue
        tile_mode(2)
        names = _kernels_of(lambda: gt.set_batch(I2, J2, V2))
        streamed += "tile_merge" in names
        total += 1
        tile_mode(0)
        names0 = _kernels_of(lambda: gr.set_batch(I2, J2, V2))
        assert "tile_merge" not in names0 and "tile_assign" not in names0
        _same_layout(gt, gr)
        for which in (0, 1):
            assert gt.info(which) == gr.info(which)
        if pol is not None:
            pol.set_batch_policy(I2, J2, V2)
            assert_matrix_equal(gt, pol)
        known = (np.concatenate([known[0], I2]), np.concatenate([known[1], J2]))
    assert total == 0 or streamed * 2 >= total, (streamed, total)   # the test is about the tile-streamed pipeline: it must have run
