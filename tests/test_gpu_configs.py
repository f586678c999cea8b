"""GPU parity at BASELINE.json's configurations (the other configs are parity-test cases, not bench lines):
C1 vector 1M keys + 100k mixed ops, C3 column generation rounds, C5 skewed inserts forcing cascading rebalances."""
import copy

import numpy as np
import pytest

import dsa_b200 as D
from oracle import oracle as O
from test_gpu_parity import BIG_WINDOW_KERNELS, RESIZE_KERNELS, _kernels_of, assert_matrix_equal, assert_vec_equal, _rel_close

pytestmark = pytest.mark.gpu


def test_config1_vector_1M_keys_100k_mixed_ops():
    """dynamicsparsevec PMA, 1M Int keys / Float64 values, 100k random inserts+deletes via one buffered flush.
    Reference side = sequential setindex! loop (oracle); GPU layout side = oracle batch policy."""
    rng = np.random.default_rng(0xD5A00001)
    keys = np.unique(rng.integers(1, 10_000_000_000, 1_000_000))            # key range of sparsevector.jl:123
    vals = rng.integers(10, 100001, len(keys)) / 10.0
    p = rng.permutation(len(keys))
    gv, seq, pol = D.dynamicsparsevec(keys[p], vals[p]), O.Vec(keys[p], vals[p]), O.Vec(keys[p], vals[p])
    assert_vec_equal(gv, seq)                                                # bulk build: layout bit-exact with the reference
    assert gv.info()["capacity"] == 1 << 21 and gv.info()["segment_capacity"] == 16 and gv.info()["height"] == 17
    nb = 100_000
    ins_k = rng.integers(1, 10_000_000_000, nb // 2)
    del_k = rng.choice(keys, nb // 2, replace=False)
    bk = np.concatenate([ins_k, del_k])
    bv = np.concatenate([rng.integers(10, 100001, nb // 2) / 10.0, np.zeros(nb // 2)])
    q = rng.permutation(nb)
    bk, bv = bk[q], bv[q]
    for k, v in zip(bk[:2000].tolist(), bv[:2000].tolist()):                 # single writes through the queue...
        gv[k] = v
    gv.set_batch(bk[2000:], bv[2000:])                                       # ...flushed in front of the batch, in order
    seq.set_many(bk, bv)
    pol.set_batch_policy(bk[:2000], bv[:2000])
    pol.set_batch_policy(bk[2000:], bv[2000:])
    assert_vec_equal(gv, pol)
    gk, gvv = gv.nonzeros()
    sk, svv = seq.items()
    assert np.array_equal(gk, sk) and np.array_equal(gvv, svv)
    probe = np.concatenate([bk[:5000], keys[:5000]])
    assert np.array_equal(gv.get_batch(probe), seq.get_many(probe))
    assert len(gv) == len(seq)


def test_full_size_config2_vs_oracle():
    """BASELINE.json configs[1] at FULL size, bit for bit: PCSR 1e5 x 1e5 / 1e7 nnz built from the bench's own COO, then the
    bench's first two 1M-update batches and its insert-only batch.  Layout + semaphores + column map against the oracle's batch
    policy, logical contents against the reference's sequential setindex! loop (oracle), SpMV <= 1e-12 both ways.
    The oracle needs ~9 s per build and ~2 s per batch."""
    import bench as B
    x, coo, batches, insert_only = B.make_workload(3)
    m, n = B.M_ROWS, B.N_COLS
    gm = D.dynamicsparse(coo[0], coo[1], coo[2], m=m, n=n)
    pol = O.Matrix(coo[0], coo[1], coo[2], m=m, n=n)
    assert_matrix_equal(gm, pol)                               # bulk build: layout bit-exact with the reference
    for which in (0, 1):
        inf = gm.info(which)
        assert (inf["capacity"], inf["segment_capacity"], inf["height"]) == (1 << 24, 16, 20)   # SURVEY §8 table
    seq = pol.clone()
    g_io, pol_io, seq_io = copy.deepcopy(gm), pol.clone(), pol.clone()
    xt = np.random.default_rng(1).random(m)
    for bi, bj, bv in batches[:2]:
        gm.set_batch(bi, bj, bv)
        pol.set_batch_policy(bi, bj, bv)
        seq.set_many(bi, bj, bv)
        assert_matrix_equal(gm, pol)                           # layout / semaphores / column map: bit-exact vs the batch policy
        assert_matrix_equal(gm, seq, layout=False)             # contents: bit-exact vs the reference's one-op-at-a-time loop
        assert _rel_close(gm.mul_dense(x), seq.mul_dense(x, m))
        assert _rel_close(gm.mul_dense(xt, trans=True), seq.mul_dense(xt, n, trans=True))
    # configs[1] as written: ONE batched insert of 1M new entries into the fresh matrix, then SpMV
    g_io.set_batch(*insert_only)
    pol_io.set_batch_policy(*insert_only)
    seq_io.set_many(*insert_only)
    assert_matrix_equal(g_io, pol_io)
    assert_matrix_equal(g_io, seq_io, layout=False)
    assert g_io.info(1)["nnz"] == B.NNZ0 - B.N_OVER + B.BATCH
    assert _rel_close(g_io.mul_dense(x), seq_io.mul_dense(x, m))
    probe = np.random.default_rng(2).integers(0, B.BATCH, 50_000)
    assert np.array_equal(g_io.get_batch(insert_only[0][probe], insert_only[1][probe]), insert_only[2][probe])


def test_config3_column_generation_rounds():
    """Coluna-style: fill mode + closefillmode! with the first columns, then rounds of {append columns x 50 nnz with
    increasing ids, deletecolumn! 5% of the live columns (never the highest), A*x and transpose(A)*pi}.  Scaled to 2k
    columns per round so that the sequential oracle (the reference semantics) replays every round."""
    rng = np.random.default_rng(0xD5A00003)
    m, cols_per_round, nnz_per_col, rounds = 20_000, 2_000, 50, 5
    gm, pol, seq = D.dynamicsparse(), O.Matrix(), O.Matrix()

    def new_columns(first_id):
        J = np.repeat(np.arange(first_id, first_id + cols_per_round), nnz_per_col)
        I = np.concatenate([rng.choice(m, nnz_per_col, replace=False) + 1 for _ in range(cols_per_round)])
        return I, J, rng.random(len(I)) + 0.01

    I, J, V = new_columns(1)
    for M_ in (gm, pol, seq):
        for i, j, v in zip(I[:3000].tolist(), J[:3000].tolist(), V[:3000].tolist()):
            M_[i, j] = v                                        # fill-mode writes (buffer.jl:20-31)
    # the rest of round 0 enters through addrow!-free bulk COO: equivalent to more fill-mode writes
    D.closefillmode(gm)
    pol.closefillmode()
    seq.closefillmode()
    gm.set_batch(I[3000:], J[3000:], V[3000:])
    pol.set_batch_policy(I[3000:], J[3000:], V[3000:])
    seq.set_many(I[3000:], J[3000:], V[3000:])
    live = list(range(1, cols_per_round + 1))
    next_id = cols_per_round + 1
    for rnd in range(1, rounds):
        I, J, V = new_columns(next_id)
        gm.set_batch(I, J, V)
        pol.set_batch_policy(I, J, V)
        seq.set_many(I, J, V)
        live += list(range(next_id, next_id + cols_per_round))
        next_id += cols_per_round
        dead = rng.choice(np.array(live[:-1]), len(live) // 20, replace=False)
        D.deletecolumn(gm, dead)
        pol.delete_columns_policy(dead)
        for c in dead:
            seq.deletecolumn(int(c))
        dead_set = set(dead.tolist())
        live = [c for c in live if c not in dead_set]
        assert_matrix_equal(gm, pol)                       # layout / semaphores / tombstones: bit-exact vs the batch policy
        assert_matrix_equal(gm, seq, layout=False)         # contents + column structure: bit-exact vs the reference semantics
        mm, nn = gm.size
        x = rng.random(nn)
        assert _rel_close(gm.mul_dense(x), seq.mul_dense(x, mm))
        pi = rng.random(mm)
        assert _rel_close(gm.mul_dense(pi, trans=True), seq.mul_dense(pi, nn, trans=True))
    assert D.nbpartitions(gm.colmajor) == len(live)


def _zipf(rng, n, size, s=1.0):
    w = 1.0 / np.arange(1, n + 1) ** s
    cdf = np.cumsum(w) / w.sum()
    return np.searchsorted(cdf, rng.random(size)) + 1


def test_config5_skewed_inserts_cascading_rebalances():
    """power-law skewed inserts (Zipf rows and columns) and a monotone variant (consecutive row ids into a few hot columns):
    hot partitions overflow their leaves, windows cascade up the tree, the radix path replaces the bucket path."""
    rng = np.random.default_rng(0xD5A00005)
    m = n = 5_000
    I, J = rng.integers(1, m + 1, 200_000), rng.integers(1, n + 1, 200_000)
    V = rng.random(200_000) + 0.01
    gm, pol = D.dynamicsparse(I, J, V, m=m, n=n), O.Matrix(I, J, V, m=m, n=n)
    names = set()
    for rnd in range(3):
        nb = 60_000
        I2, J2 = _zipf(rng, m, nb), _zipf(rng, n, nb)
        V2 = rng.random(nb) + 0.01
        names |= _kernels_of(lambda: gm.set_batch(I2, J2, V2))
        pol.set_batch_policy(I2, J2, V2)
        assert_matrix_equal(gm, pol)
    # monotone: 100 hot columns receive long runs of consecutive new row ids
    hot = rng.choice(n, 100, replace=False) + 1
    base = m + 1
    for rnd in range(3):
        I2 = np.concatenate([np.arange(base, base + 400) for _ in hot])
        J2 = np.repeat(hot, 400)
        V2 = rng.random(len(I2)) + 0.01
        base += 400
        names |= _kernels_of(lambda: gm.set_batch(I2, J2, V2))
        pol.set_batch_policy(I2, J2, V2)
        assert_matrix_equal(gm, pol)
    assert BIG_WINDOW_KERNELS <= names, sorted(names)   # windows above SMALL_CELLS cells
    seq = O.Matrix(I, J, V, m=m, n=n)          # reference semantics on the final contents (one pass is enough: contents are order-free
    # across batches only through LWW, which the policy oracle already matched batch by batch; re-check one skewed batch sequentially)
    I2, J2, V2 = _zipf(rng, m, 20_000), _zipf(rng, n, 20_000), rng.random(20_000) + 0.01
    g2, s2 = D.dynamicsparse(I, J, V, m=m, n=n), seq
    g2.set_batch(I2, J2, V2)
    s2.set_many(I2, J2, V2)
    assert_matrix_equal(g2, s2, layout=False)
    x = rng.random(gm.size[1])
    assert _rel_close(gm.mul_dense(x), pol.mul_dense(x, gm.size[0]))


def test_growth_from_empty_matches_reference_structure():
    """a matrix that starts empty keeps segment capacity 8 and doubles through _extend! (pma.jl:143-151)"""
    rng = np.random.default_rng(8)
    gm, pol, seq = D.dynamicsparse(fill_mode=False), O.Matrix(fill_mode=False), O.Matrix(fill_mode=False)
    names = set()
    for rnd in range(4):
        nb = 30_000
        I2, J2, V2 = rng.integers(1, 3000, nb), rng.integers(1, 2000, nb), rng.random(nb) + 0.01
        names |= _kernels_of(lambda: gm.set_batch(I2, J2, V2))
        pol.set_batch_policy(I2, J2, V2)
        seq.set_many(I2, J2, V2)
        assert_matrix_equal(gm, pol)
        assert_matrix_equal(gm, seq, layout=False)
    assert RESIZE_KERNELS <= names, sorted(names)
    assert gm.info(0)["segment_capacity"] == 8
