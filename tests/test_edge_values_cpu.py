"""CPU checks of the edge-value machinery of tests/test_gpu_edge_values.py: the oracle's min / max combine against Base.min /
Base.max, the chunk-coverage count, and the exact product reference on the oracle alone — the oracle's sequential sum meets
it, a fused multiply-add (computed exactly and rounded once) fails the exact check of the two-product rows."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O
from test_gpu_edge_values import (MIN_MAX_KNOWN, assert_product, bits, cancel_coo, chunk_coverage, exact_products, paired,
                                  stored_cells)


def _same_bits(a, b):
    return bits(np.array([a]))[0] == bits(np.array([b]))[0]


@pytest.mark.parametrize("comb,a,b,expect", MIN_MAX_KNOWN)
def test_oracle_min_max_combine_known_answers(comb, a, b, expect):
    v = O.Vec([3, 3], [a, b], combine=comb)
    assert _same_bits(v[3], expect), (v[3], expect)
    m = O.Matrix([3, 3], [2, 2], [a, b], combine=comb)
    for which in (0, 1):
        assert _same_bits(m.get_many([3], [2], which=which)[0], expect)


def test_chunk_coverage_counts():
    cap = 1024
    tag, key = np.zeros(cap, np.uint8), np.full(cap, 5, np.int64)
    cells = list(range(1, 11)) + list(range(264, 901)) + list(range(1001, 1011))
    sems = [0, 255, 263, 1000]
    tag[cells] = 1
    tag[sems] = 1
    key[sems] = 0
    got = chunk_coverage(dict(tag=tag, key=key))
    assert got == dict(sem_at_chunk_start=1, sem_at_chunk_end=1, sem_at_lane_end=2, partition_over_3_chunks=1, chunk_without_sem=1,
                       empty_partition=1, partial_single_chunk=0)
    assert chunk_coverage(dict(tag=tag[:128], key=key[:128]))["partial_single_chunk"] == 1


def _fused_product(om, x, trans, ny):
    """y = fma(a, x, y) cell by cell in layout order, each step exact and rounded once: what a kernel that contracts
    y += a * x into a fused multiply-add computes"""
    part, xkey, a = stored_cells(om, 0 if trans else 1)
    out = np.zeros(ny)
    for p, k, v in zip(part.tolist(), xkey.tolist(), a.tolist()):
        out[p - 1] = float(Fraction(v) * Fraction(float(x[k - 1])) + Fraction(out[p - 1]))   # Fraction -> float rounds correctly
    return out


@pytest.mark.parametrize("trans", [False, True])
def test_exact_reference_accepts_the_sequential_sum_and_rejects_a_fused_multiply_add(trans):
    rng = np.random.default_rng(12)
    m, n = 2000, 1800
    I, J, V = cancel_coo(rng, m, n, 2500)
    om = O.Matrix(I, J, V, m=m, n=n)
    nx, ny = (m, n) if trans else (n, m)
    x = paired(rng, nx)
    ref = exact_products(om, x, trans)
    assert np.sum(ref["L"] == 2) >= 50 and np.sum(ref["L"] >= 3) >= 50, np.bincount(ref["L"])[:5]
    y = om.mul_dense(x, ny, trans=trans)
    assert_product(y, ref)                          # the reference's own order of mul-then-add meets every check
    yf = _fused_product(om, x, trans, ny)
    assert np.max(np.abs(yf - y)) > 0
    with pytest.raises(AssertionError, match=r"<= 2 products"):
        assert_product(yf, ref)
    # a row of three or more products off by twice its bound fails the bound check
    big = np.nonzero((ref["L"] >= 3) & ref["finite"])[0]
    rows = ref["keys"][big]
    slack = 1.01 * ref["L"][big] * 2.0 ** -53 * ref["A"][big]
    i = int(np.argmax(ref["L"][big]))
    y2 = y.copy()
    y2[rows[i] - 1] = ref["S"][big][i] + 2 * slack[i]
    with pytest.raises(AssertionError, match="error bound"):
        assert_product(y2, ref)
