"""CPU check of phase R of k_tile_merge (csrc/tile.cuh): a re-laid leaf is written with one lane per cell, each lane working out
what lands in its own cell from (surv, insm, rop, M).

Two statements of the re-lay are compared: a walk over the leaf's cells (the next insert or the next survivor for every occupied
cell of the spread! mask, as pack! + spread! lay them) and the per-cell formula (rank r = popc(M below q); an
insert's if bit r of insm is set, else survivor number r - popc(insm below r), found through the group's survivor index).  They
must give the same (kind, source) for every cell, the same leaf count and the same semaphore positions.  The spread! mask comes
from the library's dsa_spread_dest, as in test_tile_logic.py.  The kernel itself is pinned bit for bit by tests/test_gpu_tile.py."""
import ctypes as C
import itertools

import numpy as np
import pytest

GAP = ("gap", None)


def _lib():
    import dsa_b200 as D
    L = D.lib()
    L.dsa_spread_dest.restype = C.c_int64
    return L


def _bounds(L, S, height=12):
    mn, mx = np.zeros(40, np.int64), np.zeros(40, np.int64)
    assert L.dsa_level_bounds(C.c_int64(S), C.c_int64(height), mn.ctypes.data_as(C.c_void_p), mx.ctypes.data_as(C.c_void_p)) == 0
    return int(mn[0]), int(mx[0])


def _masks(L, S, mn0, mx0):
    """leafmask[m]: the cells spread! occupies when it lays m elements over a leaf of S cells"""
    out = {}
    for m in range(mn0, mx0 + 1):
        M = 0
        for r in range(m):
            M |= 1 << int(L.dsa_spread_dest(C.c_int64(S), C.c_int64(m), C.c_int64(r)))
        assert bin(M).count("1") == m
        out[m] = M
    return out


def _popc(x):
    return bin(x).count("1")


def walk(S, surv, ni, insm, rop, M):
    """one thread per re-laid leaf, cell by cell: the next insert or the next survivor for every occupied cell of the mask"""
    cells, r, sv = [None] * S, 0, surv
    for q in range(S):
        if (M >> q) & 1:
            if (insm >> r) & 1:
                cells[q] = ("op", rop[r])
            else:
                c = (sv & -sv).bit_length() - 1   # __ffs(surv) - 1
                cells[q] = ("surv", c)
                sv &= sv - 1
            r += 1
        else:
            cells[q] = GAP
    return cells, _popc(surv) + ni


def phase_r(S, surv, ni, insm, rop, M):
    """one lane per cell (phase R): every lane q of the leaf's group computes its own cell"""
    sidx = [None] * S
    for c in range(S):                                       # lane c writes its survivor number
        if (surv >> c) & 1:
            sidx[_popc(surv & ((1 << c) - 1))] = c
    cells = [None] * S
    for q in range(S):                                       # __syncwarp, then every lane on its own
        if not (M >> q) & 1:
            cells[q] = GAP
            continue
        r = _popc(M & ((1 << q) - 1))
        if (insm >> r) & 1:
            cells[q] = ("op", rop[r])
        else:
            cells[q] = ("surv", sidx[r - _popc(insm & ((1 << r) - 1))])
    return cells, _popc(M)                                   # the leaf count phase D stores is m = popc(M)


def _semaphores(cells, keys):
    """old cell -> new cell of every semaphore (key 0) that moves; inserts have keys >= 1"""
    return {cell[1]: q for q, cell in enumerate(cells) if cell and cell[0] == "surv" and keys[cell[1]] == 0}


def _check(S, surv, m, insm, Mmask, rng):
    ni = m - _popc(surv)
    rop = list(rng.permutation(256)[:S])                     # op index of every merged rank (only the insert ranks are read)
    keys = [0 if rng.random() < 0.2 else int(rng.integers(1, 1 << 40)) for _ in range(S)]
    a = walk(S, surv, ni, insm, rop, Mmask)
    b = phase_r(S, surv, ni, insm, rop, Mmask)
    assert a == b, (S, bin(surv), m, bin(insm))
    assert _semaphores(a[0], keys) == _semaphores(b[0], keys)
    got = [c for c in a[0] if c != GAP]                      # every survivor and every insert lands exactly once
    assert len(got) == m and len(set(got)) == m


def test_phase_r_equals_the_cell_walk_exhaustive_s8():
    L = _lib()
    S = 8
    mn0, mx0 = _bounds(L, S)
    masks = _masks(L, S, mn0, mx0)
    rng = np.random.default_rng(11)
    cases = 0
    for surv in range(1 << S):
        ns = _popc(surv)
        for m in range(max(mn0, ns + 1), mx0 + 1):          # re-laid: at least one insert, m inside the leaf's bounds
            for ranks in itertools.combinations(range(m), m - ns):
                insm = sum(1 << r for r in ranks)
                _check(S, surv, m, insm, masks[m], rng)
                cases += 1
    assert cases > 10000


@pytest.mark.parametrize("S", [16, 32])
def test_phase_r_equals_the_cell_walk_sampled(S):
    L = _lib()
    mn0, mx0 = _bounds(L, S)
    masks = _masks(L, S, mn0, mx0)
    rng = np.random.default_rng(100 + S)
    for m in range(mn0, mx0 + 1):
        for _ in range(300):
            ni = int(rng.integers(1, m + 1))                  # inserts
            ns = m - ni                                      # survivors, on random cells
            surv = sum(1 << int(c) for c in rng.choice(S, ns, replace=False))
            insm = sum(1 << int(r) for r in rng.choice(m, ni, replace=False))
            _check(S, surv, m, insm, masks[m], rng)


def test_relay_list_takes_every_relaid_leaf_once():
    """phase D: per warp a ballot of the 're-laid here' flags, one atomicAdd of its popcount, each flagged lane at base + its
    rank among the flagged lanes below it; the warps arrive in any order"""
    rng = np.random.default_rng(5)
    for NL in (32, 64, 128):
        for _ in range(200):
            mod = rng.random(NL) < rng.random()
            lst, nmod = [None] * NL, 0
            for w in rng.permutation(NL // 32):
                flags = mod[32 * w: 32 * w + 32]
                b = sum(1 << lane for lane in range(32) if flags[lane])
                base, nmod = nmod, nmod + _popc(b)
                for lane in range(32):
                    if flags[lane]:
                        lst[base + _popc(b & ((1 << lane) - 1))] = 32 * w + lane
            assert sorted(lst[:nmod]) == list(np.flatnonzero(mod)) and all(x is None for x in lst[nmod:])
