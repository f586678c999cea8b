"""TEST INFRASTRUCTURE — the compressed snapshot restated on a raw layout dump: a numpy compaction of export(which) (the
device's or the oracle's), against which dsa_matrix_compress[_dense][_d] is checked."""
import numpy as np


def compact(e):
    """(part_keys, ptr, keys, vals) of an export dict: the occupied cells in array order, semaphore cells (key 0, value =
    partition id) turned into the pointer, gaps dropped"""
    occ = e["tag"].astype(bool)
    key, val = e["key"][occ], e["val"][occ]
    sem = key == 0
    heads = np.nonzero(sem)[0]
    part_keys = e["col_keys"][val[sem].astype(np.int64) - 1]
    ptr = np.append(heads - np.arange(len(heads)), int((~sem).sum())).astype(np.int64)
    return part_keys.astype(np.int64), ptr, key[~sem], val[~sem]


def in_bounds(part_keys, ptr, keys, dim, idim):
    """no entry in a partition with key > dim, no in-array key > idim (empty partitions above dim do not count)"""
    held = np.diff(ptr) > 0
    return not (part_keys[held] > dim).any() and not (keys > idim).any()


def dense(part_keys, ptr, keys, dim, base):
    """dense-pointer form of a sparse-pointer one (in bounds): ptr_dense[k] = base + ptr[first partition with key >= k + 1]"""
    pd = base + ptr[np.searchsorted(part_keys, np.arange(1, dim + 2), side="left")]
    return pd.astype(np.int64), (keys - 1 + base).astype(np.int64)
