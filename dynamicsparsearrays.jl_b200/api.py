"""Host-side mirror of DynamicSparseArrays.jl's public API (src/DynamicSparseArrays.jl:5-16) over libdsa's C ABI.

Julia is not installed in the build image, so this Python layer is the executable statement of the glue a maintainer
writes in vector.jl / matrix.jl / buffer.jl (julia/DynamicSparseArraysB200.jl holds the same calls as `ccall`s):
same names, same argument meaning, same error behaviour; the structures themselves live in HBM behind opaque handles.

    reference (Julia)                         here (Python)
    dynamicsparsevec(I, V[, combine, n])      dynamicsparsevec(I, V, combine="+", n=None)
    dynamicsparse(I, J, V[, m, n])            dynamicsparse(I, J, V, m=None, n=None)
    dynamicsparse(Ti, Tj, Tv; fill_mode)      dynamicsparse(fill_mode=True)
    v[k] / v[k] = x / m[i, j] / m[i, j] = x   same (single writes are queued and flushed as one batch before any read)
    deletecolumn!(m, j) / deleterow!(m, i)    deletecolumn(m, j) / deleterow(m, i)   (lists accepted: one bulk call)
    addrow!(m, i, cols, vals)                 addrow(m, i, cols, vals)
    closefillmode!(m)                         closefillmode(m)
    view(m, :, j) / view(m, i, :)             m.col(j) / m.row(i)  -> (keys, vals) in ascending key order
    m * v, transpose(m) * v, v * m, ...       m @ v, m.T @ v, v @ m, v @ m.T -> SparseVector
    nnz, nbpartitions, shrink_size!           nnz(x), nbpartitions(m.colmajor), shrink_size(v)
    u + v, u - v, -v (SparseArrays generics)  same operators -> SparseVector (math.jl:53-93)
    Char / other isbits keys                  KeyCodec: order-preserving map onto the device's Int64 keys (CharCodec is
                                              picked automatically for one-character string keys, sparsematrix.jl:302-336)
"""
import ctypes as C
import os
import sys

import numpy as np

from . import _lib
from ._lib import ArgumentError, ErrorException, check, lib

__all__ = ["DynamicSparseVector", "DynamicSparseMatrix", "DynamicMatrixColView", "SparseVector", "dynamicsparsevec",
           "dynamicsparse", "nbpartitions", "deletepartition", "deletecolumn", "deleterow", "addrow", "closefillmode",
           "shrink_size", "nnz", "KeyCodec", "CharCodec", "to_coo", "save_checkpoint", "load_checkpoint", "PackedCSC"]


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _combine(c):
    if callable(c):
        import operator
        c = {operator.add: "+", operator.mul: "*", max: "max", min: "min"}.get(c, c)
    if c not in _lib.COMBINE:
        raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"unsupported combine operator {c!r}; supported: {sorted(_lib.COMBINE)}")
    return _lib.COMBINE[c]


class KeyCodec:
    """Order-preserving map between a caller's key type and the device's Int64 keys (SURVEY.md §8f-4).  The device stores and
    compares Int64 only; any key type whose order an injective, monotone `encode` preserves (Char, Int32, UInt32, enums,
    dates) goes through the same kernels.  Encoded keys must be >= 1: 0 is the semaphore key (pcsr.jl:23)."""

    identity = False

    def __init__(self, encode, decode):
        self._enc, self._dec = encode, decode

    def encode(self, keys):
        out = _i64([self._enc(k) for k in keys])
        if len(out) and out.min() < 1:
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "encoded keys must be >= 1 (0 is the semaphore key)")
        return out

    def encode1(self, key):
        return int(self.encode([key])[0])

    def decode(self, codes):
        return [self._dec(int(c)) for c in codes]

    def decode1(self, code):
        return self._dec(int(code))


class _IdentityCodec(KeyCodec):
    identity = True

    def __init__(self):
        pass

    def encode(self, keys):
        return _i64(keys)

    def encode1(self, key):
        return int(key)

    def decode(self, codes):
        return codes

    def decode1(self, code):
        return int(code)


class CharCodec(KeyCodec):
    """Julia `Char` keys (one-character strings here): the code point, which is Char's own ordering."""

    def __init__(self):
        super().__init__(ord, chr)


_IDENTITY = _IdentityCodec()


def _codec_for(keys):
    """CharCodec for one-character string keys, identity for integers (what `dynamicsparse(I, J, V)` infers from eltype)."""
    if isinstance(keys, np.ndarray):
        return CharCodec() if keys.dtype.kind in "US" else _IDENTITY
    for k in keys:
        return CharCodec() if isinstance(k, str) else _IDENTITY
    return _IDENTITY


def _sv_binary(ka, va, kb, vb, sign):
    """Merge of two sorted (index, value) lists: a + sign * b, entries that come out 0 are not stored (what SparseArrays'
    `_binarymap` does for + and -; the reference has no method of its own and falls back to it, math.jl:53-93)."""
    keys = np.union1d(ka, kb)
    out = np.zeros(len(keys), np.float64)
    out[np.searchsorted(keys, ka)] = va
    ib = np.searchsorted(keys, kb)
    out[ib] = out[ib] + vb if sign > 0 else out[ib] - vb
    keep = out != 0.0
    return keys[keep].astype(np.int64), out[keep]


def _as_sorted_pairs(x):
    if isinstance(x, DynamicSparseVector):
        k, v = x._raw_nonzeros()
        return len(x), k, v
    if isinstance(x, SparseVector):
        return x.n, _i64(x.nzind), _f64(x.nzval)
    return None


def _sv_arith(a, b, sign):
    pa, pb = _as_sorted_pairs(a), _as_sorted_pairs(b)
    if pa is None or pb is None:
        return NotImplemented
    if pa[0] != pb[0]:   # SparseArrays: DimensionMismatch
        raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"dimension mismatch: {pa[0]} != {pb[0]}")
    k, v = _sv_binary(pa[1], pa[2], pb[1], pb[2], sign)
    return SparseVector(pa[0], k, v)


class SparseVector:
    """Result of a product (SparseArrays.SparseVector in the reference, operations.jl:11-12): sorted indices + values."""

    def __init__(self, n, nzind, nzval):
        self.n, self.nzind, self.nzval = int(n), nzind, nzval

    def __len__(self):
        return self.n

    def __getitem__(self, k):
        i = np.searchsorted(self.nzind, k)
        return float(self.nzval[i]) if i < len(self.nzind) and self.nzind[i] == k else 0.0

    def todense(self):
        y = np.zeros(self.n)
        m = (self.nzind >= 1) & (self.nzind <= self.n)
        y[self.nzind[m] - 1] = self.nzval[m]
        return y

    def __eq__(self, other):   # SparseArrays `==` ignores stored zeros
        if isinstance(other, DynamicSparseVector):
            n, k, v = _as_sorted_pairs(other)
            other = SparseVector(n, k, v)
        return self.n == other.n and np.array_equal(self.todense(), other.todense())

    __hash__ = None

    def __add__(self, other):
        return _sv_arith(self, other, +1)

    def __sub__(self, other):
        return _sv_arith(self, other, -1)

    def __neg__(self):
        return SparseVector(self.n, _i64(self.nzind).copy(), -_f64(self.nzval))


class _PendingWrites:
    """Single setindex! calls are queued on the host and applied as ONE batched call before any read.  The batch is
    last-writer-wins in arrival order, so the result equals the reference's loop of setindex! (matrix.jl:119-121)."""

    def __init__(self):
        self.a, self.b, self.v = [], [], []

    def __len__(self):
        return len(self.v)

    def clear(self):
        self.a, self.b, self.v = [], [], []


class DynamicSparseVector:
    """DynamicSparseVector{K,Float64} (vector.jl:1-4) backed by a device PMA (Int64 keys; other K through a KeyCodec)."""

    def __init__(self, handle, owner=True, key_codec=None):
        self._h = handle
        self._L = lib()                  # the library that owns the handle (destroy goes back to it)
        self._kc = key_codec or _IDENTITY
        self._pending = _PendingWrites()
        self.flush_threshold = 1 << 20

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._L.dsa_vec_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # -- writes -------------------------------------------------------------------------------
    def __setitem__(self, key, value):   # vector.jl:76-81
        k = int(self._kc.encode1(key))
        if k == -(1 << 63):              # the error fires at the offending write, like the reference's setindex! would
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "key typemin(Int64) is reserved")
        self._pending.a.append(k)
        self._pending.v.append(float(value))
        if len(self._pending) >= self.flush_threshold:
            self.flush()

    def set_batch(self, keys, vals):
        """Batched setindex!: last writer wins, 0.0 deletes (pma.jl:196-213)."""
        self.flush()
        keys, vals = self._kc.encode(keys), _f64(vals)
        if len(keys) != len(vals):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "keys & values must have same length.")
        check(lib().dsa_vec_set_batch(self._h, _p(keys), _p(vals), C.c_int64(len(keys))))

    def flush(self):
        if len(self._pending):
            k, v = _i64(self._pending.a), _f64(self._pending.v)
            check(lib().dsa_vec_set_batch(self._h, _p(k), _p(v), C.c_int64(len(k))))
            self._pending.clear()        # only once the library has applied them: a failed flush loses nothing

    # -- reads --------------------------------------------------------------------------------
    def __getitem__(self, key):   # vector.jl:72-73
        if isinstance(key, slice) and key == slice(None):
            return self
        return float(self.get_batch([key])[0])

    def get_batch(self, keys):
        self.flush()
        keys = self._kc.encode(keys)
        out = np.zeros(len(keys), np.float64)
        check(lib().dsa_vec_get_batch(self._h, _p(keys), C.c_int64(len(keys)), _p(out)))
        return out

    def info(self):
        self.flush()
        out = np.zeros(6, np.int64)
        check(lib().dsa_vec_info(self._h, _p(out)))
        return dict(capacity=int(out[0]), segment_capacity=int(out[1]), nb_segments=int(out[2]), nnz=int(out[3]),
                    height=int(out[4]), n=int(out[5]))

    def __len__(self):       # vector.jl:68
        return self.info()["n"]

    @property
    def size(self):          # vector.jl:69
        return (len(self),)

    def nonzeros(self):
        """(nonzeroinds, nonzeros) = iteration order of the PMA (vector.jl:93-109, pma.jl:165-180)."""
        k, v = self._raw_nonzeros()
        return self._kc.decode(k), v

    def _raw_nonzeros(self):
        self.flush()
        n = self.info()["nnz"]
        k, v = np.zeros(max(n, 1), np.int64), np.zeros(max(n, 1), np.float64)
        cnt = C.c_int64()
        check(lib().dsa_vec_nonzeros(self._h, _p(k), _p(v), C.c_int64(n), C.byref(cnt)))
        return k[:cnt.value], v[:cnt.value]

    def __iter__(self):      # vector.jl:71
        k, v = self.nonzeros()
        return iter(zip(k.tolist() if hasattr(k, "tolist") else k, v.tolist()))

    def export(self):
        """Raw layout (occupied, keys, vals) for parity checks."""
        cap = self.info()["capacity"]
        occ, k, v = np.zeros(cap, np.uint8), np.zeros(cap, np.int64), np.zeros(cap, np.float64)
        check(lib().dsa_vec_export(self._h, _p(occ), _p(k), _p(v)))
        return occ, k, v

    def __eq__(self, other):   # vector.jl:85-87 + pma.jl:262-266: same length, same stored sequence
        if isinstance(other, SparseVector):   # AbstractSparseVector `==`: same length, same non-zero content
            return other.__eq__(self)
        if not isinstance(other, DynamicSparseVector):
            return NotImplemented
        if len(self) != len(other):
            return False
        (ka, va), (kb, vb) = self._raw_nonzeros(), other._raw_nonzeros()
        return np.array_equal(ka, kb) and np.array_equal(va, vb)

    __hash__ = None

    def __copy__(self):        # vector.jl:90
        raise ErrorException(_lib.DSA_ERR_ERROR, "copy of a dynamic sparse vector not implemented.")

    def __deepcopy__(self, memo):
        self.flush()
        h = C.c_void_p()
        check(lib().dsa_vec_clone(self._h, C.byref(h)))
        return DynamicSparseVector(h, key_codec=self._kc)

    # +, -, unary -: the reference defines none and falls back to SparseArrays' generic methods through
    # nonzeroinds / nonzeros (vector.jl:93-109); the result is a SparseVector (math.jl:53-93)
    def __add__(self, other):
        return _sv_arith(self, other, +1)

    def __sub__(self, other):
        return _sv_arith(self, other, -1)

    def __neg__(self):
        k, v = self._raw_nonzeros()
        return SparseVector(len(self), k.copy(), -v)

    def filter(self, f):       # pma.jl:224-234
        k, v = self._raw_nonzeros()
        keep = [i for i, e in enumerate(zip(self._kc.decode(k.tolist()), v.tolist())) if f(e)]
        return dynamicsparsevec(k[keep], v[keep], key_codec=self._kc if not self._kc.identity else None, _encoded=True)

    def __matmul__(self, mat):   # v * mat / v * transpose(mat)  (operations.jl:38-60)
        if isinstance(mat, _Transposed):
            return mat.array._mul(self, trans=False, n=mat.array._dims()[0])
        if isinstance(mat, DynamicSparseMatrix):
            return mat._mul(self, trans=True, n=mat._dims()[1])
        return NotImplemented


def dynamicsparsevec(I, V, combine="+", n=None, key_codec=None, _encoded=False):
    """dynamicsparsevec(I, V, [combine, n]) (vector.jl:44-62)."""
    if not _encoded:
        key_codec = key_codec or _codec_for(I)
        I = key_codec.encode(I)
        n = None if n is None else key_codec.encode1(n)
    I, V = _i64(I), _f64(V)
    if len(I) != len(V):
        raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "keys & nonzeros vectors must have same length.")
    h = C.c_void_p()
    check(lib().dsa_vec_build(_p(I), _p(V), C.c_int64(len(I)), C.c_int(_combine(combine)), C.c_int64(0 if n is None else n),
                              C.c_int(0 if n is None else 1), C.byref(h)))
    return DynamicSparseVector(h, key_codec=key_codec)


def shrink_size(v):   # shrink_size! (vector.jl:64)
    v.flush()
    out = C.c_int64()
    check(lib().dsa_vec_shrink_size(v._h, C.byref(out)))
    return out.value


# ---------------------------------------------------------------------------------------------
class Buffer:
    """Fill-mode write buffer (buffer.jl:1-50): a host dict row -> (colids, vals); flushed as COO by closefillmode!."""

    def __init__(self):
        self.rowmajor_coo = {}
        self.length = 0

    def addrow(self, rowid, colids, vals):   # buffer.jl:10-18
        if rowid in self.rowmajor_coo:
            raise ErrorException(_lib.DSA_ERR_ERROR, f"Row with id {rowid} already written in dynamic sparse matrix buffer.")
        colids, vals = _i64(colids), _f64(vals)
        p = np.argsort(colids, kind="stable")
        self.rowmajor_coo[rowid] = (colids[p].tolist(), vals[p].tolist())
        self.length += len(vals)

    def addelem(self, rowid, colid, val):    # buffer.jl:20-31
        r = self.rowmajor_coo.setdefault(rowid, ([], []))
        r[0].append(int(colid))
        r[1].append(float(val))
        self.length += 1

    def get_rowids_colids_vals(self):        # buffer.jl:33-50
        rows = np.zeros(self.length, np.int64)
        cols = np.zeros(self.length, np.int64)
        vals = np.zeros(self.length, np.float64)
        cur = 0
        for rowid, (bc, bv) in self.rowmajor_coo.items():
            k = len(bv)
            rows[cur:cur + k] = rowid
            cols[cur:cur + k] = bc
            vals[cur:cur + k] = bv
            cur += k
        return rows, cols, vals

    def row(self, row):                      # view(buffer, row, :)  (views.jl:44-49): combined with +
        bc, bv = self.rowmajor_coo.get(row, ([], []))
        out = {}
        for c, v in sorted(zip(bc, bv), key=lambda e: e[0]):
            out[c] = out.get(c, 0.0) + v
        return _i64(list(out.keys())), _f64(list(out.values()))


class _Orientation:
    """Read-only facade of one MappedPackedCSC (matrix.colmajor / matrix.rowmajor, matrix.jl:6-7)."""

    def __init__(self, matrix, which):
        self._m, self.which = matrix, which

    def info(self):
        return self._m.info(self.which)

    def export(self):
        return self._m.export(self.which)

    def __getitem__(self, idx):
        a, b = idx
        r, c = (a, b) if self.which == _lib.COLMAJOR else (b, a)
        return float(self._m.get_batch([r], [c], which=self.which)[0])


class DynamicMatrixColView:
    """view(matrix, :, col) / view(matrix, row, :) (views.jl:3-35): iterates (key, value) over the stored cells."""

    def __init__(self, keys, vals):
        self.keys, self.vals = keys, vals

    def __iter__(self):
        keys = self.keys.tolist() if hasattr(self.keys, "tolist") else self.keys   # decoded keys of a codec are a list
        return iter(zip(keys, self.vals.tolist()))

    def __len__(self):
        return len(self.keys)


class _Transposed:   # operations.jl:1-9
    def __init__(self, array):
        self.array = array

    @property
    def size(self):
        return tuple(reversed(self.array.size))

    def __getitem__(self, idx):
        return self.array[idx[1], idx[0]]

    def __setitem__(self, idx, val):
        self.array[idx[1], idx[0]] = val

    def __matmul__(self, v):   # transpose(mat) * v  (operations.jl:26-36)
        return self.array._mul(v, trans=True, n=self.array._dims()[1])


class DynamicSparseMatrix:
    """DynamicSparseMatrix{K,L,Float64} (matrix.jl:1-8): both orientations live on the device with Int64 keys; other key
    types K / L go through an order-preserving KeyCodec per axis (identity for integers)."""

    def __init__(self, handle=None, fill_mode=False, row_codec=None, col_codec=None):
        self._h = handle
        self._L = lib()                  # the library that owns the handle (destroy goes back to it)
        self._rc, self._cc = row_codec or _IDENTITY, col_codec or _IDENTITY
        self.fillmode = fill_mode
        self.buffer = Buffer() if fill_mode else None
        self._m = self._n = 0            # dims while in fill mode (matrix.jl:44-47)
        self._pending = _PendingWrites()
        self._staged = []                # host arrays of the batches staged in the library, oldest first
        self.flush_threshold = 1 << 20
        self.colmajor = _Orientation(self, _lib.COLMAJOR)
        self.rowmajor = _Orientation(self, _lib.ROWMAJOR)

    def __del__(self):
        try:
            if getattr(self, "_h", None) and getattr(self, "_owner", True):   # _owner = False: a borrowed handle (DistMatrix.local)
                self._L.dsa_matrix_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # -- writes -------------------------------------------------------------------------------
    def __setitem__(self, idx, val):   # matrix.jl:43-62
        row, col = int(self._rc.encode1(idx[0])), int(self._cc.encode1(idx[1]))
        val = float(val)
        if not self.fillmode and (row < 1 or col < 1):   # device contract (DESIGN.md §3); raised at the offending write
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "row and column keys must be >= 1 (each is an in-array key of one "
                                                       "orientation; key 0 is the semaphore key, pcsr.jl:23)")
        if self.fillmode:
            if val != 0.0:
                self._m, self._n = max(self._m, row), max(self._n, col)
            self.buffer.addelem(row, col, val)
            return
        self._pending.a.append(int(row))
        self._pending.b.append(int(col))
        self._pending.v.append(val)
        if len(self._pending) >= self.flush_threshold:
            self.flush()

    def set_batch(self, rows, cols, vals):
        """Batched setindex! on both orientations: last writer wins, 0.0 deletes, absent rows/columns are created."""
        self._not_fillmode("Cannot apply a batch in fill mode")
        self.flush()
        rows, cols, vals = self._rc.encode(rows), self._cc.encode(cols), _f64(vals)
        if not (len(rows) == len(cols) == len(vals)):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "rows, columns, and nonzeros do not have same length.")
        check(lib().dsa_matrix_set_batch(self._h, _p(rows), _p(cols), _p(vals), C.c_int64(len(rows))))

    def flush(self):
        """Everything written so far becomes visible, in arrival order: staged batches first (they were submitted before any
        write still sitting in the queue: stage_batch flushes the queue in front of itself), then the queued single writes."""
        while self._staged:
            self.apply_staged()
        if len(self._pending):
            r, c, v = _i64(self._pending.a), _i64(self._pending.b), _f64(self._pending.v)
            check(lib().dsa_matrix_set_batch(self._h, _p(r), _p(c), _p(v), C.c_int64(len(r))))
            self._pending.clear()        # only once the library has applied them: a failed flush loses nothing

    def stage_batch(self, rows, cols, vals):
        """Start the host->device copy of a batch and return at once; apply_staged() applies it (double-buffered flush).
        The arrays must stay alive (and should be pinned) until the matching apply_staged() returns."""
        self._not_fillmode("Cannot apply a batch in fill mode")
        if len(self._pending):           # earlier single writes go first (flush also drains the batches staged before them)
            self.flush()
        rows, cols, vals = self._rc.encode(rows), self._cc.encode(cols), _f64(vals)
        if not (len(rows) == len(cols) == len(vals)):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "rows, columns, and nonzeros do not have same length.")
        check(lib().dsa_matrix_stage_batch(self._h, _p(rows), _p(cols), _p(vals), C.c_int64(len(rows))))
        self._staged.append((rows, cols, vals))   # keep the host arrays alive until the copy has been consumed

    def apply_staged(self):
        """Apply the oldest staged batch.  Reads, single writes, deletes and copies drain the staged batches themselves
        (flush), so arrival order — last writer wins — holds whatever the caller interleaves."""
        check(lib().dsa_matrix_apply_staged(self._h))
        if self._staged:
            self._staged.pop(0)

    def _not_fillmode(self, msg):
        if self.fillmode:
            raise ErrorException(_lib.DSA_ERR_ERROR, msg)

    # -- reads --------------------------------------------------------------------------------
    def __getitem__(self, idx):   # matrix.jl:64-68
        row, col = idx
        if self.fillmode:
            if isinstance(col, slice):       # buffer[row, :] (buffer.jl:52-55): PMA of the row, duplicates NOT combined
                bc, bv = self.buffer.rowmajor_coo[self._rc.encode1(row)]
                return dynamicsparsevec(bc, bv, combine="last")
            raise ErrorException(_lib.DSA_ERR_ERROR, "getindex(row, col) is not available in fill mode")
        if isinstance(col, slice):           # keys of the returned vector are the encoded (Int64) column keys
            k, v = self._span(lib().dsa_matrix_row, self._rc.encode1(row))
            return dynamicsparsevec(k, v)
        if isinstance(row, slice):
            k, v = self._span(lib().dsa_matrix_column, self._cc.encode1(col))
            return dynamicsparsevec(k, v)
        return float(self.get_batch([row], [col])[0])

    def get_batch(self, rows, cols, which=_lib.COLMAJOR):
        self._not_fillmode("Matrix is in fill mode")
        self.flush()
        rows, cols = self._rc.encode(rows), self._cc.encode(cols)
        out = np.zeros(len(rows), np.float64)
        check(lib().dsa_matrix_get_batch(self._h, C.c_int(which), _p(rows), _p(cols), C.c_int64(len(rows)), _p(out)))
        return out

    def _span(self, fn, key):
        self.flush()
        cnt = C.c_int64()
        check(fn(self._h, C.c_int64(key), None, None, C.c_int64(0), C.byref(cnt)))
        n = cnt.value
        k, v = np.zeros(max(n, 1), np.int64), np.zeros(max(n, 1), np.float64)
        if n:
            check(fn(self._h, C.c_int64(key), _p(k), _p(v), C.c_int64(n), C.byref(cnt)))
        return k[:n], v[:n]

    def col(self, col):
        """view(matrix, :, col) (matrix.jl:83-88)."""
        self._not_fillmode("View of a column not available in fill mode.")
        k, v = self._span(lib().dsa_matrix_column, self._cc.encode1(col))
        return self._rc.decode(k), v

    def row(self, row):
        """view(matrix, row, :) (matrix.jl:70-81), served from the row-major twin."""
        self._not_fillmode("Matrix is in fill mode, cannot create a view. However, you can use the view method on the buffer.")
        k, v = self._span(lib().dsa_matrix_row, self._rc.encode1(row))
        return self._cc.decode(k), v

    def view(self, row, col):
        if isinstance(row, slice):
            return DynamicMatrixColView(*self.col(col))
        return DynamicMatrixColView(*self.row(row))

    def info(self, which=_lib.COLMAJOR):
        self.flush()
        out = np.zeros(10, np.int64)
        check(lib().dsa_matrix_info(self._h, C.c_int(which), _p(out)))
        return dict(capacity=int(out[0]), segment_capacity=int(out[1]), nb_segments=int(out[2]), nb_elements=int(out[3]),
                    height=int(out[4]), nb_partitions=int(out[5]), nb_semaphores=int(out[6]), m=int(out[7]), n=int(out[8]),
                    nnz=int(out[9]))

    def export(self, which=_lib.COLMAJOR):
        inf = self.info(which)
        cap, ns = inf["capacity"], inf["nb_semaphores"]
        occ, k, v = np.zeros(cap, np.uint8), np.zeros(cap, np.int64), np.zeros(cap, np.float64)
        sem, ck, cl = np.zeros(max(ns, 1), np.int64), np.zeros(max(ns, 1), np.int64), np.zeros(max(ns, 1), np.uint8)
        check(lib().dsa_matrix_export(self._h, C.c_int(which), _p(occ), _p(k), _p(v), _p(sem), _p(ck), _p(cl)))
        return dict(tag=occ, key=k, val=v, semaphores=sem[:ns], col_keys=ck[:ns], col_live=cl[:ns], **inf)

    @property
    def size(self):   # matrix.jl:92; with a codec the dimensions are keys too: size(matrix) == (5, 'e') (sparsematrix.jl:317)
        if self.fillmode:
            m, n = self._m, self._n
        else:
            inf = self.info()
            m, n = inf["m"], inf["n"]
        return (self._rc.decode1(m) if m or self._rc.identity else None, self._cc.decode1(n) if n or self._cc.identity else None)

    def _dims(self):
        """encoded (Int64) dimensions"""
        if self.fillmode:
            return self._m, self._n
        inf = self.info()
        return inf["m"], inf["n"]

    @property
    def T(self):      # transpose (operations.jl:5)
        return _Transposed(self)

    def __deepcopy__(self, memo):
        self._not_fillmode("deepcopy in fill mode is not supported")
        self.flush()
        h = C.c_void_p()
        check(lib().dsa_matrix_clone(self._h, C.byref(h)))
        return DynamicSparseMatrix(h, row_codec=self._rc, col_codec=self._cc)

    # -- products -----------------------------------------------------------------------------
    def _mul(self, x, trans, n):
        self._not_fillmode("Matrix is in fill mode")
        self.flush()
        xcodec, ycodec = (self._rc, self._cc) if trans else (self._cc, self._rc)
        if isinstance(x, DynamicSparseVector):   # its key type is the matrix's key type on that axis: same codec
            xk, xv = x._raw_nonzeros()
        elif isinstance(x, SparseVector):
            xk, xv = x.nzind, x.nzval
        elif isinstance(x, dict):            # a vector over non-integer keys
            xk = xcodec.encode(list(x.keys()))
            o = np.argsort(xk, kind="stable")
            xk, xv = xk[o], _f64(list(x.values()))[o]
        else:
            xk, xv = x
        xk, xv = _i64(xk), _f64(xv)
        cap = self.info(_lib.COLMAJOR if trans else _lib.ROWMAJOR)["nb_semaphores"]
        yk, yv = np.zeros(max(cap, 1), np.int64), np.zeros(max(cap, 1), np.float64)
        cnt = C.c_int64()
        check(lib().dsa_matrix_spmv(self._h, C.c_int(1 if trans else 0), _p(xk), _p(xv), C.c_int64(len(xk)), _p(yk), _p(yv),
                                    C.c_int64(cap), C.byref(cnt)))
        if not ycodec.identity:   # _mul_output for non-integer keys: the Dict itself (operations.jl:11; test/unit/spmv.jl:19-24)
            return dict(zip(ycodec.decode(yk[:cnt.value]), yv[:cnt.value].tolist()))
        return SparseVector(n, yk[:cnt.value].copy(), yv[:cnt.value].copy())

    def __matmul__(self, x):   # mat * v  (operations.jl:14-24)
        return self._mul(x, trans=False, n=self._dims()[0])

    def mul_dense(self, x, trans=False):
        """Dense-x product: x[j-1] for every j in 1..len(x); returns dense y of length size[0] (or size[1] if trans).
        A 2-D x of shape (nx, k) holds k right-hand sides, multiplied in one pass over the matrix per 32 columns: the result
        is (ny, k), and its column c equals mul_dense(x[:, c]) bit for bit.  A torch CUDA tensor (1-D or 2-D) stays on the
        device: the product runs after the work already queued on torch's current stream, and the float64 result tensor is
        ready on that stream."""
        self._not_fillmode("Matrix is in fill mode")
        self.flush()
        torch = sys.modules.get("torch")
        if torch is not None and isinstance(x, torch.Tensor) and x.is_cuda:
            return self._mul_dense_cuda(torch, x, trans)
        x = _f64(x)
        if x.ndim > 2:
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"mul_dense takes a vector or an (nx, k) matrix, not a {x.ndim}-D array")
        ny = self._dims()[1] if trans else self._dims()[0]
        if x.ndim == 2:
            nx, k = x.shape
            y = np.zeros((max(ny, 1), k), np.float64)
            check(lib().dsa_matrix_spmm_dense(self._h, C.c_int(1 if trans else 0), _p(x), C.c_int64(nx), C.c_int64(k), C.c_int64(k),
                                              _p(y), C.c_int64(ny), C.c_int64(k)))
            return y[:ny]
        y = np.zeros(max(ny, 1), np.float64)
        check(lib().dsa_matrix_spmv_dense(self._h, C.c_int(1 if trans else 0), _p(x), C.c_int64(len(x)), _p(y), C.c_int64(ny)))
        return y[:ny]

    def _mul_dense_cuda(self, torch, x, trans):
        if x.dim() not in (1, 2):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"mul_dense takes a vector or an (nx, k) matrix, not a {x.dim()}-D tensor")
        ny = self._dims()[1] if trans else self._dims()[0]
        x = x.to(torch.float64)
        if x.dim() == 1 or x.stride(1) != 1 or x.stride(0) < x.shape[1]:   # a row-major view (any row stride) is read in place
            x = x.contiguous()
        y = torch.empty((max(ny, 1),) + tuple(x.shape[1:]), dtype=torch.float64, device=x.device)
        st = C.c_void_p()
        check(lib().dsa_matrix_get_stream(self._h, C.byref(st)))
        # the handle keeps its own stream (its priority orders the update pipeline): order it against torch's both ways
        cur = torch.cuda.current_stream(x.device)
        hs = torch.cuda.ExternalStream(st.value or 0, device=x.device)
        hs.wait_stream(cur)
        t = C.c_int(1 if trans else 0)
        xp, yp = C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr())
        if x.dim() == 1:
            check(lib().dsa_matrix_spmv_dense_d(self._h, t, xp, C.c_int64(x.shape[0]), yp, C.c_int64(ny)))
        else:
            nx, k = x.shape
            check(lib().dsa_matrix_spmm_dense_d(self._h, t, xp, C.c_int64(nx), C.c_int64(k), C.c_int64(x.stride(0)), yp, C.c_int64(ny),
                                                C.c_int64(k)))
        cur.wait_stream(hs)
        return y[:ny]

    # -- compressed snapshot ------------------------------------------------------------------
    def compressed(self, which=_lib.COLMAJOR):
        """(part_keys, ptr, keys, vals) of one orientation, compacted on the device: the live partitions in ascending key (empty
        ones included), 0-based offsets ptr[len(part_keys) + 1], then the entries of each partition in ascending in-array key
        (stored zeros kept, values bit for bit).  COLMAJOR: partitions are columns, keys rows (CSC); ROWMAJOR: the transpose
        (CSR).  Keys are decoded through the matrix's codecs."""
        self._not_fillmode("Matrix is in fill mode, cannot take a compressed snapshot.")
        self.flush()
        cnt = np.zeros(2, np.int64)
        check(lib().dsa_matrix_compress(self._h, C.c_int(which), None, None, None, None, C.c_int64(0), C.c_int64(0), _p(cnt)))
        npart, nnz = int(cnt[0]), int(cnt[1])
        pk, ptr = np.zeros(max(npart, 1), np.int64), np.zeros(npart + 1, np.int64)
        k, v = np.zeros(max(nnz, 1), np.int64), np.zeros(max(nnz, 1), np.float64)
        check(lib().dsa_matrix_compress(self._h, C.c_int(which), _p(pk), _p(ptr), _p(k), _p(v), C.c_int64(npart), C.c_int64(nnz),
                                        _p(cnt)))
        pc, kc = (self._cc, self._rc) if which == _lib.COLMAJOR else (self._rc, self._cc)
        return np.asarray(pc.decode(pk[:npart])), ptr, np.asarray(kc.decode(k[:nnz])), v[:nnz]

    def _dense_form(self, which, what):
        """checks shared by to_csr / to_csc / to_torch: (m, n, dim, idim) of the orientation"""
        self._not_fillmode(f"Matrix is in fill mode, cannot convert it {what}.")
        if not (self._rc.identity and self._cc.identity):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"conversion {what} needs integer row and column keys (this matrix has a key codec): "
                                                       "use compressed() for the keys themselves")
        self.flush()
        m, n = self._dims()
        return (m, n) + ((n, m) if which == _lib.COLMAJOR else (m, n))

    def _compress_dense_host(self, which, what):
        m, n, dim, idim = self._dense_form(which, what)
        cnt = C.c_int64()
        check(lib().dsa_matrix_compress_dense(self._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(0), None, None, None,
                                              C.c_int64(0), C.byref(cnt)))
        nnz = cnt.value
        ptr, ind, v = np.zeros(dim + 1, np.int64), np.zeros(max(nnz, 1), np.int64), np.zeros(max(nnz, 1), np.float64)
        check(lib().dsa_matrix_compress_dense(self._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(0), _p(ptr), _p(ind),
                                              _p(v), C.c_int64(nnz), C.byref(cnt)))
        return (m, n), ptr, ind[:nnz], v[:nnz]

    def to_csr(self):
        """scipy.sparse.csr_matrix of shape size, from the row-major orientation (canonical: sorted indices, no duplicates,
        stored zeros kept).  BoundsError if an entry lies outside size (dynamicsparse(I, J, V, m, n) with m < max(I))."""
        import scipy.sparse as sp
        shape, ptr, ind, v = self._compress_dense_host(_lib.ROWMAJOR, "to CSR")
        return sp.csr_matrix((v, ind, ptr), shape=shape)

    def to_csc(self):
        """scipy.sparse.csc_matrix of shape size, from the column-major orientation (see to_csr)."""
        import scipy.sparse as sp
        shape, ptr, ind, v = self._compress_dense_host(_lib.COLMAJOR, "to CSC")
        return sp.csc_matrix((v, ind, ptr), shape=shape)

    def to_torch(self, layout=None, device=None):
        """torch sparse CSR (layout=torch.sparse_csr, the default) or CSC (torch.sparse_csc) tensor of shape size with int64
        indices, filled on the device into tensors torch allocates.  The compaction runs after the work already queued on
        torch's current stream, and the tensor is ready on that stream (no host synchronisation, unless entries outside size
        may be stored: then BoundsError is decided before anything is written)."""
        import torch
        layout = torch.sparse_csr if layout is None else layout
        if layout not in (torch.sparse_csr, torch.sparse_csc):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"to_torch: layout must be torch.sparse_csr or torch.sparse_csc, not {layout}")
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if device.type != "cuda":
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"to_torch: the matrix lives on a CUDA device, not {device}")
        which = _lib.ROWMAJOR if layout == torch.sparse_csr else _lib.COLMAJOR
        m, n, dim, idim = self._dense_form(which, "to torch")
        cnt = C.c_int64()
        check(lib().dsa_matrix_compress_dense_d(self._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(0), None, None, None,
                                                C.c_int64(0), C.byref(cnt)))
        nnz = cnt.value
        ptr = torch.empty(dim + 1, dtype=torch.int64, device=device)
        ind = torch.empty(nnz, dtype=torch.int64, device=device)
        v = torch.empty(nnz, dtype=torch.float64, device=device)
        st = C.c_void_p()
        check(lib().dsa_matrix_get_stream(self._h, C.byref(st)))
        # the handle keeps its own stream: order it against torch's both ways (as _mul_dense_cuda does)
        cur = torch.cuda.current_stream(device)
        hs = torch.cuda.ExternalStream(st.value or 0, device=device)
        hs.wait_stream(cur)
        check(lib().dsa_matrix_compress_dense_d(self._h, C.c_int(which), C.c_int64(dim), C.c_int64(idim), C.c_int(0),
                                                C.c_void_p(ptr.data_ptr()), C.c_void_p(ind.data_ptr()), C.c_void_p(v.data_ptr()),
                                                C.c_int64(nnz), C.byref(cnt)))
        cur.wait_stream(hs)
        ctor = torch.sparse_csr_tensor if which == _lib.ROWMAJOR else torch.sparse_csc_tensor
        return ctor(ptr, ind, v, size=(m, n))


def dynamicsparse(I=None, J=None, V=None, m=None, n=None, fill_mode=True, combine="+", row_codec=None, col_codec=None):
    """dynamicsparse(I, J, V, [m, n]) (matrix.jl:15-19) or dynamicsparse(Ti, Tj, Tv; fill_mode) (matrix.jl:31-41)."""
    if I is None:
        if fill_mode:
            return DynamicSparseMatrix(None, fill_mode=True, row_codec=row_codec, col_codec=col_codec)
        h = C.c_void_p()
        check(lib().dsa_matrix_create(C.byref(h)))
        return DynamicSparseMatrix(h, row_codec=row_codec, col_codec=col_codec)
    row_codec, col_codec = row_codec or _codec_for(I), col_codec or _codec_for(J)
    I, J, V = row_codec.encode(I), col_codec.encode(J), _f64(V)
    m = None if m is None else row_codec.encode1(m)
    n = None if n is None else col_codec.encode1(n)
    if not (len(I) == len(J) == len(V)):
        raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "rows, columns, and nonzeros do not have same length.")
    h = C.c_void_p()
    given = m is not None or n is not None
    if given:   # each missing dimension defaults on its own: m = _guess_length(I), n = _guess_length(J)  (matrix.jl:15, vector.jl:6)
        m = int(m) if m is not None else (int(I.max()) if len(I) else 0)
        n = int(n) if n is not None else (int(J.max()) if len(J) else 0)
    check(lib().dsa_matrix_build_coo(_p(I), _p(J), _p(V), C.c_int64(len(I)), C.c_int64(m or 0), C.c_int64(n or 0),
                                     C.c_int(1 if given else 0), C.c_int(_combine(combine)), C.byref(h)))
    return DynamicSparseMatrix(h, row_codec=row_codec, col_codec=col_codec)


def closefillmode(matrix):   # closefillmode! (matrix.jl:126-134)
    if not matrix.fillmode:
        raise ErrorException(_lib.DSA_ERR_ERROR, "Cannot close fill mode because matrix is not in fill mode.")
    I, J, V = matrix.buffer.get_rowids_colids_vals()
    h = C.c_void_p()
    check(lib().dsa_matrix_build_coo(_p(I), _p(J), _p(V), C.c_int64(len(I)), C.c_int64(matrix._m), C.c_int64(matrix._n),
                                     C.c_int(1), C.c_int(_lib.COMBINE["+"]), C.byref(h)))
    matrix._h = h
    matrix.fillmode = False
    matrix.buffer = None
    return True


def addrow(matrix, row, colids, vals):   # addrow! (matrix.jl:113-124)
    if matrix.fillmode:
        # like the reference, addrow! in fill mode does not touch the dimensions (matrix.jl:116-117)
        matrix.buffer.addrow(matrix._rc.encode1(row), matrix._cc.encode(colids), vals)
    else:
        for c, v in zip(colids, vals):
            matrix[row, c] = v
    return True


def _as_list(x):
    return [x] if np.isscalar(x) or isinstance(x, str) else list(x)


def deletecolumn(matrix, col):   # deletecolumn! (matrix.jl:95-102); a list deletes in one bulk call
    matrix._not_fillmode("Cannot delete a column in fill mode")
    matrix.flush()
    ids = matrix._cc.encode(_as_list(col))
    check(lib().dsa_matrix_delete_columns(matrix._h, _p(ids), C.c_int64(len(ids))))
    return True


def deleterow(matrix, row):      # deleterow! (matrix.jl:104-111)
    matrix._not_fillmode("Cannot delete a row in fill mode")
    matrix.flush()
    ids = matrix._rc.encode(_as_list(row))
    check(lib().dsa_matrix_delete_rows(matrix._h, _p(ids), C.c_int64(len(ids))))
    return True


def deletepartition(orientation, key):   # deletepartition!(pcsc, id) (pcsr.jl:188-204) on the PackedCSC facade; a single
    if isinstance(orientation, PackedCSC):   # orientation of a matrix cannot lose a column on its own:
        return orientation.deletepartition(key)
    raise ErrorException(_lib.DSA_ERR_ERROR, "deletepartition! on a single orientation would desynchronise the twin; "
                                             "use deletecolumn / deleterow on the matrix")


def nbpartitions(orientation):   # pcsr.jl:21-22
    if isinstance(orientation, PackedCSC):
        return orientation.nbpartitions
    return orientation.info()["nb_partitions"]


def to_coo(matrix):
    """(rows, cols, vals) of every stored entry (explicit zeros included), column by column in ascending row order: the
    column-major array with gaps and semaphores removed (what iterating the reference's colmajor PMA yields, pcsr.jl:269-283).
    Keys are the device's Int64 keys (encoded if the matrix has codecs)."""
    e = matrix.export(_lib.COLMAJOR)
    occ = np.nonzero(e["tag"])[0]
    key, val = e["key"][occ], e["val"][occ]
    is_sem = key == 0                                         # semaphore cell: value = partition id (pcsr.jl:23, 26-63)
    last_sem = np.maximum.accumulate(np.where(is_sem, np.arange(len(occ)), -1))
    elem = ~is_sem
    part = val[last_sem[elem]].astype(np.int64)               # partition id of the column each element belongs to
    return key[elem], e["col_keys"][part - 1], val[elem]


def save_checkpoint(x, path):
    """Checkpoint of a vector or matrix as a compressed .npz of its entries (SURVEY.md §8f-4).  The content is exact (keys,
    Float64 bits, explicit zeros, dimensions); the gapped layout and deleted-column tombstones are not stored —
    load_checkpoint rebuilds the canonical bulk-build layout, which is what the reference's own constructors produce."""
    if isinstance(x, DynamicSparseVector):
        k, v = x._raw_nonzeros()
        np.savez_compressed(path, kind="vector", keys=k, vals=v, n=len(x))
    elif isinstance(x, DynamicSparseMatrix):
        x._not_fillmode("Cannot checkpoint a matrix in fill mode")
        I, J, V = to_coo(x)
        m, n = x._dims()
        ec, er = x.export(_lib.COLMAJOR), x.export(_lib.ROWMAJOR)
        # live partitions, empty ones included (a column created by a zero write, or emptied entry by entry, stays a live
        # partition: nbpartitions and deletecolumn! see it, test/functional/sparsematrix.jl:266-268)
        np.savez_compressed(path, kind="matrix", rows=I, cols=J, vals=V, m=m, n=n,
                            live_cols=ec["col_keys"][ec["col_live"].astype(bool)], live_rows=er["col_keys"][er["col_live"].astype(bool)])
    else:
        raise TypeError(type(x))


def load_checkpoint(path, key_codec=None, row_codec=None, col_codec=None):
    path = str(path)
    if not path.endswith(".npz") and not os.path.exists(path):   # np.savez appends the suffix on save
        path += ".npz"
    z = np.load(path)
    if str(z["kind"]) == "vector":
        return dynamicsparsevec(z["keys"], z["vals"], n=int(z["n"]), key_codec=key_codec, _encoded=True)
    h = C.c_void_p()
    I, J, V = _i64(z["rows"]), _i64(z["cols"]), _f64(z["vals"])
    check(lib().dsa_matrix_build_coo(_p(I), _p(J), _p(V), C.c_int64(len(I)), C.c_int64(int(z["m"])), C.c_int64(int(z["n"])),
                                     C.c_int(1), C.c_int(_lib.COMBINE["+"]), C.byref(h)))
    A = DynamicSparseMatrix(h, row_codec=row_codec, col_codec=col_codec)
    if "live_cols" in z.files:   # re-create the live partitions that hold no entry: a zero write creates its column / row
        lc, lr = _i64(z["live_cols"]), _i64(z["live_rows"])   # (pcsr.jl:341-347 calls addcolumn! before looking at the value)
        ec = np.setdiff1d(lc, np.unique(J))
        er = np.setdiff1d(lr, np.unique(I))
        if len(ec) and len(lr):
            check(lib().dsa_matrix_set_batch(A._h, _p(np.full(len(ec), lr[0], np.int64)), _p(ec), _p(np.zeros(len(ec))), C.c_int64(len(ec))))
        if len(er) and len(lc):
            check(lib().dsa_matrix_set_batch(A._h, _p(er), _p(np.full(len(er), lc[0], np.int64)), _p(np.zeros(len(er))), C.c_int64(len(er))))
    return A


class PackedCSC:
    """The reference's partition-id addressed PackedCSC (pcsr.jl:4-63): `pcsc[key, partition]`, partitions numbered 1..n in
    creation order, empty partitions allowed, deleting a partition is irreversible (pcsr.jl:188-204, 294-310).

    The device has no separate entry point for it — every caller in the reference goes through MappedPackedCSC — so this is a
    facade over a DynamicSparseMatrix whose column key IS the partition id: what the facade adds is the host-side bookkeeping
    that distinguishes the two types (creation of all partitions up to the written id, `_add_partitions!` pcsr.jl:312-319; the
    error on a deleted partition, pcsr.jl:299)."""

    def __init__(self, keys=None, values=None, combine="+", _matrix=None, _nparts=0, _deleted=()):
        if _matrix is not None:
            self._m, self._nparts, self._deleted = _matrix, _nparts, set(_deleted)
            return
        keys, values = keys or [], values or []
        if len(keys) != len(values):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "keys & values must have same length.")
        I = [k for part in keys for k in part]
        J = [p + 1 for p, part in enumerate(keys) for _ in part]
        V = [v for part in values for v in part]
        if len(I) != len(V):
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, "keys & values must have same length.")
        self._m = dynamicsparse(I, J, V, combine=combine) if I else dynamicsparse(fill_mode=False)
        self._nparts, self._deleted = 0, set()
        self._ensure_partitions(len(keys), existing={p + 1 for p, part in enumerate(keys) if len(part)})

    def _ensure_partitions(self, upto, existing=()):
        """partitions nparts+1 .. upto exist afterwards (empty unless `existing`): a zero write creates the column (pcsr.jl:341-347)"""
        for p in range(self._nparts + 1, upto + 1):
            if p not in existing:
                self._m[1, p] = 0.0
        self._nparts = max(self._nparts, upto)

    def __setitem__(self, idx, val):   # pcsr.jl:294-310
        key, part = idx
        if part in self._deleted:
            raise ErrorException(_lib.DSA_ERR_ERROR, f"The partition {part} has been deleted.")
        self._ensure_partitions(part - 1)
        self._m[key, part] = val
        self._nparts = max(self._nparts, part)

    def __getitem__(self, idx):        # pcsr.jl:222-291
        key, part = idx
        if isinstance(key, slice):
            return self._m[:, part]
        if isinstance(part, slice):
            return self._m[key, :]
        return self._m[key, part]

    def deletepartition(self, part):   # pcsr.jl:188-204
        if part < 1 or part > self._nparts:
            raise _lib.BoundsError(_lib.DSA_ERR_BOUNDS, f"partition {part} out of bounds 1:{self._nparts}")
        if part in self._deleted:
            raise ArgumentError(_lib.DSA_ERR_ARGUMENT, f"partition {part} does not exist.")
        deletecolumn(self._m, part)
        self._deleted.add(part)
        return True

    @property
    def nbpartitions(self):            # pcsr.jl:21
        return self._nparts - len(self._deleted)

    @property
    def nnz(self):                     # pcsr.jl:11
        return nnz(self._m)

    ndim = 2

    def __deepcopy__(self, memo):      # PackedCSC(pcsc) (pcsr.jl:65-71)
        import copy
        return PackedCSC(_matrix=copy.deepcopy(self._m), _nparts=self._nparts, _deleted=self._deleted)


def nnz(x):   # pma.jl:163, pcsr.jl:11, matrix.jl:91
    if isinstance(x, DynamicSparseVector):
        return x.info()["nnz"]
    if isinstance(x, DynamicSparseMatrix):
        return x.info(_lib.ROWMAJOR)["nnz"]
    if isinstance(x, _Orientation):
        return x.info()["nnz"]
    if isinstance(x, SparseVector):
        return len(x.nzind)
    if isinstance(x, PackedCSC):
        return x.nnz
    raise TypeError(type(x))
