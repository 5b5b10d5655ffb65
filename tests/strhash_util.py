"""Helpers shared by the StrHashMap tests (TEST INFRASTRUCTURE): key columns in MatrixOne layout, and the C restatement of the key path
(tests/oracle_strhash.c: og_pack_str_keys, og_str_group_ids, og_str_join_find) with calls in the shape of ops.pack_str_keys / StrGroupTable."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_lib as O
from matrixone_b200.vector import bitmap_from_bools, varlena_column

_vp, _i32, _i64 = C.c_void_p, C.c_int32, C.c_int64
_lib = None


def strhash():
    """tests/oracle_strhash.c compiled with the oracle's flags (oracle/build.py) into the temp directory on first use (the checkout may be
    read-only); the file name carries a digest of the source, so an edited source is rebuilt"""
    global _lib
    if _lib is None:
        src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_strhash.c")
        tag = hashlib.sha1(open(src, "rb").read()).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), "mo_b200_oracle_strhash_%s_%d.so" % (tag, os.getuid()))
        if not os.path.exists(out):
            tmp = out + ".%d.tmp" % os.getpid()
            subprocess.run(["gcc", "-std=gnu11", "-O2", "-fno-fast-math", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-o", tmp, src],
                           check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
            os.replace(tmp, out)
        lib = C.CDLL(out)
        lib.og_pack_str_keys.restype = _i64
        lib.og_pack_str_keys.argtypes = [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp]
        lib.og_str_group_ids.restype = _i64
        lib.og_str_group_ids.argtypes = [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _i64, _i64, _vp]
        lib.og_str_join_find.restype = None
        lib.og_str_join_find.argtypes = [_vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp]
        _lib = lib
    return _lib

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "strhash_kat.json")
NP = {1: np.int8, 2: np.int16, 4: np.int32, 8: np.int64}


def kat_columns(case, rows):
    cols, kinds = [], []
    for c in case["columns"]:
        if c["width"]:
            cols.append(np.arange(rows, dtype=NP[c["width"]]))
        else:
            cols.append(varchar([str(i) for i in range(rows)]))
        kinds.append(c["width"])
    nulls = None
    if case["null_rows"]:
        nb = bitmap_from_bools(np.isin(np.arange(rows), case["null_rows"]))
        nulls = [nb] * len(cols)
    return cols, kinds, nulls


def varchar(values):
    """(cells uint8[24 * n], area) for a list of bytes / str values"""
    rows = [np.frombuffer(v.encode() if isinstance(v, str) else bytes(v), dtype=np.uint8) for v in values]
    return varlena_column(rows, dtype=np.uint8)


def oracle_pack(cols, kinds, nulls=None, has_null=True, const=None, n=None):
    """og_pack_str_keys over the same column description as ops.pack_str_keys: (offsets, bytes, skip words or None)"""
    ncols = len(cols)
    const = const or [False] * ncols
    keep, data, areas, nls = [], [], [], []
    for k, c in enumerate(cols):
        if kinds[k]:
            d, a = np.ascontiguousarray(c).view(np.uint8).reshape(-1), None
        else:
            d, a = np.ascontiguousarray(c[0], dtype=np.uint8), np.ascontiguousarray(c[1], dtype=np.uint8)
            if a.size == 0:
                a = np.zeros(1, np.uint8)
        if n is None and not const[k]:
            n = d.nbytes // (kinds[k] or 24)
        nb = None if nulls is None or nulls[k] is None else np.ascontiguousarray(nulls[k], dtype=np.uint64)
        keep += [d, a, nb]
        data.append(O.p(d)); areas.append(O.p(a)); nls.append(O.p(nb))
    n = 1 if n is None else n
    P = lambda xs: (C.c_void_p * ncols)(*xs)
    width = np.asarray(kinds, dtype=np.int32)
    cst = np.asarray([1 if c else 0 for c in const], dtype=np.int32)
    offsets = np.zeros(n + 1, dtype=np.int64)
    skip = None if has_null else np.zeros(max((n + 63) // 64, 1), dtype=np.uint64)
    need = strhash().og_pack_str_keys(ncols, 1 if has_null else 0, O.p(width), P(data), P(areas), P(nls), O.p(cst), n, O.p(offsets), None, 0, O.p(skip))
    out = np.zeros(max(need, 1), dtype=np.uint8)
    strhash().og_pack_str_keys(ncols, 1 if has_null else 0, O.p(width), P(data), P(areas), P(nls), O.p(cst), n, O.p(offsets), O.p(out), need, O.p(skip))
    return offsets, out[:need], (skip[:(n + 63) // 64] if skip is not None else None)


class OracleStrTable:
    """og_str_group_ids with a persisted table"""

    def __init__(self, capacity, byte_capacity):
        self.toff = np.zeros(capacity + 1, np.int64)
        self.tbytes = np.zeros(max(byte_capacity, 1), np.uint8)
        self.ngroups = 0

    def insert(self, offsets, key_bytes, skip=None):
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        kb = np.ascontiguousarray(key_bytes, dtype=np.uint8)
        n = off.shape[0] - 1
        groups = np.zeros(n, np.uint64)
        need = np.zeros(2, np.int64)
        sk = None if skip is None else np.ascontiguousarray(skip, dtype=np.uint64)
        r = strhash().og_str_group_ids(O.p(off), O.p(kb) if kb.size else None, O.p(sk), n, O.p(groups), O.p(self.toff), O.p(self.tbytes), self.ngroups,
                                         self.toff.shape[0] - 1, self.tbytes.shape[0], O.p(need))
        assert r >= 0, "oracle table too small"
        self.ngroups = int(r)
        return groups

    def table(self):
        return self.toff[:self.ngroups + 1].copy(), self.tbytes[:int(self.toff[self.ngroups]) if self.ngroups else 0].copy()


def oracle_find(toff, tbytes, offsets, key_bytes, skip=None):
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    kb = np.ascontiguousarray(key_bytes, dtype=np.uint8)
    n = off.shape[0] - 1
    vals = np.zeros(n, np.uint64)
    sk = None if skip is None else np.ascontiguousarray(skip, dtype=np.uint64)
    tb = np.ascontiguousarray(tbytes, dtype=np.uint8)
    strhash().og_str_join_find(O.p(np.ascontiguousarray(toff, dtype=np.int64)), O.p(tb) if tb.size else None, len(toff) - 1,
                                 O.p(off), O.p(kb) if kb.size else None, O.p(sk), n, O.p(vals))
    return vals


def dict_ids(offsets, key_bytes, skip_rows=None, seen=None):
    """first-seen ids from a Python dict over the key bytes (seen persists across batches)"""
    seen = {} if seen is None else seen
    kb = bytes(np.ascontiguousarray(key_bytes, dtype=np.uint8))
    out = np.zeros(len(offsets) - 1, np.uint64)
    for i in range(len(offsets) - 1):
        if skip_rows is not None and skip_rows[i]:
            continue
        k = kb[offsets[i]:offsets[i + 1]]
        g = seen.get(k)
        if g is None:
            g = seen[k] = len(seen) + 1
        out[i] = g
    return out, seen
