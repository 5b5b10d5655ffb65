"""The StrHashMap key path of the oracle (tests/oracle_strhash.c) against the reference's own known answers (TestIterator,
pkg/common/hashmap/strhashmap_test.go:60-136, transcribed into tests/golden/strhash_kat.json) and hand-checked byte layouts of
encodeHashKeys (strhashmap.go:92-385).  CPU only."""
import json
import struct

import numpy as np

from matrixone_b200.vector import bitmap_from_bools
import oracle_lib as O
from strhash_util import GOLDEN, OracleStrTable, kat_columns, oracle_find, oracle_pack, strhash, varchar


def test_oracle_reproduces_test_iterator():
    kat = json.load(open(GOLDEN))
    assert len(kat["cases"]) == 3
    for case in kat["cases"]:
        cols, kinds, nulls = kat_columns(case, kat["rows"])
        off, kb, skip = oracle_pack(cols, kinds, nulls, case["has_null"])
        t = OracleStrTable(64, 4096)
        ids = t.insert(off, kb, skip)
        assert ids.tolist() == case["want_ids"]
        toff, tb = t.table()
        assert oracle_find(toff, tb, off, kb, skip).tolist() == case["want_ids"]      # Find returns what Insert did


def _pack1(rows_of_cols, kinds, has_null=True, nulls=None, const=None):
    off, kb, skip = oracle_pack(rows_of_cols, kinds, nulls, has_null, const)
    return [kb[off[i]:off[i + 1]].tobytes() for i in range(len(off) - 1)], skip


def pad(b):
    return b + bytes(max(0, 16 - len(b)))


def test_split_strings_get_different_keys():
    for has_null in (True, False):
        keys, _ = _pack1([varchar(["a", "ab"]), varchar(["bc", "c"])], [0, 0], has_null)
        assert keys[0] != keys[1]
        t = OracleStrTable(8, 256)
        off = np.array([0, len(keys[0]), len(keys[0]) + len(keys[1])], np.int64)
        assert t.insert(off, np.frombuffer(keys[0] + keys[1], np.uint8)).tolist() == [1, 2]


def test_byte_layouts():
    # fixed width, has_null: marker 0 + value bytes; NULL: marker 1 only; then zero padding to 16
    keys, _ = _pack1([np.array([0x0102, 7], np.int16), np.array([5, 6], np.int8)], [2, 1], True, [bitmap_from_bools([False, True]), None])
    assert keys[0] == pad(b"\x00\x02\x01" + b"\x00\x05")
    assert keys[1] == pad(b"\x01" + b"\x00\x06")
    # fixed width, no has_null: value bytes only; a NULL skips the row and appends nothing for that column
    keys, skip = _pack1([np.array([0x0102, 7], np.int16), np.array([5, 6], np.int8)], [2, 1], False, [bitmap_from_bools([False, True]), None])
    assert keys[0] == pad(b"\x02\x01\x05") and keys[1] == pad(b"\x06")
    assert int(skip[0]) == 0b10
    # varlena, has_null: marker 0 + uint16 length + bytes; NULL: marker 1
    keys, _ = _pack1([varchar(["hello", ""])], [0], True, [bitmap_from_bools([False, True])])
    assert keys[0] == pad(b"\x00\x05\x00hello") and keys[1] == pad(b"\x01")
    # varlena, no has_null, a value in the area (> 23 bytes): uint16 length + bytes, no padding past 16
    s = b"x" * 30
    keys, _ = _pack1([varchar([s])], [0], False)
    assert keys[0] == struct.pack("<H", 30) + s
    # const vector repeats element 0; const NULL: marker 1 (has_null) or every row skipped
    keys, _ = _pack1([np.array([1, 2, 3], np.int32), np.array([9], np.int64)], [4, 8], True, None, [False, True])
    assert keys[2] == b"\x00\x03\x00\x00\x00" + b"\x00" + struct.pack("<q", 9) + bytes(2)
    keys, _ = _pack1([np.array([1, 2], np.int32), np.array([9], np.int64)], [4, 8], True, [None, np.array([1], np.uint64)], [False, True])
    assert keys[1] == pad(b"\x00\x02\x00\x00\x00\x01")
    keys, skip = _pack1([np.array([1, 2], np.int32), np.array([9], np.int64)], [4, 8], False, [None, np.array([1], np.uint64)], [False, True])
    assert int(skip[0]) == 0b11 and keys[0] == pad(b"\x01\x00\x00\x00")
    # a 16-byte fixed width (Decimal128) and a 24-byte one (Rowid) are copied whole
    d = np.arange(4, dtype=np.uint64).reshape(2, 2)
    keys, _ = _pack1([d], [16], False)
    assert keys[1] == d[1].tobytes()


def test_length_over_65535_wraps():
    s = bytes(range(256)) * 257                        # 65792 bytes
    keys, _ = _pack1([varchar([s])], [0], True)
    assert keys[0][:3] == b"\x00" + struct.pack("<H", len(s) & 0xFFFF)
    assert keys[0][3:] == s and len(keys[0]) == 3 + len(s)


def test_overflow_leaves_the_table_unchanged():
    keys = [pad(b"k%d" % i) for i in range(10)]
    off = np.concatenate([[0], np.cumsum([len(k) for k in keys])]).astype(np.int64)
    kb = np.frombuffer(b"".join(keys), np.uint8)
    t = OracleStrTable(4, 1024)
    t.insert(off[:3] - 0, kb[:off[2]])
    before = (t.toff.copy(), t.tbytes.copy(), t.ngroups)
    need = np.zeros(2, np.int64); groups = np.zeros(10, np.uint64)
    r = strhash().og_str_group_ids(O.p(off), O.p(kb), None, 10, O.p(groups), O.p(t.toff), O.p(t.tbytes), t.ngroups, 4, 1024, O.p(need))
    assert r == -1 and need.tolist() == [10, 160]
    assert (t.toff == before[0]).all() and (t.tbytes == before[1]).all()
