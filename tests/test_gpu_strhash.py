"""The StrHashMap path on the GPU (csrc/strhash.cu): PACK_STR_KEYS byte for byte against og_pack_str_keys (encodeHashKeys,
strhashmap.go:92-385), STR_GROUP_IDS against the reference's TestIterator answers and first-seen ids of a Python dict over the key bytes,
STR_JOIN_FIND / STR_JOIN_PROBE against the oracle's Find and emission loop (hashjoin/join.go:383-628), and a varchar + int32 GROUP BY
through GROUP_AGG against og_sum_int64 / og_count."""
import json

import numpy as np
import pytest

import oracle_lib as O
from matrixone_b200 import capi, ops
from matrixone_b200.vector import DeviceBuffer, Vector, bitmap_from_bools, bitmap_to_bools, xcall
from strhash_util import GOLDEN, OracleStrTable, dict_ids, kat_columns, oracle_find, oracle_pack, varchar

pytestmark = pytest.mark.gpu


def inline_varchar(strings):
    """(cells, empty area) for values of at most 23 bytes, vectorised"""
    s = np.asarray(strings, dtype="S")
    n, w = s.shape[0], s.dtype.itemsize
    assert w <= 23
    cells = np.zeros((n, 24), np.uint8)
    cells[:, 0] = np.char.str_len(s)
    cells[:, 1:1 + w] = s.view(np.uint8).reshape(n, w)
    return cells.reshape(-1), np.zeros(0, np.uint8)


def random_columns(rng, n, ncols, has_null):
    """a mix of every column kind: fixed widths 1/2/4/8/16/24, inline and area varlena, const, const NULL, nullable"""
    kinds_pool = [1, 2, 4, 8, 16, 24, 0, 0]
    cols, kinds, nulls, const = [], [], [], []
    for k in range(ncols):
        w = kinds_pool[k % len(kinds_pool)]
        is_const = k % 5 == 4
        rows = 1 if is_const else n
        if w:
            cols.append(rng.integers(0, 256, rows * w, dtype=np.uint8))
        else:
            lens = rng.integers(0, 24, rows) if k % 2 == 0 else np.where(rng.random(rows) < 0.02, rng.integers(24, 4097, rows), rng.integers(24, 80, rows))
            cols.append(varchar([rng.integers(0, 256, l, dtype=np.uint8).tobytes() for l in lens]))
        kinds.append(w)
        const.append(is_const)
        if is_const:
            nulls.append(np.array([1 if k % 10 == 9 else 0], np.uint64))          # every other const column is a const NULL
        else:
            nulls.append(bitmap_from_bools(rng.random(rows) < 0.1) if k % 3 != 1 else None)
    return cols, kinds, nulls, const


@pytest.mark.parametrize("n", [0, 1, 63, 64, 65, 100_003])
@pytest.mark.parametrize("has_null", [True, False])
def test_pack_is_byte_exact(gpu, n, has_null):
    rng = np.random.default_rng(n * 2 + has_null)
    cols, kinds, nulls, const = random_columns(rng, n, 10, has_null)
    off, kb, skip = ops.pack_str_keys(cols, kinds, nulls, has_null, const, length=n)
    woff, wkb, wskip = oracle_pack(cols, kinds, nulls, has_null, const, n)
    assert np.array_equal(off, woff)
    assert kb.tobytes() == wkb.tobytes()
    if not has_null and n:
        assert np.array_equal(bitmap_to_bools(skip, n), bitmap_to_bools(wskip, n))


@pytest.mark.parametrize("ncols", [1, 2, 7, 16])
def test_pack_column_counts(gpu, ncols):
    rng = np.random.default_rng(ncols)
    for has_null in (True, False):
        cols, kinds, nulls, const = random_columns(rng, 1000, ncols, has_null)
        off, kb, skip = ops.pack_str_keys(cols, kinds, nulls, has_null, const, length=1000)
        woff, wkb, _ = oracle_pack(cols, kinds, nulls, has_null, const, 1000)
        assert np.array_equal(off, woff) and kb.tobytes() == wkb.tobytes()


def test_pack_value_over_65535_bytes(gpu):
    big = bytes(range(256)) * 300                               # 76800 bytes: the uint16 length wraps, every byte is kept
    vals = [b"a", big, b"x" * 40, b""]
    for has_null in (True, False):
        off, kb, _ = ops.pack_str_keys([varchar(vals), np.arange(4, dtype=np.int32)], [0, 4], has_null=has_null)
        woff, wkb, _ = oracle_pack([varchar(vals), np.arange(4, dtype=np.int32)], [0, 4], None, has_null)
        assert np.array_equal(off, woff) and kb.tobytes() == wkb.tobytes()
        assert off[2] - off[1] == (3 + len(big) + 1 + 4 if has_null else 2 + len(big) + 4)    # marker + uint16 + bytes, then the int32 column


def test_pack_capacity_protocol(gpu):
    cols = [varchar(["k%05d" % i for i in range(500)]), np.arange(500, dtype=np.int64)]
    woff, wkb, _ = oracle_pack(cols, [0, 8], None, True)
    offsets = np.zeros(501, np.int64)
    small = np.zeros(100, np.uint8)
    prm = capi.StrKeyParams(2, 1)
    prm.width[0], prm.width[1] = 0, 8
    vecs = [Vector(data=offsets, length=500), Vector(data=small, length=100), ops._params_vec(prm),
            Vector(data=cols[0][0], area=cols[0][1], length=500), Vector(data=cols[1].view(np.uint8), length=500)]
    rc, _ = xcall(capi.XCALL_PACK_STR_KEYS, vecs, 500, raise_on_error=False)
    assert rc == capi.RC_OUT_OF_RANGE and offsets[500] == len(wkb)
    with pytest.raises(capi.MoError):
        ops.pack_str_keys(cols, [0, 8], capacity=100)
    off, kb, _ = ops.pack_str_keys(cols, [0, 8])               # grows to offsets[n] and repeats
    assert kb.tobytes() == wkb.tobytes()


def test_group_ids_test_iterator(gpu):
    kat = json.load(open(GOLDEN))
    for case in kat["cases"]:
        cols, kinds, nulls = kat_columns(case, kat["rows"])
        off, kb, skip = ops.pack_str_keys(cols, kinds, nulls, case["has_null"])
        tab = ops.StrGroupTable(16, 1024)
        assert tab.insert(off, kb, skip).tolist() == case["want_ids"]
        jm = ops.StrJoinMap(off, kb, skip)
        assert jm.find(off, kb, skip).tolist() == case["want_ids"]
        jm.release()


def _keys(ids, salt=0):
    """varchar("k<id>") + int32 key columns for group ids"""
    return [inline_varchar(np.char.mod("k%d", ids)), ((ids * 7 + salt) % 1000).astype(np.int32)], [0, 4]


@pytest.mark.parametrize("card", [1, 37, 10_000, 1_000_000])
def test_group_ids_first_seen_across_batches(gpu, card):
    rng = np.random.default_rng(card)
    tab = ops.StrGroupTable(64, 1024)                          # small on purpose: the batches make it grow
    seen = None
    nb = 3 if card < 1_000_000 else 2
    for b in range(nb):
        n = 300_000 if card < 1_000_000 else 700_000
        ids = rng.integers(0, card, n)
        cols, kinds = _keys(ids)
        nulls = [bitmap_from_bools(rng.random(n) < 0.01), None]
        off, kb, skip = ops.pack_str_keys(cols, kinds, nulls, has_null=(b % 2 == 0))
        got = tab.insert(off, kb, skip)
        want, seen = dict_ids(off, kb, bitmap_to_bools(skip, n) if skip is not None else None, seen)
        assert np.array_equal(got, want)
    assert tab.ngroups == len(seen)
    toff, tb = tab.table()
    assert [tb[toff[g]:toff[g + 1]].tobytes() for g in range(min(tab.ngroups, 1000))] == list(seen)[:1000]


def test_group_ids_near_duplicates(gpu):
    rng = np.random.default_rng(3)
    prefix = b"p" * 700
    vals = [prefix + bytes([i & 255, i >> 8]) for i in range(2000)] + [b"abc%d" % (i % 256) + bytes([i % 7]) for i in range(3000)]
    order = rng.permutation(len(vals))
    vals = [vals[i] for i in order] * 2
    off, kb, _ = ops.pack_str_keys([varchar(vals)], [0], has_null=False)
    got = ops.StrGroupTable(16, 256).insert(off, kb)
    want, seen = dict_ids(off, kb)
    assert np.array_equal(got, want) and len(seen) == 2000 + 256 * 7


def test_group_ids_overflow_protocol(gpu):
    ids = np.arange(5000) % 1234
    cols, kinds = _keys(ids)
    off, kb, _ = ops.pack_str_keys(cols, kinds)
    want, seen = dict_ids(off, kb)
    first = ops.StrGroupTable(2000, 1 << 20)
    assert np.array_equal(first.insert(off[:1001], kb[:off[1000]]), want[:1000])
    state0 = first.state.copy()
    groups = np.zeros(5000, np.uint64)
    small_off, small_b = first.offsets[:1001].copy(), first.bytes[:int(state0[1]) + 100].copy()
    small_off_before, small_b_before = small_off.copy(), small_b.copy()
    st = state0.copy()
    vecs = [Vector(data=groups, length=5000), Vector(data=st, length=4), Vector(data=small_off, length=1001), Vector(data=small_b, length=len(small_b)),
            Vector(data=off, length=5000), Vector(data=kb, length=len(kb))]
    rc, _ = xcall(capi.XCALL_STR_GROUP_IDS, vecs, 5000, raise_on_error=False)
    assert rc == capi.RC_OUT_OF_RANGE
    assert st[0] == state0[0] and st[1] == state0[1] and st[2] == len(seen)
    assert st[3] == sum(len(k) for k in seen)
    assert np.array_equal(small_off, small_off_before) and np.array_equal(small_b, small_b_before)
    # StrGroupTable grows and repeats: the same ids as one large call
    grow = ops.StrGroupTable(8, 64)
    got = np.concatenate([grow.insert(off[:1001], kb[:off[1000]]), grow.insert(off[1000:] - off[1000], kb[off[1000]:])])
    assert np.array_equal(got, want)
    one = ops.StrGroupTable(5000, 1 << 20).insert(off, kb)
    assert np.array_equal(one, want)


def test_resident_group_ids(gpu):
    n = 200_000
    ids = np.random.default_rng(9).integers(0, 5000, n)
    cols, kinds = _keys(ids)
    woff, wkb, _ = oracle_pack(cols, kinds, None, False)
    d_cells, d_int = DeviceBuffer.from_numpy(cols[0][0]), DeviceBuffer.from_numpy(cols[1])
    d_off, d_kb = DeviceBuffer(8 * (n + 1)), DeviceBuffer(len(wkb))
    prm = capi.StrKeyParams(2, 0)
    prm.width[0], prm.width[1] = 0, 4
    xcall(capi.XCALL_PACK_STR_KEYS, [Vector(data_ptr=d_off.ptr, data_nbytes=d_off.nbytes, length=n), Vector(data_ptr=d_kb.ptr, data_nbytes=d_kb.nbytes, length=n),
                                     ops._params_vec(prm), Vector(data_ptr=d_cells.ptr, data_nbytes=d_cells.nbytes, length=n),
                                     Vector(data_ptr=d_int.ptr, data_nbytes=d_int.nbytes, length=n)], n)
    assert np.array_equal(d_off.to_numpy(np.int64), woff) and d_kb.to_numpy(np.uint8).tobytes() == wkb.tobytes()
    d_groups, d_state = DeviceBuffer(8 * n), DeviceBuffer.from_numpy(np.zeros(4, np.int64))
    d_toff, d_tb = DeviceBuffer.from_numpy(np.zeros(5001, np.int64)), DeviceBuffer(5000 * 64)
    xcall(capi.XCALL_STR_GROUP_IDS, [Vector(data_ptr=d_groups.ptr, data_nbytes=d_groups.nbytes, length=n), Vector(data_ptr=d_state.ptr, data_nbytes=32, length=4),
                                     Vector(data_ptr=d_toff.ptr, data_nbytes=d_toff.nbytes, length=5001), Vector(data_ptr=d_tb.ptr, data_nbytes=d_tb.nbytes, length=1),
                                     Vector(data_ptr=d_off.ptr, data_nbytes=d_off.nbytes, length=n), Vector(data_ptr=d_kb.ptr, data_nbytes=d_kb.nbytes, length=n)], n)
    want, seen = dict_ids(woff, wkb)
    assert np.array_equal(d_groups.to_numpy(np.uint64), want)
    st = d_state.to_numpy(np.int64)
    assert st[0] == len(seen) and st[1] == sum(len(k) for k in seen)
    toff = d_toff.to_numpy(np.int64)[:len(seen) + 1]
    tb = d_tb.to_numpy(np.uint8)
    assert b"".join(seen) == tb[:toff[-1]].tobytes()
    for b in (d_cells, d_int, d_off, d_kb, d_groups, d_state, d_toff, d_tb):
        b.free()


def _oracle_str_join(boff, bkb, bskip, poff, pkb, pskip, jt):
    nb = len(boff) - 1
    t = OracleStrTable(max(nb, 1), max(int(boff[-1]), 1))
    ids = t.insert(boff, bkb, bskip)
    toff, tb = t.table()
    ng = t.ngroups
    offsets = np.zeros(ng + 2, np.int32); sels = np.zeros(max(nb, 1), np.int32)
    m = O.go().og_join_sels(O.p(ids), nb, ng, O.p(offsets), O.p(sels))
    vals = oracle_find(toff, tb, poff, pkb, pskip)
    unique = ng == nb
    npr = len(poff) - 1
    cap = npr * 8 + nb * 4 + 1024
    while True:
        op, ob = np.zeros(cap, np.int64), np.zeros(cap, np.int64)
        r = O.go().og_join_probe(O.p(vals), npr, None if unique else O.p(offsets), None if unique else O.p(sels), jt, O.p(op), O.p(ob), cap)
        if r <= cap:
            return toff, tb, offsets, sels[:m], vals, op[:r], ob[:r]
        cap = r


@pytest.mark.parametrize("nbuild,card,nprobe", [(1, 1, 5), (1000, 1000, 3000), (5000, 37, 2000), (200_000, 50_000, 300_000), (70_000, 3, 100), (100_000, 100_000, 100_000)])
@pytest.mark.parametrize("jt", [capi.JOIN_INNER, capi.JOIN_LEFT, capi.JOIN_SEMI, capi.JOIN_ANTI])
def test_str_join_matches_the_reference_emission_order(gpu, nbuild, card, nprobe, jt):
    rng = np.random.default_rng(nbuild * 7 + card + jt)
    pool = rng.permutation(card * 4)[:card]
    bids = rng.permutation(pool) if card == nbuild else pool[rng.integers(0, card, nbuild)]
    pids = np.where(rng.random(nprobe) < 0.6, pool[rng.integers(0, card, nprobe)], rng.integers(card * 4, card * 8 + 10, nprobe))
    bcols, kinds = _keys(bids)
    pcols, _ = _keys(pids)
    bnull = [bitmap_from_bools(rng.random(nbuild) < 0.05), None] if nbuild > 10 else None
    pnull = [None, bitmap_from_bools(rng.random(nprobe) < 0.05)]
    boff, bkb, bskip = ops.pack_str_keys(bcols, kinds, bnull, has_null=False)     # join keys: a NULL never matches (zValues = 0)
    poff, pkb, pskip = ops.pack_str_keys(pcols, kinds, pnull, has_null=False)
    toff, tb, offsets, sels, vals, op, ob = _oracle_str_join(boff, bkb, bskip, poff, pkb, pskip, jt)
    jm = ops.StrJoinMap(boff, bkb, bskip, prepare=(nbuild % 2 == 0))
    assert jm.ngroups == len(toff) - 1 and np.array_equal(jm.key_offsets, toff) and jm.key_bytes.tobytes() == tb.tobytes()
    if jm.ngroups != nbuild:
        assert not jm.hash_on_unique()
        assert np.array_equal(jm.offsets, offsets) and np.array_equal(jm.sels, sels)
    assert np.array_equal(jm.find(poff, pkb, pskip), vals)
    gp, gb = jm.probe(poff, pkb, jt, pskip)
    assert len(gp) == len(op) and np.array_equal(gp, op) and np.array_equal(gb, ob)
    jm.release()


def test_str_join_capacity_and_empty_sides(gpu):
    bvals = ["hot"] * 5000 + ["warm"] * 33 + ["k%d" % i for i in range(2000)]
    boff, bkb, _ = ops.pack_str_keys([varchar(bvals)], [0])
    poff, pkb, _ = ops.pack_str_keys([varchar(["hot", "warm", "none", "hot", "k5"])], [0])
    _, _, _, _, _, op, ob = _oracle_str_join(boff, bkb, None, poff, pkb, None, capi.JOIN_LEFT)
    jm = ops.StrJoinMap(boff, bkb)
    gp, gb = jm.probe(poff, pkb, capi.JOIN_LEFT)                 # the default capacity is too small: the count comes back and the call is repeated
    assert np.array_equal(gp, op) and np.array_equal(gb, ob) and len(gp) > 10_000
    with pytest.raises(capi.MoError):
        jm.probe(poff, pkb, capi.JOIN_INNER, capacity=100)
    jm.release()
    empty = ops.StrJoinMap(np.zeros(1, np.int64), np.zeros(0, np.uint8))
    p, b = empty.probe(poff, pkb, capi.JOIN_LEFT)
    assert np.array_equal(p, np.arange(5)) and (b == -1).all()
    assert len(empty.probe(poff, pkb, capi.JOIN_INNER)[0]) == 0


def test_group_by_varchar_int_sum_count(gpu):
    rng = np.random.default_rng(11)
    n = 300_000
    ids = rng.integers(0, 20_000, n)
    cols, kinds = _keys(ids, salt=3)
    nulls = [bitmap_from_bools(rng.random(n) < 0.02), bitmap_from_bools(rng.random(n) < 0.02)]
    val = rng.integers(-1000, 1000, n).astype(np.int32)
    vnull = bitmap_from_bools(rng.random(n) < 0.05)
    off, kb, skip = ops.pack_str_keys(cols, kinds, nulls, has_null=True)              # GROUP BY keeps NULL keys as their own groups
    groups = ops.StrGroupTable(1024, 1 << 16).insert(off, kb, skip)
    woff, wkb, _ = oracle_pack(cols, kinds, nulls, True)
    oids = OracleStrTable(n, len(wkb)).insert(woff, wkb)
    assert np.array_equal(groups, oids)
    ng = int(oids.max())
    want = np.zeros(ng, np.int64); wnull = np.ones(ng, np.uint8); wcnt = np.zeros(ng, np.int64)
    assert O.go().og_sum_int64(capi.T_INT32, O.p(val), O.p(vnull), 0, O.p(oids), n, O.p(want), O.p(wnull), O.p(wcnt), None) == 0
    state = np.zeros(ng, np.int64); snull = bitmap_from_bools(np.ones(ng, bool))
    assert ops.group_agg(capi.AGG_SUM, capi.T_INT32, state, snull, None, groups, val, vnull) == 0
    live = wnull == 0
    assert np.array_equal(bitmap_to_bools(snull, ng), ~live) and np.array_equal(state[live], want[live])
    wc = np.zeros(ng, np.int64)
    O.go().og_count(0, O.p(vnull), 0, O.p(oids), n, O.p(wc))
    cs = np.zeros(ng, np.int64)
    assert ops.group_agg(capi.AGG_COUNT, capi.T_INT32, cs, None, None, groups, val, vnull, n) == 0
    assert np.array_equal(cs, wc)
