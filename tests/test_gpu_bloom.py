"""The bloom filter entry points of libmo_b200.so (include/mo_b200_bloom.h) against the reference's own cgo/bloom.c compiled UNCHANGED with the
xxHash it pins (oracle/_ref/libbloom_ref.so, its results recorded in tests/golden/ref_test_gpu_bloom.npz): same results row by row and the
same filter BYTES after every mutating call."""
import ctypes as C
import os

import numpy as np
import pytest

from matrixone_b200 import capi
from matrixone_b200.vector import bitmap_from_bools, varlena_column
from ref_tape import digest, original

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_vp, _sz, _u64, _u32 = C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32


def _proto(lib):
    lib.bloomfilter_init_with_seed.restype = _vp; lib.bloomfilter_init_with_seed.argtypes = [_u64, _u32, _u64]
    lib.bloomfilter_init.restype = _vp; lib.bloomfilter_init.argtypes = [_u64, _u32]
    lib.bloomfilter_free.restype = None; lib.bloomfilter_free.argtypes = [_vp]
    lib.bloomfilter_add.restype = None; lib.bloomfilter_add.argtypes = [_vp, _vp, _sz]
    lib.bloomfilter_test.restype = C.c_bool; lib.bloomfilter_test.argtypes = [_vp, _vp, _sz]
    lib.bloomfilter_test_and_add.restype = C.c_bool; lib.bloomfilter_test_and_add.argtypes = [_vp, _vp, _sz]
    lib.bloomfilter_add_fixed.restype = None; lib.bloomfilter_add_fixed.argtypes = [_vp, _vp, _sz, _sz, _sz, _vp, _sz]
    for n in ("bloomfilter_test_fixed", "bloomfilter_test_and_add_fixed"):
        getattr(lib, n).restype = None; getattr(lib, n).argtypes = [_vp, _vp, _sz, _sz, _sz, _vp, _sz, _vp]
    lib.bloomfilter_add_varlena_4b.restype = None; lib.bloomfilter_add_varlena_4b.argtypes = [_vp, _vp, _sz, _sz, _vp, _sz]
    for n in ("bloomfilter_test_varlena_4b", "bloomfilter_test_and_add_varlena_4b"):
        getattr(lib, n).restype = None; getattr(lib, n).argtypes = [_vp, _vp, _sz, _sz, _vp, _sz, _vp]
    lib.bloomfilter_add_varlena.restype = None; lib.bloomfilter_add_varlena.argtypes = [_vp, _vp, _sz, _sz, _sz, _vp, _sz, _vp, _sz]
    for n in ("bloomfilter_test_varlena", "bloomfilter_test_and_add_varlena"):
        getattr(lib, n).restype = None; getattr(lib, n).argtypes = [_vp, _vp, _sz, _sz, _sz, _vp, _sz, _vp, _sz, _vp]
    lib.bloomfilter_marshal.restype = _vp; lib.bloomfilter_marshal.argtypes = [_vp, C.POINTER(_sz)]
    lib.bloomfilter_unmarshal.restype = _vp; lib.bloomfilter_unmarshal.argtypes = [_vp, _sz]
    lib.bloomfilter_or.restype = C.c_int; lib.bloomfilter_or.argtypes = [_vp, _vp, _vp]
    return lib


@pytest.fixture(scope="module")
def libs(gpu):
    p = os.path.join(ROOT, "oracle", "_ref", "libbloom_ref.so")
    return _proto(capi.load_library()), original(lambda: _proto(C.CDLL(p)) if os.path.exists(p) else None)


def _bytes(lib, bf):
    n = _sz()
    p = lib.bloomfilter_marshal(bf, C.byref(n))
    return C.string_at(p, n.value)[:-8]      # sizeof(bloomfilter_t) counts bitmap[1] once more: the reference's last 8 marshalled bytes are uninitialised


def _p(a):
    return a.ctypes.data if a is not None and a.size else None


@pytest.mark.parametrize("dtype", [np.int8, np.int16, np.int32, np.int64, np.uint64, np.float64])
@pytest.mark.parametrize("k,nbits", [(3, 1 << 16), (7, 100_000), (1, 64)])
def test_fixed_add_test_and_bytes(libs, ref_tape, dtype, k, nbits):
    ours, ref = libs
    rng = np.random.default_rng(k * 131 + nbits)
    n = 20_000
    info = np.iinfo(dtype) if np.issubdtype(dtype, np.integer) else None
    keys = rng.integers(info.min, info.max, n, dtype=dtype, endpoint=True) if info else rng.standard_normal(n).astype(dtype)
    probe = np.concatenate([keys[: n // 2], (rng.integers(info.min, info.max, n // 2, dtype=dtype, endpoint=True) if info else rng.standard_normal(n // 2).astype(dtype))])
    nulls = bitmap_from_bools(rng.random(n) < 0.1)
    a, b = ours.bloomfilter_init_with_seed(nbits, k, 12345), ref_tape.live(lambda: ref.bloomfilter_init_with_seed(nbits, k, 12345))
    es = keys.itemsize
    ours.bloomfilter_add_fixed(a, _p(keys), keys.nbytes, es, n, _p(nulls), nulls.nbytes)
    ref_tape.live(lambda: ref.bloomfilter_add_fixed(b, _p(keys), keys.nbytes, es, n, _p(nulls), nulls.nbytes))
    assert digest(_bytes(ours, a)) == ref_tape(lambda: _bytes(ref, b))
    ra, rb = np.full(n, 7, np.uint8), np.full(n, 7, np.uint8)
    ours.bloomfilter_test_fixed(a, _p(probe), probe.nbytes, es, n, _p(nulls), nulls.nbytes, _p(ra))
    _, drb = ref_tape(lambda: (ref.bloomfilter_test_fixed(b, _p(probe), probe.nbytes, es, n, _p(nulls), nulls.nbytes, _p(rb)), rb))
    assert digest(ra) == drb
    # no nullmap: every added key is found
    ours.bloomfilter_add_fixed(a, _p(keys), keys.nbytes, es, n, None, 0)
    ours.bloomfilter_test_fixed(a, _p(keys), keys.nbytes, es, n, None, 0, _p(ra))
    assert ra.all()
    ours.bloomfilter_free(a); ref_tape.live(lambda: ref.bloomfilter_free(b))


def test_equal_values_of_different_widths_share_their_bits(libs):
    ours, _ = libs
    a = ours.bloomfilter_init_with_seed(1 << 14, 4, 99)
    v8 = np.array([-5, 7, 100], np.int8)
    ours.bloomfilter_add_fixed(a, _p(v8), v8.nbytes, 1, 3, None, 0)
    for dt in (np.int16, np.int32, np.int64):
        v = v8.astype(dt); r = np.zeros(3, np.uint8)
        ours.bloomfilter_test_fixed(a, _p(v), v.nbytes, v.itemsize, 3, None, 0, _p(r))
        assert r.all()
    ours.bloomfilter_free(a)


@pytest.mark.parametrize("k,nbits,n", [(3, 1 << 12, 5000), (5, 1 << 20, 50_000), (2, 64, 300)])
def test_test_and_add_keeps_the_sequential_semantics(libs, ref_tape, k, nbits, n):
    ours, ref = libs
    rng = np.random.default_rng(n)
    keys = rng.integers(0, n // 3 + 2, n, dtype=np.int64)        # many repeats: a repeat is "seen" only after its first occurrence
    nulls = bitmap_from_bools(rng.random(n) < 0.05)
    a, b = ours.bloomfilter_init_with_seed(nbits, k, 777), ref_tape.live(lambda: ref.bloomfilter_init_with_seed(nbits, k, 777))
    pre = rng.integers(0, 1000, 50, dtype=np.int64) + 10_000_000
    ours.bloomfilter_add_fixed(a, _p(pre), pre.nbytes, 8, 50, None, 0); ref_tape.live(lambda: ref.bloomfilter_add_fixed(b, _p(pre), pre.nbytes, 8, 50, None, 0))
    for rep in range(2):   # the second round sees the first round's bits
        ra, rb = np.full(n, 9, np.uint8), np.full(n, 9, np.uint8)
        ours.bloomfilter_test_and_add_fixed(a, _p(keys), keys.nbytes, 8, n, _p(nulls), nulls.nbytes, _p(ra))
        _, drb = ref_tape(lambda: (ref.bloomfilter_test_and_add_fixed(b, _p(keys), keys.nbytes, 8, n, _p(nulls), nulls.nbytes, _p(rb)), rb))
        assert digest(ra) == drb, rep
        assert digest(_bytes(ours, a)) == ref_tape(lambda: _bytes(ref, b))
    ours.bloomfilter_free(a); ref_tape.live(lambda: ref.bloomfilter_free(b))


def _rows(rng, n):
    lens = rng.choice([0, 1, 2, 3, 4, 5, 8, 9, 16, 17, 23, 24, 31, 32, 33, 64, 100, 128, 129, 200, 240, 241, 300, 1000, 1500], n)
    return [rng.integers(0, 256, int(l), dtype=np.uint8) for l in lens]


def test_varlena_cells_all_length_classes(libs, ref_tape):
    ours, ref = libs
    rng = np.random.default_rng(5)
    n = 3000
    rows = _rows(rng, n)
    cells, area = varlena_column(rows, dtype=np.uint8)
    probe_rows = rows[: n // 2] + _rows(rng, n - n // 2)
    pcells, parea = varlena_column(probe_rows, dtype=np.uint8)
    nulls = bitmap_from_bools(rng.random(n) < 0.1)
    a, b = ours.bloomfilter_init_with_seed(1 << 18, 6, 4242), ref_tape.live(lambda: ref.bloomfilter_init_with_seed(1 << 18, 6, 4242))
    ours.bloomfilter_add_varlena(a, _p(cells), cells.nbytes, 24, n, _p(area), area.nbytes, _p(nulls), nulls.nbytes)
    ref_tape.live(lambda: ref.bloomfilter_add_varlena(b, _p(cells), cells.nbytes, 24, n, _p(area), area.nbytes, _p(nulls), nulls.nbytes))
    assert digest(_bytes(ours, a)) == ref_tape(lambda: _bytes(ref, b))
    ra, rb = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    ours.bloomfilter_test_varlena(a, _p(pcells), pcells.nbytes, 24, n, _p(parea), parea.nbytes, _p(nulls), nulls.nbytes, _p(ra))
    _, drb = ref_tape(lambda: (ref.bloomfilter_test_varlena(b, _p(pcells), pcells.nbytes, 24, n, _p(parea), parea.nbytes, _p(nulls), nulls.nbytes, _p(rb)), rb))
    assert digest(ra) == drb
    ours.bloomfilter_test_and_add_varlena(a, _p(pcells), pcells.nbytes, 24, n, _p(parea), parea.nbytes, None, 0, _p(ra))
    _, drb, dbytes = ref_tape(lambda: (ref.bloomfilter_test_and_add_varlena(b, _p(pcells), pcells.nbytes, 24, n, _p(parea), parea.nbytes, None, 0, _p(rb)), rb, _bytes(ref, b)))
    assert digest(ra) == drb and digest(_bytes(ours, a)) == dbytes
    ours.bloomfilter_free(a); ref_tape.live(lambda: ref.bloomfilter_free(b))


def test_length_prefixed_stream_single_keys_marshal_or(libs, ref_tape):
    ours, ref = libs
    rng = np.random.default_rng(6)
    rows = _rows(rng, 500)
    stream = np.concatenate([np.concatenate([np.array([len(r)], np.uint32).view(np.uint8), r]) for r in rows])
    a, b = ours.bloomfilter_init_with_seed(1 << 15, 3, 1), ref_tape.live(lambda: ref.bloomfilter_init_with_seed(1 << 15, 3, 1))
    ours.bloomfilter_add_varlena_4b(a, _p(stream), stream.nbytes, 500, None, 0); ref_tape.live(lambda: ref.bloomfilter_add_varlena_4b(b, _p(stream), stream.nbytes, 500, None, 0))
    assert digest(_bytes(ours, a)) == ref_tape(lambda: _bytes(ref, b))
    cut = stream[: stream.nbytes - 7]     # a truncated stream: rows past the cut are not touched
    ra, rb = np.full(500, 5, np.uint8), np.full(500, 5, np.uint8)
    ours.bloomfilter_test_varlena_4b(a, _p(cut), cut.nbytes, 500, None, 0, _p(ra))
    _, drb = ref_tape(lambda: (ref.bloomfilter_test_varlena_4b(b, _p(cut), cut.nbytes, 500, None, 0, _p(rb)), rb))
    assert digest(ra) == drb
    # single-key entry points
    for r in rows[:20] + [np.frombuffer(b"not there", np.uint8)]:
        assert ours.bloomfilter_test(a, _p(r), r.nbytes) == ref_tape(lambda: ref.bloomfilter_test(b, _p(r), r.nbytes))
    k1 = np.frombuffer(b"a brand new key", np.uint8)
    assert ours.bloomfilter_test_and_add(a, _p(k1), k1.nbytes) == ref_tape(lambda: ref.bloomfilter_test_and_add(b, _p(k1), k1.nbytes)) == False
    assert ours.bloomfilter_test_and_add(a, _p(k1), k1.nbytes) == ref_tape(lambda: ref.bloomfilter_test_and_add(b, _p(k1), k1.nbytes)) == True
    k2 = np.array([123456789], np.int64)
    ours.bloomfilter_add(a, _p(k2), 8); ref_tape.live(lambda: ref.bloomfilter_add(b, _p(k2), 8))
    assert digest(_bytes(ours, a)) == ref_tape(lambda: _bytes(ref, b))
    # marshal -> unmarshal -> probe; or
    raw = np.frombuffer(_bytes(ours, a), np.uint8).copy()
    u = ours.bloomfilter_unmarshal(_p(raw), raw.nbytes)
    assert u == raw.ctypes.data
    for r in rows[:20]:
        assert ours.bloomfilter_test(u, _p(r), r.nbytes)
    c, d = ours.bloomfilter_init_with_seed(1 << 15, 3, 1), ref_tape.live(lambda: ref.bloomfilter_init_with_seed(1 << 15, 3, 1))
    more = rng.integers(0, 1 << 40, 1000, dtype=np.int64)
    ours.bloomfilter_add_fixed(c, _p(more), more.nbytes, 8, 1000, None, 0); ref_tape.live(lambda: ref.bloomfilter_add_fixed(d, _p(more), more.nbytes, 8, 1000, None, 0))
    assert ours.bloomfilter_or(a, a, c) == ref_tape(lambda: ref.bloomfilter_or(b, b, d)) == 0      # Merge: dst == a (cbloomfilter.go:435)
    assert digest(_bytes(ours, a)) == ref_tape(lambda: _bytes(ref, b))
    e = ours.bloomfilter_init_with_seed(1 << 16, 3, 1)
    assert ours.bloomfilter_or(a, a, e) == 1
    f = ours.bloomfilter_init_with_seed(1 << 15, 3, 2)
    assert ours.bloomfilter_or(a, a, f) == 2
    g = ours.bloomfilter_init_with_seed(1 << 15, 4, 1)
    assert ours.bloomfilter_or(a, a, g) == 3
    for x in (a, c, e, f, g):
        ours.bloomfilter_free(x)
    for x in (b, d):
        ref_tape.live(lambda: ref.bloomfilter_free(x))


def test_device_resident_keys_and_results(libs, ref_tape):
    from matrixone_b200.vector import DeviceBuffer
    ours, ref = libs
    rng = np.random.default_rng(8)
    n = 1_000_000
    keys = rng.integers(0, 1 << 62, n, dtype=np.int64)
    a, b = ours.bloomfilter_init_with_seed(1 << 24, 3, 5), ref_tape.live(lambda: ref.bloomfilter_init_with_seed(1 << 24, 3, 5))
    dk = DeviceBuffer.from_numpy(keys); dr = DeviceBuffer(n)
    ours.bloomfilter_add_fixed(a, dk.ptr, keys.nbytes, 8, n // 2, None, 0)
    ref_tape.live(lambda: ref.bloomfilter_add_fixed(b, _p(keys), keys.nbytes, 8, n // 2, None, 0))
    ours.bloomfilter_test_fixed(a, dk.ptr, keys.nbytes, 8, n, None, 0, dr.ptr)
    rb = np.zeros(n, np.uint8)
    _, drb = ref_tape(lambda: (ref.bloomfilter_test_fixed(b, _p(keys), keys.nbytes, 8, n, None, 0, _p(rb)), rb))
    assert digest(dr.to_numpy(np.uint8)) == drb
    assert digest(_bytes(ours, a)) == ref_tape(lambda: _bytes(ref, b))
    ours.bloomfilter_free(a); ref_tape.live(lambda: ref.bloomfilter_free(b)); dk.free(); dr.free()
