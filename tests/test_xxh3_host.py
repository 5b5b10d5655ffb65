"""The device hash header (matrixone_b200/csrc/xxh3_128.cuh, compiled for the host by oracle/build.py) against the REAL xxHash 0.8.3 of the
tarball the reference pins (thirdparties/Makefile:26), exported by oracle/_ref/libbloom_ref.so (its results recorded in
tests/golden/ref_test_xxh3_host.npz): every input-length class of XXH3_128bits_withSeed, several seeds, and the 8-byte integer path
cgo/bloom.c:31-37 uses.  No GPU needed."""
import ctypes as C
import os

import numpy as np

from oracle import build as oracle_build
from ref_tape import digest, original

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _libs():
    ref_path = os.path.join(ROOT, "oracle", "_ref", "libbloom_ref.so")
    ref = original(lambda: C.CDLL(ref_path) if os.path.exists(ref_path) else None)
    mine = C.CDLL(oracle_build.build_xxh3_host())
    if ref is not None:
        ref.ref_xxh3_128.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p]
    mine.mob_xxh3_128_bytes.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p]
    mine.mob_xxh3_128_u64.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p]
    return ref, mine


def test_every_length_class_matches_real_xxhash(ref_tape):
    ref, mine = _libs()
    rng = np.random.default_rng(1)
    buf = rng.integers(0, 256, 6000, dtype=np.uint8)
    lengths = list(range(0, 1100)) + [2047, 2048, 2049, 4096, 5990]
    for seed in (0, 1, 0x9E3779B185EBCA87, 0xFFFFFFFFFFFFFFFF, int(rng.integers(0, 2 ** 63))):
        def hashes(fn):
            out = np.zeros((len(lengths), 2), np.uint64)
            for i, n in enumerate(lengths):
                fn(buf.ctypes.data + 3, n, seed, out[i].ctypes.data)          # + 3: unaligned input
            return out
        assert digest(hashes(mine.mob_xxh3_128_bytes)) == ref_tape(lambda: hashes(ref.ref_xxh3_128)), seed


def test_integer_key_path_matches_real_xxhash(ref_tape):
    ref, mine = _libs()
    rng = np.random.default_rng(2)
    for seed in (0, 7, 0xDEADBEEFCAFEF00D):
        keys = list(rng.integers(0, 2 ** 64, 500, dtype=np.uint64)) + [0, 1, 2 ** 64 - 1, 2 ** 63]
        got = np.zeros((len(keys), 2), np.uint64)
        for i, k in enumerate(keys):
            mine.mob_xxh3_128_u64(int(k), seed, got[i].ctypes.data)

        def want():
            out = np.zeros((len(keys), 2), np.uint64)
            for i, k in enumerate(keys):
                kk = np.array([k], np.uint64)
                ref.ref_xxh3_128(kk.ctypes.data, 8, seed, out[i].ctypes.data)
            return out
        assert digest(got) == ref_tape(want), seed
