"""Recorded results of the original project's own C code, so that the tests comparing with it run without it.

The original's C (oracle/_ref/*, compiled by oracle/build.py from the original sources) exists only where those sources do.  A test
that compares with it takes the `ref_tape` fixture and wraps every call of the original code in `ref_tape(fn)`:

    rc1, d1 = ref_tape(lambda: (ref.SignedInt_VecAdd(...), r1))       # what the original returned, digest of what it wrote
    assert rc1 == rc2 and d1 == digest(r2)

By default `fn` is not called: its results come from tests/golden/ref_<test module>.npz, in call order.  With MO_B200_RECORD_REF=<dir>
the original is called and its results are written to <dir>/ref_<test module>.npz when the module ends (run whole modules; copy the
files to tests/golden/ to update the recording).

`fn` returns an int / bool / None, an ndarray / bytes, or a tuple of those.  Arrays are kept as a 64-bit digest (`digest`); with
keep=True they are stored whole, for comparisons within a tolerance.
"""
import hashlib
import os

import numpy as np

RECORD_DIR = os.environ.get("MO_B200_RECORD_REF") or None
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_MASK = (1 << 64) - 1
_INT, _DIGEST, _ARRAY = 0, 1, 2


def recording():
    return RECORD_DIR is not None


def original(load):
    """the original's library while recording (load() must find it under oracle/_ref); None when replaying"""
    if not recording():
        return None
    lib = load()
    assert lib is not None, "recording needs oracle/_ref, which oracle/build.py builds from the original sources"
    return lib


def digest(a):
    """64-bit digest of an array's dtype, shape and values.  Floats are canonical first: every NaN is the same NaN and -0.0 is 0.0, so
    equal digests mean what np.array_equal(..., equal_nan=True) means."""
    if isinstance(a, (bytes, bytearray)):
        a = np.frombuffer(bytes(a), np.uint8)
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), a.dtype.type(np.nan), a + a.dtype.type(0))
    h = hashlib.blake2b(digest_size=8)
    h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return int.from_bytes(h.digest(), "little")


def _signed(v):
    return v - (1 << 64) if v >> 63 else v


class Tape:
    def __init__(self, store, node):
        self.node = node
        self.store = store
        if recording():
            self.flat, self.arrays = [], {}
        else:
            if node not in store:
                raise KeyError("no recording of the original's results for %s; record them with MO_B200_RECORD_REF=<dir>" % node)
            self.flat = [int(x) for x in store[node]]
            self.pos = 0

    def live(self, fn):
        """calls fn only while recording (set-up and clean-up of the original's objects); None otherwise"""
        return fn() if recording() else None

    def __call__(self, fn, keep=False):
        if recording():
            res = fn()
            items = res if isinstance(res, tuple) else (res,)
            out = []
            self.flat.append(len(items))
            for it in items:
                if isinstance(it, (np.ndarray, bytes, bytearray)):
                    if keep:
                        key = "%s#%d" % (self.node, len(self.arrays))
                        self.arrays[key] = np.array(np.frombuffer(bytes(it), np.uint8) if not isinstance(it, np.ndarray) else it, copy=True)
                        self.flat += [_ARRAY, len(self.arrays) - 1]
                        out.append(self.arrays[key])
                    else:
                        d = digest(it)
                        self.flat += [_DIGEST, d]
                        out.append(d)
                else:
                    v = 0 if it is None else int(it)
                    self.flat += [_INT, v & _MASK]
                    out.append(v)
        else:
            assert self.pos < len(self.flat), "%s calls the original more often than the recording holds" % self.node
            n = self.flat[self.pos]
            self.pos += 1
            out = []
            for _ in range(n):
                kind, v = self.flat[self.pos], self.flat[self.pos + 1]
                self.pos += 2
                if kind == _ARRAY:
                    out.append(self.store["%s#%d" % (self.node, v)])
                elif kind == _DIGEST:
                    out.append(v)
                else:
                    out.append(_signed(v))
        return tuple(out) if len(out) > 1 else out[0]

    def close(self):
        if recording():
            self.store.update(self.arrays)
            self.store[self.node] = np.array(self.flat, dtype=np.uint64)
        else:
            assert self.pos == len(self.flat), "%s called the original fewer times than recorded" % self.node


def module_store(module_name):
    if recording():
        return {}
    path = os.path.join(GOLDEN, "ref_%s.npz" % module_name)
    if not os.path.exists(path):
        return {}
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def write_store(module_name, store):
    if recording() and store:
        os.makedirs(RECORD_DIR, exist_ok=True)
        np.savez_compressed(os.path.join(RECORD_DIR, "ref_%s.npz" % module_name), **store)
