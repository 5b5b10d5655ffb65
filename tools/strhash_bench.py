"""Time the StrHashMap entry points (csrc/strhash.cu) on resident inputs larger than L2 and print one JSON line.

    python tools/strhash_bench.py [--rows 50000000] [--reps 3] [--out FILE]

Keys: varchar (lengths uniform in 5..40, so both inline and area cells) + int32, nullable (has_null mode), at cardinality 16, 65 536 and
4 194 304; plus a long-key case (~512-byte varchar).  Per case: PACK_STR_KEYS, STR_GROUP_IDS on a fresh table (first batch) and again into
the populated table (second batch), STR_JOIN_FIND and STR_JOIN_PROBE (INNER) against a prepared map of the distinct keys.  Times are CUDA
events around each synchronous call after one warm-up, median of --reps.  Rates use algorithmic bytes: what each call must read and write
once (key columns, offsets, packed key bytes, ids / pairs).  The one-core time of the C oracle (tests/oracle_strhash.c) is reported for
context only: it is this project's restatement with an exact byte-compare hash set, not the reference's AES-hashed StringHashMap.
"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from matrixone_b200 import capi, ops  # noqa: E402
from matrixone_b200.vector import DeviceBuffer, Vector, xcall  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        name, pl, pmax = [x.strip() for x in out.split(",")]
        return {"card": name, "power_limit": pl, "power_max_limit": pmax}
    except Exception as e:  # noqa: BLE001
        return {"card": "unknown", "power_limit": "unknown (%s)" % e}


def key_columns(rng, n, card, min_len=5, max_len=40):
    """varchar of group g: 5 base-26 digits of g then filler, length min_len + (g * 2654435761) % (max_len - min_len + 1); int32 = g ^ 0x5bd1e995"""
    g = np.arange(card, dtype=np.int64)
    lens = min_len + (g * 2654435761) % (max_len - min_len + 1)
    width = int(lens.max())
    txt = np.empty((card, width), np.uint8)
    for j in range(width):
        txt[:, j] = (97 + (g // 26 ** j) % 26) if j < 5 else (97 + (g * 31 + j * 7) % 26)
    gcells = np.zeros((card, 24), np.uint8)
    small = lens <= 23
    for L in np.unique(lens[small]):
        m = lens == L
        gcells[m, 0] = L
        gcells[m, 1:1 + L] = txt[m, :L]
    u32 = gcells.view(np.uint32)
    u32[~small, 0] = 0xFFFFFFFF
    u32[~small, 1] = (g[~small] * width).astype(np.uint32)
    u32[~small, 2] = lens[~small].astype(np.uint32)
    area = txt.reshape(-1)
    gid = rng.integers(0, card, n)
    cells = gcells[gid]
    ints = (gid ^ 0x5BD1E995).astype(np.int32)
    alg_col_bytes = int(n) * (24 + 4) + int(np.where(small[gid], 0, lens[gid]).sum())
    return cells.reshape(-1), area, ints, alg_col_bytes


class Timer:
    def __init__(self, lib):
        self.lib = lib

    def run(self, fn, reps, setup=None):
        if setup:
            setup()
        fn()                                                     # warm-up
        ts = []
        for _ in range(reps):
            if setup:
                setup()
            capi.check(self.lib.MoB200_TimerStart(), self.lib)
            fn()
            ms = C.c_float()
            capi.check(self.lib.MoB200_TimerStop(C.byref(ms)), self.lib)
            ts.append(ms.value)
        return float(np.median(ts))


def dv(buf, nbytes=None, length=1, nulls=None):
    return Vector(data_ptr=buf.ptr, data_nbytes=buf.nbytes if nbytes is None else nbytes, length=length, nulls_ptr=nulls)


def bench_case(lib, T, n, card, reps, min_len=5, max_len=40):
    rng = np.random.default_rng(card)
    cells, area, ints, col_bytes = key_columns(rng, n, card, min_len, max_len)
    d_cells, d_area, d_ints = DeviceBuffer.from_numpy(cells), DeviceBuffer.from_numpy(area), DeviceBuffer.from_numpy(ints)
    del cells, ints
    prm = capi.StrKeyParams(2, 1)
    prm.width[0], prm.width[1] = 0, 4
    d_off = DeviceBuffer(8 * (n + 1))
    cap = n * (8 + max_len) + 64
    d_kb = DeviceBuffer(cap)
    cols = [Vector(data_ptr=d_cells.ptr, data_nbytes=d_cells.nbytes, area_ptr=d_area.ptr, area_nbytes=d_area.nbytes, length=n), dv(d_ints, length=n)]
    pack = lambda: xcall(capi.XCALL_PACK_STR_KEYS, [dv(d_off, length=n), dv(d_kb, length=n), ops._params_vec(prm)] + cols, n)
    t_pack = T.run(pack, reps)
    key_bytes = int(d_off.to_numpy(np.int64, n + 1)[n])
    d_groups = DeviceBuffer(8 * n)
    d_state = DeviceBuffer(32)
    d_toff = DeviceBuffer(8 * (card + 1))
    d_tb = DeviceBuffer(card * (8 + max_len) + 64)
    zero_state = lambda: capi.check(lib.MoB200_Upload(d_state.ptr, np.zeros(4, np.int64).ctypes.data, 32), lib)
    gid_args = lambda: [dv(d_groups, length=n), dv(d_state, 32, 4), dv(d_toff, length=card + 1), dv(d_tb), dv(d_off, length=n), dv(d_kb, key_bytes, n)]
    insert = lambda: xcall(capi.XCALL_STR_GROUP_IDS, gid_args(), n)
    t_first = T.run(insert, reps, setup=zero_state)
    zero_state(); insert()
    state = d_state.to_numpy(np.int64)
    ng, tbytes = int(state[0]), int(state[1])
    populated = lambda: capi.check(lib.MoB200_Upload(d_state.ptr, state.ctypes.data, 32), lib)
    t_second = T.run(insert, reps, setup=populated)
    assert int(d_state.to_numpy(np.int64)[0]) == ng
    capi.check(lib.MoB200_StrJoinMapPrepare(d_toff.ptr, d_tb.ptr, ng), lib)
    tab = [dv(d_toff, 8 * (ng + 1), ng + 1), dv(d_tb, tbytes)]
    find = lambda: xcall(capi.XCALL_STR_JOIN_FIND, [dv(d_groups, length=n)] + tab + [dv(d_off, length=n), dv(d_kb, key_bytes, n)], n)
    t_find = T.run(find, reps)
    d_pp, d_pb, d_cnt = DeviceBuffer(8 * n), DeviceBuffer(8 * n), DeviceBuffer(8)
    jp = np.array([capi.JOIN_INNER, 0], np.int32)
    probe = lambda: xcall(capi.XCALL_STR_JOIN_PROBE, [dv(d_pp, length=n), dv(d_pb, length=n), dv(d_cnt), Vector(data=jp.view(np.uint8), length=1)] + tab +
                          [Vector(length=0), Vector(length=0), dv(d_off, length=n), dv(d_kb, key_bytes, n)], n)
    t_probe = T.run(probe, reps)
    pairs = int(d_cnt.to_numpy(np.int64)[0])
    capi.check(lib.MoB200_StrJoinMapRelease(d_toff.ptr), lib)
    for b in (d_cells, d_area, d_ints, d_off, d_kb, d_groups, d_state, d_toff, d_tb, d_pp, d_pb, d_cnt):
        b.free()
    keyed = 8 * (n + 1) + key_bytes                          # packed offsets + key bytes, read once

    def rate(ms, nbytes):
        return {"ms": round(ms, 3), "rows_per_s": round(n / (ms * 1e-3), 1), "alg_GB_per_s": round(nbytes / (ms * 1e-3) / 1e9, 2)}
    return {"rows": n, "cardinality": card, "groups": ng, "key_len": [min_len, max_len], "packed_key_bytes": key_bytes,
            "key_bytes_per_s_pack": round(key_bytes / (t_pack * 1e-3), 1),
            "pack": rate(t_pack, col_bytes + keyed), "group_ids_first": rate(t_first, keyed + 8 * n + tbytes),
            "group_ids_second": rate(t_second, keyed + 8 * n + tbytes), "find": rate(t_find, keyed + 8 * n + tbytes),
            "probe_inner": dict(rate(t_probe, keyed + 16 * pairs + tbytes), pairs=pairs)}


def oracle_one_core(n, card):
    """one-core C restatement (tests/oracle_strhash.c), pack + insert, for context"""
    import oracle_lib as O
    from strhash_util import oracle_pack, strhash
    rng = np.random.default_rng(7)
    cells, area, ints, _ = key_columns(rng, n, card)
    t0 = time.perf_counter()
    off, kb, _ = oracle_pack([(cells, area), ints], [0, 4], None, True)
    t1 = time.perf_counter()
    toff, tb = np.zeros(n + 1, np.int64), np.zeros(len(kb), np.uint8)
    groups, need = np.zeros(n, np.uint64), np.zeros(2, np.int64)
    strhash().og_str_group_ids(O.p(off), O.p(kb), None, n, O.p(groups), O.p(toff), O.p(tb), 0, n, len(tb), O.p(need))
    t2 = time.perf_counter()
    return {"label": "C oracle restatement, one CPU core (context only: byte-compare hash set, not the reference's AES StringHashMap); "
                     "pack time includes a sizing pass", "rows": n, "cardinality": card,
            "pack_rows_per_s": round(n / (t1 - t0), 1), "group_ids_rows_per_s": round(n / (t2 - t1), 1)}


def main():
    rows = int(sys.argv[sys.argv.index("--rows") + 1]) if "--rows" in sys.argv else 50_000_000
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 3
    lib = capi.load_library()
    capi.check(lib.MoB200_Init(0), lib)
    T = Timer(lib)
    res = {"bench": "strhash", "method": "CUDA events around each synchronous call, 1 warm-up, median of %d; resident inputs" % reps}
    res.update(gpu_info())
    res["cases"] = [bench_case(lib, T, rows, card, reps) for card in (16, 65_536, 4_194_304)]
    res["cases"].append(dict(bench_case(lib, T, rows // 10, 65_536, reps, 500, 524), long_keys=True))
    res["oracle_one_core"] = oracle_one_core(2_000_000, 65_536)
    line = json.dumps(res)
    print(line)
    if "--out" in sys.argv:
        with open(sys.argv[sys.argv.index("--out") + 1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
