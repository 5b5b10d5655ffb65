"""Pin the CPU oracle (oracle/oracle_go.c) against the reference's own known-answer tests (tests/golden/*.json,
transcribed from the Go test files by tests/golden/extract_goldens.py) and against the reference C compiled unchanged
(oracle/_ref).  CPU only."""
import ctypes as C
import json
import os

import numpy as np

import oracle_lib as O
from ref_tape import digest, original

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


def _call64(fn, v1, v2):
    a = np.asarray(v1, dtype=np.float64); b = np.asarray(v2, dtype=np.float64)
    return fn(O.p(a), O.p(b), len(a))


def test_metric_kats_exact_f64():
    """distance_func_test.go:158-496 -- the Go tests use != on float64, so do we."""
    k = load("metric_kat.json")
    lib = O.go()
    for key, fn in (("l2", lib.og_l2_f64), ("l1", lib.og_l1_f64), ("cosine_distance", lib.og_cosdist_f64),
                    ("inner_product", lib.og_ip_f64), ("l2sq", lib.og_l2sq_f64)):
        for c in k[key]:
            got = _call64(fn, c["v1"], c["v2"])
            assert got == c["want"], (key, c, got)
    z = k["zero_vector_cosine_distance"]
    assert _call64(lib.og_cosdist_f64, z["v1"], z["v2"]) == 1.0
    a = np.zeros(3, dtype=np.float32)
    assert lib.og_cosdist_f32(O.p(a), O.p(a), 3) == np.float32(1.0)


def test_moarray_kats():
    """moarray/external_test.go:584-870 (InEpsilonF64).  The f32 and f64 L2 goldens differ (33.6749153137207 vs
    33.67491648096547): this pins 'accumulator type == element type'."""
    k = load("moarray_kat.json")
    lib = O.go()
    err = np.zeros(1, dtype=np.int32)
    for c in k["l2"]:
        if c["dtype"] == "f32":
            a = np.asarray(c["v1"], dtype=np.float32); b = np.asarray(c["v2"], dtype=np.float32)
            got = float(lib.og_l2_f32(O.p(a), O.p(b), len(a)))
        else:
            got = _call64(lib.og_l2_f64, c["v1"], c["v2"])
        assert got == c["want"], (c, got)   # exact: the goldens were printed by the reference itself
    for c in k["inner_product"]:
        if c["dtype"] == "f32":
            a = np.asarray(c["v1"], dtype=np.float32); b = np.asarray(c["v2"], dtype=np.float32)
            got = float(lib.og_ip_f32(O.p(a), O.p(b), len(a)))
        else:
            got = _call64(lib.og_ip_f64, c["v1"], c["v2"])
        assert got == c["want"]
    for c in k["cosine_similarity"]:
        if c["dtype"] == "f32":
            a = np.asarray(c["v1"], dtype=np.float32); b = np.asarray(c["v2"], dtype=np.float32)
            got = lib.og_moarray_cossim_f32(O.p(a), O.p(b), len(a), O.p(err))
        else:
            a = np.asarray(c["v1"], dtype=np.float64); b = np.asarray(c["v2"], dtype=np.float64)
            got = lib.og_moarray_cossim_f64(O.p(a), O.p(b), len(a), O.p(err))
        assert abs(got - c["want"]) <= 1e-9 * max(1.0, abs(c["want"])), (c, got)
    for c in k["cosine_distance"]:
        if c["dtype"] == "f32":
            a = np.asarray(c["v1"], dtype=np.float32); b = np.asarray(c["v2"], dtype=np.float32)
            got = float(lib.og_cosdist_f32(O.p(a), O.p(b), len(a)))
        else:
            got = _call64(lib.og_cosdist_f64, c["v1"], c["v2"])
        assert abs(got - c["want"]) <= 1e-6, (c, got)
    for c in k["normalize_l2"]:
        dt = np.float32 if c["dtype"] == "f32" else np.float64
        v = np.asarray(c["v"], dtype=dt); out = np.zeros_like(v)
        fn = lib.og_normalize_l2_f32 if dt == np.float32 else lib.og_normalize_l2_f64
        assert fn(O.p(v), O.p(out), len(v)) == 0
        np.testing.assert_allclose(out, np.asarray(c["want"], dtype=dt), rtol=1e-6 if dt == np.float32 else 1e-15)


def test_fast_max_heap_kat():
    """index_test.go:215-249: pushes (10,5,20,1,8) with limit 3 pop as 8,5,1 => ascending output 1,5,8."""
    k = load("heap_kat.json")
    d = np.asarray([x["dist"] for x in k["pushes"]], dtype=np.float32)
    keys = np.asarray([x["key"] for x in k["pushes"]], dtype=np.int64)
    ok = np.zeros(k["limit"], dtype=np.int64); od = np.zeros(k["limit"], dtype=np.float32)
    O.go().og_heap_topk_f32(O.p(d), O.p(keys), len(d), k["limit"], O.p(ok), O.p(od))
    pops = k["pops_in_order"]  # largest first
    assert list(ok[::-1]) == [x["key"] for x in pops]
    assert list(od[::-1]) == [x["dist"] for x in pops]


def test_bruteforce_self_match_and_padding():
    """brute_force_test.go:76-146: querying the dataset with itself returns key == i and distance == 0.0 exactly;
    brute_force.go:319-331: fewer rows than limit pads (-1, 0) at the FRONT."""
    rng = np.random.default_rng(5)
    ds = rng.standard_normal((500, 128)).astype(np.float32)
    keys, dists = O.bruteforce(ds, ds, 3)
    keys = keys.reshape(-1, 3); dists = dists.reshape(-1, 3)
    assert (keys[:, 0] == np.arange(500)).all()
    assert (dists[:, 0] == 0.0).all()
    assert (np.diff(dists, axis=1) >= 0).all()
    keys, dists = O.bruteforce(ds[:2], ds[:1], 5)
    assert list(keys[:3]) == [-1, -1, -1] and list(dists[:3]) == [0, 0, 0] and keys[3] == 0 and dists[3] == 0.0


def test_bruteforce_vs_naive_sort():
    """brute_force_test.go:156-232: random 1000x16 against a naive full sort, limits {1,5,50,1000}."""
    rng = np.random.default_rng(6)
    ds = rng.standard_normal((1000, 16)).astype(np.float32)
    qs = rng.standard_normal((7, 16)).astype(np.float32)
    full = ((qs[:, None, :].astype(np.float64) - ds[None, :, :].astype(np.float64)) ** 2).sum(-1)
    for limit in (1, 5, 50, 1000):
        keys, dists = O.bruteforce(ds, qs, limit)
        keys = keys.reshape(7, limit); dists = dists.reshape(7, limit)
        for q in range(7):
            order = np.argsort(full[q], kind="stable")[:limit]
            np.testing.assert_allclose(dists[q], full[q][order], rtol=1e-5)
            assert (np.diff(dists[q]) >= 0).all()
            assert set(keys[q]) == set(order) or np.allclose(np.sort(full[q][keys[q]]), full[q][order], rtol=1e-6)


def test_aggregate_kats():
    """sumavg2_test.go / count2_test.go: values 1..10 with and without nulls."""
    k = load("agg_kat.json")
    lib = O.go()
    for T, dt in ((20, np.int8), (22, np.int32), (23, np.int64)):
        v = np.asarray(k["values"], dtype=dt)
        s = np.zeros(1, dtype=np.int64); nul = np.ones(1, dtype=np.uint8); c = np.zeros(1, dtype=np.int64)
        assert lib.og_sum_int64(T, O.p(v), None, 0, None, len(v), O.p(s), O.p(nul), O.p(c), None) == 0
        assert s[0] == k["sum_all"] and c[0] == k["count_all"] and nul[0] == 0
        mask = np.zeros(len(v), dtype=bool); mask[k["null_rows_example"]] = True
        from matrixone_b200.vector import bitmap_from_bools
        bm = bitmap_from_bools(mask)
        s[:] = 0; nul[:] = 1; c[:] = 0
        lib.og_sum_int64(T, O.p(v), O.p(bm), 0, None, len(v), O.p(s), O.p(nul), O.p(c), None)
        assert s[0] == k["sum_with_nulls"] and c[0] == k["count_with_nulls"]
    for T, dt in ((30, np.float32), (31, np.float64)):
        v = np.asarray(k["values"], dtype=dt)
        s = np.zeros(1, dtype=np.float64); nul = np.ones(1, dtype=np.uint8); c = np.zeros(1, dtype=np.int64)
        lib.og_sum_float64(T, O.p(v), None, 0, None, len(v), O.p(s), O.p(nul), O.p(c))
        assert abs(s[0] - k["sum_all"]) < k["tolerance_abs"] and abs(s[0] / c[0] - k["avg_all"]) < k["tolerance_abs"]


def test_sum_int64_overflow_is_prefix_order_dependent():
    """int64OfCheck (sumavg2.go:89-94) fires on the running sum: [MAX, 1, -5] errors although the total fits."""
    lib = O.go()
    v = np.asarray([np.iinfo(np.int64).max, 1, -5], dtype=np.int64)
    s = np.zeros(1, dtype=np.int64); nul = np.ones(1, dtype=np.uint8); row = np.zeros(1, dtype=np.int64)
    assert lib.og_sum_int64(23, O.p(v), None, 0, None, 3, O.p(s), O.p(nul), None, O.p(row)) == 20201 and row[0] == 1
    v2 = np.asarray([np.iinfo(np.int64).max, -5, 1], dtype=np.int64)
    s[:] = 0
    assert lib.og_sum_int64(23, O.p(v2), None, 0, None, 3, O.p(s), O.p(nul), None, None) == 0
    assert s[0] == np.iinfo(np.int64).max - 4


def test_go_arith_overflow_semantics():
    """arithmetic_overflow_check.go: exact detection, error at the FIRST offending row, later rows untouched."""
    lib = O.go()
    a = np.asarray([1, 100, 100, 3], dtype=np.int8); b = np.asarray([2, 27, 28, 4], dtype=np.int8)
    r = np.full(4, -7, dtype=np.int8); rn = np.zeros(1, dtype=np.uint64); row = np.full(1, -1, dtype=np.int64)
    rc = lib.og_arith(0, 20, O.p(r), O.p(a), O.p(b), 4, 0, 0, None, None, O.p(rn), 0, O.p(row))
    assert rc == 20201 and row[0] == 2 and list(r) == [3, 127, -7, -7]
    # int16 multiply IS detected by the Go path (the C path never trips, SURVEY appendix)
    a = np.asarray([300], dtype=np.int16); b = np.asarray([300], dtype=np.int16); r = np.zeros(1, dtype=np.int16); rn[:] = 0
    assert lib.og_arith(2, 21, O.p(r), O.p(a), O.p(b), 1, 0, 0, None, None, O.p(rn), 0, O.p(row)) == 20201


def test_three_valued_logic_truth_tables():
    """logicalOperator.go:36-168 against the SQL truth tables printed in cgo/logic.c:19-31,95-108."""
    lib = O.go()
    T, F, N = 1, 0, None
    vals = [T, F, N]
    for is_or in (0, 1):
        a_vals, b_vals, want = [], [], []
        for x in vals:
            for y in vals:
                a_vals.append(x); b_vals.append(y)
                if is_or:
                    want.append(T if (x == T or y == T) else (N if (x is N or y is N) else F))
                else:
                    want.append(F if (x == F or y == F) else (N if (x is N or y is N) else T))
        n = len(a_vals)
        a = np.asarray([v or 0 for v in a_vals], dtype=np.uint8); b = np.asarray([v or 0 for v in b_vals], dtype=np.uint8)
        from matrixone_b200.vector import bitmap_from_bools, bitmap_to_bools
        an = bitmap_from_bools([v is N for v in a_vals]); bn = bitmap_from_bools([v is N for v in b_vals])
        r = np.zeros(n, dtype=np.uint8); rn = np.zeros(1, dtype=np.uint64)
        cols = (C.c_void_p * 2)(O.p(a), O.p(b)); nulls = (C.c_void_p * 2)(O.p(an), O.p(bn)); kind = (C.c_int32 * 2)(0, 0)
        lib.og_multi_logic(is_or, O.p(r), O.p(rn), 2, cols, nulls, kind, n)
        rnb = bitmap_to_bools(rn, n)
        for i in range(n):
            if want[i] is N:
                assert rnb[i], (is_or, a_vals[i], b_vals[i])
            else:
                assert not rnb[i] and r[i] == want[i], (is_or, a_vals[i], b_vals[i])


def test_q6_pipeline_matches_direct_formula_and_threads():
    from matrixone_b200 import datagen
    n = 100_000
    cols = datagen.lineitem(10, 0, n)
    P = datagen.q6_params()
    s1, ns1, nul1 = O.q6(cols, n, P, nthreads=1)
    m = ((cols["shipdate"] >= P[0]) & (cols["shipdate"] < P[1]) & (cols["discount"] >= P[2]) & (cols["discount"] <= P[3]) & (cols["quantity"] < P[4]))
    prod = cols["extendedprice"][m] * cols["discount"][m]
    serial = 0.0
    for x in prod:
        serial += x
    assert ns1 == int(m.sum()) and s1 == serial and not nul1          # single pipeline == strict serial order
    s4, ns4, _ = O.q6(cols, n, P, nthreads=4)
    assert ns4 == ns1 and abs(s4 - s1) <= 1e-9 * abs(s1)              # worker partials re-associate
    assert 0.01 < ns1 / n < 0.03                                       # ~1.8 % selectivity (SURVEY 8(d))


def test_q1_pipeline_groups_and_counts():
    from matrixone_b200 import datagen
    n = 200_000
    cols = datagen.lineitem(11, 0, n)
    g1 = O.q1(cols, n, datagen.Q1_CUTOFF, nthreads=1)
    assert 3 <= len(g1) <= 6
    m = cols["shipdate"] <= datagen.Q1_CUTOFF
    assert sum(g["count_order"] for g in g1) == int(m.sum())
    for g in g1:
        sel = m & (cols["returnflag"] == g["returnflag"]) & (cols["linestatus"] == g["linestatus"])
        assert g["count_order"] == int(sel.sum())
        assert g["first_row"] == int(np.flatnonzero(sel)[0])
        np.testing.assert_allclose(g["sum_qty"], cols["quantity"][sel].sum(), rtol=1e-12)
        ch = cols["extendedprice"][sel] * (1 - cols["discount"][sel]) * (1 + cols["tax"][sel])
        np.testing.assert_allclose(g["sum_charge"], ch.sum(), rtol=1e-11)
    g3 = O.q1(cols, n, datagen.Q1_CUTOFF, nthreads=3)
    assert [(g["returnflag"], g["linestatus"], g["count_order"]) for g in g3] == [(g["returnflag"], g["linestatus"], g["count_order"]) for g in g1]


def test_reference_c_agrees_with_restatement_where_semantics_coincide(ref_tape):
    """libmo_ref.so (reference C, unchanged; its results recorded in tests/golden/ref_test_oracle_golden.npz) vs the Go restatement:
    float add/sub/mul are single IEEE ops in both."""
    ref, lib = original(O.ref), O.go()
    rng = np.random.default_rng(1)
    a = rng.standard_normal(8192); b = rng.standard_normal(8192)
    for name, op in (("Float_VecAdd", 0), ("Float_VecSub", 1), ("Float_VecMul", 2)):
        r1 = np.zeros(8192); r2 = np.zeros(8192); rn = np.zeros(128, dtype=np.uint64)
        rc1, d1 = ref_tape(lambda: (getattr(ref, name)(O.p(r1), O.p(a), O.p(b), 8192, None, 0, 8), r1))
        assert rc1 == 0
        assert lib.og_arith(op, 31, O.p(r2), O.p(a), O.p(b), 8192, 0, 0, None, None, O.p(rn), 0, None) == 0
        assert d1 == digest(r2)
    # the XCall L2 of the reference (double accumulation) stays within 1e-6 of the Go f32-accumulating metric
    from matrixone_b200.vector import varlena_column_from_matrix, Vector
    from matrixone_b200 import capi
    m1 = rng.standard_normal((64, 768)).astype(np.float32); m2 = rng.standard_normal((64, 768)).astype(np.float32)
    c1, a1 = varlena_column_from_matrix(m1); c2, a2 = varlena_column_from_matrix(m2)
    res = np.zeros(64)
    args = (capi.XCallArgs * 3)(Vector(data=res, length=64).fill_raw_ptr_len(), Vector(data=c1, area=a1, length=64).fill_raw_ptr_len(),
                                Vector(data=c2, area=a2, length=64).fill_raw_ptr_len())
    err = (C.c_uint8 * 256)()
    rc, res = ref_tape(lambda: (ref.XCall(0, 2, err, C.cast(args, C.c_void_p), 64), res), keep=True)
    assert rc == 0
    want = np.zeros(64)
    lib.og_distance_rows_f32(4, O.p(want), O.p(m1), 768, O.p(m2), 768, 768, 64, None)
    np.testing.assert_allclose(res, want, rtol=1e-5)


def test_usearch_exact_search_agrees_on_l2sq_ranking(ref_tape):
    """UsearchBruteForceIndex.Search -> usearch_exact_search (brute_force.go:143-221): same neighbours as the Go index."""
    us = original(O.usearch)
    rng = np.random.default_rng(3)
    ds = rng.standard_normal((2000, 64)).astype(np.float32); qs = rng.standard_normal((16, 64)).astype(np.float32)
    k = 5
    keys = np.zeros((16, k), dtype=np.uint64); dist = np.zeros((16, k), dtype=np.float32)

    def search():
        err = C.c_char_p()
        # scalar_kind f32 = 2? metric l2sq: resolved from the header enum order (usearch.h): unknown=0, f32=1 ... ; metric: unknown=0, cos=1, ip=2, l2sq=3
        us.usearch_exact_search(O.p(ds), 2000, 64 * 4, O.p(qs), 16, 64 * 4, 1, 64, 3, k, 1, O.p(keys), k * 8, O.p(dist), k * 4, C.byref(err))
        return bool(err.value), keys, dist
    failed, keys, dist = ref_tape(search, keep=True)
    assert not failed
    gk, gd = O.bruteforce(ds, qs, k)
    gk = gk.reshape(16, k); gd = gd.reshape(16, k)
    np.testing.assert_allclose(dist, gd, rtol=1e-5)
    assert (keys.astype(np.int64) == gk).mean() > 0.98
