"""GPU parity: row-wise distances behind XCall.  Reference ids 0..3 against the reference C (oracle/_ref, its results recorded in
tests/golden/ref_test_gpu_distance.npz; 1e-5 relative --
the C accumulates in double under -ffast-math); new Go-semantics ids 100..109 BIT-EXACT against the oracle restatement
of pkg/vectorindex/metric/distance_func.go, plus the reference's golden vectors."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle_lib as O
from matrixone_b200 import capi
from matrixone_b200.vector import DeviceBuffer, Vector, bitmap_from_bools, varlena_column, varlena_column_from_matrix, xcall
from ref_tape import original

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _cols(m):
    cells, area = varlena_column_from_matrix(m) if m.shape[1] * m.itemsize > 23 else varlena_column(list(m), m.dtype)
    return Vector(data=cells, area=area, length=m.shape[0])


def _go_rows(kind, a, b, rnulls=None):
    n = a.shape[0]
    out = np.zeros(n)
    fn = O.go().og_distance_rows_f32 if a.dtype == np.float32 else O.go().og_distance_rows_f64
    fn(kind, O.p(out), O.p(a), a.shape[1], O.p(b), 0 if b.shape[0] == 1 else b.shape[1], a.shape[1], n, O.p(rnulls))
    return out


GO_IDS = {np.float32: {0: capi.XCALL_GO_L2_F32, 4: capi.XCALL_GO_L2SQ_F32, 1: capi.XCALL_GO_IP_F32, 2: capi.XCALL_GO_COSDIST_F32, 3: capi.XCALL_GO_L1_F32},
          np.float64: {0: capi.XCALL_GO_L2_F64, 4: capi.XCALL_GO_L2SQ_F64, 1: capi.XCALL_GO_IP_F64, 2: capi.XCALL_GO_COSDIST_F64, 3: capi.XCALL_GO_L1_F64}}


@pytest.mark.parametrize("dim", [1, 3, 4, 5, 8, 9, 31, 128, 257, 768, 1027])
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_go_semantics_distances_bit_exact(gpu, dim, dt):
    rng = np.random.default_rng(dim)
    n = 300
    a = rng.standard_normal((n, dim)).astype(dt); b = rng.standard_normal((n, dim)).astype(dt)
    a[7] = b[7]            # identical rows: l2 == 0 exactly
    a[9] = 0; b[9] = 0     # zero vectors: cosine distance 1
    for kind, fid in GO_IDS[dt].items():
        for bb, const in ((b, False), (b[:1], True)):
            want = _go_rows(kind, a, bb)
            res = np.zeros(n)
            vb = _cols(bb); vb.const = const
            xcall(fid, [Vector(data=res, length=n), _cols(a), vb], n)
            assert (res == want).all(), (kind, dim, const, np.abs(res - want).max())
            if kind in (0, 4) and not const:
                assert res[7] == 0.0
        # const FIRST argument (the kernel swaps the operand roles internally; the result must equal f(a0, b_i) evaluated in that order)
        want = _go_rows(kind, np.repeat(a[:1], n, axis=0), b)
        res = np.zeros(n)
        va = _cols(a[:1]); va.const = True
        xcall(fid, [Vector(data=res, length=n), va, _cols(b)], n)
        assert (res == want).all(), (kind, dim, "const-first", np.abs(res - want).max())


def test_reference_golden_vectors_through_xcall(gpu):
    k = json.load(open(os.path.join(G, "metric_kat.json")))
    for key, fid in (("l2", capi.XCALL_GO_L2_F64), ("l2sq", capi.XCALL_GO_L2SQ_F64), ("inner_product", capi.XCALL_GO_IP_F64),
                     ("cosine_distance", capi.XCALL_GO_COSDIST_F64), ("l1", capi.XCALL_GO_L1_F64)):
        for c in k[key]:
            a = np.asarray([c["v1"]], dtype=np.float64); b = np.asarray([c["v2"]], dtype=np.float64)
            res = np.zeros(1)
            xcall(fid, [Vector(data=res, length=1), _cols(a), _cols(b)], 1)
            assert res[0] == c["want"], (key, c, res[0])        # exact equality, like distance_func_test.go
    m = json.load(open(os.path.join(G, "moarray_kat.json")))
    for c in m["l2"]:
        dt = np.float32 if c["dtype"] == "f32" else np.float64
        res = np.zeros(1)
        xcall(capi.XCALL_GO_L2_F32 if dt == np.float32 else capi.XCALL_GO_L2_F64,
              [Vector(data=res, length=1), _cols(np.asarray([c["v1"]], dtype=dt)), _cols(np.asarray([c["v2"]], dtype=dt))], 1)
        assert res[0] == c["want"]       # 33.6749153137207 (f32 accumulate) vs 33.67491648096547 (f64)
    for c in m["cosine_similarity"]:
        dt = np.float32 if c["dtype"] == "f32" else np.float64
        res = np.zeros(1)
        xcall(capi.XCALL_GO_COSSIM_F32 if dt == np.float32 else capi.XCALL_GO_COSSIM_F64,
              [Vector(data=res, length=1), _cols(np.asarray([c["v1"]], dtype=dt)), _cols(np.asarray([c["v2"]], dtype=dt))], 1)
        assert abs(res[0] - c["want"]) <= 1e-9


def test_cosine_similarity_zero_vector_is_an_error_and_dim_mismatch(gpu):
    a = np.zeros((2, 8), dtype=np.float32); b = np.ones((2, 8), dtype=np.float32)
    res = np.zeros(2)
    rc, msg = xcall(capi.XCALL_GO_COSSIM_F32, [Vector(data=res, length=2), _cols(a), _cols(b)], 2, raise_on_error=False)
    assert rc != 0 and "zero" in msg           # distance_func.go:342-345
    rc, msg = xcall(capi.XCALL_GO_L2_F32, [Vector(data=res, length=2), _cols(a), _cols(np.ones((2, 9), dtype=np.float32))], 2, raise_on_error=False)
    assert rc == capi.RC_INVALID_ARGUMENT and "dimension" in msg


@pytest.mark.parametrize("dt,ids", [(np.float32, (0, 2)), (np.float64, (1, 3))])
def test_reference_ids_match_reference_c(gpu, ref_tape, dt, ids):
    ref = original(O.ref)
    rng = np.random.default_rng(3)
    n, dim = 1000, 768
    a = rng.standard_normal((n, dim)).astype(dt); b = rng.standard_normal((n, dim)).astype(dt)
    a[11] = b[11]
    rn = bitmap_from_bools(rng.random(n) < 0.1)
    for fid in ids:
        for bb, const in ((b, False), (b[:1], True)):
            for nulls in (None, rn):
                r1 = np.full(n, -1.0); r2 = np.full(n, -1.0)
                va, vb = _cols(a), _cols(bb)
                args = (capi.XCallArgs * 3)(Vector(data=r1, nulls=nulls, length=n).fill_raw_ptr_len(), va.fill_raw_ptr_len(), vb.fill_raw_ptr_len())
                err = (C.c_uint8 * 256)()
                rc1, want = ref_tape(lambda: (ref.XCall(0, fid, err, C.cast(args, C.c_void_p), n), r1), keep=True)
                assert rc1 == 0
                xcall(fid, [Vector(data=r2, nulls=nulls, length=n), va, vb], n, runtime_id=1)
                np.testing.assert_allclose(r2, want, rtol=1e-5, atol=0)
                if nulls is not None:
                    from matrixone_b200.vector import bitmap_to_bools
                    assert (r2[bitmap_to_bools(rn, n)] == -1.0).all()         # null rows are left unwritten (xcall.c:57)
                if not const:
                    assert r2[11] == 0.0


def test_resident_columns_and_unknown_func(gpu):
    rng = np.random.default_rng(5)
    n, dim = 4096, 768
    a = rng.standard_normal((n, dim)).astype(np.float32); q = rng.standard_normal((1, dim)).astype(np.float32)
    cells, area = varlena_column_from_matrix(a)
    dc, da = DeviceBuffer.from_numpy(cells), DeviceBuffer.from_numpy(area)
    dr = DeviceBuffer(8 * n)
    qc, qa = varlena_column_from_matrix(q)
    xcall(capi.XCALL_GO_L2SQ_F32, [Vector(data_ptr=dr.ptr, data_nbytes=8 * n, length=n),
                                   Vector(data_ptr=dc.ptr, data_nbytes=dc.nbytes, area_ptr=da.ptr, area_nbytes=da.nbytes, length=n),
                                   Vector(data=qc, area=qa, length=n, const=True)], n)
    assert (dr.to_numpy(np.float64) == _go_rows(4, a, q)).all()
    rc, _ = xcall(77, [Vector(data=np.zeros(1), length=1)], 1, raise_on_error=False)
    assert rc == -1                       # unknown funcId, cgo/mo.c:64-67
    for b in (dc, da, dr):
        b.free()
