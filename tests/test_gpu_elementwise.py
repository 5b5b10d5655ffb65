"""GPU parity: the mo.h batch operators against the reference C compiled unchanged (oracle/_ref/libmo_ref.so, its results recorded in
tests/golden/ref_test_gpu_elementwise.npz), bit-exact for results, return codes and nulls.  Host-pointer and device-pointer (resident) paths."""
import numpy as np
import pytest

import oracle_lib as O
from matrixone_b200 import capi
from matrixone_b200.vector import DeviceBuffer, bitmap_from_bools
from ref_tape import digest, original

pytestmark = pytest.mark.gpu

INT_T = {1: (np.int8, np.uint8), 2: (np.int16, np.uint16), 4: (np.int32, np.uint32), 8: (np.int64, np.uint64)}


def _rand(rng, dt, n, wide=True):
    info = np.iinfo(dt)
    if wide:
        return rng.integers(info.min, info.max, size=n, dtype=dt, endpoint=True)
    lim = int(min(info.max, 100))
    return rng.integers(max(info.min, -lim), lim, size=n, dtype=dt, endpoint=True)


@pytest.mark.parametrize("n", [1, 7, 64, 8192, 100_003])
@pytest.mark.parametrize("flag", [0, 1, 2])
def test_int_arith_bit_exact_vs_reference_c(gpu, ref_tape, n, flag):
    ref = original(O.ref)
    rng = np.random.default_rng(n * 3 + flag)
    for szof, (sdt, udt) in INT_T.items():
        for kind, dt in (("SignedInt", sdt), ("UnsignedInt", udt)):
            for op in ("Add", "Sub", "Mul", "Mod"):
                for wide in (False, True):
                    a = _rand(rng, dt, n, wide); b = _rand(rng, dt, n, wide)
                    if op == "Mod":
                        b[b == 0] = 1           # division by zero has its own test
                        if kind == "SignedInt":
                            b[b == -1] = 2      # INT_MIN % -1 traps in the reference C
                    nulls = bitmap_from_bools(rng.random(n) < 0.2) if (n % 2) else None
                    name = "%s_Vec%s" % (kind, op)
                    r0 = _rand(rng, dt, n)
                    r1 = r0.copy(); r2 = r0.copy()
                    rc1, d1 = ref_tape(lambda: (getattr(ref, name)(O.p(r1), O.p(a), O.p(b), n, O.p(nulls), flag, szof), r1))
                    rc2 = getattr(gpu, name)(O.p(r2), O.p(a), O.p(b), n, O.p(nulls), flag, szof)
                    assert rc1 == rc2, (name, szof, n, flag, wide, rc1, rc2)
                    assert d1 == digest(r2), (name, szof, n, flag, wide)


def test_mul_overflow_flag_is_decided_by_last_row_only(gpu, ref_tape):
    """arith.c:115,129 assigns opflag per element: an overflow in the middle is forgotten, one at the end is reported"""
    ref = original(O.ref)
    a = np.asarray([2**40, 2, 3], dtype=np.int64); b = np.asarray([2**40, 2, 3], dtype=np.int64)
    for arr_a, arr_b in ((a, b), (a[::-1].copy(), b[::-1].copy())):
        r1 = np.zeros(3, dtype=np.int64); r2 = np.zeros(3, dtype=np.int64)
        rc1, d1 = ref_tape(lambda: (ref.SignedInt_VecMul(O.p(r1), O.p(arr_a), O.p(arr_b), 3, None, 0, 8), r1))
        rc2 = gpu.SignedInt_VecMul(O.p(r2), O.p(arr_a), O.p(arr_b), 3, None, 0, 8)
        assert rc1 == rc2 and d1 == digest(r2)
    # equal operands never trip ((A ^ B) > 0 is false), int16 never trips: quirks kept
    x = np.asarray([100], dtype=np.int8); r = np.zeros(1, dtype=np.int8)
    assert gpu.SignedInt_VecMul(O.p(r), O.p(x), O.p(x), 1, None, 0, 1) == ref_tape(lambda: ref.SignedInt_VecMul(O.p(r), O.p(x), O.p(x), 1, None, 0, 1)) == 0
    y = np.asarray([300], dtype=np.int16); z = np.asarray([-300], dtype=np.int16); r = np.zeros(1, dtype=np.int16)
    assert gpu.SignedInt_VecMul(O.p(r), O.p(y), O.p(z), 1, None, 0, 2) == 0


@pytest.mark.parametrize("n", [5, 8192, 70_001])
def test_float_arith_vs_reference_c(gpu, ref_tape, n):
    ref = original(O.ref)
    lib = O.go()
    rng = np.random.default_rng(n)
    for szof, dt in ((4, np.float32), (8, np.float64)):
        a = rng.standard_normal(n).astype(dt) * 1000; b = rng.standard_normal(n).astype(dt)
        b[::17] = 0
        nulls = bitmap_from_bools(rng.random(n) < 0.1)
        for flag in (0, 1, 2):
            for name in ("Float_VecAdd", "Float_VecSub", "Float_VecMul", "Float_VecDiv", "Float_VecMod"):
                r1 = np.full(n, 7, dtype=dt); r2 = r1.copy()
                scalar_div = name in ("Float_VecDiv",) and flag == 2
                rc1, out1 = ref_tape(lambda: (getattr(ref, name)(O.p(r1), O.p(a), O.p(b), n, O.p(nulls), flag, szof), r1), keep=scalar_div)
                rc2 = getattr(gpu, name)(O.p(r2), O.p(a), O.p(b), n, O.p(nulls), flag, szof)
                assert rc1 == rc2, (name, flag, rc1, rc2)
                if scalar_div:
                    # -ffast-math turns x / scalar into x * (1/scalar) in the reference build: 1 ulp apart; IEEE here
                    np.testing.assert_allclose(r2, out1, rtol=4 * np.finfo(dt).eps)
                else:
                    assert out1 == digest(r2), (name, flag, szof)
        # integer division of floats
        bb = b.copy(); bb[bb == 0] = 3
        r1 = np.zeros(n, dtype=np.int64); r2 = np.zeros(n, dtype=np.int64)
        rc1, d1 = ref_tape(lambda: (ref.Float_VecIntegerDiv(O.p(r1), O.p(a), O.p(bb), n, None, 0, szof), r1))
        assert rc1 == gpu.Float_VecIntegerDiv(O.p(r2), O.p(a), O.p(bb), n, None, 0, szof) == 0
        assert d1 == digest(r2)
        # quotients outside int64 / NaN: the reference's cvttsd2si yields INT64_MIN ("integer indefinite"), not a saturated value
        big = np.array([1e30, -1e30, np.inf, -np.inf, np.nan, 9.3e18, -9.3e18, 5.0], dtype=dt); one = np.array([1e-3, 1e-3, 1, 1, 1, 1, 1, 2], dtype=dt)
        q1 = np.zeros(8, dtype=np.int64); q2 = np.zeros(8, dtype=np.int64)
        rc1, d1 = ref_tape(lambda: (ref.Float_VecIntegerDiv(O.p(q1), O.p(big), O.p(one), 8, None, 0, szof), q1))
        assert rc1 == gpu.Float_VecIntegerDiv(O.p(q2), O.p(big), O.p(one), 8, None, 0, szof) == 0
        assert d1 == digest(q2), q2
        # division: bit-exact against the IEEE restatement of the Go "/" operator (null on zero divisor)
        rn = np.zeros((n + 63) // 64, dtype=np.uint64); rg = np.full(n, 7, dtype=dt); r2 = np.full(n, 7, dtype=dt)
        lib.og_arith(3, 30 if szof == 4 else 31, O.p(rg), O.p(a), O.p(b), n, 0, 0, None, None, O.p(rn), 1, None)
        assert gpu.Float_VecDiv(O.p(r2), O.p(a), O.p(b), n, None, 0, szof) == capi.RC_DIVISION_BY_ZERO
        assert np.array_equal(rg, r2, equal_nan=True)


def test_div_and_mod_by_zero_rc(gpu, ref_tape):
    ref = original(O.ref)
    a = np.asarray([10, 20, 30], dtype=np.int32); b = np.asarray([3, 0, 7], dtype=np.int32)
    r1 = np.full(3, -9, dtype=np.int32); r2 = r1.copy()
    rc1, d1 = ref_tape(lambda: (ref.SignedInt_VecMod(O.p(r1), O.p(a), O.p(b), 3, None, 0, 4), r1))
    assert rc1 == gpu.SignedInt_VecMod(O.p(r2), O.p(a), O.p(b), 3, None, 0, 4) == capi.RC_DIVISION_BY_ZERO
    assert d1 == digest(r2) and r2[1] == -9     # the offending row keeps its old value
    assert gpu.SignedInt_VecAdd(O.p(r2), O.p(a), O.p(b), 3, None, 0, 3) == capi.RC_INVALID_ARGUMENT   # bad szof


CMP_TYPES = [(capi.T_INT8, np.int8), (capi.T_INT16, np.int16), (capi.T_INT32, np.int32), (capi.T_INT64, np.int64),
             (capi.T_UINT8, np.uint8), (capi.T_UINT16, np.uint16), (capi.T_UINT32, np.uint32), (capi.T_UINT64, np.uint64),
             (capi.T_FLOAT32, np.float32), (capi.T_FLOAT64, np.float64), (capi.T_DATE, np.int32), (capi.T_TIME, np.int64),
             (capi.T_DATETIME, np.int64), (capi.T_TIMESTAMP, np.int64), (capi.T_BOOL, np.uint8)]


@pytest.mark.parametrize("n", [3, 8192, 50_001])
def test_compare_bit_exact_vs_reference_c(gpu, ref_tape, n):
    ref = original(O.ref)
    rng = np.random.default_rng(n + 9)
    for T, dt in CMP_TYPES:
        if T == capi.T_BOOL:
            a = rng.integers(0, 2, n).astype(np.uint8); b = rng.integers(0, 2, n).astype(np.uint8)
        elif np.issubdtype(dt, np.floating):
            a = rng.integers(-5, 5, n).astype(dt); b = rng.integers(-5, 5, n).astype(dt)
        else:
            a = rng.integers(0, 6, n).astype(dt); b = rng.integers(0, 6, n).astype(dt)
        nulls = bitmap_from_bools(rng.random(n) < 0.15)
        for flag in (0, 1, 2):
            for op in ("Eq", "Ne", "Gt", "Ge", "Lt", "Le"):
                for nl in (None, nulls):
                    r1 = np.full(n, 5, dtype=np.uint8); r2 = r1.copy()
                    rc1, d1 = ref_tape(lambda: (getattr(ref, "Numeric_Vec" + op)(O.p(r1), O.p(a), O.p(b), n, O.p(nl), flag, T), r1))
                    rc2 = getattr(gpu, "Numeric_Vec" + op)(O.p(r2), O.p(a), O.p(b), n, O.p(nl), flag, T)
                    assert rc1 == rc2 == 0 and d1 == digest(r2), (T, op, flag)
    r = np.zeros(4, dtype=np.uint8)
    assert gpu.Numeric_VecEq(O.p(r), O.p(r), O.p(r), 4, None, 0, 99) == capi.RC_INVALID_ARGUMENT


@pytest.mark.parametrize("n", [9, 64, 200, 8192, 33_333])
def test_three_valued_logic_bit_exact_vs_reference_c(gpu, ref_tape, n):
    ref = original(O.ref)
    rng = np.random.default_rng(n + 77)
    a = rng.integers(0, 2, n).astype(np.uint8); b = rng.integers(0, 2, n).astype(np.uint8)
    an = bitmap_from_bools(rng.random(n) < 0.3); bn = bitmap_from_bools(rng.random(n) < 0.3)
    for name in ("Logic_VecAnd", "Logic_VecOr"):
        for flag in (0, 1, 2):
            for (xa, xb) in ((an, bn), (an, None), (None, bn), (None, None)):
                rn0 = np.zeros_like(an)
                if xa is not None: rn0 |= xa
                if xb is not None: rn0 |= xb
                if flag:  # scalar operand: the caller pre-fills rnulls with the vector side's nulls
                    rn0 = (bn if flag == 1 else an).copy()
                r1 = np.full(n, 9, dtype=np.uint8); r2 = r1.copy(); rn1 = rn0.copy(); rn2 = rn0.copy()
                rc1, d1, dn1 = ref_tape(lambda: (getattr(ref, name)(O.p(r1), O.p(a), O.p(b), n, O.p(xa), O.p(xb), O.p(rn1), flag), r1, rn1))
                rc2 = getattr(gpu, name)(O.p(r2), O.p(a), O.p(b), n, O.p(xa), O.p(xb), O.p(rn2), flag)
                assert rc1 == rc2 == 0 and d1 == digest(r2) and dn1 == digest(rn2), (name, flag)
    for flag in (0, 1, 2):
        r1 = np.full(n, 9, dtype=np.uint8); r2 = r1.copy()
        _, d1 = ref_tape(lambda: (ref.Logic_VecXor(O.p(r1), O.p(a), O.p(b), n, None, flag), r1)); gpu.Logic_VecXor(O.p(r2), O.p(a), O.p(b), n, None, flag)
        assert d1 == digest(r2)
    for flag in (0, 1):
        r1 = np.full(n, 9, dtype=np.uint8); r2 = r1.copy()
        _, d1 = ref_tape(lambda: (ref.Logic_VecNot(O.p(r1), O.p(a), n, None, flag), r1)); gpu.Logic_VecNot(O.p(r2), O.p(a), n, None, flag)
        assert d1 == digest(r2)      # scalar flag writes only r[0] (logic.c:214-216)


@pytest.mark.parametrize("nbits", [1, 63, 64, 65, 8192, 100_001])
def test_bitmap_ops_bit_exact_vs_reference_c(gpu, ref_tape, nbits):
    ref = original(O.ref)
    rng = np.random.default_rng(nbits)
    nw = (nbits + 63) // 64
    a = rng.integers(0, 2**63, nw, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, nw, dtype=np.uint64)
    b = rng.integers(0, 2**63, nw, dtype=np.uint64)
    assert gpu.Bitmap_Count(O.p(a), nbits) == ref_tape(lambda: ref.Bitmap_Count(O.p(a), nbits))        # last word masked (bitmap.h:110-131)
    z = np.zeros(nw, dtype=np.uint64)
    assert gpu.Bitmap_IsEmpty(O.p(z), nbits) and not gpu.Bitmap_IsEmpty(O.p(a | np.uint64(1)), nbits)
    for name in ("Bitmap_And", "Bitmap_Or"):
        d1 = np.zeros(nw, dtype=np.uint64); d2 = np.zeros(nw, dtype=np.uint64)
        _, w = ref_tape(lambda: (getattr(ref, name)(O.p(d1), O.p(a), O.p(b), nbits), d1)); getattr(gpu, name)(O.p(d2), O.p(a), O.p(b), nbits)
        assert w == digest(d2)
    d1 = np.zeros(nw, dtype=np.uint64); d2 = np.zeros(nw, dtype=np.uint64)
    _, w = ref_tape(lambda: (ref.Bitmap_Not(O.p(d1), O.p(a), nbits), d1)); gpu.Bitmap_Not(O.p(d2), O.p(a), nbits)
    assert w == digest(d2)
    w1 = a.copy(); w2 = a.copy()
    pos = nbits - 1
    _, w = ref_tape(lambda: (ref.Bitmap_Add(O.p(w1), pos), w1)); gpu.Bitmap_Add(O.p(w2), pos)
    assert w == digest(w2) and gpu.Bitmap_Contains(O.p(w2), pos)
    _, w = ref_tape(lambda: (ref.Bitmap_Remove(O.p(w1), pos), w1)); gpu.Bitmap_Remove(O.p(w2), pos)
    assert w == digest(w2) and not gpu.Bitmap_Contains(O.p(w2), pos) and not gpu.Bitmap_Contains(None, 3)


def test_resident_device_pointers_zero_copy(gpu, ref_tape):
    """the same entry points on DEVICE pointers (resident columns): nothing is staged, results stay in HBM"""
    ref = original(O.ref)
    rng = np.random.default_rng(4)
    n = 1 << 20
    a = rng.integers(-1000, 1000, n).astype(np.int64); b = rng.integers(-1000, 1000, n).astype(np.int64)
    da, db = DeviceBuffer.from_numpy(a), DeviceBuffer.from_numpy(b)
    dr = DeviceBuffer(8 * n); dc = DeviceBuffer(n)
    assert gpu.SignedInt_VecAdd(dr.ptr, da.ptr, db.ptr, n, None, 0, 8) == 0
    assert (dr.to_numpy(np.int64) == a + b).all()
    assert gpu.Numeric_VecLt(dc.ptr, da.ptr, db.ptr, n, None, 0, capi.T_INT64) == 0
    r1 = np.zeros(n, dtype=np.uint8)
    _, d1 = ref_tape(lambda: (ref.Numeric_VecLt(O.p(r1), O.p(a), O.p(b), n, None, 0, capi.T_INT64), r1))
    assert digest(dc.to_numpy(np.uint8)) == d1
    for x in (da, db, dr, dc):
        x.free()
