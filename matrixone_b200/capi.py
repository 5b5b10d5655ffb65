"""ctypes binding of libmo_b200.so (include/mo_b200.h).

The product has NO CPU path: if the shared library is missing, or no CUDA device is present, calls fail loudly
(ImportError / MoError) -- nothing here falls back to numpy or to the oracle.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmo_b200.so")

# return codes (cgo/mo_impl.h:26-35)
RC_SUCCESS = 0
RC_INTERNAL_ERROR = 20101
RC_DIVISION_BY_ZERO = 20200
RC_OUT_OF_RANGE = 20201
RC_INVALID_ARGUMENT = 20203

# types.T ids (pkg/container/types/types.go:35-67)
T_BOOL, T_INT8, T_INT16, T_INT32, T_INT64 = 10, 20, 21, 22, 23
T_UINT8, T_UINT16, T_UINT32, T_UINT64 = 25, 26, 27, 28
T_FLOAT32, T_FLOAT64 = 30, 31
T_DATE, T_TIME, T_DATETIME, T_TIMESTAMP = 50, 51, 52, 53
NP_OF_T = {T_BOOL: np.uint8, T_INT8: np.int8, T_INT16: np.int16, T_INT32: np.int32, T_INT64: np.int64,
           T_UINT8: np.uint8, T_UINT16: np.uint16, T_UINT32: np.uint32, T_UINT64: np.uint64,
           T_FLOAT32: np.float32, T_FLOAT64: np.float64, T_DATE: np.int32, T_TIME: np.int64,
           T_DATETIME: np.int64, T_TIMESTAMP: np.int64}

# XCall funcIds
XCALL_L2DISTANCE_F32, XCALL_L2DISTANCE_F64, XCALL_L2DISTANCE_SQ_F32, XCALL_L2DISTANCE_SQ_F64 = 0, 1, 2, 3
XCALL_GO_L2_F32, XCALL_GO_L2_F64, XCALL_GO_L2SQ_F32, XCALL_GO_L2SQ_F64 = 100, 101, 102, 103
XCALL_GO_IP_F32, XCALL_GO_IP_F64, XCALL_GO_COSDIST_F32, XCALL_GO_COSDIST_F64 = 104, 105, 106, 107
XCALL_GO_COSSIM_F32, XCALL_GO_COSSIM_F64 = 108, 109
XCALL_GO_L1_F32, XCALL_GO_L1_F64 = 110, 111
XCALL_GO_NORMALIZE_L2_F32, XCALL_GO_NORMALIZE_L2_F64 = 112, 113
AGG_SUM, AGG_COUNT, AGG_MIN, AGG_MAX, AGG_AVG = 0, 1, 2, 3, 4


def XCALL_AGG(op, T):
    return 0x1000 + (op << 8) + T


def XCALL_AGG_MERGE(op, T):
    return 0x1800 + (op << 8) + T


XCALL_FILTER_SELS, XCALL_PACK_KEYS, XCALL_GROUP_IDS = 0x6000, 0x6001, 0x6002
XCALL_JOIN_SELS, XCALL_JOIN_FIND, XCALL_JOIN_PROBE = 0x6010, 0x6011, 0x6012
XCALL_PACK_STR_KEYS, XCALL_STR_GROUP_IDS = 0x6003, 0x6004
XCALL_STR_JOIN_FIND, XCALL_STR_JOIN_PROBE = 0x6013, 0x6014
STR_KEY_MAX_COLS = 16
XCALL_KMEANS_ELKAN_F32, XCALL_KMEANS_ELKAN_F64 = 0x6020, 0x6021
XCALL_LZ4_DECODE = 0x6030
XCALL_VECTOR_UNMARSHAL = 0x6031
JOIN_INNER, JOIN_LEFT, JOIN_SEMI, JOIN_ANTI = 0, 1, 2, 3


def XCALL_SHUFFLE(szof):
    return 0x6100 + szof


def XCALL_GROUP_AGG(op, T):
    return 0x6400 + (op << 8) + T


XCALL_Q6_FILTER_SUM = 0x2000
XCALL_Q1_GROUP_AGG = 0x2001
XCALL_Q6_MERGE = 0x2002
XCALL_Q1_MERGE = 0x2003
AGG_STATE_BYTES = 24
XCALL_BRUTEFORCE_TOPK_F32 = 0x3000
XCALL_IVF_TOPK_F32 = 0x3001
XCALL_TOPK_MERGE = 0x3002
METRIC_L2, METRIC_IP, METRIC_COS, METRIC_L1, METRIC_L2SQ = 0, 1, 2, 3, 4


def XCALL_GO_ARITH(op, T):
    return 0x4000 + (op << 8) + T


def XCALL_GO_COMPARE(op, T):
    return 0x4800 + (op << 8) + T


def XCALL_GO_COMPARE_F32_SCALE(op, scale):
    return 0x5200 + (op << 8) + scale


def XCALL_GO_BETWEEN(T):
    return 0x5000 + T


XCALL_GO_MULTI_AND, XCALL_GO_MULTI_OR = 0x5100, 0x5101
Q1_MAX_GROUPS = 8


class XCallArgs(C.Structure):
    """mo_xcall_args_t == cgo/xcall.h:24-31"""
    _fields_ = [("pnulls", C.c_void_p), ("nullCnt", C.c_uint64), ("pdata", C.c_void_p), ("dataSz", C.c_uint64),
                ("parea", C.c_void_p), ("areaSz", C.c_uint64)]


class StrKeyParams(C.Structure):
    """mo_str_key_params_t: width[k] = fixed element bytes of key column k, 0 = varlena"""
    _fields_ = [("ncols", C.c_int32), ("has_null", C.c_int32), ("width", C.c_int32 * STR_KEY_MAX_COLS)]


class Q6Params(C.Structure):
    _fields_ = [("date_lo", C.c_int32), ("date_hi", C.c_int32), ("disc_lo", C.c_double), ("disc_hi", C.c_double),
                ("qty_hi", C.c_double)]


class Q1Group(C.Structure):
    _fields_ = [("returnflag", C.c_uint8), ("linestatus", C.c_uint8), ("pad", C.c_uint8 * 6), ("first_row", C.c_int64),
                ("sum_qty", C.c_double), ("sum_base_price", C.c_double), ("sum_disc_price", C.c_double),
                ("sum_charge", C.c_double), ("avg_qty", C.c_double), ("avg_price", C.c_double), ("avg_disc", C.c_double),
                ("sum_disc", C.c_double), ("count_order", C.c_int64)]


class Q1Result(C.Structure):
    _fields_ = [("ngroups", C.c_int64), ("groups", Q1Group * Q1_MAX_GROUPS)]


class Q1Params(C.Structure):
    _fields_ = [("cutoff", C.c_int32), ("reserved", C.c_int32), ("row_base", C.c_int64)]


class SearchParams(C.Structure):
    _fields_ = [("n", C.c_int64), ("dim", C.c_int64), ("nq", C.c_int64), ("k", C.c_int32), ("metric", C.c_int32),
                ("nprobe", C.c_int32), ("sqrt_out", C.c_int32), ("nlist", C.c_int64), ("key_base", C.c_int64)]


_vp, _u64, _i32, _i64 = C.c_void_p, C.c_uint64, C.c_int32, C.c_int64
_ARITH = [_vp, _vp, _vp, _u64, _vp, _i32, _i32]

# name -> (restype, argtypes): every symbol include/mo_b200.h declares
PROTOTYPES = {
    "Bitmap_Add": (None, [_vp, _u64]), "Bitmap_Remove": (None, [_vp, _u64]), "Bitmap_Contains": (C.c_bool, [_vp, _u64]),
    "Bitmap_IsEmpty": (C.c_bool, [_vp, _u64]), "Bitmap_Count": (_u64, [_vp, _u64]),
    "Bitmap_And": (None, [_vp, _vp, _vp, _u64]), "Bitmap_Or": (None, [_vp, _vp, _vp, _u64]), "Bitmap_Not": (None, [_vp, _vp, _u64]),
    "Logic_VecAnd": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp, _vp, _i32]), "Logic_VecOr": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp, _vp, _i32]),
    "Logic_VecXor": (_i32, [_vp, _vp, _vp, _u64, _vp, _i32]), "Logic_VecNot": (_i32, [_vp, _vp, _u64, _vp, _i32]),
    "XCall": (_i32, [_i64, _i64, _vp, _vp, _u64]),
    "MoB200_Init": (_i32, [_i32]), "MoB200_Version": (C.c_char_p, []), "MoB200_DeviceCount": (_i32, []),
    "MoB200_DeviceAlloc": (_i32, [_u64, C.POINTER(_vp)]), "MoB200_DeviceFree": (_i32, [_vp]),
    "MoB200_HostAlloc": (_i32, [_u64, C.POINTER(_vp)]), "MoB200_HostFree": (_i32, [_vp]),
    "MoB200_HostRegister": (_i32, [_vp, _u64]), "MoB200_HostUnregister": (_i32, [_vp]),
    "MoB200_Upload": (_i32, [_vp, _vp, _u64]), "MoB200_Download": (_i32, [_vp, _vp, _u64]), "MoB200_Memset": (_i32, [_vp, _i32, _u64]),
    "MoB200_ColumnCacheConfigure": (_i32, [_u64]), "MoB200_ColumnPin": (_i32, [_vp, _u64, _u64]), "MoB200_ColumnUnpin": (_i32, [_vp]),
    "MoB200_ColumnCacheStats": (_i32, [C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64)]),
    "MoB200_JoinMapPrepare": (_i32, [_vp, _u64]), "MoB200_JoinMapRelease": (_i32, [_vp]),
    "MoB200_StrJoinMapPrepare": (_i32, [_vp, _vp, _u64]), "MoB200_StrJoinMapRelease": (_i32, [_vp]),
    "MoB200_DownloadAsync": (_i32, [_vp, _vp, _u64]), "MoB200_UploadAsync": (_i32, [_vp, _vp, _u64]),
    "MoB200_Sync": (_i32, []), "MoB200_SetStream": (_i32, [_vp]), "MoB200_TimerStart": (_i32, []),
    "MoB200_TimerStop": (_i32, [C.POINTER(C.c_float)]), "MoB200_KernelLaunchCount": (_u64, []), "MoB200_LastKernelMs": (_i32, [C.POINTER(C.c_float)]),
    "MoB200_LastError": (_i32, [C.c_char_p, _u64]), "MoB200_FlushL2": (_i32, []), "MoB200_SetTuning": (_i32, [C.c_char_p, _i32]), "MoB200_DebugBuffer": (_vp, []),
    "MoB200_GenLineitem": (_i32, [_u64, _u64, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "MoB200_GenInt64": (_i32, [_u64, _u64, _u64, _vp, _vp, C.c_uint32]),
    "MoB200_GenVectorsF32": (_i32, [_u64, _u64, _u64, _i64, _vp, _vp, _i64, C.c_float]),
    "MoB200_GatherRowsF32": (_i32, [_vp, _vp, _vp, _u64, _i64]),
    "MoB200_SearchPrepare": (_i32, [_vp, _u64, _i64]),
    "MoB200_SearchPrepareMetric": (_i32, [_vp, _u64, _i64, _i32]),
    "MoB200_SearchPrepareIvf": (_i32, [_vp, _u64, _i64, _vp, _u64, _vp]),
    "MoB200_SearchRelease": (_i32, [_vp]),
}
for _k in ("SignedInt", "UnsignedInt", "Float"):
    for _op in ("Add", "Sub", "Mul", "Mod"):
        PROTOTYPES["%s_Vec%s" % (_k, _op)] = (_i32, _ARITH)
PROTOTYPES["Float_VecDiv"] = (_i32, _ARITH)
PROTOTYPES["Float_VecIntegerDiv"] = (_i32, _ARITH)
for _op in ("Eq", "Ne", "Gt", "Ge", "Lt", "Le"):
    PROTOTYPES["Numeric_Vec%s" % _op] = (_i32, _ARITH)


class MoError(RuntimeError):
    def __init__(self, rc, msg=""):
        super().__init__("mo_b200 rc=%d %s" % (rc, msg))
        self.rc = rc


_lib = None


def load_library(path=None):
    """dlopen libmo_b200.so and attach prototypes.  Raises ImportError when the library has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ImportError("libmo_b200.so not found at %s -- run `python -m matrixone_b200.build` "
                          "(there is no CPU fallback)" % p)
    lib = C.CDLL(p)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def last_error(lib=None):
    lib = lib or load_library()
    buf = C.create_string_buffer(512)
    lib.MoB200_LastError(buf, 512)
    return buf.value.decode(errors="replace")


def check(rc, lib=None):
    if rc != 0:
        raise MoError(rc, last_error(lib))
    return rc


# ---- the generic fused operator (include/mo_b200.h MO_XCALL_PLAN)
XCALL_PLAN = 0x2100
PLAN_MAX_COLS, PLAN_MAX_PREDS, PLAN_MAX_INSTR, PLAN_MAX_KEYS, PLAN_MAX_AGGS = 12, 8, 16, 4, 12
PLAN_OP_COL, PLAN_OP_CONST, PLAN_OP_ADD, PLAN_OP_SUB, PLAN_OP_MUL, PLAN_OP_DIV = 0, 1, 2, 3, 4, 5
PLAN_CMP = {"==": 0, "!=": 1, ">": 2, ">=": 3, "<": 4, "<=": 5, "between": 6}


class PlanPred(C.Structure):
    _fields_ = [("col", C.c_int32), ("op", C.c_int32), ("lo", C.c_double), ("hi", C.c_double)]


class PlanInstr(C.Structure):
    _fields_ = [("op", C.c_int32), ("a", C.c_int32), ("b", C.c_int32), ("reserved", C.c_int32), ("imm", C.c_double)]


class PlanAgg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("value", C.c_int32)]


class Plan(C.Structure):
    _fields_ = [("ncols", C.c_int32), ("npreds", C.c_int32), ("ninstr", C.c_int32), ("nkeys", C.c_int32), ("naggs", C.c_int32), ("has_null_keys", C.c_int32),
                ("row_base", C.c_int64), ("col_type", C.c_int32 * PLAN_MAX_COLS), ("pred", PlanPred * PLAN_MAX_PREDS), ("instr", PlanInstr * PLAN_MAX_INSTR),
                ("key_col", C.c_int32 * PLAN_MAX_KEYS), ("agg", PlanAgg * PLAN_MAX_AGGS)]


class PlanHeader(C.Structure):
    _fields_ = [("ngroups", C.c_int64), ("sorted", C.c_int32), ("overflow", C.c_int32), ("reserved", C.c_int64)]


def XCALL_DEC_ARITH(op, width):
    return 0x7000 + (op << 8) + width


def XCALL_DEC_SUM(width):
    return 0x7400 + width


class DecParams(C.Structure):
    _fields_ = [("scale1", C.c_int32), ("scale2", C.c_int32), ("err_row", C.c_int64)]
