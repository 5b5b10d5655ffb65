"""C-ABI checks that need no GPU: the library loads, exports every symbol include/mo_b200.h declares, struct layouts
match the header, and -- with no CUDA device -- every entry point FAILS LOUDLY instead of computing on the CPU."""
import ctypes as C
import glob
import os
import re

import numpy as np
import pytest

from matrixone_b200 import capi
from matrixone_b200.vector import Vector, xcall
from oracle import build as oracle_build
from ref_tape import original

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mo_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?(?:void|bool|int32_t|uint64_t|char)\s*\*?\s*([A-Z][A-Za-z0-9_]+)\s*\(", src, flags=re.M)
    return sorted(set(names))


def test_header_symbols_all_exported(lib):
    names = declared_symbols()
    assert len(names) >= 50, names
    for n in names:
        assert hasattr(lib, n), "declared in mo_b200.h but not exported: " + n
    # and the Python prototypes cover the whole header
    assert set(names) == set(capi.PROTOTYPES), set(names) ^ set(capi.PROTOTYPES)


def test_reference_mo_h_surface_is_complete(lib, ref_tape):
    """every prototype of the reference's cgo/mo.h:24-73 (listed here by name) is exported with that exact name"""
    ref_names = ["Bitmap_Add", "Bitmap_Remove", "Bitmap_Contains", "Bitmap_IsEmpty", "Bitmap_Count", "Bitmap_And", "Bitmap_Or", "Bitmap_Not",
                 "SignedInt_VecAdd", "UnsignedInt_VecAdd", "Float_VecAdd", "SignedInt_VecSub", "UnsignedInt_VecSub", "Float_VecSub",
                 "SignedInt_VecMul", "UnsignedInt_VecMul", "Float_VecMul", "Float_VecDiv", "Float_VecIntegerDiv",
                 "SignedInt_VecMod", "UnsignedInt_VecMod", "Float_VecMod",
                 "Numeric_VecEq", "Numeric_VecNe", "Numeric_VecGt", "Numeric_VecGe", "Numeric_VecLt", "Numeric_VecLe",
                 "Logic_VecAnd", "Logic_VecOr", "Logic_VecXor", "Logic_VecNot", "XCall"]
    for n in ref_names:
        assert hasattr(lib, n)
    def prototypes():    # the real header, recorded in tests/golden/ref_test_abi.npz
        src = open(os.path.join(original(lambda: oracle_build.REF), "cgo", "mo.h")).read()
        return np.array(re.findall(r"^\s*(?:void|bool|int32_t|uint64_t)\s+([A-Za-z_0-9]+)\s*\(", src, flags=re.M))
    found = ref_tape(prototypes, keep=True)
    assert sorted(found) == sorted(ref_names)


def test_struct_layouts():
    assert C.sizeof(capi.XCallArgs) == 48            # cgo/xcall.h:24-31: 6 x 8 bytes
    assert C.sizeof(capi.Q6Params) == 32
    assert C.sizeof(capi.Q1Group) == 88
    assert C.sizeof(capi.Q1Result) == 8 + 8 * 88
    assert C.sizeof(capi.SearchParams) == 56


def test_version_and_launch_counter(lib):
    assert b"sm_100a" in lib.MoB200_Version()
    assert lib.MoB200_KernelLaunchCount() >= 0


@pytest.mark.skipif(bool(glob.glob("/dev/nvidia[0-9]*")), reason="a GPU is present; the no-device behaviour is tested on CPU boxes")
def test_no_gpu_fails_loudly(lib):
    """no CUDA device => rc != 0 and an error text; results are never produced by a CPU path"""
    assert lib.MoB200_DeviceCount() == 0
    assert lib.MoB200_Init(-1) == capi.RC_INTERNAL_ERROR
    a = np.arange(8, dtype=np.int32); b = np.ones(8, dtype=np.int32); r = np.full(8, -1, dtype=np.int32)
    rc = lib.SignedInt_VecAdd(r.ctypes.data, a.ctypes.data, b.ctypes.data, 8, None, 0, 4)
    assert rc == capi.RC_INTERNAL_ERROR and (r == -1).all()
    assert "no CUDA device" in capi.last_error(lib)
    res = np.zeros(1, dtype=np.int64)
    rc, msg = xcall(capi.XCALL_AGG(capi.AGG_SUM, capi.T_INT64), [Vector(data=res, length=1), Vector(data=np.arange(4, dtype=np.int64))], 4,
                    raise_on_error=False)
    assert rc == capi.RC_INTERNAL_ERROR and "no CUDA device" in msg    # Pascal errStr, cxcall.go:76-89
    rc, _ = xcall(999999, [Vector(data=res, length=1)], 1, raise_on_error=False)
    assert rc in (-1, capi.RC_INTERNAL_ERROR)


def test_missing_library_raises_importerror(tmp_path):
    with pytest.raises(ImportError):
        capi.load_library(str(tmp_path / "libmo_b200.so"))


def test_bloom_header_symbols_exported_and_match_the_reference_header(lib, ref_tape):
    """include/mo_b200_bloom.h == the prototypes of the reference's cgo/bloom.h, every one exported; the host-only entry points (init, marshal,
    unmarshal, free: no GPU work) behave like cgo/bloom.c:98-135,321-339"""
    def protos(path):
        src = re.sub(r"/\*.*?\*/", "", open(path).read(), flags=re.S)
        return sorted(set(re.findall(r"^\s*(?:const\s+)?(?:void|bool|int|uint8_t|bloomfilter_t)\s*\*?\s*(bloomfilter_[a-z0-9_]+)\s*\(", src, flags=re.M)))
    names = protos(os.path.join(ROOT, "include", "mo_b200_bloom.h"))
    assert len(names) == 18, names
    for n in names:
        assert hasattr(lib, n), n
    ref_names = ref_tape(lambda: np.array(protos(os.path.join(original(lambda: oracle_build.REF), "cgo", "bloom.h"))), keep=True)
    assert [n for n in ref_names if not n.startswith("bloomfilter_get_")] == names
    lib.bloomfilter_init_with_seed.restype = C.c_void_p; lib.bloomfilter_init_with_seed.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64]
    lib.bloomfilter_marshal.restype = C.c_void_p; lib.bloomfilter_marshal.argtypes = [C.c_void_p, C.POINTER(C.c_size_t)]
    lib.bloomfilter_unmarshal.restype = C.c_void_p; lib.bloomfilter_unmarshal.argtypes = [C.c_void_p, C.c_size_t]
    lib.bloomfilter_free.restype = None; lib.bloomfilter_free.argtypes = [C.c_void_p]
    bf = lib.bloomfilter_init_with_seed(1000, 3, 42)        # nbits rounds up to a power of two (bloom.c:119)
    n = C.c_size_t()
    p = lib.bloomfilter_marshal(bf, C.byref(n))
    raw = C.string_at(p, n.value)
    assert n.value == 32 + 1024 // 8 and raw[:4] == b"XXBF"
    hdr = np.frombuffer(raw[:24], dtype=np.uint8)
    assert hdr[4:8].view(np.uint32)[0] == 3 and hdr[8:16].view(np.uint64)[0] == 1024 and hdr[16:24].view(np.uint64)[0] == 42
    assert not any(raw[24:24 + 128])
    assert lib.bloomfilter_init_with_seed(64, 65, 0) is None          # k > MAX_K_SEED
    buf = np.frombuffer(raw, np.uint8).copy()
    assert lib.bloomfilter_unmarshal(buf.ctypes.data, buf.nbytes) == buf.ctypes.data
    assert lib.bloomfilter_unmarshal(buf.ctypes.data, 8) is None
    buf[0] = 0
    assert lib.bloomfilter_unmarshal(buf.ctypes.data, buf.nbytes) is None
    lib.bloomfilter_free(bf)
