// xcall.cu -- the XCall dispatcher (replaces cgo/mo.c:54-68).
// Error convention of the reference (cgo/cuda/cuda.cpp:45-58, pkg/sql/plan/function/cxcall.go:76-89): non-zero return
// code + Pascal string in the caller's 256-byte errStr (errStr[0] = length, text from errStr[1]).
#include "common.cuh"
#include <cstring>
#include <cstdio>

namespace mob {
int xcall_rowdist(int64_t funcId, mo_xcall_args_t *args, uint64_t len);
int xcall_agg(int op, int T, mo_xcall_args_t *args, uint64_t len);
int xcall_q6(mo_xcall_args_t *args, uint64_t len);
int xcall_go_elementwise(int64_t funcId, mo_xcall_args_t *args, uint64_t len);
int xcall_q1(mo_xcall_args_t *args, uint64_t len);
int xcall_q6_merge(mo_xcall_args_t *args, uint64_t len);
int xcall_q1_merge(mo_xcall_args_t *args, uint64_t len);
int xcall_agg_merge(int op, int T, mo_xcall_args_t *args, uint64_t len);
int xcall_plan(mo_xcall_args_t *args, uint64_t len);
int xcall_dec_arith(int op, int width, mo_xcall_args_t *args, uint64_t len);
int xcall_dec_sum(int width, mo_xcall_args_t *args, uint64_t len);
int xcall_filter_sels(mo_xcall_args_t *args, uint64_t len);
int xcall_shuffle(int szof, mo_xcall_args_t *args, uint64_t len);
int xcall_pack_keys(mo_xcall_args_t *args, uint64_t len);
int xcall_group_ids(mo_xcall_args_t *args, uint64_t len);
int xcall_join_sels(mo_xcall_args_t *args, uint64_t len);
int xcall_kmeans(int64_t funcId, mo_xcall_args_t *args, uint64_t len);
int xcall_lz4_decode(mo_xcall_args_t *args, uint64_t len);
int xcall_vector_unmarshal(mo_xcall_args_t *args, uint64_t len);
int xcall_join_find(mo_xcall_args_t *args, uint64_t len);
int xcall_join_probe(mo_xcall_args_t *args, uint64_t len);
int xcall_group_agg(int op, int T, mo_xcall_args_t *args, uint64_t len);
int xcall_pack_str_keys(mo_xcall_args_t *args, uint64_t len);
int xcall_str_group_ids(mo_xcall_args_t *args, uint64_t len);
int xcall_str_join_find(mo_xcall_args_t *args, uint64_t len);
int xcall_str_join_probe(mo_xcall_args_t *args, uint64_t len);
int xcall_bruteforce(mo_xcall_args_t *args, uint64_t len);
int xcall_ivf(mo_xcall_args_t *args, uint64_t len);
int xcall_topk_merge(mo_xcall_args_t *args, uint64_t len);
int tuning_set(const char *name, int value);
unsigned long long *q1_debug_buffer();
}  // namespace mob

using namespace mob;

static void fill_err(uint8_t *errStr, int rc) {
    if (!errStr) return;
    ThreadCtx &t = tctx();
    char msg[256];
    int n = snprintf(msg, sizeof msg, "mo_b200 rc=%d: %s", rc, t.err[0] ? t.err : "error");
    if (n < 0) n = 0;
    if (n > 254) n = 254;
    errStr[0] = (uint8_t)n;
    memcpy(errStr + 1, msg, (size_t)n);
}

extern "C" int32_t XCall(int64_t runtimeId, int64_t funcId, uint8_t *errStr, uint64_t *args, uint64_t len) {
    (void)runtimeId;  // "C" and "CUDA" both run on the GPU here: this library has no CPU implementation
    ThreadCtx &t = tctx();
    if (!t.ready) { fill_err(errStr, MO_RC_INTERNAL_ERROR); return MO_RC_INTERNAL_ERROR; }
    t.err[0] = 0;
    mo_xcall_args_t *a = reinterpret_cast<mo_xcall_args_t *>(args);
    int rc;
    if ((funcId >= 0 && funcId <= 3) || (funcId >= 100 && funcId <= 113)) rc = xcall_rowdist(funcId, a, len);
    else if (funcId >= 0x1000 && funcId < 0x1000 + (5 << 8)) rc = xcall_agg((int)((funcId - 0x1000) >> 8), (int)((funcId - 0x1000) & 0xff), a, len);
    else if (funcId >= 0x1800 && funcId < 0x1800 + (5 << 8)) rc = xcall_agg_merge((int)((funcId - 0x1800) >> 8), (int)((funcId - 0x1800) & 0xff), a, len);
    else if (funcId == MO_XCALL_PLAN) rc = xcall_plan(a, len);
    else if (funcId >= 0x7000 && funcId < 0x7300) rc = xcall_dec_arith((int)((funcId - 0x7000) >> 8), (int)(funcId & 0xff), a, len);
    else if (funcId >= 0x7400 && funcId < 0x7500) rc = xcall_dec_sum((int)(funcId & 0xff), a, len);
    else if (funcId == MO_XCALL_FILTER_SELS) rc = xcall_filter_sels(a, len);
    else if (funcId == MO_XCALL_PACK_KEYS) rc = xcall_pack_keys(a, len);
    else if (funcId == MO_XCALL_GROUP_IDS) rc = xcall_group_ids(a, len);
    else if (funcId == MO_XCALL_JOIN_SELS) rc = xcall_join_sels(a, len);
    else if (funcId == MO_XCALL_LZ4_DECODE) rc = xcall_lz4_decode(a, len);
    else if (funcId == MO_XCALL_VECTOR_UNMARSHAL) rc = xcall_vector_unmarshal(a, len);
    else if (funcId == MO_XCALL_KMEANS_ELKAN_F32 || funcId == MO_XCALL_KMEANS_ELKAN_F64) rc = xcall_kmeans(funcId, a, len);
    else if (funcId == MO_XCALL_JOIN_FIND) rc = xcall_join_find(a, len);
    else if (funcId == MO_XCALL_JOIN_PROBE) rc = xcall_join_probe(a, len);
    else if (funcId == MO_XCALL_PACK_STR_KEYS) rc = xcall_pack_str_keys(a, len);
    else if (funcId == MO_XCALL_STR_GROUP_IDS) rc = xcall_str_group_ids(a, len);
    else if (funcId == MO_XCALL_STR_JOIN_FIND) rc = xcall_str_join_find(a, len);
    else if (funcId == MO_XCALL_STR_JOIN_PROBE) rc = xcall_str_join_probe(a, len);
    else if (funcId > 0x6100 && funcId <= 0x6100 + 24) rc = xcall_shuffle((int)(funcId - 0x6100), a, len);
    else if (funcId >= 0x6400 && funcId < 0x6400 + (5 << 8)) rc = xcall_group_agg((int)((funcId - 0x6400) >> 8), (int)((funcId - 0x6400) & 0xff), a, len);
    else if (funcId == MO_XCALL_Q6_MERGE) rc = xcall_q6_merge(a, len);
    else if (funcId == MO_XCALL_Q1_MERGE) rc = xcall_q1_merge(a, len);
    else if (funcId >= 0x4000 && funcId < 0x5800) rc = xcall_go_elementwise(funcId, a, len);
    else if (funcId == MO_XCALL_Q6_FILTER_SUM) rc = xcall_q6(a, len);
    else if (funcId == MO_XCALL_Q1_GROUP_AGG) rc = xcall_q1(a, len);
    else if (funcId == MO_XCALL_BRUTEFORCE_TOPK_F32) rc = xcall_bruteforce(a, len);
    else if (funcId == MO_XCALL_IVF_TOPK_F32) rc = xcall_ivf(a, len);
    else if (funcId == MO_XCALL_TOPK_MERGE) rc = xcall_topk_merge(a, len);
    else return -1;  // unknown funcId, cgo/mo.c:64-67
    if (rc != 0) fill_err(errStr, rc);
    return rc;
}

extern "C" int32_t MoB200_SetTuning(const char *name, int32_t value) { return tuning_set(name, value); }

// debug aid for tools/q1_phases.py: device address of the per-CTA phase timestamps (8 x uint64 per CTA), or NULL
extern "C" void *MoB200_DebugBuffer(void) { return q1_debug_buffer(); }
