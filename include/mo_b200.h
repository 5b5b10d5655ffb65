/*
 * mo_b200.h -- C-ABI of libmo_b200.so, the B200 (sm_100a) implementation of MatrixOne's per-block batch
 * operators and vector-distance kernels.
 *
 * PART 1 is the reference's cgo surface, byte for byte the same prototypes as /root/reference/cgo/mo.h:24-73
 * (Bitmap_*, {SignedInt,UnsignedInt,Float}_Vec*, Numeric_Vec*, Logic_Vec*, XCall), so the Go side
 * (pkg/common/bitmap/cbitmap.go:33-50, pkg/sql/plan/function/cxcall.go:78-83) binds to it unchanged.
 * Rules kept from cgo/README.md:12-16: only fixed-width ints, float/double and pointers cross the boundary.
 *
 * Every pointer argument may be either a HOST pointer (pageable or pinned; the library stages it through the
 * calling thread's stream) or a DEVICE pointer obtained from MoB200_DeviceAlloc (zero-copy, the resident path).
 * The library classifies each pointer with cudaPointerGetAttributes.  All pointers of one call must live on the
 * same side unless stated otherwise.  Buffers stay owned by the caller (cgo/README.md:21-23).
 *
 * PART 2 declares the XCall argument block (reference cgo/xcall.h:24-31) and the funcIds this library adds
 * (>= 100; ids 0..3 keep the reference meaning, cgo/mo.c:49-52).
 *
 * PART 3 is the residency/runtime extension (device + pinned allocation, copies, stream adoption, timers).
 */
#ifndef _MO_B200_H_
#define _MO_B200_H_

#include <stdint.h>
#include <stdbool.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ======================================================================================================
 * PART 1 -- reference ABI (cgo/mo.h)
 * ==================================================================================================== */

/* Bitmap ops -- replaces cgo/mo.c:19-47 (bodies in cgo/bitmap.h:47-149).  LSB-first uint64 words, set = NULL. */
void Bitmap_Add(uint64_t *p, uint64_t pos);
void Bitmap_Remove(uint64_t *p, uint64_t pos);
bool Bitmap_Contains(uint64_t *p, uint64_t pos);
bool Bitmap_IsEmpty(uint64_t *p, uint64_t nbits);
uint64_t Bitmap_Count(uint64_t *p, uint64_t nbits);
void Bitmap_And(uint64_t *dst, uint64_t *a, uint64_t *b, uint64_t nbits);
void Bitmap_Or(uint64_t *dst, uint64_t *a, uint64_t *b, uint64_t nbits);
void Bitmap_Not(uint64_t *dst, uint64_t *a, uint64_t nbits);

/* Vector arithmetic -- replaces cgo/arith.c:316-580.  flag&1: a is scalar, flag&2: b is scalar
 * (cgo/mo_impl.h:37-38).  Rows whose bit is set in `nulls` are skipped (r[i] untouched).
 * Return codes as cgo/mo_impl.h:26-35 (see MO_RC_* below); overflow-flag quirks of arith.c are reproduced. */
int32_t SignedInt_VecAdd(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t UnsignedInt_VecAdd(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t Float_VecAdd(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);

int32_t SignedInt_VecSub(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t UnsignedInt_VecSub(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t Float_VecSub(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);

int32_t SignedInt_VecMul(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t UnsignedInt_VecMul(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t Float_VecMul(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);

int32_t Float_VecDiv(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t Float_VecIntegerDiv(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);

int32_t SignedInt_VecMod(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t UnsignedInt_VecMod(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);
int32_t Float_VecMod(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t szof);

/* Compare -- replaces cgo/compare.c:153-383.  r is bool[n] (1 byte each); `type` is a types.T id (MO_T_*). */
int32_t Numeric_VecEq(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t type);
int32_t Numeric_VecNe(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t type);
int32_t Numeric_VecGt(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t type);
int32_t Numeric_VecGe(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t type);
int32_t Numeric_VecLt(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t type);
int32_t Numeric_VecLe(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag, int32_t type);

/* Three-valued logic -- replaces cgo/logic.c:33-221.  The caller pre-fills rnulls = anulls | bnulls;
 * And/Or clear the bits where the other operand dominates. */
int32_t Logic_VecAnd(void *r, void *a, void *b, uint64_t n, uint64_t *anulls, uint64_t *bnulls, uint64_t *rnulls, int32_t flag);
int32_t Logic_VecOr(void *r, void *a, void *b, uint64_t n, uint64_t *anulls, uint64_t *bnulls, uint64_t *rnulls, int32_t flag);
int32_t Logic_VecXor(void *r, void *a, void *b, uint64_t n, uint64_t *nulls, int32_t flag);
int32_t Logic_VecNot(void *r, void *a, uint64_t n, uint64_t *nulls, int32_t flag);

/* XCall -- replaces cgo/mo.c:54-68.  runtimeId: 0 = "C", 1 = "CUDA" (cgo/xcall.h:44-45); this library runs every
 * funcId on the GPU for BOTH runtime ids (there is no CPU implementation inside it).  errStr is the reference's
 * 256-byte Pascal string: errStr[0] = length, text from errStr[1] (cgo/cuda/cuda.cpp:45-58, cxcall.go:76-89).
 * args -> xcall_args_t[]: index 0 = result vector, 1..k = inputs.  Unknown funcId returns -1. */
int32_t XCall(int64_t runtimeId, int64_t funcId, uint8_t *errStr, uint64_t *args, uint64_t len);

/* ======================================================================================================
 * PART 2 -- XCall argument block, type ids, return codes, funcIds
 * ==================================================================================================== */

/* cgo/xcall.h:24-31; filled by Vector.FillRawPtrLen, pkg/container/vector/vector.go:5161-5172 */
typedef struct mo_xcall_args_t {
    uint64_t *pnulls;  /* nulls bitmap words or NULL */
    uint64_t nullCnt;  /* bitmap length IN BITS (field misnamed in the reference) */
    uint8_t *pdata;    /* fixed-width values, or 24-byte varlena cells */
    uint64_t dataSz;   /* bytes; typeSize*1 for a const vector */
    uint8_t *parea;    /* varlena payload area or NULL */
    uint64_t areaSz;
} mo_xcall_args_t;

#define MO_VARLENA_SZ 24         /* cgo/xcall.h:33 */
#define MO_VARLENA_INLINE_SZ 23

#define MO_RUNTIME_C 0
#define MO_RUNTIME_CUDA 1

/* return codes, cgo/mo_impl.h:26-35 */
#define MO_RC_SUCCESS 0
#define MO_RC_INTERNAL_ERROR 20101
#define MO_RC_DIVISION_BY_ZERO 20200
#define MO_RC_OUT_OF_RANGE 20201
#define MO_RC_DATA_TRUNCATED 20202
#define MO_RC_INVALID_ARGUMENT 20203

/* types.T ids, pkg/container/types/types.go:35-67 == cgo/compare.c:20-38 */
#define MO_T_BOOL 10
#define MO_T_INT8 20
#define MO_T_INT16 21
#define MO_T_INT32 22
#define MO_T_INT64 23
#define MO_T_UINT8 25
#define MO_T_UINT16 26
#define MO_T_UINT32 27
#define MO_T_UINT64 28
#define MO_T_FLOAT32 30
#define MO_T_FLOAT64 31
#define MO_T_DATE 50
#define MO_T_TIME 51
#define MO_T_DATETIME 52
#define MO_T_TIMESTAMP 53

/* reference funcIds, cgo/mo.c:49-52 == cxcall.go:33-38.  args: [0] f64 result, [1] vec col, [2] vec col
 * (varlena cells; either side may be const: dataSz == 24).  Semantics of cgo/xcall.c:23-134:
 * float diff, squares accumulated in double, optional sqrt. */
#define MO_XCALL_L2DISTANCE_F32 0
#define MO_XCALL_L2DISTANCE_F64 1
#define MO_XCALL_L2DISTANCE_SQ_F32 2
#define MO_XCALL_L2DISTANCE_SQ_F64 3

/* --- new: row-wise distances with the Go semantics of pkg/vectorindex/metric/distance_func.go (accumulator type =
 * element type, 8-way unrolled association), i.e. what the SQL builtins l2_distance / l2_distance_sq / inner_product /
 * cosine_distance / cosine_similarity compute (pkg/vectorize/moarray/external.go:171-260).  Same 3-arg layout as
 * ids 0..3, result float64[len].  Bit-exact with the Go loops.  dim mismatch -> MO_RC_INVALID_ARGUMENT. */
#define MO_XCALL_GO_L2_F32 100
#define MO_XCALL_GO_L2_F64 101
#define MO_XCALL_GO_L2SQ_F32 102
#define MO_XCALL_GO_L2SQ_F64 103
#define MO_XCALL_GO_IP_F32 104
#define MO_XCALL_GO_IP_F64 105
#define MO_XCALL_GO_COSDIST_F32 106
#define MO_XCALL_GO_COSDIST_F64 107
#define MO_XCALL_GO_COSSIM_F32 108
#define MO_XCALL_GO_COSSIM_F64 109
#define MO_XCALL_GO_L1_F32 110   /* metric.L1Distance, distance_func.go:112-154 (l1_norm of the difference) */
#define MO_XCALL_GO_L1_F64 111
/* normalize_l2(v): moarray.NormalizeL2 (pkg/vectorize/moarray/external.go:262-285): a VECTOR-valued result.
 * args: [0] the result varlena vector (pdata -> 24 * len cells, parea / areaSz -> its area, at least as large as the
 * argument's: the result area MIRRORS the argument's layout -- cell i gets the same (offset, length), inline cells
 * stay inline; pnulls = the result nulls, rows set there are skipped and get an empty cell) ; [1] the argument vector
 * (dataSz == 24: const).  sumSquares in float64 in index order, normalized[i] = T(float64(v[i]) / norm), norm == 0
 * copies the row; an empty non-null vector -> MO_RC_INTERNAL_ERROR "cannot normalize empty vector". */
#define MO_XCALL_GO_NORMALIZE_L2_F32 112
#define MO_XCALL_GO_NORMALIZE_L2_F64 113

/* --- new: single-column aggregates (aggexec sumavg2.go / count2.go / minmax2.go semantics, no group-by = H0).
 * funcId = MO_XCALL_AGG(op, T).  args: [0] result: pdata -> one 8-byte value (int64 / uint64 / float64, or the
 * column type for MIN/MAX, zero-extended), pnulls -> 1-word bitmap, bit 0 set when the result is NULL
 * (all-null input); [1] the column (fixed width, pnulls optional).  len = rows.
 * SUM over signed ints returns MO_RC_OUT_OF_RANGE exactly when the serial Go loop would (int64OfCheck). */
#define MO_AGG_SUM 0
#define MO_AGG_COUNT 1   /* COUNT(col): non-null rows; result int64 */
#define MO_AGG_MIN 2
#define MO_AGG_MAX 3
#define MO_AGG_AVG 4     /* result float64 = sum/cnt, NULL when cnt == 0 */
#define MO_XCALL_AGG(op, T) (0x1000 + ((op) << 8) + (T))
/* Wider results: dataSz >= 16 adds the non-null row count at pdata+8; dataSz >= 24 makes the result a PARTIAL STATE
 * mo_agg_state_t {value bits (SUM/AVG: the sum in the SUM return type; AVG is NOT divided yet), non-null rows, rc} -- what a partial
 * Group hands to MergeGroup (pkg/sql/colexec/group/mergeGroup.go:132-247).
 * Asynchronous form: when the column AND the result (pdata, pnulls) are DEVICE pointers the call only enqueues work on the calling
 * thread's stream and returns MO_RC_SUCCESS at once; errors detected on the device (SUM overflow) are reported in state.rc. */
typedef struct mo_agg_state_t { uint64_t bits; int64_t count; int64_t rc; } mo_agg_state_t;
/* MergeGroup for these aggregates: args [0] result (8 / 16 / 24 bytes as above, + nulls word) ; [1] len partial states (24 bytes each),
 * folded in order with the reference's BatchMerge rules (sumavg2.go:205-248 incl. int64OfCheck / uint64OfCheck, minmax2.go:90-110).
 * Device pointers on both sides: asynchronous as above. */
#define MO_XCALL_AGG_MERGE(op, T) (0x1800 + ((op) << 8) + (T))

/* --- new: fused TPC-H Q6 shape  SUM(a*b) WHERE d in [d_lo,d_hi) AND b BETWEEN b_lo AND b_hi AND c < c_hi
 * args: [0] result f64 (+ 1-word nulls bitmap, bit0 = no row qualified) ; [1] d int32/DATE col ; [2] b f64 col
 * (discount) ; [3] c f64 col (quantity) ; [4] a f64 col (extendedprice) ; [5] params: pdata -> mo_q6_params_t.
 * Optional second result word: if args[0].dataSz >= 16 the qualifying row count (int64) is written at pdata+8. */
/* ---- The Go elementwise engine's conventions (pkg/sql/plan/function/baseTemplate.go:457-728, arithmetic.go:222-762,
 * func_compare.go:285-1185, operator_between.go:138-199, logicalOperator.go:36-168) -- the LIVE per-batch path of the reference;
 * the mo.h symbols above keep the C kernels' conventions.  Differences: rows whose RESULT null bit is set on entry are skipped
 * (the caller pre-fills args[0].pnulls with NOT selectList, baseTemplate.go:473-486); on return it holds rnulls | n1 | n2 (plus
 * the rows a zero divisor nulled); a const operand is a 1-element vector (dataSz == sizeof(T)), a const NULL operand nulls every
 * row; the FIRST offending row in row order fails the call (MO_RC_OUT_OF_RANGE with "data out of range: data type int64, value
 * '(a + b)'" / MO_RC_DIVISION_BY_ZERO) and its index is stored in the parameter block; rows before it hold their results.
 *   ARITH(op, T)   op: 0 + 1 - 2 * 3 / (floats) 4 %     args: [0] result T[len] + pnulls (in/out)  [1] a  [2] b  [3] mo_go_params_t
 *   COMPARE(op, T) op: 0 == 1 != 2 > 3 >= 4 < 5 <=      args: [0] result bool[len] + pnulls (in/out)  [1] a  [2] b
 *   BETWEEN(T)                                           args: [0] result bool[len] + pnulls (in/out)  [1] column (+ pnulls)  [2] lo  [3] hi
 *                                                        null input -> result false AND null bit set
 *   MULTI_AND / MULTI_OR                                 args: [0] result bool[len] + pnulls (out)  [1] int32 operand count n (<= 16)
 *                                                              [2 .. 2 + n) bool operands (+ pnulls); const = 1 byte
 * T = types.T id (MO_T_*); DATE compares as int32, TIME / DATETIME / TIMESTAMP as int64. */
typedef struct { int32_t div0_null; int32_t reserved; int64_t err_row; } mo_go_params_t;   /* err_row: out, -1 = no error */
#define MO_XCALL_GO_ARITH(op, T) (0x4000 + ((op) << 8) + (T))
#define MO_XCALL_GO_COMPARE(op, T) (0x4800 + ((op) << 8) + (T))
/* float32 columns declared with scale > 0 compare after rounding both sides to `scale` decimals (func_compare.go:207-216,725-734,
 * 852-861,979-988,1106-1115,1233-1242): same args as COMPARE(op, MO_T_FLOAT32), scale 1..22 */
#define MO_XCALL_GO_COMPARE_F32_SCALE(op, scale) (0x5200 + ((op) << 8) + (scale))
#define MO_XCALL_GO_BETWEEN(T) (0x5000 + (T))
#define MO_XCALL_GO_MULTI_AND 0x5100
#define MO_XCALL_GO_MULTI_OR 0x5101

/* ---- the standalone column operators of the colexec pipeline (csrc/colops.cu).  Host or device pointers; with device pointers on
 * every vector FILTER_SELS and SHUFFLE only enqueue work (asynchronous form, as MO_XCALL_AGG).
 *
 * FILTER_SELS  Filter.Call inner loop (filter.go:116-152): rows with (!null && true), ascending.
 *              args: [0] sels int64[] (a host buffer only has to hold the selected rows) ; [1] count int64[1] ; [2] bool vector (+pnulls).  len = rows
 * SHUFFLE(sz)  Vector.Shrink / Union / shuffle.FixedLengthShuffle (vector.go:1014,2583 ; shuffle.go:21-26) with nulls.Filter
 *              (nulls.go:237-281) fused: dst[i] = src[sels[i]], dst null bit i = src null bit sels[i].  sz = element bytes: 1, 2, 4, 8, 16, 24 (varlena cell).
 *              args: [0] dst (+pnulls out) ; [1] src (+pnulls, nullCnt = its length in bits) ; [2] sels int64[len].  len = selected rows
 * PACK_KEYS    intHashMapIterator.encodeHashKeys / fillKeys (inthashmap.go:92-183): up to 8 key bytes per row from fixed-width columns, in
 *              has_null mode a marker byte (0 / 1) precedes every column's value bytes and a NULL contributes the marker only.
 *              args: [0] keys uint64[len] (+pnulls out, has_null = 0: rows with a NULL key join no group) ; [1] host params {int32 ncols, int32 has_null}
 *              ; [2 .. 2+ncols) key columns (+pnulls; a const vector holds one element)
 * GROUP_IDS    IntHashMap insert as driven by Group.buildOneBatch (exec2.go:325-362): 1-based group ids in FIRST-SEEN order; the table persists across
 *              calls through (ngroups, table_keys).  The hash function is not observable (random seeds, hashtable/hash.go:41-47), the ids are.
 *              args: [0] groups uint64[len] ; [1] int64 ngroups (in/out) ; [2] table_keys uint64[capacity] (in: keys of groups 1..ngroups ; out: + new groups)
 *              ; [3] keys uint64[len] (+pnulls: such rows get id 0 = GroupNotMatched)
 * GROUP_AGG(op, T)  sumAvgExec / countColumnExec / minMaxExecFixed .BatchFill (sumavg2.go:133-199, count2.go:120-146, minmax2.go:49-80) into a
 *              caller-owned state that persists across batches: SUM into int64 / uint64 / float64 (overflow -> MO_RC_OUT_OF_RANGE exactly when
 *              the serial loop would fail), AVG = SUM + counts, COUNT into int64, MIN / MAX in 8-byte slots (value in the low bytes) with the
 *              first-value-initialises / strict-compare rule incl. NaN.  A group is NULL until its first value (state pnulls, in/out).
 *              args: [0] state 8 bytes per group (+pnulls) ; [1] counts int64 per group (AVG: required) ; [2] groups uint64[len] ; [3] column (+pnulls)
 * float64 group sums are accumulated with atomics: the association order is not fixed, results agree with the serial loop to ~1e-13 relative. */
#define MO_XCALL_FILTER_SELS 0x6000
#define MO_XCALL_PACK_KEYS 0x6001
#define MO_XCALL_GROUP_IDS 0x6002
#define MO_XCALL_SHUFFLE(szof) (0x6100 + (szof))
/* ---- Elkan k-means, dense variant (csrc/kmeans.cu): ElkanClusterer.Cluster from given initial centroids
 * (pkg/vectorindex/ivfflat/kmeans/elkans/clusterer.go:330-392; distance = metric.L2Distance for every metric, distance_func.go:452-476).
 * Centroids bit for bit, assignments and iteration count as the reference computes them (serial row-order sums, Go-order distances).
 * InitCentroids (initializer.go: draws from Go's PCG) stays with the caller.  args: [0] centroids T[k * dim] (in: initial, out: final) ;
 * [1] assignments int64[n] (out) ; [2] int64 iterations (out) ; [3] host mo_kmeans_params_t ; [4] vectors T[n * dim] ;
 * [5] rnd float32[] (optional): the rnd.Float32() stream an EMPTY cluster re-seeds its centroid from (clusterer.go:700-707), consumed in
 * cluster order, dim values per empty cluster; running out of it fails the call with MO_RC_INVALID_ARGUMENT. */
/* ---- LZ4 block decompression of column blocks (csrc/lz4.cu): compress.Decompress = lz4.UncompressBlock (pkg/compress/compress.go:37-47), one
 * warp per block.  args: [0] dst bytes ; [1] src bytes ; [2] int64[4 * len] descriptors {src_off, src_len, dst_off, dst_len} per block (dst_len = the
 * decoded size the object metadata records; a block that decodes to anything else, or is malformed, fails the call with MO_RC_INVALID_ARGUMENT and
 * the block number in the error text).  len = number of blocks. */
#define MO_XCALL_LZ4_DECODE 0x6030
/* ---- a decompressed column block -> a resident vector (csrc/vecdecode.cu): Vector.UnmarshalBinary (pkg/container/vector/vector.go:766-819) on the device.
 * args: [0] mo_vector_view_t (out) ; [1] data bytes (out: capacity >= dataLen, aligned) ; [2] area bytes (out) ; [3] nulls uint64 words (out:
 * (length + 63) / 64 words; pdata NULL when not wanted) ; [4] the marshalled bytes (dataSz = their length; when they are device memory the buffer
 * must be readable 8 bytes past that length).  Malformed bytes or too small output buffers -> MO_RC_INVALID_ARGUMENT. */
typedef struct mo_vector_view_t {
    int32_t vclass;        /* 0 FLAT, 1 CONSTANT */
    int32_t oid;           /* types.T */
    int32_t size, width, scale;
    uint32_t length;       /* rows */
    uint64_t data_len, area_len;
    int64_t null_count;    /* bitmap.count as marshalled */
    uint64_t nulls_words;
    int32_t sorted, bad;
} mo_vector_view_t;
#define MO_XCALL_VECTOR_UNMARSHAL 0x6031
typedef struct mo_kmeans_params_t { int64_t n, dim, k, max_iter; } mo_kmeans_params_t;
#define MO_XCALL_KMEANS_ELKAN_F32 0x6020
#define MO_XCALL_KMEANS_ELKAN_F64 0x6021
/* ---- hash join, equality conditions over <= 8-byte packed keys (csrc/join.cu).  The build side inserts its keys with GROUP_IDS (IntHashMap insert):
 *   JOIN_SELS   GroupSels.Insert + Finalize (pkg/vm/message/joinMapMsg.go:72-125) as driven by HashmapBuilder.BuildHashmap (hashbuild/hashmap.go:395-412):
 *               the build rows of every group, ascending.  args: [0] offsets int32[ngroups + 2] (out: [k] = start of 0-based group k, [ngroups] =
 *               [ngroups + 1] = count) ; [1] vals int32[len] (out) ; [2] int64 count (out: rows that have a group) ; [3] groups uint64[len] (the ids
 *               GROUP_IDS returned for the build rows; 0 = the row has a NULL key and joins nothing).  len = build rows (< 2^31).
 *               (The reference keeps no sels when every row got its own group -- HashOnUnique, joinMapMsg.go:83-89,203-205: pass pdata NULL below.)
 *   JOIN_FIND   intHashMapIterator.Find (pkg/common/hashmap/inthashmap.go): vals[i] = 1-based group id of probe key i, 0 = absent or NULL key.
 *               args: [0] vals uint64[len] ; [1] table_keys uint64[ngroups] (GROUP_IDS's key table: key of group g at [g - 1]) ; [2] keys uint64[len] (+pnulls)
 *   JOIN_PROBE  the emission loop of hashjoin container.probe (pkg/sql/colexec/hashjoin/join.go:383-628) without a non-equality condition: result rows
 *               as (probe row, build row) pairs in the reference's order -- probe rows ascending, per probe row its group's sels ascending.
 *               join_type INNER: matches only; LEFT: + (row, -1) for a probe row without a match; SEMI: (row, -1) once per matching probe row;
 *               ANTI: (row, -1) per probe row WITHOUT a match.  args: [0] probe_rows int64[cap] ; [1] build_rows int64[cap] ; [2] int64 count (out; when
 *               it exceeds cap the call fails with MO_RC_OUT_OF_RANGE and the count is still written) ; [3] host mo_join_params_t ; [4] table_keys ;
 *               [5] sels offsets int32[ngroups + 2] (pdata NULL: unique map, build row = id - 1) ; [6] sels vals int32[] ; [7] probe keys uint64[len] (+pnulls)
 * The device hash table is rebuilt from table_keys per call unless MoB200_JoinMapPrepare(table_keys, ngroups) cached it (keyed by that pointer). */
#define MO_JOIN_INNER 0
#define MO_JOIN_LEFT 1
#define MO_JOIN_SEMI 2
#define MO_JOIN_ANTI 3
typedef struct mo_join_params_t { int32_t join_type; int32_t reserved; } mo_join_params_t;
#define MO_XCALL_JOIN_SELS 0x6010
#define MO_XCALL_JOIN_FIND 0x6011
#define MO_XCALL_JOIN_PROBE 0x6012
#define MO_XCALL_GROUP_AGG(op, T) (0x6400 + ((op) << 8) + (T))

/* ---- group-by and hash join on keys wider than 8 bytes: the StrHashMap path (csrc/strhash.cu).  The reference takes it for any varchar / char
 * key, any composite key wider than 8 bytes (a nullable column costs one byte more, group/exec2.go:73-94,167-188) and any join whose equality
 * columns are wider than 8 bytes (hashbuild/hashmap.go:258-277).  A packed key table is "offsets int64[ngroups + 1] + bytes": the key of 1-based
 * group g is bytes[offsets[g - 1] .. offsets[g]).  Everything behind the ids is shared with the 8-byte path: GROUP_AGG, DEC_SUM, JOIN_SELS.
 * All four calls are synchronous; pointers as everywhere (host or device).
 *   PACK_STR_KEYS   strHashmapIterator.encodeHashKeys (pkg/common/hashmap/strhashmap.go:92-385), the exact bytes.  Per column, in column order:
 *                   fixed width w, has_null: marker 0 + the w value bytes, a NULL appends marker 1 only ; fixed, no has_null: the w value bytes,
 *                   a NULL makes the row skip (zValues = 0) and the column appends nothing ; varlena, has_null: marker 0 + length as little-endian
 *                   uint16 + the bytes, a NULL appends marker 1 ; varlena, no has_null: uint16 length + bytes, a NULL skips the row.  The length
 *                   field is truncated to 16 bits, the bytes are not.  A const vector repeats element 0, a const NULL appends marker 1 (has_null)
 *                   or skips every row.  Keys shorter than 16 bytes are zero-padded to 16 (hashtable.StrKeyPadding).
 *                   args: [0] offsets int64[len + 1] (out; + pnulls out, no has_null mode: the rows that join no group) ; [1] key bytes (out;
 *                   capacity = dataSz) ; [2] host mo_str_key_params_t ; [3 .. 3 + ncols) the key columns (+pnulls): fixed width = width[k] bytes
 *                   per row (any width >= 1: Decimal128, uuid, Rowid), varlena (width 0) = 24-byte cells with parea.  A const vector holds one
 *                   element.  When the bytes do not fit, the call fails with MO_RC_OUT_OF_RANGE and offsets[len] holds the bytes needed.
 *   STR_GROUP_IDS   strHashmapIterator.Insert as driven by Group.buildOneBatch (exec2.go:325-362, string_hash_map.go:97-158): 1-based group ids
 *                   in FIRST-SEEN order, 0 for a skipped row.  Two keys are one group when their bytes are equal (the reference compares 192-bit
 *                   hash states; the ids are the same).  The table persists across calls in caller-owned buffers.
 *                   args: [0] groups uint64[len] ; [1] state int64[4] = {ngroups (in/out), key bytes used (in/out), groups needed (out), bytes
 *                   needed (out)} ; [2] table offsets int64[capacity + 1] ; [3] table bytes (capacity = dataSz) ; [4] packed key offsets
 *                   int64[len + 1] (+pnulls: rows that get id 0) ; [5] packed key bytes.  More groups than the capacity or more key bytes than the
 *                   table holds: MO_RC_OUT_OF_RANGE with state[2], state[3] set, and ngroups, bytes used and the table left unchanged; the caller
 *                   grows its buffers and repeats the call.
 *   STR_JOIN_FIND   strHashmapIterator.Find: vals[i] = 1-based group id of probe key i, 0 = absent, NULL or skipped.
 *                   args: [0] vals uint64[len] ; [1] table offsets int64[ngroups + 1] ; [2] table bytes ; [3] probe key offsets (+pnulls) ; [4] probe key bytes
 *   STR_JOIN_PROBE  JOIN_PROBE over string keys: same join types, emission order, capacity protocol and sels.  args: [0 .. 3] as JOIN_PROBE ;
 *                   [4] table offsets ; [5] table bytes ; [6] sels offsets ; [7] sels vals ; [8] probe key offsets (+pnulls) ; [9] probe key bytes
 * The device hash table is rebuilt from the key table per call (like GROUP_IDS) unless MoB200_StrJoinMapPrepare cached it for FIND / PROBE.
 * Not provided here: string keys inside MO_XCALL_PLAN, the grouping-set marker 2 (ROLLUP / CUBE), non-equality join conditions, right joins. */
#define MO_STR_KEY_MAX_COLS 16
typedef struct mo_str_key_params_t { int32_t ncols; int32_t has_null; int32_t width[MO_STR_KEY_MAX_COLS]; /* 0 = varlena */ } mo_str_key_params_t;
#define MO_XCALL_PACK_STR_KEYS 0x6003
#define MO_XCALL_STR_GROUP_IDS 0x6004
#define MO_XCALL_STR_JOIN_FIND 0x6013
#define MO_XCALL_STR_JOIN_PROBE 0x6014

/* ---- Decimal64 / Decimal128 (csrc/decimal.cu): the reference's native TPC-H column type is DECIMAL(15,2).  Decimal64 = int64 unscaled value,
 * Decimal128 = 16 bytes two's complement {B0_63, B64_127}; scales travel in the parameter block.  Conventions of the Go engine (as GO_ARITH).
 *   DEC_ARITH(op, width)  op 0 + 1 - 2 * ; width 64 / 128 = operand type.  d64Add/d64Sub/d64Mul/d128Add/d128Sub/d128Mul,
 *                         pkg/sql/plan/function/arith_decimal_fast.go:111-733,3618-4095.  + - : the lower-scale operand is scaled up, result
 *                         scale = max(scale1, scale2), result type = operand type; * : result Decimal128 with scale
 *                         min(scale1 + scale2, max(12, scale1, scale2)), scaled down with round-half-up when that is smaller than scale1 + scale2.
 *                         The first row that overflows fails the call with MO_RC_INVALID_ARGUMENT (moerr ErrInvalidInput) and err_row is set.
 *                         args: [0] result (+pnulls in/out) ; [1] a ; [2] b (const = one element) ; [3] host mo_dec_params_t
 *   DEC_SUM(width)        SUM / AVG accumulation of a decimal column into Decimal128 sums + int64 counts per group (count 0 = NULL; AVG divides at
 *                         Flush), sumDecimal64FastExec / sumDecimal128FastExec.batchFill, pkg/sql/colexec/aggexec/sum_decimal_fast.go -- exact and
 *                         order independent.  args: [0] sums Decimal128 per group (in/out) ; [1] counts int64 per group (in/out) ;
 *                         [2] groups uint64[len] (1-based, 0 = skip) or pdata NULL for one group ; [3] the column (+pnulls) */
typedef struct mo_dec_params_t { int32_t scale1, scale2; int64_t err_row; } mo_dec_params_t;
#define MO_XCALL_DEC_ARITH(op, width) (0x7000 + ((op) << 8) + (width))
#define MO_XCALL_DEC_SUM(width) (0x7400 + (width))

/* ---- the generic fused operator: scan -> filter -> project -> (hash) group -> aggregate in ONE pass over the columns (csrc/plan.cu).
 * What the colexec pipeline runs per block as table_scan -> filter -> projection -> group (filter.go:87-153, evalExpression.go:575-640,
 * group/exec2.go:296-367, aggexec/*), described by a host-side mo_plan_t:
 *   columns      args[2 .. 2+ncols): fixed-width columns of col_type[c] (MO_T_*), each with an optional nulls bitmap
 *   predicates   conjunction of  col OP lo  (OP: 0 == 1 != 2 > 3 >= 4 < 5 <=)  or  col BETWEEN lo AND hi (op 6); a NULL operand rejects the row
 *   instructions SSA program: value slot ncols + i = COL(a) | CONST(imm) | slot a (+ - * /) slot b; slots 0..ncols-1 are the columns.  float64
 *                arithmetic, one rounding per instruction (the reference evaluates one node at a time); integer columns are converted (exact
 *                below 2^53); NULL in -> NULL out; x / 0 -> NULL
 *   keys         nkeys columns packed into <= 8 bytes exactly like fillKeys (inthashmap.go:92-183; has_null_keys: marker byte per column)
 *   aggregates   kind MO_AGG_SUM / COUNT / MIN / MAX / AVG over value slot `value`; value = -1 with MO_AGG_COUNT is COUNT(*)
 * Result: mo_plan_result_header_t followed by ngroups records {mo_plan_group_t, naggs x mo_plan_agg_value_t}, groups in first-seen row order
 * (the reference's group-id order) when header.sorted (up to 8192 groups; beyond that in table order, first_row is there to sort by).  An
 * aggregate with count 0 is NULL.  No group-by (nkeys = 0): one group, present only if a row qualified.  header.overflow = more groups than the
 * result buffer holds (synchronous form: MO_RC_INVALID_ARGUMENT).  Device columns AND a device result: asynchronous form (as MO_XCALL_AGG).
 * float64 sums are accumulated with atomics: the association order is not fixed (agreement with the serial loop ~1e-13 relative); MIN / MAX
 * ignore NaN.  The TPC-H Q6 / Q1 shapes below are hand-specialised instances of this operator that reach the HBM roofline. */
#define MO_XCALL_PLAN 0x2100
#define MO_PLAN_MAX_COLS 12
#define MO_PLAN_MAX_PREDS 8
#define MO_PLAN_MAX_INSTR 16
#define MO_PLAN_MAX_KEYS 4
#define MO_PLAN_MAX_AGGS 12
#define MO_PLAN_OP_COL 0
#define MO_PLAN_OP_CONST 1
#define MO_PLAN_OP_ADD 2
#define MO_PLAN_OP_SUB 3
#define MO_PLAN_OP_MUL 4
#define MO_PLAN_OP_DIV 5
typedef struct mo_plan_pred_t { int32_t col; int32_t op; double lo; double hi; } mo_plan_pred_t;
typedef struct mo_plan_instr_t { int32_t op; int32_t a; int32_t b; int32_t reserved; double imm; } mo_plan_instr_t;
typedef struct mo_plan_agg_t { int32_t kind; int32_t value; } mo_plan_agg_t;
typedef struct mo_plan_t {
    int32_t ncols, npreds, ninstr, nkeys, naggs, has_null_keys;
    int64_t row_base;                       /* added to first_row (block-range offset of a shard) */
    int32_t col_type[MO_PLAN_MAX_COLS];
    mo_plan_pred_t pred[MO_PLAN_MAX_PREDS];
    mo_plan_instr_t instr[MO_PLAN_MAX_INSTR];
    int32_t key_col[MO_PLAN_MAX_KEYS];
    mo_plan_agg_t agg[MO_PLAN_MAX_AGGS];
} mo_plan_t;
typedef struct mo_plan_result_header_t { int64_t ngroups; int32_t sorted; int32_t overflow; int64_t reserved; } mo_plan_result_header_t;
typedef struct mo_plan_group_t { uint64_t key; int64_t first_row; int64_t rows; } mo_plan_group_t;
typedef struct mo_plan_agg_value_t { double value; int64_t count; } mo_plan_agg_value_t;

#define MO_XCALL_Q6_FILTER_SUM 0x2000
typedef struct mo_q6_params_t {
    int32_t date_lo, date_hi;  /* date_lo <= d < date_hi */
    double disc_lo, disc_hi;   /* disc_lo <= b <= disc_hi (BETWEEN) */
    double qty_hi;             /* c < qty_hi */
} mo_q6_params_t;

/* Asynchronous form: device columns AND a device result (pdata 16 bytes = {f64 sum, i64 qualifying rows}, pnulls device or NULL): the
 * call enqueues the kernel on the calling thread's stream and returns at once.
 * MO_XCALL_Q6_MERGE (MergeGroup): args [0] result as above ; [1] len partial results of 16 bytes each, added in order; an empty partial
 * (count 0) is NULL and skipped (sumavg2.go:222-236). */
#define MO_XCALL_Q6_MERGE 0x2002

/* --- new: fused TPC-H Q1 shape: filter d <= cutoff, group by two 1-byte keys, 8 aggregates (q1.sql:5-12).
 * args: [0] result: pdata -> mo_q1_result_t ; [1] shipdate int32 ; [2] quantity f64 ; [3] extendedprice f64 ;
 * [4] discount f64 ; [5] tax f64 ; [6] returnflag ; [7] linestatus ; [8] params: pdata -> int32 cutoff.
 * Key columns: dataSz == len -> packed uint8 column; dataSz == 24*len -> MatrixOne varlena cells (inline char(1)). */
#define MO_XCALL_Q1_GROUP_AGG 0x2001
/* args[8] may also hold mo_q1_params_t (dataSz >= 16): row_base is added to every first_row (the block-range offset of this shard), so
 * partial results of different shards order their groups globally.  Asynchronous form as for Q6 (device columns + device result);
 * there "more than MO_Q1_MAX_GROUPS keys" is reported as ngroups = -1 instead of MO_RC_INVALID_ARGUMENT.
 * MO_XCALL_Q1_MERGE (MergeGroup): args [0] mo_q1_result_t ; [1] len partial mo_q1_result_t, merged in order, groups re-sorted by
 * first_row, averages recomputed from the merged sums and counts. */
#define MO_XCALL_Q1_MERGE 0x2003
typedef struct mo_q1_params_t { int32_t cutoff; int32_t reserved; int64_t row_base; } mo_q1_params_t;
#define MO_Q1_MAX_GROUPS 8
typedef struct mo_q1_group_t {
    uint8_t returnflag, linestatus; uint8_t pad[6];
    int64_t first_row;      /* global row index of the first qualifying row of the group (first-seen order) */
    double sum_qty, sum_base_price, sum_disc_price, sum_charge, avg_qty, avg_price, avg_disc;
    double sum_disc;        /* numerator of avg_disc (partials for a cross-GPU reduce) */
    int64_t count_order;
} mo_q1_group_t;
typedef struct mo_q1_result_t {
    int64_t ngroups;        /* groups sorted by first_row (= reference first-seen group-id order) */
    mo_q1_group_t groups[MO_Q1_MAX_GROUPS];
} mo_q1_result_t;

/* --- new: brute-force top-k (GoBruteForceIndex.Search, pkg/vectorindex/brute_force/brute_force.go:248-341).
 * args: [0] result keys int64[nq*k] ; [1] result distances f64[nq*k] ; [2] dataset f32 row-major (dataSz = n*dim*4)
 * ; [3] queries f32 row-major (dataSz = nq*dim*4) ; [4] params: pdata -> mo_search_params_t.  len = nq.
 * Distances are bit-exact with the Go metric functions; ties between equal distances resolve to the lower row id. */
#define MO_XCALL_BRUTEFORCE_TOPK_F32 0x3000
/* IVF-flat probe (IvfflatSearchIndex.Search, pkg/vectorindex/ivfflat/search.go:509-630):
 * args as above plus [5] centroids f32 (nlist*dim) ; [6] list offsets int64[nlist+1] into a list-ordered dataset ;
 * [7] row ids int64[n] (original pk of each list-ordered row). */
#define MO_XCALL_IVF_TOPK_F32 0x3001
typedef struct mo_search_params_t {
    int64_t n, dim, nq;
    int32_t k;        /* RuntimeConfig.Limit */
    int32_t metric;   /* MO_METRIC_* */
    int32_t nprobe;   /* IVF only */
    int32_t sqrt_out; /* DistanceTransformIvfflat: sqrt on the final k (user asked l2_distance) */
    int64_t nlist;    /* IVF only */
    int64_t key_base; /* added to row ordinals (dataset shard offset in a multi-GPU run) */
} mo_search_params_t;
#define MO_METRIC_L2 0      /* metric/types.go MetricType: both L2 variants search with L2sq (distance_func.go:507-524) */
#define MO_METRIC_IP 1
#define MO_METRIC_COS 2
#define MO_METRIC_L1 3
#define MO_METRIC_L2SQ 4

/* merge of per-shard top-k lists (MergeTop / hnsw sub-index merge, pkg/vectorindex/hnsw/search.go:89-135):
 * args: [0] out keys int64[nq*k] ; [1] out dist f64[nq*k] ; [2] in keys int64[nshards*nq*k] ; [3] in dist f64[...] ;
 * [4] params mo_search_params_t (n = nshards, nq, k). */
#define MO_XCALL_TOPK_MERGE 0x3002

/* ======================================================================================================
 * PART 3 -- runtime / residency extension
 * ==================================================================================================== */
int32_t MoB200_Init(int32_t device);          /* idempotent; device < 0 -> $MO_B200_DEVICE, $LOCAL_RANK or 0 */
const char *MoB200_Version(void);
int32_t MoB200_DeviceCount(void);
int32_t MoB200_DeviceAlloc(uint64_t bytes, void **dptr);
int32_t MoB200_DeviceFree(void *dptr);
int32_t MoB200_HostAlloc(uint64_t bytes, void **hptr);  /* pinned host memory (replaces malloc.CAllocator) */
int32_t MoB200_HostFree(void *hptr);
int32_t MoB200_HostRegister(void *hptr, uint64_t bytes);
int32_t MoB200_HostUnregister(void *hptr);
int32_t MoB200_Upload(void *dst_dev, const void *src_host, uint64_t bytes);   /* on the calling thread's stream, synchronous */
int32_t MoB200_Download(void *dst_host, const void *src_dev, uint64_t bytes);
int32_t MoB200_DownloadAsync(void *dst_host, const void *src_dev, uint64_t bytes);  /* stream-ordered, NO synchronise (pinned host memory) */
int32_t MoB200_UploadAsync(void *dst_dev, const void *src_host, uint64_t bytes);
int32_t MoB200_Memset(void *dst_dev, int32_t value, uint64_t bytes);
/* Device column cache (off by default).  The ABI hands the library HOST vectors; re-uploading a column on every call makes every call
 * PCIe-bound (the reference's CUDA shim re-allocates and re-copies per call, cgo/cuda/cuda.cpp:123-201).  A caller that knows a host range is
 * immutable -- the column of a decoded block, an index's dataset -- pins it once: ColumnPin uploads [host, host + bytes) and from then on EVERY
 * entry point that is handed a host pointer inside that range reads the device copy instead of staging it.  `generation` distinguishes reuses of
 * the same buffer (block id / version): pinning the same address with another generation replaces the copy.  LRU eviction beyond the capacity. */
int32_t MoB200_ColumnCacheConfigure(uint64_t capacity_bytes);   /* 0 = off (drops everything) */
int32_t MoB200_ColumnPin(const void *host, uint64_t bytes, uint64_t generation);
int32_t MoB200_ColumnUnpin(const void *host);
int32_t MoB200_ColumnCacheStats(uint64_t *hits, uint64_t *misses, uint64_t *bytes);

/* prepared join maps: build the probe-side device hash table of a JoinMap once (the JoinMap message lives for the whole probe phase,
 * pkg/vm/message/joinMapMsg.go:127-160); JOIN_FIND / JOIN_PROBE calls whose table_keys pointer equals `table_keys` reuse it. */
int32_t MoB200_JoinMapPrepare(const void *table_keys, uint64_t ngroups);
int32_t MoB200_JoinMapRelease(const void *table_keys);
/* the same for a string-keyed JoinMap (MO_XCALL_STR_JOIN_FIND / STR_JOIN_PROBE): the key table (offsets int64[ngroups + 1] + bytes) is copied to
 * the device with its hash table; calls whose table offsets pointer equals `key_offsets` (and whose group count matches) use the prepared copy. */
int32_t MoB200_StrJoinMapPrepare(const void *key_offsets, const void *key_bytes, uint64_t ngroups);
int32_t MoB200_StrJoinMapRelease(const void *key_offsets);
int32_t MoB200_Sync(void);                    /* synchronize the calling thread's stream */
int32_t MoB200_SetStream(void *cuda_stream);  /* adopt an external cudaStream_t for the calling thread (NULL = own) */
int32_t MoB200_TimerStart(void);              /* CUDA event on the calling thread's stream */
int32_t MoB200_TimerStop(float *ms);          /* records, synchronizes, returns elapsed milliseconds */
uint64_t MoB200_KernelLaunchCount(void);      /* kernels launched by this library since load (all threads) */
int32_t MoB200_LastKernelMs(float *ms);       /* device time of the dominant kernel of the calling thread's last call (CUDA events) */
int32_t MoB200_LastError(char *buf, uint64_t buflen);  /* thread-local last error text */
int32_t MoB200_FlushL2(void);                 /* write a >L2-sized scratch buffer (bench hygiene) */
int32_t MoB200_SetTuning(const char *name, int32_t value);
void *MoB200_DebugBuffer(void);               /* per-CTA phase timestamps of the last Q1 launch when SetTuning("q1_debug",1) */  /* kernel-variant knobs used by tools/tune.py; returns 0 if known */

/* synthetic column generators used by bench.py / tests (counter-based, reproducible on the host: see
 * matrixone_b200/datagen.py).  All write DEVICE memory, rows [row0, row0+n). */
int32_t MoB200_GenLineitem(uint64_t seed, uint64_t row0, uint64_t n, int32_t *shipdate, double *quantity,
                           double *extendedprice, double *discount, double *tax, uint8_t *returnflag, uint8_t *linestatus);
int32_t MoB200_GenInt64(uint64_t seed, uint64_t row0, uint64_t n, int64_t *out, uint64_t *nulls, uint32_t null_per_mille);
int32_t MoB200_GenVectorsF32(uint64_t seed, uint64_t row0, uint64_t n, int64_t dim, float *out,
                             const float *centers, int64_t ncenters, float sigma);
int32_t MoB200_GatherRowsF32(float *dst, const float *src, const int64_t *idx, uint64_t m, int64_t dim);  /* device pointers */

/* Index load hooks (brute_force.go:104-123 Load / ivfflat/search.go:216-290 LoadIndex build the reference's in-memory index once;
 * Destroy frees it).  SearchPrepare splits a RESIDENT float32 dataset [n][dim] into the tensor-core operand of
 * MO_XCALL_BRUTEFORCE_TOPK_F32 / MO_XCALL_IVF_TOPK_F32 once, instead of once per search; the rows must not change until
 * SearchRelease(data).  Optional: searches return identical results with or without it.  Costs 6*dim bytes of HBM per row. */
int32_t MoB200_SearchPrepare(const void *data, uint64_t n, int64_t dim);   /* = SearchPrepareMetric(..., MO_METRIC_L2) */
/* MO_METRIC_L2 / L2SQ / IP share one operand; MO_METRIC_COS keeps the rows normalised; other metrics have nothing to prepare */
int32_t MoB200_SearchPrepareMetric(const void *data, uint64_t n, int64_t dim, int32_t metric);
/* IVF-flat: the list-ordered entries are split as residuals against their list's centroid (centroids [nlist][dim] float32,
 * offsets [nlist + 1] int64, device pointers; the same buffers MO_XCALL_IVF_TOPK_F32 is later called with). */
int32_t MoB200_SearchPrepareIvf(const void *data, uint64_t n, int64_t dim, const void *centroids, uint64_t nlist, const void *offsets);
int32_t MoB200_SearchRelease(const void *data);

#ifdef __cplusplus
}
#endif
#endif /* _MO_B200_H_ */
