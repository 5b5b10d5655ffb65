// colops.cu -- the standalone column operators of the colexec pipeline, one kernel family per reference operator:
//
//   MO_XCALL_FILTER_SELS      Filter.Call inner loop: bool vector (+nulls) -> ascending sels     pkg/sql/colexec/filter/filter.go:116-152
//   MO_XCALL_SHUFFLE(szof)    Vector.Shrink / Union / shuffle.FixedLengthShuffle + nulls.Filter   pkg/container/vector/vector.go:1014,2583,
//                                                                                                 pkg/vectorize/shuffle/shuffle.go:21-26,
//                                                                                                 pkg/container/nulls/nulls.go:237-281
//   MO_XCALL_PACK_KEYS        intHashMapIterator.encodeHashKeys / fillKeys (<= 8 key bytes)       pkg/common/hashmap/inthashmap.go:92-183
//   MO_XCALL_GROUP_IDS        IntHashMap insert: 1-based group ids in FIRST-SEEN order            pkg/common/hashmap/iterator.go:127-148,
//                                                                                                 pkg/container/hashtable/int64_hash_map.go:92-158
//   MO_XCALL_GROUP_AGG(op,T)  sumAvgExec / countColumnExec / minMaxExecFixed .BatchFill           pkg/sql/colexec/aggexec/{sumavg2,count2,minmax2}.go
//
// These are what the fused plans (tpch.cu, plan.cu) are built from; exposed on their own they make every operator of the chain
// available on resident columns.  All are HBM- or atomic-throughput bound integer/byte kernels: coalesced 128-bit loads, warp
// ballots for bitmaps, a single-pass decoupled look-back scan for the order-preserving compaction.
#include "hashops.cuh"
#include <cstring>

using namespace mob;

namespace {

int type_size(int T) {
    switch (T) {
    case MO_T_BOOL: case MO_T_INT8: case MO_T_UINT8: return 1;
    case MO_T_INT16: case MO_T_UINT16: return 2;
    case MO_T_INT32: case MO_T_UINT32: case MO_T_FLOAT32: case MO_T_DATE: return 4;
    case MO_T_INT64: case MO_T_UINT64: case MO_T_FLOAT64: case MO_T_TIME: case MO_T_DATETIME: case MO_T_TIMESTAMP: return 8;
    }
    return 0;
}

constexpr int kThreads = 256;

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
}

// =========================================================================================================
// order-preserving compaction: indices of the flagged rows, ascending.  Single pass over the flags (decoupled look-back):
// a CTA takes the next tile (atomic ticket, so every predecessor tile is already running), counts its flagged rows, publishes
// (aggregate | inclusive prefix) in one 64-bit status word, and walks back over its predecessors' words for its exclusive prefix.
// =========================================================================================================
constexpr int kSelThreads = 256, kSelRows = 32, kSelTile = kSelThreads * kSelRows;   // 8192 rows per tile = one MatrixOne block
constexpr unsigned long long kFlagA = 1ull << 62, kFlagP = 2ull << 62, kValMask = (1ull << 62) - 1;

template <typename OutT>
__global__ void __launch_bounds__(kSelThreads)
select_kernel(const uint8_t *__restrict__ v, const uint64_t *__restrict__ nulls, uint64_t n, OutT *__restrict__ sels,
              unsigned long long *status, unsigned *ticket, unsigned long long *total, int aligned) {
    __shared__ unsigned s_tile;
    __shared__ unsigned s_warp[kSelThreads / 32];
    __shared__ unsigned long long s_prefix;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const unsigned tile = s_tile;
    const uint64_t ntiles = (n + kSelTile - 1) / kSelTile;
    const uint64_t row0 = (uint64_t)tile * kSelTile + (uint64_t)threadIdx.x * kSelRows;
    unsigned mask = 0;
    if (row0 + kSelRows <= n && aligned) {
        const int4 x0 = ld_stream16(v + row0), x1 = ld_stream16(v + row0 + 16);
        const unsigned w[8] = {(unsigned)x0.x, (unsigned)x0.y, (unsigned)x0.z, (unsigned)x0.w, (unsigned)x1.x, (unsigned)x1.y, (unsigned)x1.z, (unsigned)x1.w};
#pragma unroll
        for (int j = 0; j < 32; j++) mask |= (((w[j >> 2] >> (8 * (j & 3))) & 0xffu) ? 1u : 0u) << j;
    } else {
        for (int j = 0; j < kSelRows; j++) if (row0 + j < n && v[row0 + j]) mask |= 1u << j;
    }
    if (nulls && row0 < n) mask &= ~(unsigned)((nulls[row0 >> 6] >> (row0 & 63)) & 0xffffffffu);   // 32 rows never straddle a word
    const unsigned cnt = __popc(mask);
    // CTA exclusive scan of cnt
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned inc = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    unsigned wbase = 0, agg = 0;
#pragma unroll
    for (int w = 0; w < kSelThreads / 32; w++) { if (w < warp) wbase += s_warp[w]; agg += s_warp[w]; }
    if (threadIdx.x == 0) {
        unsigned long long excl = 0;
        if (tile == 0) {
            atomicExch(&status[0], kFlagP | (unsigned long long)agg);
        } else {
            atomicExch(&status[tile], kFlagA | (unsigned long long)agg);
            for (long long p = (long long)tile - 1; p >= 0; p--) {
                unsigned long long s;
                do { s = *((volatile unsigned long long *)&status[p]); } while ((s >> 62) == 0);
                excl += s & kValMask;
                if ((s >> 62) == 2) break;
            }
            atomicExch(&status[tile], kFlagP | (excl + agg));
        }
        s_prefix = excl;
        if (tile == ntiles - 1) *total = excl + agg;
    }
    // the selected rows of the tile are first listed in shared memory (16-bit offsets inside the tile, at their rank), then written out by the
    // whole CTA with consecutive threads on consecutive slots: one coalesced stream instead of 256 interleaved per-thread runs
    __shared__ unsigned short s_list[kSelTile];
    unsigned lpos = wbase + (inc - cnt);
    const unsigned tbase = threadIdx.x * kSelRows;
    while (mask) { const int j = __ffs(mask) - 1; mask &= mask - 1; s_list[lpos++] = (unsigned short)(tbase + j); }
    __syncthreads();
    const unsigned long long out0 = s_prefix;
    const uint64_t tile_row0 = (uint64_t)tile * kSelTile;
    for (unsigned i = threadIdx.x; i < agg; i += kSelThreads) sels[out0 + i] = (OutT)(tile_row0 + s_list[i]);
}

}  // namespace

namespace mob {
// launches the compaction; *dtotal (device) receives the count.  status/ticket scratch comes from the arena.
template <typename OutT>
int launch_select(ThreadCtx &t, const uint8_t *v, const uint64_t *nulls, uint64_t n, OutT *sels, unsigned long long *dtotal) {
    if (n == 0) { MOB_CUDA_TRY(cudaMemsetAsync(dtotal, 0, 8, t.stream)); return MO_RC_SUCCESS; }
    const uint64_t ntiles = (n + kSelTile - 1) / kSelTile;
    unsigned long long *status = (unsigned long long *)arena_alloc(t, ntiles * 8 + 16);
    if (!status) return MO_RC_INTERNAL_ERROR;
    MOB_CUDA_TRY(cudaMemsetAsync(status, 0, ntiles * 8 + 16, t.stream));
    unsigned *ticket = (unsigned *)(status + ntiles);
    select_kernel<OutT><<<(unsigned)ntiles, kSelThreads, 0, t.stream>>>(v, nulls, n, sels, status, ticket, dtotal, (((uintptr_t)v) & 15) == 0 ? 1 : 0);
    MOB_LAUNCH_CHECK();
    return MO_RC_SUCCESS;
}
template int launch_select<int64_t>(ThreadCtx &, const uint8_t *, const uint64_t *, uint64_t, int64_t *, unsigned long long *);
template int launch_select<uint32_t>(ThreadCtx &, const uint8_t *, const uint64_t *, uint64_t, uint32_t *, unsigned long long *);
}  // namespace mob

namespace {

// =========================================================================================================
// gather (Shrink / Union / FixedLengthShuffle) with nulls.Filter fused: dst[i] = src[sels[i]], dst null bit i = src null bit sels[i]
// =========================================================================================================
template <typename E>
__global__ void __launch_bounds__(kThreads)
gather_kernel(E *__restrict__ dst, const E *__restrict__ src, const int64_t *__restrict__ sels, uint64_t nsel,
              const uint64_t *__restrict__ snulls, uint64_t snull_bits, uint32_t *__restrict__ dnulls32) {
    const uint64_t n64 = (nsel + 63) & ~63ull;   // whole uint64 words of the destination bitmap are written (zero past nsel)
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n64; i += (uint64_t)gridDim.x * kThreads) {
        bool isnull = false;
        if (i < nsel) {
            const uint64_t s = (uint64_t)sels[i];
            dst[i] = src[s];
            isnull = snulls && s < snull_bits && ((snulls[s >> 6] >> (s & 63)) & 1ull);
        }
        if (dnulls32) {
            const unsigned m = __ballot_sync(0xffffffffu, isnull);
            if ((threadIdx.x & 31) == 0) dnulls32[i >> 5] = m;
        }
    }
}
struct Cell24 { uint64_t a, b, c; };
struct Cell16 { uint64_t a, b; };

// =========================================================================================================
// key packing (fillKeys): column k contributes [marker byte (has_null mode)] + its value bytes at the row's running offset
// =========================================================================================================
constexpr int kMaxKeyCols = 8;
struct KeyCols { const uint8_t *col[kMaxKeyCols]; const uint64_t *nulls[kMaxKeyCols]; int size[kMaxKeyCols]; int cst[kMaxKeyCols]; int n; };

__global__ void __launch_bounds__(kThreads)
pack_keys_kernel(uint64_t *__restrict__ keys, uint32_t *__restrict__ skip32, uint64_t n, KeyCols K, int has_null) {
    const uint64_t n32 = (n + 63) & ~63ull;
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n32; i += (uint64_t)gridDim.x * kThreads) {
        bool skip = false;
        if (i < n) {
            uint64_t key = 0; int off = 0;
            for (int k = 0; k < K.n; k++) {
                const uint64_t r = K.cst[k] ? 0 : i;
                const bool isnull = K.nulls[k] && ((K.nulls[k][r >> 6] >> (r & 63)) & 1ull);
                if (has_null) {
                    if (isnull) { key |= 1ull << (8 * off); off += 1; continue; }   // marker 1, no value bytes (inthashmap.go:161-163)
                    off += 1;                                                          // marker 0
                } else if (isnull) { skip = true; continue; }                         // zValues[i] = 0: the row joins no group
                uint64_t val = 0;
                const uint8_t *p = K.col[k] + r * (uint64_t)K.size[k];
                for (int b = 0; b < K.size[k]; b++) val |= (uint64_t)p[b] << (8 * b);
                if (off < 8) key |= val << (8 * off);
                off += K.size[k];
            }
            keys[i] = key;
        }
        if (skip32) {
            const unsigned m = __ballot_sync(0xffffffffu, skip);
            if ((threadIdx.x & 31) == 0) skip32[i >> 5] = m;
        }
    }
}

// =========================================================================================================
// group ids in first-seen order
// =========================================================================================================
// "virtual row" v: v < nexist is existing group v (its key comes from table_keys), v >= nexist is batch row v - nexist.  Every
// distinct key remembers the smallest virtual row that carries it; ranking the keys by that row reproduces the reference's ids:
// existing groups keep theirs, new groups are numbered in the order their first row appears.
constexpr uint64_t kEmptyKey = 0xffffffffffffffffull;
constexpr uint32_t kNoSlot = 0xffffffffu;

struct GidTable { uint64_t *key; unsigned long long *minrow; uint64_t *id; uint64_t mask; /* capacity - 1; slot capacity = sentinel-key slot */ };

__global__ void __launch_bounds__(kThreads)
gid_init_kernel(GidTable T) {
    for (uint64_t s = blockIdx.x * (uint64_t)kThreads + threadIdx.x; s <= T.mask + 1; s += (uint64_t)gridDim.x * kThreads) {
        T.key[s] = kEmptyKey; T.minrow[s] = ~0ull; T.id[s] = 0;
    }
}

__global__ void __launch_bounds__(kThreads)
gid_insert_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ knulls, uint64_t n, const uint64_t *__restrict__ table_keys,
                  uint64_t nexist, GidTable T, uint32_t *__restrict__ rowslot, unsigned *overflow) {
    const uint64_t total = n + nexist;
    for (uint64_t v = blockIdx.x * (uint64_t)kThreads + threadIdx.x; v < total; v += (uint64_t)gridDim.x * kThreads) {
        uint64_t key;
        if (v < nexist) key = table_keys[v];
        else {
            const uint64_t i = v - nexist;
            if (knulls && ((knulls[i >> 6] >> (i & 63)) & 1ull)) { rowslot[v] = kNoSlot; continue; }
            key = keys[i];
        }
        uint64_t slot;
        if (key == kEmptyKey) { slot = T.mask + 1; T.key[slot] = key; }
        else {
            slot = mix64(key) & T.mask;
            uint64_t probes = 0;
            for (;;) {
                uint64_t cur = T.key[slot];
                if (cur == key) break;
                if (cur == kEmptyKey) {
                    cur = atomicCAS((unsigned long long *)&T.key[slot], (unsigned long long)kEmptyKey, (unsigned long long)key);
                    if (cur == kEmptyKey || cur == key) break;
                }
                slot = (slot + 1) & T.mask;
                if (++probes > T.mask) { *overflow = 1; slot = kNoSlot; break; }
            }
            if (slot == kNoSlot) { rowslot[v] = kNoSlot; continue; }
        }
        // monotone: a stale read can only be larger than the truth, so skipping when it is already <= v is safe -- after the first few
        // rows of a group almost every row skips the atomic
        if (*((volatile unsigned long long *)&T.minrow[slot]) > v) atomicMin(&T.minrow[slot], (unsigned long long)v);
        rowslot[v] = (uint32_t)slot;
    }
}

__global__ void __launch_bounds__(kThreads)
gid_flag_kernel(uint64_t total, GidTable T, const uint32_t *__restrict__ rowslot, uint8_t *__restrict__ isfirst) {
    for (uint64_t v = blockIdx.x * (uint64_t)kThreads + threadIdx.x; v < total; v += (uint64_t)gridDim.x * kThreads) {
        const uint32_t s = rowslot[v];
        isfirst[v] = (s != kNoSlot && T.minrow[s] == v) ? 1 : 0;
    }
}

__global__ void __launch_bounds__(kThreads)
gid_assign_kernel(const uint32_t *__restrict__ firsts, const unsigned long long *count, GidTable T, const uint32_t *__restrict__ rowslot,
                  uint64_t *__restrict__ table_keys, uint64_t table_cap, uint64_t nexist, int64_t *ngroups_out, unsigned *overflow) {
    const uint64_t cnt = *count;
    for (uint64_t j = blockIdx.x * (uint64_t)kThreads + threadIdx.x; j < cnt; j += (uint64_t)gridDim.x * kThreads) {
        const uint32_t s = rowslot[firsts[j]];
        T.id[s] = j + 1;
        if (j >= nexist) { if (j < table_cap) table_keys[j] = T.key[s]; else *overflow = 2; }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *ngroups_out = (int64_t)cnt;
}

__global__ void __launch_bounds__(kThreads)
gid_emit_kernel(uint64_t *__restrict__ groups, uint64_t n, uint64_t nexist, GidTable T, const uint32_t *__restrict__ rowslot) {
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        const uint32_t s = rowslot[nexist + i];
        groups[i] = s == kNoSlot ? 0ull : T.id[s];
    }
}

// =========================================================================================================
// grouped aggregates (BatchFill): per-group temporaries accumulated with atomics -- in shared memory (replicated per lane group so
// equal group ids of one warp do not collide) when there are few groups, directly in global memory otherwise -- then folded into the
// caller's persistent state with the reference's rules (overflow checks, NULL until the first value, strict compare for MIN/MAX).
// =========================================================================================================
enum AggKind { G_SUM_SIGNED = 0, G_SUM_UNSIGNED = 1, G_SUM_FLOAT = 2, G_COUNT = 3, G_MIN_INT = 4, G_MAX_INT = 5, G_MIN_UINT = 6, G_MAX_UINT = 7, G_MIN_FLT = 8, G_MAX_FLT = 9 };
constexpr int kSmemSlots = 1024;   // group x replica slots kept in shared memory (4 arrays x 8 bytes = 32 KB)

// total order on non-NaN doubles as unsigned integers; -0.0 is folded onto +0.0 (they compare equal in the reference too)
__device__ __forceinline__ unsigned long long flt_key(double d) {
    if (d == 0.0) d = 0.0;
    unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b >> 63) ? ~b : (b | (1ull << 63));
}
__device__ __forceinline__ double flt_unkey(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & ~(1ull << 63)) : ~k;
    return __longlong_as_double((long long)b);
}

template <int KIND> __device__ __forceinline__ unsigned long long a0_identity() {
    if (KIND == G_MIN_INT) return (unsigned long long)INT64_MAX;
    if (KIND == G_MAX_INT) return (unsigned long long)INT64_MIN;
    if (KIND == G_MIN_UINT || KIND == G_MIN_FLT) return ~0ull;
    return 0ull;
}

struct AggTemp { unsigned long long *a0, *a1, *a2, *cnt; };

template <typename T, int KIND>
__device__ __forceinline__ void agg_update(unsigned long long *a0, unsigned long long *a1, unsigned long long *a2, unsigned long long *cnt, T v, uint64_t row) {
    if (KIND == G_SUM_SIGNED) {
        const int64_t x = (int64_t)v;
        const uint64_t m = x < 0 ? (0ull - (uint64_t)x) : (uint64_t)x;
        atomicAdd(a0, (unsigned long long)x);
        atomicAdd(a1, (unsigned long long)(m & 0xffffffffull));
        if (m >> 32) atomicAdd(a2, (unsigned long long)(m >> 32));
    } else if (KIND == G_SUM_UNSIGNED) {
        const uint64_t x = (uint64_t)v;
        atomicAdd(a1, (unsigned long long)(x & 0xffffffffull));
        if (x >> 32) atomicAdd(a2, (unsigned long long)(x >> 32));
    } else if (KIND == G_SUM_FLOAT) {
        atomicAdd(reinterpret_cast<double *>(a0), (double)v);
    } else if (KIND == G_MIN_INT) atomicMin(reinterpret_cast<long long *>(a0), (long long)v);
    else if (KIND == G_MAX_INT) atomicMax(reinterpret_cast<long long *>(a0), (long long)v);
    else if (KIND == G_MIN_UINT) atomicMin(a0, (unsigned long long)v);
    else if (KIND == G_MAX_UINT) atomicMax(a0, (unsigned long long)v);
    else if (KIND == G_MIN_FLT || KIND == G_MAX_FLT) {
        const double d = (double)v;
        if (d == d) { if (KIND == G_MIN_FLT) atomicMin(a0, flt_key(d)); else atomicMax(a0, flt_key(d)); }
        atomicMin(a1, (unsigned long long)row);   // first non-null row of the group in this batch (the NaN rule needs it)
    }
    atomicAdd(cnt, 1ull);
}

template <int KIND>
__global__ void __launch_bounds__(kThreads)
agg_temp_init_kernel(AggTemp A, uint64_t ngroups) {
    for (uint64_t g = blockIdx.x * (uint64_t)kThreads + threadIdx.x; g < ngroups; g += (uint64_t)gridDim.x * kThreads) {
        A.a0[g] = a0_identity<KIND>(); A.a1[g] = (KIND == G_MIN_FLT || KIND == G_MAX_FLT) ? ~0ull : 0ull; A.a2[g] = 0; A.cnt[g] = 0;
    }
}

template <typename T, int KIND, bool SMEM>
__global__ void __launch_bounds__(kThreads)
group_agg_kernel(const uint64_t *__restrict__ groups, const T *__restrict__ col, const uint64_t *__restrict__ nulls, uint64_t n,
                 uint64_t ngroups, int rep_shift, AggTemp A, unsigned *bad_group) {
    __shared__ unsigned long long s0[SMEM ? kSmemSlots : 1], s1[SMEM ? kSmemSlots : 1], s2[SMEM ? kSmemSlots : 1], sc[SMEM ? kSmemSlots : 1];
    const int rep_mask = (1 << rep_shift) - 1;
    if (SMEM) {
        for (int s = threadIdx.x; s < (int)(ngroups << rep_shift); s += kThreads) {
            s0[s] = a0_identity<KIND>(); s1[s] = (KIND == G_MIN_FLT || KIND == G_MAX_FLT) ? ~0ull : 0ull; s2[s] = 0; sc[s] = 0;
        }
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        const uint64_t g = groups[i];
        if (g == 0) continue;                       // GroupNotMatched
        if (g > ngroups) { *bad_group = 1; continue; }
        if (nulls && ((nulls[i >> 6] >> (i & 63)) & 1ull)) continue;
        T v = KIND == G_COUNT ? T(0) : col[i];
        if (SMEM) { const int s = (int)((g - 1) << rep_shift) + (lane & rep_mask); agg_update<T, KIND>(&s0[s], &s1[s], &s2[s], &sc[s], v, i); }
        else agg_update<T, KIND>(&A.a0[g - 1], &A.a1[g - 1], &A.a2[g - 1], &A.cnt[g - 1], v, i);
    }
    if (SMEM) {
        __syncthreads();
        for (int s = threadIdx.x; s < (int)(ngroups << rep_shift); s += kThreads) {
            if (sc[s] == 0) continue;
            const uint64_t g = (uint64_t)s >> rep_shift;
            if (KIND == G_SUM_SIGNED) { atomicAdd(&A.a0[g], s0[s]); atomicAdd(&A.a1[g], s1[s]); atomicAdd(&A.a2[g], s2[s]); }
            else if (KIND == G_SUM_UNSIGNED) { atomicAdd(&A.a1[g], s1[s]); atomicAdd(&A.a2[g], s2[s]); }
            else if (KIND == G_SUM_FLOAT) atomicAdd(reinterpret_cast<double *>(&A.a0[g]), __longlong_as_double((long long)s0[s]));
            else if (KIND == G_MIN_INT) atomicMin(reinterpret_cast<long long *>(&A.a0[g]), (long long)s0[s]);
            else if (KIND == G_MAX_INT) atomicMax(reinterpret_cast<long long *>(&A.a0[g]), (long long)s0[s]);
            else if (KIND == G_MIN_UINT || KIND == G_MIN_FLT) atomicMin(&A.a0[g], s0[s]);
            else if (KIND == G_MAX_UINT || KIND == G_MAX_FLT) atomicMax(&A.a0[g], s0[s]);
            if (KIND == G_MIN_FLT || KIND == G_MAX_FLT) atomicMin(&A.a1[g], s1[s]);
            atomicAdd(&A.cnt[g], sc[s]);
        }
    }
}

// fold the batch temporaries into the caller's state.  status[0] = rc, status[1] = first group (0-based) needing the exact serial check
template <typename T, int KIND>
__global__ void __launch_bounds__(kThreads)
agg_fold_kernel(uint64_t *__restrict__ state, uint64_t *__restrict__ snulls, int64_t *__restrict__ counts, uint64_t ngroups, AggTemp A,
                const T *__restrict__ col, int is_avg, unsigned long long *status, uint8_t *needs_serial) {
    for (uint64_t g = blockIdx.x * (uint64_t)kThreads + threadIdx.x; g < ngroups; g += (uint64_t)gridDim.x * kThreads) {
        const unsigned long long c = A.cnt[g];
        if (KIND == G_COUNT) { state[g] = (uint64_t)((int64_t)state[g] + (int64_t)c); continue; }
        if (c == 0) continue;
        bool was_null = snulls ? ((snulls[g >> 6] >> (g & 63)) & 1ull) != 0 : false;
        if (is_avg && counts) was_null = counts[g] == 0;
        if (KIND == G_SUM_SIGNED) {
            const __int128 mag = ((__int128)A.a2[g] << 32) + (__int128)A.a1[g];
            const int64_t cur = was_null ? 0 : (int64_t)state[g];
            const __int128 bound = mag + (cur < 0 ? -(__int128)cur : (__int128)cur);
            if (bound <= (__int128)INT64_MAX) state[g] = (uint64_t)(cur + (int64_t)A.a0[g]);   // no prefix can leave int64
            else { needs_serial[g] = 1; atomicMin(&status[1], (unsigned long long)g); }
        } else if (KIND == G_SUM_UNSIGNED) {
            const unsigned __int128 tot = ((unsigned __int128)A.a2[g] << 32) + (unsigned __int128)A.a1[g] + (unsigned __int128)(was_null ? 0ull : state[g]);
            if (tot >> 64) atomicMax(&status[0], (unsigned long long)MO_RC_OUT_OF_RANGE);   // prefixes are monotone: overflow iff the total overflows
            state[g] = (uint64_t)tot;
        } else if (KIND == G_SUM_FLOAT) {
            const double cur = was_null ? 0.0 : __longlong_as_double((long long)state[g]);
            state[g] = (uint64_t)__double_as_longlong(cur + __longlong_as_double((long long)A.a0[g]));
        } else if (KIND == G_MIN_INT || KIND == G_MAX_INT) {
            const int64_t b = (int64_t)A.a0[g], cur = (int64_t)state[g];
            if (was_null || (KIND == G_MIN_INT ? b < cur : b > cur)) state[g] = (uint64_t)b;
        } else if (KIND == G_MIN_UINT || KIND == G_MAX_UINT) {
            const uint64_t b = A.a0[g], cur = state[g];
            if (was_null || (KIND == G_MIN_UINT ? b < cur : b > cur)) state[g] = b;
        } else {   // float MIN / MAX with the Go NaN rule (minmax2.go:69-75): the first value initialises, `<` never replaces a NaN
            const double first = (double)col[A.a1[g]];
            double cur = was_null ? first : (sizeof(T) == 4 ? (double)__uint_as_float((unsigned)state[g]) : __longlong_as_double((long long)state[g]));
            if (cur == cur) {
                const bool any = KIND == G_MIN_FLT ? A.a0[g] != ~0ull : A.a0[g] != 0ull;
                if (any) { const double b = flt_unkey(A.a0[g]); if (KIND == G_MIN_FLT ? b < cur : b > cur) cur = b; }
            }
            if (sizeof(T) == 4) state[g] = (uint64_t)__float_as_uint((float)cur); else state[g] = (uint64_t)__double_as_longlong(cur);
        }
        if (snulls) atomicAnd((unsigned long long *)&snulls[g >> 6], ~(1ull << (g & 63)));
        if (counts) counts[g] += (int64_t)c;
    }
}

// exact serial-order check for the (pathological) groups whose magnitude sum does not fit int64: one thread per flagged group walks
// the batch in row order with int64OfCheck (sumavg2.go:89-94)
template <typename T>
__global__ void agg_serial_signed_kernel(const uint64_t *__restrict__ groups, const T *__restrict__ col, const uint64_t *__restrict__ nulls, uint64_t n,
                                         uint64_t ngroups, uint64_t *state, uint64_t *snulls, int64_t *counts, int is_avg, const uint8_t *needs_serial,
                                         unsigned long long *status) {
    const uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (g >= ngroups || !needs_serial[g]) return;
    bool was_null = snulls ? ((snulls[g >> 6] >> (g & 63)) & 1ull) != 0 : false;
    if (is_avg && counts) was_null = counts[g] == 0;
    int64_t s = was_null ? 0 : (int64_t)state[g];
    int64_t c = 0;
    for (uint64_t i = 0; i < n; i++) {
        if (groups[i] != g + 1) continue;
        if (nulls && ((nulls[i >> 6] >> (i & 63)) & 1ull)) continue;
        const int64_t v = (int64_t)col[i];
        const int64_t r = (int64_t)((uint64_t)s + (uint64_t)v);
        if ((s > 0 && v > 0 && r <= 0) || (s < 0 && v < 0 && r >= 0)) { atomicMax(&status[0], (unsigned long long)MO_RC_OUT_OF_RANGE); return; }
        s = r; c++;
    }
    state[g] = (uint64_t)s;
    if (snulls && c) atomicAnd((unsigned long long *)&snulls[g >> 6], ~(1ull << (g & 63)));
    if (counts) counts[g] += c;
}

template <typename T, int KIND>
int run_group_agg(ThreadCtx &t, mo_xcall_args_t *args, uint64_t len, int is_avg) {
    const uint64_t ngroups = args[0].dataSz / 8;
    if (ngroups == 0) return MO_RC_SUCCESS;
    const uint64_t nwords = (len + 63) / 64, gwords = (ngroups + 63) / 64;
    Stager st(t);
    uint64_t *state = (uint64_t *)st.out(args[0].pdata, ngroups * 8, true);
    uint64_t *snulls = (uint64_t *)st.out(args[0].pnulls, args[0].pnulls ? gwords * 8 : 0, true);
    int64_t *counts = (int64_t *)st.out(args[1].pdata, args[1].pdata ? ngroups * 8 : 0, true);
    const uint64_t *groups = (const uint64_t *)st.in(args[2].pdata, len * 8);
    const T *col = (const T *)st.in(args[3].pdata, KIND == G_COUNT ? 0 : len * sizeof(T));
    const uint64_t *nulls = (const uint64_t *)st.in(args[3].pnulls, args[3].pnulls ? nwords * 8 : 0);
    unsigned long long *tmp = (unsigned long long *)st.tmp(ngroups * 8 * 4 + ngroups + 64);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    AggTemp A{tmp, tmp + ngroups, tmp + 2 * ngroups, tmp + 3 * ngroups};
    uint8_t *needs_serial = (uint8_t *)(tmp + 4 * ngroups);
    unsigned long long *status = (unsigned long long *)(needs_serial + ((ngroups + 15) & ~15ull));
    unsigned *bad = (unsigned *)(status + 2);
    const int ggrid = (int)((ngroups + kThreads - 1) / kThreads > 2048 ? 2048 : (ngroups + kThreads - 1) / kThreads);
    agg_temp_init_kernel<KIND><<<ggrid, kThreads, 0, t.stream>>>(A, ngroups);
    MOB_LAUNCH_CHECK();
    MOB_CUDA_TRY(cudaMemsetAsync(needs_serial, 0, ((ngroups + 15) & ~15ull) + 32, t.stream));
    MOB_CUDA_TRY(cudaMemsetAsync(status + 1, 0xff, 8, t.stream));
    if (len) {
        int grid = num_sms() * 8;
        const uint64_t work = (len + kThreads - 1) / kThreads;
        if ((uint64_t)grid > work) grid = (int)work;
        cudaEventRecord(t.kev0, t.stream);
        if (ngroups <= (uint64_t)kSmemSlots) {
            int rep_shift = 0;
            while (rep_shift < 5 && (ngroups << (rep_shift + 1)) <= (uint64_t)kSmemSlots) rep_shift++;
            group_agg_kernel<T, KIND, true><<<grid, kThreads, 0, t.stream>>>(groups, col, nulls, len, ngroups, rep_shift, A, bad);
        } else {
            group_agg_kernel<T, KIND, false><<<grid, kThreads, 0, t.stream>>>(groups, col, nulls, len, ngroups, 0, A, bad);
        }
        cudaEventRecord(t.kev1, t.stream);
        MOB_LAUNCH_CHECK();
    }
    agg_fold_kernel<T, KIND><<<ggrid, kThreads, 0, t.stream>>>(state, snulls, counts, ngroups, A, col, is_avg, status, needs_serial);
    MOB_LAUNCH_CHECK();
    unsigned long long hst[3];
    int rc = read_back(t, hst, status, 24);
    if (rc) { st.finish(); return rc; }
    if (((unsigned *)&hst[2])[0]) { st.finish(); set_error("group agg: a group id exceeds the state's group count %llu", (unsigned long long)ngroups); return MO_RC_INVALID_ARGUMENT; }
    if (KIND == G_SUM_SIGNED && hst[1] != ~0ull) {
        agg_serial_signed_kernel<T><<<(unsigned)((ngroups + 63) / 64), 64, 0, t.stream>>>(groups, col, nulls, len, ngroups, state, snulls, counts, is_avg, needs_serial, status);
        MOB_LAUNCH_CHECK();
        rc = read_back(t, hst, status, 8);
        if (rc) { st.finish(); return rc; }
    }
    int frc = st.finish();
    if (hst[0]) { set_error("data out of range: grouped SUM overflows its 64-bit state"); return (int)hst[0]; }
    return frc;
}

template <int KIND_INT_S, int KIND_INT_U, int KIND_F>
int dispatch_minmax(ThreadCtx &t, int T, mo_xcall_args_t *args, uint64_t len) {
    switch (T) {
    case MO_T_BOOL: case MO_T_UINT8: return run_group_agg<uint8_t, KIND_INT_U>(t, args, len, 0);
    case MO_T_INT8: return run_group_agg<int8_t, KIND_INT_S>(t, args, len, 0);
    case MO_T_INT16: return run_group_agg<int16_t, KIND_INT_S>(t, args, len, 0);
    case MO_T_UINT16: return run_group_agg<uint16_t, KIND_INT_U>(t, args, len, 0);
    case MO_T_INT32: case MO_T_DATE: return run_group_agg<int32_t, KIND_INT_S>(t, args, len, 0);
    case MO_T_UINT32: return run_group_agg<uint32_t, KIND_INT_U>(t, args, len, 0);
    case MO_T_INT64: case MO_T_TIME: case MO_T_DATETIME: case MO_T_TIMESTAMP: return run_group_agg<int64_t, KIND_INT_S>(t, args, len, 0);
    case MO_T_UINT64: return run_group_agg<uint64_t, KIND_INT_U>(t, args, len, 0);
    case MO_T_FLOAT32: return run_group_agg<float, KIND_F>(t, args, len, 0);
    case MO_T_FLOAT64: return run_group_agg<double, KIND_F>(t, args, len, 0);
    }
    set_error("group agg: unsupported type %d", T);
    return MO_RC_INVALID_ARGUMENT;
}

}  // namespace

namespace mob {

// MO_XCALL_FILTER_SELS: args [0] sels int64[>= count] ; [1] count int64[1] ; [2] bool vector (+pnulls).  len = rows.
int xcall_filter_sels(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!args[1].pdata || args[1].dataSz < 8 || args[2].dataSz < len) { set_error("filter sels: count needs 8 bytes, the bool vector len bytes"); return MO_RC_INVALID_ARGUMENT; }
    const bool dev = is_device_ptr(args[0].pdata) && is_device_ptr(args[1].pdata) && (len == 0 || is_device_ptr(args[2].pdata));
    Stager st(t);
    const uint8_t *v = (const uint8_t *)st.in(args[2].pdata, len);
    const uint64_t *nulls = (const uint64_t *)st.in(args[2].pnulls, args[2].pnulls ? ((len + 63) / 64) * 8 : 0);
    // a host caller's sels buffer only has to hold the selected rows: compact into scratch, copy back `count` entries
    const bool host_out = !is_device_ptr(args[0].pdata);
    int64_t *sels = host_out ? (int64_t *)st.tmp(len * 8 + 8) : (int64_t *)args[0].pdata;
    unsigned long long *dcount = (unsigned long long *)st.out(args[1].pdata, 8);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    cudaEventRecord(t.kev0, t.stream);
    int rc = launch_select<int64_t>(t, v, nulls, len, sels, dcount);
    cudaEventRecord(t.kev1, t.stream);
    if (rc) { st.finish(); return rc; }
    if (dev) { st.release_async(); return MO_RC_SUCCESS; }   // asynchronous form: everything stays on the device
    unsigned long long cnt = 0;
    rc = read_back(t, &cnt, dcount, 8);
    if (rc) { st.finish(); return rc; }
    if (host_out) {
        if (cnt * 8 > args[0].dataSz) { st.finish(); set_error("filter sels: %llu rows selected, the sels buffer holds %llu", cnt, (unsigned long long)(args[0].dataSz / 8)); return MO_RC_INVALID_ARGUMENT; }
        if (cnt) MOB_CUDA_TRY(cudaMemcpyAsync(args[0].pdata, sels, cnt * 8, cudaMemcpyDeviceToHost, t.stream));
    }
    return st.finish();
}

// MO_XCALL_SHUFFLE(szof): args [0] dst (szof bytes x len, + pnulls out) ; [1] src (+pnulls, nullCnt = its bit length) ; [2] sels int64[len]
int xcall_shuffle(int szof, mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (szof != 1 && szof != 2 && szof != 4 && szof != 8 && szof != 16 && szof != 24) { set_error("shuffle: element size %d (1, 2, 4, 8, 16 or 24 = varlena cell)", szof); return MO_RC_INVALID_ARGUMENT; }
    if (args[0].dataSz < (uint64_t)szof * len || args[2].dataSz < 8 * len) { set_error("shuffle: dst / sels shorter than len"); return MO_RC_INVALID_ARGUMENT; }
    if (len == 0) return MO_RC_SUCCESS;
    const bool dev = is_device_ptr(args[0].pdata) && is_device_ptr(args[1].pdata) && is_device_ptr(args[2].pdata);
    Stager st(t);
    void *dst = st.out(args[0].pdata, (size_t)szof * len);
    const void *src = st.in(args[1].pdata, args[1].dataSz);
    const uint64_t src_rows = args[1].dataSz / (uint64_t)szof;
    const uint64_t snull_bits = args[1].pnulls ? (args[1].nullCnt ? args[1].nullCnt : src_rows) : 0;
    const uint64_t *snulls = (const uint64_t *)st.in(args[1].pnulls, args[1].pnulls ? ((snull_bits + 63) / 64) * 8 : 0);
    const int64_t *sels = (const int64_t *)st.in(args[2].pdata, 8 * len);
    uint32_t *dnulls = (uint32_t *)st.out(args[0].pnulls, args[0].pnulls ? ((len + 63) / 64) * 8 : 0);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    int grid = num_sms() * 8;
    const uint64_t work = (len + kThreads - 1) / kThreads;
    if ((uint64_t)grid > work) grid = (int)work;
    cudaEventRecord(t.kev0, t.stream);
    switch (szof) {
    case 1: gather_kernel<uint8_t><<<grid, kThreads, 0, t.stream>>>((uint8_t *)dst, (const uint8_t *)src, sels, len, snulls, snull_bits, dnulls); break;
    case 2: gather_kernel<uint16_t><<<grid, kThreads, 0, t.stream>>>((uint16_t *)dst, (const uint16_t *)src, sels, len, snulls, snull_bits, dnulls); break;
    case 4: gather_kernel<uint32_t><<<grid, kThreads, 0, t.stream>>>((uint32_t *)dst, (const uint32_t *)src, sels, len, snulls, snull_bits, dnulls); break;
    case 8: gather_kernel<uint64_t><<<grid, kThreads, 0, t.stream>>>((uint64_t *)dst, (const uint64_t *)src, sels, len, snulls, snull_bits, dnulls); break;
    case 16: gather_kernel<Cell16><<<grid, kThreads, 0, t.stream>>>((Cell16 *)dst, (const Cell16 *)src, sels, len, snulls, snull_bits, dnulls); break;
    default: gather_kernel<Cell24><<<grid, kThreads, 0, t.stream>>>((Cell24 *)dst, (const Cell24 *)src, sels, len, snulls, snull_bits, dnulls); break;
    }
    cudaEventRecord(t.kev1, t.stream);
    MOB_LAUNCH_CHECK();
    if (dev) { st.release_async(); return MO_RC_SUCCESS; }
    return st.finish();
}

// MO_XCALL_PACK_KEYS: args [0] keys uint64[len] (+ pnulls out: rows that join no group, has_null = 0 only) ; [1] params {int32 ncols, int32 has_null} ;
// [2 .. 2+ncols) fixed-width key columns (element size = dataSz / len, or a const vector), + pnulls
int xcall_pack_keys(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    int32_t prm[2] = {0, 1};
    if (!args[1].pdata || args[1].dataSz < 4 || is_device_ptr(args[1].pdata)) { set_error("pack keys: host params {ncols, has_null} missing"); return MO_RC_INVALID_ARGUMENT; }
    memcpy(prm, args[1].pdata, args[1].dataSz >= 8 ? 8 : 4);
    if (prm[0] < 1 || prm[0] > kMaxKeyCols || args[0].dataSz < 8 * len) { set_error("pack keys: 1..%d key columns, keys buffer of 8*len bytes", kMaxKeyCols); return MO_RC_INVALID_ARGUMENT; }
    if (len == 0) return MO_RC_SUCCESS;
    Stager st(t);
    KeyCols K; K.n = prm[0];
    int total = 0;
    for (int k = 0; k < K.n; k++) {
        const mo_xcall_args_t &a = args[2 + k];
        int sz = (int)(a.dataSz / len);
        const bool cst = a.dataSz < len || (a.dataSz <= 8 && len > 8);   // a const vector holds one element
        if (cst) sz = (int)a.dataSz;
        if (sz != 1 && sz != 2 && sz != 4 && sz != 8) { st.finish(); set_error("pack keys: column %d element size %d", k, sz); return MO_RC_INVALID_ARGUMENT; }
        K.size[k] = sz; K.cst[k] = cst ? 1 : 0;
        K.col[k] = (const uint8_t *)st.in(a.pdata, cst ? (size_t)sz : (size_t)sz * len);
        K.nulls[k] = (const uint64_t *)st.in(a.pnulls, a.pnulls ? (cst ? 8 : ((len + 63) / 64) * 8) : 0);
        total += sz + (prm[1] ? 1 : 0);
    }
    if (total > 8) { st.finish(); set_error("pack keys: %d key bytes exceed the 8-byte IntHashMap key (group/exec2.go:73-118)", total); return MO_RC_INVALID_ARGUMENT; }
    uint64_t *keys = (uint64_t *)st.out(args[0].pdata, 8 * len);
    uint32_t *skip = (uint32_t *)st.out(args[0].pnulls, args[0].pnulls ? ((len + 63) / 64) * 8 : 0);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    int grid = num_sms() * 8;
    const uint64_t work = (len + kThreads - 1) / kThreads;
    if ((uint64_t)grid > work) grid = (int)work;
    pack_keys_kernel<<<grid, kThreads, 0, t.stream>>>(keys, skip, len, K, prm[1]);
    MOB_LAUNCH_CHECK();
    return st.finish();
}

// MO_XCALL_GROUP_IDS: args [0] groups uint64[len] ; [1] state: pdata -> int64 ngroups (in/out) ; [2] table_keys uint64[cap] (in: the keys of the
// existing groups by id, out: + the new groups) ; [3] keys uint64[len] (+pnulls: rows that get id 0) ; optional [4] params {int64 expected_groups}
int xcall_group_ids(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!args[1].pdata || args[1].dataSz < 8 || args[0].dataSz < 8 * len || args[3].dataSz < 8 * len) { set_error("group ids: buffers too small"); return MO_RC_INVALID_ARGUMENT; }
    int64_t nexist = 0;
    if (is_device_ptr(args[1].pdata)) { int rc = read_back(t, &nexist, args[1].pdata, 8); if (rc) return rc; } else memcpy(&nexist, args[1].pdata, 8);
    const uint64_t table_cap = args[2].dataSz / 8;
    if (nexist < 0 || (uint64_t)nexist > table_cap) { set_error("group ids: ngroups %lld exceeds the key table (%llu)", (long long)nexist, (unsigned long long)table_cap); return MO_RC_INVALID_ARGUMENT; }
    const uint64_t total = len + (uint64_t)nexist;
    if (total >= 0x7fffffffull) { set_error("group ids: at most 2^31 rows per call"); return MO_RC_INVALID_ARGUMENT; }
    uint64_t want = total < table_cap ? total : table_cap;   // distinct keys <= min(rows, key table): the caller bounds the scratch through the table size
    if (want < 16) want = 16;
    uint64_t cap = 32;
    while (cap < 2 * want) cap <<= 1;
    Stager st(t);
    uint64_t *groups = (uint64_t *)st.out(args[0].pdata, 8 * len);
    uint64_t *table_keys = (uint64_t *)st.out(args[2].pdata, table_cap * 8, true);
    const uint64_t *keys = (const uint64_t *)st.in(args[3].pdata, 8 * len);
    const uint64_t *knulls = (const uint64_t *)st.in(args[3].pnulls, args[3].pnulls ? ((len + 63) / 64) * 8 : 0);
    int64_t *dng = (int64_t *)st.out(args[1].pdata, 8);
    GidTable T;
    T.key = (uint64_t *)st.tmp((cap + 1) * 8); T.minrow = (unsigned long long *)st.tmp((cap + 1) * 8); T.id = (uint64_t *)st.tmp((cap + 1) * 8);
    T.mask = cap - 1;
    uint32_t *rowslot = (uint32_t *)st.tmp(total * 4 + 16);
    uint8_t *isfirst = (uint8_t *)st.tmp(total + 16);
    uint32_t *firsts = (uint32_t *)st.tmp(total * 4 + 16);
    unsigned long long *dcount = (unsigned long long *)st.tmp(16);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    unsigned *overflow = (unsigned *)(dcount + 1);
    MOB_CUDA_TRY(cudaMemsetAsync(dcount, 0, 16, t.stream));
    auto grid_for = [&](uint64_t items) { uint64_t g = (items + kThreads - 1) / kThreads; uint64_t mx = (uint64_t)num_sms() * 8; return (unsigned)(g > mx ? mx : (g ? g : 1)); };
    gid_init_kernel<<<grid_for(cap + 1), kThreads, 0, t.stream>>>(T);
    MOB_LAUNCH_CHECK();
    cudaEventRecord(t.kev0, t.stream);
    gid_insert_kernel<<<grid_for(total), kThreads, 0, t.stream>>>(keys, knulls, len, table_keys, (uint64_t)nexist, T, rowslot, overflow);
    cudaEventRecord(t.kev1, t.stream);
    MOB_LAUNCH_CHECK();
    gid_flag_kernel<<<grid_for(total), kThreads, 0, t.stream>>>(total, T, rowslot, isfirst);
    MOB_LAUNCH_CHECK();
    int rc = launch_select<uint32_t>(t, isfirst, nullptr, total, firsts, dcount);
    if (rc) { st.finish(); return rc; }
    gid_assign_kernel<<<grid_for(total < 1 ? 1 : (total < (1u << 20) ? total : (1u << 20))), kThreads, 0, t.stream>>>(firsts, dcount, T, rowslot, table_keys, table_cap, (uint64_t)nexist, dng, overflow);
    MOB_LAUNCH_CHECK();
    gid_emit_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(groups, len, (uint64_t)nexist, T, rowslot);
    MOB_LAUNCH_CHECK();
    unsigned hov = 0;
    rc = read_back(t, &hov, overflow, 4);
    int frc = st.finish();
    if (rc) return rc;
    if (hov) { set_error("group ids: more distinct keys than the key table holds (%llu)", (unsigned long long)table_cap); return MO_RC_INVALID_ARGUMENT; }
    return frc;
}

// MO_XCALL_GROUP_AGG(op, T): args [0] state: 8 bytes per group (+pnulls: group is NULL, in/out) ; [1] counts int64 per group (AVG: required;
// others: optional) ; [2] groups uint64[len] (1-based, 0 = skip) ; [3] the column (+pnulls).  len = rows.
int xcall_group_agg(int op, int T, mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    const int sz = type_size(T);
    if (!sz) { set_error("group agg: unsupported type %d", T); return MO_RC_INVALID_ARGUMENT; }
    if (args[2].dataSz < 8 * len || (op != MO_AGG_COUNT && args[3].dataSz < (uint64_t)sz * len)) { set_error("group agg: groups / column shorter than len"); return MO_RC_INVALID_ARGUMENT; }
    if (op == MO_AGG_AVG && !args[1].pdata) { set_error("group agg: AVG needs the counts vector"); return MO_RC_INVALID_ARGUMENT; }
    if (args[1].pdata && args[1].dataSz < args[0].dataSz) { set_error("group agg: counts shorter than the state"); return MO_RC_INVALID_ARGUMENT; }
    const bool is_signed = T >= MO_T_INT8 && T <= MO_T_INT64, is_unsigned = T >= MO_T_UINT8 && T <= MO_T_UINT64;
    const int is_avg = op == MO_AGG_AVG;
    switch (op) {
    case MO_AGG_COUNT: return run_group_agg<uint8_t, G_COUNT>(t, args, len, 0);
    case MO_AGG_MIN: return dispatch_minmax<G_MIN_INT, G_MIN_UINT, G_MIN_FLT>(t, T, args, len);
    case MO_AGG_MAX: return dispatch_minmax<G_MAX_INT, G_MAX_UINT, G_MAX_FLT>(t, T, args, len);
    case MO_AGG_SUM: case MO_AGG_AVG:
        if (is_signed) switch (sz) {
            case 1: return run_group_agg<int8_t, G_SUM_SIGNED>(t, args, len, is_avg);
            case 2: return run_group_agg<int16_t, G_SUM_SIGNED>(t, args, len, is_avg);
            case 4: return run_group_agg<int32_t, G_SUM_SIGNED>(t, args, len, is_avg);
            default: return run_group_agg<int64_t, G_SUM_SIGNED>(t, args, len, is_avg);
        }
        if (is_unsigned) switch (sz) {
            case 1: return run_group_agg<uint8_t, G_SUM_UNSIGNED>(t, args, len, is_avg);
            case 2: return run_group_agg<uint16_t, G_SUM_UNSIGNED>(t, args, len, is_avg);
            case 4: return run_group_agg<uint32_t, G_SUM_UNSIGNED>(t, args, len, is_avg);
            default: return run_group_agg<uint64_t, G_SUM_UNSIGNED>(t, args, len, is_avg);
        }
        if (T == MO_T_FLOAT32) return run_group_agg<float, G_SUM_FLOAT>(t, args, len, is_avg);
        if (T == MO_T_FLOAT64) return run_group_agg<double, G_SUM_FLOAT>(t, args, len, is_avg);
    }
    set_error("group agg: operator %d is not defined for type %d", op, T);
    return MO_RC_INVALID_ARGUMENT;
}

}  // namespace mob
