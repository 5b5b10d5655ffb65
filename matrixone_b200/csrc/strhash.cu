// strhash.cu -- the reference's StrHashMap path behind XCall: group-by and hash join on keys wider than 8 bytes (any varchar / char key, any
// composite key over 8 bytes, group/exec2.go:73-94,167-188 and hashbuild/hashmap.go:258-277).
//
//   MO_XCALL_PACK_STR_KEYS   strHashmapIterator.encodeHashKeys (pkg/common/hashmap/strhashmap.go:92-385): the exact key bytes, padding included.
//                            Row lengths -> exclusive scan -> write; short rows are written by their own thread, long rows by their whole warp.
//   MO_XCALL_STR_GROUP_IDS   strHashmapIterator.Insert (string_hash_map.go:97-158) as Group.buildOneBatch drives it: 1-based ids in first-seen
//                            order.  "Virtual rows" exactly like gid_* in colops.cu: v < nexist is existing group v (its key from the table),
//                            v >= nexist is batch row v - nexist; every distinct key keeps its smallest virtual row and an order-preserving
//                            compaction of those first rows ranks them, so the ids do not depend on the hash or on scheduling.
//   MO_XCALL_STR_JOIN_FIND   strHashmapIterator.Find.
//   MO_XCALL_STR_JOIN_PROBE  JOIN_PROBE with string keys: only the lookup is new, the scan and the emission are join.cu's (hashops.cuh).
// Matching is exact: a 64-bit hash picks the slot and 32 of its bits are kept in the slot as a filter, but two keys are one group only when
// their bytes are equal.  The reference compares 192-bit AES hash states; the ids it hands out are the same.
// Algorithmic bytes per row: the key columns once and the packed key twice (write, then read by insert / find) + 8 per offset + 8 per id.
#include "hashops.cuh"
#include <cstring>
#include <mutex>
#include <shared_mutex>
#include <unordered_map>

namespace mob {

namespace {

constexpr int kThreads = 256;
constexpr int kMaxCols = MO_STR_KEY_MAX_COLS;
constexpr uint64_t kPadTo = 16;           // hashtable.StrKeyPadding: shorter keys are zero-padded to 16 bytes
constexpr uint64_t kWarpRow = 64;         // packed rows longer than this are written by their whole warp
constexpr uint32_t kNoSlot = 0xffffffffu;
constexpr uint64_t kMaxRows = 1ull << 30; // virtual rows per call: slot indices and row ids stay below 2^31

__device__ __forceinline__ uint64_t mix64(uint64_t x) { x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; return x ^ (x >> 33); }

__device__ __forceinline__ uint64_t ld64u(const uint8_t *p) {   // unaligned little-endian load
    uint64_t w = 0;
#pragma unroll
    for (int b = 0; b < 8; b++) w |= (uint64_t)p[b] << (8 * b);
    return w;
}

// slot choice only: equality is decided by the bytes
__device__ __forceinline__ uint64_t key_hash(const uint8_t *p, uint64_t n) {
    uint64_t h = 0x9e3779b97f4a7c15ull ^ n;
    uint64_t j = 0;
    for (; j + 8 <= n; j += 8) {
        const uint64_t x = h ^ mix64(ld64u(p + j));
        h = ((x << 27) | (x >> 37)) * 0x9e3779b97f4a7c15ull + 0x52dce729ull;
    }
    uint64_t w = 0;
    for (int b = 0; j < n; j++, b++) w |= (uint64_t)p[j] << (8 * b);
    return mix64(h ^ mix64(w ^ 0x27d4eb2f165667c5ull));
}

__device__ __forceinline__ bool key_eq(const uint8_t *a, uint64_t an, const uint8_t *b, uint64_t bn) {
    if (an != bn) return false;
    for (uint64_t j = 0; j < an; j++) if (a[j] != b[j]) return false;
    return true;
}

// key i of a packed key set (offsets + bytes); false for offsets that are not increasing or leave the bytes
struct Packed { const int64_t *off; const uint8_t *bytes; uint64_t nbytes; };
__device__ __forceinline__ bool packed_key(const Packed &K, uint64_t i, const uint8_t **p, uint64_t *n) {
    const int64_t o0 = K.off[i], o1 = K.off[i + 1];
    if (o0 < 0 || o1 < o0 || (uint64_t)o1 > K.nbytes) return false;
    *p = K.bytes + o0; *n = (uint64_t)(o1 - o0);
    return true;
}

// =========================================================================================================
// PACK_STR_KEYS
// =========================================================================================================
struct StrCols {
    const uint8_t *col[kMaxCols]; const uint64_t *nulls[kMaxCols]; const uint8_t *area[kMaxCols]; uint64_t area_len[kMaxCols];
    int width[kMaxCols]; int cst[kMaxCols]; int n; int has_null;
};

// what column k appends for row i: hdr_len header bytes (marker / uint16 length, little-endian in hdr), then the n value bytes at p
struct Piece { const uint8_t *p; uint64_t n; uint32_t hdr; int hdr_len; bool skip; bool bad; };

__device__ __forceinline__ Piece piece_of(const StrCols &K, int k, uint64_t i) {
    Piece c; c.p = nullptr; c.n = 0; c.hdr = 0; c.hdr_len = 0; c.skip = false; c.bad = false;
    const uint64_t r = K.cst[k] ? 0 : i;
    if (bm_test(K.nulls[k], r)) {                                   // marker 1 (hasNull) or zValues[i] = 0 (strhashmap.go:164-176,318-330)
        if (K.has_null) { c.hdr = 1; c.hdr_len = 1; } else c.skip = true;
        return c;
    }
    if (K.width[k]) {                                               // fillGroupStr: [marker 0] + TypeSize() bytes
        c.p = K.col[k] + r * (uint64_t)K.width[k]; c.n = (uint64_t)K.width[k];
        c.hdr_len = K.has_null ? 1 : 0;
    } else {                                                        // fillStringGroupStr: [marker 0] + uint16(len) + bytes
        if (!varlena_bytes(K.col[k] + r * MO_VARLENA_SZ, K.area[k], K.area_len[k], &c.p, &c.n)) { c.bad = true; c.n = 0; }
        const uint32_t l16 = (uint32_t)(c.n & 0xffffu);            // the length field wraps, the bytes do not
        if (K.has_null) { c.hdr = l16 << 8; c.hdr_len = 3; } else { c.hdr = l16; c.hdr_len = 2; }
    }
    return c;
}

__global__ void __launch_bounds__(kThreads) sk_len_kernel(StrCols K, uint64_t n, uint64_t *__restrict__ len, uint32_t *__restrict__ skip32, unsigned *bad) {
    const uint64_t n64 = (n + 63) & ~63ull;
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n64; i += (uint64_t)gridDim.x * kThreads) {
        bool skip = false;
        if (i < n) {
            uint64_t L = 0;
            for (int k = 0; k < K.n; k++) {
                const Piece c = piece_of(K, k, i);
                if (c.bad) *bad = 1;
                skip |= c.skip;
                L += (uint64_t)c.hdr_len + c.n;
            }
            len[i] = L < kPadTo ? kPadTo : L;
        }
        if (skip32) {
            const unsigned m = __ballot_sync(0xffffffffu, skip);
            if ((threadIdx.x & 31) == 0) skip32[i >> 5] = m;
        }
    }
}

// row i's packed key into dst[0 .. L): by one thread (lane 0, step 1) or by a whole warp (lane, step 32)
__device__ __forceinline__ void write_row(const StrCols &K, uint64_t i, uint8_t *dst, uint64_t L, unsigned lane, unsigned step) {
    uint64_t o = 0;
    for (int k = 0; k < K.n; k++) {
        const Piece c = piece_of(K, k, i);
        if (c.skip || c.bad) continue;
        for (int b = (int)lane; b < c.hdr_len; b += (int)step) dst[o + b] = (uint8_t)(c.hdr >> (8 * b));
        o += (uint64_t)c.hdr_len;
        for (uint64_t j = lane; j < c.n; j += step) dst[o + j] = c.p[j];
        o += c.n;
    }
    for (uint64_t j = o + lane; j < L; j += step) dst[j] = 0;   // StrKeyPadding
}

__global__ void __launch_bounds__(kThreads) sk_write_kernel(StrCols K, uint64_t n, const int64_t *__restrict__ off, uint8_t *__restrict__ bytes) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t nrounds = (n + 31) / 32;
    for (uint64_t w = (blockIdx.x * (uint64_t)kThreads + threadIdx.x) >> 5; w < nrounds; w += ((uint64_t)gridDim.x * kThreads) >> 5) {
        const uint64_t i = w * 32 + lane;
        uint64_t o = 0, L = 0;
        if (i < n) { o = (uint64_t)off[i]; L = (uint64_t)off[i + 1] - o; }
        if (i < n && L <= kWarpRow) write_row(K, i, bytes + o, L, 0, 1);
        unsigned heavy = __ballot_sync(0xffffffffu, i < n && L > kWarpRow);
        while (heavy) {                                   // long keys: the whole warp copies, coalesced
            const int src = __ffs(heavy) - 1; heavy &= heavy - 1;
            const uint64_t hi = __shfl_sync(0xffffffffu, i, src), ho = __shfl_sync(0xffffffffu, o, src), hL = __shfl_sync(0xffffffffu, L, src);
            write_row(K, hi, bytes + ho, hL, lane, 32);
        }
    }
}

// =========================================================================================================
// STR_GROUP_IDS
// =========================================================================================================
// a slot holds (upper 32 hash bits << 32) | (virtual row + 1) of the key that claimed it; 0 = empty
struct VKeys { Packed table; uint64_t nexist; Packed batch; const uint64_t *skip; };

__device__ __forceinline__ bool vkey(const VKeys &V, uint64_t v, const uint8_t **p, uint64_t *n) {
    return v < V.nexist ? packed_key(V.table, v, p, n) : packed_key(V.batch, v - V.nexist, p, n);
}

__global__ void __launch_bounds__(kThreads) sg_insert_kernel(VKeys V, uint64_t total, unsigned long long *slot, unsigned *minrow, uint64_t mask,
                                                             uint32_t *__restrict__ rowslot, unsigned *bad) {
    for (uint64_t v = blockIdx.x * (uint64_t)kThreads + threadIdx.x; v < total; v += (uint64_t)gridDim.x * kThreads) {
        const uint8_t *p; uint64_t n;
        if (v >= V.nexist && bm_test(V.skip, v - V.nexist)) { rowslot[v] = kNoSlot; continue; }   // InsertStringBatchWithRing skips zValues == 0
        if (!vkey(V, v, &p, &n)) { *bad = 1; rowslot[v] = kNoSlot; continue; }
        const uint64_t h = key_hash(p, n);
        const unsigned long long tag = h & 0xffffffff00000000ull;
        uint64_t s = h & mask;
        for (;;) {                                        // at least half the slots stay empty: the probe ends
            unsigned long long cur = *((volatile unsigned long long *)&slot[s]);
            if (cur == 0) {
                cur = atomicCAS(&slot[s], 0ull, tag | (v + 1));
                if (cur == 0) break;
            }
            if ((cur & 0xffffffff00000000ull) == tag) {
                const uint8_t *q; uint64_t qn;
                if (vkey(V, (cur & 0xffffffffull) - 1, &q, &qn) && key_eq(p, n, q, qn)) break;
            }
            s = (s + 1) & mask;
        }
        if (*((volatile unsigned *)&minrow[s]) > (unsigned)v) atomicMin(&minrow[s], (unsigned)v);   // monotone: see gid_insert_kernel
        rowslot[v] = (uint32_t)s;
    }
}

__global__ void __launch_bounds__(kThreads) sg_flag_kernel(uint64_t total, const unsigned *__restrict__ minrow, const uint32_t *__restrict__ rowslot, uint8_t *__restrict__ isfirst) {
    for (uint64_t v = blockIdx.x * (uint64_t)kThreads + threadIdx.x; v < total; v += (uint64_t)gridDim.x * kThreads) {
        const uint32_t s = rowslot[v];
        isfirst[v] = (s != kNoSlot && minrow[s] == (unsigned)v) ? 1 : 0;
    }
}

// key length of every new group (rank j >= nexist), 0 past the group count
__global__ void __launch_bounds__(kThreads) sg_newlen_kernel(VKeys V, const uint32_t *__restrict__ firsts, const unsigned long long *count, uint64_t maxnew, uint64_t *__restrict__ nlen) {
    const uint64_t cnt = *count;
    for (uint64_t j = blockIdx.x * (uint64_t)kThreads + threadIdx.x; j < maxnew; j += (uint64_t)gridDim.x * kThreads) {
        const uint64_t g = V.nexist + j;
        uint64_t n = 0;
        if (g < cnt) { const uint8_t *p; vkey(V, firsts[g], &p, &n); }
        nlen[j] = n;
    }
}

// state = {ngroups, bytes used, groups needed, bytes needed}: the table only grows when everything fits
__global__ void sg_decide_kernel(const unsigned long long *count, const uint64_t *newbytes, uint64_t cap, uint64_t byte_cap, uint64_t nexist,
                                 int64_t *state, int64_t *toff, unsigned *ok, const unsigned *bad) {
    const uint64_t cnt = *count, used = (uint64_t)state[1], need = used + *newbytes;
    state[2] = (int64_t)cnt; state[3] = (int64_t)need;
    const bool fits = cnt <= cap && need <= byte_cap && !*bad;   // (broken key offsets fail the call: nothing is appended)
    *ok = fits ? 1u : 0u;
    if (fits) { state[0] = (int64_t)cnt; state[1] = (int64_t)need; toff[nexist] = (int64_t)used; }
}

// one warp per group rank j: id of its slot (minrow is reused as the id array), and for a new group its key appended to the table
__global__ void __launch_bounds__(kThreads) sg_assign_kernel(VKeys V, const uint32_t *__restrict__ firsts, const unsigned long long *count, const uint32_t *__restrict__ rowslot,
                                                             unsigned *id, const uint64_t *__restrict__ pos, uint64_t used, const unsigned *ok, int64_t *toff, uint8_t *tbytes) {
    const uint64_t cnt = *count;
    const bool append = *ok != 0;
    const unsigned lane = threadIdx.x & 31;
    for (uint64_t j = (blockIdx.x * (uint64_t)kThreads + threadIdx.x) >> 5; j < cnt; j += ((uint64_t)gridDim.x * kThreads) >> 5) {
        const uint32_t v = firsts[j];
        if (lane == 0) id[rowslot[v]] = (unsigned)(j + 1);
        if (!append || j < V.nexist) continue;
        const uint8_t *p; uint64_t n;
        vkey(V, v, &p, &n);
        const uint64_t o = used + pos[j - V.nexist];
        for (uint64_t b = lane; b < n; b += 32) tbytes[o + b] = p[b];
        if (lane == 0) toff[j + 1] = (int64_t)(o + n);
    }
}

__global__ void __launch_bounds__(kThreads) sg_emit_kernel(uint64_t *__restrict__ groups, uint64_t n, uint64_t nexist, const unsigned *__restrict__ id, const uint32_t *__restrict__ rowslot, const unsigned *ok) {
    const bool fits = *ok != 0;
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        const uint32_t s = rowslot[nexist + i];
        groups[i] = (!fits || s == kNoSlot) ? 0ull : (uint64_t)id[s];
    }
}

// =========================================================================================================
// the probe-side table of a string-keyed JoinMap
// =========================================================================================================
struct StrTable { unsigned long long *slot; uint64_t mask; Packed keys; uint64_t ngroups; };

__global__ void __launch_bounds__(kThreads) st_init_kernel(unsigned long long *slot, uint64_t slots) {
    for (uint64_t s = blockIdx.x * (uint64_t)kThreads + threadIdx.x; s < slots; s += (uint64_t)gridDim.x * kThreads) slot[s] = 0;
}
__global__ void __launch_bounds__(kThreads) st_build_kernel(StrTable T, unsigned *bad) {
    for (uint64_t g = blockIdx.x * (uint64_t)kThreads + threadIdx.x; g < T.ngroups; g += (uint64_t)gridDim.x * kThreads) {
        const uint8_t *p; uint64_t n;
        if (!packed_key(T.keys, g, &p, &n)) { *bad = 1; continue; }
        const uint64_t h = key_hash(p, n);
        uint64_t s = h & T.mask;
        for (;;) {                                        // the key table of STR_GROUP_IDS holds distinct keys: one writer per slot
            if (atomicCAS(&T.slot[s], 0ull, (h & 0xffffffff00000000ull) | (g + 1)) == 0) break;
            s = (s + 1) & T.mask;
        }
    }
}
__device__ __forceinline__ uint32_t st_find(const StrTable &T, const uint8_t *p, uint64_t n) {
    const uint64_t h = key_hash(p, n);
    const unsigned long long tag = h & 0xffffffff00000000ull;
    uint64_t s = h & T.mask;
    for (;;) {
        const unsigned long long cur = T.slot[s];
        if (cur == 0) return 0;
        if ((cur & 0xffffffff00000000ull) == tag) {
            const uint8_t *q; uint64_t qn;
            const uint32_t g1 = (uint32_t)(cur & 0xffffffffull);
            if (packed_key(T.keys, g1 - 1, &q, &qn) && key_eq(p, n, q, qn)) return g1;
        }
        s = (s + 1) & T.mask;
    }
}
// id of probe row i (0: skipped / NULL, absent, or offsets outside the bytes)
__device__ __forceinline__ uint32_t probe_id(const StrTable &T, const Packed &K, const uint64_t *skip, uint64_t i, unsigned *bad) {
    if (bm_test(skip, i)) return 0;
    const uint8_t *p; uint64_t n;
    if (!packed_key(K, i, &p, &n)) { *bad = 1; return 0; }
    return st_find(T, p, n);
}
__global__ void __launch_bounds__(kThreads) st_find_kernel(StrTable T, Packed K, const uint64_t *__restrict__ skip, uint64_t n, uint64_t *__restrict__ vals, unsigned *bad) {
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) vals[i] = probe_id(T, K, skip, i, bad);
}
__global__ void __launch_bounds__(kThreads) st_probe_count_kernel(StrTable T, Packed K, const uint64_t *__restrict__ skip, uint64_t n, const int32_t *__restrict__ offsets,
                                                                  int join_type, uint32_t *__restrict__ vals, uint64_t *__restrict__ cnt, unsigned *bad) {
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        uint32_t v = probe_id(T, K, skip, i, bad);
        cnt[i] = probe_row_count(&v, offsets, join_type);
        vals[i] = v;
    }
}

struct StrDevTable { unsigned long long *slot = nullptr; int64_t *off = nullptr; uint8_t *bytes = nullptr; uint64_t nbytes = 0, mask = 0, ngroups = 0; };
std::shared_mutex g_sjm_mu;
std::unordered_map<const void *, StrDevTable> g_sjm;   // prepared string join maps, by key offsets pointer

StrTable view_of(const StrDevTable &D) { return StrTable{D.slot, D.mask, Packed{D.off, D.bytes, D.nbytes}, D.ngroups}; }

void free_table(StrDevTable &D) { if (D.slot) cudaFree(D.slot); if (D.off) cudaFree(D.off); if (D.bytes) cudaFree(D.bytes); D = StrDevTable(); }

// hash table over ngroups keys (device offsets + bytes) in the arena or, persistent, in its own allocation; *bad (device) flags broken offsets
int build_str_table(ThreadCtx &t, const int64_t *doff, const uint8_t *dbytes, uint64_t nbytes, uint64_t ngroups, bool persistent, unsigned *bad, StrDevTable *out) {
    uint64_t slots = 64;
    while (slots < 2 * ngroups) slots <<= 1;
    StrDevTable D;
    D.mask = slots - 1; D.ngroups = ngroups; D.nbytes = nbytes;
    if (persistent) {
        if (cudaMalloc(&D.slot, slots * 8) != cudaSuccess || cudaMalloc(&D.off, (ngroups + 1) * 8) != cudaSuccess || cudaMalloc(&D.bytes, nbytes ? nbytes : 1) != cudaSuccess) {
            set_error("string join map: cudaMalloc of a %llu-slot table failed", (unsigned long long)slots);
            free_table(D);
            return MO_RC_INTERNAL_ERROR;
        }
        MOB_CUDA_TRY(cudaMemcpyAsync(D.off, doff, (ngroups + 1) * 8, cudaMemcpyDeviceToDevice, t.stream));
        if (nbytes) MOB_CUDA_TRY(cudaMemcpyAsync(D.bytes, dbytes, nbytes, cudaMemcpyDeviceToDevice, t.stream));
    } else {
        D.slot = (unsigned long long *)arena_alloc(t, slots * 8);
        if (!D.slot) return MO_RC_INTERNAL_ERROR;
        D.off = const_cast<int64_t *>(doff); D.bytes = const_cast<uint8_t *>(dbytes);
    }
    st_init_kernel<<<grid_for(slots), kThreads, 0, t.stream>>>(D.slot, slots);
    MOB_LAUNCH_CHECK();
    if (ngroups) {
        st_build_kernel<<<grid_for(ngroups), kThreads, 0, t.stream>>>(view_of(D), bad);
        MOB_LAUNCH_CHECK();
    }
    *out = D;
    return MO_RC_SUCCESS;
}

uint64_t groups_of(const mo_xcall_args_t &offs) { return offs.dataSz >= 8 ? offs.dataSz / 8 - 1 : 0; }

// the table for this call: the prepared one (by the caller's offsets pointer) or a scratch one in the arena
int str_table_for(ThreadCtx &t, Stager &st, const mo_xcall_args_t &offs, const mo_xcall_args_t &bytes, unsigned *bad, StrTable *T,
                  std::shared_lock<std::shared_mutex> &lk) {
    const uint64_t ngroups = groups_of(offs);
    if (ngroups >= kMaxRows) { set_error("string join: at most 2^30 groups"); return MO_RC_INVALID_ARGUMENT; }
    lk = std::shared_lock<std::shared_mutex>(g_sjm_mu);
    auto it = g_sjm.find(offs.pdata);
    if (it != g_sjm.end() && it->second.ngroups == ngroups) { *T = view_of(it->second); return MO_RC_SUCCESS; }
    lk.unlock();
    const int64_t *doff = ngroups ? (const int64_t *)st.in(offs.pdata, (ngroups + 1) * 8) : nullptr;
    const uint8_t *dbytes = (const uint8_t *)st.in(bytes.pdata, bytes.pdata ? bytes.dataSz : 0);
    if (st.failed) return MO_RC_INTERNAL_ERROR;
    StrDevTable D;
    int rc = build_str_table(t, doff, dbytes, bytes.pdata ? bytes.dataSz : 0, ngroups, false, bad, &D);
    if (rc) return rc;
    *T = view_of(D);
    return MO_RC_SUCCESS;
}

int check_bad(ThreadCtx &t, const unsigned *bad, const char *what) {
    unsigned hb = 0;
    int rc = read_back(t, &hb, bad, 4);
    if (rc) return rc;
    if (hb) { set_error("%s", what); return MO_RC_INVALID_ARGUMENT; }
    return MO_RC_SUCCESS;
}

}  // namespace

// MO_XCALL_PACK_STR_KEYS: args [0] offsets int64[len + 1] (+pnulls out: skipped rows) ; [1] key bytes (capacity = dataSz) ; [2] host mo_str_key_params_t ;
// [3 .. 3 + ncols) key columns (+pnulls; width 0 = varlena cells + parea; a const vector holds one element)
int xcall_pack_str_keys(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!args[2].pdata || args[2].dataSz < 8 || is_device_ptr(args[2].pdata)) { set_error("pack str keys: host mo_str_key_params_t missing"); return MO_RC_INVALID_ARGUMENT; }
    mo_str_key_params_t P;
    memset(&P, 0, sizeof P);
    memcpy(&P, args[2].pdata, args[2].dataSz < sizeof P ? args[2].dataSz : sizeof P);
    if (P.ncols < 1 || P.ncols > kMaxCols || args[2].dataSz < 8 + 4 * (uint64_t)P.ncols) { set_error("pack str keys: 1..%d key columns, one width each", kMaxCols); return MO_RC_INVALID_ARGUMENT; }
    if (!args[0].pdata || args[0].dataSz < 8 * (len + 1)) { set_error("pack str keys: offsets need len + 1 entries"); return MO_RC_INVALID_ARGUMENT; }
    Stager st(t);
    StrCols K;
    memset(&K, 0, sizeof K);
    K.n = P.ncols; K.has_null = P.has_null ? 1 : 0;
    for (int k = 0; k < K.n; k++) {
        const mo_xcall_args_t &a = args[3 + k];
        const int w = P.width[k];
        const uint64_t esz = w > 0 ? (uint64_t)w : (uint64_t)MO_VARLENA_SZ;
        if (w < 0) { st.finish(); set_error("pack str keys: column %d width %d", k, w); return MO_RC_INVALID_ARGUMENT; }
        bool cst;
        if (a.dataSz >= esz * len) cst = false;
        else if (a.dataSz >= esz) cst = true;                 // a const vector holds one element
        else { st.finish(); set_error("pack str keys: column %d holds %llu bytes, %llu rows of %llu", k, (unsigned long long)a.dataSz, (unsigned long long)len, (unsigned long long)esz); return MO_RC_INVALID_ARGUMENT; }
        K.width[k] = w; K.cst[k] = cst ? 1 : 0;
        const uint64_t rows = cst ? 1 : len;
        K.col[k] = (const uint8_t *)st.in(a.pdata, rows ? esz * rows : 0);
        K.nulls[k] = (const uint64_t *)st.in(a.pnulls, a.pnulls && rows ? ((rows + 63) / 64) * 8 : 0);
        if (!w) { K.area[k] = (const uint8_t *)st.in(a.parea, a.parea ? a.areaSz : 0); K.area_len[k] = a.parea ? a.areaSz : 0; }
    }
    int64_t *offs = (int64_t *)st.out(args[0].pdata, 8 * (len + 1));
    uint32_t *skip = (uint32_t *)st.out(args[0].pnulls, args[0].pnulls && len ? ((len + 63) / 64) * 8 : 0);
    unsigned *bad = (unsigned *)st.tmp(16);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    MOB_CUDA_TRY(cudaMemsetAsync(bad, 0, 16, t.stream));
    cudaEventRecord(t.kev0, t.stream);
    sk_len_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(K, len, (uint64_t *)offs, skip, bad);
    MOB_LAUNCH_CHECK();
    int rc = exclusive_scan(t, (const uint64_t *)offs, len, (uint64_t *)offs, (uint64_t *)offs + len);   // offsets[len] = bytes needed
    if (rc) { st.finish(); return rc; }
    rc = check_bad(t, bad, "pack str keys: a varlena cell points outside its area");
    if (rc) { st.finish(); return rc; }
    int64_t need = 0;
    rc = read_back(t, &need, offs + len, 8);
    if (rc) { st.finish(); return rc; }
    if ((uint64_t)need > args[1].dataSz) {
        int frc = st.finish();
        if (frc) return frc;
        set_error("pack str keys: %lld key bytes exceed the buffer (%llu); offsets[len] holds the size, call again with a larger buffer", (long long)need, (unsigned long long)args[1].dataSz);
        return MO_RC_OUT_OF_RANGE;
    }
    uint8_t *bytes = (uint8_t *)st.out(args[1].pdata, (size_t)need);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    if (len) {
        sk_write_kernel<<<grid_for(len), kThreads, 0, t.stream>>>(K, len, offs, bytes);
        MOB_LAUNCH_CHECK();
    }
    cudaEventRecord(t.kev1, t.stream);
    return st.finish();
}

// MO_XCALL_STR_GROUP_IDS: args [0] groups uint64[len] ; [1] state int64[4] ; [2] table offsets int64[cap + 1] ; [3] table bytes ; [4] packed key offsets
// int64[len + 1] (+pnulls: rows that get id 0) ; [5] packed key bytes
int xcall_str_group_ids(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!args[1].pdata || args[1].dataSz < 32 || args[0].dataSz < 8 * len || args[2].dataSz < 8 || args[4].dataSz < 8 * (len + 1)) { set_error("str group ids: buffers too small"); return MO_RC_INVALID_ARGUMENT; }
    int64_t hs[4] = {0, 0, 0, 0};
    if (is_device_ptr(args[1].pdata)) { int rc = read_back(t, hs, args[1].pdata, 16); if (rc) return rc; } else memcpy(hs, args[1].pdata, 16);
    const uint64_t cap = args[2].dataSz / 8 - 1, byte_cap = args[3].pdata ? args[3].dataSz : 0;
    if (hs[0] < 0 || (uint64_t)hs[0] > cap || hs[1] < 0 || (uint64_t)hs[1] > byte_cap) { set_error("str group ids: state {%lld groups, %lld bytes} exceeds the table (%llu, %llu)", (long long)hs[0], (long long)hs[1], (unsigned long long)cap, (unsigned long long)byte_cap); return MO_RC_INVALID_ARGUMENT; }
    const uint64_t nexist = (uint64_t)hs[0], used = (uint64_t)hs[1];
    const uint64_t total = len + nexist;
    if (total >= kMaxRows) { set_error("str group ids: at most 2^30 rows + groups per call"); return MO_RC_INVALID_ARGUMENT; }
    uint64_t slots = 64;
    while (slots < 2 * total) slots <<= 1;
    Stager st(t);
    uint64_t *groups = (uint64_t *)st.out(args[0].pdata, 8 * len);
    int64_t *state = (int64_t *)st.out(args[1].pdata, 32, true);
    int64_t *toff = (int64_t *)st.out(args[2].pdata, (cap + 1) * 8, true);
    uint8_t *tbytes = (uint8_t *)st.out(args[3].pdata, byte_cap, true);
    VKeys V;
    V.table = Packed{toff, tbytes, used};
    V.nexist = nexist;
    V.batch = Packed{(const int64_t *)st.in(args[4].pdata, 8 * (len + 1)), (const uint8_t *)st.in(args[5].pdata, args[5].pdata ? args[5].dataSz : 0), args[5].pdata ? args[5].dataSz : 0};
    V.skip = (const uint64_t *)st.in(args[4].pnulls, args[4].pnulls && len ? ((len + 63) / 64) * 8 : 0);
    unsigned long long *slot = (unsigned long long *)st.tmp(slots * 8);
    unsigned *minrow = (unsigned *)st.tmp(slots * 4);
    uint32_t *rowslot = (uint32_t *)st.tmp(total * 4 + 16);
    uint8_t *isfirst = (uint8_t *)st.tmp(total + 16);
    uint32_t *firsts = (uint32_t *)st.tmp(total * 4 + 16);
    uint64_t *nlen = (uint64_t *)st.tmp(len * 8 + 16);
    unsigned long long *scal = (unsigned long long *)st.tmp(32);   // [0] group count, [1] new key bytes, [2] ok | bad
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    unsigned *ok = (unsigned *)(scal + 2), *bad = ok + 1;
    MOB_CUDA_TRY(cudaMemsetAsync(scal, 0, 32, t.stream));
    MOB_CUDA_TRY(cudaMemsetAsync(slot, 0, slots * 8, t.stream));
    MOB_CUDA_TRY(cudaMemsetAsync(minrow, 0xff, slots * 4, t.stream));
    cudaEventRecord(t.kev0, t.stream);
    sg_insert_kernel<<<grid_for(total), kThreads, 0, t.stream>>>(V, total, slot, minrow, slots - 1, rowslot, bad);
    cudaEventRecord(t.kev1, t.stream);
    MOB_LAUNCH_CHECK();
    sg_flag_kernel<<<grid_for(total), kThreads, 0, t.stream>>>(total, minrow, rowslot, isfirst);
    MOB_LAUNCH_CHECK();
    int rc = launch_select<uint32_t>(t, isfirst, nullptr, total, firsts, scal);
    if (rc) { st.finish(); return rc; }
    sg_newlen_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(V, firsts, scal, len, nlen);
    MOB_LAUNCH_CHECK();
    rc = exclusive_scan(t, nlen, len, nlen, (uint64_t *)(scal + 1));
    if (rc) { st.finish(); return rc; }
    sg_decide_kernel<<<1, 1, 0, t.stream>>>(scal, (const uint64_t *)(scal + 1), cap, byte_cap, nexist, state, toff, ok, bad);
    MOB_LAUNCH_CHECK();
    sg_assign_kernel<<<grid_for(total * 32), kThreads, 0, t.stream>>>(V, firsts, scal, rowslot, minrow, nlen, used, ok, toff, tbytes);
    MOB_LAUNCH_CHECK();
    sg_emit_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(groups, len, nexist, minrow, rowslot, ok);
    MOB_LAUNCH_CHECK();
    unsigned flags[2] = {0, 0};
    rc = read_back(t, flags, ok, 8);
    int64_t need[4] = {0, 0, 0, 0};
    if (!rc) rc = read_back(t, need, state, 32);
    int frc = st.finish();
    if (rc) return rc;
    if (flags[1]) { set_error("str group ids: key offsets are not increasing or point past the key bytes"); return MO_RC_INVALID_ARGUMENT; }
    if (!flags[0]) {
        set_error("str group ids: %lld groups / %lld key bytes exceed the table (%llu groups, %llu bytes); the state holds the sizes, grow the table and call again",
                  (long long)need[2], (long long)need[3], (unsigned long long)cap, (unsigned long long)byte_cap);
        return MO_RC_OUT_OF_RANGE;
    }
    return frc;
}

// MO_XCALL_STR_JOIN_FIND: args [0] vals uint64[len] ; [1] table offsets int64[ngroups + 1] ; [2] table bytes ; [3] probe key offsets (+pnulls) ; [4] probe key bytes
int xcall_str_join_find(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (args[0].dataSz < 8 * len || args[3].dataSz < 8 * (len + 1)) { set_error("str join find: buffers too small"); return MO_RC_INVALID_ARGUMENT; }
    Stager st(t);
    unsigned *bad = (unsigned *)st.tmp(16);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    MOB_CUDA_TRY(cudaMemsetAsync(bad, 0, 16, t.stream));
    StrTable T;
    std::shared_lock<std::shared_mutex> lk;
    int rc = str_table_for(t, st, args[1], args[2], bad, &T, lk);
    if (rc) { st.finish(); return rc; }
    uint64_t *vals = (uint64_t *)st.out(args[0].pdata, 8 * len);
    const Packed K{(const int64_t *)st.in(args[3].pdata, 8 * (len + 1)), (const uint8_t *)st.in(args[4].pdata, args[4].pdata ? args[4].dataSz : 0), args[4].pdata ? args[4].dataSz : 0};
    const uint64_t *skip = (const uint64_t *)st.in(args[3].pnulls, args[3].pnulls && len ? ((len + 63) / 64) * 8 : 0);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    cudaEventRecord(t.kev0, t.stream);
    st_find_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(T, K, skip, len, vals, bad);
    cudaEventRecord(t.kev1, t.stream);
    MOB_LAUNCH_CHECK();
    rc = check_bad(t, bad, "str join find: key offsets are not increasing or point past the key bytes");
    int frc = st.finish();
    return rc ? rc : frc;
}

// MO_XCALL_STR_JOIN_PROBE: args [0] probe_rows int64[cap] ; [1] build_rows int64[cap] ; [2] int64 count (out) ; [3] host mo_join_params_t ;
// [4] table offsets ; [5] table bytes ; [6] sels offsets int32[ngroups + 2] (pdata NULL: unique map) ; [7] sels vals ; [8] probe key offsets (+pnulls) ;
// [9] probe key bytes
int xcall_str_join_probe(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!args[3].pdata || args[3].dataSz < sizeof(mo_join_params_t) || is_device_ptr(args[3].pdata)) { set_error("str join probe: host mo_join_params_t missing"); return MO_RC_INVALID_ARGUMENT; }
    mo_join_params_t P;
    memcpy(&P, args[3].pdata, sizeof P);
    if (P.join_type < MO_JOIN_INNER || P.join_type > MO_JOIN_ANTI) { set_error("str join probe: join type %d", P.join_type); return MO_RC_INVALID_ARGUMENT; }
    const uint64_t cap = args[0].dataSz / 8;
    if (args[1].dataSz / 8 < cap || !args[2].pdata || args[2].dataSz < 8 || args[8].dataSz < 8 * (len + 1)) { set_error("str join probe: buffers too small"); return MO_RC_INVALID_ARGUMENT; }
    const uint64_t ngroups = groups_of(args[4]);
    const bool multi = args[6].pdata != nullptr;
    if (multi && args[6].dataSz < (ngroups + 2) * 4) { set_error("str join probe: sels offsets shorter than the group count + 2"); return MO_RC_INVALID_ARGUMENT; }
    Stager st(t);
    unsigned *bad = (unsigned *)st.tmp(16);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    MOB_CUDA_TRY(cudaMemsetAsync(bad, 0, 16, t.stream));
    StrTable T;
    std::shared_lock<std::shared_mutex> lk;
    int rc = str_table_for(t, st, args[4], args[5], bad, &T, lk);
    if (rc) { st.finish(); return rc; }
    int64_t *out_probe = (int64_t *)st.out(args[0].pdata, cap * 8);
    int64_t *out_build = (int64_t *)st.out(args[1].pdata, cap * 8);
    int64_t *count = (int64_t *)st.out(args[2].pdata, 8);
    const int32_t *offsets = multi ? (const int32_t *)st.in(args[6].pdata, (ngroups + 2) * 4) : nullptr;
    const int32_t *sels = multi ? (const int32_t *)st.in(args[7].pdata, args[7].dataSz) : nullptr;
    const Packed K{(const int64_t *)st.in(args[8].pdata, 8 * (len + 1)), (const uint8_t *)st.in(args[9].pdata, args[9].pdata ? args[9].dataSz : 0), args[9].pdata ? args[9].dataSz : 0};
    const uint64_t *skip = (const uint64_t *)st.in(args[8].pnulls, args[8].pnulls && len ? ((len + 63) / 64) * 8 : 0);
    uint32_t *vals = (uint32_t *)st.tmp(len * 4 + 4);
    uint64_t *cnt = (uint64_t *)st.tmp((len + 1) * 8);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    cudaEventRecord(t.kev0, t.stream);
    st_probe_count_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(T, K, skip, len, offsets, P.join_type, vals, cnt, bad);
    MOB_LAUNCH_CHECK();
    int64_t produced = 0;
    rc = probe_scan_emit(t, len, vals, cnt, offsets, sels, P.join_type, cap, out_probe, out_build, count, &produced);
    if (!rc) rc = check_bad(t, bad, "str join probe: key offsets are not increasing or point past the key bytes");
    int frc = st.finish();
    if (rc) return rc;
    if ((uint64_t)produced > cap) { set_error("str join probe: %lld result rows exceed the output capacity (%llu); the count is reported, call again with larger buffers", (long long)produced, (unsigned long long)cap); return MO_RC_OUT_OF_RANGE; }
    return frc;
}

}  // namespace mob

// ---- prepared string join maps (as MoB200_JoinMapPrepare: the JoinMap lives for the whole probe phase, message/joinMapMsg.go:127-160) -------------
extern "C" int32_t MoB200_StrJoinMapPrepare(const void *key_offsets, const void *key_bytes, uint64_t ngroups) {
    using namespace mob;
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!key_offsets || ngroups >= kMaxRows) { set_error("string join map: key offsets missing or more than 2^30 groups"); return MO_RC_INVALID_ARGUMENT; }
    int64_t nbytes = 0;
    if (is_device_ptr(key_offsets)) { int rc = read_back(t, &nbytes, (const int64_t *)key_offsets + ngroups, 8); if (rc) return rc; }
    else memcpy(&nbytes, (const int64_t *)key_offsets + ngroups, 8);
    if (nbytes < 0 || (nbytes > 0 && !key_bytes)) { set_error("string join map: key offsets[ngroups] = %lld", (long long)nbytes); return MO_RC_INVALID_ARGUMENT; }
    Stager st(t);
    const int64_t *doff = (const int64_t *)st.in(key_offsets, (ngroups + 1) * 8);
    const uint8_t *dbytes = (const uint8_t *)st.in(key_bytes, (size_t)nbytes);
    unsigned *bad = (unsigned *)st.tmp(16);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    MOB_CUDA_TRY(cudaMemsetAsync(bad, 0, 16, t.stream));
    StrDevTable D;
    int rc = build_str_table(t, doff, dbytes, (uint64_t)nbytes, ngroups, true, bad, &D);
    if (!rc) rc = check_bad(t, bad, "string join map: key offsets are not increasing or point past the key bytes");
    int frc = st.finish();
    if (rc || frc) { free_table(D); return rc ? rc : frc; }
    std::unique_lock<std::shared_mutex> lk(g_sjm_mu);
    auto it = g_sjm.find(key_offsets);
    if (it != g_sjm.end()) free_table(it->second);
    g_sjm[key_offsets] = D;
    return MO_RC_SUCCESS;
}

extern "C" int32_t MoB200_StrJoinMapRelease(const void *key_offsets) {
    using namespace mob;
    std::unique_lock<std::shared_mutex> lk(g_sjm_mu);
    auto it = g_sjm.find(key_offsets);
    if (it == g_sjm.end()) return MO_RC_SUCCESS;
    // (probes hold the shared lock until their stream has drained, so nothing is reading the table once the unique lock is ours)
    free_table(it->second);
    g_sjm.erase(it);
    return MO_RC_SUCCESS;
}
