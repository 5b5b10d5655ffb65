// join.cu -- the data-parallel pieces of the reference's hash join (pkg/sql/colexec/hashbuild/hashmap.go:237-488, pkg/vm/message/joinMapMsg.go:32-132,
// pkg/sql/colexec/hashjoin/join.go:383-628) behind XCall, over the <= 8-byte packed keys of MO_XCALL_PACK_KEYS and the group ids of MO_XCALL_GROUP_IDS.
//
//   build side   GROUP_IDS over the build keys (IntHashMap insert, first-seen ids) gives vals[i]; JOIN_SELS turns them into the JoinMap's GroupSels:
//                offsets int32[groupCount + 2], vals int32[n] -- rows of group k (0-based) at vals[offsets[k] .. offsets[k + 1]), ASCENDING row ids,
//                exactly what GroupSels.Insert + Finalize (joinMapMsg.go:72-125: count, prefix sum, stable scatter) leave behind.
//                Here: order-preserving compaction of the rows with an id, then a stable LSD radix sort by group id (8 bits per pass, one warp per
//                1024-row tile ranks with __match_any_sync so equal digits keep their order), offsets from a histogram + exclusive scan.
//   probe side   JOIN_FIND = intHashMapIterator.Find (vals[i] = group id or 0; a NULL key never matches, zvals == 0).
//                JOIN_PROBE = the emission loop of container.probe for the equality-only joins: per probe row the matched build rows in sels order
//                (unique maps: build row = id - 1), for inner / left outer / left semi / left anti.  Output pairs (probe row, build row | -1) in
//                exactly the order the reference appends them: probe rows ascending, within a row the sels ascending.  Counts -> exclusive scan ->
//                positions; rows with >= 32 matches are written by their whole warp.
//   The hash table itself is not observable in the reference (random seeds): ids and pairs are.  The device table is rebuilt from table_keys per
//   call (O(groups)) unless it was prepared with MoB200_JoinMapPrepare (cached per table_keys pointer).
// All passes stream their inputs once; algorithmic bytes per probe row: 8 (key) + 16 per emitted pair + one random 8-byte table probe.
#include "hashops.cuh"
#include <cstring>
#include <mutex>
#include <shared_mutex>
#include <unordered_map>

namespace mob {

namespace {

constexpr int kThreads = 256;
constexpr uint64_t kEmptyKey = 0xffffffffffffffffull;

__device__ __forceinline__ uint64_t mix64(uint64_t x) { x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; return x ^ (x >> 33); }

// ---- exclusive scan of uint64 (three kernels: tile sums, scan of the sums by one CTA, apply) ---------------------------------------------------
constexpr int kScanTile = 2048;   // 256 threads x 8
__global__ void __launch_bounds__(kThreads) scan_sums_kernel(const uint64_t *__restrict__ in, uint64_t n, uint64_t *__restrict__ sums) {
    __shared__ uint64_t sw[kThreads / 32];
    const uint64_t base = (uint64_t)blockIdx.x * kScanTile;
    uint64_t s = 0;
    for (int j = 0; j < 8; j++) { const uint64_t i = base + (uint64_t)j * kThreads + threadIdx.x; if (i < n) s += in[i]; }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sw[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { uint64_t t = 0; for (int w = 0; w < kThreads / 32; w++) t += sw[w]; sums[blockIdx.x] = t; }
}
__global__ void __launch_bounds__(1024) scan_of_sums_kernel(uint64_t *sums, uint64_t nb, uint64_t *total) {
    __shared__ uint64_t sw[32];
    __shared__ uint64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint64_t b0 = 0; b0 < nb; b0 += 1024) {
        const uint64_t i = b0 + threadIdx.x;
        const uint64_t v = i < nb ? sums[i] : 0;
        uint64_t inc = v;
        for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
        if (lane == 31) sw[warp] = inc;
        __syncthreads();
        uint64_t wbase = 0;
        for (int w = 0; w < warp; w++) wbase += sw[w];
        const uint64_t c = carry;
        if (i < nb) sums[i] = c + wbase + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + wbase + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}
__global__ void __launch_bounds__(kThreads) scan_apply_kernel(const uint64_t *__restrict__ in, uint64_t n, const uint64_t *__restrict__ sums, uint64_t *__restrict__ out) {
    // tile layout for the apply pass: thread t owns 8 CONSECUTIVE items, so its exclusive prefix is a register scan
    __shared__ uint64_t sw[kThreads / 32];
    const uint64_t base = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * 8;
    uint64_t v[8], s = 0;
    for (int j = 0; j < 8; j++) { v[j] = base + j < n ? in[base + j] : 0; s += v[j]; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t inc = s;
    for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) sw[warp] = inc;
    __syncthreads();
    uint64_t run = sums[blockIdx.x] + inc - s;
    for (int w = 0; w < warp; w++) run += sw[w];
    for (int j = 0; j < 8; j++) { if (base + j < n) out[base + j] = run; run += v[j]; }
}
}  // namespace

// out[i] = sum of in[0 .. i); *total (device) = sum of all.  in == out allowed.  sums scratch from the arena.
int exclusive_scan(ThreadCtx &t, const uint64_t *in, uint64_t n, uint64_t *out, uint64_t *total) {
    if (n == 0) { MOB_CUDA_TRY(cudaMemsetAsync(total, 0, 8, t.stream)); return MO_RC_SUCCESS; }
    const uint64_t nb = (n + kScanTile - 1) / kScanTile;
    uint64_t *sums = (uint64_t *)arena_alloc(t, nb * 8);
    if (!sums) return MO_RC_INTERNAL_ERROR;
    scan_sums_kernel<<<(unsigned)nb, kThreads, 0, t.stream>>>(in, n, sums);
    MOB_LAUNCH_CHECK();
    scan_of_sums_kernel<<<1, 1024, 0, t.stream>>>(sums, nb, total);
    MOB_LAUNCH_CHECK();
    scan_apply_kernel<<<(unsigned)nb, kThreads, 0, t.stream>>>(in, n, sums, out);
    MOB_LAUNCH_CHECK();
    return MO_RC_SUCCESS;
}

namespace {

// ---- JOIN_SELS ------------------------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) sels_flag_kernel(const uint64_t *__restrict__ groups, uint64_t n, uint64_t ngroups, uint64_t *__restrict__ flag, uint64_t *__restrict__ cnt, unsigned *bad) {
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        const uint64_t g = groups[i];
        if (g > ngroups) { *bad = 1; flag[i] = 0; continue; }
        flag[i] = g ? 1 : 0;
        if (g) atomicAdd((unsigned long long *)&cnt[g - 1], 1ull);
    }
}
__global__ void __launch_bounds__(kThreads) sels_compact_kernel(const uint64_t *__restrict__ groups, const uint64_t *__restrict__ pos, uint64_t n, uint64_t ngroups, uint32_t *__restrict__ key, uint32_t *__restrict__ row) {
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        const uint64_t g = groups[i];
        if (g && g <= ngroups) { key[pos[i]] = (uint32_t)(g - 1); row[pos[i]] = (uint32_t)i; }
    }
}
// one radix pass, 8 bits at `shift`: tiles of 1024 items, ONE WARP per tile
constexpr int kRadixTile = 1024;
__global__ void __launch_bounds__(32) radix_hist_kernel(const uint32_t *__restrict__ key, const uint64_t *__restrict__ m_ptr, int shift, uint64_t *__restrict__ hist, uint64_t nblocks_cap) {
    __shared__ unsigned h[256];
    const uint64_t m = *m_ptr;
    const uint64_t nblocks = (m + kRadixTile - 1) / kRadixTile;
    for (uint64_t b = blockIdx.x; b < nblocks_cap; b += gridDim.x) {
        for (int d = threadIdx.x; d < 256; d += 32) h[d] = 0;
        __syncwarp();
        if (b < nblocks) {
            for (int r = 0; r < kRadixTile / 32; r++) {
                const uint64_t i = b * kRadixTile + (uint64_t)r * 32 + threadIdx.x;
                if (i < m) atomicAdd(&h[(key[i] >> shift) & 255u], 1u);
            }
        }
        __syncwarp();
        for (int d = threadIdx.x; d < 256; d += 32) hist[(uint64_t)d * nblocks_cap + b] = h[d];   // digit-major: the scan orders (digit, tile)
        __syncwarp();
    }
}
__global__ void __launch_bounds__(32) radix_scatter_kernel(const uint32_t *__restrict__ key, const uint32_t *__restrict__ row, const uint64_t *__restrict__ m_ptr, int shift,
                                                           const uint64_t *__restrict__ base, uint64_t nblocks_cap, uint32_t *__restrict__ okey, uint32_t *__restrict__ orow) {
    __shared__ uint64_t run[256];
    const uint64_t m = *m_ptr;
    const uint64_t nblocks = (m + kRadixTile - 1) / kRadixTile;
    const unsigned lane = threadIdx.x;
    for (uint64_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
        for (int d = lane; d < 256; d += 32) run[d] = base[(uint64_t)d * nblocks_cap + b];
        __syncwarp();
        for (int r = 0; r < kRadixTile / 32; r++) {
            const uint64_t i = b * kRadixTile + (uint64_t)r * 32 + lane;
            const bool live = i < m;
            const uint32_t k = live ? key[i] : 0u, rw = live ? row[i] : 0u;
            const unsigned d = live ? ((k >> shift) & 255u) : 256u;            // 256: the dead lanes of the last round match only each other
            const unsigned peers = __match_any_sync(0xffffffffu, d);
            const unsigned rank = __popc(peers & ((1u << lane) - 1u));
            uint64_t pos = 0;
            if (live) pos = run[d] + rank;
            __syncwarp();
            if (live && rank == 0) run[d] += __popc(peers);                  // the lowest lane of every digit class advances its cursor
            __syncwarp();
            if (live) { okey[pos] = k; orow[pos] = rw; }
        }
        __syncwarp();
    }
}
__global__ void __launch_bounds__(kThreads) sels_offsets_kernel(const uint64_t *__restrict__ starts, uint64_t ngroups, const uint64_t *__restrict__ total, int32_t *__restrict__ offsets) {
    // offsets has ngroups + 2 entries: [k] = start of group k, [ngroups] = [ngroups + 1] = n (joinMapMsg.go:89-121)
    for (uint64_t k = blockIdx.x * (uint64_t)kThreads + threadIdx.x; k < ngroups + 2; k += (uint64_t)gridDim.x * kThreads)
        offsets[k] = (int32_t)(k < ngroups ? starts[k] : *total);
}
__global__ void __launch_bounds__(kThreads) copy_rows_kernel(const uint32_t *__restrict__ row, const uint64_t *__restrict__ m_ptr, int32_t *__restrict__ vals, int64_t *count_out) {
    const uint64_t m = *m_ptr;
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < m; i += (uint64_t)gridDim.x * kThreads) vals[i] = (int32_t)row[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) *count_out = (int64_t)m;
}

// ---- the probe-side hash table -----------------------------------------------------------------------------------------------------------------------
struct JoinTable { uint64_t *key; uint32_t *id; uint64_t mask; uint32_t sentinel_id; /* id of the key 0xff..ff (stored outside the table) */ };

__global__ void __launch_bounds__(kThreads) jt_init_kernel(uint64_t *key, uint32_t *id, uint64_t slots) {
    for (uint64_t s = blockIdx.x * (uint64_t)kThreads + threadIdx.x; s < slots; s += (uint64_t)gridDim.x * kThreads) { key[s] = kEmptyKey; id[s] = 0; }
}
__global__ void __launch_bounds__(kThreads) jt_build_kernel(const uint64_t *__restrict__ table_keys, uint64_t ngroups, uint64_t *key, uint32_t *id, uint64_t mask, uint32_t *sentinel_id) {
    for (uint64_t g = blockIdx.x * (uint64_t)kThreads + threadIdx.x; g < ngroups; g += (uint64_t)gridDim.x * kThreads) {
        const uint64_t k = table_keys[g];
        if (k == kEmptyKey) { *sentinel_id = (uint32_t)(g + 1); continue; }
        uint64_t s = mix64(k) & mask;
        for (;;) {
            const uint64_t cur = atomicCAS((unsigned long long *)&key[s], (unsigned long long)kEmptyKey, (unsigned long long)k);
            if (cur == kEmptyKey || cur == k) { id[s] = (uint32_t)(g + 1); break; }   // table_keys are distinct: one writer per slot
            s = (s + 1) & mask;
        }
    }
}
__device__ __forceinline__ uint32_t jt_find(const uint64_t *__restrict__ key, const uint32_t *__restrict__ id, uint64_t mask, const uint32_t *sentinel_id, uint64_t k) {
    if (k == kEmptyKey) return *sentinel_id;
    uint64_t s = mix64(k) & mask;
    for (;;) {
        const uint64_t cur = key[s];
        if (cur == k) return id[s];
        if (cur == kEmptyKey) return 0;
        s = (s + 1) & mask;
    }
}
__global__ void __launch_bounds__(kThreads) jt_find_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ knulls, uint64_t n, const uint64_t *__restrict__ tkey,
                                                           const uint32_t *__restrict__ tid, uint64_t mask, const uint32_t *sentinel_id, uint64_t *__restrict__ vals) {
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        const bool isnull = knulls && ((knulls[i >> 6] >> (i & 63)) & 1ull);
        vals[i] = isnull ? 0ull : (uint64_t)jt_find(tkey, tid, mask, sentinel_id, keys[i]);
    }
}

struct DevTable { uint64_t *key = nullptr; uint32_t *id = nullptr; uint32_t *sentinel = nullptr; uint64_t mask = 0; uint64_t ngroups = 0; bool cached = false; };
std::shared_mutex g_jm_mu;
std::unordered_map<const void *, DevTable> g_jm;   // prepared join maps, by table_keys pointer

int build_table(ThreadCtx &t, const uint64_t *dkeys, uint64_t ngroups, bool persistent, DevTable *out) {
    uint64_t slots = 64;
    while (slots < 2 * ngroups) slots <<= 1;
    DevTable T;
    if (persistent) {
        if (cudaMalloc(&T.key, slots * 8) != cudaSuccess || cudaMalloc(&T.id, slots * 4) != cudaSuccess || cudaMalloc(&T.sentinel, 4) != cudaSuccess) {
            set_error("join map: cudaMalloc of a %llu-slot table failed", (unsigned long long)slots);
            if (T.key) cudaFree(T.key);
            if (T.id) cudaFree(T.id);
            return MO_RC_INTERNAL_ERROR;
        }
    } else {
        T.key = (uint64_t *)arena_alloc(t, slots * 8); T.id = (uint32_t *)arena_alloc(t, slots * 4); T.sentinel = (uint32_t *)arena_alloc(t, 4);
        if (!T.key || !T.id || !T.sentinel) return MO_RC_INTERNAL_ERROR;
    }
    T.mask = slots - 1; T.ngroups = ngroups; T.cached = persistent;
    MOB_CUDA_TRY(cudaMemsetAsync(T.sentinel, 0, 4, t.stream));
    jt_init_kernel<<<grid_for(slots), kThreads, 0, t.stream>>>(T.key, T.id, slots);
    MOB_LAUNCH_CHECK();
    if (ngroups) {
        jt_build_kernel<<<grid_for(ngroups), kThreads, 0, t.stream>>>(dkeys, ngroups, T.key, T.id, T.mask, T.sentinel);
        MOB_LAUNCH_CHECK();
    }
    *out = T;
    return MO_RC_SUCCESS;
}

// the table for this call: the prepared one (by the caller's table_keys pointer) or a scratch one in the arena
int table_for(ThreadCtx &t, Stager &st, const mo_xcall_args_t &a, DevTable *T, std::shared_lock<std::shared_mutex> &lk) {
    const uint64_t ngroups = a.dataSz / 8;
    lk = std::shared_lock<std::shared_mutex>(g_jm_mu);
    auto it = g_jm.find(a.pdata);
    if (it != g_jm.end() && it->second.ngroups == ngroups) { *T = it->second; return MO_RC_SUCCESS; }
    lk.unlock();
    const uint64_t *dkeys = (const uint64_t *)st.in(a.pdata, ngroups * 8);
    if (st.failed) return MO_RC_INTERNAL_ERROR;
    return build_table(t, dkeys, ngroups, false, T);
}

// ---- JOIN_PROBE -----------------------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) probe_count_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ knulls, uint64_t n, const uint64_t *__restrict__ tkey,
                                                               const uint32_t *__restrict__ tid, uint64_t mask, const uint32_t *sentinel_id, const int32_t *__restrict__ offsets,
                                                               int join_type, uint32_t *__restrict__ vals, uint64_t *__restrict__ cnt) {
    for (uint64_t i = blockIdx.x * (uint64_t)kThreads + threadIdx.x; i < n; i += (uint64_t)gridDim.x * kThreads) {
        const bool isnull = knulls && ((knulls[i >> 6] >> (i & 63)) & 1ull);
        uint32_t v = isnull ? 0u : jt_find(tkey, tid, mask, sentinel_id, keys[i]);
        cnt[i] = probe_row_count(&v, offsets, join_type);
        vals[i] = v;
    }
}
__global__ void __launch_bounds__(kThreads) probe_emit_kernel(uint64_t n, const uint32_t *__restrict__ vals, const uint64_t *__restrict__ pos, const uint64_t *__restrict__ total,
                                                              const int32_t *__restrict__ offsets, const int32_t *__restrict__ sels, int join_type, uint64_t cap,
                                                              int64_t *__restrict__ out_probe, int64_t *__restrict__ out_build, int64_t *count_out) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t nrounds = (n + 31) / 32;
    for (uint64_t w = (blockIdx.x * (uint64_t)kThreads + threadIdx.x) >> 5; w < nrounds; w += ((uint64_t)gridDim.x * kThreads) >> 5) {
        const uint64_t i = w * 32 + lane;
        uint32_t v = 0; uint64_t p = 0, c = 0;
        if (i < n) { v = vals[i]; p = pos[i]; c = (i + 1 < n ? pos[i + 1] : *total) - p; }
        const bool pairs = (join_type == MO_JOIN_INNER || join_type == MO_JOIN_LEFT) && v;
        const int32_t s0 = (pairs && offsets) ? offsets[v - 1] : 0;
        if (c && c < 32) {
            for (uint64_t j = 0; j < c; j++) {
                if (p + j >= cap) break;
                out_probe[p + j] = (int64_t)i;
                out_build[p + j] = pairs ? (offsets ? (int64_t)sels[s0 + j] : (int64_t)v - 1) : -1;
            }
        }
        unsigned heavy = __ballot_sync(0xffffffffu, c >= 32);
        while (heavy) {                                   // rows with many matches are written by the whole warp, coalesced
            const int src = __ffs(heavy) - 1; heavy &= heavy - 1;
            const uint64_t hi = __shfl_sync(0xffffffffu, i, src), hp = __shfl_sync(0xffffffffu, p, src), hc = __shfl_sync(0xffffffffu, c, src);
            const int32_t hs0 = __shfl_sync(0xffffffffu, s0, src);
            for (uint64_t j = lane; j < hc; j += 32) {
                if (hp + j >= cap) break;
                out_probe[hp + j] = (int64_t)hi;
                out_build[hp + j] = (int64_t)sels[hs0 + j];      // >= 32 matches only happens with sels
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *count_out = (int64_t)*total;
}

}  // namespace

int probe_scan_emit(ThreadCtx &t, uint64_t n, const uint32_t *vals, uint64_t *cnt, const int32_t *offsets, const int32_t *sels, int join_type,
                    uint64_t cap, int64_t *out_probe, int64_t *out_build, int64_t *count_out, int64_t *produced) {
    uint64_t *total = (uint64_t *)arena_alloc(t, 8);
    if (!total) return MO_RC_INTERNAL_ERROR;
    int rc = exclusive_scan(t, cnt, n, cnt, total);
    if (rc) return rc;
    probe_emit_kernel<<<grid_for(n ? n : 1), kThreads, 0, t.stream>>>(n, vals, cnt, total, offsets, sels, join_type, cap, out_probe, out_build, count_out);
    cudaEventRecord(t.kev1, t.stream);
    MOB_LAUNCH_CHECK();
    return read_back(t, produced, total, 8);
}

// Stable grouping of rows by their 1-based group id (0 = the row takes no part): *starts = uint64[ngroups + 1] (start of every 0-based group in
// *rows), *rows = uint32[n] row ids, ascending inside every group, *scal[0] = how many rows have a group, scal[2] (as unsigned) != 0 = an id exceeded
// ngroups.  Everything lives in the call's arena.  Used by JOIN_SELS and by the k-means centroid update (kmeans.cu).
int group_rows_stable(ThreadCtx &t, const uint64_t *groups, uint64_t len, uint64_t ngroups, uint64_t **starts, uint32_t **rows, uint64_t **scal_out) {
    uint64_t *flag = (uint64_t *)arena_alloc(t, (len + 1) * 8), *cnt = (uint64_t *)arena_alloc(t, (ngroups + 1) * 8);
    uint32_t *k0 = (uint32_t *)arena_alloc(t, len * 4 + 4), *r0 = (uint32_t *)arena_alloc(t, len * 4 + 4), *k1 = (uint32_t *)arena_alloc(t, len * 4 + 4), *r1 = (uint32_t *)arena_alloc(t, len * 4 + 4);
    const uint64_t nblocks_cap = (len + kRadixTile - 1) / kRadixTile + 1;
    uint64_t *hist = (uint64_t *)arena_alloc(t, 256 * nblocks_cap * 8);
    uint64_t *scal = (uint64_t *)arena_alloc(t, 32);     // [0] rows with a group, [1] scratch total, [2] bad flag
    if (!flag || !cnt || !k0 || !r0 || !k1 || !r1 || !hist || !scal) return MO_RC_INTERNAL_ERROR;
    MOB_CUDA_TRY(cudaMemsetAsync(cnt, 0, (ngroups + 1) * 8, t.stream));
    MOB_CUDA_TRY(cudaMemsetAsync(scal, 0, 32, t.stream));
    sels_flag_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(groups, len, ngroups, flag, cnt, (unsigned *)(scal + 2));
    MOB_LAUNCH_CHECK();
    int rc = exclusive_scan(t, flag, len, flag, scal);                 // flag -> position among the rows that have a group ; scal[0] = m
    if (rc) return rc;
    sels_compact_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(groups, flag, len, ngroups, k0, r0);
    MOB_LAUNCH_CHECK();
    int bits = 0;
    while (bits < 32 && (1ull << bits) < ngroups) bits++;
    uint32_t *ka = k0, *ra = r0, *kb = k1, *rb = r1;
    for (int shift = 0; shift < bits; shift += 8) {
        const unsigned g = grid_for(nblocks_cap, 1);
        radix_hist_kernel<<<g, 32, 0, t.stream>>>(ka, scal, shift, hist, nblocks_cap);
        MOB_LAUNCH_CHECK();
        rc = exclusive_scan(t, hist, 256 * nblocks_cap, hist, scal + 1);
        if (rc) return rc;
        radix_scatter_kernel<<<g, 32, 0, t.stream>>>(ka, ra, scal, shift, hist, nblocks_cap, kb, rb);
        MOB_LAUNCH_CHECK();
        uint32_t *x = ka; ka = kb; kb = x; x = ra; ra = rb; rb = x;
    }
    rc = exclusive_scan(t, cnt, ngroups, cnt, scal + 1);               // cnt[k] -> start of group k
    if (rc) return rc;
    MOB_CUDA_TRY(cudaMemcpyAsync(cnt + ngroups, scal, 8, cudaMemcpyDeviceToDevice, t.stream));   // starts[ngroups] = m
    *starts = cnt; *rows = ra; *scal_out = scal;
    return MO_RC_SUCCESS;
}

// MO_XCALL_JOIN_SELS: args [0] offsets int32[ngroups + 2] ; [1] vals int32[len] ; [2] int64 count (out: rows that have a group) ; [3] groups uint64[len]
int xcall_join_sels(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!args[0].pdata || args[0].dataSz < 8 || !args[2].pdata || args[2].dataSz < 8 || args[1].dataSz < 4 * len || args[3].dataSz < 8 * len) { set_error("join sels: buffers too small"); return MO_RC_INVALID_ARGUMENT; }
    if (len >= 0x7fffffffull) { set_error("join sels: at most 2^31 build rows (row ids are int32, joinMapMsg.go:32-40)"); return MO_RC_INVALID_ARGUMENT; }
    const uint64_t ngroups = args[0].dataSz / 4 - 2;
    Stager st(t);
    int32_t *offsets = (int32_t *)st.out(args[0].pdata, (ngroups + 2) * 4);
    int32_t *vals = (int32_t *)st.out(args[1].pdata, 4 * len);
    int64_t *count = (int64_t *)st.out(args[2].pdata, 8);
    const uint64_t *groups = (const uint64_t *)st.in(args[3].pdata, 8 * len);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    cudaEventRecord(t.kev0, t.stream);
    uint64_t *starts, *scal; uint32_t *rows;
    int rc = group_rows_stable(t, groups, len, ngroups, &starts, &rows, &scal);
    if (rc) { st.finish(); return rc; }
    sels_offsets_kernel<<<grid_for(ngroups + 2), kThreads, 0, t.stream>>>(starts, ngroups, scal, offsets);
    MOB_LAUNCH_CHECK();
    copy_rows_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(rows, scal, vals, count);
    cudaEventRecord(t.kev1, t.stream);
    MOB_LAUNCH_CHECK();
    unsigned bad = 0;
    rc = read_back(t, &bad, scal + 2, 4);
    int frc = st.finish();
    if (rc) return rc;
    if (bad) { set_error("join sels: a group id exceeds the group count (%llu)", (unsigned long long)ngroups); return MO_RC_INVALID_ARGUMENT; }
    return frc;
}

// MO_XCALL_JOIN_FIND: args [0] vals uint64[len] ; [1] table_keys uint64[ngroups] ; [2] probe keys uint64[len] (+pnulls)
int xcall_join_find(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (args[0].dataSz < 8 * len || args[2].dataSz < 8 * len) { set_error("join find: buffers too small"); return MO_RC_INVALID_ARGUMENT; }
    Stager st(t);
    DevTable T;
    std::shared_lock<std::shared_mutex> lk;
    int rc = table_for(t, st, args[1], &T, lk);
    if (rc) { st.finish(); return rc; }
    uint64_t *vals = (uint64_t *)st.out(args[0].pdata, 8 * len);
    const uint64_t *keys = (const uint64_t *)st.in(args[2].pdata, 8 * len);
    const uint64_t *kn = (const uint64_t *)st.in(args[2].pnulls, args[2].pnulls ? ((len + 63) / 64) * 8 : 0);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    cudaEventRecord(t.kev0, t.stream);
    jt_find_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(keys, kn, len, T.key, T.id, T.mask, T.sentinel, vals);
    cudaEventRecord(t.kev1, t.stream);
    MOB_LAUNCH_CHECK();
    return st.finish();
}

// MO_XCALL_JOIN_PROBE: args [0] probe_rows int64[cap] ; [1] build_rows int64[cap] ; [2] int64 count (out) ; [3] host mo_join_params_t ; [4] table_keys uint64[ngroups]
// ; [5] sels offsets int32[ngroups + 2] (pdata NULL: unique map, build row = id - 1) ; [6] sels vals int32[] ; [7] probe keys uint64[len] (+pnulls)
int xcall_join_probe(mo_xcall_args_t *args, uint64_t len) {
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    if (!args[3].pdata || args[3].dataSz < sizeof(mo_join_params_t) || is_device_ptr(args[3].pdata)) { set_error("join probe: host mo_join_params_t missing"); return MO_RC_INVALID_ARGUMENT; }
    mo_join_params_t P;
    memcpy(&P, args[3].pdata, sizeof P);
    if (P.join_type < MO_JOIN_INNER || P.join_type > MO_JOIN_ANTI) { set_error("join probe: join type %d", P.join_type); return MO_RC_INVALID_ARGUMENT; }
    const uint64_t cap = args[0].dataSz / 8;
    if (args[1].dataSz / 8 < cap || !args[2].pdata || args[2].dataSz < 8 || args[7].dataSz < 8 * len) { set_error("join probe: buffers too small"); return MO_RC_INVALID_ARGUMENT; }
    const uint64_t ngroups = args[4].dataSz / 8;
    const bool multi = args[5].pdata != nullptr;
    if (multi && args[5].dataSz < (ngroups + 2) * 4) { set_error("join probe: sels offsets shorter than the group count + 2"); return MO_RC_INVALID_ARGUMENT; }
    Stager st(t);
    DevTable T;
    std::shared_lock<std::shared_mutex> lk;
    int rc = table_for(t, st, args[4], &T, lk);
    if (rc) { st.finish(); return rc; }
    int64_t *out_probe = (int64_t *)st.out(args[0].pdata, cap * 8);
    int64_t *out_build = (int64_t *)st.out(args[1].pdata, cap * 8);
    int64_t *count = (int64_t *)st.out(args[2].pdata, 8);
    const int32_t *offsets = multi ? (const int32_t *)st.in(args[5].pdata, (ngroups + 2) * 4) : nullptr;
    const int32_t *sels = multi ? (const int32_t *)st.in(args[6].pdata, args[6].dataSz) : nullptr;
    const uint64_t *keys = (const uint64_t *)st.in(args[7].pdata, 8 * len);
    const uint64_t *kn = (const uint64_t *)st.in(args[7].pnulls, args[7].pnulls ? ((len + 63) / 64) * 8 : 0);
    uint32_t *vals = (uint32_t *)st.tmp(len * 4 + 4);
    uint64_t *cnt = (uint64_t *)st.tmp((len + 1) * 8);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    cudaEventRecord(t.kev0, t.stream);
    probe_count_kernel<<<grid_for(len ? len : 1), kThreads, 0, t.stream>>>(keys, kn, len, T.key, T.id, T.mask, T.sentinel, offsets, P.join_type, vals, cnt);
    MOB_LAUNCH_CHECK();
    int64_t produced = 0;
    rc = probe_scan_emit(t, len, vals, cnt, offsets, sels, P.join_type, cap, out_probe, out_build, count, &produced);
    int frc = st.finish();
    if (rc) return rc;
    if ((uint64_t)produced > cap) { set_error("join probe: %lld result rows exceed the output capacity (%llu); the count is reported, call again with larger buffers", (long long)produced, (unsigned long long)cap); return MO_RC_OUT_OF_RANGE; }
    return frc;
}

}  // namespace mob

// ---- prepared join maps (the JoinMap message lives for the whole probe phase: message/joinMapMsg.go:127-160) ---------------------------------------
extern "C" int32_t MoB200_JoinMapPrepare(const void *table_keys, uint64_t ngroups) {
    using namespace mob;
    ThreadCtx &t = tctx();
    if (!t.ready) return MO_RC_INTERNAL_ERROR;
    Stager st(t);
    const uint64_t *dkeys = (const uint64_t *)st.in(table_keys, ngroups * 8);
    if (st.failed) { st.finish(); return MO_RC_INTERNAL_ERROR; }
    DevTable T;
    int rc = build_table(t, dkeys, ngroups, true, &T);
    int frc = st.finish();
    if (rc || frc) { if (!rc) { cudaFree(T.key); cudaFree(T.id); cudaFree(T.sentinel); } return rc ? rc : frc; }
    std::unique_lock<std::shared_mutex> lk(g_jm_mu);
    auto it = g_jm.find(table_keys);
    if (it != g_jm.end()) { cudaFree(it->second.key); cudaFree(it->second.id); cudaFree(it->second.sentinel); }
    g_jm[table_keys] = T;
    return MO_RC_SUCCESS;
}

extern "C" int32_t MoB200_JoinMapRelease(const void *table_keys) {
    using namespace mob;
    std::unique_lock<std::shared_mutex> lk(g_jm_mu);
    auto it = g_jm.find(table_keys);
    if (it == g_jm.end()) return MO_RC_SUCCESS;
    // (probes hold the shared lock until their stream has drained, so nothing is reading the table once the unique lock is ours)
    cudaFree(it->second.key); cudaFree(it->second.id); cudaFree(it->second.sentinel);
    g_jm.erase(it);
    return MO_RC_SUCCESS;
}
