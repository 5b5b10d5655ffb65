// hashops.cuh -- internal helpers shared by the group-by and join translation units (colops.cu, join.cu, strhash.cu).
// Not part of the C-ABI.
#pragma once
#include "common.cuh"

namespace mob {

// grid for a grid-stride loop over `items` work items of `per_block` each, capped at a few waves
inline unsigned grid_for(uint64_t items, int per_block = 256) {
    uint64_t g = (items + per_block - 1) / per_block;
    const uint64_t mx = (uint64_t)num_sms() * (per_block == 1 ? 32 : 16);
    return (unsigned)(g > mx ? mx : (g ? g : 1));
}

// join.cu: out[i] = sum of in[0 .. i); *total (device) = sum of all.  in == out allowed.  Scratch from the arena.
int exclusive_scan(ThreadCtx &t, const uint64_t *in, uint64_t n, uint64_t *out, uint64_t *total);

// colops.cu: order-preserving compaction -- the indices of the rows with v[i] != 0 (and no bit in nulls), ascending; *dtotal (device) = count
template <typename OutT>
int launch_select(ThreadCtx &t, const uint8_t *v, const uint64_t *nulls, uint64_t n, OutT *sels, unsigned long long *dtotal);

// join.cu, the emission half of JOIN_PROBE: per probe row the matched group id vals[i] (0 = no match) and its result-row count cnt[i]
// (probe_row_count); cnt is turned into positions in place, then the (probe row, build row) pairs are written in the reference's order.
// *produced (host) = result rows, also written to *count_out (device); rows past `cap` are not written.
int probe_scan_emit(ThreadCtx &t, uint64_t n, const uint32_t *vals, uint64_t *cnt, const int32_t *offsets, const int32_t *sels, int join_type,
                    uint64_t cap, int64_t *out_probe, int64_t *out_build, int64_t *count_out, int64_t *produced);

}  // namespace mob

#ifdef __CUDACC__
namespace mob {

// result rows of one probe row whose key found group v (0 = none): matches m = the group's sels (unique map: 1), then per join type
// (hashjoin/join.go:383-628).  *v is cleared when the row has no match.
__device__ __forceinline__ uint64_t probe_row_count(uint32_t *v, const int32_t *__restrict__ offsets, int join_type) {
    uint64_t m = 0;
    if (*v) m = offsets ? (uint64_t)(offsets[*v] - offsets[*v - 1]) : 1ull;
    if (!m) *v = 0;
    switch (join_type) {
    case MO_JOIN_INNER: return m;
    case MO_JOIN_LEFT: return m ? m : 1;        // EmitUnmatchedProbe: one row with the build side NULL
    case MO_JOIN_SEMI: return m ? 1 : 0;
    default: return m ? 0 : 1;                   // anti
    }
}

}  // namespace mob
#endif
