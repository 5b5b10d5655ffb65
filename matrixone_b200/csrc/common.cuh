// common.cuh -- runtime plumbing shared by every translation unit of libmo_b200.so.
//
// One ThreadCtx per calling OS thread (the reference calls the cgo surface from arbitrary goroutines pinned to
// arbitrary OS threads, pkg/sql/compile/scope.go:442-499): its own CUDA stream, timing events, a device scratch
// arena and a small pinned staging buffer, so concurrent callers never share mutable state.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <vector>
#include <atomic>
#include <memory>
#include "../../include/mo_b200.h"

namespace mob {

constexpr int kSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

struct ArenaBlock { char *p; size_t size; };

struct ThreadCtx {
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    bool ready = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t kev0 = nullptr, kev1 = nullptr;  // bracket the dominant kernel of the last call (MoB200_LastKernelMs)
    std::vector<ArenaBlock> blocks;  // device scratch arena (bump allocated, reset per call)
    size_t cur_block = 0, cur_off = 0;
    int kev_prio = 0;                // priority of the kernel kev0/kev1 currently bracket within this call (reset with the arena)
    uint64_t arena_epoch = 0;        // bumped by arena_reset: per-call caches of arena pointers key on it
    char *pinned = nullptr;          // small pinned staging (scalar results, status words)
    size_t pinned_sz = 0;
    unsigned *ctrl = nullptr;        // 64 device words, zero between calls ("last CTA done" tickets, atomicInc wraps)
    char err[256] = {0};
};

ThreadCtx &tctx();                      // lazily initialises the runtime and the calling thread's context
int runtime_init(int device);           // idempotent
void set_error(const char *fmt, ...);
extern std::atomic<uint64_t> g_launches;
int num_sms();

// cudaPointerGetAttributes classification
bool is_device_ptr(const void *p);

// prepared search operands (tcsearch.cu) that read [p, p + bytes) are dropped: called by every library entry point that WRITES device memory
void search_invalidate(const void *p, uint64_t bytes);

// --- device scratch arena -------------------------------------------------------------------------------
void *arena_alloc(ThreadCtx &t, size_t bytes);   // 256-byte aligned; nullptr on failure (error set)
void arena_reset(ThreadCtx &t);                  // called at the end of every API call
// scoped scratch inside one call (loops that need temporaries per iteration): everything allocated after the mark is handed back by the rewind
struct ArenaMark { size_t block, off; };
inline ArenaMark arena_mark(ThreadCtx &t) { return ArenaMark{t.cur_block, t.cur_off}; }
inline void arena_rewind(ThreadCtx &t, ArenaMark m) { t.cur_block = m.block; t.cur_off = m.off; }

// --- Stager: makes every pointer argument a device pointer for the duration of one call -------------------
struct Stager {
    ThreadCtx &t;
    struct Back { void *host; const void *dev; size_t bytes; };
    std::vector<Back> backs;
    std::vector<std::shared_ptr<void>> pins;   // column-cache blocks this call reads (kept alive until finish())
    bool failed = false;
    bool finished = false;   // set by finish(); the destructor cleans up otherwise
    explicit Stager(ThreadCtx &tc) : t(tc) {}
    // input: device pointers pass through, host pointers are copied into the arena (async on t.stream)
    const void *in(const void *p, size_t bytes);
    // output: device pointers pass through; host pointers get an arena buffer that is copied back by finish().
    // preload=true first uploads the host content (needed when the kernel writes only some rows).
    void *out(void *p, size_t bytes, bool preload = false);
    // device temp
    void *tmp(size_t bytes) { void *q = arena_alloc(t, bytes); if (!q) failed = true; return q; }
    // copy-backs + stream sync + arena reset. Returns MO_RC_SUCCESS or MO_RC_INTERNAL_ERROR.
    int finish();
    // asynchronous form (every pointer was a device pointer): nothing to copy back, no synchronise; the scratch is handed back in stream order
    void release_async() { backs.clear(); arena_reset(t); finished = true; }   // (no cached host blocks on this path: every pointer was a device pointer)
    ~Stager();
};

#define MOB_CUDA_TRY(expr)                                                                    \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            mob::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return MO_RC_INTERNAL_ERROR;                                                      \
        }                                                                                     \
    } while (0)

// count + check a kernel launch
#define MOB_LAUNCH_CHECK()                                                                    \
    do {                                                                                      \
        mob::g_launches.fetch_add(1, std::memory_order_relaxed);                              \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess) {                                                              \
            mob::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
            return MO_RC_INTERNAL_ERROR;                                                      \
        }                                                                                     \
    } while (0)

// read one small device value back through the pinned staging buffer (synchronises the stream)
int read_back(ThreadCtx &t, void *host_dst, const void *dev_src, size_t bytes);

}  // namespace mob

// =========================================================================================================
// device helpers
// =========================================================================================================
#ifdef __CUDACC__
namespace mob {

// 128-bit streaming loads: read-only path, do not allocate in L1 (each byte is touched once)
__device__ __forceinline__ int4 ld_stream16(const void *p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ int2 ld_stream8(const void *p) {
    int2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.s32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream16(void *p, int4 v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}

__device__ __forceinline__ bool bm_test(const uint64_t *p, uint64_t i) { return p && ((p[i >> 6] >> (i & 63)) & 1ull); }

// the bytes of one MatrixOne varlena cell (pkg/container/types/bytes.go:61-115): c[0] <= 23 -> inline, bytes c[1 .. 1 + c[0]); otherwise
// uint32 offset at c + 4 and uint32 length at c + 8 into the area.  false when a big cell points outside [area, area + area_len).
__device__ __forceinline__ bool varlena_bytes(const uint8_t *c, const uint8_t *area, uint64_t area_len, const uint8_t **p, uint64_t *n) {
    if (c[0] <= MO_VARLENA_INLINE_SZ) { *p = c + 1; *n = c[0]; return true; }
    const uint32_t off = (uint32_t)c[4] | ((uint32_t)c[5] << 8) | ((uint32_t)c[6] << 16) | ((uint32_t)c[7] << 24);
    const uint32_t ln = (uint32_t)c[8] | ((uint32_t)c[9] << 8) | ((uint32_t)c[10] << 16) | ((uint32_t)c[11] << 24);
    if (!area || (uint64_t)off + ln > area_len) return false;
    *p = area + off; *n = ln;
    return true;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// fixed-order butterfly: every lane ends with the same value, association independent of data
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = v + __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace mob
#endif
