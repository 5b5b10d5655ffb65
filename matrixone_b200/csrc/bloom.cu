// bloom.cu -- the reference's C bloom filter (cgo/bloom.h:40-159, cgo/bloom.c) on the GPU, same symbols, same struct, same bits.
//
//   bloomfilter_t is the reference's host struct (magic "XXBF", k, nbits, seed, bitmap[]): init / init_with_seed malloc it, marshal hands its
//   bytes out, unmarshal adopts a caller buffer without a copy, free() releases it -- exactly cgo/bloom.c:98-135,321-339.  What changes is WHERE
//   the bitmap is worked on: every filter gets a DEVICE MIRROR of its bitmap on first use (uploaded once), all add / test / test_and_add / or
//   calls run as kernels against the mirror, and the host copy is refreshed only when somebody asks for the bytes (marshal).  A probe of an
//   8192-row block therefore moves the keys in and one byte per key out, not the filter.
//
//   Bit positions: (h1 + i * h2) & (nbits - 1), i < k, with (h1, h2) = XXH3_128bits_withSeed(key, len, seed) (bloom.c:31-74); 1/2/4-byte keys are
//   sign-extended to int64 first and 8-byte keys hashed as they are (bloom.c:46-55).  The hash is xxh3_128.cuh (pinned to the real xxHash).
//   NULL rows: test -> false, add -> skipped (bloom.c:152-156,203-209).
//
//   test_and_add is SEQUENTIAL in the reference (row i sees the bits rows < i set, bloom.c:241-275).  Here: kernel 1 inserts every (position, row)
//   into a scratch hash table keeping the MINIMUM row per position together with the position's bit before the call; kernel 2 answers
//   result[i] = all positions (bit was set before the call || first row to set it < i) -- which is what the sequential loop computes -- and sets
//   the bits.  Bit-exact, order-independent.
//
//   Kernel shape: one thread per key; the filter words are random 8-byte reads (L2-resident for filters up to ~100 MB), keys stream coalesced.
//   Algorithmic bytes per key: elemsz + 1 result byte + k x 32-byte sectors of the filter.
#include "common.cuh"
#include "xxh3_128.cuh"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <vector>

using namespace mob;

#include "../../include/mo_b200_bloom.h"

namespace {

constexpr int kMaxK = 64;   // MAX_K_SEED, bloom.h:25

struct Mirror { uint64_t *dbits = nullptr; size_t words = 0; bool dev_newer = false; };
std::mutex g_mu;
std::unordered_map<const void *, Mirror> g_mirrors;

[[noreturn]] void bloom_fatal(const char *what) {
    // the reference's entry points return void / bool: there is no error channel, and a silent no-op would corrupt a join.  Fail loudly.
    char msg[512];
    MoB200_LastError(msg, sizeof msg);
    fprintf(stderr, "libmo_b200 bloomfilter: %s failed: %s\n", what, msg);
    abort();
}

inline size_t bitmap_words(uint64_t nbits) { return (size_t)((nbits + 63) / 64); }
inline uint64_t next_pow2_64(uint64_t v) { v--; v |= v >> 1; v |= v >> 2; v |= v >> 4; v |= v >> 8; v |= v >> 16; v |= v >> 32; return v + 1; }

// device mirror of bf's bitmap (created + uploaded on first use).  Returns nullptr (error set) on failure.
uint64_t *mirror_of(ThreadCtx &t, const bloomfilter_t *bf, bool will_write) {
    std::lock_guard<std::mutex> lk(g_mu);
    Mirror &m = g_mirrors[bf];
    const size_t words = bitmap_words(bf->nbits);
    if (!m.dbits || m.words != words) {
        if (m.dbits) cudaFree(m.dbits);
        m.dbits = nullptr; m.words = words; m.dev_newer = false;
        if (cudaMalloc(&m.dbits, words ? words * 8 : 8) != cudaSuccess) { set_error("bloom: cudaMalloc of %zu filter bytes failed", words * 8); g_mirrors.erase(bf); return nullptr; }
        if (words && cudaMemcpyAsync(m.dbits, bf->bitmap, words * 8, cudaMemcpyHostToDevice, t.stream) != cudaSuccess) { set_error("bloom: filter upload failed"); return nullptr; }
        if (cudaStreamSynchronize(t.stream) != cudaSuccess) { set_error("bloom: filter upload failed"); return nullptr; }
    }
    if (will_write) m.dev_newer = true;
    return m.dbits;
}

__device__ __forceinline__ xxh3::Hash128 key_hash(const uint8_t *p, size_t len, uint64_t seed) {
    // bloom_calculate_hash, bloom.c:43-66: narrow integers are widened so that equal values of different widths share their hash
    switch (len) {
    case 1: return xxh3::hash_u64((uint64_t)(int64_t)(int8_t)p[0], seed);
    case 2: return xxh3::hash_u64((uint64_t)(int64_t)(int16_t)((uint16_t)p[0] | ((uint16_t)p[1] << 8)), seed);
    case 4: return xxh3::hash_u64((uint64_t)(int64_t)(int32_t)xxh3::rd32(p), seed);
    case 8: return xxh3::hash_u64(xxh3::rd64(p), seed);
    default: return xxh3::hash_bytes(p, len, seed);
    }
}

struct KeySrc {   // where row i's key bytes are
    const uint8_t *keys; uint64_t len; uint64_t elemsz;      // fixed: keys + i * elemsz ; varlena: 24-byte cells (elemsz = stride)
    const uint8_t *area; uint64_t area_len; int varlena;     // varlena: big cells point into area
    const uint64_t *offs;                                     // 4-byte-length-prefixed stream: byte offset of row i's payload, ~0 = past the end
};
__device__ __forceinline__ bool key_of(const KeySrc &K, uint64_t i, const uint8_t **p, uint64_t *n) {
    if (K.offs) {
        const uint64_t o = K.offs[i];
        if (o == ~0ull) return false;
        *p = K.keys + o; *n = xxh3::rd32(K.keys + o - 4);
        return true;
    }
    if (i * K.elemsz + (K.varlena ? (uint64_t)MO_VARLENA_SZ : K.elemsz) > K.len) return false;   // the reference's  j < len  loop bound (a trailing partial element is not read)
    if (!K.varlena) { *p = K.keys + i * K.elemsz; *n = K.elemsz; return true; }
    return varlena_bytes(K.keys + i * K.elemsz, K.area, K.area_len, p, n);   // (a big cell outside the area: the reference would read out of bounds; such a row is skipped)
}

// MODE 0: add, 1: test
template <int MODE>
__global__ void __launch_bounds__(256)
bloom_kernel(uint64_t *__restrict__ bits, uint64_t nbits, uint32_t k, uint64_t seed, KeySrc K, uint64_t nitem, const uint64_t *__restrict__ nullmap,
             uint8_t *__restrict__ result) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < nitem; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint8_t *p; uint64_t n;
        const bool have = key_of(K, i, &p, &n);
        if (!have) continue;                                                    // rows past the end of the key buffer are not touched (bloom.c loop bounds)
        const bool isnull = nullmap && ((nullmap[i >> 6] >> (i & 63)) & 1ull);
        if (isnull || nbits == 0) { if (MODE == 1) result[i] = 0; continue; }
        const xxh3::Hash128 h = key_hash(p, n, seed);
        if (MODE == 0) {
            for (uint32_t j = 0; j < k; j++) {
                const uint64_t pos = (h.lo + (uint64_t)j * h.hi) & (nbits - 1);
                const uint64_t bit = 1ull << (pos & 63);
                if (!(bits[pos >> 6] & bit)) atomicOr((unsigned long long *)&bits[pos >> 6], (unsigned long long)bit);
            }
        } else {
            bool all = true;   // (issuing all k probes before looking at any was measured: 6 % slower -- the early exit saves more sectors than the overlap gains)
            for (uint32_t j = 0; j < k && all; j++) {
                const uint64_t pos = (h.lo + (uint64_t)j * h.hi) & (nbits - 1);
                all = (__ldg(&bits[pos >> 6]) >> (pos & 63)) & 1ull;
            }
            result[i] = all ? 1 : 0;
        }
    }
}

// ---- test_and_add ------------------------------------------------------------------------------------------------------------------------
constexpr uint64_t kEmpty = ~0ull;
__device__ __forceinline__ uint64_t mix64(uint64_t x) { x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; return x ^ (x >> 33); }

__global__ void __launch_bounds__(256)
taa_insert_kernel(const uint64_t *__restrict__ bits, uint64_t nbits, uint32_t k, uint64_t seed, KeySrc K, uint64_t nitem, const uint64_t *__restrict__ nullmap,
                  uint64_t *__restrict__ tkey, unsigned *__restrict__ trow, uint64_t tmask) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < nitem; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint8_t *p; uint64_t n;
        if (!key_of(K, i, &p, &n)) continue;
        if (nbits == 0 || (nullmap && ((nullmap[i >> 6] >> (i & 63)) & 1ull))) continue;
        const xxh3::Hash128 h = key_hash(p, n, seed);
        for (uint32_t j = 0; j < k; j++) {
            const uint64_t pos = (h.lo + (uint64_t)j * h.hi) & (nbits - 1);
            // the entry's key carries the position's bit BEFORE the call in its top bit (the filter is not modified by this kernel, so every
            // inserter of a position builds the same key)
            const uint64_t was = (bits[pos >> 6] >> (pos & 63)) & 1ull;
            const uint64_t key = pos | (was << 63);
            uint64_t s = mix64(pos) & tmask;
            for (;;) {
                uint64_t cur = tkey[s];
                if (cur == kEmpty) cur = atomicCAS((unsigned long long *)&tkey[s], (unsigned long long)kEmpty, (unsigned long long)key);
                if (cur == kEmpty || cur == key) { atomicMin(&trow[s], (unsigned)i); break; }
                s = (s + 1) & tmask;
            }
        }
    }
}

__global__ void __launch_bounds__(256)
taa_finish_kernel(uint64_t *__restrict__ bits, uint64_t nbits, uint32_t k, uint64_t seed, KeySrc K, uint64_t nitem, const uint64_t *__restrict__ nullmap,
                  const uint64_t *__restrict__ tkey, const unsigned *__restrict__ trow, uint64_t tmask, uint8_t *__restrict__ result) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < nitem; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint8_t *p; uint64_t n;
        if (!key_of(K, i, &p, &n)) continue;
        if (nullmap && ((nullmap[i >> 6] >> (i & 63)) & 1ull)) { result[i] = 0; continue; }
        if (nbits == 0) { result[i] = 0; continue; }
        const xxh3::Hash128 h = key_hash(p, n, seed);
        bool all = true;
        for (uint32_t j = 0; j < k; j++) {
            const uint64_t pos = (h.lo + (uint64_t)j * h.hi) & (nbits - 1);
            uint64_t s = mix64(pos) & tmask;
            while ((tkey[s] & ~(1ull << 63)) != pos) s = (s + 1) & tmask;      // present: kernel 1 inserted it
            const bool was = tkey[s] >> 63;
            if (!was && !(trow[s] < (unsigned)i)) all = false;                    // nobody before row i had set it
            if (!was && trow[s] == (unsigned)i) atomicOr((unsigned long long *)&bits[pos >> 6], 1ull << (pos & 63));   // the first setter writes the bit
        }
        result[i] = all ? 1 : 0;
    }
}

__global__ void taa_init_kernel(uint64_t *tkey, unsigned *trow, uint64_t slots) {
    for (uint64_t s = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; s < slots; s += (uint64_t)gridDim.x * blockDim.x) { tkey[s] = kEmpty; trow[s] = 0xffffffffu; }
}

// offsets of a [u32 length][payload] stream (bloom.c:159-176): inherently sequential; one thread walks it (this format is not used by the Go side)
__global__ void walk_4b_kernel(const uint8_t *keys, uint64_t len, uint64_t nitem, uint64_t *offs) {
    if (blockIdx.x || threadIdx.x) return;
    uint64_t o = 0, i = 0;
    for (; i < nitem; i++) {
        if (o + 4 > len) break;
        const uint32_t n = xxh3::rd32(keys + o);
        o += 4;
        if (o + n > len) break;
        offs[i] = o;
        o += n;
    }
    for (; i < nitem; i++) offs[i] = ~0ull;
}

__global__ void or_kernel(uint64_t *d, const uint64_t *a, const uint64_t *b, uint64_t words) {
    for (uint64_t w = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < words; w += (uint64_t)gridDim.x * blockDim.x) d[w] = a[w] | b[w];
}

enum Op { OP_ADD = 0, OP_TEST = 1, OP_TAA = 2 };
enum Fmt { FMT_FIXED = 0, FMT_VARLENA = 1, FMT_4B = 2 };

void run(const char *what, int op, int fmt, const bloomfilter_t *bf, const void *key, size_t len, size_t elemsz, size_t nitem, const void *area, size_t area_len,
         const void *nullmap, void *result) {
    if (nitem == 0) return;
    ThreadCtx &t = tctx();
    if (!t.ready) bloom_fatal(what);
    if (memcmp(bf->magic, "XXBF", 4) != 0 || bf->k > (uint32_t)kMaxK) { set_error("bloom: not a filter (bad magic or k)"); bloom_fatal(what); }
    uint64_t *bits = mirror_of(t, bf, op != OP_TEST);
    if (!bits) bloom_fatal(what);
    Stager st(t);
    KeySrc K;
    memset(&K, 0, sizeof K);
    if (fmt == FMT_FIXED && len > elemsz * nitem) len = elemsz * nitem;
    if (fmt == FMT_VARLENA && len > elemsz * nitem) len = elemsz * nitem;
    K.keys = (const uint8_t *)st.in(key, len);
    K.len = len; K.elemsz = elemsz; K.varlena = fmt == FMT_VARLENA;
    if (fmt == FMT_VARLENA) { K.area = (const uint8_t *)st.in(area, area_len); K.area_len = area_len; }
    const uint64_t *nm = (const uint64_t *)st.in(nullmap, nullmap ? ((nitem + 63) / 64) * 8 : 0);
    uint8_t *res = op == OP_ADD ? nullptr : (uint8_t *)st.out(result, nitem, true);   // rows past the key buffer keep the caller's bytes
    unsigned grid = (unsigned)((nitem + 255) / 256);
    if (grid > (unsigned)num_sms() * 8) grid = (unsigned)num_sms() * 8;
    if (fmt == FMT_4B) {
        uint64_t *offs = (uint64_t *)st.tmp(nitem * 8);
        if (st.failed) { st.finish(); bloom_fatal(what); }
        walk_4b_kernel<<<1, 32, 0, t.stream>>>(K.keys, len, nitem, offs);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        K.offs = offs;
    }
    if (st.failed) { st.finish(); bloom_fatal(what); }
    cudaEventRecord(t.kev0, t.stream);
    if (op == OP_ADD) {
        bloom_kernel<0><<<grid, 256, 0, t.stream>>>(bits, bf->nbits, bf->k, bf->seed, K, nitem, nm, nullptr);
        g_launches.fetch_add(1, std::memory_order_relaxed);
    } else if (op == OP_TEST) {
        bloom_kernel<1><<<grid, 256, 0, t.stream>>>(bits, bf->nbits, bf->k, bf->seed, K, nitem, nm, res);
        g_launches.fetch_add(1, std::memory_order_relaxed);
    } else {
        uint64_t slots = 1024;
        while (slots < 2 * (uint64_t)nitem * (bf->k ? bf->k : 1)) slots <<= 1;
        uint64_t *tkey = (uint64_t *)st.tmp(slots * 8);
        unsigned *trow = (unsigned *)st.tmp(slots * 4);
        if (st.failed) { st.finish(); bloom_fatal(what); }
        taa_init_kernel<<<num_sms() * 4, 256, 0, t.stream>>>(tkey, trow, slots);
        taa_insert_kernel<<<grid, 256, 0, t.stream>>>(bits, bf->nbits, bf->k, bf->seed, K, nitem, nm, tkey, trow, slots - 1);
        taa_finish_kernel<<<grid, 256, 0, t.stream>>>(bits, bf->nbits, bf->k, bf->seed, K, nitem, nm, tkey, trow, slots - 1, res);
        g_launches.fetch_add(3, std::memory_order_relaxed);
    }
    cudaEventRecord(t.kev1, t.stream);
    if (cudaGetLastError() != cudaSuccess) { set_error("bloom: kernel launch failed"); st.finish(); bloom_fatal(what); }
    if (st.finish() != MO_RC_SUCCESS) bloom_fatal(what);
}

}  // namespace

// ---- the reference's symbols (cgo/bloom.h) -------------------------------------------------------------------------------------------------
extern "C" {

bloomfilter_t *bloomfilter_init_with_seed(uint64_t nbits, uint32_t k, uint64_t seed) {   // bloom.c:118-130
    const uint64_t nb = next_pow2_64(nbits);
    if (k > (uint32_t)kMaxK) return nullptr;
    const size_t nbytes = bitmap_words(nb) * 8;
    bloomfilter_t *bf = (bloomfilter_t *)malloc(sizeof(bloomfilter_t) + nbytes);
    if (!bf) return nullptr;
    memset(bf, 0, sizeof(bloomfilter_t) + nbytes);   // (the reference leaves the last 8 marshalled bytes -- past the bitmap -- uninitialised)
    memcpy(bf->magic, "XXBF", 4);
    bf->nbits = nb; bf->k = k; bf->seed = seed;
    {   // the allocator may hand out an address a mirror is still registered for (a buffer released without bloomfilter_free)
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_mirrors.find(bf);
        if (it != g_mirrors.end()) { if (it->second.dbits) cudaFree(it->second.dbits); g_mirrors.erase(it); }
    }
    return bf;
}

bloomfilter_t *bloomfilter_init(uint64_t nbits, uint32_t k) {   // bloom.c:98-116: a random 64-bit seed from four 16-bit draws
    uint64_t seed = 0;
    for (int j = 0; j < 4; j++) seed = (seed << 16) | (uint64_t)(rand() & 0xFFFF);
    return bloomfilter_init_with_seed(nbits, k, seed);
}

void bloomfilter_free(bloomfilter_t *bf) {
    if (!bf) return;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_mirrors.find(bf);
        if (it != g_mirrors.end()) { if (it->second.dbits) cudaFree(it->second.dbits); g_mirrors.erase(it); }
    }
    free(bf);
}

void bloomfilter_add(bloomfilter_t *bf, const void *key, size_t len) {   // one key = one variable-length row
    // a [u32 length][payload] stream of one row keeps arbitrary lengths exact (a fixed row of len 1/2/4/8 would be widened the same way: bloom_calculate_hash switches on len)
    std::vector<uint8_t> buf(4 + len);
    const uint32_t n = (uint32_t)len;
    memcpy(buf.data(), &n, 4);
    if (len) memcpy(buf.data() + 4, key, len);
    run("bloomfilter_add", OP_ADD, FMT_4B, bf, buf.data(), buf.size(), 0, 1, nullptr, 0, nullptr, nullptr);
}

bool bloomfilter_test(const bloomfilter_t *bf, const void *key, size_t len) {
    std::vector<uint8_t> buf(4 + len);
    const uint32_t n = (uint32_t)len;
    memcpy(buf.data(), &n, 4);
    if (len) memcpy(buf.data() + 4, key, len);
    uint8_t r = 0;
    run("bloomfilter_test", OP_TEST, FMT_4B, bf, buf.data(), buf.size(), 0, 1, nullptr, 0, nullptr, &r);
    return r != 0;
}

bool bloomfilter_test_and_add(bloomfilter_t *bf, const void *key, size_t len) {
    std::vector<uint8_t> buf(4 + len);
    const uint32_t n = (uint32_t)len;
    memcpy(buf.data(), &n, 4);
    if (len) memcpy(buf.data() + 4, key, len);
    uint8_t r = 0;
    run("bloomfilter_test_and_add", OP_TAA, FMT_4B, bf, buf.data(), buf.size(), 0, 1, nullptr, 0, nullptr, &r);
    return r != 0;
}

void bloomfilter_add_fixed(bloomfilter_t *bf, const void *key, size_t len, size_t elemsz, size_t nitem, const void *nullmap, size_t nullmaplen) {
    (void)nullmaplen;
    if (elemsz == 0) return;
    run("bloomfilter_add_fixed", OP_ADD, FMT_FIXED, bf, key, len, elemsz, nitem, nullptr, 0, nullmap, nullptr);
}
void bloomfilter_test_fixed(const bloomfilter_t *bf, const void *key, size_t len, size_t elemsz, size_t nitem, const void *nullmap, size_t nullmaplen, void *result) {
    (void)nullmaplen;
    if (elemsz == 0) return;
    run("bloomfilter_test_fixed", OP_TEST, FMT_FIXED, bf, key, len, elemsz, nitem, nullptr, 0, nullmap, result);
}
void bloomfilter_test_and_add_fixed(bloomfilter_t *bf, const void *key, size_t len, size_t elemsz, size_t nitem, const void *nullmap, size_t nullmaplen, void *result) {
    (void)nullmaplen;
    if (elemsz == 0) return;
    run("bloomfilter_test_and_add_fixed", OP_TAA, FMT_FIXED, bf, key, len, elemsz, nitem, nullptr, 0, nullmap, result);
}

void bloomfilter_add_varlena_4b(bloomfilter_t *bf, const void *key, size_t len, size_t nitem, const void *nullmap, size_t nullmaplen) {
    (void)nullmaplen;
    run("bloomfilter_add_varlena_4b", OP_ADD, FMT_4B, bf, key, len, 0, nitem, nullptr, 0, nullmap, nullptr);
}
void bloomfilter_test_varlena_4b(const bloomfilter_t *bf, const void *key, size_t len, size_t nitem, const void *nullmap, size_t nullmaplen, void *result) {
    (void)nullmaplen;
    run("bloomfilter_test_varlena_4b", OP_TEST, FMT_4B, bf, key, len, 0, nitem, nullptr, 0, nullmap, result);
}
void bloomfilter_test_and_add_varlena_4b(bloomfilter_t *bf, const void *key, size_t len, size_t nitem, const void *nullmap, size_t nullmaplen, void *result) {
    (void)nullmaplen;
    run("bloomfilter_test_and_add_varlena_4b", OP_TAA, FMT_4B, bf, key, len, 0, nitem, nullptr, 0, nullmap, result);
}

void bloomfilter_add_varlena(bloomfilter_t *bf, const void *keys, size_t len, size_t elemsz, size_t nitem, const void *area, size_t area_len, const void *nullmap, size_t nullmaplen) {
    (void)nullmaplen;
    if (elemsz < MO_VARLENA_SZ) return;
    run("bloomfilter_add_varlena", OP_ADD, FMT_VARLENA, bf, keys, len, elemsz, nitem, area, area_len, nullmap, nullptr);
}
void bloomfilter_test_varlena(const bloomfilter_t *bf, const void *keys, size_t len, size_t elemsz, size_t nitem, const void *area, size_t area_len, const void *nullmap, size_t nullmaplen, void *result) {
    (void)nullmaplen;
    if (elemsz < MO_VARLENA_SZ) return;
    run("bloomfilter_test_varlena", OP_TEST, FMT_VARLENA, bf, keys, len, elemsz, nitem, area, area_len, nullmap, result);
}
void bloomfilter_test_and_add_varlena(bloomfilter_t *bf, const void *keys, size_t len, size_t elemsz, size_t nitem, const void *area, size_t area_len, const void *nullmap, size_t nullmaplen, void *result) {
    (void)nullmaplen;
    if (elemsz < MO_VARLENA_SZ) return;
    run("bloomfilter_test_and_add_varlena", OP_TAA, FMT_VARLENA, bf, keys, len, elemsz, nitem, area, area_len, nullmap, result);
}

uint8_t *bloomfilter_marshal(const bloomfilter_t *bf, size_t *len) {   // bloom.c:321-328; the host bytes are refreshed from the mirror first
    if (memcmp(bf->magic, "XXBF", 4) != 0) { *len = 0; return nullptr; }
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_mirrors.find(bf);
        if (it != g_mirrors.end() && it->second.dev_newer && it->second.words) {
            if (cudaMemcpy(const_cast<uint64_t *>(bf->bitmap), it->second.dbits, it->second.words * 8, cudaMemcpyDeviceToHost) != cudaSuccess) {
                set_error("bloom: filter download failed");
                bloom_fatal("bloomfilter_marshal");
            }
            it->second.dev_newer = false;
        }
    }
    *len = sizeof(bloomfilter_t) + bitmap_words(bf->nbits) * 8;
    return (uint8_t *)bf;
}

bloomfilter_t *bloomfilter_unmarshal(const uint8_t *buf, size_t len) {   // bloom.c:330-339: adopts the buffer, no copy
    if (len < sizeof(bloomfilter_t)) return nullptr;
    bloomfilter_t *bf = (bloomfilter_t *)buf;
    if (memcmp(bf->magic, "XXBF", 4) != 0) return nullptr;
    {   // a buffer address may be reused by a new filter: forget a stale mirror
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_mirrors.find(bf);
        if (it != g_mirrors.end()) { if (it->second.dbits) cudaFree(it->second.dbits); g_mirrors.erase(it); }
    }
    return bf;
}

int bloomfilter_or(bloomfilter_t *dst, const bloomfilter_t *a, const bloomfilter_t *b) {   // bloom.c:341-357
    if (!(a->nbits == b->nbits && a->nbits == dst->nbits)) return 1;
    if (!(a->seed == b->seed && a->seed == dst->seed)) return 2;
    if (!(a->k == b->k && a->k == dst->k)) return 3;
    ThreadCtx &t = tctx();
    if (!t.ready) bloom_fatal("bloomfilter_or");
    const uint64_t *da = mirror_of(t, a, false), *db = mirror_of(t, b, false);
    uint64_t *dd = mirror_of(t, dst, true);
    if (!da || !db || !dd) bloom_fatal("bloomfilter_or");
    const uint64_t words = bitmap_words(dst->nbits);
    if (words) {
        unsigned grid = (unsigned)((words + 255) / 256);
        if (grid > (unsigned)num_sms() * 8) grid = (unsigned)num_sms() * 8;
        or_kernel<<<grid, 256, 0, t.stream>>>(dd, da, db, words);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(t.stream) != cudaSuccess) { set_error("bloom: or kernel failed"); bloom_fatal("bloomfilter_or"); }
    }
    return 0;
}

}  // extern "C"
