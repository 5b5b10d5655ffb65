/* oracle_strhash.c -- C restatement of the reference's StrHashMap key path (TEST INFRASTRUCTURE ONLY, never linked into the product):
 *
 *   og_pack_str_keys    strHashmapIterator.encodeHashKeys, pkg/common/hashmap/strhashmap.go:92-106, with fillGroupStr (:311-385) for fixed-width
 *                       columns and fillStringGroupStr / fillStringGroupStrForConstVec (:108-309) for varlena columns, padding to 16 bytes with
 *                       hashtable.StrKeyPadding (pkg/container/hashtable/string_hash_map.go:37)
 *   og_str_group_ids    strHashmapIterator.Insert (strhashmap.go, string_hash_map.go:97-158 InsertStringBatchWithRing): ids 1, 2, ... in
 *                       first-seen order, rows with zValues == 0 skipped; the table persists as offsets + bytes (key of group g at
 *                       bytes[offsets[g - 1] .. offsets[g]))
 *   og_str_join_find    strHashmapIterator.Find (string_hash_map.go FindStringBatch): the group id, 0 for an absent or skipped key
 *
 * The reference identifies a key by its 192-bit AES hash state; this restatement compares the key bytes, which gives the same ids.
 * Built by tests/oracle_lib.py (strhash()) with the flags of oracle/build.py.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static int bm(const uint64_t *b, int64_t i) { return b && ((b[i >> 6] >> (i & 63)) & 1u); }

/* varlena cell, pkg/container/types/bytes.go:61-115: c[0] <= 23 inline, else uint32 offset at +4 and length at +8 into the area */
static const uint8_t *cell_bytes(const uint8_t *c, const uint8_t *area, uint64_t *n) {
    if (c[0] <= 23) { *n = c[0]; return c + 1; }
    uint32_t off, len;
    memcpy(&off, c + 4, 4); memcpy(&len, c + 8, 4);
    *n = len;
    return area + off;
}

typedef struct { uint8_t *p; uint64_t n, cap; } buf_t;
static void put(buf_t *b, const void *src, uint64_t n) {
    if (b->n + n > b->cap) {
        while (b->n + n > b->cap) b->cap = b->cap ? 2 * b->cap : 256;
        b->p = (uint8_t *)realloc(b->p, b->cap);
    }
    if (n) memcpy(b->p + b->n, src, n);
    b->n += n;
}
static void put1(buf_t *b, uint8_t v) { put(b, &v, 1); }

/* returns the bytes needed; the bytes are written only when they fit in cap.  offsets int64[n + 1]; skip (may be NULL) gets a bit per row
 * with zValues == 0.  cols[k]: fixed-width values (width[k] bytes each) or 24-byte cells (width[k] == 0) with areas[k]; is_const[k]: one element. */
int64_t og_pack_str_keys(int32_t ncols, int32_t has_null, const int32_t *width, const void *const *cols, const void *const *areas, const void *const *nulls,
                         const int32_t *is_const, int64_t n, int64_t *offsets, uint8_t *out, int64_t cap, uint64_t *skip) {
    static const uint8_t pad[16] = {0};
    buf_t row = {0, 0, 0};
    int64_t pos = 0;
    if (skip) memset(skip, 0, (size_t)((n + 63) / 64) * 8);
    for (int64_t i = 0; i < n; i++) {
        row.n = 0;
        int zero = 0;
        for (int k = 0; k < ncols; k++) {
            const int64_t r = is_const[k] ? 0 : i;
            const uint64_t *nb = (const uint64_t *)nulls[k];
            if (bm(nb, r)) {                       /* NULL (a const NULL vector too): marker 1, or zValues[i] = 0 and nothing appended */
                if (has_null) put1(&row, 1); else zero = 1;
                continue;
            }
            if (width[k] > 0) {                    /* fillGroupStr */
                if (has_null) put1(&row, 0);
                put(&row, (const uint8_t *)cols[k] + r * width[k], (uint64_t)width[k]);
            } else {                               /* fillStringGroupStr: uint16 length (truncated), then every byte */
                uint64_t len;
                const uint8_t *b = cell_bytes((const uint8_t *)cols[k] + r * 24, (const uint8_t *)areas[k], &len);
                const uint16_t l16 = (uint16_t)len;
                if (has_null) put1(&row, 0);
                put(&row, &l16, 2);
                put(&row, b, len);
            }
        }
        if (row.n < 16) put(&row, pad, 16 - row.n);
        if (zero && skip) skip[i >> 6] |= 1ull << (i & 63);
        offsets[i] = pos;
        if (pos + (int64_t)row.n <= cap) memcpy(out + pos, row.p, row.n);
        pos += (int64_t)row.n;
    }
    offsets[n] = pos;
    free(row.p);
    return pos;
}

/* ---- exact string set: open addressing over FNV-1a, an entry is a 1-based group id ---- */
typedef struct { uint32_t *slot; uint64_t mask; } set_t;
static uint64_t fnv(const uint8_t *p, uint64_t n) {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t j = 0; j < n; j++) { h ^= p[j]; h *= 1099511628211ull; }
    return h ^ (h >> 29);
}
static void set_init(set_t *s, uint64_t items) {
    uint64_t sl = 64;
    while (sl < 2 * items) sl <<= 1;
    s->slot = (uint32_t *)calloc(sl, 4); s->mask = sl - 1;
}
typedef struct { const int64_t *off; const uint8_t *b; } keys_t;
/* slot of key (p, n): an existing group or the empty slot where it goes; the group of a slot g has its key at K(g) */
static uint64_t set_find(const set_t *s, const uint8_t *p, uint64_t n, const keys_t *t, const keys_t *extra, int64_t nt) {
    uint64_t i = fnv(p, n) & s->mask;
    for (;;) {
        const uint32_t g = s->slot[i];
        if (!g) return i;
        const keys_t *K = (int64_t)g <= nt ? t : extra;
        const int64_t gi = (int64_t)g <= nt ? g - 1 : g - 1 - nt;
        const uint64_t qn = (uint64_t)(K->off[gi + 1] - K->off[gi]);
        if (qn == n && memcmp(K->b + K->off[gi], p, n) == 0) return i;
        i = (i + 1) & s->mask;
    }
}

/* Insert: groups[i] = id of row i (0 = skipped).  The table holds ngroups keys on entry; on success it holds the new groups too and the new
 * count is returned.  When more than cap groups or byte_cap key bytes would be needed, the table is left unchanged, need = {groups, bytes}
 * and -1 is returned. */
int64_t og_str_group_ids(const int64_t *koff, const uint8_t *kbytes, const uint64_t *skip, int64_t n, uint64_t *groups, int64_t *toff, uint8_t *tbytes,
                         int64_t ngroups, int64_t cap, int64_t byte_cap, int64_t *need) {
    set_t s;
    set_init(&s, (uint64_t)(ngroups + n));
    const keys_t T = {toff, tbytes};
    int64_t *noff = (int64_t *)malloc((size_t)(n + 1) * 8);   /* the new groups' keys, appended after the table's */
    buf_t nb = {0, 0, 0};
    noff[0] = 0;
    keys_t N = {noff, NULL};
    for (int64_t g = 0; g < ngroups; g++) {
        const uint64_t i = set_find(&s, tbytes + toff[g], (uint64_t)(toff[g + 1] - toff[g]), &T, &N, ngroups);
        s.slot[i] = (uint32_t)(g + 1);
    }
    int64_t ng = ngroups, nnew = 0;
    for (int64_t r = 0; r < n; r++) {
        if (bm(skip, r)) { groups[r] = 0; continue; }
        const uint8_t *p = kbytes + koff[r];
        const uint64_t len = (uint64_t)(koff[r + 1] - koff[r]);
        N.b = nb.p;
        const uint64_t i = set_find(&s, p, len, &T, &N, ngroups);
        if (!s.slot[i]) {
            put(&nb, p, len);
            nnew++;
            noff[nnew] = (int64_t)nb.n;
            s.slot[i] = (uint32_t)(++ng);
        }
        groups[r] = s.slot[i];
    }
    const int64_t used = ngroups ? toff[ngroups] : 0;
    need[0] = ng; need[1] = used + (int64_t)nb.n;
    int64_t rc = ng;
    if (ng > cap || need[1] > byte_cap) rc = -1;
    else {
        toff[ngroups] = used;
        if (nb.n) memcpy(tbytes + used, nb.p, nb.n);
        for (int64_t j = 1; j <= nnew; j++) toff[ngroups + j] = used + noff[j];
    }
    free(nb.p); free(noff); free(s.slot);
    return rc;
}

/* Find: vals[i] = group id of probe key i, 0 when absent or skipped */
void og_str_join_find(const int64_t *toff, const uint8_t *tbytes, int64_t ngroups, const int64_t *koff, const uint8_t *kbytes, const uint64_t *skip,
                      int64_t n, uint64_t *vals) {
    set_t s;
    set_init(&s, (uint64_t)ngroups);
    const keys_t T = {toff, tbytes};
    for (int64_t g = 0; g < ngroups; g++) {
        const uint64_t i = set_find(&s, tbytes + toff[g], (uint64_t)(toff[g + 1] - toff[g]), &T, &T, ngroups);
        if (!s.slot[i]) s.slot[i] = (uint32_t)(g + 1);
    }
    for (int64_t r = 0; r < n; r++) {
        if (bm(skip, r)) { vals[r] = 0; continue; }
        vals[r] = s.slot[set_find(&s, kbytes + koff[r], (uint64_t)(koff[r + 1] - koff[r]), &T, &T, ngroups)];
    }
    free(s.slot);
}
