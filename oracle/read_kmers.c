/* TEST INFRASTRUCTURE -- CPU oracle of the read k-mer table (OpenMP).  PARITY UNPINNED.
 *
 * R1 of oracle.c without the restriction to the database: every canonical K-mer of the reads counted -- the whole
 * `kmc -k60 -ci2 -cs3` database (scripts/select_db.py:50-52 of the reference; reads_60mers.kmc_*) that the product's
 * read k-mer table (metalign_b200/csrc/readkmers.cu) writes.  Built differently from it on purpose: unsigned __int128
 * rolling k-mers, a host hash map claimed slot by slot with a state word, a bucketed qsort for the output.
 *
 * Only tests/ and scripts/bench_read_kmers.py load this library (oracle/read_kmers.py builds it).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <omp.h>

typedef unsigned __int128 u128;
#define ORC_API __attribute__((visibility("default")))

static inline uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33; return x;
}
static inline uint64_t hash128(u128 k) { return mix64((uint64_t)k ^ mix64((uint64_t)(k >> 64) + 0x632BE59BD9B4E019ull)); }

/* bucketed parallel sort: partition on the top 12 bits of a `bits`-wide key, qsort the buckets */
#define NBKT 4096
static void psort(void* base, uint64_t n, size_t sz, int (*cmp)(const void*, const void*), u128 (*keyof)(const void*), uint32_t bits) {
    if (n < (1u << 16) || bits < 12) { qsort(base, n, sz, cmp); return; }
    uint64_t* cnt = (uint64_t*)calloc(NBKT + 1, sizeof(uint64_t));
    char* src = (char*)base;
    uint32_t sh = bits - 12;
    for (uint64_t i = 0; i < n; ++i) cnt[(uint32_t)(keyof(src + i * sz) >> sh) + 1]++;
    for (uint32_t b = 0; b < NBKT; ++b) cnt[b + 1] += cnt[b];
    uint64_t* pos = (uint64_t*)malloc(NBKT * sizeof(uint64_t));
    memcpy(pos, cnt, NBKT * sizeof(uint64_t));
    char* tmp = (char*)malloc(n * sz);
    for (uint64_t i = 0; i < n; ++i) {
        uint32_t b = (uint32_t)(keyof(src + i * sz) >> sh);
        memcpy(tmp + pos[b]++ * sz, src + i * sz, sz);
    }
#pragma omp parallel for schedule(dynamic, 8)
    for (uint32_t b = 0; b < NBKT; ++b)
        qsort(tmp + cnt[b] * sz, cnt[b + 1] - cnt[b], sz, cmp);
    memcpy(base, tmp, n * sz);
    free(tmp); free(pos); free(cnt);
}

/* ---------------------------------------------------------------- R1': every read k-mer */
/* An open-addressing map from canonical key to count.  A slot is claimed by a CAS on its state word (0 empty, 1 being
 * written, 2 set); the map is resized between chunks of reads so that it stays at most 70 % full. */
typedef struct { uint64_t hi, lo; uint32_t count, state; } rkslot;
typedef struct orc_rk { uint32_t K; u128 mask; uint64_t cap, n; rkslot* s; } orc_rk;

static int rk_put(rkslot* s, uint64_t cap, u128 c, uint32_t add) {
    uint64_t h = hash128(c) & (cap - 1);
    const uint64_t hi = (uint64_t)(c >> 64), lo = (uint64_t)c;
    for (;;) {
        rkslot* x = &s[h];
        uint32_t st = __atomic_load_n(&x->state, __ATOMIC_ACQUIRE);
        if (st == 0) {
            uint32_t e = 0;
            if (__atomic_compare_exchange_n(&x->state, &e, 1u, 0, __ATOMIC_ACQ_REL, __ATOMIC_ACQUIRE)) {
                x->hi = hi; x->lo = lo; x->count = add;
                __atomic_store_n(&x->state, 2u, __ATOMIC_RELEASE);
                return 1;
            }
            st = e;
        }
        while (st == 1) st = __atomic_load_n(&x->state, __ATOMIC_ACQUIRE);
        if (x->hi == hi && x->lo == lo) { __atomic_fetch_add(&x->count, add, __ATOMIC_RELAXED); return 0; }
        h = (h + 1) & (cap - 1);
    }
}
static void rk_reserve(orc_rk* t, uint64_t more) {
    if ((double)(t->n + more) <= 0.7 * (double)t->cap) return;
    uint64_t cap = t->cap;
    while ((double)(t->n + more) > 0.7 * (double)cap) cap *= 2;
    rkslot* ns = (rkslot*)calloc(cap, sizeof(rkslot));
#pragma omp parallel for schedule(static)
    for (uint64_t i = 0; i < t->cap; ++i)
        if (t->s[i].state == 2) rk_put(ns, cap, (((u128)t->s[i].hi) << 64) | t->s[i].lo, t->s[i].count);
    free(t->s); t->s = ns; t->cap = cap;
}

ORC_API orc_rk* orc_rk_begin(uint32_t K) {
    if (K < 1 || K > 63) return NULL;
    orc_rk* t = (orc_rk*)calloc(1, sizeof(orc_rk));
    t->K = K; t->mask = (((u128)1) << (2 * K)) - 1; t->cap = 1u << 16;
    t->s = (rkslot*)calloc(t->cap, sizeof(rkslot));
    return t;
}
ORC_API void orc_rk_free(orc_rk* t) { if (t) { free(t->s); free(t); } }

#define RK_CHUNK (1u << 18)
/* same inputs as orc_query_push_ascii / orc_query_push_packed (text: off given; packed: off or fixed read_len) */
static void rk_push(orc_rk* t, const char* text, const uint8_t* bases, const uint8_t* nmask, const uint64_t* off, uint64_t nreads,
                    uint32_t read_len) {
    const uint32_t K = t->K; const u128 mask = t->mask;
    for (uint64_t r0 = 0; r0 < nreads; r0 += RK_CHUNK) {
        const uint64_t r1 = nreads - r0 < RK_CHUNK ? nreads : r0 + RK_CHUNK;
        const uint64_t b0 = off ? off[r0] : r0 * (uint64_t)read_len, b1 = off ? off[r1] : r1 * (uint64_t)read_len;
        rk_reserve(t, b1 - b0);                  /* windows <= bases */
        uint64_t added = 0;
#pragma omp parallel for schedule(dynamic, 256) reduction(+ : added)
        for (uint64_t r = r0; r < r1; ++r) {
            uint64_t p0 = off ? off[r] : r * (uint64_t)read_len, p1 = off ? off[r + 1] : (r + 1) * (uint64_t)read_len;
            u128 fwd = 0, rcv = 0; uint32_t run = 0;
            for (uint64_t p = p0; p < p1; ++p) {
                uint32_t b;
                if (text) {
                    switch (text[p]) {
                        case 'A': case 'a': b = 0; break;
                        case 'C': case 'c': b = 1; break;
                        case 'G': case 'g': b = 2; break;
                        case 'T': case 't': b = 3; break;
                        default: b = 4; break;
                    }
                } else {
                    b = (nmask && ((nmask[p >> 3] >> (7 - (p & 7))) & 1)) ? 4u : (bases[p >> 2] >> (6 - 2 * (p & 3))) & 3u;
                }
                if (b == 4) { run = 0; fwd = 0; rcv = 0; continue; }
                fwd = ((fwd << 2) | b) & mask;
                rcv = (rcv >> 2) | (((u128)(3u - b)) << (2 * (K - 1)));
                if (++run >= K) added += rk_put(t->s, t->cap, fwd < rcv ? fwd : rcv, 1);
            }
        }
        t->n += added;
    }
}
ORC_API void orc_rk_push_ascii(orc_rk* t, const char* text, const uint64_t* off, uint64_t nreads) {
    rk_push(t, text, NULL, NULL, off, nreads, 0);
}
ORC_API void orc_rk_push_packed(orc_rk* t, const uint8_t* bases, const uint8_t* nmask, const uint64_t* off, uint64_t nreads,
                                uint32_t read_len) {
    rk_push(t, NULL, bases, nmask, off, nreads, read_len);
}

typedef struct { u128 key; uint32_t count; } rkrec;
static int cmp_rkrec(const void* a, const void* b) {
    u128 x = ((const rkrec*)a)->key, y = ((const rkrec*)b)->key; return x < y ? -1 : (x > y);
}
static u128 keyof_rkrec(const void* p) { return ((const rkrec*)p)->key; }
ORC_API uint64_t orc_rk_distinct(const orc_rk* t) { return t->n; }
/* the keys counted >= min_count times, ascending, as (hi, lo) pairs with their counts saturated at counter_max; returns
 * their number (writes at most cap) */
ORC_API uint64_t orc_rk_result(const orc_rk* t, uint32_t min_count, uint32_t counter_max, uint64_t* keys, uint8_t* counts,
                               uint64_t cap) {
    rkrec* v = (rkrec*)malloc((t->n ? t->n : 1) * sizeof(rkrec));
    uint64_t m = 0;
    for (uint64_t i = 0; i < t->cap; ++i)
        if (t->s[i].state == 2 && t->s[i].count >= min_count) {
            v[m].key = (((u128)t->s[i].hi) << 64) | t->s[i].lo; v[m].count = t->s[i].count; m++;
        }
    psort(v, m, sizeof(rkrec), cmp_rkrec, keyof_rkrec, 2 * t->K);
    for (uint64_t i = 0; i < m && i < cap; ++i) {
        keys[2 * i] = (uint64_t)(v[i].key >> 64); keys[2 * i + 1] = (uint64_t)v[i].key;
        counts[i] = (uint8_t)(v[i].count < counter_max ? v[i].count : counter_max);
    }
    free(v);
    return m;
}
