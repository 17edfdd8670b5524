// Read k-mer table (include/metalign_b200.h, mlg_query_enable_read_kmers): every canonical K-mer (K <= 60) of the pushed
// reads with a saturating 8-bit count -- the counting part of `kmc -k<K> -ci<min> -cs<max>` -- and the KMC database files
// written from it and from the query's intersection.  The count kernel runs beside K1 on the compute stream, over the same
// staged batch; K1 itself does not know the table exists.  The key-range mode (mlg_query_enable_read_kmer_passes, at the
// end of this file) counts a device copy of the reads at output time instead, one interval of the key order per pass.
// DESIGN.md section 10.
#include <cub/cub.cuh>
#include <errno.h>
#include <fcntl.h>
#include <stdio.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <chrono>
#include <deque>
#include <functional>
#include "mlg_internal.h"

namespace {

constexpr int RK_TPB = 256;                             // windows per tile == threads per CTA
constexpr unsigned long long CNT_ONE = 1ull << 56;      // count in the top byte of hi; the key lives in the low 2K <= 120 bits
constexpr unsigned long long KEY_HI = CNT_ONE - 1;
constexpr double RK_LOAD = 0.7;
constexpr unsigned long long RK_MIN_SLOTS = 1ull << 12;

// one 16-byte slot, laid out as the unsigned __int128 (lo, hi) the CAS works on; all zero = empty (a stored count is >= 1)
struct __align__(16) Slot { unsigned long long lo, hi; };

__host__ __device__ __forceinline__ unsigned long long rk_hash(unsigned long long hi, unsigned long long lo) {
    unsigned long long x = lo ^ (hi * 0x9E3779B97F4A7C15ull);
    x ^= x >> 32; x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32; x *= 0xD6E8FEB86659FD93ull;
    return x ^ (x >> 32);
}

// 64-bit word w of a packed stream with the first byte in the top bits (words past the buffer read as 0)
__device__ __forceinline__ unsigned long long be_word(const unsigned long long* p, unsigned long long w, unsigned long long n) {
    if (w >= n) return 0ull;
    const unsigned long long x = p[w];
    return ((unsigned long long)__byte_perm((unsigned)x, 0, 0x0123) << 32) | __byte_perm((unsigned)(x >> 32), 0, 0x0123);
}

// saturating +1 on the count byte; h = a value of the slot's hi word seen before (possibly stale)
__device__ __forceinline__ void bump(Slot* s, unsigned long long h) {
    while ((h >> 56) < 255ull) {
        const unsigned long long old = atomicCAS(&s->hi, h, h + CNT_ONE);
        if (old == h) return;
        h = old;
    }
}

// Open addressing over 128-byte lines of 8 slots: start at a hashed slot of a hashed line, go round the line, then on to
// the next line.  Only the 8-byte hi word is read plainly (it cannot tear, and its key bits never change once set) and
// only to pass by slots of other keys; whether the slot is empty, ours or someone else's is decided from what the 16-byte
// CAS returns, or from a non-zero lo word (lo is written once, from 0, by that CAS).  Returns 1 when the key was new.
__device__ __forceinline__ int rk_insert(Slot* tab, unsigned long long line_mask, unsigned long long khi, unsigned long long klo,
                                         unsigned long long* full) {
    const unsigned long long h = rk_hash(khi, klo);
    unsigned long long line = h & line_mask;
    const unsigned s0 = (unsigned)(h >> 61);
    const unsigned __int128 mine = ((unsigned __int128)(khi | CNT_ONE) << 64) | klo;
    for (unsigned long long n = 0; n <= line_mask; ++n, line = (line + 1) & line_mask) {
        for (unsigned i = 0; i < 8; ++i) {
            Slot* s = tab + line * 8 + ((s0 + i) & 7u);
            const unsigned long long sh = __ldcg(&s->hi);
            if (sh != 0 && (sh & KEY_HI) != khi) continue;
            if (sh != 0) {
                const unsigned long long sl = __ldcg(&s->lo);
                if (sl != 0) {
                    if (sl != klo) continue;
                    bump(s, sh);
                    return 0;
                }
            }
            const unsigned __int128 old = atomicCAS(reinterpret_cast<unsigned __int128*>(s), (unsigned __int128)0, mine);
            if (old == 0) return 1;
            const unsigned long long oh = (unsigned long long)(old >> 64);
            if ((oh & KEY_HI) == khi && (unsigned long long)old == klo) { bump(s, oh); return 0; }
        }
    }
    atomicOr(full, 1ull);          // cannot happen below the load bound; recorded instead of looping forever
    return 0;
}

struct CountArgs {
    const unsigned long long* bases; const unsigned long long* nmask; const unsigned long long* off;
    uint32_t read_len, K;
    unsigned long long base_words, nmask_words, r_begin, r_end;
    Slot* tab; unsigned long long line_mask;
    unsigned long long* ctr;       // [0] distinct keys, [1] windows counted, [2] table full
    key128 range_lo, range_hi;     // ranged count (key-range passes): only the keys in [range_lo, range_hi)
};

// Window enumeration, shared by the count and the histogram kernels.  A CTA takes the 256 consecutive base positions
// from p0; the thread at p = p0 + threadIdx.x gets the canonical key of the window starting there when that window lies
// inside one read and holds no N.  The read of a position is found by a binary search inside the few reads the tile
// spans.  ok = whether there is such a window; the result is on_key(key) for it, 0 without one.  Every thread of the CTA
// calls tile_window (it holds a barrier), and the caller puts a barrier between two calls: s_r is read after the first.
template <class F>
__device__ __forceinline__ int tile_window(const CountArgs& a, unsigned K, unsigned long long p0, unsigned long long b1,
                                           unsigned long long* s_r, bool& ok_out, F&& on_key) {
    const unsigned long long p = p0 + threadIdx.x;
    if (a.off && threadIdx.x < 2) {            // reads holding the tile's first and last position
        const unsigned long long q = threadIdx.x ? min(p0 + RK_TPB - 1, b1 - 1) : p0;
        unsigned long long lo = a.r_begin, hi = a.r_end;      // last read r with off[r] <= q
        while (hi - lo > 1) { const unsigned long long m = (lo + hi) / 2; if (a.off[m] <= q) lo = m; else hi = m; }
        s_r[threadIdx.x] = lo;
    }
    __syncthreads();
    bool ok = p + K <= b1;
    if (ok) {
        unsigned long long end;
        if (a.off) {
            unsigned long long lo = s_r[0], hi = s_r[1] + 1;
            while (hi - lo > 1) { const unsigned long long m = (lo + hi) / 2; if (a.off[m] <= p) lo = m; else hi = m; }
            end = a.off[lo + 1];
        } else {
            end = (p / a.read_len + 1) * (unsigned long long)a.read_len;
        }
        ok = p + K <= end;
    }
    if (ok && a.nmask) {
        const unsigned long long w = p >> 6; const unsigned b = (unsigned)(p & 63);
        unsigned long long m = be_word(a.nmask, w, a.nmask_words) << b;
        if (b) m |= be_word(a.nmask, w + 1, a.nmask_words) >> (64 - b);
        ok = (m >> (64 - K)) == 0;
    }
    int r = 0;
    if (ok) {
        const unsigned long long w = p >> 5; const unsigned b = (unsigned)(p & 31) * 2;
        const unsigned long long x = be_word(a.bases, w, a.base_words), y = be_word(a.bases, w + 1, a.base_words),
                                 z = be_word(a.bases, w + 2, a.base_words);
        key128 t;
        t.hi = b ? (x << b) | (y >> (64 - b)) : x;
        t.lo = b ? (y << b) | (z >> (64 - b)) : y;
        r = on_key(key_canon(key_shr(t, 128 - 2 * K), K));
    }
    ok_out = ok;
    return r;
}

// One thread per window start, so the work is the same per window whatever the read lengths are.  RANGED: only the keys
// in [a.range_lo, a.range_hi) go into the table (one pass of the key-range mode); the push-time table counts every key.
template <bool RANGED>
__global__ void __launch_bounds__(RK_TPB) k_count_read_kmers(CountArgs a) {
    __shared__ unsigned long long s_r[2];
    const unsigned long long b0 = a.off ? a.off[a.r_begin] : a.r_begin * (unsigned long long)a.read_len;
    const unsigned long long b1 = a.off ? a.off[a.r_end] : a.r_end * (unsigned long long)a.read_len;
    const unsigned K = a.K;
    unsigned long long n_new = 0, n_win = 0;
    for (unsigned long long p0 = b0 + (unsigned long long)blockIdx.x * RK_TPB; p0 < b1; p0 += (unsigned long long)gridDim.x * RK_TPB) {
        bool ok;
        const int fresh = tile_window(a, K, p0, b1, s_r, ok, [&](const key128& c) {
            return (!RANGED || (!key_lt(c, a.range_lo) && key_lt(c, a.range_hi))) ? rk_insert(a.tab, a.line_mask, c.hi, c.lo, a.ctr + 2) : 0;
        });
        const int nf = __syncthreads_count(fresh), nw = __syncthreads_count(ok);
        n_new += nf; n_win += nw;
    }
    if (threadIdx.x == 0 && (n_new | n_win)) { atomicAdd(a.ctr, n_new); atomicAdd(a.ctr + 1, n_win); }
}

// Windows per bin of the key space: the canonical keys c whose leading bases equal `prefix` (c >> pshift == prefix;
// pshift = 2K takes every key) are binned by the bits below it, bins[(c >> shift) & mask]
__global__ void __launch_bounds__(RK_TPB) k_kmer_histogram(CountArgs a, unsigned pshift, key128 prefix, unsigned shift,
                                                            unsigned long long mask, unsigned long long* bins) {
    __shared__ unsigned long long s_r[2];
    const unsigned long long b0 = a.off ? a.off[a.r_begin] : a.r_begin * (unsigned long long)a.read_len;
    const unsigned long long b1 = a.off ? a.off[a.r_end] : a.r_end * (unsigned long long)a.read_len;
    for (unsigned long long p0 = b0 + (unsigned long long)blockIdx.x * RK_TPB; p0 < b1; p0 += (unsigned long long)gridDim.x * RK_TPB) {
        bool ok;
        tile_window(a, a.K, p0, b1, s_r, ok, [&](const key128& c) {
            if (key_eq(key_shr(c, pshift), prefix)) atomicAdd(bins + (key_shr(c, shift).lo & mask), 1ull);
            return 0;
        });
        __syncthreads();        // every thread is done with s_r before the next tile overwrites it (the count kernel's
                                // __syncthreads_count calls do this there)
    }
}

__global__ void k_rehash(const Slot* from, unsigned long long n_from, Slot* to, unsigned long long line_mask, unsigned long long* full) {
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n_from; i += (unsigned long long)gridDim.x * blockDim.x) {
        const Slot v = from[i];
        if (!v.hi) continue;
        const unsigned long long h = rk_hash(v.hi & KEY_HI, v.lo);
        unsigned long long line = h & line_mask;
        const unsigned s0 = (unsigned)(h >> 61);
        const unsigned __int128 val = ((unsigned __int128)v.hi << 64) | v.lo;
        bool done = false;
        for (unsigned long long n = 0; n <= line_mask && !done; ++n, line = (line + 1) & line_mask)
            for (unsigned j = 0; j < 8 && !done; ++j) {
                Slot* s = to + line * 8 + ((s0 + j) & 7u);
                if (__ldcg(&s->hi)) continue;
                done = atomicCAS(reinterpret_cast<unsigned __int128*>(s), (unsigned __int128)0, val) == 0;
            }
        if (!done) atomicOr(full, 1ull);
    }
}

struct AtLeast {
    unsigned long long min_count;
    __host__ __device__ bool operator()(const Slot& s) const { return (s.hi >> 56) >= min_count; }
};
__global__ void k_split_slots(const Slot* s, uint32_t n, unsigned long long* hi, unsigned long long* lo, uint32_t* cnt) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    hi[i] = s[i].hi & KEY_HI; lo[i] = s[i].lo; cnt[i] = (uint32_t)(s[i].hi >> 56);
}
__global__ void k_split_keys(const key128* k, const unsigned char* c8, uint32_t n, unsigned long long* hi, unsigned long long* lo, uint32_t* cnt) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    hi[i] = k[i].hi; lo[i] = k[i].lo; cnt[i] = c8[i];
}
// KMC prefix table of sorted keys: lut[i] = records before prefix i (the exclusive scan of the prefix histogram, read off
// the sorted order by a lower bound per prefix); lut[4^p] = n
__global__ void k_kmc_lut(const key128* keys, uint32_t n, uint32_t K, uint32_t p, unsigned long long* lut) {
    const unsigned long long np = 1ull << (2 * p);
    const unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (i > np) return;
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t m = (lo + hi) / 2;
        if (key_shr(keys[m], 2 * (K - p)).lo < i) lo = m + 1; else hi = m;
    }
    lut[i] = lo;
}
// .kmc_suf records: (K - p) / 4 suffix bytes, first base in the top bits, then one count byte
__global__ void k_kmc_records(const key128* keys, const uint32_t* cnt, uint32_t n, uint32_t K, uint32_t p, uint32_t counter_max,
                              unsigned char* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t sb = (K - p) / 4, rec = sb + 1;
    const key128 k = keys[i];
    unsigned char* o = out + (unsigned long long)i * rec;
    for (uint32_t j = 0; j < sb; ++j) o[j] = (unsigned char)key_shr(k, 8 * (sb - 1 - j)).lo;
    o[sb] = (unsigned char)min(cnt[i], counter_max);
}

// slots of a table that holds b keys at <= RK_LOAD (a power of two: the probe masks the hash)
inline unsigned long long slots_for(unsigned long long b) { unsigned long long s = RK_MIN_SLOTS; while ((double)s * RK_LOAD < (double)b) s *= 2; return s; }

inline unsigned grid_for(unsigned long long n, int cap) { return (unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>((n + RK_TPB - 1) / RK_TPB, (unsigned long long)cap)); }

}  // namespace

struct ReadKmerTable {
    mlg_ctx* ctx = nullptr;
    uint32_t K = 0;
    unsigned long long budget = 0;
    DevBuf<Slot> tab, retired;               // retired: the table before the last rehash, freed once the rehash has run
    cudaEvent_t retired_ev = nullptr;
    unsigned long long nslots = 0;
    DevBuf<unsigned long long> ctr;          // [0] distinct keys, [1] windows counted, [2] a probe found the table full
    unsigned long long* occ = nullptr;       // pinned: [s] = distinct keys after the last batch of staging set s
    cudaEvent_t occ_ev[2] = {nullptr, nullptr};
    unsigned long long occ_w[2] = {0, 0};    // windows bound pushed up to that copy
    unsigned long long windows_bound = 0, known_occ = 0, known_w = 0;
    bool overflowed = false;
    unsigned long long bytes_needed = 0;
    uint32_t grows = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> count_ev, rehash_ev;
    ~ReadKmerTable() {
        for (auto& e : count_ev) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
        for (auto& e : rehash_ev) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
        for (auto& e : occ_ev) if (e) cudaEventDestroy(e);
        if (retired_ev) cudaEventDestroy(retired_ev);
        if (occ) cudaFreeHost(occ);
    }
};

int rk_create(mlg_ctx* ctx, uint32_t K, unsigned long long max_table_bytes, ReadKmerTable** out) {
    if (K < 1 || K > 60) { mlg_set_error("the read k-mer table needs K <= 60 (the count lives in the top byte of the key); this database has K = %u", K); return MLG_ERR_ARG; }
    ReadKmerTable* t = new ReadKmerTable();
    t->ctx = ctx; t->K = K; t->budget = max_table_bytes;
    int rc = t->ctr.alloc(4);
    if (rc == MLG_OK && (cudaMemsetAsync(t->ctr.p, 0, 32, ctx->s_comp) != cudaSuccess || cudaMallocHost(&t->occ, 16) != cudaSuccess ||
                         cudaEventCreateWithFlags(&t->occ_ev[0], cudaEventDisableTiming) != cudaSuccess ||
                         cudaEventCreateWithFlags(&t->occ_ev[1], cudaEventDisableTiming) != cudaSuccess ||
                         cudaEventCreateWithFlags(&t->retired_ev, cudaEventDisableTiming) != cudaSuccess)) {
        mlg_set_error("read k-mer table set-up failed: %s", cudaGetErrorString(cudaGetLastError())); rc = MLG_ERR_CUDA;
    }
    if (rc != MLG_OK) { delete t; return rc; }
    *out = t;
    return MLG_OK;
}
void rk_destroy(ReadKmerTable* t) { delete t; }

static void rk_overflow(ReadKmerTable* t, unsigned long long bytes) {
    t->overflowed = true; t->bytes_needed = bytes;
    t->tab.release(); t->retired.release(); t->nslots = 0;
}

// Growth, without a host sync on the common path: the distinct keys cannot exceed the last occupancy the host has seen
// plus every window pushed since (the windows of this batch included).  When that bound passes the load limit the table
// is rehashed into one at least twice as large on the compute stream.  Only a table that would pass the byte budget looks
// at the exact occupancy (one join) before it gives up.
int rk_before_batch(ReadKmerTable* t, unsigned long long batch_windows, uint32_t* launches) {
    if (t->overflowed) return MLG_OK;
    cudaStream_t st = t->ctx->s_comp;
    for (int s = 0; s < 2; ++s)
        if (t->occ_w[s] > t->known_w && cudaEventQuery(t->occ_ev[s]) == cudaSuccess) { t->known_occ = t->occ[s]; t->known_w = t->occ_w[s]; }
    cudaGetLastError();
    if (t->retired.p && cudaEventQuery(t->retired_ev) == cudaSuccess) t->retired.release();
    cudaGetLastError();
    t->windows_bound += batch_windows;
    unsigned long long bound = t->known_occ + (t->windows_bound - t->known_w);
    if ((double)bound <= RK_LOAD * (double)t->nslots) return MLG_OK;
    unsigned long long want = std::max(slots_for(bound), 2 * t->nslots);
    if (t->budget && want * sizeof(Slot) > t->budget) {
        unsigned long long occ = 0;
        CUDA_TRY(cudaMemcpyAsync(t->occ, t->ctr.p, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        occ = t->occ[0];
        t->known_occ = occ; t->known_w = t->windows_bound - batch_windows;
        bound = occ + batch_windows;
        if ((double)bound <= RK_LOAD * (double)t->nslots) return MLG_OK;
        want = slots_for(bound);
        if (want * sizeof(Slot) > t->budget) { rk_overflow(t, want * sizeof(Slot)); return MLG_OK; }
    }
    if (t->retired.p) { CUDA_TRY(cudaEventSynchronize(t->retired_ev)); t->retired.release(); }
    DevBuf<Slot> nt;
    if (nt.alloc(want) != MLG_OK) {
        CUDA_TRY(cudaStreamSynchronize(st));          // the old table may still be counted into: join before it is freed
        rk_overflow(t, want * sizeof(Slot));
        return MLG_OK;
    }
    CUDA_TRY(cudaMemsetAsync(nt.p, 0, want * sizeof(Slot), st));
    if (t->nslots) {
        cudaEvent_t e0, e1;
        CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
        CUDA_TRY(cudaEventRecord(e0, st));
        k_rehash<<<grid_for(t->nslots, t->ctx->sm_count * 8), RK_TPB, 0, st>>>(t->tab.p, t->nslots, nt.p, want / 8 - 1, t->ctr.p + 2);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(e1, st));
        t->rehash_ev.emplace_back(e0, e1);
        t->grows += 1; *launches += 1;
        std::swap(t->retired.p, t->tab.p); std::swap(t->retired.n, t->tab.n);
        CUDA_TRY(cudaEventRecord(t->retired_ev, st));
    }
    t->tab.release();
    std::swap(t->tab.p, nt.p); std::swap(t->tab.n, nt.n);
    t->nslots = want;
    return MLG_OK;
}

int rk_count_range(ReadKmerTable* t, const ProbeArgs& pa, unsigned long long batch_bases, uint32_t* launches) {
    if (t->overflowed || !t->nslots) return MLG_OK;       // no table yet: the batch has no window
    cudaStream_t st = t->ctx->s_comp;
    CountArgs a{};
    a.bases = pa.bases; a.nmask = pa.nmask; a.off = pa.off; a.read_len = pa.read_len; a.K = t->K;
    a.base_words = pa.base_words; a.nmask_words = pa.nmask_words; a.r_begin = pa.r_begin; a.r_end = pa.r_end;
    a.tab = t->tab.p; a.line_mask = t->nslots / 8 - 1; a.ctr = t->ctr.p;
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, st));
    k_count_read_kmers<false><<<grid_for(batch_bases, t->ctx->sm_count * 16), RK_TPB, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(e1, st));
    t->count_ev.emplace_back(e0, e1);
    *launches += 1;
    return MLG_OK;
}

// the occupancy after this batch, copied to a pinned word for the next batch's bound (staging set s: the copy of the
// batch before on the same set has long been consumed)
int rk_after_batch(ReadKmerTable* t, int s) {
    if (t->overflowed) return MLG_OK;
    cudaStream_t st = t->ctx->s_comp;
    CUDA_TRY(cudaMemcpyAsync(t->occ + s, t->ctr.p, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(t->occ_ev[s], st));
    t->occ_w[s] = t->windows_bound;
    return MLG_OK;
}

int rk_check(ReadKmerTable* t) {
    if (t->overflowed) {
        mlg_set_error("the read k-mer table outgrew its budget: %llu bytes needed, %llu allowed", t->bytes_needed, t->budget);
        return MLG_ERR_NOMEM;
    }
    unsigned long long full = 0;
    CUDA_TRY(cudaStreamSynchronize(t->ctx->s_copy));
    CUDA_TRY(cudaMemcpyAsync(&full, t->ctr.p + 2, 8, cudaMemcpyDeviceToHost, t->ctx->s_comp));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->s_comp));
    if (t->retired.p) t->retired.release();
    if (full) { mlg_set_error("read k-mer table: a key found no free slot"); return MLG_ERR_STATE; }
    return MLG_OK;
}

int rk_stats(ReadKmerTable* t, mlg_read_kmer_stats* o) {
    unsigned long long c[2] = {0, 0};
    CUDA_TRY(cudaStreamSynchronize(t->ctx->s_copy));
    CUDA_TRY(cudaMemcpyAsync(c, t->ctr.p, 16, cudaMemcpyDeviceToHost, t->ctx->s_comp));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->s_comp));
    memset(o, 0, sizeof(*o));
    o->windows = c[1]; o->distinct = c[0]; o->slots = t->nslots; o->bytes = t->nslots * sizeof(Slot);
    o->bytes_needed = t->bytes_needed; o->grows = t->grows; o->overflowed = t->overflowed ? 1 : 0;
    float ms = 0;
    for (auto& e : t->count_ev) if (cudaEventElapsedTime(&ms, e.first, e.second) == cudaSuccess) o->ms_count += ms;
    for (auto& e : t->rehash_ev) if (cudaEventElapsedTime(&ms, e.first, e.second) == cudaSuccess) o->ms_rehash += ms;
    return MLG_OK;
}

// the keys of a table seen >= min_count times, sorted, with their counts (saturated at 255); *distinct_out = the keys in it
static int collect_slots(mlg_ctx* ctx, const Slot* tab, unsigned long long nslots, const unsigned long long* d_distinct, uint32_t K,
                         uint32_t min_count, DevBuf<key128>& keys, DevBuf<uint32_t>& cnt, uint32_t* n_out, KmcOutStats* ws,
                         unsigned long long* distinct_out = nullptr) {
    cudaStream_t st = ctx->s_comp;
    cudaEvent_t e0, e1, e2;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1)); CUDA_TRY(cudaEventCreate(&e2));
    struct Ev { cudaEvent_t* e; ~Ev() { for (int i = 0; i < 3; ++i) cudaEventDestroy(e[i]); } };
    cudaEvent_t evs[3] = {e0, e1, e2}; Ev guard{evs};
    CUDA_TRY(cudaEventRecord(e0, st));
    unsigned long long distinct = 0;
    CUDA_TRY(cudaMemcpyAsync(&distinct, d_distinct, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (distinct_out) *distinct_out = distinct;
    if (distinct >= (1ull << 32)) { mlg_set_error("%llu distinct read k-mers: more than the output stage sorts (2^32)", distinct); return MLG_ERR_ARG; }
    DevBuf<Slot> sel; MLG_TRY(sel.alloc(distinct));
    DevBuf<unsigned long long> d_n; MLG_TRY(d_n.alloc(1));
    unsigned long long n = 0;
    const unsigned long long CH = 1ull << 30;                 // cub's item count is an int
    for (unsigned long long s0 = 0; s0 < nslots; s0 += CH) {
        const int m = (int)std::min(CH, nslots - s0);
        size_t tb = 0;
        CUDA_TRY(cub::DeviceSelect::If(nullptr, tb, tab + s0, sel.p + n, d_n.p, m, AtLeast{min_count}, st));
        DevBuf<unsigned char> tmp; MLG_TRY(tmp.alloc(tb ? tb : 1));
        CUDA_TRY(cub::DeviceSelect::If(tmp.p, tb, tab + s0, sel.p + n, d_n.p, m, AtLeast{min_count}, st));
        unsigned long long got = 0;
        CUDA_TRY(cudaMemcpyAsync(&got, d_n.p, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        n += got;
    }
    CUDA_TRY(cudaEventRecord(e1, st));
    *n_out = (uint32_t)n;
    if (n) {
        DevBuf<unsigned long long> hi, lo; DevBuf<uint32_t> c;
        MLG_TRY(hi.alloc(n)); MLG_TRY(lo.alloc(n)); MLG_TRY(c.alloc(n));
        k_split_slots<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(sel.p, (uint32_t)n, hi.p, lo.p, c.p);
        sel.release();
        MLG_TRY(keys.alloc(n)); MLG_TRY(cnt.alloc(n));
        MLG_TRY(sort_keys128(hi.p, lo.p, c.p, (uint32_t)n, K, keys.p, cnt.p, st));
    }
    CUDA_TRY(cudaEventRecord(e2, st));
    CUDA_TRY(cudaEventSynchronize(e2));
    float ms = 0;
    if (ws && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) ws->ms_compact += ms;
    if (ws && cudaEventElapsedTime(&ms, e1, e2) == cudaSuccess) ws->ms_sort += ms;
    return MLG_OK;
}

int rk_collect(ReadKmerTable* t, uint32_t min_count, DevBuf<key128>& keys, DevBuf<uint32_t>& cnt, uint32_t* n_out, KmcOutStats* ws) {
    return collect_slots(t->ctx, t->tab.p, t->nslots, t->ctr.p, t->K, min_count, keys, cnt, n_out, ws);
}

int rk_sort_pairs(mlg_ctx* ctx, const key128* k, const unsigned char* c8, uint32_t n, uint32_t K, DevBuf<key128>& keys, DevBuf<uint32_t>& cnt) {
    if (!n) return MLG_OK;
    cudaStream_t st = ctx->s_comp;
    DevBuf<unsigned long long> hi, lo; DevBuf<uint32_t> c;
    MLG_TRY(hi.alloc(n)); MLG_TRY(lo.alloc(n)); MLG_TRY(c.alloc(n));
    k_split_keys<<<(n + 255) / 256, 256, 0, st>>>(k, c8, n, hi.p, lo.p, c.p);
    MLG_TRY(keys.alloc(n)); MLG_TRY(cnt.alloc(n));
    return sort_keys128(hi.p, lo.p, c.p, n, K, keys.p, cnt.p, st);
}

// KMC's prefix length for a k: the smallest p >= 4 (p >= 1 below k = 8) with a whole number of suffix bytes
static uint32_t kmc_prefix_len(uint32_t K) {
    uint32_t p = K > 8 ? 4 : (K > 4 ? K - 4 : 1);
    while ((K - p) % 4) ++p;
    return p;
}

// <prefix>.kmc_pre / .kmc_suf, version-0 layout (one sorted table, as kmc_tools writes it), written as a sequence of sorted
// chunks whose keys ascend from one chunk to the next: kmc_begin opens the suffix file, every kmc_append packs one chunk's
// records on the device (counts saturated at counter_max), copies them back in pieces through two pinned buffers, each
// piece's fwrite overlapping the next piece's copy, and adds the chunk's prefix table into the running one; kmc_end writes
// the prefix file.  One chunk gives the files of one sorted table.  A writer that does not reach the end of kmc_end
// removes both files.
struct KmcWriter {
    mlg_ctx* ctx = nullptr;
    std::string pre_path, suf_path;
    uint32_t K = 0, p = 0, rec = 0, min_count = 0, counter_max = 0;
    FILE* fs = nullptr;
    bool ok = true;
    std::vector<unsigned long long> lut;     // records before each prefix, summed over the chunks; lut[4^p] = records
    unsigned long long records = 0, sbytes = 0;
    unsigned char* pin[2] = {nullptr, nullptr};
    unsigned long long pin_bytes = 0;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    KmcOutStats* ws = nullptr;
    bool created = false, finished = false;
    ~KmcWriter() {
        if (fs) fclose(fs);
        for (int i = 0; i < 2; ++i) { if (pin[i]) cudaFreeHost(pin[i]); if (ev[i]) cudaEventDestroy(ev[i]); }
        if (created && !finished) { remove(suf_path.c_str()); remove(pre_path.c_str()); }   // no partial database is left
    }
};

static double seconds_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

static int kmc_begin(KmcWriter& w, mlg_ctx* ctx, const char* prefix, uint32_t K, uint32_t min_count, uint32_t counter_max, KmcOutStats* ws) {
    if (K < 5 || K > 60) { mlg_set_error("KMC files need 5 <= K <= 60 here (K = %u)", K); return MLG_ERR_ARG; }
    const auto t0 = std::chrono::steady_clock::now();
    w.ctx = ctx; w.K = K; w.min_count = min_count; w.counter_max = counter_max; w.ws = ws;
    w.p = kmc_prefix_len(K); w.rec = (K - w.p) / 4 + 1;
    w.lut.assign((1ull << (2 * w.p)) + 1, 0);
    w.pre_path = std::string(prefix) + ".kmc_pre"; w.suf_path = std::string(prefix) + ".kmc_suf";
    w.fs = fopen(w.suf_path.c_str(), "wb");
    if (!w.fs) { mlg_set_error("cannot create %s", w.suf_path.c_str()); return MLG_ERR_IO; }
    w.created = true;
    w.ok = fwrite("KMCS", 1, 4, w.fs) == 4;
    if (ws) ws->s_write += seconds_since(t0);
    return MLG_OK;
}

static int kmc_append(KmcWriter& w, const key128* keys, const uint32_t* cnt, uint32_t n) {
    if (!n) return MLG_OK;
    cudaStream_t st = w.ctx->s_comp;
    const unsigned long long np = 1ull << (2 * w.p), sbytes = (unsigned long long)n * w.rec;
    DevBuf<unsigned long long> d_lut; MLG_TRY(d_lut.alloc(np + 1));
    DevBuf<unsigned char> d_rec; MLG_TRY(d_rec.alloc(sbytes));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    struct Ev { cudaEvent_t a, b; ~Ev() { cudaEventDestroy(a); cudaEventDestroy(b); } } guard{e0, e1};
    CUDA_TRY(cudaEventRecord(e0, st));
    k_kmc_lut<<<(unsigned)((np + 256) / 256), 256, 0, st>>>(keys, n, w.K, w.p, d_lut.p);
    k_kmc_records<<<(n + 255) / 256, 256, 0, st>>>(keys, cnt, n, w.K, w.p, w.counter_max, d_rec.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(e1, st));
    std::vector<unsigned long long> lut(np + 1);
    CUDA_TRY(cudaMemcpyAsync(lut.data(), d_lut.p, (np + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    float ms = 0;
    if (w.ws && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) w.ws->ms_encode += ms;
    for (unsigned long long i = 0; i <= np; ++i) w.lut[i] += lut[i];

    const auto t0 = std::chrono::steady_clock::now();
    const unsigned long long CH = 32ull << 20;
    if (w.pin_bytes < std::min(CH, sbytes)) {
        for (int i = 0; i < 2; ++i) if (w.pin[i]) { cudaFreeHost(w.pin[i]); w.pin[i] = nullptr; }
        w.pin_bytes = std::min(CH, sbytes);
        if (cudaMallocHost(&w.pin[0], w.pin_bytes) != cudaSuccess || cudaMallocHost(&w.pin[1], w.pin_bytes) != cudaSuccess ||
            (!w.ev[0] && cudaEventCreateWithFlags(&w.ev[0], cudaEventDisableTiming) != cudaSuccess) ||
            (!w.ev[1] && cudaEventCreateWithFlags(&w.ev[1], cudaEventDisableTiming) != cudaSuccess)) {
            mlg_set_error("pinned staging for %s failed: %s", w.suf_path.c_str(), cudaGetErrorString(cudaGetLastError())); return MLG_ERR_CUDA;
        }
    }
    const unsigned long long pc_bytes = w.pin_bytes, nch = (sbytes + pc_bytes - 1) / pc_bytes;
    int rc = MLG_OK;
    for (unsigned long long c = 0; rc == MLG_OK && c <= nch; ++c) {
        if (c < nch) {
            const unsigned long long b = std::min(pc_bytes, sbytes - c * pc_bytes);
            if (cudaMemcpyAsync(w.pin[c & 1], d_rec.p + c * pc_bytes, b, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaEventRecord(w.ev[c & 1], st) != cudaSuccess) { mlg_set_error("copy of %s failed", w.suf_path.c_str()); rc = MLG_ERR_CUDA; break; }
        }
        if (c > 0) {
            const unsigned long long pc = c - 1, b = std::min(pc_bytes, sbytes - pc * pc_bytes);
            if (cudaEventSynchronize(w.ev[pc & 1]) != cudaSuccess) { mlg_set_error("copy of %s failed", w.suf_path.c_str()); rc = MLG_ERR_CUDA; break; }
            w.ok = w.ok && fwrite(w.pin[pc & 1], 1, b, w.fs) == b;
        }
    }
    cudaStreamSynchronize(st);
    w.records += n; w.sbytes += sbytes;
    if (w.ws) w.ws->s_write += seconds_since(t0);
    return rc;
}

// .kmc_pre: "KMCP" | LUT (+ guard) | header | header bytes | "KMCP"   (csrc/kmcdb.h), version 0.  The one writer of this
// file: kmc_end and kmc_concat both go through it.
struct KmcHeader {
    uint32_t K = 0, mode = 0, counter_size = 1, p = 0, min_count = 0;
    unsigned long long max_count = 0, total = 0;
    unsigned char strands = 0;               // 0: both strands (canonical k-mers)
};
static int kmc_write_pre(const std::string& path, const std::vector<unsigned long long>& lut, const KmcHeader& h, unsigned long long* bytes) {
    std::vector<unsigned char> pre;
    auto put = [&](const void* v, size_t b) { const unsigned char* c = (const unsigned char*)v; pre.insert(pre.end(), c, c + b); };
    auto u32 = [&](uint32_t v) { put(&v, 4); };
    put("KMCP", 4);
    put(lut.data(), lut.size() * 8);
    const size_t h0 = pre.size();
    u32(h.K); u32(h.mode); u32(h.counter_size); u32(h.p);           // k, mode (counters), counter_size, lut_prefix_length
    u32(h.min_count); u32((uint32_t)h.max_count);
    put(&h.total, 8);
    const unsigned char hdr_tail[4] = {h.strands, 0, 0, 0}; put(hdr_tail, 4);   // strands + 3 pad bytes
    u32((uint32_t)(h.max_count >> 32));                              // max_count, high word
    const unsigned char reserved[20] = {}; put(reserved, 20);
    u32(0);                                                          // kmc_version 0
    u32((uint32_t)(pre.size() - h0));
    put("KMCP", 4);
    FILE* fp = fopen(path.c_str(), "wb");
    if (!fp) { mlg_set_error("cannot create %s", path.c_str()); return MLG_ERR_IO; }
    bool ok = fwrite(pre.data(), 1, pre.size(), fp) == pre.size();
    ok = (fclose(fp) == 0) && ok;
    if (!ok) { mlg_set_error("%s: short write", path.c_str()); return MLG_ERR_IO; }
    *bytes = pre.size();
    return MLG_OK;
}

static int kmc_end(KmcWriter& w) {
    const auto t0 = std::chrono::steady_clock::now();
    bool ok = w.ok && fwrite("KMCS", 1, 4, w.fs) == 4;
    ok = (fclose(w.fs) == 0) && ok;
    w.fs = nullptr;
    if (!ok) { mlg_set_error("%s: short write", w.suf_path.c_str()); return MLG_ERR_IO; }
    KmcHeader h;
    h.K = w.K; h.p = w.p; h.min_count = w.min_count; h.max_count = w.counter_max; h.total = w.records;
    unsigned long long pre_bytes = 0;
    MLG_TRY(kmc_write_pre(w.pre_path, w.lut, h, &pre_bytes));
    w.finished = true;
    if (w.ws) {
        w.ws->records = w.records; w.ws->bytes = pre_bytes + w.sbytes + 8;
        w.ws->s_write += seconds_since(t0);
    }
    return MLG_OK;
}

int kmc_write(mlg_ctx* ctx, const char* prefix, const key128* keys, const uint32_t* cnt, uint32_t n, uint32_t K, uint32_t min_count,
              uint32_t counter_max, KmcOutStats* ws) {
    KmcWriter w;
    MLG_TRY(kmc_begin(w, ctx, prefix, K, min_count, counter_max, ws));
    MLG_TRY(kmc_append(w, keys, cnt, n));
    return kmc_end(w);
}

// ---------------------------------------------------------------- key-range passes (mlg_query_enable_read_kmer_passes)
// The pushes only copy the reads into a device archive.  Each output call plans contiguous intervals of the 2K-bit key
// order from a histogram of the archive, counts each interval in its own table by replaying the archive, and hands each
// interval's sorted records on (to the chunked KMC writer, or to the caller's buffers): the concatenation is the sorted
// table of every key.  DESIGN.md section 10.
namespace {

constexpr uint32_t RK_BIN_BASES = 10;                   // bases per histogram level: <= 4^10 u64 counters, 8 MB, L2-resident
// Output-stage device bytes per key of a pass beside its table (collect_slots + sort_keys128 at 2K > 64): the selection
// buffer (16), split hi / lo / count (20), sorted keys and counts (20), sort_keys128's lo_s, iota, perm1, hi_g, hi_s and
// perm2 (36), and the alternate buffers inside CUB's temp storage for one SortPairs (12).
constexpr unsigned long long RK_OUT_BYTES_PER_KEY = 16 + 20 + 20 + 36 + 12;
constexpr unsigned long long RK_FREE_MARGIN = 1ull << 30;   // budget 0: device memory left to CUB, the prefix tables and the driver

typedef unsigned __int128 u128;
inline key128 to_key(u128 x) { key128 k; k.hi = (unsigned long long)(x >> 64); k.lo = (unsigned long long)x; return k; }

// device bytes of one pass whose keys are bounded by `bound`
inline unsigned long long pass_bytes(unsigned long long bound) { return slots_for(bound) * sizeof(Slot) + bound * RK_OUT_BYTES_PER_KEY; }

struct ArchivedBatch {
    DevBuf<unsigned long long> bases, nmask, off;       // nmask: none when the push had no N; off: none with a fixed read_len
    unsigned long long n_reads = 0, nbases = 0, base_words = 0, nmask_words = 0;
    uint32_t read_len = 0;
};

struct KeyRange { u128 lo, hi; unsigned long long bound; };

}  // namespace

struct ReadKmerPasses {
    mlg_ctx* ctx = nullptr;
    uint32_t K = 0;
    unsigned long long budget = 0;
    std::deque<ArchivedBatch> batches;
    unsigned long long archive_bytes = 0, bytes_needed = 0;
    bool overflowed = false;
    int overflowed_rank = -1;                // a peer's blob came flagged: that rank's archive overflowed
    // rank `rank` of a `world`-rank count (mlg_query_read_kmer_archive): the output calls count share `rank` of the key
    // order over this rank's batches and every peer's
    uint32_t rank = 0, world = 1, peers = 0;
    std::vector<char> added;                 // per rank: its batches are in the archive
    DevBuf<unsigned char> blob;              // this rank's blob, until the first output call
    std::vector<unsigned long long> blob_head;
    mlg_read_kmer_plan plan{};               // of the last output call
    mlg_read_kmer_stats st{};                // windows, distinct, slots, bytes, ms_count of the last output call
};

int rkp_create(mlg_ctx* ctx, uint32_t K, unsigned long long max_bytes, ReadKmerPasses** out) {
    if (K < 1 || K > 60) { mlg_set_error("read k-mer counting needs K <= 60 (the count lives in the top byte of the key); this database has K = %u", K); return MLG_ERR_ARG; }
    ReadKmerPasses* t = new ReadKmerPasses();
    t->ctx = ctx; t->K = K; t->budget = max_bytes;
    *out = t;
    return MLG_OK;
}
void rkp_destroy(ReadKmerPasses* t) { delete t; }

// Enqueued on the compute stream after the batch's last probe range, before the staging set's `done` event: copies of
// what the probe read (whole 16-byte units of bases, the N mask as it saw it, the offsets).  No kernel.
// the archive stops: batches freed, the output calls return MLG_ERR_NOMEM; bytes_needed = what it would have needed
static int rkp_overflow(ReadKmerPasses* t, unsigned long long add) {
    cudaGetLastError();                                   // a failed allocation is recorded here, not an error of the query
    CUDA_TRY(cudaStreamSynchronize(t->ctx->s_comp));      // copies into the archive may still be in flight
    t->batches.clear();
    t->overflowed = true; t->bytes_needed = t->archive_bytes + add; t->archive_bytes = 0;
    return MLG_OK;
}

int rkp_archive(ReadKmerPasses* t, const ProbeArgs& a, unsigned long long n_reads, unsigned long long nbases) {
    const unsigned long long add = a.base_words * 8 + (a.nmask ? a.nmask_words * 8 : 0) + (a.off ? (n_reads + 1) * 8 : 0);
    if (t->overflowed) { t->bytes_needed += add; return MLG_OK; }     // what the whole archive would have needed
    cudaStream_t st = t->ctx->s_comp;
    auto overflow = [&]() -> int { return rkp_overflow(t, add); };
    if (t->budget && t->archive_bytes + add > t->budget) return overflow();
    t->batches.emplace_back();
    ArchivedBatch& b = t->batches.back();
    if (b.bases.alloc(a.base_words) != MLG_OK || (a.nmask && b.nmask.alloc(a.nmask_words) != MLG_OK) ||
        (a.off && b.off.alloc(n_reads + 1) != MLG_OK)) return overflow();
    CUDA_TRY(cudaMemcpyAsync(b.bases.p, a.bases, a.base_words * 8, cudaMemcpyDeviceToDevice, st));
    if (a.nmask) CUDA_TRY(cudaMemcpyAsync(b.nmask.p, a.nmask, a.nmask_words * 8, cudaMemcpyDeviceToDevice, st));
    if (a.off) CUDA_TRY(cudaMemcpyAsync(b.off.p, a.off, (n_reads + 1) * 8, cudaMemcpyDeviceToDevice, st));
    b.n_reads = n_reads; b.nbases = nbases; b.base_words = a.base_words; b.nmask_words = a.nmask_words; b.read_len = a.read_len;
    t->archive_bytes += add;
    return MLG_OK;
}

int rkp_check(ReadKmerPasses* t) {
    if (t->overflowed && t->overflowed_rank >= 0) {
        mlg_set_error("rank %d's device copy of the reads outgrew its read k-mer budget", t->overflowed_rank);
        return MLG_ERR_NOMEM;
    }
    if (t->overflowed) {
        mlg_set_error("the device copy of the reads outgrew the read k-mer budget: %llu bytes needed, %llu allowed", t->bytes_needed, t->budget);
        return MLG_ERR_NOMEM;
    }
    CUDA_TRY(cudaStreamSynchronize(t->ctx->s_copy));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->s_comp));
    return MLG_OK;
}

static CountArgs batch_args(const ReadKmerPasses* t, const ArchivedBatch& b) {
    CountArgs a{};
    a.bases = b.bases.p; a.nmask = b.nmask.p; a.off = b.off.p; a.read_len = b.read_len; a.K = t->K;
    a.base_words = b.base_words; a.nmask_words = b.nmask_words; a.r_begin = 0; a.r_end = b.n_reads;
    return a;
}

namespace {

// The plan: bins of the leading bases of the canonical key (RK_BIN_BASES per level), each bounded by min(windows, keys
// it can hold), grouped in key order into passes that fit the cap; a bin that alone does not fit is split by a histogram
// over its next bases.  A bin that covers the whole k-mer holds one key, so the recursion ends.
// Share r of a W-rank count: the top-level bins [s_r, s_{r+1}) with s_r = the first bin i such that W * (windows of the
// bins before i) >= r * T, T = every window, and s_W = the number of bins.  Every rank holds the same reads, so every
// rank finds the same boundaries.  A share holds fewer than T / W + (the largest bin) windows.
void share_bins(const std::vector<unsigned long long>& h, uint32_t world, uint32_t rank, unsigned long long* b0, unsigned long long* b1) {
    unsigned long long T = 0;
    for (unsigned long long x : h) T += x;
    auto bound = [&](uint32_t r) -> unsigned long long {
        if (r >= world) return h.size();
        unsigned long long before = 0;
        for (unsigned long long i = 0; i < h.size(); before += h[i], ++i)
            if ((u128)world * before >= (u128)r * T) return i;
        return h.size();
    };
    *b0 = bound(rank); *b1 = bound(rank + 1);
}

struct Planner {
    ReadKmerPasses* t;
    unsigned long long cap;
    std::vector<KeyRange> passes;
    KeyRange cur{};
    bool open = false;
    DevBuf<unsigned long long> d_bins;
    std::vector<unsigned long long> bins;
    float ms = 0;

    bool fits(unsigned long long bound) const { return bound < (1ull << 32) && pass_bytes(bound) <= cap; }
    void add(u128 lo, u128 hi, unsigned long long bound) {
        if (open && !fits(cur.bound + bound)) { passes.push_back(cur); open = false; }
        if (!open) { cur = KeyRange{lo, hi, bound}; open = true; }
        else { cur.hi = hi; cur.bound += bound; }
    }
    // windows per bin of the keys that start with the `depth` bases `prefix`, by their next b bases
    int histogram(uint32_t depth, u128 prefix, uint32_t b) {
        cudaStream_t st = t->ctx->s_comp;
        const unsigned long long nb = 1ull << (2 * b);
        CUDA_TRY(cudaMemsetAsync(d_bins.p, 0, nb * 8, st));
        cudaEvent_t e0, e1;
        CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
        struct Ev { cudaEvent_t a, b; ~Ev() { cudaEventDestroy(a); cudaEventDestroy(b); } } guard{e0, e1};
        CUDA_TRY(cudaEventRecord(e0, st));
        for (const ArchivedBatch& ab : t->batches)
            k_kmer_histogram<<<grid_for(ab.nbases, t->ctx->sm_count * 16), RK_TPB, 0, st>>>(
                batch_args(t, ab), 2 * (t->K - depth), to_key(prefix), 2 * (t->K - depth - b), nb - 1, d_bins.p);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(e1, st));
        bins.resize(nb);
        CUDA_TRY(cudaMemcpyAsync(bins.data(), d_bins.p, nb * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        float m = 0;
        if (cudaEventElapsedTime(&m, e0, e1) == cudaSuccess) ms += m;
        return MLG_OK;
    }
    int visit(uint32_t depth, u128 prefix, unsigned long long* windows) {
        const uint32_t b = std::min(RK_BIN_BASES, t->K - depth), rest = t->K - depth - b;
        MLG_TRY(histogram(depth, prefix, b));
        const std::vector<unsigned long long> h = bins;       // the recursion reuses `bins`
        const unsigned long long keys_per_bin = 2 * rest >= 64 ? ~0ull : 1ull << (2 * rest);
        unsigned long long i0 = 0, i1 = h.size();               // this rank's share of the top-level bins
        if (depth == 0) {
            share_bins(h, t->world, t->rank, &i0, &i1);
            t->plan.share_first_bin = i0; t->plan.share_end_bin = i1;
        }
        for (unsigned long long i = 0; i < h.size(); ++i) {
            if (windows) *windows += h[i];
            if (i < i0 || i >= i1) continue;
            if (depth == 0) t->plan.share_windows += h[i];
            const u128 sub = (prefix << (2 * b)) | i;
            const unsigned long long bound = std::min(h[i], keys_per_bin);
            if (fits(bound)) { add(sub << (2 * rest), (sub + 1) << (2 * rest), bound); continue; }
            t->plan.refined_bins += 1;
            MLG_TRY(visit(depth + b, sub, nullptr));
        }
        return MLG_OK;
    }
};

}  // namespace

// The passes of an output call, before anything is allocated for them or written (the plan's NOMEM leaves no file)
static int rkp_plan_passes(ReadKmerPasses* t, std::vector<KeyRange>& passes) {
    mlg_ctx* ctx = t->ctx;
    mlg_read_kmer_plan& pl = t->plan;
    pl = mlg_read_kmer_plan{};
    t->st = mlg_read_kmer_stats{};
    t->blob.release();                                     // the peers have their copies: rkp_check joined the stream
    pl.archive_bytes = t->archive_bytes;
    pl.rank = t->rank; pl.world = t->world; pl.peers_added = t->peers;
    Planner P{t, 0};
    MLG_TRY(P.d_bins.alloc(1ull << (2 * RK_BIN_BASES)));
    if (t->budget) {
        P.cap = t->budget > t->archive_bytes ? t->budget - t->archive_bytes : 0;
    } else {
        mlg_pool_trim(ctx->device);                        // cached blocks count as free here: the passes take them
        size_t fr = 0, tot = 0;
        CUDA_TRY(cudaMemGetInfo(&fr, &tot));
        P.cap = fr > RK_FREE_MARGIN ? fr - RK_FREE_MARGIN : 0;
    }
    pl.pass_cap_bytes = P.cap;
    if (!P.fits(1)) {
        mlg_set_error("%llu bytes are left for a read k-mer pass beside the %llu-byte device copy of the reads; the smallest pass needs %llu",
                      P.cap, t->archive_bytes, pass_bytes(1));
        return MLG_ERR_NOMEM;
    }
    unsigned long long windows = 0;
    MLG_TRY(P.visit(0, 0, &windows));
    if (P.open) P.passes.push_back(P.cur);
    P.d_bins.release();
    pl.ms_histogram = P.ms;
    pl.passes = (uint32_t)P.passes.size();
    t->st.windows = windows;
    passes.swap(P.passes);
    return MLG_OK;
}

// Every pass: a table sized from the pass's bound, the ranged count over every archived batch, then the selection and
// sort of collect_slots; the table is freed before the sorted records go to `sink`.
static int rkp_run(ReadKmerPasses* t, const std::vector<KeyRange>& passes, uint32_t min_count,
                   const std::function<int(const key128*, const uint32_t*, uint32_t)>& sink, KmcOutStats* ws) {
    mlg_ctx* ctx = t->ctx;
    cudaStream_t st = ctx->s_comp;
    mlg_read_kmer_plan& pl = t->plan;

    DevBuf<unsigned long long> ctr; MLG_TRY(ctr.alloc(4));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    struct Ev { cudaEvent_t a, b; ~Ev() { cudaEventDestroy(a); cudaEventDestroy(b); } } guard{e0, e1};
    for (const KeyRange& r : passes) {
        pl.max_pass_bound = std::max<uint64_t>(pl.max_pass_bound, r.bound);
        const unsigned long long nslots = slots_for(r.bound);
        DevBuf<Slot> tab;
        if (tab.alloc(nslots) != MLG_OK) {
            cudaGetLastError();
            mlg_set_error("a read k-mer pass could not allocate its %llu-byte table", nslots * sizeof(Slot));
            return MLG_ERR_NOMEM;
        }
        CUDA_TRY(cudaMemsetAsync(tab.p, 0, nslots * sizeof(Slot), st));
        CUDA_TRY(cudaMemsetAsync(ctr.p, 0, 32, st));
        CUDA_TRY(cudaEventRecord(e0, st));
        for (const ArchivedBatch& ab : t->batches) {
            CountArgs a = batch_args(t, ab);
            a.tab = tab.p; a.line_mask = nslots / 8 - 1; a.ctr = ctr.p; a.range_lo = to_key(r.lo); a.range_hi = to_key(r.hi);
            k_count_read_kmers<true><<<grid_for(ab.nbases, ctx->sm_count * 16), RK_TPB, 0, st>>>(a);
        }
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(e1, st));
        KmcOutStats po;
        DevBuf<key128> keys; DevBuf<uint32_t> cnt;
        uint32_t n = 0;
        unsigned long long distinct = 0, full = 0;
        MLG_TRY(collect_slots(ctx, tab.p, nslots, ctr.p, t->K, min_count, keys, cnt, &n, &po, &distinct));
        CUDA_TRY(cudaMemcpyAsync(&full, ctr.p + 2, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (full) { mlg_set_error("read k-mer pass: a key found no free slot"); return MLG_ERR_STATE; }
        tab.release();
        float ms = 0;
        if (cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) t->st.ms_count += ms;
        t->st.distinct += distinct;
        if (nslots > t->st.slots) { t->st.slots = nslots; t->st.bytes = nslots * sizeof(Slot); }
        if (ws) { ws->ms_compact += po.ms_compact; ws->ms_sort += po.ms_sort; }
        const double enc0 = ws ? ws->ms_encode : 0;
        MLG_TRY(sink(keys.p, cnt.p, n));
        pl.ms_output += po.ms_compact + po.ms_sort + (ws ? ws->ms_encode - enc0 : 0);
    }
    pl.distinct = t->st.distinct;
    pl.ms_count = t->st.ms_count;
    return MLG_OK;
}

int rkp_read_kmers(ReadKmerPasses* t, uint32_t min_count, uint32_t counter_max, uint64_t* keys_out, uint8_t* counts_out, uint64_t cap,
                   uint64_t* n_total, KmcOutStats* ws) {
    cudaStream_t st = t->ctx->s_comp;
    uint64_t at = 0;
    std::vector<uint32_t> hc;
    std::vector<KeyRange> passes;
    MLG_TRY(rkp_plan_passes(t, passes));
    MLG_TRY(rkp_run(t, passes, min_count, [&](const key128* keys, const uint32_t* cnt, uint32_t n) -> int {
        const uint64_t c = at < cap ? std::min<uint64_t>(cap - at, n) : 0;
        if (c) {
            hc.resize(c);
            if (keys_out) CUDA_TRY(cudaMemcpyAsync(keys_out + 2 * at, keys, c * sizeof(key128), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(hc.data(), cnt, c * 4, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (counts_out) for (uint64_t i = 0; i < c; ++i) counts_out[at + i] = (uint8_t)std::min(hc[i], counter_max);
        }
        at += n;
        return MLG_OK;
    }, ws));
    *n_total = at;
    if (ws) ws->records = at;
    return MLG_OK;
}

int rkp_write_kmc(ReadKmerPasses* t, const char* prefix, uint32_t min_count, uint32_t counter_max, KmcOutStats* ws) {
    std::vector<KeyRange> passes;
    MLG_TRY(rkp_plan_passes(t, passes));
    KmcWriter w;
    MLG_TRY(kmc_begin(w, t->ctx, prefix, t->K, min_count, counter_max, ws));
    MLG_TRY(rkp_run(t, passes, min_count, [&](const key128* keys, const uint32_t* cnt, uint32_t n) { return kmc_append(w, keys, cnt, n); }, ws));
    return kmc_end(w);
}

int rkp_stats(ReadKmerPasses* t, mlg_read_kmer_stats* o) {
    *o = t->st;
    o->overflowed = t->overflowed ? 1 : 0; o->bytes_needed = t->bytes_needed;
    return MLG_OK;
}
int rkp_plan(ReadKmerPasses* t, mlg_read_kmer_plan* o) { *o = t->plan; return MLG_OK; }

// ---------------------------------------------------------------- the read k-mer count across ranks
// Each rank packs its archive into one device blob; every rank appends every peer's blob to its archive and then counts
// its own share of the key order over all the reads.  Blob layout (8-byte words, all little endian):
//   header   magic, BUILD_TAG | K << 32, rank | world << 32, overflowed, batches, bytes     (RKA_HEAD_WORDS)
//   per batch n_reads, nbases, read_len, base_words, nmask_words, flags (1: N mask, 2: offsets)   (RKA_DESC_WORDS)
//   data     per batch: bases (base_words words), N mask (nmask_words words), offsets (n_reads + 1 words)
// DESIGN.md section 10.
namespace {

constexpr unsigned long long RKA_MAGIC = 0x3130414B52474C4Dull;      // "MLGRKA01"
constexpr unsigned long long RKA_HEAD_WORDS = 6, RKA_DESC_WORDS = 6;
constexpr unsigned long long RKA_MASK = 1, RKA_OFF = 2;
constexpr unsigned long long RKA_FIRST_READ = 64 << 10;               // bytes of the first header copy

inline unsigned long long rka_data_words(unsigned long long n_reads, unsigned long long base_words, unsigned long long nmask_words,
                                         unsigned long long flags) {
    return base_words + ((flags & RKA_MASK) ? nmask_words : 0) + ((flags & RKA_OFF) ? n_reads + 1 : 0);
}

// a peer's offsets before they are trusted: off[0] = 0, non-decreasing, off[n_reads] = nbases (bad[0] = 1 otherwise)
__global__ void k_check_offsets(const unsigned long long* off, unsigned long long n_reads, unsigned long long nbases, unsigned long long* bad) {
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i <= n_reads; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long v = off[i];
        if ((i == 0 && v != 0) || (i == n_reads && v != nbases) || (i < n_reads && off[i + 1] < v)) atomicOr(bad, 1ull);
    }
}

}  // namespace

int rkp_pack_archive(ReadKmerPasses* t, uint32_t rank, uint32_t world, const void** d_blob, uint64_t* bytes) {
    cudaStream_t st = t->ctx->s_comp;
    const unsigned long long nb = t->overflowed ? 0 : t->batches.size();     // an overflowed archive sends its flag only
    std::vector<unsigned long long>& h = t->blob_head;                       // kept: the copy below is asynchronous
    h.assign(RKA_HEAD_WORDS + nb * RKA_DESC_WORDS, 0);
    unsigned long long words = h.size();
    for (unsigned long long i = 0; i < nb; ++i) {
        const ArchivedBatch& b = t->batches[i];
        unsigned long long* d = h.data() + RKA_HEAD_WORDS + i * RKA_DESC_WORDS;
        d[0] = b.n_reads; d[1] = b.nbases; d[2] = b.read_len; d[3] = b.base_words; d[4] = b.nmask_words;
        d[5] = (b.nmask.p ? RKA_MASK : 0) | (b.off.p ? RKA_OFF : 0);
        words += rka_data_words(d[0], d[3], d[4], d[5]);
    }
    h[0] = RKA_MAGIC; h[1] = MLG_BUILD_TAG | (unsigned long long)t->K << 32; h[2] = rank | (unsigned long long)world << 32;
    h[3] = t->overflowed ? 1 : 0; h[4] = nb; h[5] = words * 8;
    DevBuf<unsigned char> blob;
    if (blob.alloc(words * 8) != MLG_OK) {
        cudaGetLastError();
        mlg_set_error("no device memory for the %llu-byte blob of the read archive", words * 8);
        return MLG_ERR_NOMEM;
    }
    unsigned char* p = blob.p;
    CUDA_TRY(cudaMemcpyAsync(p, h.data(), h.size() * 8, cudaMemcpyHostToDevice, st));
    p += h.size() * 8;
    for (unsigned long long i = 0; i < nb; ++i) {
        const ArchivedBatch& b = t->batches[i];
        CUDA_TRY(cudaMemcpyAsync(p, b.bases.p, b.base_words * 8, cudaMemcpyDeviceToDevice, st)); p += b.base_words * 8;
        if (b.nmask.p) { CUDA_TRY(cudaMemcpyAsync(p, b.nmask.p, b.nmask_words * 8, cudaMemcpyDeviceToDevice, st)); p += b.nmask_words * 8; }
        if (b.off.p) { CUDA_TRY(cudaMemcpyAsync(p, b.off.p, (b.n_reads + 1) * 8, cudaMemcpyDeviceToDevice, st)); p += (b.n_reads + 1) * 8; }
    }
    std::swap(t->blob.p, blob.p); std::swap(t->blob.n, blob.n);
    t->rank = rank; t->world = world; t->peers = 0;
    t->added.assign(world, 0); t->added[rank] = 1;
    *d_blob = t->blob.p; *bytes = words * 8;
    return MLG_OK;
}

// A peer's blob comes from outside the query: everything the count kernels rely on is checked before anything changes.
int rkp_add_archive(ReadKmerPasses* t, const void* d_blob, uint64_t bytes, uint32_t* launches) {
    cudaStream_t st = t->ctx->s_comp;
    const unsigned char* blob = (const unsigned char*)d_blob;
    if ((uintptr_t)d_blob % 8) { mlg_set_error("a read archive blob must start on an 8-byte boundary"); return MLG_ERR_ARG; }
    if (bytes < RKA_HEAD_WORDS * 8 || bytes % 8) { mlg_set_error("a read archive blob has %llu bytes: not a blob", (unsigned long long)bytes); return MLG_ERR_ARG; }
    std::vector<unsigned long long> h(std::min<unsigned long long>(bytes, RKA_FIRST_READ) / 8);
    CUDA_TRY(cudaMemcpyAsync(h.data(), blob, h.size() * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const uint32_t tag = (uint32_t)h[1], K = (uint32_t)(h[1] >> 32), rank = (uint32_t)h[2], world = (uint32_t)(h[2] >> 32);
    const unsigned long long nb = h[4];
    if (h[0] != RKA_MAGIC || tag != MLG_BUILD_TAG) { mlg_set_error("not a read archive blob of this library version"); return MLG_ERR_ARG; }
    if (K != t->K || world != t->world) { mlg_set_error("read archive blob of K = %u, %u ranks; this query has K = %u, %u ranks", K, world, t->K, t->world); return MLG_ERR_ARG; }
    if (rank >= world || rank == t->rank || t->added[rank]) { mlg_set_error("read archive blob of rank %u: out of range, this rank's own, or already added", rank); return MLG_ERR_ARG; }
    if (h[5] != bytes || h[3] > 1 || (h[3] && nb) || nb > (bytes / 8 - RKA_HEAD_WORDS) / RKA_DESC_WORDS) {
        mlg_set_error("read archive blob of rank %u: its header does not match its %llu bytes", rank, (unsigned long long)bytes); return MLG_ERR_ARG;
    }
    const unsigned long long head = RKA_HEAD_WORDS + nb * RKA_DESC_WORDS;
    if (head > h.size()) {
        h.resize(head);
        CUDA_TRY(cudaMemcpyAsync(h.data(), blob, head * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    u128 words = head;
    for (unsigned long long i = 0; i < nb; ++i) {
        const unsigned long long* d = h.data() + RKA_HEAD_WORDS + i * RKA_DESC_WORDS;
        const unsigned long long n_reads = d[0], nbases = d[1], read_len = d[2], bw = d[3], mw = d[4], fl = d[5];
        bool ok = fl <= (RKA_MASK | RKA_OFF) && read_len < (1ull << 32) && bw <= bytes / 8 && mw <= bytes / 8 && n_reads < bytes / 8 &&
                  (u128)bw * 32 >= nbases && (!(fl & RKA_MASK) || (u128)mw * 64 >= nbases);
        if (ok && !(fl & RKA_OFF)) ok = (u128)n_reads * read_len == nbases && (read_len || !n_reads);
        if (!ok) { mlg_set_error("read archive blob of rank %u: batch %llu has an inconsistent descriptor", rank, i); return MLG_ERR_ARG; }
        words += rka_data_words(n_reads, bw, mw, fl);
    }
    if (words * 8 != bytes) { mlg_set_error("read archive blob of rank %u: its batches do not add up to its %llu bytes", rank, (unsigned long long)bytes); return MLG_ERR_ARG; }
    // the offsets, on the device: a bad one would send the count kernels' read search out of the batch
    std::vector<const unsigned long long*> data(nb);
    {
        const unsigned char* p = blob + head * 8;
        for (unsigned long long i = 0; i < nb; ++i) {
            const unsigned long long* d = h.data() + RKA_HEAD_WORDS + i * RKA_DESC_WORDS;
            data[i] = (const unsigned long long*)p;
            p += rka_data_words(d[0], d[3], d[4], d[5]) * 8;
        }
    }
    DevBuf<unsigned long long> bad; MLG_TRY(bad.alloc(1));
    CUDA_TRY(cudaMemsetAsync(bad.p, 0, 8, st));
    for (unsigned long long i = 0; i < nb; ++i) {
        const unsigned long long* d = h.data() + RKA_HEAD_WORDS + i * RKA_DESC_WORDS;
        if (!(d[5] & RKA_OFF)) continue;
        const unsigned long long* off = data[i] + d[3] + ((d[5] & RKA_MASK) ? d[4] : 0);
        k_check_offsets<<<grid_for(d[0] + 1, t->ctx->sm_count * 4), RK_TPB, 0, st>>>(off, d[0], d[1], bad.p);
        CUDA_TRY(cudaGetLastError());
        *launches += 1;
    }
    unsigned long long flag = 0;
    CUDA_TRY(cudaMemcpyAsync(&flag, bad.p, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (flag) { mlg_set_error("read archive blob of rank %u: read offsets that do not start at 0, ascend and end at the batch's bases", rank); return MLG_ERR_ARG; }

    t->added[rank] = 1; t->peers += 1;
    const unsigned long long add = bytes - head * 8;
    if (h[3]) {                                           // that rank's archive overflowed: so does the count on every rank
        if (!t->overflowed) MLG_TRY(rkp_overflow(t, 0));
        t->overflowed_rank = (int)rank;
        return MLG_OK;
    }
    if (t->overflowed) { t->bytes_needed += add; return MLG_OK; }
    if (t->budget && t->archive_bytes + add > t->budget) return rkp_overflow(t, add);
    for (unsigned long long i = 0; i < nb; ++i) {
        const unsigned long long* d = h.data() + RKA_HEAD_WORDS + i * RKA_DESC_WORDS;
        t->batches.emplace_back();
        ArchivedBatch& b = t->batches.back();
        const bool m = d[5] & RKA_MASK, o = d[5] & RKA_OFF;
        if (b.bases.alloc(d[3]) != MLG_OK || (m && b.nmask.alloc(d[4]) != MLG_OK) || (o && b.off.alloc(d[0] + 1) != MLG_OK)) return rkp_overflow(t, add);
        const unsigned long long* p = data[i];
        CUDA_TRY(cudaMemcpyAsync(b.bases.p, p, d[3] * 8, cudaMemcpyDeviceToDevice, st)); p += d[3];
        if (m) { CUDA_TRY(cudaMemcpyAsync(b.nmask.p, p, d[4] * 8, cudaMemcpyDeviceToDevice, st)); p += d[4]; }
        if (o) CUDA_TRY(cudaMemcpyAsync(b.off.p, p, (d[0] + 1) * 8, cudaMemcpyDeviceToDevice, st));
        b.n_reads = d[0]; b.nbases = d[1]; b.read_len = (uint32_t)d[2]; b.base_words = d[3]; b.nmask_words = d[4];
    }
    t->archive_bytes += add;
    return MLG_OK;
}

uint32_t rkp_peers_missing(const ReadKmerPasses* t) { return t->world - 1 - t->peers; }

// ---------------------------------------------------------------- mlg_kmc_concat
// Version-0 KMC databases whose keys ascend from one to the next, joined into one: the suffix bodies streamed one after
// the other (copy_file_range, or reads and writes of 64 MiB), the prefix tables summed, the header of the parts with the
// summed total.  Only the prefix files, the first and last record of each part and the file sizes are read to check them.
namespace {

constexpr unsigned long long KMC_HEADER_BYTES = 64;      // version 0: k .. kmc_version

struct KmcPart {
    std::string pre, suf;
    KmcHeader h;
    std::vector<unsigned long long> lut;
    unsigned long long rec = 0;
    u128 first = 0, last = 0;
    struct stat st_pre{}, st_suf{};
};

bool slurp(const std::string& path, std::vector<unsigned char>& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    bool ok = fseek(f, 0, SEEK_END) == 0;
    const long n = ok ? ftell(f) : -1;
    ok = ok && n >= 0 && fseek(f, 0, SEEK_SET) == 0;
    if (ok) { out.resize((size_t)n); ok = fread(out.data(), 1, out.size(), f) == out.size(); }
    fclose(f);
    return ok;
}

bool pread_all(int fd, void* buf, size_t n, off_t at) {
    unsigned char* b = (unsigned char*)buf;
    while (n) {
        const ssize_t r = pread(fd, b, n, at);
        if (r <= 0) return false;
        b += r; n -= (size_t)r; at += r;
    }
    return true;
}

// the key of record r of a part: its prefix from the prefix table, its suffix bytes from the suffix file
bool record_key(const KmcPart& P, int fd, unsigned long long r, u128* key) {
    const unsigned long long np = P.lut.size() - 1;
    unsigned long long lo = 0, hi = np;              // the prefix i with lut[i] <= r < lut[i + 1]
    while (hi - lo > 1) { const unsigned long long m = (lo + hi) / 2; if (P.lut[m] <= r) lo = m; else hi = m; }
    const uint32_t sb = (P.h.K - P.h.p) / 4;
    unsigned char b[16];
    if (!pread_all(fd, b, sb, 4 + (off_t)(r * P.rec))) return false;
    u128 k = lo;
    for (uint32_t j = 0; j < sb; ++j) k = (k << 8) | b[j];
    *key = k;
    return true;
}

int read_part(const char* prefix, KmcPart& P) {
    P.pre = std::string(prefix) + ".kmc_pre"; P.suf = std::string(prefix) + ".kmc_suf";
    std::vector<unsigned char> pre;
    if (!slurp(P.pre, pre) || stat(P.pre.c_str(), &P.st_pre) != 0) { mlg_set_error("cannot read %s", P.pre.c_str()); return MLG_ERR_IO; }
    auto u32 = [&](size_t at) { uint32_t v; memcpy(&v, pre.data() + at, 4); return v; };
    const size_t n = pre.size();
    if (n < 8 + 8 + KMC_HEADER_BYTES + 8 || memcmp(pre.data(), "KMCP", 4) || memcmp(pre.data() + n - 4, "KMCP", 4) ||
        u32(n - 8) != KMC_HEADER_BYTES || u32(n - 12) != 0) {
        mlg_set_error("%s is not the prefix file of a version-0 KMC database", P.pre.c_str()); return MLG_ERR_ARG;
    }
    const size_t h0 = n - 8 - KMC_HEADER_BYTES;
    KmcHeader& h = P.h;
    h.K = u32(h0); h.mode = u32(h0 + 4); h.counter_size = u32(h0 + 8); h.p = u32(h0 + 12); h.min_count = u32(h0 + 16);
    memcpy(&h.total, pre.data() + h0 + 24, 8);
    h.strands = pre[h0 + 32];
    h.max_count = u32(h0 + 20) | (unsigned long long)u32(h0 + 36) << 32;
    const bool shape = h.p >= 1 && h.p <= 15 && h.K > h.p && h.K <= 64 && (h.K - h.p) % 4 == 0 && h.counter_size >= 1 && h.counter_size <= 4 &&
                       h0 == 4 + ((1ull << (2 * h.p)) + 1) * 8;
    if (!shape) { mlg_set_error("%s: k = %u, lut_prefix_length = %u, counter_size = %u and its prefix table do not fit together", P.pre.c_str(), h.K, h.p, h.counter_size); return MLG_ERR_ARG; }
    P.lut.resize((1ull << (2 * h.p)) + 1);
    memcpy(P.lut.data(), pre.data() + 4, P.lut.size() * 8);
    bool mono = P.lut[0] == 0 && P.lut.back() == h.total;
    for (size_t i = 1; mono && i < P.lut.size(); ++i) mono = P.lut[i - 1] <= P.lut[i];
    if (!mono) { mlg_set_error("%s: the prefix table does not ascend to the total of %llu k-mers", P.pre.c_str(), h.total); return MLG_ERR_ARG; }
    P.rec = (h.K - h.p) / 4 + h.counter_size;
    const int fd = open(P.suf.c_str(), O_RDONLY);
    if (fd < 0) { mlg_set_error("cannot read %s", P.suf.c_str()); return MLG_ERR_IO; }
    struct Fd { int f; ~Fd() { close(f); } } guard{fd};
    char m0[4], m1[4];
    if (fstat(fd, &P.st_suf) != 0 || (u128)P.st_suf.st_size != 8 + (u128)h.total * P.rec || !pread_all(fd, m0, 4, 0) ||
        !pread_all(fd, m1, 4, P.st_suf.st_size - 4) || memcmp(m0, "KMCS", 4) || memcmp(m1, "KMCS", 4)) {
        mlg_set_error("%s does not hold the %llu records of %s", P.suf.c_str(), h.total, P.pre.c_str()); return MLG_ERR_ARG;
    }
    if (h.total && (!record_key(P, fd, 0, &P.first) || !record_key(P, fd, h.total - 1, &P.last))) { mlg_set_error("cannot read %s", P.suf.c_str()); return MLG_ERR_IO; }
    return MLG_OK;
}

// bytes [at, at + n) of `in` appended to `out`
bool copy_range(int in, off_t at, unsigned long long n, int out, std::vector<unsigned char>& buf) {
    bool plain = false;
    while (n) {
        const size_t c = (size_t)std::min<unsigned long long>(n, 1ull << 30);
        ssize_t r = -1;
        if (!plain) {
            loff_t a = at;
            r = copy_file_range(in, &a, out, nullptr, c, 0);
            if (r < 0 && (errno == EXDEV || errno == ENOSYS || errno == EINVAL || errno == EOPNOTSUPP || errno == EBADF)) { plain = true; continue; }
        } else {
            if (buf.empty()) buf.resize(64ull << 20);
            const size_t m = std::min(c, buf.size());
            if (!pread_all(in, buf.data(), m, at)) return false;
            for (size_t w = 0; w < m;) { const ssize_t k = write(out, buf.data() + w, m - w); if (k <= 0) return false; w += (size_t)k; }
            r = (ssize_t)m;
        }
        if (r <= 0) return false;
        at += r; n -= (unsigned long long)r;
    }
    return true;
}

}  // namespace

int kmc_concat(const char* prefix, const char* const* parts, uint32_t n_parts) {
    std::vector<KmcPart> P(n_parts);
    for (uint32_t i = 0; i < n_parts; ++i) {
        MLG_TRY(read_part(parts[i], P[i]));
        const KmcHeader &a = P[0].h, &b = P[i].h;
        if (a.K != b.K || a.mode != b.mode || a.counter_size != b.counter_size || a.p != b.p || a.min_count != b.min_count ||
            a.max_count != b.max_count || a.strands != b.strands) {
            mlg_set_error("%s: its header (k, mode, counter size, lut_prefix_length, min / max count or strands) differs from %s's", parts[i], parts[0]);
            return MLG_ERR_ARG;
        }
    }
    const KmcPart* prev = nullptr;
    for (const KmcPart& x : P) {
        if (!x.h.total) continue;
        if (prev && !(prev->last < x.first)) { mlg_set_error("%s does not start after the last k-mer of %s", x.pre.c_str(), prev->pre.c_str()); return MLG_ERR_ARG; }
        prev = &x;
    }
    const std::string pre_path = std::string(prefix) + ".kmc_pre", suf_path = std::string(prefix) + ".kmc_suf";
    for (const std::string& o : {pre_path, suf_path}) {
        struct stat so;
        if (stat(o.c_str(), &so) != 0) continue;
        for (const KmcPart& x : P)
            for (const struct stat* sp : {&x.st_pre, &x.st_suf})
                if (sp->st_dev == so.st_dev && sp->st_ino == so.st_ino) { mlg_set_error("%s is one of the parts", o.c_str()); return MLG_ERR_ARG; }
    }
    KmcHeader h = P[0].h;
    h.total = 0;
    std::vector<unsigned long long> lut(P[0].lut.size(), 0);
    for (const KmcPart& x : P) {
        h.total += x.h.total;
        for (size_t i = 0; i < lut.size(); ++i) lut[i] += x.lut[i];
    }
    struct Out { std::string pre, suf; int fd = -1; bool done = false;
                 ~Out() { if (fd >= 0) close(fd); if (!done) { remove(suf.c_str()); remove(pre.c_str()); } } } out{pre_path, suf_path};
    out.fd = open(suf_path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (out.fd < 0) { mlg_set_error("cannot create %s", suf_path.c_str()); return MLG_ERR_IO; }
    std::vector<unsigned char> buf;
    bool ok = write(out.fd, "KMCS", 4) == 4;
    for (const KmcPart& x : P) {
        if (!ok || !x.h.total) continue;
        const int in = open(x.suf.c_str(), O_RDONLY);
        ok = in >= 0 && copy_range(in, 4, x.h.total * x.rec, out.fd, buf);
        if (in >= 0) close(in);
    }
    ok = ok && write(out.fd, "KMCS", 4) == 4;
    ok = (close(out.fd) == 0) && ok;
    out.fd = -1;
    if (!ok) { mlg_set_error("%s: short write (%s)", suf_path.c_str(), strerror(errno)); return MLG_ERR_IO; }
    unsigned long long pre_bytes = 0;
    MLG_TRY(kmc_write_pre(pre_path, lut, h, &pre_bytes));
    out.done = true;
    return MLG_OK;
}
