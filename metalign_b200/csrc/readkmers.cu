// Read k-mer table (include/metalign_b200.h, mlg_query_enable_read_kmers): every canonical K-mer (K <= 60) of the pushed
// reads with a saturating 8-bit count -- the counting part of `kmc -k<K> -ci<min> -cs<max>` -- and the KMC database files
// written from it and from the query's intersection.  The count kernel runs beside K1 on the compute stream, over the same
// staged batch; K1 itself does not know the table exists.  DESIGN.md section 10.
#include <cub/cub.cuh>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <chrono>
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
};

// One thread per window start: a CTA takes 256 consecutive base positions of the range, so the work is the same per
// window whatever the read lengths are.  The read of a position is found by a binary search inside the few reads the
// tile spans.
__global__ void __launch_bounds__(RK_TPB) k_count_read_kmers(CountArgs a) {
    __shared__ unsigned long long s_r[2];
    const unsigned long long b0 = a.off ? a.off[a.r_begin] : a.r_begin * (unsigned long long)a.read_len;
    const unsigned long long b1 = a.off ? a.off[a.r_end] : a.r_end * (unsigned long long)a.read_len;
    const unsigned K = a.K;
    unsigned long long n_new = 0, n_win = 0;
    for (unsigned long long p0 = b0 + (unsigned long long)blockIdx.x * RK_TPB; p0 < b1; p0 += (unsigned long long)gridDim.x * RK_TPB) {
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
        int fresh = 0;
        if (ok) {
            const unsigned long long w = p >> 5; const unsigned b = (unsigned)(p & 31) * 2;
            const unsigned long long x = be_word(a.bases, w, a.base_words), y = be_word(a.bases, w + 1, a.base_words),
                                     z = be_word(a.bases, w + 2, a.base_words);
            key128 t;
            t.hi = b ? (x << b) | (y >> (64 - b)) : x;
            t.lo = b ? (y << b) | (z >> (64 - b)) : y;
            const key128 c = key_canon(key_shr(t, 128 - 2 * K), K);
            fresh = rk_insert(a.tab, a.line_mask, c.hi, c.lo, a.ctr + 2);
        }
        const int nf = __syncthreads_count(fresh), nw = __syncthreads_count(ok);
        n_new += nf; n_win += nw;
    }
    if (threadIdx.x == 0 && (n_new | n_win)) { atomicAdd(a.ctr, n_new); atomicAdd(a.ctr + 1, n_win); }
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
    auto slots_for = [](unsigned long long b) { unsigned long long s = RK_MIN_SLOTS; while ((double)s * RK_LOAD < (double)b) s *= 2; return s; };
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
    k_count_read_kmers<<<grid_for(batch_bases, t->ctx->sm_count * 16), RK_TPB, 0, st>>>(a);
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

// the table's keys seen >= min_count times, sorted, with their counts (saturated at 255)
int rk_collect(ReadKmerTable* t, uint32_t min_count, DevBuf<key128>& keys, DevBuf<uint32_t>& cnt, uint32_t* n_out, KmcOutStats* ws) {
    cudaStream_t st = t->ctx->s_comp;
    cudaEvent_t e0, e1, e2;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1)); CUDA_TRY(cudaEventCreate(&e2));
    struct Ev { cudaEvent_t* e; ~Ev() { for (int i = 0; i < 3; ++i) cudaEventDestroy(e[i]); } };
    cudaEvent_t evs[3] = {e0, e1, e2}; Ev guard{evs};
    CUDA_TRY(cudaEventRecord(e0, st));
    unsigned long long distinct = 0;
    CUDA_TRY(cudaMemcpyAsync(&distinct, t->ctr.p, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (distinct >= (1ull << 32)) { mlg_set_error("%llu distinct read k-mers: more than the output stage sorts (2^32)", distinct); return MLG_ERR_ARG; }
    DevBuf<Slot> sel; MLG_TRY(sel.alloc(distinct));
    DevBuf<unsigned long long> d_n; MLG_TRY(d_n.alloc(1));
    unsigned long long n = 0;
    const unsigned long long CH = 1ull << 30;                 // cub's item count is an int
    for (unsigned long long s0 = 0; s0 < t->nslots; s0 += CH) {
        const int m = (int)std::min(CH, t->nslots - s0);
        size_t tb = 0;
        CUDA_TRY(cub::DeviceSelect::If(nullptr, tb, t->tab.p + s0, sel.p + n, d_n.p, m, AtLeast{min_count}, st));
        DevBuf<unsigned char> tmp; MLG_TRY(tmp.alloc(tb ? tb : 1));
        CUDA_TRY(cub::DeviceSelect::If(tmp.p, tb, t->tab.p + s0, sel.p + n, d_n.p, m, AtLeast{min_count}, st));
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
        MLG_TRY(sort_keys128(hi.p, lo.p, c.p, (uint32_t)n, t->K, keys.p, cnt.p, st));
    }
    CUDA_TRY(cudaEventRecord(e2, st));
    CUDA_TRY(cudaEventSynchronize(e2));
    float ms = 0;
    if (ws && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) ws->ms_compact = ms;
    if (ws && cudaEventElapsedTime(&ms, e1, e2) == cudaSuccess) ws->ms_sort = ms;
    return MLG_OK;
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

// <prefix>.kmc_pre / .kmc_suf, version-0 layout (one sorted table, as kmc_tools writes it): n sorted keys with counts,
// counts saturated at counter_max; the records are packed on the device and copied back in chunks through two pinned
// buffers, each chunk's fwrite overlapping the next chunk's copy
int kmc_write(mlg_ctx* ctx, const char* prefix, const key128* keys, const uint32_t* cnt, uint32_t n, uint32_t K, uint32_t min_count,
              uint32_t counter_max, KmcOutStats* ws) {
    if (K < 5 || K > 60) { mlg_set_error("KMC files need 5 <= K <= 60 here (K = %u)", K); return MLG_ERR_ARG; }
    cudaStream_t st = ctx->s_comp;
    const uint32_t p = kmc_prefix_len(K), rec = (K - p) / 4 + 1;
    const unsigned long long np = 1ull << (2 * p), sbytes = (unsigned long long)n * rec;
    DevBuf<unsigned long long> d_lut; MLG_TRY(d_lut.alloc(np + 1));
    DevBuf<unsigned char> d_rec; MLG_TRY(d_rec.alloc(sbytes));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, st));
    k_kmc_lut<<<(unsigned)((np + 256) / 256), 256, 0, st>>>(keys, n, K, p, d_lut.p);
    if (n) k_kmc_records<<<(n + 255) / 256, 256, 0, st>>>(keys, cnt, n, K, p, counter_max, d_rec.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(e1, st));
    std::vector<unsigned long long> lut(np + 1);
    CUDA_TRY(cudaMemcpyAsync(lut.data(), d_lut.p, (np + 1) * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    float ms = 0;
    if (ws && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) ws->ms_encode = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);

    const auto t0 = std::chrono::steady_clock::now();
    const std::string pre_path = std::string(prefix) + ".kmc_pre", suf_path = std::string(prefix) + ".kmc_suf";
    FILE* fs = fopen(suf_path.c_str(), "wb");
    if (!fs) { mlg_set_error("cannot create %s", suf_path.c_str()); return MLG_ERR_IO; }
    bool ok = fwrite("KMCS", 1, 4, fs) == 4;
    const unsigned long long CH = 32ull << 20;
    unsigned char* pin[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    int rc = MLG_OK;
    if (sbytes) {
        if (cudaMallocHost(&pin[0], std::min(CH, sbytes)) != cudaSuccess || cudaMallocHost(&pin[1], std::min(CH, sbytes)) != cudaSuccess ||
            cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming) != cudaSuccess) {
            mlg_set_error("pinned staging for %s failed: %s", suf_path.c_str(), cudaGetErrorString(cudaGetLastError())); rc = MLG_ERR_CUDA;
        }
        const unsigned long long nch = (sbytes + CH - 1) / CH;
        for (unsigned long long c = 0; rc == MLG_OK && c <= nch; ++c) {
            if (c < nch) {
                const unsigned long long b = std::min(CH, sbytes - c * CH);
                if (cudaMemcpyAsync(pin[c & 1], d_rec.p + c * CH, b, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                    cudaEventRecord(ev[c & 1], st) != cudaSuccess) { mlg_set_error("copy of %s failed", suf_path.c_str()); rc = MLG_ERR_CUDA; break; }
            }
            if (c > 0) {
                const unsigned long long pc = c - 1, b = std::min(CH, sbytes - pc * CH);
                if (cudaEventSynchronize(ev[pc & 1]) != cudaSuccess) { mlg_set_error("copy of %s failed", suf_path.c_str()); rc = MLG_ERR_CUDA; break; }
                ok = ok && fwrite(pin[pc & 1], 1, b, fs) == b;
            }
        }
        cudaStreamSynchronize(st);
        for (int i = 0; i < 2; ++i) { if (pin[i]) cudaFreeHost(pin[i]); if (ev[i]) cudaEventDestroy(ev[i]); }
    }
    ok = ok && fwrite("KMCS", 1, 4, fs) == 4;
    ok = (fclose(fs) == 0) && ok;
    if (rc != MLG_OK) return rc;
    if (!ok) { mlg_set_error("%s: short write", suf_path.c_str()); return MLG_ERR_IO; }

    // .kmc_pre: "KMCP" | LUT (+ guard) | header | header bytes | "KMCP"   (csrc/kmcdb.h)
    std::vector<unsigned char> pre;
    auto put = [&](const void* v, size_t b) { const unsigned char* c = (const unsigned char*)v; pre.insert(pre.end(), c, c + b); };
    auto u32 = [&](uint32_t v) { put(&v, 4); };
    put("KMCP", 4);
    put(lut.data(), lut.size() * 8);
    const size_t h0 = pre.size();
    u32(K); u32(0); u32(1); u32(p);                                 // k, mode (counters), counter_size, lut_prefix_length
    u32(min_count); u32(counter_max);
    const unsigned long long total = n; put(&total, 8);
    const unsigned char hdr_tail[4] = {0, 0, 0, 0}; put(hdr_tail, 4);  // both strands (canonical) + 3 pad bytes
    u32(0);                                                          // max_count, high word
    const unsigned char reserved[20] = {}; put(reserved, 20);
    u32(0);                                                          // kmc_version 0
    u32((uint32_t)(pre.size() - h0));
    put("KMCP", 4);
    FILE* fp = fopen(pre_path.c_str(), "wb");
    if (!fp) { mlg_set_error("cannot create %s", pre_path.c_str()); return MLG_ERR_IO; }
    ok = fwrite(pre.data(), 1, pre.size(), fp) == pre.size();
    ok = (fclose(fp) == 0) && ok;
    if (!ok) { mlg_set_error("%s: short write", pre_path.c_str()); return MLG_ERR_IO; }
    if (ws) {
        ws->records = n; ws->bytes = pre.size() + sbytes + 8;
        ws->s_write = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    }
    return MLG_OK;
}
