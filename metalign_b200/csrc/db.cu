// Database build: turns G*n sketch slots (stored-orientation K-mers, '' = empty) into the
// HBM-resident structures the query kernels use.  Replaces, for this path, CMash's training HDF5 +
// marisa-trie `.tst` + hydra Bloom prefilter (scripts/select_db.py:69-70) and the KMC database of the
// dumped sketch k-mers (scripts/select_db.py:44; local_tests/retrain_and_test_metalign.sh:49-66).
//
//   P   all non-empty slots sorted by key + slot id payload, with a bucket index on the top bits of
//       the key ("bucketed binary search": a k-prefix query is a key range, every k served by one array)
//   rep per queried k: representative slot of each (genome, k-prefix) class -> numerators dedupe by
//       prefix exactly like CMash's per-genome `unique_kmers` set; class counts are the denominators
//   D   distinct canonical keys, sorted by a 64-bit hash; level-1 table of 16/32-byte buckets of 31-bit
//       fingerprints so that a read k-mer that is NOT in the database (>99.9 % of them) costs exactly
//       one DRAM sector; bstart maps a bucket back to its run of D for exact verification
//
// Everything runs on the device (CUB radix sorts / scans + small kernels).
#include <cub/cub.cuh>
#include <math.h>
#include <algorithm>
#include <stdlib.h>
#include <string.h>
#include "mlg_internal.h"

namespace {

constexpr int TPB = 256;
inline unsigned nblk(unsigned long long n) { return (unsigned)((n + TPB - 1) / TPB); }

// ---------------------------------------------------------------- small kernels
__global__ void k_mark_nonempty(const key128* keys, unsigned long long total, uint32_t n, unsigned char* flag,
                                unsigned char* has_empty) {
    unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (s >= total) return;
    bool e = key_is_empty(keys[s]);
    flag[s] = e ? 0 : 1;
    if (e) has_empty[s / n] = 1;
}
__global__ void k_gather_split(const key128* keys, const uint32_t* slots, uint32_t np, unsigned long long* hi,
                               unsigned long long* lo) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    key128 k = keys[slots[i]];
    hi[i] = k.hi; lo[i] = k.lo;
}
__global__ void k_iota(uint32_t* a, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = i;
}
__global__ void k_gather_u64(const unsigned long long* src, const uint32_t* idx, uint32_t n, unsigned long long* dst) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[idx[i]];
}
__global__ void k_gather_u32(const uint32_t* src, const uint32_t* idx, uint32_t n, uint32_t* dst) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[idx[i]];
}
// out[i] = {hi[i], lo_sorted[perm[i]]}
__global__ void k_zip_keys(const unsigned long long* hi, const unsigned long long* lo_sorted, const uint32_t* perm,
                           uint32_t n, key128* out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    key128 k; k.hi = hi[i]; k.lo = lo_sorted[perm ? perm[i] : i];
    out[i] = k;
}
__global__ void k_pbucket_hist(const key128* P, uint32_t np, uint32_t K, uint32_t pbits, uint32_t* counts) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    key128 b = key_shr(P[i], 2 * K - pbits);
    atomicAdd(&counts[(uint32_t)b.lo], 1u);
}
__global__ void k_slot_to_genome(const uint32_t* slot, uint32_t np, uint32_t n, uint32_t* g) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < np) g[i] = slot[i] / n;
}
// q-order = entries sorted by (genome, key).  A (genome, k-prefix) class is a run in q-order; its
// representative is the slot of the run head.
__global__ void k_rep_classes(const key128* P, const uint32_t* P_slot, const uint32_t* q2p, uint32_t np, uint32_t n,
                              uint32_t K, uint32_t k, uint32_t ki, uint32_t nk, uint32_t* rep_k, long long* den_real) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= np) return;
    uint32_t i = q2p[q];
    uint32_t slot = P_slot[i];
    uint32_t g = slot / n;
    key128 pre = key_prefix(P[i], K, k);
    uint32_t h = q;
    while (h > 0) {
        uint32_t ip = q2p[h - 1];
        if (P_slot[ip] / n != g) break;
        if (!key_eq(key_prefix(P[ip], K, k), pre)) break;
        --h;
    }
    rep_k[slot] = P_slot[q2p[h]];
    if (h == q) atomicAdd((unsigned long long*)&den_real[(size_t)g * nk + ki], 1ull);
}
__global__ void k_canon_split(const key128* P, uint32_t np, uint32_t K, unsigned long long* hi, unsigned long long* lo) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    key128 c = key_canon(P[i], K);
    hi[i] = c.hi; lo[i] = c.lo;
}
__global__ void k_flag_heads(const key128* a, uint32_t n, unsigned char* flag) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flag[i] = (i == 0 || !key_eq(a[i], a[i - 1])) ? 1 : 0;
}
// length of the run of equal keys that starts at every head, saturating at 255 (the number of sketch slots that hold the K-mer)
__global__ void k_run_lengths(const unsigned char* head, uint32_t n, unsigned char* len) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t l = 0;
    if (head[i]) { l = 1; while (l < 255u && i + l < n && !head[i + l]) ++l; }
    len[i] = (unsigned char)l;
}
__global__ void k_gather_u8(const unsigned char* src, const uint32_t* idx, uint32_t n, unsigned char* dst) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[idx[i]];
}
__global__ void k_hash_keys(const key128* a, uint32_t n, uint32_t K, uint32_t layout, uint32_t bbits, unsigned long long* h) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) h[i] = layout == 2 ? key_hash_mz(a[i], K) : layout == 1 ? key_hash_sk(a[i], K, bbits) : key_hash(a[i], K);
}
// layout 2: level-1 bits of the identities of every K-mer's leftmost and rightmost minimum (kmer.cuh), and the alias
// entries of the K-mers whose two identities differ (pass 0 counts them, pass 1 writes them)
__global__ void k_fill_mzbits(const key128* D, uint32_t nd, uint32_t K, uint32_t fbits, uint32_t* MB, int pass,
                              unsigned long long* alias_z, uint32_t* alias_i, uint32_t* alias_bloom, unsigned long long* counter) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nd) return;
    unsigned long long zL, zR;
    key_mz(D[i], K, &zL, &zR);
    if (pass == 0) {
        const unsigned long long bl = mz_bit_index(zL, fbits), br = mz_bit_index(zR, fbits);
        atomicOr(&MB[bl >> 5], (1u << (bl & 31ull)) | (1u << mz_bit2((uint32_t)(zL >> 32))));
        if (zR != zL) { atomicOr(&MB[br >> 5], (1u << (br & 31ull)) | (1u << mz_bit2((uint32_t)(zR >> 32)))); atomicAdd(counter, 1ull); }
    } else if (zR != zL) {
        const unsigned long long j = atomicAdd(counter, 1ull);
        alias_z[j] = zR; alias_i[j] = i;
        const uint32_t zlo = (uint32_t)zR;
        atomicOr(&alias_bloom[(zlo & 0xFFFFu) >> 5], 1u << (zlo & 31u));
    }
}
__global__ void k_gather_key(const key128* src, const uint32_t* idx, uint32_t n, key128* dst) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[idx[i]];
}
__global__ void k_hbucket_hist(const unsigned long long* h, uint32_t nd, uint32_t bbits, uint32_t* counts) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nd) atomicAdd(&counts[hash_bucket(h[i], bbits)], 1u);
}
__global__ void k_fill_filter(const unsigned long long* h, uint32_t nd, uint32_t nfw, uint32_t fk, uint32_t* F) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nd) atomicOr(&F[filter_word(h[i], nfw)], filter_mask(h[i], fk));
}
__global__ void k_fill_t1(const unsigned long long* h, uint32_t nd, uint32_t bbits, const uint32_t* bstart,
                          uint32_t slots, uint32_t layout, uint32_t* T1) {
    uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nd) return;
    unsigned long long b = hash_bucket(h[e], bbits);
    uint32_t s = e - bstart[b];
    uint32_t c = bstart[b + 1] - bstart[b];
    if (s < slots) {
        uint32_t v = hash_fp(h[e]);
        // more entries than slots: the probe must take the exact path.  Layout 0 flags it in bit 31 of the first slot;
        // layout 1 needs no flag, it treats every FULL bucket as overflowed
        if (s == 0 && c > slots && layout == 0) v |= 0x80000000u;
        T1[b * slots + s] = v;
    }
}

struct IsNonEmpty {
    const unsigned char* flag;
    __host__ __device__ bool operator()(const uint32_t& s) const { return flag[s] != 0; }
};

// exclusive prefix sum of counts[0..m) into out[0..m], out[m] = total
int exclusive_scan_u32(uint32_t* counts_inout_m_plus_1, size_t m, cudaStream_t st) {
    // counts has m+1 entries with counts[m] == 0; in-place exclusive sum over m+1 entries gives the bucket starts
    void* tmp = nullptr; size_t tb = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, counts_inout_m_plus_1, counts_inout_m_plus_1, m + 1, st));
    CUDA_TRY(cudaMalloc(&tmp, tb ? tb : 1));
    cudaError_t e = cub::DeviceScan::ExclusiveSum(tmp, tb, counts_inout_m_plus_1, counts_inout_m_plus_1, m + 1, st);
    cudaStreamSynchronize(st);
    cudaFree(tmp);
    if (e != cudaSuccess) { mlg_set_error("DeviceScan failed: %s", cudaGetErrorString(e)); return MLG_ERR_CUDA; }
    return MLG_OK;
}

// stable radix sort of (u64 key, u32 value) pairs; results land in keys_out / vals_out
int sort_pairs_u64(const unsigned long long* keys_in, unsigned long long* keys_out, const uint32_t* vals_in,
                   uint32_t* vals_out, uint32_t n, int begin_bit, int end_bit, cudaStream_t st) {
    void* tmp = nullptr; size_t tb = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tb, keys_in, keys_out, vals_in, vals_out, (int)n, begin_bit, end_bit, st));
    CUDA_TRY(cudaMalloc(&tmp, tb ? tb : 1));
    cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, tb, keys_in, keys_out, vals_in, vals_out, (int)n, begin_bit, end_bit, st);
    cudaStreamSynchronize(st);
    cudaFree(tmp);
    if (e != cudaSuccess) { mlg_set_error("DeviceRadixSort failed: %s", cudaGetErrorString(e)); return MLG_ERR_CUDA; }
    return MLG_OK;
}
int sort_pairs_u32(const uint32_t* keys_in, uint32_t* keys_out, const uint32_t* vals_in, uint32_t* vals_out, uint32_t n,
                   int end_bit, cudaStream_t st) {
    void* tmp = nullptr; size_t tb = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tb, keys_in, keys_out, vals_in, vals_out, (int)n, 0, end_bit, st));
    CUDA_TRY(cudaMalloc(&tmp, tb ? tb : 1));
    cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, tb, keys_in, keys_out, vals_in, vals_out, (int)n, 0, end_bit, st);
    cudaStreamSynchronize(st);
    cudaFree(tmp);
    if (e != cudaSuccess) { mlg_set_error("DeviceRadixSort failed: %s", cudaGetErrorString(e)); return MLG_ERR_CUDA; }
    return MLG_OK;
}

}  // namespace

// Sort n 2K-bit keys given as split (hi, lo) arrays; on return out[i] is the i-th smallest key and, if
// vals is non-null, vals_out[i] the value that travelled with it.  LSD: by lo, then stably by hi.
int sort_keys128(unsigned long long* hi, unsigned long long* lo, const uint32_t* vals, uint32_t n, uint32_t K,
                 key128* out, uint32_t* vals_out, cudaStream_t st) {
    if (n == 0) return MLG_OK;
    DevBuf<unsigned long long> lo_s, hi_g, hi_s;
    DevBuf<uint32_t> iota, perm1, perm2;
    MLG_TRY(lo_s.alloc(n)); MLG_TRY(iota.alloc(n)); MLG_TRY(perm1.alloc(n));
    k_iota<<<nblk(n), TPB, 0, st>>>(iota.p, n);
    int lo_bits = (2 * K < 64) ? (int)(2 * K) : 64;
    MLG_TRY(sort_pairs_u64(lo, lo_s.p, iota.p, perm1.p, n, 0, lo_bits, st));
    const uint32_t* final_perm = perm1.p;   // position in sorted order -> original index
    if (2 * K > 64) {
        MLG_TRY(hi_g.alloc(n)); MLG_TRY(hi_s.alloc(n)); MLG_TRY(perm2.alloc(n));
        k_gather_u64<<<nblk(n), TPB, 0, st>>>(hi, perm1.p, n, hi_g.p);
        MLG_TRY(sort_pairs_u64(hi_g.p, hi_s.p, iota.p, perm2.p, n, 0, (int)(2 * K - 64), st));
        // perm2[i] = position in the lo-sorted order
        k_zip_keys<<<nblk(n), TPB, 0, st>>>(hi_s.p, lo_s.p, perm2.p, n, out);
        if (vals_out) {
            // original index = perm1[perm2[i]]
            k_gather_u32<<<nblk(n), TPB, 0, st>>>(perm1.p, perm2.p, n, iota.p);   // iota reused as composed perm
            final_perm = iota.p;
        }
    } else {
        DevBuf<unsigned long long> zero; MLG_TRY(zero.alloc(n));
        CUDA_TRY(cudaMemsetAsync(zero.p, 0, (size_t)n * 8, st));
        k_zip_keys<<<nblk(n), TPB, 0, st>>>(zero.p, lo_s.p, nullptr, n, out);
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    if (vals_out) {
        if (vals) k_gather_u32<<<nblk(n), TPB, 0, st>>>(vals, final_perm, n, vals_out);
        else CUDA_TRY(cudaMemcpyAsync(vals_out, final_perm, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}

namespace {

// level-1 table geometry from the number of distinct keys: slots per bucket and number of buckets (a power of two)
void choose_buckets(DbView& v, uint32_t nd) {
    uint32_t slots_per_bucket = 8;
    if (const char* s = getenv("MLG_BUCKET_SLOTS")) { int x = atoi(s); if (x == 4 || x == 8) slots_per_bucket = (uint32_t)x; }
    double load = slots_per_bucket * 0.3125;  // upper bound on the mean entries per bucket (2.5 of 8 slots)
    if (const char* s = getenv("MLG_BUCKET_LOAD")) { double x = atof(s); if (x > 0.01 && x <= slots_per_bucket) load = x; }
    uint32_t bbits = 1;                       // at least two buckets: the probe kernel shifts by 32 - bbits
    if (v.layout == 1) {
        // k-mers that share a minimizer share a bucket PAIR (kmer.cuh), so occupancy is clumpier than a plain hash's;
        // mean load <= 1.25 per 8-slot half keeps the overflowing halves rare
        slots_per_bucket = 8; load = 1.25; bbits = 2;
        if (const char* s = getenv("MLG_SK_LOAD")) { double x = atof(s); if (x > 0.01 && x <= 8) load = x; }
    }
    if (v.layout == 2) {
        // the bucket index only serves the exact compare of the few super-k-mers whose minimizer is in the database
        slots_per_bucket = 8; load = 2.5; bbits = 1;
        if (const char* s = getenv("MLG_MZ_LOAD")) { double x = atof(s); if (x > 0.01 && x <= 64) load = x; }
    }
    while (bbits < 31 && (double)(1ull << bbits) * load < (double)nd) ++bbits;
    v.nbuckets = 1ull << bbits; v.bbits = bbits; v.slots = slots_per_bucket;
}


// ---------------------------------------------------------------- memory-lean build helpers
// one chunk of genomes: non-empty slots flagged, emptiness noted per genome
__global__ void k_mark_nonempty_chunk(const key128* keys, unsigned long long total, uint32_t n, uint32_t g0, unsigned char* flag,
                                      unsigned char* has_empty) {
    unsigned long long s = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (s >= total) return;
    bool e = key_is_empty(keys[s]);
    flag[s] = e ? 0 : 1;
    if (e) has_empty[g0 + s / n] = 1;
}
// the chunk's non-empty keys appended to the builder's split arrays; slot ids are global (g * n + j)
__global__ void k_append_split(const key128* keys, const uint32_t* sel, uint32_t cnt, uint32_t slot0, unsigned long long* hi,
                               unsigned long long* lo, uint32_t* slot) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt) return;
    const key128 k = keys[sel[i]];
    hi[i] = k.hi; lo[i] = k.lo; slot[i] = slot0 + sel[i];
}
__global__ void k_canon_split2(const unsigned long long* hi, const unsigned long long* lo, uint32_t np, uint32_t K,
                               unsigned long long* chi, unsigned long long* clo) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    key128 k; k.hi = hi[i]; k.lo = lo[i];
    const key128 c = key_canon(k, K);
    chi[i] = c.hi; clo[i] = c.lo;
}
__global__ void k_flag_heads2(const unsigned long long* hi, const unsigned long long* lo, uint32_t n, unsigned char* flag) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    flag[i] = (i == 0 || hi[i] != hi[i - 1] || lo[i] != lo[i - 1]) ? 1 : 0;
}
__global__ void k_hash_keys2(const unsigned long long* hi, const unsigned long long* lo, uint32_t n, uint32_t K, uint32_t layout,
                             uint32_t bbits, unsigned long long* h) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    key128 a; a.hi = hi[i]; a.lo = lo[i];
    h[i] = layout == 2 ? key_hash_mz(a, K) : layout == 1 ? key_hash_sk(a, K, bbits) : key_hash(a, K);
}
__global__ void k_gather_key2(const unsigned long long* hi, const unsigned long long* lo, const uint32_t* idx, uint32_t n, key128* dst) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    key128 k; k.hi = hi[idx[i]]; k.lo = lo[idx[i]];
    dst[i] = k;
}

// Two buffers a radix sort ping-pongs between (cub::DoubleBuffer): the sort then needs no scratch of the input's size,
// which is what lets a 2e9-slot database build inside 180 GB.
template <typename T>
struct PingPong {
    DevBuf<T> buf[2];
    int sel = 0;
    T* cur() { return buf[sel].p; }
    T* alt() { return buf[sel ^ 1].p; }
    int alloc_alt(size_t n) { return buf[sel ^ 1].alloc(n); }
    void adopt(DevBuf<T>& src) { buf[0].release(); buf[0].p = src.p; buf[0].n = src.n; src.p = nullptr; src.n = 0; sel = 0; }
    void drop_alt() { buf[sel ^ 1].release(); }
    void drop() { buf[0].release(); buf[1].release(); }
};
// scratch for the CUB calls comes from the pool (which gives cached blocks back to the driver before it fails)
template <typename KeyT, typename ValT>
int radix_pairs(PingPong<KeyT>& k, PingPong<ValT>& v, uint32_t n, int begin_bit, int end_bit, cudaStream_t st) {
    if (n == 0 || end_bit <= begin_bit) return MLG_OK;
    cub::DoubleBuffer<KeyT> dk(k.cur(), k.alt());
    cub::DoubleBuffer<ValT> dv(v.cur(), v.alt());
    size_t tb = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tb, dk, dv, (int)n, begin_bit, end_bit, st));
    DevBuf<unsigned char> tmp; MLG_TRY(tmp.alloc(tb ? tb : 1));
    cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp.p, tb, dk, dv, (int)n, begin_bit, end_bit, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { mlg_set_error("DeviceRadixSort failed: %s", cudaGetErrorString(e)); return MLG_ERR_CUDA; }
    k.sel = dk.Current() == k.buf[0].p ? 0 : 1;
    v.sel = dv.Current() == v.buf[0].p ? 0 : 1;
    return MLG_OK;
}
template <typename T>
int select_flagged(const T* in, const unsigned char* flags, T* out, unsigned long long* d_count, uint32_t n, cudaStream_t st) {
    size_t tb = 0;
    CUDA_TRY(cub::DeviceSelect::Flagged(nullptr, tb, in, flags, out, d_count, (int)n, st));
    DevBuf<unsigned char> tmp; MLG_TRY(tmp.alloc(tb ? tb : 1));
    cudaError_t e = cub::DeviceSelect::Flagged(tmp.p, tb, in, flags, out, d_count, (int)n, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { mlg_set_error("DeviceSelect failed: %s", cudaGetErrorString(e)); return MLG_ERR_CUDA; }
    return MLG_OK;
}

}  // namespace

// ---- the builder: genomes arrive in chunks (the caller never has to hold all G*n keys on the device), the non-empty
// slots are kept as split (hi, lo, slot) arrays, and finish() derives the device structures from them stage by stage,
// every stage releasing what the next one does not read.  Peak device memory for 2e9 slots: ~145 GB (the radix sorts
// ping-pong between two buffers instead of taking scratch of the input's size, D is built before P, and the hit records
// are only precomputed when they fit beside P and the class representatives).
struct mlg_db_builder {
    mlg_ctx* ctx = nullptr;
    uint32_t G = 0, n = 0, K = 0, nk = 0, ks[MLG_MAX_KS] = {};
    DevBuf<unsigned long long> hi, lo;
    DevBuf<uint32_t> slot;
    DevBuf<unsigned char> has_empty;
    uint32_t np = 0, next_g = 0;
};

int mlg_db_builder_create_impl(mlg_ctx* ctx, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks, uint32_t nk, mlg_db_builder** out) {
    if (!ctx || !out || !ks) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (K < 1 || K > 63) { mlg_set_error("K=%u out of range 1..63", K); return MLG_ERR_ARG; }
    if (nk < 1 || nk > MLG_MAX_KS) { mlg_set_error("nk=%u out of range 1..%d", nk, MLG_MAX_KS); return MLG_ERR_ARG; }
    for (uint32_t i = 0; i < nk; ++i)
        if (ks[i] < 1 || ks[i] > K || (i && ks[i] <= ks[i - 1])) { mlg_set_error("ks must be ascending and within 1..K"); return MLG_ERR_ARG; }
    if (K - ks[0] + 1 > 64) { mlg_set_error("K - ks[0] + 1 must be <= 64"); return MLG_ERR_ARG; }
    const unsigned long long total = (unsigned long long)G * n;
    if (G == 0 || n == 0 || total >= 0x7FFFFFF0ull) { mlg_set_error("G*n=%llu out of range (1 .. 2^31-16)", total); return MLG_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(ctx->device));
    mlg_db_builder* b = new mlg_db_builder();
    b->ctx = ctx; b->G = G; b->n = n; b->K = K; b->nk = nk;
    for (uint32_t i = 0; i < nk; ++i) b->ks[i] = ks[i];
    int rc = b->hi.alloc(total);
    if (rc == MLG_OK) rc = b->lo.alloc(total);
    if (rc == MLG_OK) rc = b->slot.alloc(total);
    if (rc == MLG_OK) rc = b->has_empty.alloc(G);
    if (rc == MLG_OK && cudaMemsetAsync(b->has_empty.p, 0, G, ctx->s_comp) != cudaSuccess) { mlg_set_error("memset failed"); rc = MLG_ERR_CUDA; }
    if (rc != MLG_OK) { delete b; return rc; }
    *out = b;
    return MLG_OK;
}

int mlg_db_builder_add_impl(mlg_db_builder* b, const key128* d_keys, uint32_t g0, uint32_t count) {
    if (!b || !d_keys) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (g0 != b->next_g || count == 0 || (unsigned long long)g0 + count > b->G) {
        mlg_set_error("genomes must be added in order without gaps (expected genome %u, got %u..%u of %u)", b->next_g, g0, g0 + count, b->G);
        return MLG_ERR_ARG;
    }
    CUDA_TRY(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->ctx->s_comp;
    const unsigned long long total = (unsigned long long)count * b->n;
    DevBuf<unsigned char> flag; MLG_TRY(flag.alloc(total));
    DevBuf<uint32_t> sel; MLG_TRY(sel.alloc(total));
    DevBuf<unsigned long long> d_cnt; MLG_TRY(d_cnt.alloc(1));
    k_mark_nonempty_chunk<<<nblk(total), TPB, 0, st>>>(d_keys, total, b->n, g0, flag.p, b->has_empty.p);
    {
        cub::CountingInputIterator<uint32_t> it(0);
        IsNonEmpty pred{flag.p};
        size_t tb = 0;
        CUDA_TRY(cub::DeviceSelect::If(nullptr, tb, it, sel.p, d_cnt.p, (int)total, pred, st));
        DevBuf<unsigned char> tmp; MLG_TRY(tmp.alloc(tb ? tb : 1));
        cudaError_t e = cub::DeviceSelect::If(tmp.p, tb, it, sel.p, d_cnt.p, (int)total, pred, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { mlg_set_error("DeviceSelect failed: %s", cudaGetErrorString(e)); return MLG_ERR_CUDA; }
    }
    unsigned long long c64 = 0;
    CUDA_TRY(cudaMemcpy(&c64, d_cnt.p, 8, cudaMemcpyDeviceToHost));
    const uint32_t c = (uint32_t)c64;
    if (c) k_append_split<<<nblk(c), TPB, 0, st>>>(d_keys, sel.p, c, g0 * b->n, b->hi.p + b->np, b->lo.p + b->np, b->slot.p + b->np);
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    b->np += c;
    b->next_g = g0 + count;
    return MLG_OK;
}

void mlg_db_builder_destroy_impl(mlg_db_builder* b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    delete b;
}

int mlg_db_builder_finish_impl(mlg_db_builder* b, mlg_db** out) {
    if (!b || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (b->next_g != b->G) { mlg_set_error("only %u of %u genomes were added", b->next_g, b->G); return MLG_ERR_STATE; }
    mlg_ctx* ctx = b->ctx;
    const uint32_t G = b->G, n = b->n, K = b->K, nk = b->nk, np = b->np;
    const uint32_t* ks = b->ks;
    const unsigned long long total = (unsigned long long)G * n;
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->s_comp;
    cudaEvent_t e0, e1; CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, st));

    mlg_db* db = new mlg_db();
    db->ctx = ctx;
    struct Guard { mlg_db* d; ~Guard() { if (d) delete d; } } guard{db};
    DbView& v = db->v;
    v.G = G; v.n = n; v.K = K; v.nk = nk; v.np = np;
    // Metalign's K = 60 gets the minimizer-bitmap layout (kmer.cuh); other K keep the whole-k-mer hash layout.
    // MLG_LAYOUT=0 / 1 force the whole-k-mer hash layout / the fingerprint-pair super-k-mer layout (A/B measurements).
    v.layout = (K == 60) ? 2u : 0u;
    if (const char* s = getenv("MLG_LAYOUT")) { int x = atoi(s); if (x == 0 || (x == 1 && K == 60)) v.layout = (uint32_t)x; }
    for (uint32_t i = 0; i < MLG_MAX_KS; ++i) v.ks[i] = i < nk ? ks[i] : 0;
    db->has_empty.p = b->has_empty.p; db->has_empty.n = b->has_empty.n; b->has_empty.p = nullptr; b->has_empty.n = 0;
    DevBuf<unsigned long long> d_cnt; MLG_TRY(d_cnt.alloc(1));
    const int lo_bits = (2 * K < 64) ? (int)(2 * K) : 64, hi_bits = (2 * K > 64) ? (int)(2 * K - 64) : 0;
    const bool verbose = getenv("MLG_VERBOSE_BUILD") != nullptr;
    auto stage = [&](const char* what) {      // MLG_VERBOSE_BUILD=1: device memory in use after every stage (stderr)
        if (!verbose) return;
        cudaStreamSynchronize(st);
        mlg_pool_trim(ctx->device);
        size_t f = 0, t = 0; cudaMemGetInfo(&f, &t);
        fprintf(stderr, "[mlg build] %-28s in use %.1f GB of %.1f\n", what, (double)(t - f) / 1e9, (double)t / 1e9);
    };
    stage("builder arrays");

    // 1. D first (it only reads the builder's arrays): distinct canonical keys with their multiplicities, hash-ordered
    uint32_t nd = 0;
    DevBuf<unsigned long long> hsorted;
    if (np) {
        PingPong<unsigned long long> chi, clo;
        MLG_TRY(chi.buf[0].alloc(np)); MLG_TRY(clo.buf[0].alloc(np));
        k_canon_split2<<<nblk(np), TPB, 0, st>>>(b->hi.p, b->lo.p, np, K, chi.cur(), clo.cur());
        MLG_TRY(chi.alloc_alt(np)); MLG_TRY(clo.alloc_alt(np));
        MLG_TRY(radix_pairs(clo, chi, np, 0, lo_bits, st));           // LSD: by the low word carrying the high one ...
        MLG_TRY(radix_pairs(chi, clo, np, 0, hi_bits, st));           // ... then stably by the high word
        chi.drop_alt(); clo.drop_alt();
        DevBuf<unsigned char> head; MLG_TRY(head.alloc(np));
        k_flag_heads2<<<nblk(np), TPB, 0, st>>>(chi.cur(), clo.cur(), np, head.p);
        // how many sketch slots hold each distinct K-mer (what `kmc -ci0` of the sketches' dump counts)
        DevBuf<unsigned char> runlen; MLG_TRY(runlen.alloc(np));
        k_run_lengths<<<nblk(np), TPB, 0, st>>>(head.p, np, runlen.p);
        // upper bound of nd is np; the exact size is known after the first select, so select the smallest array first
        DevBuf<unsigned char> multu_big; MLG_TRY(multu_big.alloc(np));
        MLG_TRY(select_flagged(runlen.p, head.p, multu_big.p, d_cnt.p, np, st));
        unsigned long long nd64 = 0;
        CUDA_TRY(cudaMemcpy(&nd64, d_cnt.p, 8, cudaMemcpyDeviceToHost));
        nd = (uint32_t)nd64;
        runlen.release();
        DevBuf<unsigned long long> dhi, dlo;
        MLG_TRY(dhi.alloc(nd)); MLG_TRY(select_flagged(chi.cur(), head.p, dhi.p, d_cnt.p, np, st)); chi.drop();
        MLG_TRY(dlo.alloc(nd)); MLG_TRY(select_flagged(clo.cur(), head.p, dlo.p, d_cnt.p, np, st)); clo.drop();
        head.release();
        // order by hash
        choose_buckets(v, nd);
        PingPong<unsigned long long> h; PingPong<uint32_t> perm;
        MLG_TRY(h.buf[0].alloc(nd)); MLG_TRY(perm.buf[0].alloc(nd));
        k_hash_keys2<<<nblk(nd), TPB, 0, st>>>(dhi.p, dlo.p, nd, K, v.layout, v.bbits, h.cur());
        k_iota<<<nblk(nd), TPB, 0, st>>>(perm.cur(), nd);
        MLG_TRY(h.alloc_alt(nd)); MLG_TRY(perm.alloc_alt(nd));
        MLG_TRY(radix_pairs(h, perm, nd, 0, 64, st));
        h.drop_alt(); perm.drop_alt();
        MLG_TRY(db->D_key.alloc((size_t)nd + 1));
        CUDA_TRY(cudaMemsetAsync(db->D_key.p + nd, 0, sizeof(key128), st));
        k_gather_key2<<<nblk(nd), TPB, 0, st>>>(dhi.p, dlo.p, perm.cur(), nd, db->D_key.p);
        MLG_TRY(db->D_mult.alloc(nd));
        k_gather_u8<<<nblk(nd), TPB, 0, st>>>(multu_big.p, perm.cur(), nd, db->D_mult.p);
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaGetLastError());
        // hsorted = the sorted hashes (bucket histogram and level-1 fill below)
        hsorted.p = h.buf[h.sel].p; hsorted.n = h.buf[h.sel].n; h.buf[h.sel].p = nullptr; h.buf[h.sel].n = 0;
    } else {
        MLG_TRY(db->D_key.alloc(1)); MLG_TRY(hsorted.alloc(1));
    }
    v.nd = nd; v.D_key = db->D_key.p;
    {
        if (!nd) choose_buckets(v, nd);
        const uint32_t slots_per_bucket = v.slots, bbits = v.bbits;
        const unsigned long long nb = v.nbuckets;
        MLG_TRY(db->bstart.alloc(nb + 1));
        CUDA_TRY(cudaMemsetAsync(db->bstart.p, 0, (nb + 1) * 4, st));
        if (nd) k_hbucket_hist<<<nblk(nd), TPB, 0, st>>>(hsorted.p, nd, bbits, db->bstart.p);
        MLG_TRY(exclusive_scan_u32(db->bstart.p, nb, st));
        // layout 2 has no fingerprint table: its level 1 is the minimizer bitmap
        const unsigned long long t1_words = v.layout == 2 ? 8ull : nb * slots_per_bucket + 8;
        MLG_TRY(db->T1.alloc(t1_words));
        CUDA_TRY(cudaMemsetAsync(db->T1.p, 0, t1_words * 4, st));
        if (nd && v.layout != 2) k_fill_t1<<<nblk(nd), TPB, 0, st>>>(hsorted.p, nd, bbits, db->bstart.p, slots_per_bucket, v.layout, db->T1.p);
        v.bstart = db->bstart.p; v.T1 = db->T1.p;
        // One-bit-per-key prefilter sized to stay L2-resident: MLG_FILTER_MB MiB at most (default 64), 16 bits per
        // key at most; below 1.5 bits per key it would pass most probes and is left out.
        double max_mb = 64.0;
        if (const char* s = getenv("MLG_FILTER_MB")) max_mb = atof(s);
        unsigned long long nfw = 0;                       // 32-bit words
        if (nd && max_mb > 0 && v.layout == 0) {
            unsigned long long want = ((unsigned long long)nd * 16ull + 31ull) / 32ull;
            unsigned long long cap = (unsigned long long)(max_mb * 1048576.0 / 4.0);
            nfw = want < cap ? want : cap;
            if (nfw > 0xFFFFFFF0ull) nfw = 0xFFFFFFF0ull;
            if ((double)nfw * 32.0 < 1.5 * (double)nd) nfw = 0;
        }
        if (v.layout == 2) {
            // level-1 bit array: at least 32 bits per K-mer, two bits set per K-mer (density <= 1/16, false-positive rate
            // of a run ~ density^2 <= 0.4 %; every false positive costs an exact compare of ~11 windows), 2^20 .. 2^36 bits
            uint32_t fbits = 20;
            while (fbits < 36 && (1ull << fbits) < 32ull * nd) ++fbits;
            if (const char* s = getenv("MLG_MZ_FBITS")) { int x = atoi(s); if (x >= 10 && x <= 36) fbits = (uint32_t)x; }
            v.fbits = fbits;
            nfw = 1ull << (fbits - 5);
        }
        v.nfw = (uint32_t)nfw; v.F = nullptr;
        v.fk = ((double)nfw * 32.0 >= 3.0 * (double)nd) ? 2u : 1u;     // two probe bits pay off above ~3 bits per key
        if (const char* s = getenv("MLG_FILTER_K")) { int x = atoi(s); if (x == 1 || x == 2) v.fk = (uint32_t)x; }
        if (v.layout == 2) {
            MLG_TRY(db->F.alloc(nfw));
            CUDA_TRY(cudaMemsetAsync(db->F.p, 0, nfw * 4, st));
            v.F = db->F.p;
            v.n_alias = 0; v.alias_z = nullptr; v.alias_i = nullptr;
            MLG_TRY(db->alias_bloom.alloc(2048));
            CUDA_TRY(cudaMemsetAsync(db->alias_bloom.p, 0, 2048 * 4, st));
            v.alias_bloom = db->alias_bloom.p;
            if (nd) {
                CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, 8, st));
                k_fill_mzbits<<<nblk(nd), TPB, 0, st>>>(db->D_key.p, nd, K, v.fbits, db->F.p, 0, nullptr, nullptr, nullptr, d_cnt.p);
                unsigned long long na = 0;
                CUDA_TRY(cudaMemcpyAsync(&na, d_cnt.p, 8, cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                if (na) {
                    DevBuf<unsigned long long> az; DevBuf<uint32_t> ai;
                    MLG_TRY(az.alloc(na)); MLG_TRY(ai.alloc(na));
                    MLG_TRY(db->alias_z.alloc(na)); MLG_TRY(db->alias_i.alloc(na));
                    CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, 8, st));
                    k_fill_mzbits<<<nblk(nd), TPB, 0, st>>>(db->D_key.p, nd, K, v.fbits, db->F.p, 1, az.p, ai.p, db->alias_bloom.p, d_cnt.p);
                    MLG_TRY(sort_pairs_u64(az.p, db->alias_z.p, ai.p, db->alias_i.p, (uint32_t)na, 0, 64, st));
                    v.n_alias = (uint32_t)na; v.alias_z = db->alias_z.p; v.alias_i = db->alias_i.p;
                }
            }
        } else if (nfw) {
            MLG_TRY(db->F.alloc(nfw));
            CUDA_TRY(cudaMemsetAsync(db->F.p, 0, nfw * 4, st));
            k_fill_filter<<<nblk(nd), TPB, 0, st>>>(hsorted.p, nd, (uint32_t)nfw, v.fk, db->F.p);
            v.F = db->F.p;
            // pin the prefilter in L2: grow the persisting carve-out (default 24 MB of the 79 MB this part allows) and
            // put a persisting access-policy window over F on the compute stream.  MLG_L2_PERSIST=0 leaves the
            // device limits alone (the kernel's evict_last / evict_first load policies still apply).
            const char* pe = getenv("MLG_L2_PERSIST");
            if (!pe || atoi(pe) > 0) {
                cudaDeviceProp prop;
                if (cudaGetDeviceProperties(&prop, ctx->device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
                    size_t fbytes = (size_t)nfw * 4;
                    size_t carve = fbytes < (size_t)prop.persistingL2CacheMaxSize ? fbytes : (size_t)prop.persistingL2CacheMaxSize;
                    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
                    cudaStreamAttrValue attr;
                    memset(&attr, 0, sizeof(attr));
                    attr.accessPolicyWindow.base_ptr = (void*)db->F.p;
                    attr.accessPolicyWindow.num_bytes = fbytes < (size_t)prop.accessPolicyMaxWindowSize ? fbytes : (size_t)prop.accessPolicyMaxWindowSize;
                    attr.accessPolicyWindow.hitRatio = (float)((double)carve / (double)fbytes);
                    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
                    attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
                    if (cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
                }
            }
        }
    }
    hsorted.release();
    mlg_pool_trim(ctx->device);
    stage("D, level 1");

    // 2. P: the non-empty slots in stored orientation sorted by key, slot id as payload
    if (np) {
        PingPong<unsigned long long> klo; PingPong<uint32_t> p1;
        klo.adopt(b->lo);
        MLG_TRY(p1.buf[0].alloc(np));
        k_iota<<<nblk(np), TPB, 0, st>>>(p1.cur(), np);
        MLG_TRY(klo.alloc_alt(np)); MLG_TRY(p1.alloc_alt(np));
        MLG_TRY(radix_pairs(klo, p1, np, 0, lo_bits, st));
        klo.drop_alt(); p1.drop_alt();                        // klo.cur() = low words sorted, p1.cur() = position -> builder index
        if (hi_bits) {
            PingPong<unsigned long long> khi; PingPong<uint32_t> p2;
            MLG_TRY(khi.buf[0].alloc(np));
            k_gather_u64<<<nblk(np), TPB, 0, st>>>(b->hi.p, p1.cur(), np, khi.cur());
            CUDA_TRY(cudaStreamSynchronize(st));
            b->hi.release();
            MLG_TRY(p2.buf[0].alloc(np));
            k_iota<<<nblk(np), TPB, 0, st>>>(p2.cur(), np);
            MLG_TRY(khi.alloc_alt(np)); MLG_TRY(p2.alloc_alt(np));
            MLG_TRY(radix_pairs(khi, p2, np, 0, hi_bits, st));
            khi.drop_alt(); p2.drop_alt();                    // p2.cur() = position -> position in the low-word order
            MLG_TRY(db->P_key.alloc(np));
            k_zip_keys<<<nblk(np), TPB, 0, st>>>(khi.cur(), klo.cur(), p2.cur(), np, db->P_key.p);
            CUDA_TRY(cudaStreamSynchronize(st));
            khi.drop(); klo.drop();
            DevBuf<uint32_t> fin; MLG_TRY(fin.alloc(np));
            k_gather_u32<<<nblk(np), TPB, 0, st>>>(p1.cur(), p2.cur(), np, fin.p);      // builder index = p1[p2[i]]
            CUDA_TRY(cudaStreamSynchronize(st));
            p1.drop(); p2.drop();
            MLG_TRY(db->P_slot.alloc(np));
            k_gather_u32<<<nblk(np), TPB, 0, st>>>(b->slot.p, fin.p, np, db->P_slot.p);
            CUDA_TRY(cudaStreamSynchronize(st));
        } else {
            b->hi.release();
            DevBuf<unsigned long long> zero; MLG_TRY(zero.alloc(np));
            CUDA_TRY(cudaMemsetAsync(zero.p, 0, (size_t)np * 8, st));
            MLG_TRY(db->P_key.alloc(np));
            k_zip_keys<<<nblk(np), TPB, 0, st>>>(zero.p, klo.cur(), nullptr, np, db->P_key.p);
            MLG_TRY(db->P_slot.alloc(np));
            k_gather_u32<<<nblk(np), TPB, 0, st>>>(b->slot.p, p1.cur(), np, db->P_slot.p);
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        CUDA_TRY(cudaGetLastError());
    } else {
        MLG_TRY(db->P_key.alloc(1)); MLG_TRY(db->P_slot.alloc(1));
    }
    b->hi.release(); b->lo.release(); b->slot.release();
    v.P_key = db->P_key.p; v.P_slot = db->P_slot.p;
    mlg_pool_trim(ctx->device);
    stage("P");

    // 3. bucket index on the top pbits of the key
    {
        uint32_t pbits = 8;
        while (pbits < 28 && (1ull << pbits) < np) ++pbits;
        if (pbits > 2 * K) pbits = 2 * K;
        v.pbits = pbits;
        size_t m = (size_t)1 << pbits;
        MLG_TRY(db->pidx.alloc(m + 1));
        CUDA_TRY(cudaMemsetAsync(db->pidx.p, 0, (m + 1) * 4, st));
        if (np) k_pbucket_hist<<<nblk(np), TPB, 0, st>>>(db->P_key.p, np, K, pbits, db->pidx.p);
        MLG_TRY(exclusive_scan_u32(db->pidx.p, m, st));
        v.pidx = db->pidx.p;
    }

    // 4. (genome, k-prefix) classes and denominators
    MLG_TRY(db->rep.alloc((size_t)nk * total));
    CUDA_TRY(cudaMemsetAsync(db->rep.p, 0xFF, (size_t)nk * total * 4, st));
    MLG_TRY(db->den_real.alloc((size_t)G * nk));
    CUDA_TRY(cudaMemsetAsync(db->den_real.p, 0, (size_t)G * nk * 8, st));
    if (np) {
        PingPong<uint32_t> gkey, q2p;
        MLG_TRY(gkey.buf[0].alloc(np)); MLG_TRY(q2p.buf[0].alloc(np));
        k_slot_to_genome<<<nblk(np), TPB, 0, st>>>(db->P_slot.p, np, n, gkey.cur());
        k_iota<<<nblk(np), TPB, 0, st>>>(q2p.cur(), np);
        int gbits = 1; while (gbits < 32 && (1ull << gbits) < G) ++gbits;
        MLG_TRY(gkey.alloc_alt(np)); MLG_TRY(q2p.alloc_alt(np));
        MLG_TRY(radix_pairs(gkey, q2p, np, 0, gbits, st));
        gkey.drop(); q2p.drop_alt();
        for (uint32_t ki = 0; ki < nk; ++ki)
            k_rep_classes<<<nblk(np), TPB, 0, st>>>(db->P_key.p, db->P_slot.p, q2p.cur(), np, n, K, ks[ki], ki, nk,
                                                    db->rep.p + (size_t)ki * total, db->den_real.p);
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaGetLastError());
    }
    v.rep = db->rep.p;
    mlg_pool_trim(ctx->device);
    stage("classes");

    // 6. hit records: what a present k-mer of D contributes to the per-genome table is a static function of the
    //    database, so it is expanded once here (same code as the on-the-fly kernel) and replayed per query.  Two passes:
    //    tally (sizes; the common one-slot records are complete after it) -> offsets -> fill.  Afterwards P, its bucket
    //    index and the class representatives -- 60 % of the database's footprint -- have no reader left and are released.
    //    MLG_PRECOMPUTE_HITS=0 skips all this (every query expands on the fly); MLG_HIT_CAP_WORDS=n drops the records
    //    beyond word n (their k-mers are expanded on the fly: the mixed path, for tests); MLG_KEEP_P=1 keeps P regardless.
    {
        const char* pe = getenv("MLG_PRECOMPUTE_HITS");
        if (nd && (!pe || atoi(pe) != 0)) {
            unsigned long long drop_from = ~0ull;
            if (const char* s = getenv("MLG_HIT_CAP_WORDS")) { unsigned long long x = strtoull(s, nullptr, 10); if (x >= 16) drop_from = x; }
            const unsigned long long groups = ((unsigned long long)nd + (1ull << MLG_HGROUP_SHIFT) - 1) >> MLG_HGROUP_SHIFT;
            DevBuf<uint32_t> summary;
            MLG_TRY(summary.alloc(2ull * nd)); MLG_TRY(db->hoff.alloc(nd)); MLG_TRY(db->hbase.alloc(groups + 1));
            MLG_TRY(launch_tally_hits(v, summary.p, st));
            CUDA_TRY(cudaMemsetAsync(db->hbase.p, 0, (groups + 1) * 8, st));
            MLG_TRY(launch_hit_group_sums(summary.p, nd, db->hbase.p, st));
            {
                void* tmp = nullptr; size_t tb = 0;
                CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb, db->hbase.p, db->hbase.p, (int)(groups + 1), st));
                CUDA_TRY(cudaMalloc(&tmp, tb ? tb : 1));
                cudaError_t e = cub::DeviceScan::ExclusiveSum(tmp, tb, db->hbase.p, db->hbase.p, (int)(groups + 1), st);
                cudaStreamSynchronize(st); cudaFree(tmp);
                if (e != cudaSuccess) { mlg_set_error("DeviceScan failed: %s", cudaGetErrorString(e)); return MLG_ERR_CUDA; }
            }
            MLG_TRY(launch_hit_offsets(summary.p, nd, db->hoff.p, st));
            unsigned long long total_words = 0;
            CUDA_TRY(cudaMemcpyAsync(&total_words, db->hbase.p + groups, 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            CUDA_TRY(cudaGetLastError());
            const unsigned long long keep_words = total_words < drop_from ? total_words : drop_from;
            // The records have to fit BESIDE P and the class representatives, which the fill still reads (afterwards those
            // go, and a query's own tables take their place).  When they do not (2e9 slots: P + rep are 73 GB), the
            // database keeps P and every query expands its present k-mers on the fly -- |I| x 240 sectors, well under a
            // millisecond more per query -- instead of failing.  MLG_HIT_BUDGET_BYTES overrides the free-memory figure (tests).
            mlg_pool_trim(ctx->device);
            size_t free_b = 0, total_b = 0;
            CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
            if (const char* s = getenv("MLG_HIT_BUDGET_BYTES")) free_b = (size_t)strtoull(s, nullptr, 10);
            const unsigned long long need = (keep_words + 2 + MLG_MAX_KS) * 4ull + (256ull << 20);
            if (verbose) fprintf(stderr, "[mlg build] hit records need %.1f GB, free %.1f GB\n", (double)need / 1e9, (double)free_b / 1e9);
            if (need > free_b) {
                summary.release(); db->hoff.release(); db->hbase.release();
                db->hit_words = 0;
                db->hits_skipped_bytes = need;
            } else {
                MLG_TRY(db->hits.alloc(keep_words + 2 + MLG_MAX_KS));
                MLG_TRY(launch_fill_hits(v, summary.p, db->hoff.p, db->hbase.p, db->hits.p, drop_from, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                CUDA_TRY(cudaGetLastError());
                db->hit_words = keep_words;
                const char* kp = getenv("MLG_KEEP_P");
                if (drop_from == ~0ull && !(kp && atoi(kp) != 0)) {
                    db->P_key.release(); db->P_slot.release(); db->pidx.release(); db->rep.release();
                    v.P_key = nullptr; v.P_slot = nullptr; v.pidx = nullptr; v.rep = nullptr;
                    db->p_dropped = true;
                }
            }
        }
    }
    stage("hit records");
    CUDA_TRY(cudaEventRecord(e1, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1); db->build_ms = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    guard.d = nullptr;
    delete b;
    mlg_pool_trim(ctx->device);   // the build's multi-GB temporaries should not stay cached
    *out = db;
    return MLG_OK;
}

int mlg_db_build_device(mlg_ctx* ctx, const key128* d_keys, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks,
                        uint32_t nk, mlg_db** out) {
    if (!ctx || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    mlg_db_builder* b = nullptr;
    MLG_TRY(mlg_db_builder_create_impl(ctx, G, n, K, ks, nk, &b));
    // in chunks, so that the scratch of the compaction stays small beside the caller's keys
    const uint32_t step = std::max<uint32_t>(1u, (uint32_t)std::min<unsigned long long>(G, (256ull << 20) / n));
    for (uint32_t g0 = 0; g0 < G; g0 += step) {
        const uint32_t c = std::min<uint32_t>(step, G - g0);
        int rc = mlg_db_builder_add_impl(b, d_keys + (size_t)g0 * n, g0, c);
        if (rc != MLG_OK) { mlg_db_builder_destroy_impl(b); return rc; }
    }
    int rc = mlg_db_builder_finish_impl(b, out);
    if (rc != MLG_OK) mlg_db_builder_destroy_impl(b);
    return rc;
}
