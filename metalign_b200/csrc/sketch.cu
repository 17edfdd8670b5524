// Sketch builder: the bottom-n MinHash sketch of every genome, as CMash's
//   MakeStreamingDNADatabase.py <list of genome files> <out.h5> -n 1000 -k 60
// builds it for Metalign's training database (local_tests/retrain_and_test_metalign.sh:49; SURVEY.md A.2):
// every N-free K-long window of the genome, forward strand only (rev_comp=False), upper-cased, is hashed with
// MurmurHash3_x64_128 (seed 0, first 64-bit word: khmer's hash_no_rc_murmur3) modulo a prime; the sketch keeps the n
// smallest DISTINCT hash values in ascending order, each with the first k-mer that produced it and the number of times
// it occurred; unused slots keep (prime, 0, '').  The reference does this one k-mer at a time in Python
// (MinHash.CountEstimator.add: bisect + list insert); here it is
//   S0  k_valid_mask      one thread per byte: is it A/C/G/T (either case)?  warp ballot -> one bit per base
//   S1  k_hash_windows    one thread per window: 60 valid bits in a row? -> the K bytes as little-endian 64-bit words
//                         (9 aligned loads, L1-resident overlap with the neighbours) -> MurmurHash3 -> mod prime
//                         (Barrett) -> windows below the genome's threshold T_g are appended to a candidate list.
//                         T_g = prime * 4n / windows(g): the n-th smallest of L uniform values sits near prime * n / L,
//                         so ~4n candidates per genome survive out of millions of windows
//   S2  CUB radix sort of the candidates by (genome, hash)
//   S3  k_heads + scan + k_emit   distinct hashes, their rank inside the genome, occurrence count, first position
// A genome that ends up with fewer than n distinct candidates although T_g < prime (repeats) is redone with 8 T_g.
// Instruction-bound (two 64-bit multiplies per 8 bytes), not HBM-bound: every base is read once from DRAM.
#include <cub/cub.cuh>
#include <algorithm>
#include <stdlib.h>
#include <string.h>
#include "mlg_internal.h"

#ifndef MLG_API
#define MLG_API extern "C" __attribute__((visibility("default")))
#endif

namespace {

constexpr int TPB = 256;
constexpr uint32_t TILE = 4096;           // windows per CTA pass
constexpr unsigned HBITS = 44;            // hash values are < prime < 2^44
// device text of one pass, separators and 64 bytes of padding included, stays below this: positions are 32-bit
constexpr unsigned long long PASS_LIMIT = 0xFFFFFFF0ull;

__device__ __forceinline__ unsigned long long rotl64(unsigned long long x, int r) { return (x << r) | (x >> (64 - r)); }
__device__ __forceinline__ unsigned long long fmix64(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}
// first word of MurmurHash3_x64_128(key, len, seed 0); key as little-endian 64-bit words, zero beyond len (len <= 64)
__device__ __forceinline__ unsigned long long murmur3_x64_h1(const unsigned long long (&w)[8], uint32_t len) {
    const unsigned long long c1 = 0x87c37b91114253d5ull, c2 = 0x4cf5ad432745937full;
    unsigned long long h1 = 0, h2 = 0;
    const uint32_t nblocks = len >> 4;
#pragma unroll
    for (uint32_t i = 0; i < 4; ++i) {
        if (i < nblocks) {
            unsigned long long k1 = w[2 * i], k2 = w[2 * i + 1];
            k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
            h1 = rotl64(h1, 27); h1 += h2; h1 = h1 * 5 + 0x52dce729ull;
            k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
            h2 = rotl64(h2, 31); h2 += h1; h2 = h2 * 5 + 0x38495ab5ull;
        }
    }
    // tail: the bytes beyond len are zero, and mixing a zero word changes nothing, so no switch on len & 15 is needed
    unsigned long long k1 = 0, k2 = 0;
#pragma unroll
    for (uint32_t i = 0; i < 4; ++i)
        if (i == nblocks) { k1 = w[2 * i]; k2 = w[2 * i + 1]; }
    k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
    k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
    h1 ^= len; h2 ^= len;
    h1 += h2; h2 += h1;
    h1 = fmix64(h1); h2 = fmix64(h2);
    h1 += h2;
    return h1;
}

__device__ __forceinline__ bool is_acgt(unsigned char c) {
    c &= 0xDFu;                            // fold case: only 'a'..'z' / 'A'..'Z' land on a letter
    return c == 'A' || c == 'C' || c == 'G' || c == 'T';
}
// S0: bit i of vmask (bit i % 32 of word i / 32) = text[i] is A/C/G/T in either case
__global__ void k_valid_mask(const unsigned char* text, unsigned long long nbytes, uint32_t* vmask) {
    const unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    const bool v = i < nbytes && is_acgt(text[i]);
    const unsigned b = __ballot_sync(0xFFFFFFFFu, v);
    if ((threadIdx.x & 31u) == 0 && i < nbytes + 32) vmask[i >> 5] = b;
}

struct SketchArgs {
    const unsigned long long* text8;       // the text as aligned 64-bit words (padded)
    const uint32_t* vmask;
    const uint32_t* tile_g;                // genome of each tile
    const unsigned long long* tile_pos;    // first window (byte position) of each tile
    const unsigned long long* g_end;       // per genome: one past its last window start
    const unsigned long long* g_T;         // per genome: candidates are the windows with hash < T
    uint32_t K;
    unsigned long long prime, barrett;     // barrett = floor((2^64 - 1) / prime)
    unsigned long long* cand_key;          // genome << HBITS | hash
    uint32_t* cand_pos;
    unsigned long long cap;
    unsigned long long* counters;          // [0] candidates appended, [1] valid windows
};

// S1
__global__ void __launch_bounds__(TPB) k_hash_windows(SketchArgs a) {
    const uint32_t g = a.tile_g[blockIdx.x];
    const unsigned long long p0 = a.tile_pos[blockIdx.x], pend = a.g_end[g], T = a.g_T[g];
    const uint32_t K = a.K;
    unsigned long long nvalid = 0;
    for (uint32_t t = threadIdx.x; t < TILE; t += TPB) {
        const unsigned long long p = p0 + t;
        if (p >= pend) break;
        // K valid bases in a row from p?
        const unsigned long long wi = p >> 5;
        const unsigned sh = (unsigned)(p & 31ull);
        const uint32_t m0 = a.vmask[wi], m1 = a.vmask[wi + 1], m2 = a.vmask[wi + 2];
        const unsigned long long lo = ((unsigned long long)m1 << 32) | m0;
        unsigned long long bits = sh ? ((lo >> sh) | ((unsigned long long)m2 << (64 - sh))) : lo;   // validity of bases p .. p+63
        const unsigned long long need = K >= 64 ? ~0ull : ((1ull << K) - 1ull);
        if ((bits & need) != need) continue;
        ++nvalid;
        // the K bytes as little-endian words, case folded, zero beyond K
        const unsigned long long q = p >> 3;
        const unsigned bs = 8u * (unsigned)(p & 7ull);
        unsigned long long w[8];
        unsigned long long prev = a.text8[q];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const unsigned long long next = a.text8[q + k + 1];
            const unsigned long long v = bs ? ((prev >> bs) | (next << (64 - bs))) : prev;
            prev = next;
            const int nb = (int)K - 8 * k;                 // bytes of this word inside the k-mer
            const unsigned long long keep = nb >= 8 ? ~0ull : (nb <= 0 ? 0ull : ((1ull << (8 * nb)) - 1ull));
            w[k] = v & 0xDFDFDFDFDFDFDFDFull & keep;
        }
        unsigned long long h = murmur3_x64_h1(w, K);
        // h mod prime
        const unsigned long long qq = __umul64hi(h, a.barrett);
        h -= qq * a.prime;
        while (h >= a.prime) h -= a.prime;
        if (h < T) {
            const unsigned long long i = atomicAdd(a.counters, 1ull);
            if (i < a.cap) { a.cand_key[i] = ((unsigned long long)g << HBITS) | h; a.cand_pos[i] = (uint32_t)p; }
        }
    }
    for (int o = 16; o > 0; o >>= 1) nvalid += __shfl_down_sync(0xFFFFFFFFu, nvalid, o);
    if ((threadIdx.x & 31u) == 0 && nvalid) atomicAdd(a.counters + 1, nvalid);
}

// S3a: heads of runs of equal (genome, hash), and the first candidate of every genome
__global__ void k_heads(const unsigned long long* key, uint32_t nc, uint32_t* head, uint32_t* g_first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nc) return;
    const bool h = i == 0 || key[i] != key[i - 1];
    head[i] = h ? 1u : 0u;
    if (i == 0 || (key[i] >> HBITS) != (key[i - 1] >> HBITS)) g_first[key[i] >> HBITS] = i;
}
// S3b: every head = one distinct hash; its rank inside the genome decides whether it is in the sketch
__global__ void k_emit(const unsigned long long* key, const uint32_t* pos, const uint32_t* head, const uint32_t* rank_excl, uint32_t nc,
                       const uint32_t* g_first, uint32_t n, uint32_t K, const unsigned char* text, unsigned long long* mins,
                       uint32_t* counts, unsigned char* kmers, uint32_t* g_distinct, uint32_t* g_seen_all, uint32_t* g_last) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nc || !head[i]) return;
    const unsigned long long k = key[i];
    const uint32_t g = (uint32_t)(k >> HBITS);
    const uint32_t rank = rank_excl[i] - rank_excl[g_first[g]];
    atomicMax(&g_distinct[g], rank + 1u);
    if (rank >= n) return;
    uint32_t cnt = 0, first = 0xFFFFFFFFu;
    for (uint32_t j = i; j < nc && key[j] == k; ++j) { ++cnt; first = min(first, pos[j]); }
    const size_t slot = (size_t)g * n + rank;
    mins[slot] = k & ((1ull << HBITS) - 1ull);
    counts[slot] = cnt;
    // for the count of the sketch's LAST element (k_fix_last): where the n-1 smaller ones are all in, and where its run is
    if (rank + 1u < n) atomicMax(&g_seen_all[g], first); else g_last[g] = i;
    for (uint32_t b = 0; b < K; ++b) kmers[slot * K + b] = text[first + b] & 0xDFu;
}
// CountEstimator.add() returns early on `h >= mins[-1]`: while a hash is the LARGEST of a full sketch its repeats are not
// counted.  Only the final last element can ever be in that position -- from the moment the n-1 smaller hashes have
// all appeared -- so its count is the number of its occurrences before that moment (at least the one that inserted it).
__global__ void k_fix_last(const unsigned long long* key, const uint32_t* pos, uint32_t nc, uint32_t ng, uint32_t n,
                           const uint32_t* g_distinct, const uint32_t* g_seen_all, const uint32_t* g_last, uint32_t* counts) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ng || g_distinct[g] < n) return;
    const uint32_t i = g_last[g], full_at = n > 1 ? g_seen_all[g] : 0u;
    const unsigned long long k = key[i];
    uint32_t cnt = 0;
    for (uint32_t j = i; j < nc && key[j] == k; ++j) cnt += pos[j] < full_at ? 1u : 0u;
    counts[(size_t)g * n + (n - 1)] = cnt ? cnt : 1u;
}
__global__ void k_fill_u64(unsigned long long* a, size_t n, unsigned long long v) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}

inline unsigned nblk(unsigned long long n) { return (unsigned)((n + TPB - 1) / TPB); }

}  // namespace

// one pass over the genomes idx[0..ng): their text goes to the device with one 'N' between genomes; results land in the
// host arrays at the genomes' own slots; genomes that need a larger threshold are returned in `redo`
static int sketch_pass(mlg_ctx* ctx, const char* text, const uint64_t* off, const std::vector<uint32_t>& idx, std::vector<double>& tmul,
                       uint32_t n, uint32_t K, unsigned long long prime, uint64_t* mins, uint32_t* counts, char* kmers,
                       mlg_sketch_stats* st, std::vector<uint32_t>& redo) {
    cudaStream_t s = ctx->s_comp;
    const uint32_t ng = (uint32_t)idx.size();
    // device text layout: genome i at d_off[i], followed by one 'N'; 64 bytes of 'N' padding at the end
    std::vector<unsigned long long> d_off(ng + 1), g_end(ng), g_T(ng), tile_pos;
    std::vector<uint32_t> tile_g;
    unsigned long long total = 0, nwin_total = 0;
    for (uint32_t i = 0; i < ng; ++i) {
        const unsigned long long len = off[idx[i] + 1] - off[idx[i]];
        d_off[i] = total;
        const unsigned long long nwin = len >= K ? len - K + 1 : 0;
        g_end[i] = total + nwin;
        double frac = nwin ? tmul[idx[i]] * 4.0 * (double)n / (double)nwin : 1.0;
        g_T[i] = frac >= 1.0 ? prime : (unsigned long long)((double)prime * frac) + 1ull;
        for (unsigned long long p = 0; p < nwin; p += TILE) { tile_g.push_back(i); tile_pos.push_back(total + p); }
        nwin_total += nwin;
        total += len + 1;
    }
    d_off[ng] = total;
    if (total + 64 >= PASS_LIMIT) { mlg_set_error("sketch batch of %llu bytes is too large (< 4 GB per pass)", total); return MLG_ERR_ARG; }
    const unsigned long long padded = (total + 128 + 15) & ~15ull;
    std::vector<unsigned char> h_text(padded, (unsigned char)'N');
    for (uint32_t i = 0; i < ng; ++i) memcpy(h_text.data() + d_off[i], text + off[idx[i]], off[idx[i] + 1] - off[idx[i]]);

    DevBuf<unsigned char> d_text, d_kmers; DevBuf<uint32_t> d_vmask, d_tile_g, d_cpos, d_cpos_s, d_head, d_rank, d_gfirst, d_gdist, d_counts, d_gseen, d_glast;
    DevBuf<unsigned long long> d_tile_pos, d_gend, d_gT, d_ckey, d_ckey_s, d_cnt, d_mins;
    MLG_TRY(d_text.alloc(padded)); MLG_TRY(d_vmask.alloc(padded / 32 + 4));
    MLG_TRY(d_tile_g.alloc(tile_g.size())); MLG_TRY(d_tile_pos.alloc(tile_pos.size()));
    MLG_TRY(d_gend.alloc(ng)); MLG_TRY(d_gT.alloc(ng)); MLG_TRY(d_cnt.alloc(2));
    MLG_TRY(d_gfirst.alloc(ng)); MLG_TRY(d_gdist.alloc(ng)); MLG_TRY(d_gseen.alloc(ng)); MLG_TRY(d_glast.alloc(ng));
    const size_t slots = (size_t)ng * n;
    MLG_TRY(d_mins.alloc(slots)); MLG_TRY(d_counts.alloc(slots)); MLG_TRY(d_kmers.alloc(slots * K));
    CUDA_TRY(cudaMemcpyAsync(d_text.p, h_text.data(), padded, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemsetAsync(d_vmask.p, 0, (padded / 32 + 4) * 4, s));
    if (!tile_g.empty()) {
        CUDA_TRY(cudaMemcpyAsync(d_tile_g.p, tile_g.data(), tile_g.size() * 4, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(d_tile_pos.p, tile_pos.data(), tile_pos.size() * 8, cudaMemcpyHostToDevice, s));
    }
    CUDA_TRY(cudaMemcpyAsync(d_gend.p, g_end.data(), ng * 8ull, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(d_gT.p, g_T.data(), ng * 8ull, cudaMemcpyHostToDevice, s));
    // kernel time only: event pairs around the launches, allocations and host round trips outside them
    cudaEvent_t e0, e1; CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    float ms_sum = 0;
    auto lap = [&]() { float ms = 0; if (cudaEventSynchronize(e1) == cudaSuccess && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) ms_sum += ms; };
    CUDA_TRY(cudaEventRecord(e0, s));
    k_valid_mask<<<nblk(padded), TPB, 0, s>>>(d_text.p, padded, d_vmask.p);
    k_fill_u64<<<nblk(slots), TPB, 0, s>>>(d_mins.p, slots, prime);
    CUDA_TRY(cudaMemsetAsync(d_counts.p, 0, slots * 4, s));
    CUDA_TRY(cudaMemsetAsync(d_kmers.p, 0, slots * K, s));
    CUDA_TRY(cudaMemsetAsync(d_gdist.p, 0, ng * 4ull, s));
    CUDA_TRY(cudaMemsetAsync(d_gfirst.p, 0, ng * 4ull, s));
    CUDA_TRY(cudaMemsetAsync(d_gseen.p, 0, ng * 4ull, s));
    CUDA_TRY(cudaMemsetAsync(d_glast.p, 0, ng * 4ull, s));
    CUDA_TRY(cudaEventRecord(e1, s));
    lap();

    // candidates: ~4n per genome are expected (more when k-mers repeat); grow and redo the pass if the list overflows
    unsigned long long cap = std::min<unsigned long long>(nwin_total, (unsigned long long)ng * 8ull * n + 4096ull);
    unsigned long long cnt[2] = {0, 0};
    for (int attempt = 0;; ++attempt) {
        if (cap == 0) cap = 1;
        MLG_TRY(d_ckey.alloc(cap)); MLG_TRY(d_cpos.alloc(cap));
        CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, 16, s));
        CUDA_TRY(cudaEventRecord(e0, s));
        if (!tile_g.empty()) {
            SketchArgs a{reinterpret_cast<const unsigned long long*>(d_text.p), d_vmask.p, d_tile_g.p, d_tile_pos.p, d_gend.p, d_gT.p, K, prime,
                         ~0ull / prime, d_ckey.p, d_cpos.p, cap, d_cnt.p};
            k_hash_windows<<<(unsigned)tile_g.size(), TPB, 0, s>>>(a);
            CUDA_TRY(cudaGetLastError());
        }
        CUDA_TRY(cudaEventRecord(e1, s));
        CUDA_TRY(cudaMemcpyAsync(cnt, d_cnt.p, 16, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        lap();
        if (cnt[0] <= cap) break;
        if (attempt >= 3) { mlg_set_error("sketch: candidate list overflow (%llu > %llu)", cnt[0], cap); return MLG_ERR_STATE; }
        cap = cnt[0] + 1024;
    }
    const uint32_t nc = (uint32_t)cnt[0];
    if (st) { st->n_windows += cnt[1]; st->n_candidates += nc; st->passes += 1; }
    std::vector<uint32_t> h_gdist(ng, 0);
    if (nc) {
        MLG_TRY(d_ckey_s.alloc(nc)); MLG_TRY(d_cpos_s.alloc(nc)); MLG_TRY(d_head.alloc(nc)); MLG_TRY(d_rank.alloc(nc));
        int gbits = 1; while (gbits < 20 && (1u << gbits) < ng) ++gbits;
        size_t tb_sort = 0, tb_scan = 0;
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tb_sort, d_ckey.p, d_ckey_s.p, d_cpos.p, d_cpos_s.p, (int)nc, 0, (int)HBITS + gbits, s));
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tb_scan, d_head.p, d_rank.p, (int)nc, s));
        DevBuf<unsigned char> d_tmp; MLG_TRY(d_tmp.alloc(std::max(tb_sort, tb_scan) + 16));
        CUDA_TRY(cudaEventRecord(e0, s));
        CUDA_TRY(cub::DeviceRadixSort::SortPairs(d_tmp.p, tb_sort, d_ckey.p, d_ckey_s.p, d_cpos.p, d_cpos_s.p, (int)nc, 0, (int)HBITS + gbits, s));
        k_heads<<<nblk(nc), TPB, 0, s>>>(d_ckey_s.p, nc, d_head.p, d_gfirst.p);
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb_scan, d_head.p, d_rank.p, (int)nc, s));
        k_emit<<<nblk(nc), TPB, 0, s>>>(d_ckey_s.p, d_cpos_s.p, d_head.p, d_rank.p, nc, d_gfirst.p, n, K, d_text.p, d_mins.p, d_counts.p,
                                         d_kmers.p, d_gdist.p, d_gseen.p, d_glast.p);
        k_fix_last<<<nblk(ng), TPB, 0, s>>>(d_ckey_s.p, d_cpos_s.p, nc, ng, n, d_gdist.p, d_gseen.p, d_glast.p, d_counts.p);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(e1, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        lap();
        CUDA_TRY(cudaMemcpyAsync(h_gdist.data(), d_gdist.p, ng * 4ull, cudaMemcpyDeviceToHost, s));
    }
    std::vector<unsigned long long> h_mins(slots); std::vector<uint32_t> h_counts(slots); std::vector<char> h_kmers(slots * K);
    CUDA_TRY(cudaMemcpyAsync(h_mins.data(), d_mins.p, slots * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h_counts.data(), d_counts.p, slots * 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(h_kmers.data(), d_kmers.p, slots * K, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (st) st->ms_kernels += ms_sum;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    for (uint32_t i = 0; i < ng; ++i) {
        const uint32_t g = idx[i];
        if (h_gdist[i] < n && g_T[i] < prime) { tmul[g] *= 8.0; redo.push_back(g); continue; }   // too few distinct candidates: widen
        memcpy(mins + (size_t)g * n, h_mins.data() + (size_t)i * n, (size_t)n * 8);
        memcpy(counts + (size_t)g * n, h_counts.data() + (size_t)i * n, (size_t)n * 4);
        memcpy(kmers + (size_t)g * n * K, h_kmers.data() + (size_t)i * n * K, (size_t)n * K);
    }
    return MLG_OK;
}

MLG_API int mlg_sketch_genomes(mlg_ctx* ctx, const char* text, const uint64_t* genome_off, uint32_t G, uint32_t n, uint32_t K,
                               uint64_t prime, uint64_t* mins, uint32_t* counts, char* kmers, mlg_sketch_stats* st) {
    if (!ctx || !text || !genome_off || !mins || !counts || !kmers) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (K < 1 || K > 64) { mlg_set_error("K=%u out of range 1..64", K); return MLG_ERR_ARG; }
    if (n < 1 || G < 1 || G >= (1u << 20)) { mlg_set_error("need n >= 1 and 1 <= G < 2^20 genomes per call"); return MLG_ERR_ARG; }
    if (prime == 0) prime = 9999999999971ull;
    if (prime < 2 || prime >= (1ull << HBITS)) { mlg_set_error("prime must be below 2^44"); return MLG_ERR_ARG; }
    // a genome is never split: each one has to fit in one pass (its separator and the padding included)
    const unsigned long long max_len = PASS_LIMIT - 66;
    for (uint32_t g = 0; g < G; ++g) {
        if (genome_off[g + 1] < genome_off[g]) { mlg_set_error("genome_off decreases at genome %u", g); return MLG_ERR_ARG; }
        if (genome_off[g + 1] - genome_off[g] > max_len) { mlg_set_error("genome %u is too large (< 4 GB per genome)", g); return MLG_ERR_ARG; }
    }
    // bytes of text per pass; MLG_SKETCH_PASS_BYTES (experiment and test knob, read on every call): any value >= 1
    unsigned long long pass_bytes = 1ull << 30;
    if (const char* e = getenv("MLG_SKETCH_PASS_BYTES")) {
        const unsigned long long v = strtoull(e, nullptr, 10);
        if (v >= 1) pass_bytes = std::min(v, max_len);
    }
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (st) memset(st, 0, sizeof(*st));
    std::vector<double> tmul(G, 1.0);
    std::vector<uint32_t> todo(G), redo;
    for (uint32_t g = 0; g < G; ++g) todo[g] = g;
    // passes of at most pass_bytes of text (a genome larger than that gets a pass of its own)
    while (!todo.empty()) {
        redo.clear();
        size_t i = 0;
        while (i < todo.size()) {
            std::vector<uint32_t> batch;
            unsigned long long bytes = 0;
            while (i < todo.size()) {
                const unsigned long long len = genome_off[todo[i] + 1] - genome_off[todo[i]];
                if (!batch.empty() && bytes + len > pass_bytes) break;
                batch.push_back(todo[i]); bytes += len + 1; ++i;
            }
            MLG_TRY(sketch_pass(ctx, text, genome_off, batch, tmul, n, K, prime, mins, counts, kmers, st, redo));
        }
        todo = redo;
    }
    mlg_pool_trim(ctx->device);
    return MLG_OK;
}
