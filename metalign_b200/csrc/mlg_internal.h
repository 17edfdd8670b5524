// Internal declarations shared by the translation units of libmetalign_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include "kmer.cuh"
#include "../../include/metalign_b200.h"

#define MLG_MAX_KS 8
#define MLG_MAX_RANKS 16        // ranks of one exchange (one NVSwitch domain)
#define MLG_TILE_WORDS 256u     // 64-base words per K1 tile == threads per CTA
// version of the device structures in built .mlgdb files and of the read archives ranks exchange: minimizer identity =
// min/max multiply-add + xor-shift; hit records v2
#define MLG_BUILD_TAG 0x20261017u

void mlg_set_error(const char* fmt, ...);

#define CUDA_TRY(expr)                                                                            \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            mlg_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return MLG_ERR_CUDA;                                                                  \
        }                                                                                         \
    } while (0)

#define MLG_TRY(expr)                \
    do {                             \
        int _r = (expr);             \
        if (_r != MLG_OK) return _r; \
    } while (0)

// Device memory comes from a small per-device caching pool (capi.cu): a query allocates and frees a dozen
// buffers, and cudaMalloc/cudaFree would otherwise cost more than the kernels on small batches.  Blocks are
// only returned to the pool after the stream work that used them has been joined.
void* mlg_pool_alloc(size_t bytes);
void mlg_pool_free(void* p);
void mlg_pool_trim(int device);

// owning device buffer
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() {}
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() { if (p) mlg_pool_free(p); p = nullptr; n = 0; }
    int alloc(size_t count) {
        release();
        if (count == 0) count = 1;
        p = (T*)mlg_pool_alloc(count * sizeof(T));
        if (!p) return MLG_ERR_NOMEM;
        n = count;
        return MLG_OK;
    }
    int ensure(size_t count) { return (count <= n && p) ? MLG_OK : alloc(count); }
};

struct mlg_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t s_comp = nullptr;   // kernels
    cudaStream_t s_copy = nullptr;   // host<->device copies
};

// device view of a database (plain pointers, passed to kernels by value)
struct DbView {
    uint32_t G, n, K, nk;
    uint32_t ks[MLG_MAX_KS];
    uint32_t np;                 // non-empty sketch entries
    uint32_t nd;                 // distinct canonical k-mers
    // P: stored-orientation entries sorted by key
    const key128* P_key;
    const uint32_t* P_slot;      // g*n + j
    uint32_t pbits;              // bucket index on the top pbits bits of the 2K-bit key
    const uint32_t* pidx;        // 2^pbits + 1
    const uint32_t* rep;         // nk * (G*n): representative slot of the (genome, k-prefix) class
    // D: distinct canonical keys sorted by hash; level-1 fingerprint buckets
    const key128* D_key;
    const uint32_t* bstart;      // nbuckets + 1
    const uint32_t* T1;          // nbuckets * slots
    unsigned long long nbuckets; // 2^bbits
    uint32_t bbits;
    uint32_t slots;              // 4 (16-byte buckets) or 8 (32-byte buckets)
    // L2-resident prefilter over D: nfw 32-bit words, one bit per key (nfw == 0: disabled)
    const uint32_t* F;
    uint32_t nfw;
    uint32_t fk;                 // bits per key in the prefilter (1 or 2)
    // 0: bucket = hash of the whole k-mer (+ L2 prefilter); 1: fingerprint bucket pair by 16-base minimizer (K = 60);
    // 2: bit array over the identities of 32-base minimizers (K = 60 default; F holds the 2^fbits bits)
    uint32_t layout;
    uint32_t fbits;
    // layout 2: K-mers whose leftmost and rightmost minimum differ, by the identity of the rightmost one (sorted)
    const unsigned long long* alias_z;
    const uint32_t* alias_i;     // index in D
    const uint32_t* alias_bloom; // 2^16 bits over the low identity bits of the aliases
    uint32_t n_alias;
};

struct mlg_db {
    mlg_ctx* ctx = nullptr;
    DbView v{};
    DevBuf<key128> P_key;
    DevBuf<uint32_t> P_slot, pidx, rep, bstart, T1;
    DevBuf<uint32_t> F;
    DevBuf<unsigned long long> alias_z;
    DevBuf<uint32_t> alias_i, alias_bloom;
    DevBuf<key128> D_key;
    DevBuf<unsigned char> D_mult;    // per k-mer of D: sketch slots that hold it (either strand), saturating at 255 -- its count in the KMC database
                                     // of the sketches (retrain_and_test_metalign.sh:66); only mlg_query_dump_intersection reads it
    DevBuf<uint32_t> hoff, hits;     // precomputed hit records per k-mer of D (hoff.p == nullptr: not built)
    DevBuf<unsigned long long> hbase; // 64-bit word offset of every group of 2^MLG_HGROUP_SHIFT k-mers' records
    unsigned long long hit_words = 0;
    bool p_dropped = false;          // P / pidx / rep were released after the hit records were built
    unsigned long long hits_skipped_bytes = 0;   // != 0: the hit records (this many bytes) did not fit beside P; queries expand on the fly
    DevBuf<unsigned char> clean_cnt8; // an all-zero counter table handed from one finished query to the next (no 0.16 GB memset per query)
    DevBuf<long long> den_real;      // G*nk
    DevBuf<unsigned char> has_empty; // G
    double build_ms = 0;
};

int mlg_db_build_device(mlg_ctx* ctx, const key128* d_keys, uint32_t G, uint32_t n, uint32_t K,
                        const uint32_t* ks, uint32_t nk, mlg_db** out);
// the same build fed chunk by chunk (db.cu): the caller never holds all G*n keys on the device
struct mlg_db_builder;
int mlg_db_builder_create_impl(mlg_ctx* ctx, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks, uint32_t nk, mlg_db_builder** out);
int mlg_db_builder_add_impl(mlg_db_builder* b, const key128* d_keys, uint32_t g0, uint32_t count);
int mlg_db_builder_finish_impl(mlg_db_builder* b, mlg_db** out);      // frees the builder on success
void mlg_db_builder_destroy_impl(mlg_db_builder* b);
void mlg_db_builder_shape(const mlg_db_builder* b, mlg_ctx** ctx, uint32_t* G, uint32_t* n, uint32_t* K, uint32_t* next_g);
// genome files sketched on the device and appended to the builder (sketch.cu)
int mlg_db_builder_add_fasta_impl(mlg_db_builder* b, const void* bytes, const uint64_t* file_off, uint32_t nfiles, uint64_t prime,
                                  mlg_fasta_stats* st);
// .mlgdb files (dbfile.cu): version 1 = source keys (built on load), version 2 = the built structures
int mlg_db_load_file(mlg_ctx* ctx, const char* path, mlg_db** out);
int mlg_db_save_file(const mlg_db* db, const char* path, const char* names, uint64_t names_bytes);

// ---- kernels' host launchers (probe.cu / query.cu) ----
struct ProbeArgs {
    const unsigned long long* bases;    // packed stream as 8-byte words (32 bases each, stream byte order)
    const unsigned long long* nmask;    // N mask as 8-byte words (64 bases each), may be null
    const unsigned long long* off;      // read offsets in bases (n_reads + 1), or null: every read is read_len long
    uint32_t read_len;
    unsigned long long base_words;      // readable 8-byte words of `bases` (loads are clamped to it)
    unsigned long long nmask_words;     // readable 8-byte words of `nmask`
    unsigned long long r_begin, r_end;  // reads of this launch
    unsigned char* cnt8;                // nd saturating occurrence counters
    uint32_t ci_min;                    // a counter reaching ci_min appends its index to present[]
    uint32_t* present;                  // nd entries
    unsigned long long* n_present;      // device cursors: [0] of present[], [1] of touched[]
    uint32_t* touched;                  // nd entries: counters that left zero
    unsigned long long* tile_counter;   // layout 1: next 32-read tile to hand out (zeroed before every launch)
    unsigned long long* n_kmers;        // device accumulators: [0] valid windows, [1] level-1 bucket fetches (layout 1)
};
int launch_probe(const mlg_ctx* ctx, const DbView& db, const ProbeArgs& a, cudaStream_t st);
int launch_pack_ascii(const unsigned char* text, unsigned long long nbases, unsigned char* bases, unsigned char* nmask,
                      cudaStream_t st);
int launch_ascii_to_keys(const unsigned char* text, unsigned long long nslots, uint32_t K, key128* keys, cudaStream_t st);

int launch_clamp_counts(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp, cudaStream_t st);
int launch_pack_touched(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp,
                        unsigned long long* out, cudaStream_t st);
int launch_merge_sparse(unsigned char* cnt8, const unsigned long long* entries, unsigned long long n, uint32_t nd, uint32_t ci_min,
                        uint32_t* present, uint32_t* touched, unsigned long long* d_cursors, cudaStream_t st);
int launch_pack_exchange(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp,
                         unsigned long long* out, unsigned long long cap, unsigned long long* own_count, cudaStream_t st);
int launch_push_peers(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp,
                      unsigned long long* const* boxes, uint32_t n_peers, unsigned long long cap, unsigned long long epoch,
                      unsigned int* done_ctas, unsigned long long* own_count, cudaStream_t st);
int launch_merge_exchange(unsigned char* cnt8, const unsigned long long* recv, unsigned long long stride_words, uint32_t world, uint32_t rank,
                          unsigned long long cap, uint32_t nd, uint32_t ci_min, uint32_t* present, uint32_t* touched,
                          unsigned long long* d_cursors, unsigned long long* d_status, unsigned long long epoch,
                          unsigned long long timeout_ns, cudaStream_t st);
int launch_compact_present(const unsigned char* cnt8, uint32_t nd, uint32_t ci_min, uint32_t* out, unsigned long long* d_cursor,
                           cudaStream_t st);
int launch_expand_hits(const DbView& db, const uint32_t* present, const unsigned long long* d_n_present, int gate_none,
                       uint32_t* hitbits, unsigned long long words_per_k, unsigned long long* num, cudaStream_t st);
// precomputed hit lists (built once per database, replayed per query); HOFF_NONE = no list, expand on the fly
#define HOFF_NONE 0xFFFFFFFFu
int launch_apply_hits(const DbView& db, const uint32_t* present, const unsigned long long* d_n_present, int gate_none,
                      uint32_t* hitbits, unsigned long long words_per_k, unsigned long long* num, const uint32_t* hoff,
                      const unsigned long long* hbase, const uint32_t* hits, uint32_t* fallback, unsigned long long* d_n_fallback,
                      cudaStream_t st);
// hit-record build (db.cu): tally -> sizes -> offsets (32-bit, relative to a 64-bit base per MLG_HGROUP k-mers) -> fill
#define MLG_HGROUP_SHIFT 16
int launch_tally_hits(const DbView& db, uint32_t* summary, cudaStream_t st);
int launch_hit_group_sums(const uint32_t* summary, uint32_t nd, unsigned long long* gsum, cudaStream_t st);
int launch_hit_offsets(const uint32_t* summary, uint32_t nd, uint32_t* hoff, cudaStream_t st);
int launch_fill_hits(const DbView& db, const uint32_t* summary, uint32_t* hoff, const unsigned long long* hbase,
                     uint32_t* hits, unsigned long long drop_from, cudaStream_t st);
int launch_scatter_nruns(const uint32_t* d_runs, unsigned long long n_runs, unsigned long long nbases, unsigned char* nmask,
                         cudaStream_t st);
int launch_finalize(const unsigned long long* num, const long long* den_real, const unsigned char* has_empty, uint32_t G,
                    uint32_t nk, int count_empty, long long* out_num, long long* out_den, double* out_ci, cudaStream_t st);
int launch_finalize_sparse(const unsigned long long* num, const long long* den_real, const unsigned char* has_empty, uint32_t G, uint32_t nk,
                           int count_empty, uint32_t* out_g, long long* out_num, long long* out_den, double* out_ci, unsigned long long cap,
                           unsigned long long* d_counter, cudaStream_t st);
int launch_clear_touched(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, cudaStream_t st);
int launch_gather_keys(const key128* D_key, const uint32_t* present, uint32_t n_present, key128* out, cudaStream_t st);
int launch_gather_hit_flags(const uint32_t* hitbits, unsigned long long words_per_k, const uint32_t* genomes, uint32_t m, uint32_t n,
                            uint32_t nk, unsigned char* out, cudaStream_t st);
int launch_gather_counts(const unsigned char* cnt8, const unsigned char* D_mult, const uint32_t* present, uint32_t n_present, uint32_t cap,
                         unsigned char* out, cudaStream_t st);

// sort of split 2K-bit keys (db.cu), shared by the database build and the KMC writers
int sort_keys128(unsigned long long* hi, unsigned long long* lo, const uint32_t* vals, uint32_t n, uint32_t K,
                 key128* out, uint32_t* vals_out, cudaStream_t st);

// ---- read k-mer table and KMC database writers (readkmers.cu) ----
struct ReadKmerTable;
struct KmcOutStats { double ms_compact = 0, ms_sort = 0, ms_encode = 0, s_write = 0; unsigned long long records = 0, bytes = 0; };
int rk_create(mlg_ctx* ctx, uint32_t K, unsigned long long max_table_bytes, ReadKmerTable** out);
void rk_destroy(ReadKmerTable* t);
int rk_before_batch(ReadKmerTable* t, unsigned long long batch_windows, uint32_t* launches);   // growth (may launch a rehash)
int rk_count_range(ReadKmerTable* t, const ProbeArgs& a, unsigned long long batch_bases, uint32_t* launches);   // a.r_begin..a.r_end
int rk_after_batch(ReadKmerTable* t, int staging_set);
int rk_check(ReadKmerTable* t);                // joins the streams; MLG_ERR_NOMEM once the table overflowed
int rk_stats(ReadKmerTable* t, mlg_read_kmer_stats* out);
int rk_collect(ReadKmerTable* t, uint32_t min_count, DevBuf<key128>& keys, DevBuf<uint32_t>& counts, uint32_t* n, KmcOutStats* ws);
int rk_sort_pairs(mlg_ctx* ctx, const key128* keys, const unsigned char* counts, uint32_t n, uint32_t K, DevBuf<key128>& keys_out,
                  DevBuf<uint32_t>& counts_out);
int kmc_write(mlg_ctx* ctx, const char* prefix, const key128* keys, const uint32_t* counts, uint32_t n, uint32_t K, uint32_t min_count,
              uint32_t counter_max, KmcOutStats* ws);
// key-range passes (mlg_query_enable_read_kmer_passes): the pushes archive the reads on the device, every output call
// counts them in passes over contiguous intervals of the key order
struct ReadKmerPasses;
int rkp_create(mlg_ctx* ctx, uint32_t K, unsigned long long max_bytes, ReadKmerPasses** out);
void rkp_destroy(ReadKmerPasses* t);
int rkp_archive(ReadKmerPasses* t, const ProbeArgs& a, unsigned long long n_reads, unsigned long long nbases);   // no kernel
int rkp_check(ReadKmerPasses* t);              // joins the streams; MLG_ERR_NOMEM once the archive overflowed
int rkp_read_kmers(ReadKmerPasses* t, uint32_t min_count, uint32_t counter_max, uint64_t* keys_out, uint8_t* counts_out, uint64_t cap,
                   uint64_t* n_total, KmcOutStats* ws);
int rkp_write_kmc(ReadKmerPasses* t, const char* prefix, uint32_t min_count, uint32_t counter_max, KmcOutStats* ws);
int rkp_stats(ReadKmerPasses* t, mlg_read_kmer_stats* out);
int rkp_plan(ReadKmerPasses* t, mlg_read_kmer_plan* out);
// the read k-mer count across ranks (mlg_query_read_kmer_archive / _add_archive): this rank's archive as one device blob,
// a peer's blob appended to the archive, and the peers still missing before the output calls may run
int rkp_pack_archive(ReadKmerPasses* t, uint32_t rank, uint32_t world, const void** d_blob, uint64_t* bytes);
int rkp_add_archive(ReadKmerPasses* t, const void* d_blob, uint64_t bytes, uint32_t* launches);
uint32_t rkp_peers_missing(const ReadKmerPasses* t);
int kmc_concat(const char* prefix, const char* const* parts, uint32_t n_parts);
