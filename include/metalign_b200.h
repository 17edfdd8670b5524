/* metalign_b200 -- C ABI of the B200-native database-selection hot path of Metalign.
 *
 * The reference (nlapier2/Metalign) has no FFI: its hot path is four subprocesses started from
 * scripts/select_db.py.  Each entry point below names the reference step it replaces:
 *
 *   mlg_db_*               the CMash training database that select_db.py:69-70 hands to
 *                          StreamingQueryDNADatabase.py (cmash_db_n1000_k60.h5 + its .tst trie + the
 *                          30-60-10 Bloom prefilter) and the KMC database of its k-mers that
 *                          select_db.py:44 hands to kmc_tools (built at
 *                          local_tests/retrain_and_test_metalign.sh:49-66 via local_tests/dump_kmers.py:7-14)
 *   mlg_query_push_*       `kmc -k60 -fq|-fa -ci2 -cs3` + `kmc_tools simple ... intersect`
 *                          (select_db.py:50-56): canonical K-mer occurrence counting of the reads,
 *                          restricted to the database's k-mers
 *   mlg_query_counts_*     (new) the seam for the one multi-GPU exchange: per-k-mer occurrence
 *                          counters, clamped to ci_min, summed over ranks by the caller (NCCL)
 *   mlg_query_finish       `kmc_dump` + the FASTA rewrite + `StreamingQueryDNADatabase.py <fa> <h5> <csv>
 *                          30-60-10 -c 0 -r 1000000 -v -f <bf> --sensitive` (select_db.py:58-76) up to, but
 *                          not including, the pandas filter/sort/to_csv tail, which stays on the host
 *   mlg_query_intersection the contents of `60mers_intersection_dump` (select_db.py:58-59)
 *   mlg_sketch_genomes     (offline, SURVEY.md 8f-2) CMash `MakeStreamingDNADatabase.py <list> <h5> -n 1000 -k 60`
 *                          (local_tests/retrain_and_test_metalign.sh:49): the bottom-n MinHash sketches the
 *                          database above is made of
 *
 * Conventions
 *   - every function returns MLG_OK (0) or a negative error code; mlg_last_error() gives the message
 *     (thread-local).  There is no CPU fallback: without a CUDA device every call fails.
 *   - one context == one GPU == one host thread (one process per GPU; ranks combine through
 *     mlg_query_counts_export/import).  Work is asynchronous on the context's streams and joined in
 *     mlg_query_finish / mlg_query_counts_export / mlg_query_sync.
 *   - the caller owns every buffer it passes.  Host buffers given to mlg_query_push_* must stay valid
 *     until the next push/sync/finish on that query (pinned memory makes the copies asynchronous).
 *   - k-mer key: 2K-bit integer, first base most significant, A=0 C=1 G=2 T=3, as two uint64 (hi, lo);
 *     an empty CMash sketch slot ('' in CE._kmers) is (~0, ~0).
 *   - packed read stream: reads back to back at base granularity; base i in byte i/4, bits
 *     7-2*(i%4)..6-2*(i%4); N (any non-ACGT symbol) is flagged in nmask (bit i in byte i/8, bit 7-(i%8))
 *     and its 2-bit code is ignored.  `bases` must be readable up to a multiple of 16 bytes covering
 *     ceil(nbases/64) 16-byte words, `nmask` up to a multiple of 16 bytes covering ceil(nbases/64) 8-byte words.
 */
#ifndef METALIGN_B200_H
#define METALIGN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLG_OK 0
#define MLG_ERR_CUDA (-1)
#define MLG_ERR_ARG (-2)
#define MLG_ERR_IO (-3)
#define MLG_ERR_STATE (-4)
#define MLG_ERR_NOMEM (-5)
#define MLG_ERR_RETRY (-6) /* mlg_query_finish after an exchange whose blocks were too small: repeat it with a larger one */

#define MLG_GATE_EXACT 0 /* smallest-k prefilter with zero false positives (SURVEY.md 3.3 R4) */
#define MLG_GATE_NONE 1  /* no prefilter */

typedef struct mlg_ctx mlg_ctx;
typedef struct mlg_db mlg_db;
typedef struct mlg_query mlg_query;
typedef struct mlg_exchange mlg_exchange;

typedef struct mlg_stats {
    uint64_t n_reads;        /* reads pushed */
    uint64_t n_bases;        /* bases pushed (N included) */
    uint64_t n_kmers;        /* N-free K-long windows probed (the metric's unit of work) */
    uint64_t n_intersect;    /* |I|: database k-mers seen >= ci_min times */
    uint64_t n_db_entries;   /* non-empty sketch slots */
    uint64_t n_db_distinct;  /* |D|: distinct canonical sketch k-mers */
    uint64_t n_buckets;      /* level-1 fingerprint buckets */
    uint32_t bucket_bytes;   /* bytes per level-1 fetch: one 16/32-byte bucket (layout 0), one 64-byte bucket pair (layout 1), one 32-byte sector of the minimizer bitmap (layout 2) */
    uint32_t gpu_launches;   /* kernels of this library launched for this query so far */
    uint64_t h2d_bytes;      /* host->device bytes copied for this query */
    uint64_t d2h_bytes;      /* device->host bytes copied for this query */
    double ms_probe;         /* sum of CUDA-event durations of the probe kernel launches */
    double ms_query;         /* CUDA-event duration of the finish stage (compact, expand, popcount, finalize) */
    uint32_t probe_launches; /* number of probe kernel launches in ms_probe */
    uint32_t filter_words;   /* L2 prefilter: number of 32-bit words, 0 = no prefilter */
    uint64_t n_bucket_fetches; /* level-1 fetches from HBM: one per k-mer in layout 0, one per super-k-mer in layouts 1 and 2 */
    uint32_t layout;         /* 0 = bucket by hash of the whole k-mer (+ L2 prefilter), 1 = fingerprint bucket pair by 16-base minimizer, 2 = bit array over the identities of 32-base minimizers (K = 60 default) */
    uint32_t reserved;
} mlg_stats;

const char* mlg_last_error(void);
int mlg_version(void);

/* context: one GPU */
int mlg_ctx_create(int device, mlg_ctx** out);
int mlg_ctx_destroy(mlg_ctx* ctx);
/* the context's cudaStream_t handles: kernels run on *compute_stream, host<->device copies on *copy_stream
 * (for callers that bracket work with CUDA events or order their own work against it) */
int mlg_ctx_streams(mlg_ctx* ctx, void** compute_stream, void** copy_stream);
/* pinned host memory for callers that have no other way to get it */
int mlg_host_alloc(void** out, uint64_t bytes);
int mlg_host_free(void* p);

/* database: G genomes x n sketch slots of K-mers, queried at nk prefix lengths ks[] (ascending, ks[nk-1] <= K) */
int mlg_db_from_keys(mlg_ctx* ctx, const uint64_t* keys /* host, G*n (hi,lo) pairs */, uint32_t G, uint32_t n,
                     uint32_t K, const uint32_t* ks, uint32_t nk, mlg_db** out);
int mlg_db_from_keys_device(mlg_ctx* ctx, const uint64_t* d_keys /* device, 16-byte aligned */, uint32_t G, uint32_t n,
                            uint32_t K, const uint32_t* ks, uint32_t nk, mlg_db** out);
int mlg_db_from_ascii(mlg_ctx* ctx, const char* kmers /* host, G*n*K chars; a slot starting with NUL is empty */,
                      uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks, uint32_t nk, mlg_db** out);
/* The same build fed in chunks of whole genomes, in order (first_genome = the number of genomes added so far): the caller
 * never holds all G*n keys on the device, which is what lets a 2e9-slot database (BASELINE configs[4]) build inside 180 GB.
 * mlg_db_builder_finish frees the builder when it succeeds; after a failure call mlg_db_builder_destroy.  A database whose
 * precomputed hit records would not fit beside its other structures keeps the prefix index instead and expands every
 * query's present k-mers on the fly (same results). */
typedef struct mlg_db_builder mlg_db_builder;
int mlg_db_builder_create(mlg_ctx* ctx, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks, uint32_t nk, mlg_db_builder** out);
int mlg_db_builder_add_device(mlg_db_builder* b, const uint64_t* d_keys /* device, n_genomes*n (hi,lo) pairs */,
                              uint32_t first_genome, uint32_t n_genomes);
int mlg_db_builder_finish(mlg_db_builder* b, mlg_db** out);
int mlg_db_builder_destroy(mlg_db_builder* b);
/* .mlgdb file: the source form (sketch keys; the device structures are built on load) or the built form written by
 * mlg_db_save (the device structures themselves: loading is a file read).  names = the '\n'-joined genome names the
 * file's head carries for the host side (metalign_b200/dbformat.py). */
int mlg_db_load(mlg_ctx* ctx, const char* path /* .mlgdb file */, mlg_db** out);
int mlg_db_save(const mlg_db* db, const char* path, const char* names, uint64_t names_bytes);
int mlg_db_info(const mlg_db* db, uint32_t* G, uint32_t* n, uint32_t* K, uint32_t* nk, uint32_t* ks /* 8 */,
                uint64_t* n_entries, uint64_t* n_distinct);
/* static denominators: distinct k-prefixes per genome (+1 for '' where the genome has an empty slot) */
int mlg_db_denominators(const mlg_db* db, int count_empty_in_den, int64_t* den /* host, G*nk */);
int mlg_db_free(mlg_db* db);

/* query */
int mlg_query_begin(mlg_ctx* ctx, mlg_db* db, int ci_min, int gate_mode, int count_empty_in_den, mlg_query** out);
/* host buffers; read_off (n_reads+1 entries, in bases) or NULL with every read read_len long */
int mlg_query_push_packed(mlg_query* q, const uint8_t* bases, const uint8_t* nmask_or_null,
                          const uint64_t* read_off_or_null, uint64_t n_reads, uint32_t read_len);
/* same, with N given as n_runs sorted, non-overlapping (start, length) pairs of uint32 in batch base coordinates
 * instead of a bit mask (NULL / 0: the batch has no N).  N is rare in real reads, so this format moves 1/3 fewer
 * bytes over PCIe than the mask does; the mask is rebuilt on the device.  A batch must hold < 2^32 bases. */
int mlg_query_push_packed_nruns(mlg_query* q, const uint8_t* bases, const uint32_t* nruns_or_null, uint64_t n_runs,
                                const uint64_t* read_off_or_null, uint64_t n_reads, uint32_t read_len);
/* same as mlg_query_push_packed, buffers already on the device (16-byte aligned); they must stay valid until the next sync/finish */
int mlg_query_push_packed_device(mlg_query* q, const uint8_t* d_bases, const uint8_t* d_nmask_or_null,
                                 const uint64_t* d_read_off_or_null, uint64_t n_reads, uint32_t read_len);
/* host ASCII: read i = text[read_off[i] .. read_off[i+1]); anything outside ACGTacgt is N */
int mlg_query_push_ascii(mlg_query* q, const char* text, const uint64_t* read_off, uint64_t n_reads);
int mlg_query_sync(mlg_query* q);
/* multi-GPU seam: device pointer to the |D| uint8 occurrence counters, clamped to ci_min, work joined.
 * After the caller has summed them over ranks in place, mlg_query_counts_import() tells the query to
 * derive presence from the summed table. */
int mlg_query_counts_export(mlg_query* q, uint8_t** d_counts, uint64_t* n_counts);
int mlg_query_counts_import(mlg_query* q);
/* the same seam in sparse form (the counter table is >99.9 % zeros): *d_entries = device array of one 64-bit entry per
 * non-zero counter, index | min(count, ci_min) << 32, work joined; the caller all-gathers the ranks' arrays and hands
 * every OTHER rank's array to mlg_query_counts_merge_sparse(), which adds it into this rank's counters.  Entries with
 * count 0 (padding) are ignored.  After the first merge no more reads can be pushed. */
int mlg_query_counts_export_sparse(mlg_query* q, uint64_t** d_entries, uint64_t* n_entries);
int mlg_query_counts_merge_sparse(mlg_query* q, const uint64_t* d_entries, uint64_t n_entries);
/* The same exchange WITHOUT a host round trip (everything below is queued on the context's compute stream; nothing
 * synchronises the host).  An mlg_exchange is one rank's end: persistent buffers sized for cap_entries non-zero
 * counters per rank.  A rank's contribution is one block of *block_words uint64: [0] its number of non-zero counters,
 * [1] unused, then the entries.
 *   all-gather form:  mlg_query_exchange_pack() fills *d_send; the caller all-gathers every rank's block into *d_recv
 *                     (world blocks, rank order; e.g. ncclAllGather / torch.distributed on the compute stream);
 *                     mlg_query_exchange_merge() adds the other ranks' blocks into this rank's counters.
 *   direct form:      mlg_query_exchange_p2p() stores the block straight into every peer's mailbox over NVLink
 *                     (peer-mapped memory: exchange the 64-byte handles of mlg_exchange_local_handle() between the
 *                     ranks once, then mlg_exchange_connect()), publishes it with a system-scope release, waits on the
 *                     device for the peers' blocks and merges them -- no NCCL call, no host involvement.  Collective:
 *                     every rank must call it once per query, in the same order.
 *   dense form:       mlg_query_exchange_dense() = mlg_query_counts_export() + _import() without the host join.
 * If some rank had more than cap_entries non-zero counters, nothing is merged on any rank and mlg_query_finish()
 * returns MLG_ERR_RETRY: repeat the exchange with a larger mlg_exchange and call finish again.  Every rank judges all
 * world counts, its own included, so every rank gets the same answer, and the error message names the largest count.
 * Every form leaves the same counters on every rank: the sum over ranks of min(count, ci_min).  The pack calls
 * (mlg_query_counts_export*, mlg_query_exchange_pack / _p2p / _dense) clamp the rank's own counters to ci_min in place. */
int mlg_exchange_create(mlg_ctx* ctx, uint32_t world, uint32_t rank, uint64_t cap_entries, mlg_exchange** out);
int mlg_exchange_destroy(mlg_exchange* ex);
int mlg_exchange_buffers(mlg_exchange* ex, uint64_t** d_send, uint64_t** d_recv, uint64_t* block_words);
int mlg_exchange_local_handle(mlg_exchange* ex, void* handle64 /* 64 bytes out */);
int mlg_exchange_connect(mlg_exchange* ex, const void* handles /* world * 64 bytes, rank order */);
int mlg_query_exchange_pack(mlg_query* q, mlg_exchange* ex);
int mlg_query_exchange_merge(mlg_query* q, mlg_exchange* ex);
int mlg_query_exchange_p2p(mlg_query* q, mlg_exchange* ex);
int mlg_query_exchange_dense(mlg_query* q, uint8_t** d_counts, uint64_t* n_counts);
/* num/den: int64 [G*nk]; ci: double [G*nk] (num/den where num > 0, else 0.0); any pointer may be NULL */
int mlg_query_finish(mlg_query* q, int64_t* num, int64_t* den, double* ci, uint64_t* n_intersect);
/* the same result in sparse form: one row per genome with a hit at any k (in no particular order) -- genome index, and
 * nk values each of num / den / ci per row; any output pointer may be NULL.  *n_rows = the number of rows; if it exceeds
 * cap_rows the call fails with MLG_ERR_ARG and can be repeated with larger buffers.  Everything select_db.py keeps is in
 * these rows: CMash's tail drops the genomes whose containment at the largest k is 0 (SURVEY.md 3.3 R6). */
int mlg_query_finish_sparse(mlg_query* q, uint32_t* genomes, int64_t* num, int64_t* den, double* ci, uint64_t cap_rows,
                            uint64_t* n_rows, uint64_t* n_intersect);
/* after finish: for each of the m genomes listed, nk*n bytes, out[(i*nk + ki)*n + j] = 1 where sketch slot j of genomes[i] is
 * the representative of a (genome, ks[ki]-prefix) class the query hit (one slot per class carries the flag).  This is what
 * CMash's post-processing works on when --sensitive is NOT given (it re-filters the hits to k-mers unique to one organism;
 * Metalign always passes --sensitive, select_db.py:76, so the drop-in never calls this); the host side of it is
 * metalign_b200/cmash_tail.py: refilter_unique. */
int mlg_query_hit_flags(mlg_query* q, const uint32_t* genomes, uint32_t m, uint8_t* out);
/* after finish: I as (hi,lo) canonical keys in increasing order; writes at most cap pairs, *n = |I| */
int mlg_query_intersection(mlg_query* q, uint64_t* keys_out, uint64_t cap, uint64_t* n);
/* after finish: `kmc_dump <temp>/60mers_intersection <temp>/60mers_intersection_dump` and the FASTA rewrite that follows it
 * (scripts/select_db.py:58-65) as files: one "<k-mer>\t<count>" line per k-mer of I in lexicographic order, and, if asked
 * for, the ">seq" / k-mer records of 60mers_intersection_dump.fa.  count = what `kmc_tools simple ... intersect` keeps: the
 * smaller of the k-mer's occurrences in the reads and the number of sketch slots that hold it, both saturated at
 * counter_max (the reference builds both KMC databases with -cs3: select_db.py:50, retrain_and_test_metalign.sh:66).
 * Exact for a query whose reads were all pushed here; after a multi-GPU exchange, in every form and on every rank, the
 * read counter is the sum over ranks of the per-rank counters clamped to ci_min. */
int mlg_query_dump_intersection(mlg_query* q, const char* dump_path, const char* fasta_path_or_null, uint32_t counter_max);
int mlg_query_stats(mlg_query* q, mlg_stats* out);
int mlg_query_free(mlg_query* q);

/* Read k-mer table (off unless enabled): every canonical K-mer of the pushed reads with a count saturating at 255, the
 * counting part of `kmc -k<K> -ci<min_count> -cs<counter_max>` (select_db.py:50-52), so that the two KMC databases the
 * reference leaves in its temp dir (reads_60mers, 60mers_intersection) can be written.  The table lives on this rank's GPU
 * and grows with the reads; max_table_bytes caps it (0 = no cap).  A table that would pass the cap, or whose allocation
 * fails, stops counting: the query itself is unaffected and the read k-mer calls return MLG_ERR_NOMEM.  After any counter
 * exchange (mlg_query_counts_*, mlg_query_exchange_*) they return MLG_ERR_STATE: the table is not merged across ranks.
 * (The key-range passes below count across ranks instead: mlg_query_read_kmer_archive.)  Without the table they return
 * MLG_ERR_STATE too. */
typedef struct mlg_read_kmer_stats {
    uint64_t windows;        /* N-free K-long windows counted */
    uint64_t distinct;       /* distinct canonical k-mers in the table */
    uint64_t slots;          /* 16-byte slots of the table */
    uint64_t bytes;          /* device bytes of the table */
    uint64_t bytes_needed;   /* overflowed: the bytes the table would have needed */
    uint32_t grows;          /* rehashes into a larger table */
    uint32_t overflowed;     /* 1: the table passed its budget or could not be allocated */
    double ms_count;         /* CUDA-event time of the count kernel launches */
    double ms_rehash;        /* CUDA-event time of the rehash launches */
    /* the last mlg_query_read_kmers / mlg_query_write_reads_kmc call */
    uint64_t out_records;    /* k-mers selected */
    uint64_t out_bytes;      /* bytes written (both files) */
    double ms_compact;       /* selection of the slots >= min_count */
    double ms_sort;          /* sort by key */
    double ms_encode;        /* prefix table and .kmc_suf records */
    double s_write;          /* seconds of copying back and writing the files */
} mlg_read_kmer_stats;
/* before the first push: also count every canonical K-mer of the pushed reads (K <= 60); max_table_bytes 0 = no cap */
int mlg_query_enable_read_kmers(mlg_query* q, uint64_t max_table_bytes);
/* after sync or finish: the read k-mers seen >= min_count times, counts saturated at counter_max, keys ascending; writes
 * at most cap (hi,lo) pairs and counts, *n = their number */
int mlg_query_read_kmers(mlg_query* q, uint32_t min_count, uint32_t counter_max, uint64_t* keys_out /* (hi,lo) */,
                         uint8_t* counts_out, uint64_t cap, uint64_t* n);
/* `kmc -k<K> -ci<min_count> -cs<counter_max>` of the pushed reads as <prefix>.kmc_pre / <prefix>.kmc_suf */
int mlg_query_write_reads_kmc(mlg_query* q, const char* prefix, uint32_t min_count, uint32_t counter_max);
/* Key-range passes: a second mode of the same calls for read sets whose table would not fit.  Enabled before the first
 * push instead of mlg_query_enable_read_kmers (either after the other, or after a push: MLG_ERR_STATE).  The pushes only
 * copy the reads into a device archive (0.375 bytes per base; no kernel launch).  Every mlg_query_read_kmers /
 * mlg_query_write_reads_kmc call then plans contiguous intervals of the canonical key order from a histogram of the
 * archive and counts each interval in a table of its own, one after the other; the results are those of the single
 * table.  max_bytes caps the archive plus one pass (0 = the free device memory at the output call, less 1 GiB).  An
 * archive that would pass it, or whose allocation fails, stops archiving: the query is unaffected and the output calls
 * return MLG_ERR_NOMEM, as they do when the cap leaves no room for the smallest pass.  Passes lift the 2^32 limit on the
 * records of one call (each pass sorts < 2^32 keys).  In this mode mlg_read_kmer_stats describes the last output call:
 * windows (from the histogram), distinct (summed over the passes), slots / bytes (of the largest pass), ms_count (summed),
 * out_* as in the other mode; grows and ms_rehash are 0; bytes_needed, once the archive overflowed, what the archive of
 * every batch pushed would need.  A failed mlg_query_write_reads_kmc leaves neither file behind. */
int mlg_query_enable_read_kmer_passes(mlg_query* q, uint64_t max_bytes);
typedef struct mlg_read_kmer_plan {
    uint32_t passes;         /* key-range passes of the last output call */
    uint32_t refined_bins;   /* histogram bins that alone passed the cap and were split by their next bases */
    uint64_t archive_bytes;  /* device copy of the reads */
    uint64_t pass_cap_bytes; /* device bytes one pass may use: table + output stage */
    uint64_t max_pass_bound; /* largest bound on the distinct keys of one pass */
    uint64_t distinct;       /* distinct canonical k-mers, summed over the passes */
    double ms_histogram;     /* CUDA-event time of the histogram launches */
    double ms_count;         /* CUDA-event time of the ranged count launches */
    double ms_output;        /* CUDA-event time of selection, sort and encoding */
    /* the count across ranks (mlg_query_read_kmer_archive); a query that never called it is rank 0 of 1 */
    uint32_t rank;           /* this rank: its output holds share `rank` of the key order */
    uint32_t world;          /* ranks */
    uint32_t peers_added;    /* peer archives added */
    uint32_t reserved;
    uint64_t share_first_bin; /* the share: top-level bins [first, end) of the min(K, 10) leading bases of the canonical key */
    uint64_t share_end_bin;
    uint64_t share_windows;  /* windows of the share's bins (mlg_read_kmer_stats.windows stays the total over every archive) */
} mlg_read_kmer_plan;
/* the plan of the last output call in passes mode (MLG_ERR_STATE in any other mode) */
int mlg_query_read_kmer_plan(mlg_query* q, mlg_read_kmer_plan* out);
/* The read k-mers of reads sharded over W ranks, in passes mode only: every rank receives every other rank's archive, and
 * rank r counts share r of the canonical key order over all the reads, so its counts are global and exact.  Share r is
 * a contiguous run of the top-level histogram bins (DESIGN.md section 10); the shares of ranks 0..W-1, in rank order,
 * are the whole key order, and so are the KMC databases the ranks write (mlg_kmc_concat joins them into the file one
 * query over all the reads writes).
 *   mlg_query_read_kmer_archive   after the last push: this rank's archive packed into one device blob the query owns
 *                                 (copies on the compute stream, no host join; valid until the first output call or
 *                                 mlg_query_free, so a peer's copy of it must be ordered on this context's compute stream
 *                                 before that call).  From then on the query is rank `rank` of `world` (1..16) and
 *                                 refuses pushes.  An archive that outgrew its budget sends a header flagged overflowed.
 *                                 MLG_ERR_STATE without passes or on a second call; MLG_ERR_ARG for rank >= world or world > 16.
 *   mlg_query_read_kmer_add_archive  a peer's blob (device memory of this GPU, 8-byte aligned), copied into the archive: it counts
 *                                 against the budget.  The blob is checked first -- header (magic, library version, K,
 *                                 world, sizes that add up to `bytes`), its rank (not this one, not one already added,
 *                                 < world) and, by a kernel, every batch's read offsets -- and a blob that fails returns
 *                                 MLG_ERR_ARG and changes nothing.  A flagged blob, or one past the budget, makes the
 *                                 output calls return MLG_ERR_NOMEM on this rank too, so every rank reaches the same verdict.
 * mlg_query_read_kmers / mlg_query_write_reads_kmc return MLG_ERR_STATE until every one of the world - 1 peers has been
 * added, and then return / write the share's keys only; a counter exchange no longer makes them refuse. */
int mlg_query_read_kmer_archive(mlg_query* q, uint32_t rank, uint32_t world, const void** d_blob, uint64_t* bytes);
int mlg_query_read_kmer_add_archive(mlg_query* q, const void* d_blob, uint64_t bytes);
/* Host only (no context): the version-0 KMC databases part_prefixes[0..n_parts) -- the same k, mode, counter size,
 * lut_prefix_length, min / max count, each one's keys above the last one's -- joined into <prefix>.kmc_pre / .kmc_suf:
 * the suffix bodies one after the other, the prefix tables and totals summed.  The parts are read in pieces and left as
 * they are; a call that fails leaves no output file behind (MLG_ERR_ARG for parts that do not fit together, MLG_ERR_IO
 * for files that cannot be read or written). */
int mlg_kmc_concat(const char* prefix, const char* const* part_prefixes, uint32_t n_parts);
/* after finish: `kmc_tools simple <reads> <db> intersect <prefix>`: the k-mers of I, count = the count column of
 * mlg_query_dump_intersection.  Needs no read k-mer table. */
int mlg_query_write_intersection_kmc(mlg_query* q, const char* prefix, uint32_t counter_max);
/* Both files are written in the version-0 layout (one sorted table, what kmc_tools writes; lut_prefix_length = the
 * smallest p >= 4 with (K - p) % 4 == 0, counter_size 1); the reads file has min_count / max_count = min_count /
 * counter_max, the intersection file 1 / counter_max.  The stats join the compute stream. */
int mlg_query_read_kmer_stats(mlg_query* q, mlg_read_kmer_stats* out);

/* Sketch builder (offline): bottom-n MinHash sketch of G genomes, CMash semantics (MinHash.CountEstimator with
 * rev_comp=False, as MakeStreamingDNADatabase.py builds Metalign's training database): every K-long window of
 * text[genome_off[g] .. genome_off[g+1]) that consists of ACGT/acgt only is upper-cased and hashed with
 * MurmurHash3_x64_128 (seed 0, first 64-bit word) modulo `prime` (0 = CMash's 9999999999971); a genome's sketch is its n
 * smallest distinct hash values in ascending order.  Records (contigs) of one genome are separated by any non-ACGT byte.
 * Outputs (host, G*n slots): mins (prime where the slot is unused), counts, kmers (K bytes per slot: the first k-mer
 * with that hash, upper case; NUL-filled where unused -- the layout mlg_db_from_ascii takes).  counts are CountEstimator's:
 * the occurrences of the hash in the genome, except in the last slot of a full sketch, whose repeats stop counting once
 * the n-1 smaller hashes have all appeared (`h >= mins[-1]` returns early): there it is the number of occurrences before
 * that moment, and at least 1 (so always 1 when n = 1); 0 where the slot is unused.
 * Refused with MLG_ERR_ARG before anything is written: null pointers, K outside 1..64, n = 0, G = 0 or G >= 2^20,
 * prime = 1 or prime >= 2^44, a genome_off that decreases anywhere, a single genome of about 4 GB or more.
 * The text goes to the device in passes of about 1 GB (whole genomes; a genome larger than that has a pass of its own);
 * the environment variable MLG_SKETCH_PASS_BYTES, read on every call, sets the bytes per pass instead (any value >= 1;
 * an experiment and test knob, the results do not depend on it). */
typedef struct mlg_sketch_stats {
    uint64_t n_windows;      /* N-free K-long windows hashed */
    uint64_t n_candidates;   /* windows below their genome's threshold (sorted and ranked) */
    double ms_kernels;       /* CUDA-event time of the kernels, all passes */
    uint32_t passes;         /* device passes (more than ceil(bytes / 1 GB) when a genome needed a wider threshold) */
    uint32_t reserved;
} mlg_sketch_stats;
int mlg_sketch_genomes(mlg_ctx* ctx, const char* text, const uint64_t* genome_off /* G+1 */, uint32_t G, uint32_t n, uint32_t K,
                       uint64_t prime, uint64_t* mins, uint32_t* counts, char* kmers, mlg_sketch_stats* stats_or_null);

#ifdef __cplusplus
}
#endif
#endif /* METALIGN_B200_H */
