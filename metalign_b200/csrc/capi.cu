// C ABI of libmetalign_b200.so (declared in include/metalign_b200.h).  Host-side orchestration only:
// buffers, streams, chunked host->device copies overlapped with the probe kernel, and the finish stage.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include "mlg_internal.h"

#define MLG_API __attribute__((visibility("default")))

static thread_local char g_err[512] = "";

void mlg_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ---------------------------------------------------------------- caching device-memory pool
#include <map>
#include <mutex>
namespace {
struct PoolBlock { void* p; size_t bytes; };
struct Pool {
    std::mutex mu;
    std::map<int, std::vector<PoolBlock>> free_blocks;   // per device
    std::map<void*, std::pair<int, size_t>> live;        // ptr -> (device, bytes)
};
Pool& pool() { static Pool* p = new Pool(); return *p; }
constexpr size_t POOL_MAX_CACHED_PER_DEVICE = 64;
}  // namespace

void* mlg_pool_alloc(size_t bytes) {
    bytes = (bytes + 511) & ~(size_t)511;
    int dev = 0;
    cudaGetDevice(&dev);
    Pool& P = pool();
    {
        std::lock_guard<std::mutex> g(P.mu);
        auto& v = P.free_blocks[dev];
        int best = -1;
        for (int i = 0; i < (int)v.size(); ++i)
            if (v[i].bytes >= bytes && v[i].bytes <= bytes + bytes / 4 + 4096 && (best < 0 || v[i].bytes < v[best].bytes)) best = i;
        if (best >= 0) {
            PoolBlock b = v[best];
            v.erase(v.begin() + best);
            P.live[b.p] = {dev, b.bytes};
            return b.p;
        }
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        mlg_pool_trim(dev);                      // give cached blocks back and retry once
        e = cudaMalloc(&p, bytes);
    }
    if (e != cudaSuccess) {
        mlg_set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        return nullptr;
    }
    std::lock_guard<std::mutex> g(P.mu);
    P.live[p] = {dev, bytes};
    return p;
}
void mlg_pool_free(void* p) {
    if (!p) return;
    Pool& P = pool();
    std::unique_lock<std::mutex> g(P.mu);
    auto it = P.live.find(p);
    if (it == P.live.end()) { g.unlock(); cudaFree(p); return; }
    int dev = it->second.first; size_t bytes = it->second.second;
    P.live.erase(it);
    auto& v = P.free_blocks[dev];
    if (v.size() >= POOL_MAX_CACHED_PER_DEVICE) {
        // evict the largest cached block rather than growing without bound
        size_t big = 0;
        for (size_t i = 1; i < v.size(); ++i) if (v[i].bytes > v[big].bytes) big = i;
        void* victim = v[big].p;
        v[big] = {p, bytes};
        g.unlock();
        cudaFree(victim);
        return;
    }
    v.push_back({p, bytes});
}
MLG_API int mlg_device_memory(int device, uint64_t* live_bytes, uint64_t* cached_bytes) {
    Pool& P = pool();
    std::lock_guard<std::mutex> g(P.mu);
    uint64_t live = 0, cached = 0;
    for (const auto& kv : P.live) if (kv.second.first == device) live += kv.second.second;
    auto it = P.free_blocks.find(device);
    if (it != P.free_blocks.end()) for (const auto& b : it->second) cached += b.bytes;
    if (live_bytes) *live_bytes = live;
    if (cached_bytes) *cached_bytes = cached;
    return MLG_OK;
}
void mlg_pool_trim(int device) {
    Pool& P = pool();
    std::vector<PoolBlock> blocks;
    {
        std::lock_guard<std::mutex> g(P.mu);
        blocks.swap(P.free_blocks[device]);
    }
    for (auto& b : blocks) cudaFree(b.p);
}

namespace {

constexpr unsigned long long CHUNK_WORDS = 2ull * 64ull * MLG_TILE_WORDS * 32ull;   // 1048576 words = 16 MiB of packed bases per copy chunk

struct Staging {
    DevBuf<unsigned char> bases, nmask;
    DevBuf<unsigned long long> off;
    DevBuf<unsigned char> text;
    DevBuf<uint32_t> nruns;
    cudaEvent_t done = nullptr;   // last kernel reading this staging set
    bool used = false;
};

inline unsigned long long round_up(unsigned long long x, unsigned long long m) { return (x + m - 1) / m * m; }

}  // namespace

// One rank's end of the multi-GPU exchange (include/metalign_b200.h, "exchange"): persistent blocks for the all-gather
// form, and the peer-mapped mailboxes of the direct (NVLink store) form.
struct mlg_exchange {
    mlg_ctx* ctx = nullptr;
    uint32_t world = 1, rank = 0;
    unsigned long long cap = 0, block_words = 0;
    DevBuf<unsigned long long> send, recv, status;     // status: [0] largest count of an overflowing exchange, [1] peer timeout,
                                                       // [2] CTA counter, [3] this rank's count at the last pack
    unsigned long long* mailbox = nullptr;             // [world senders][2 parities][block_words], cudaMalloc'ed (IPC-exportable)
    unsigned long long* peer_mailbox[MLG_MAX_RANKS] = {};   // peers' mailboxes as mapped into this process (own slot unused)
    bool connected = false;
    unsigned long long epoch = 0;
    unsigned long long timeout_ns = 20ull * 1000ull * 1000ull * 1000ull;
};

struct mlg_query {
    mlg_ctx* ctx = nullptr;
    mlg_db* db = nullptr;
    int ci_min = 2, gate = MLG_GATE_EXACT, count_empty = 1;
    int ex_clamp = 2;                              // a rank's counters are clamped to this before an exchange (>= ci_min)
    DevBuf<unsigned char> cnt8;
    DevBuf<unsigned long long> d_nkmers, d_scalar;
    Staging stg[2];
    int cur = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> probe_events;
    std::vector<cudaEvent_t> chunk_events;
    cudaEvent_t ev_q0 = nullptr, ev_q1 = nullptr;
    mlg_stats st{};
    bool finished = false, reduced = false, merged = false;
    mlg_exchange* ex_pending = nullptr;            // exchange whose status words mlg_query_finish has to look at
    DevBuf<uint32_t> fallback;                     // k-mers without a hit record (databases that kept P only)
    DevBuf<unsigned long long> d_rows;             // sparse finish: row counter
    DevBuf<unsigned long long> sparse;             // this rank's non-zero counters as index | count << 32
    unsigned long long chunk_words = CHUNK_WORDS;   // 64-base words per host->device copy chunk
    // results kept for mlg_query_intersection
    DevBuf<uint32_t> present, touched;
    uint32_t n_present = 0;
    // the finish stage's tables (hit bitmap, per-genome counts): allocated and zeroed on the COPY stream at the first push,
    // so that the 0.1 GB memset runs beside the probe kernel instead of behind it
    DevBuf<uint32_t> hitbits;
    DevBuf<unsigned long long> d_num;
    // read k-mer table (mlg_query_enable_read_kmers; null = off) and what its last output stage measured
    ReadKmerTable* rk = nullptr;
    ReadKmerPasses* rkp = nullptr;                 // the key-range mode instead (mlg_query_enable_read_kmer_passes; null = off)
    KmcOutStats rk_out;
    bool exchanged = false;                        // counters went through an exchange: the per-rank table no longer matches
    bool rk_shared = false;                        // rank of a read k-mer count across ranks (mlg_query_read_kmer_archive)
};

namespace {

int ensure_device(mlg_ctx* ctx) { CUDA_TRY(cudaSetDevice(ctx->device)); return MLG_OK; }

// device-side part common to every push: launch the probe over the batch's reads, in ranges; range i may
// start once copy event i (if any) has completed
struct ReadRange {
    unsigned long long r_end; cudaEvent_t ready;
    unsigned long long run0 = 0, run1 = 0;      // N runs [run0, run1) to scatter into the mask before this range is probed
};

int run_probe(mlg_query* q, Staging& s, const unsigned char* d_bases, const unsigned char* d_nmask,
              const unsigned long long* d_off, unsigned long long n_reads, uint32_t read_len, unsigned long long nbases,
              const std::vector<ReadRange>* ranges) {
    mlg_ctx* ctx = q->ctx;
    if (!q->present.p) {                       // first push: room for every database k-mer to become present once
        MLG_TRY(q->present.alloc((size_t)q->db->v.nd + 1));
        MLG_TRY(q->touched.alloc((size_t)q->db->v.nd + 1));
        const DbView& v = q->db->v;
        const unsigned long long words_per_k = ((unsigned long long)v.G * v.n + 31) / 32;
        MLG_TRY(q->hitbits.alloc(words_per_k * v.nk));
        MLG_TRY(q->d_num.alloc((size_t)v.G * v.nk));
        CUDA_TRY(cudaMemsetAsync(q->hitbits.p, 0, words_per_k * v.nk * 4, ctx->s_copy));      // joined at the top of the finish stage
        CUDA_TRY(cudaMemsetAsync(q->d_num.p, 0, (size_t)v.G * v.nk * 8, ctx->s_copy));
    }
    const unsigned long long nwords64 = (nbases + 63) / 64;       // 64-base words: 16 bytes of bases, 8 bytes of mask
    ProbeArgs a{};
    a.bases = reinterpret_cast<const unsigned long long*>(d_bases);
    a.nmask = reinterpret_cast<const unsigned long long*>(d_nmask);
    a.off = d_off; a.read_len = read_len;
    a.base_words = nwords64 * 2;                                  // buffers cover whole 16-byte units
    a.nmask_words = round_up(nwords64, 2);
    a.cnt8 = q->cnt8.p; a.n_kmers = q->d_nkmers.p;
    a.ci_min = (uint32_t)q->ci_min; a.present = q->present.p; a.n_present = q->d_scalar.p; a.touched = q->touched.p; a.tile_counter = q->d_scalar.p + 3;
    auto launch_range = [&](unsigned long long r0, unsigned long long r1) -> int {
        if (r1 <= r0) return MLG_OK;
        cudaEvent_t e0, e1;
        CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
        a.r_begin = r0; a.r_end = r1;
        CUDA_TRY(cudaEventRecord(e0, ctx->s_comp));
        MLG_TRY(launch_probe(ctx, q->db->v, a, ctx->s_comp));
        CUDA_TRY(cudaEventRecord(e1, ctx->s_comp));
        q->probe_events.emplace_back(e0, e1);
        q->st.gpu_launches += 1; q->st.probe_launches += 1;
        if (q->rk) MLG_TRY(rk_count_range(q->rk, a, nbases, &q->st.gpu_launches));
        return MLG_OK;
    };
    if (q->rk) {
        const uint32_t K = q->db->v.K;
        const unsigned long long windows = read_len ? n_reads * (read_len >= K ? read_len - K + 1ull : 0ull) : nbases;   // upper bound
        MLG_TRY(rk_before_batch(q->rk, windows, &q->st.gpu_launches));
    }
    if (ranges) {
        unsigned long long r0 = 0;
        for (auto& rr : *ranges) {
            CUDA_TRY(cudaStreamWaitEvent(ctx->s_comp, rr.ready, 0));
            if (rr.run1 > rr.run0) {
                MLG_TRY(launch_scatter_nruns(s.nruns.p + 2 * rr.run0, rr.run1 - rr.run0, nbases, s.nmask.p, ctx->s_comp));
                q->st.gpu_launches += 1;
            }
            MLG_TRY(launch_range(r0, rr.r_end));
            if (rr.r_end > r0) r0 = rr.r_end;
        }
    } else {
        MLG_TRY(launch_range(0, n_reads));
    }
    if (q->rk) MLG_TRY(rk_after_batch(q->rk, q->cur));
    if (q->rkp) MLG_TRY(rkp_archive(q->rkp, a, n_reads, nbases));
    if (!s.done) CUDA_TRY(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(s.done, ctx->s_comp));
    s.used = true;
    q->st.n_reads += n_reads; q->st.n_bases += nbases;
    return MLG_OK;
}

int check_push(mlg_query* q) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (q->finished) { mlg_set_error("query already finished"); return MLG_ERR_STATE; }
    if (q->reduced || q->merged) { mlg_set_error("counters were already combined across ranks; no more reads can be pushed"); return MLG_ERR_STATE; }
    if (q->rk_shared) { mlg_set_error("the read archive was handed to the other ranks; no more reads can be pushed"); return MLG_ERR_STATE; }
    return ensure_device(q->ctx);
}

// total bases of a batch; for offsets given on the host read it there, on the device copy one word back
int batch_bases_host(const uint64_t* off, uint64_t n_reads, uint32_t read_len, unsigned long long* nbases) {
    if (off) {
        if (off[0] != 0) { mlg_set_error("read_off[0] must be 0"); return MLG_ERR_ARG; }
        *nbases = off[n_reads];
    } else {
        if (read_len == 0 && n_reads) { mlg_set_error("read_len must be > 0 when read_off is NULL"); return MLG_ERR_ARG; }
        *nbases = n_reads * (unsigned long long)read_len;
    }
    return MLG_OK;
}

}  // namespace

extern "C" {

MLG_API const char* mlg_last_error(void) { return g_err; }
MLG_API int mlg_version(void) { return 100; }

MLG_API int mlg_ctx_create(int device, mlg_ctx** out) {
    if (!out) { mlg_set_error("null out pointer"); return MLG_ERR_ARG; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        mlg_set_error("no CUDA device available (%s); metalign_b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "0 devices");
        return MLG_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) { mlg_set_error("device %d out of range (0..%d)", device, ndev - 1); return MLG_ERR_ARG; }
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { mlg_set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); return MLG_ERR_CUDA; }
    // Random 32-byte probes: do not let an L2 miss fetch the neighbouring sector as well (the default
    // fetch granularity is 64 bytes, which doubles DRAM traffic for this access pattern).
    {
        size_t gran = 32;
        if (const char* s = getenv("MLG_L2_FETCH")) gran = (size_t)atoi(s);
        if (gran == 32 || gran == 64 || gran == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran);
        cudaGetLastError();
    }
    mlg_ctx* ctx = new mlg_ctx();
    ctx->device = device; ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->s_comp, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking) != cudaSuccess) {
        mlg_set_error("cudaStreamCreate failed"); delete ctx; return MLG_ERR_CUDA;
    }
    *out = ctx;
    return MLG_OK;
}
MLG_API int mlg_ctx_destroy(mlg_ctx* ctx) {
    if (!ctx) return MLG_OK;
    cudaSetDevice(ctx->device);
    if (ctx->s_comp) cudaStreamDestroy(ctx->s_comp);
    if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
    mlg_pool_trim(ctx->device);
    delete ctx;
    return MLG_OK;
}
MLG_API int mlg_ctx_streams(mlg_ctx* ctx, void** compute_stream, void** copy_stream) {
    if (!ctx) { mlg_set_error("null ctx"); return MLG_ERR_ARG; }
    if (compute_stream) *compute_stream = (void*)ctx->s_comp;
    if (copy_stream) *copy_stream = (void*)ctx->s_copy;
    return MLG_OK;
}
MLG_API int mlg_host_alloc(void** out, uint64_t bytes) {
    if (!out) { mlg_set_error("null out pointer"); return MLG_ERR_ARG; }
    CUDA_TRY(cudaMallocHost(out, bytes ? bytes : 1));
    return MLG_OK;
}
MLG_API int mlg_host_free(void* p) { if (p) CUDA_TRY(cudaFreeHost(p)); return MLG_OK; }

// ------------------------------------------------------------------ database
MLG_API int mlg_db_from_keys_device(mlg_ctx* ctx, const uint64_t* d_keys, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks,
                            uint32_t nk, mlg_db** out) {
    if (!ctx || !d_keys || !ks || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(ctx));
    return mlg_db_build_device(ctx, reinterpret_cast<const key128*>(d_keys), G, n, K, ks, nk, out);
}
// chunk-fed build (csrc/db.cu): host keys are uploaded a few thousand genomes at a time, so the device never holds the
// caller's G*n keys beside the structures built from them
MLG_API int mlg_db_builder_create(mlg_ctx* ctx, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks, uint32_t nk, mlg_db_builder** out) {
    if (!ctx || !ks || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(ctx));
    return mlg_db_builder_create_impl(ctx, G, n, K, ks, nk, out);
}
MLG_API int mlg_db_builder_add_device(mlg_db_builder* b, const uint64_t* d_keys, uint32_t first_genome, uint32_t n_genomes) {
    return mlg_db_builder_add_impl(b, reinterpret_cast<const key128*>(d_keys), first_genome, n_genomes);
}
MLG_API int mlg_db_builder_add_fasta(mlg_db_builder* b, const void* bytes, const uint64_t* file_off, uint32_t nfiles, uint64_t prime,
                                     mlg_fasta_stats* stats_or_null) {
    return mlg_db_builder_add_fasta_impl(b, bytes, file_off, nfiles, prime, stats_or_null);
}
MLG_API int mlg_db_builder_finish(mlg_db_builder* b, mlg_db** out) { return mlg_db_builder_finish_impl(b, out); }
MLG_API int mlg_db_builder_destroy(mlg_db_builder* b) { mlg_db_builder_destroy_impl(b); return MLG_OK; }

MLG_API int mlg_db_from_keys(mlg_ctx* ctx, const uint64_t* keys, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks, uint32_t nk,
                     mlg_db** out) {
    if (!ctx || !keys || !ks || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(ctx));
    mlg_db_builder* b = nullptr;
    MLG_TRY(mlg_db_builder_create_impl(ctx, G, n, K, ks, nk, &b));
    const uint32_t step = std::max<uint32_t>(1u, (uint32_t)std::min<unsigned long long>(G, (16ull << 20) / n));   // <= 256 MB of keys per upload
    DevBuf<key128> d;
    int rc = d.alloc((size_t)step * n);
    for (uint32_t g0 = 0; rc == MLG_OK && g0 < G; g0 += step) {
        const uint32_t c = std::min<uint32_t>(step, G - g0);
        // on the stream the build runs on, then joined: the build never sees a copy still in flight
        if (cudaMemcpyAsync(d.p, keys + (size_t)g0 * n * 2, (size_t)c * n * sizeof(key128), cudaMemcpyHostToDevice, ctx->s_comp) != cudaSuccess ||
            cudaStreamSynchronize(ctx->s_comp) != cudaSuccess) { mlg_set_error("upload of the sketch keys failed: %s", cudaGetErrorString(cudaGetLastError())); rc = MLG_ERR_CUDA; break; }
        rc = mlg_db_builder_add_impl(b, d.p, g0, c);
    }
    d.release();
    if (rc == MLG_OK) rc = mlg_db_builder_finish_impl(b, out);
    if (rc != MLG_OK) mlg_db_builder_destroy_impl(b);
    return rc;
}
MLG_API int mlg_db_from_ascii(mlg_ctx* ctx, const char* kmers, uint32_t G, uint32_t n, uint32_t K, const uint32_t* ks, uint32_t nk,
                      mlg_db** out) {
    if (!ctx || !kmers || !ks || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (K < 1 || K > 63) { mlg_set_error("K=%u out of range 1..63", K); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(ctx));
    size_t total = (size_t)G * n;
    DevBuf<unsigned char> t; MLG_TRY(t.alloc(total * K));
    DevBuf<key128> d; MLG_TRY(d.alloc(total));
    CUDA_TRY(cudaMemcpyAsync(t.p, kmers, total * K, cudaMemcpyHostToDevice, ctx->s_comp));
    MLG_TRY(launch_ascii_to_keys(t.p, total, K, d.p, ctx->s_comp));     // joins the stream before it returns
    t.release();
    return mlg_db_build_device(ctx, d.p, G, n, K, ks, nk, out);
}

// .mlgdb files, source form (version 1: the sketch keys; everything else is rebuilt here) or built form (version 2: the
// device structures as mlg_db_save wrote them): csrc/dbfile.cu
MLG_API int mlg_db_load(mlg_ctx* ctx, const char* path, mlg_db** out) {
    if (!ctx || !path || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(ctx));
    return mlg_db_load_file(ctx, path, out);
}
MLG_API int mlg_db_save(const mlg_db* db, const char* path, const char* names, uint64_t names_bytes) {
    if (!db || !path || (names_bytes && !names)) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(db->ctx));
    return mlg_db_save_file(db, path, names, names_bytes);
}
MLG_API int mlg_db_info(const mlg_db* db, uint32_t* G, uint32_t* n, uint32_t* K, uint32_t* nk, uint32_t* ks, uint64_t* n_entries,
                uint64_t* n_distinct) {
    if (!db) { mlg_set_error("null db"); return MLG_ERR_ARG; }
    if (G) *G = db->v.G; if (n) *n = db->v.n; if (K) *K = db->v.K; if (nk) *nk = db->v.nk;
    if (ks) for (int i = 0; i < MLG_MAX_KS; ++i) ks[i] = db->v.ks[i];
    if (n_entries) *n_entries = db->v.np; if (n_distinct) *n_distinct = db->v.nd;
    return MLG_OK;
}
MLG_API int mlg_db_denominators(const mlg_db* db, int count_empty_in_den, int64_t* den) {
    if (!db || !den) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(db->ctx));
    size_t cells = (size_t)db->v.G * db->v.nk;
    std::vector<unsigned char> he(db->v.G);
    CUDA_TRY(cudaMemcpy(den, db->den_real.p, cells * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(he.data(), db->has_empty.p, db->v.G, cudaMemcpyDeviceToHost));
    if (count_empty_in_den)
        for (uint32_t g = 0; g < db->v.G; ++g) if (he[g]) for (uint32_t k = 0; k < db->v.nk; ++k) den[(size_t)g * db->v.nk + k] += 1;
    return MLG_OK;
}
MLG_API int mlg_db_free(mlg_db* db) {
    if (!db) return MLG_OK;
    cudaSetDevice(db->ctx->device);
    delete db;
    return MLG_OK;
}

// ------------------------------------------------------------------ query
MLG_API int mlg_query_begin(mlg_ctx* ctx, mlg_db* db, int ci_min, int gate_mode, int count_empty_in_den, mlg_query** out) {
    if (!ctx || !db || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (ci_min < 1 || ci_min > 255) { mlg_set_error("ci_min=%d out of range 1..255", ci_min); return MLG_ERR_ARG; }
    if (gate_mode != MLG_GATE_EXACT && gate_mode != MLG_GATE_NONE) { mlg_set_error("bad gate_mode %d", gate_mode); return MLG_ERR_ARG; }
    if (db->ctx != ctx) { mlg_set_error("database belongs to another context"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(ctx));
    mlg_query* q = new mlg_query();
    struct Guard { mlg_query* q; ~Guard() { if (q) mlg_query_free(q); } } guard{q};
    q->ctx = ctx; q->db = db; q->ci_min = ci_min; q->ex_clamp = ci_min; q->gate = gate_mode; q->count_empty = count_empty_in_den ? 1 : 0;
    size_t cbytes = round_up((size_t)db->v.nd + 4, 16);
    if (db->clean_cnt8.p && db->clean_cnt8.n >= cbytes) {        // left all-zero by the query before (mlg_query_free)
        std::swap(q->cnt8.p, db->clean_cnt8.p); std::swap(q->cnt8.n, db->clean_cnt8.n);
    } else {
        MLG_TRY(q->cnt8.alloc(cbytes));
        CUDA_TRY(cudaMemsetAsync(q->cnt8.p, 0, cbytes, ctx->s_comp));
    }
    MLG_TRY(q->d_nkmers.alloc(2)); MLG_TRY(q->d_scalar.alloc(4));
    CUDA_TRY(cudaMemsetAsync(q->d_nkmers.p, 0, 16, ctx->s_comp));
    CUDA_TRY(cudaMemsetAsync(q->d_scalar.p, 0, 32, ctx->s_comp));
    CUDA_TRY(cudaEventCreate(&q->ev_q0)); CUDA_TRY(cudaEventCreate(&q->ev_q1));
    if (const char* e = getenv("MLG_CHUNK_MB")) {     // experiment knob: MiB of packed bases per copy chunk
        double mb = atof(e);
        if (mb >= 0.25 && mb <= 4096) q->chunk_words = std::max<unsigned long long>(1024, (unsigned long long)(mb * 65536.0));
    }
    q->st.n_db_entries = db->v.np; q->st.n_db_distinct = db->v.nd;
    q->st.n_buckets = db->v.nbuckets; q->st.bucket_bytes = db->v.layout == 2 ? 32u : db->v.layout == 1 ? 64u : db->v.slots * 4;   // layout 1 fetches bucket PAIRS, layout 2 one sector of the minimizer bitmap
    q->st.filter_words = db->v.nfw; q->st.layout = db->v.layout;
    guard.q = nullptr;
    *out = q;
    return MLG_OK;
}

MLG_API int mlg_query_push_packed_device(mlg_query* q, const uint8_t* d_bases, const uint8_t* d_nmask, const uint64_t* d_off,
                                 uint64_t n_reads, uint32_t read_len) {
    MLG_TRY(check_push(q));
    if (!n_reads) return MLG_OK;
    if (!d_bases) { mlg_set_error("null bases"); return MLG_ERR_ARG; }
    if (((uintptr_t)d_bases & 15) || ((uintptr_t)d_nmask & 15)) { mlg_set_error("device buffers must be 16-byte aligned"); return MLG_ERR_ARG; }
    unsigned long long nbases = 0;
    if (d_off) CUDA_TRY(cudaMemcpy(&nbases, d_off + n_reads, 8, cudaMemcpyDeviceToHost));
    else {
        if (!read_len) { mlg_set_error("read_len must be > 0 when read_off is NULL"); return MLG_ERR_ARG; }
        nbases = n_reads * (unsigned long long)read_len;
    }
    Staging& s = q->stg[q->cur];
    if (s.used) CUDA_TRY(cudaEventSynchronize(s.done));
    MLG_TRY(run_probe(q, s, d_bases, d_nmask, reinterpret_cast<const unsigned long long*>(d_off), n_reads, read_len, nbases, nullptr));
    q->cur ^= 1;
    return MLG_OK;
}

// host packed stream; N given either as a bit mask (nmask) or as sorted (start, length) runs (nruns), or not at all
static int push_packed_host(mlg_query* q, const uint8_t* bases, const uint8_t* nmask, const uint32_t* nruns, uint64_t n_runs,
                            const uint64_t* off, uint64_t n_reads, uint32_t read_len) {
    MLG_TRY(check_push(q));
    if (!n_reads) return MLG_OK;
    if (!bases) { mlg_set_error("null bases"); return MLG_ERR_ARG; }
    unsigned long long nbases = 0;
    MLG_TRY(batch_bases_host(off, n_reads, read_len, &nbases));
    if (!nbases) return MLG_OK;
    if (n_runs && !nruns) { mlg_set_error("null nruns"); return MLG_ERR_ARG; }
    if (n_runs && nbases > 0xFFFFFFFFull) { mlg_set_error("a batch pushed with N runs must hold < 2^32 bases"); return MLG_ERR_ARG; }
    mlg_ctx* ctx = q->ctx;
    CUDA_TRY(cudaStreamSynchronize(ctx->s_copy));          // host buffers of the previous push are free from here on
    Staging& s = q->stg[q->cur];
    if (s.used) CUDA_TRY(cudaEventSynchronize(s.done));   // previous batch that used this set has been consumed
    const unsigned long long nwords = (nbases + 63) / 64;
    const unsigned long long cap_words = round_up(nwords + 2, 2);   // 64-base words
    const bool have_mask = nmask || n_runs;
    MLG_TRY(s.bases.ensure(cap_words * 16));
    if (have_mask) MLG_TRY(s.nmask.ensure(cap_words * 8));
    if (n_runs) {
        MLG_TRY(s.nruns.ensure(2 * n_runs));
        CUDA_TRY(cudaMemsetAsync(s.nmask.p, 0, cap_words * 8, ctx->s_comp));
    }
    if (off) {
        MLG_TRY(s.off.ensure(n_reads + 1));
        CUDA_TRY(cudaMemcpyAsync(s.off.p, off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, ctx->s_copy));
        cudaEvent_t e; CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CUDA_TRY(cudaEventRecord(e, ctx->s_copy));
        CUDA_TRY(cudaStreamWaitEvent(ctx->s_comp, e, 0));
        q->chunk_events.push_back(e);
        q->st.h2d_bytes += (n_reads + 1) * 8;
    }
    // chunked copies: the reads that are complete after chunk c are probed while chunk c+1 is still in flight
    const unsigned long long bases_bytes = (nbases + 3) / 4, nmask_bytes = (nbases + 7) / 8;
    const unsigned long long chunk_words = q->chunk_words;
    std::vector<ReadRange> ready;
    unsigned long long run0 = 0;
    for (unsigned long long w0 = 0; w0 < nwords; w0 += chunk_words) {
        const unsigned long long w1 = std::min(nwords, w0 + chunk_words);
        const unsigned long long b0 = w0 * 16, b1 = std::min(bases_bytes, w1 * 16);
        CUDA_TRY(cudaMemcpyAsync(s.bases.p + b0, bases + b0, b1 - b0, cudaMemcpyHostToDevice, ctx->s_copy));
        q->st.h2d_bytes += b1 - b0;
        if (nmask) {
            const unsigned long long m0 = w0 * 8, m1 = std::min(nmask_bytes, w1 * 8);
            CUDA_TRY(cudaMemcpyAsync(s.nmask.p + m0, nmask + m0, m1 - m0, cudaMemcpyHostToDevice, ctx->s_copy));
            q->st.h2d_bytes += m1 - m0;
        }
        // N runs that START inside this chunk travel with it (a run may extend past the chunk: harmless, the mask
        // of the whole batch was cleared up front and later reads are probed later)
        unsigned long long run1 = run0;
        if (n_runs) {
            if (w1 == nwords) run1 = n_runs;
            else {
                unsigned long long lo = run0, hi = n_runs; const unsigned long long lim = w1 * 64;
                while (lo < hi) { unsigned long long mid = (lo + hi) / 2; if (nruns[2 * mid] < lim) lo = mid + 1; else hi = mid; }
                run1 = lo;
            }
            if (run1 > run0) {
                CUDA_TRY(cudaMemcpyAsync(s.nruns.p + 2 * run0, nruns + 2 * run0, (run1 - run0) * 8, cudaMemcpyHostToDevice, ctx->s_copy));
                q->st.h2d_bytes += (run1 - run0) * 8;
            }
        }
        cudaEvent_t e; CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CUDA_TRY(cudaEventRecord(e, ctx->s_copy));
        q->chunk_events.push_back(e);
        // reads whose last base has been copied (base index < 64 * w1)
        unsigned long long r_end;
        if (w1 == nwords) r_end = n_reads;
        else if (off) r_end = (unsigned long long)(std::upper_bound(off, off + n_reads + 1, (uint64_t)(w1 * 64)) - off) - 1;
        else r_end = (w1 * 64) / read_len;
        ReadRange rr; rr.r_end = r_end; rr.ready = e; rr.run0 = run0; rr.run1 = run1;
        ready.push_back(rr);
        run0 = run1;
    }
    MLG_TRY(run_probe(q, s, s.bases.p, have_mask ? s.nmask.p : nullptr, off ? s.off.p : nullptr, n_reads, read_len, nbases, &ready));
    q->cur ^= 1;
    return MLG_OK;
}
MLG_API int mlg_query_push_packed(mlg_query* q, const uint8_t* bases, const uint8_t* nmask, const uint64_t* off, uint64_t n_reads,
                          uint32_t read_len) {
    return push_packed_host(q, bases, nmask, nullptr, 0, off, n_reads, read_len);
}
MLG_API int mlg_query_push_packed_nruns(mlg_query* q, const uint8_t* bases, const uint32_t* nruns, uint64_t n_runs,
                                        const uint64_t* off, uint64_t n_reads, uint32_t read_len) {
    return push_packed_host(q, bases, nullptr, nruns, n_runs, off, n_reads, read_len);
}

MLG_API int mlg_query_push_ascii(mlg_query* q, const char* text, const uint64_t* off, uint64_t n_reads) {
    MLG_TRY(check_push(q));
    if (!n_reads) return MLG_OK;
    if (!text || !off) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (off[0] != 0) { mlg_set_error("read_off[0] must be 0"); return MLG_ERR_ARG; }
    const unsigned long long nbases = off[n_reads];
    if (!nbases) return MLG_OK;
    mlg_ctx* ctx = q->ctx;
    CUDA_TRY(cudaStreamSynchronize(ctx->s_copy));
    Staging& s = q->stg[q->cur];
    if (s.used) CUDA_TRY(cudaEventSynchronize(s.done));
    const unsigned long long nwords = (nbases + 63) / 64;
    const unsigned long long cap_words = round_up(nwords + 2, 2);   // 64-base words
    MLG_TRY(s.bases.ensure(cap_words * 16)); MLG_TRY(s.nmask.ensure(cap_words * 8));
    MLG_TRY(s.text.ensure(nbases)); MLG_TRY(s.off.ensure(n_reads + 1));
    CUDA_TRY(cudaMemcpyAsync(s.text.p, text, nbases, cudaMemcpyHostToDevice, ctx->s_copy));
    CUDA_TRY(cudaMemcpyAsync(s.off.p, off, (n_reads + 1) * 8, cudaMemcpyHostToDevice, ctx->s_copy));
    q->st.h2d_bytes += nbases + (n_reads + 1) * 8;
    cudaEvent_t e; CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(e, ctx->s_copy));
    CUDA_TRY(cudaStreamWaitEvent(ctx->s_comp, e, 0));
    q->chunk_events.push_back(e);
    MLG_TRY(launch_pack_ascii(s.text.p, nbases, s.bases.p, s.nmask.p, ctx->s_comp));
    q->st.gpu_launches += 1;
    MLG_TRY(run_probe(q, s, s.bases.p, s.nmask.p, s.off.p, n_reads, 0, nbases, nullptr));
    q->cur ^= 1;
    return MLG_OK;
}

MLG_API int mlg_query_sync(mlg_query* q) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(q->ctx));
    CUDA_TRY(cudaStreamSynchronize(q->ctx->s_copy));
    CUDA_TRY(cudaStreamSynchronize(q->ctx->s_comp));
    return MLG_OK;
}

MLG_API int mlg_query_counts_export(mlg_query* q, uint8_t** d_counts, uint64_t* n_counts) {
    if (!q || !d_counts || !n_counts) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (q->finished) { mlg_set_error("query already finished"); return MLG_ERR_STATE; }
    MLG_TRY(ensure_device(q->ctx));
    q->exchanged = true;
    if (q->touched.p) {     // nothing pushed: every counter is still zero
        MLG_TRY(launch_clamp_counts(q->cnt8.p, q->touched.p, q->d_scalar.p + 1, (uint32_t)q->ex_clamp, q->ctx->s_comp));
        q->st.gpu_launches += 1;
    }
    MLG_TRY(mlg_query_sync(q));
    *d_counts = q->cnt8.p; *n_counts = q->db->v.nd;
    return MLG_OK;
}
MLG_API int mlg_query_counts_export_sparse(mlg_query* q, uint64_t** d_entries, uint64_t* n_entries) {
    if (!q || !d_entries || !n_entries) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (q->finished) { mlg_set_error("query already finished"); return MLG_ERR_STATE; }
    if (q->merged || q->reduced) { mlg_set_error("counters were already combined across ranks"); return MLG_ERR_STATE; }
    MLG_TRY(ensure_device(q->ctx));
    q->exchanged = true;
    *d_entries = nullptr; *n_entries = 0;
    if (!q->touched.p) return MLG_OK;                      // nothing pushed: no non-zero counter
    cudaStream_t st = q->ctx->s_comp;
    CUDA_TRY(cudaStreamSynchronize(q->ctx->s_copy));
    unsigned long long nt = 0;
    CUDA_TRY(cudaMemcpyAsync(&nt, q->d_scalar.p + 1, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));                   // joins the probe kernels
    MLG_TRY(q->sparse.ensure(nt));
    MLG_TRY(launch_pack_touched(q->cnt8.p, q->touched.p, q->d_scalar.p + 1, (uint32_t)q->ex_clamp, q->sparse.p, st));
    q->st.gpu_launches += 1;
    CUDA_TRY(cudaStreamSynchronize(st));
    *d_entries = reinterpret_cast<uint64_t*>(q->sparse.p); *n_entries = nt;
    return MLG_OK;
}
MLG_API int mlg_query_counts_merge_sparse(mlg_query* q, const uint64_t* d_entries, uint64_t n_entries) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (q->finished) { mlg_set_error("query already finished"); return MLG_ERR_STATE; }
    if (q->reduced) { mlg_set_error("counters were already reduced densely"); return MLG_ERR_STATE; }
    MLG_TRY(ensure_device(q->ctx));
    q->merged = true; q->exchanged = true;
    if (!n_entries) return MLG_OK;
    if (!d_entries) { mlg_set_error("null entries"); return MLG_ERR_ARG; }
    if (!q->present.p) { MLG_TRY(q->present.alloc((size_t)q->db->v.nd + 1)); MLG_TRY(q->touched.alloc((size_t)q->db->v.nd + 1)); }
    MLG_TRY(launch_merge_sparse(q->cnt8.p, reinterpret_cast<const unsigned long long*>(d_entries), n_entries, q->db->v.nd,
                                (uint32_t)q->ci_min, q->present.p, q->touched.p, q->d_scalar.p, q->ctx->s_comp));
    q->st.gpu_launches += 1;
    return MLG_OK;
}
MLG_API int mlg_query_counts_import(mlg_query* q) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    q->reduced = true; q->exchanged = true;
    return MLG_OK;
}

MLG_API int mlg_query_set_exchange_clamp(mlg_query* q, int clamp) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (q->exchanged || q->finished) { mlg_set_error("the exchange clamp must be set before any exchange"); return MLG_ERR_STATE; }
    if (clamp < q->ci_min || clamp > 255) { mlg_set_error("exchange clamp %d out of range ci_min (%d)..255", clamp, q->ci_min); return MLG_ERR_ARG; }
    q->ex_clamp = clamp;
    return MLG_OK;
}

// ------------------------------------------------------------------ exchange (multi-GPU, no host round trip)
MLG_API int mlg_exchange_create(mlg_ctx* ctx, uint32_t world, uint32_t rank, uint64_t cap_entries, mlg_exchange** out) {
    if (!ctx || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (world < 1 || world > MLG_MAX_RANKS || rank >= world) { mlg_set_error("world=%u rank=%u out of range (1..%d ranks)", world, rank, MLG_MAX_RANKS); return MLG_ERR_ARG; }
    if (cap_entries < 1 || cap_entries > (1ull << 32)) { mlg_set_error("cap_entries out of range"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(ctx));
    mlg_exchange* ex = new mlg_exchange();
    struct Guard { mlg_exchange* e; ~Guard() { if (e) mlg_exchange_destroy(e); } } guard{ex};
    ex->ctx = ctx; ex->world = world; ex->rank = rank; ex->cap = cap_entries;
    ex->block_words = round_up(cap_entries + 2, 2);
    MLG_TRY(ex->send.alloc(ex->block_words)); MLG_TRY(ex->recv.alloc(ex->block_words * world)); MLG_TRY(ex->status.alloc(4));
    const size_t mb = (size_t)world * 2 * ex->block_words * 8;
    CUDA_TRY(cudaMalloc(&ex->mailbox, mb));
    CUDA_TRY(cudaMemsetAsync(ex->mailbox, 0, mb, ctx->s_comp));
    CUDA_TRY(cudaMemsetAsync(ex->send.p, 0, ex->block_words * 8, ctx->s_comp));
    CUDA_TRY(cudaMemsetAsync(ex->recv.p, 0, ex->block_words * world * 8, ctx->s_comp));
    CUDA_TRY(cudaMemsetAsync(ex->status.p, 0, 32, ctx->s_comp));
    CUDA_TRY(cudaStreamSynchronize(ctx->s_comp));
    guard.e = nullptr;
    *out = ex;
    return MLG_OK;
}
MLG_API int mlg_exchange_destroy(mlg_exchange* ex) {
    if (!ex) return MLG_OK;
    cudaSetDevice(ex->ctx->device);
    cudaStreamSynchronize(ex->ctx->s_comp);
    for (uint32_t w = 0; w < ex->world; ++w)
        if (w != ex->rank && ex->peer_mailbox[w]) cudaIpcCloseMemHandle(ex->peer_mailbox[w]);
    if (ex->mailbox) cudaFree(ex->mailbox);
    delete ex;
    return MLG_OK;
}
MLG_API int mlg_exchange_buffers(mlg_exchange* ex, uint64_t** d_send, uint64_t** d_recv, uint64_t* block_words) {
    if (!ex) { mlg_set_error("null exchange"); return MLG_ERR_ARG; }
    if (d_send) *d_send = reinterpret_cast<uint64_t*>(ex->send.p);
    if (d_recv) *d_recv = reinterpret_cast<uint64_t*>(ex->recv.p);
    if (block_words) *block_words = ex->block_words;
    return MLG_OK;
}
MLG_API int mlg_exchange_local_handle(mlg_exchange* ex, void* handle64) {
    if (!ex || !handle64) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI passes IPC handles as 64 opaque bytes");
    MLG_TRY(ensure_device(ex->ctx));
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, ex->mailbox));
    memcpy(handle64, &h, 64);
    return MLG_OK;
}
MLG_API int mlg_exchange_connect(mlg_exchange* ex, const void* handles) {
    if (!ex || !handles) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (ex->connected) return MLG_OK;
    MLG_TRY(ensure_device(ex->ctx));
    for (uint32_t w = 0; w < ex->world; ++w) {
        if (w == ex->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + 64 * (size_t)w, 64);
        void* p = nullptr;
        CUDA_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        ex->peer_mailbox[w] = (unsigned long long*)p;
    }
    ex->connected = true;
    return MLG_OK;
}
static int check_exchange(mlg_query* q, mlg_exchange* ex) {
    if (!q || !ex) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (q->finished) { mlg_set_error("query already finished"); return MLG_ERR_STATE; }
    if (q->reduced) { mlg_set_error("counters were already reduced densely"); return MLG_ERR_STATE; }
    if (ex->ctx != q->ctx) { mlg_set_error("exchange belongs to another context"); return MLG_ERR_ARG; }
    if ((unsigned long long)q->ex_clamp * ex->world > 255ull) { mlg_set_error("exchange clamp (%d) * world must fit the 8-bit counters", q->ex_clamp); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(q->ctx));
    if (!q->present.p) { MLG_TRY(q->present.alloc((size_t)q->db->v.nd + 1)); MLG_TRY(q->touched.alloc((size_t)q->db->v.nd + 1)); }
    q->exchanged = true;
    return MLG_OK;
}
// the probe kernels run on the compute stream, the copies feeding them on the copy stream, and every copy chunk is
// already awaited by the probe launch that consumes it: work queued on the compute stream after the last push sees
// every counter.  No host synchronisation here.
MLG_API int mlg_query_exchange_pack(mlg_query* q, mlg_exchange* ex) {
    MLG_TRY(check_exchange(q, ex));
    cudaStream_t st = q->ctx->s_comp;
    CUDA_TRY(cudaMemsetAsync(ex->status.p, 0, 16, st));
    MLG_TRY(launch_pack_exchange(q->cnt8.p, q->touched.p, q->d_scalar.p + 1, (uint32_t)q->ex_clamp, ex->send.p, ex->cap, ex->status.p + 3,
                                 st));
    q->st.gpu_launches += 1;
    return MLG_OK;
}
MLG_API int mlg_query_exchange_merge(mlg_query* q, mlg_exchange* ex) {
    MLG_TRY(check_exchange(q, ex));
    MLG_TRY(launch_merge_exchange(q->cnt8.p, ex->recv.p, ex->block_words, ex->world, ex->rank, ex->cap, q->db->v.nd, (uint32_t)q->ci_min,
                                  q->present.p, q->touched.p, q->d_scalar.p, ex->status.p, 0, 0, q->ctx->s_comp));
    q->st.gpu_launches += 1;
    q->merged = true; q->ex_pending = ex;
    return MLG_OK;
}
MLG_API int mlg_query_exchange_p2p(mlg_query* q, mlg_exchange* ex) {
    MLG_TRY(check_exchange(q, ex));
    if (ex->world > 1 && !ex->connected) { mlg_set_error("mlg_exchange_connect has not been called"); return MLG_ERR_STATE; }
    cudaStream_t st = q->ctx->s_comp;
    const unsigned long long epoch = ++ex->epoch;
    if (epoch >= (1ull << 23)) { mlg_set_error("exchange epoch counter exhausted; create a new exchange"); return MLG_ERR_STATE; }
    const unsigned long long parity = epoch & 1ull;
    unsigned long long* boxes[MLG_MAX_RANKS];
    uint32_t np = 0;
    for (uint32_t w = 0; w < ex->world; ++w)
        if (w != ex->rank) boxes[np++] = ex->peer_mailbox[w] + ((unsigned long long)ex->rank * 2ull + parity) * ex->block_words;
    CUDA_TRY(cudaMemsetAsync(ex->status.p, 0, 16, st));
    MLG_TRY(launch_push_peers(q->cnt8.p, q->touched.p, q->d_scalar.p + 1, (uint32_t)q->ex_clamp, boxes, np, ex->cap, epoch,
                              reinterpret_cast<unsigned int*>(ex->status.p + 2), ex->status.p + 3, st));
    MLG_TRY(launch_merge_exchange(q->cnt8.p, ex->mailbox + parity * ex->block_words, 2ull * ex->block_words, ex->world, ex->rank, ex->cap,
                                  q->db->v.nd, (uint32_t)q->ci_min, q->present.p, q->touched.p, q->d_scalar.p, ex->status.p, epoch,
                                  ex->timeout_ns, st));
    q->st.gpu_launches += 2;
    q->merged = true; q->ex_pending = ex;
    return MLG_OK;
}
// dense form without the host join of mlg_query_counts_export: the counters are clamped on the compute stream and the
// caller's all-reduce must be ordered after it on that stream
MLG_API int mlg_query_exchange_dense(mlg_query* q, uint8_t** d_counts, uint64_t* n_counts) {
    if (!q || !d_counts || !n_counts) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (q->finished) { mlg_set_error("query already finished"); return MLG_ERR_STATE; }
    if (q->merged) { mlg_set_error("counters were already merged sparsely"); return MLG_ERR_STATE; }
    MLG_TRY(ensure_device(q->ctx));
    if (q->touched.p) {
        MLG_TRY(launch_clamp_counts(q->cnt8.p, q->touched.p, q->d_scalar.p + 1, (uint32_t)q->ex_clamp, q->ctx->s_comp));
        q->st.gpu_launches += 1;
    }
    *d_counts = q->cnt8.p; *n_counts = q->db->v.nd;
    q->reduced = true; q->exchanged = true;
    return MLG_OK;
}

// from the present k-mers to the hit bitmap and the per-genome counts (both zeroed by the caller)
static int replay_hits(mlg_query* q, uint32_t* hitbits, unsigned long long words_per_k, unsigned long long* d_num) {
    mlg_db* db = q->db; const DbView& v = db->v;
    cudaStream_t st = q->ctx->s_comp;
    if (db->hoff.p) {
        // replay the precomputed hit records; k-mers without one (only a database that kept P has any) are listed and
        // expanded on the fly
        if (v.P_key && !q->fallback.p) MLG_TRY(q->fallback.alloc((size_t)v.nd + 1));
        MLG_TRY(launch_apply_hits(v, q->present.p, q->d_scalar.p, q->gate == MLG_GATE_NONE, hitbits, words_per_k, d_num,
                                  db->hoff.p, db->hbase.p, db->hits.p, q->fallback.p, q->d_scalar.p + 2, st));
        q->st.gpu_launches += 1;
    } else {
        MLG_TRY(launch_expand_hits(v, q->present.p, q->d_scalar.p, q->gate == MLG_GATE_NONE, hitbits, words_per_k, d_num, st));
    }
    return MLG_OK;
}

// the finish stage, shared by the dense and the sparse form of the result
struct SparseOut { uint32_t* genomes; int64_t* num; int64_t* den; double* ci; uint64_t cap; uint64_t* n_rows; };
static int finish_impl(mlg_query* q, int64_t* num, int64_t* den, double* ci, const SparseOut* sp, uint64_t* n_intersect) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (q->finished) { mlg_set_error("query already finished"); return MLG_ERR_STATE; }
    mlg_ctx* ctx = q->ctx; mlg_db* db = q->db; const DbView& v = db->v;
    MLG_TRY(ensure_device(ctx));
    cudaStream_t st = ctx->s_comp;
    CUDA_TRY(cudaStreamSynchronize(ctx->s_copy));
    if (!q->present.p) { MLG_TRY(q->present.alloc((size_t)v.nd + 1)); MLG_TRY(q->touched.alloc((size_t)v.nd + 1)); }   // nothing was pushed
    CUDA_TRY(cudaEventRecord(q->ev_q0, st));
    // I = database k-mers seen >= ci_min times.  Single GPU: the probe kernel appended each one when its counter
    // reached ci_min.  After a cross-rank reduction the list is rebuilt from the summed counters.
    if (q->reduced) {
        MLG_TRY(launch_compact_present(q->cnt8.p, v.nd, (uint32_t)q->ci_min, q->present.p, q->d_scalar.p, st));
        q->st.gpu_launches += 1;
    }
    // hit bitmap: nk planes of G*n bits; the kernel that sets a bit first also counts it
    const unsigned long long total = (unsigned long long)v.G * v.n;
    const unsigned long long words_per_k = (total + 31) / 32;
    const size_t cells = (size_t)v.G * v.nk;
    DevBuf<uint32_t>& hitbits = q->hitbits;
    DevBuf<unsigned long long>& d_num = q->d_num;
    if (!hitbits.p) {                                  // nothing was pushed: the tables were not set up beside a probe
        MLG_TRY(hitbits.alloc(words_per_k * v.nk)); MLG_TRY(d_num.alloc(cells));
        CUDA_TRY(cudaMemsetAsync(hitbits.p, 0, words_per_k * v.nk * 4, st));
        CUDA_TRY(cudaMemsetAsync(d_num.p, 0, cells * 8, st));
    }
    MLG_TRY(replay_hits(q, hitbits.p, words_per_k, d_num.p));
    q->st.gpu_launches += 2;
    DevBuf<long long> o_num, o_den; DevBuf<double> o_ci; DevBuf<uint32_t> o_g;
    unsigned long long nrows = 0;
    const uint64_t first = sp ? std::min<uint64_t>(sp->cap, 4096) : 0;     // rows copied back before their number is known
    if (!sp) {
        MLG_TRY(o_num.alloc(cells)); MLG_TRY(o_den.alloc(cells)); MLG_TRY(o_ci.alloc(cells));
        MLG_TRY(launch_finalize(d_num.p, db->den_real.p, db->has_empty.p, v.G, v.nk, q->count_empty, o_num.p, o_den.p, o_ci.p, st));
        CUDA_TRY(cudaEventRecord(q->ev_q1, st));
        if (num) { CUDA_TRY(cudaMemcpyAsync(num, o_num.p, cells * 8, cudaMemcpyDeviceToHost, st)); q->st.d2h_bytes += cells * 8; }
        if (den) { CUDA_TRY(cudaMemcpyAsync(den, o_den.p, cells * 8, cudaMemcpyDeviceToHost, st)); q->st.d2h_bytes += cells * 8; }
        if (ci) { CUDA_TRY(cudaMemcpyAsync(ci, o_ci.p, cells * 8, cudaMemcpyDeviceToHost, st)); q->st.d2h_bytes += cells * 8; }
    } else {
        const size_t rc = (size_t)std::max<uint64_t>(sp->cap, 1);
        MLG_TRY(o_g.alloc(rc)); MLG_TRY(o_num.alloc(rc * v.nk)); MLG_TRY(o_den.alloc(rc * v.nk)); MLG_TRY(o_ci.alloc(rc * v.nk));
        if (!q->d_rows.p) MLG_TRY(q->d_rows.alloc(1));
        MLG_TRY(launch_finalize_sparse(d_num.p, db->den_real.p, db->has_empty.p, v.G, v.nk, q->count_empty, o_g.p, o_num.p, o_den.p,
                                       o_ci.p, sp->cap, q->d_rows.p, st));
        CUDA_TRY(cudaEventRecord(q->ev_q1, st));
        CUDA_TRY(cudaMemcpyAsync(&nrows, q->d_rows.p, 8, cudaMemcpyDeviceToHost, st));
        if (first) {
            if (sp->genomes) CUDA_TRY(cudaMemcpyAsync(sp->genomes, o_g.p, first * 4, cudaMemcpyDeviceToHost, st));
            if (sp->num) CUDA_TRY(cudaMemcpyAsync(sp->num, o_num.p, first * v.nk * 8, cudaMemcpyDeviceToHost, st));
            if (sp->den) CUDA_TRY(cudaMemcpyAsync(sp->den, o_den.p, first * v.nk * 8, cudaMemcpyDeviceToHost, st));
            if (sp->ci) CUDA_TRY(cudaMemcpyAsync(sp->ci, o_ci.p, first * v.nk * 8, cudaMemcpyDeviceToHost, st));
        }
    }
    unsigned long long nk_host2[2] = {0, 0}, ni = 0;
    unsigned long long& nk_host = nk_host2[0];
    CUDA_TRY(cudaMemcpyAsync(nk_host2, q->d_nkmers.p, 16, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&ni, q->d_scalar.p, 8, cudaMemcpyDeviceToHost, st));
    unsigned long long xstat[2] = {0, 0};
    if (q->ex_pending) CUDA_TRY(cudaMemcpyAsync(xstat, q->ex_pending->status.p, 16, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    if (xstat[1]) { mlg_set_error("exchange: a peer's block did not arrive within the time limit"); return MLG_ERR_STATE; }
    if (xstat[0]) {
        // some rank had more non-zero counters than a block holds: nothing was merged (on any rank), so the exchange can
        // simply be repeated with larger blocks and finish called again
        q->merged = false; q->ex_pending = nullptr;
        // the tables of this attempt go back to zero: finish will be called again after the repeated exchange
        CUDA_TRY(cudaMemsetAsync(hitbits.p, 0, words_per_k * v.nk * 4, st));
        CUDA_TRY(cudaMemsetAsync(d_num.p, 0, cells * 8, st));
        mlg_set_error("exchange blocks too small: %llu entries needed", xstat[0]);
        return MLG_ERR_RETRY;
    }
    if (sp) {
        if (sp->n_rows) *sp->n_rows = nrows;
        if (nrows > sp->cap) { mlg_set_error("result has %llu rows, the buffers hold %llu", nrows, (unsigned long long)sp->cap); return MLG_ERR_ARG; }
        if (nrows > first) {                          // (rare) more rows than were copied ahead
            const size_t m = (size_t)(nrows - first);
            if (sp->genomes) CUDA_TRY(cudaMemcpyAsync(sp->genomes + first, o_g.p + first, m * 4, cudaMemcpyDeviceToHost, st));
            if (sp->num) CUDA_TRY(cudaMemcpyAsync(sp->num + first * v.nk, o_num.p + first * v.nk, m * v.nk * 8, cudaMemcpyDeviceToHost, st));
            if (sp->den) CUDA_TRY(cudaMemcpyAsync(sp->den + first * v.nk, o_den.p + first * v.nk, m * v.nk * 8, cudaMemcpyDeviceToHost, st));
            if (sp->ci) CUDA_TRY(cudaMemcpyAsync(sp->ci + first * v.nk, o_ci.p + first * v.nk, m * v.nk * 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        const uint64_t copied = std::max<uint64_t>(first, nrows);
        q->st.d2h_bytes += 8 + copied * ((sp->genomes ? 4 : 0) + ((sp->num ? 8 : 0) + (sp->den ? 8 : 0) + (sp->ci ? 8 : 0)) * v.nk);
    }
    q->n_present = (uint32_t)ni;
    q->st.n_kmers = nk_host; q->st.n_intersect = ni;
    q->st.n_bucket_fetches = v.layout >= 1 ? nk_host2[1] : nk_host;
    q->st.d2h_bytes += 16;
    // timings
    float ms = 0; double probe_ms = 0;
    for (auto& pe : q->probe_events) { if (cudaEventElapsedTime(&ms, pe.first, pe.second) == cudaSuccess) probe_ms += ms; }
    q->st.ms_probe = probe_ms;
    if (cudaEventElapsedTime(&ms, q->ev_q0, q->ev_q1) == cudaSuccess) q->st.ms_query = ms;
    if (n_intersect) *n_intersect = ni;
    q->finished = true;
    return MLG_OK;
}
MLG_API int mlg_query_finish(mlg_query* q, int64_t* num, int64_t* den, double* ci, uint64_t* n_intersect) {
    return finish_impl(q, num, den, ci, nullptr, n_intersect);
}
MLG_API int mlg_query_finish_sparse(mlg_query* q, uint32_t* genomes, int64_t* num, int64_t* den, double* ci, uint64_t cap_rows,
                                    uint64_t* n_rows, uint64_t* n_intersect) {
    if (!n_rows) { mlg_set_error("null n_rows"); return MLG_ERR_ARG; }
    SparseOut sp{genomes, num, den, ci, cap_rows, n_rows};
    return finish_impl(q, nullptr, nullptr, nullptr, &sp, n_intersect);
}

// which (genome, k-prefix) classes of the given genomes the query hit: the raw material of CMash's post-processing when
// --sensitive is absent (metalign_b200/cmash_tail.py: refilter_unique).  The bitmap is rebuilt from the present k-mers (the
// finish stage does not keep it: 0.1 GB per query for something Metalign never asks for).
MLG_API int mlg_query_hit_flags(mlg_query* q, const uint32_t* genomes, uint32_t m, uint8_t* out) {
    if (!q || (m && (!genomes || !out))) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (!q->finished) { mlg_set_error("call mlg_query_finish first"); return MLG_ERR_STATE; }
    if (!m) return MLG_OK;
    mlg_ctx* ctx = q->ctx; const DbView& v = q->db->v;
    MLG_TRY(ensure_device(ctx));
    for (uint32_t i = 0; i < m; ++i) if (genomes[i] >= v.G) { mlg_set_error("genome %u out of range (G = %u)", genomes[i], v.G); return MLG_ERR_ARG; }
    cudaStream_t st = ctx->s_comp;
    const unsigned long long total = (unsigned long long)v.G * v.n, words_per_k = (total + 31) / 32;
    const size_t cells = (size_t)v.G * v.nk, flags = (size_t)m * v.nk * v.n;
    DevBuf<uint32_t> hitbits; MLG_TRY(hitbits.alloc(words_per_k * v.nk));
    DevBuf<unsigned long long> d_num; MLG_TRY(d_num.alloc(cells));
    DevBuf<uint32_t> d_g; MLG_TRY(d_g.alloc(m));
    DevBuf<unsigned char> d_out; MLG_TRY(d_out.alloc(flags));
    CUDA_TRY(cudaMemsetAsync(hitbits.p, 0, words_per_k * v.nk * 4, st));
    CUDA_TRY(cudaMemsetAsync(d_num.p, 0, cells * 8, st));
    CUDA_TRY(cudaMemcpyAsync(d_g.p, genomes, (size_t)m * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(q->d_scalar.p + 2, 0, 8, st));          // the fallback list's cursor
    MLG_TRY(replay_hits(q, hitbits.p, words_per_k, d_num.p));
    MLG_TRY(launch_gather_hit_flags(hitbits.p, words_per_k, d_g.p, m, v.n, v.nk, d_out.p, st));
    CUDA_TRY(cudaMemcpyAsync(out, d_out.p, flags, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}

MLG_API int mlg_query_intersection(mlg_query* q, uint64_t* keys_out, uint64_t cap, uint64_t* n) {
    if (!q || !n) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (!q->finished) { mlg_set_error("call mlg_query_finish first"); return MLG_ERR_STATE; }
    MLG_TRY(ensure_device(q->ctx));
    *n = q->n_present;
    if (!keys_out || !cap || !q->n_present) return MLG_OK;
    DevBuf<key128> d; MLG_TRY(d.alloc(q->n_present));
    MLG_TRY(launch_gather_keys(q->db->D_key.p, q->present.p, q->n_present, d.p, q->ctx->s_comp));
    std::vector<key128> h(q->n_present);
    CUDA_TRY(cudaMemcpyAsync(h.data(), d.p, (size_t)q->n_present * sizeof(key128), cudaMemcpyDeviceToHost, q->ctx->s_comp));
    CUDA_TRY(cudaStreamSynchronize(q->ctx->s_comp));
    std::sort(h.begin(), h.end(), [](const key128& a, const key128& b) { return key_lt(a, b); });
    uint64_t m = std::min<uint64_t>(cap, q->n_present);
    for (uint64_t i = 0; i < m; ++i) { keys_out[2 * i] = h[i].hi; keys_out[2 * i + 1] = h[i].lo; }
    return MLG_OK;
}

// `kmc_dump <temp>/60mers_intersection <temp>/60mers_intersection_dump` and the FASTA rewrite after it
// (scripts/select_db.py:58-65), straight from the query's tables
MLG_API int mlg_query_dump_intersection(mlg_query* q, const char* dump_path, const char* fasta_path_or_null, uint32_t counter_max) {
    if (!q || !dump_path) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (!q->finished) { mlg_set_error("call mlg_query_finish first"); return MLG_ERR_STATE; }
    if (counter_max == 0 || counter_max > 255) { mlg_set_error("counter_max must be 1..255"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(q->ctx));
    const uint32_t n = q->n_present, K = q->db->v.K;
    struct Rec { key128 k; unsigned char c; };
    std::vector<Rec> recs(n);
    if (n) {
        DevBuf<key128> d; MLG_TRY(d.alloc(n));
        DevBuf<unsigned char> dc; MLG_TRY(dc.alloc(n));
        MLG_TRY(launch_gather_keys(q->db->D_key.p, q->present.p, n, d.p, q->ctx->s_comp));
        MLG_TRY(launch_gather_counts(q->cnt8.p, q->db->D_mult.p, q->present.p, n, counter_max, dc.p, q->ctx->s_comp));
        std::vector<key128> hk(n); std::vector<unsigned char> hc(n);
        CUDA_TRY(cudaMemcpyAsync(hk.data(), d.p, (size_t)n * sizeof(key128), cudaMemcpyDeviceToHost, q->ctx->s_comp));
        CUDA_TRY(cudaMemcpyAsync(hc.data(), dc.p, n, cudaMemcpyDeviceToHost, q->ctx->s_comp));
        CUDA_TRY(cudaStreamSynchronize(q->ctx->s_comp));
        for (uint32_t i = 0; i < n; ++i) recs[i] = Rec{hk[i], hc[i]};
        std::sort(recs.begin(), recs.end(), [](const Rec& a, const Rec& b) { return key_lt(a.k, b.k); });
    }
    FILE* fd = fopen(dump_path, "w");
    if (!fd) { mlg_set_error("cannot create %s", dump_path); return MLG_ERR_IO; }
    FILE* ff = fasta_path_or_null ? fopen(fasta_path_or_null, "w") : nullptr;
    if (fasta_path_or_null && !ff) { fclose(fd); mlg_set_error("cannot create %s", fasta_path_or_null); return MLG_ERR_IO; }
    std::vector<char> line(K + 1);
    bool ok = true;
    for (uint32_t i = 0; i < n && ok; ++i) {
        key128 k = recs[i].k;
        for (uint32_t j = 0; j < K; ++j) { line[K - 1 - j] = "ACGT"[k.lo & 3ull]; k = key_shr(k, 2); }
        line[K] = 0;
        ok = fprintf(fd, "%s\t%u\n", line.data(), (unsigned)recs[i].c) > 0 && (!ff || fprintf(ff, ">seq\n%s\n", line.data()) > 0);
    }
    ok = (fclose(fd) == 0) && ok;
    if (ff) ok = (fclose(ff) == 0) && ok;
    if (!ok) { mlg_set_error("%s: short write", dump_path); return MLG_ERR_IO; }
    return MLG_OK;
}

// ------------------------------------------------------------------ read k-mer table (csrc/readkmers.cu)
MLG_API int mlg_query_enable_read_kmers(mlg_query* q, uint64_t max_table_bytes) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (q->rk) return MLG_OK;
    if (q->rkp) { mlg_set_error("read k-mer passes are already enabled on this query"); return MLG_ERR_STATE; }
    if (q->finished || q->exchanged || q->stg[0].used || q->stg[1].used) {
        mlg_set_error("the read k-mer table must be enabled before the first push"); return MLG_ERR_STATE;
    }
    MLG_TRY(ensure_device(q->ctx));
    return rk_create(q->ctx, q->db->v.K, max_table_bytes, &q->rk);
}
MLG_API int mlg_query_enable_read_kmer_passes(mlg_query* q, uint64_t max_bytes) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (q->rkp) return MLG_OK;
    if (q->rk) { mlg_set_error("the read k-mer table is already enabled on this query"); return MLG_ERR_STATE; }
    if (q->finished || q->exchanged || q->stg[0].used || q->stg[1].used) {
        mlg_set_error("read k-mer passes must be enabled before the first push"); return MLG_ERR_STATE;
    }
    MLG_TRY(ensure_device(q->ctx));
    return rkp_create(q->ctx, q->db->v.K, max_bytes, &q->rkp);
}
static int check_read_kmers(mlg_query* q, uint32_t min_count, uint32_t counter_max) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (!q->rk && !q->rkp) { mlg_set_error("the read k-mer table is off (mlg_query_enable_read_kmers)"); return MLG_ERR_STATE; }
    if (q->exchanged && !q->rk_shared) { mlg_set_error("the read k-mer table is per rank and the counters went through an exchange"); return MLG_ERR_STATE; }
    if (q->rk_shared && rkp_peers_missing(q->rkp)) {
        mlg_set_error("%u peer read archives are still to be added (mlg_query_read_kmer_add_archive)", rkp_peers_missing(q->rkp)); return MLG_ERR_STATE;
    }
    if (min_count < 1 || min_count > 255 || counter_max < 1 || counter_max > 255) { mlg_set_error("min_count and counter_max must be 1..255"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(q->ctx));
    return q->rk ? rk_check(q->rk) : rkp_check(q->rkp);
}
MLG_API int mlg_query_read_kmers(mlg_query* q, uint32_t min_count, uint32_t counter_max, uint64_t* keys_out, uint8_t* counts_out,
                                 uint64_t cap, uint64_t* n) {
    if (!n) { mlg_set_error("null n"); return MLG_ERR_ARG; }
    MLG_TRY(check_read_kmers(q, min_count, counter_max));
    q->rk_out = KmcOutStats{};
    if (q->rkp) return rkp_read_kmers(q->rkp, min_count, counter_max, keys_out, counts_out, cap, n, &q->rk_out);
    DevBuf<key128> keys; DevBuf<uint32_t> cnt;
    uint32_t m = 0;
    MLG_TRY(rk_collect(q->rk, min_count, keys, cnt, &m, &q->rk_out));
    q->rk_out.records = m;
    *n = m;
    const uint64_t c = std::min<uint64_t>(cap, m);
    if (!c) return MLG_OK;
    std::vector<uint32_t> hc(c);
    if (keys_out) CUDA_TRY(cudaMemcpyAsync(keys_out, keys.p, c * sizeof(key128), cudaMemcpyDeviceToHost, q->ctx->s_comp));
    CUDA_TRY(cudaMemcpyAsync(hc.data(), cnt.p, c * 4, cudaMemcpyDeviceToHost, q->ctx->s_comp));
    CUDA_TRY(cudaStreamSynchronize(q->ctx->s_comp));
    if (counts_out) for (uint64_t i = 0; i < c; ++i) counts_out[i] = (uint8_t)std::min(hc[i], counter_max);
    return MLG_OK;
}
MLG_API int mlg_query_write_reads_kmc(mlg_query* q, const char* prefix, uint32_t min_count, uint32_t counter_max) {
    if (!prefix) { mlg_set_error("null prefix"); return MLG_ERR_ARG; }
    MLG_TRY(check_read_kmers(q, min_count, counter_max));
    q->rk_out = KmcOutStats{};
    if (q->rkp) return rkp_write_kmc(q->rkp, prefix, min_count, counter_max, &q->rk_out);
    DevBuf<key128> keys; DevBuf<uint32_t> cnt;
    uint32_t m = 0;
    MLG_TRY(rk_collect(q->rk, min_count, keys, cnt, &m, &q->rk_out));
    return kmc_write(q->ctx, prefix, keys.p, cnt.p, m, q->db->v.K, min_count, counter_max, &q->rk_out);
}
MLG_API int mlg_query_write_intersection_kmc(mlg_query* q, const char* prefix, uint32_t counter_max) {
    if (!q || !prefix) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (!q->finished) { mlg_set_error("call mlg_query_finish first"); return MLG_ERR_STATE; }
    if (counter_max == 0 || counter_max > 255) { mlg_set_error("counter_max must be 1..255"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(q->ctx));
    const uint32_t n = q->n_present;
    DevBuf<key128> d, keys; DevBuf<unsigned char> dc; DevBuf<uint32_t> cnt;
    if (n) {
        MLG_TRY(d.alloc(n)); MLG_TRY(dc.alloc(n));
        MLG_TRY(launch_gather_keys(q->db->D_key.p, q->present.p, n, d.p, q->ctx->s_comp));
        MLG_TRY(launch_gather_counts(q->cnt8.p, q->db->D_mult.p, q->present.p, n, counter_max, dc.p, q->ctx->s_comp));
        MLG_TRY(rk_sort_pairs(q->ctx, d.p, dc.p, n, q->db->v.K, keys, cnt));
    }
    return kmc_write(q->ctx, prefix, keys.p, cnt.p, n, q->db->v.K, 1, counter_max, nullptr);
}
MLG_API int mlg_query_read_kmer_stats(mlg_query* q, mlg_read_kmer_stats* out) {
    if (!q || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (!q->rk && !q->rkp) { mlg_set_error("the read k-mer table is off (mlg_query_enable_read_kmers)"); return MLG_ERR_STATE; }
    MLG_TRY(ensure_device(q->ctx));
    MLG_TRY(q->rk ? rk_stats(q->rk, out) : rkp_stats(q->rkp, out));
    out->out_records = q->rk_out.records; out->out_bytes = q->rk_out.bytes;
    out->ms_compact = q->rk_out.ms_compact; out->ms_sort = q->rk_out.ms_sort; out->ms_encode = q->rk_out.ms_encode;
    out->s_write = q->rk_out.s_write;
    return MLG_OK;
}
MLG_API int mlg_query_read_kmer_plan(mlg_query* q, mlg_read_kmer_plan* out) {
    if (!q || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (!q->rkp) { mlg_set_error("read k-mer passes are off (mlg_query_enable_read_kmer_passes)"); return MLG_ERR_STATE; }
    return rkp_plan(q->rkp, out);
}

MLG_API int mlg_query_read_kmer_archive(mlg_query* q, uint32_t rank, uint32_t world, const void** d_blob, uint64_t* bytes) {
    if (!q || !d_blob || !bytes) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    if (!q->rkp) { mlg_set_error("read k-mer passes are off (mlg_query_enable_read_kmer_passes)"); return MLG_ERR_STATE; }
    if (q->rk_shared) { mlg_set_error("this query's read archive was already packed"); return MLG_ERR_STATE; }
    if (world < 1 || world > MLG_MAX_RANKS || rank >= world) { mlg_set_error("rank %u of %u ranks: need rank < world <= %d", rank, world, MLG_MAX_RANKS); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(q->ctx));
    MLG_TRY(rkp_pack_archive(q->rkp, rank, world, d_blob, bytes));
    q->rk_shared = true;
    return MLG_OK;
}
MLG_API int mlg_query_read_kmer_add_archive(mlg_query* q, const void* d_blob, uint64_t bytes) {
    if (!q) { mlg_set_error("null query"); return MLG_ERR_ARG; }
    if (!q->rk_shared) { mlg_set_error("call mlg_query_read_kmer_archive first"); return MLG_ERR_STATE; }
    if (!d_blob) { mlg_set_error("null blob"); return MLG_ERR_ARG; }
    MLG_TRY(ensure_device(q->ctx));
    return rkp_add_archive(q->rkp, d_blob, bytes, &q->st.gpu_launches);
}
MLG_API int mlg_kmc_concat(const char* prefix, const char* const* part_prefixes, uint32_t n_parts) {
    if (!prefix || !part_prefixes || !n_parts) { mlg_set_error("null argument or no part"); return MLG_ERR_ARG; }
    for (uint32_t i = 0; i < n_parts; ++i) if (!part_prefixes[i]) { mlg_set_error("null part prefix"); return MLG_ERR_ARG; }
    return kmc_concat(prefix, part_prefixes, n_parts);
}

MLG_API int mlg_query_stats(mlg_query* q, mlg_stats* out) {
    if (!q || !out) { mlg_set_error("null argument"); return MLG_ERR_ARG; }
    *out = q->st;
    return MLG_OK;
}

MLG_API int mlg_query_free(mlg_query* q) {
    if (!q) return MLG_OK;
    cudaSetDevice(q->ctx->device);
    cudaStreamSynchronize(q->ctx->s_copy);
    cudaStreamSynchronize(q->ctx->s_comp);
    // The counter table goes to the next query of this database all-zero: only the counters this query touched are
    // visited (a dense all-reduce writes counters that are on no list, so that table is dropped instead).
    if (q->db && q->cnt8.p && !q->reduced && !q->db->clean_cnt8.p) {
        bool ok = true;
        if (q->touched.p) {
            ok = launch_clear_touched(q->cnt8.p, q->touched.p, q->d_scalar.p + 1, q->ctx->s_comp) == MLG_OK &&
                 cudaStreamSynchronize(q->ctx->s_comp) == cudaSuccess;
        }
        if (ok) { std::swap(q->cnt8.p, q->db->clean_cnt8.p); std::swap(q->cnt8.n, q->db->clean_cnt8.n); }
    }
    rk_destroy(q->rk);
    rkp_destroy(q->rkp);
    for (auto& pe : q->probe_events) { cudaEventDestroy(pe.first); cudaEventDestroy(pe.second); }
    for (auto& e : q->chunk_events) cudaEventDestroy(e);
    for (auto& s : q->stg) if (s.done) cudaEventDestroy(s.done);
    if (q->ev_q0) cudaEventDestroy(q->ev_q0);
    if (q->ev_q1) cudaEventDestroy(q->ev_q1);
    delete q;
    return MLG_OK;
}

}  // extern "C"
