// .mlgdb files: reading the source form (version 1: the G*n sketch keys, everything else rebuilt on the GPU) and
// writing / reading the BUILT form (version 2: the device structures themselves), so that a run of select_db.py pays a
// file read instead of a database build.  The reference pays the analogous cost on every run as well: CMash re-imports
// the training HDF5 and its trie, KMC re-reads its database (scripts/select_db.py:44,69-70).
//
// Version 2 layout (little endian):
//   "MLGDB002" | u32 K, n | u64 G | u32 nk, ks[8] | u64 names_bytes | names | pad to 16          (same head as version 1)
//   u32 build_tag | u32 n_sections | u64 scalars[16] | sections[n_sections] {u32 tag, u32 elem_bytes, u64 count, u64 offset}
//   section payloads, each starting at a multiple of 4096
// scalars: np, nd, layout, fbits, bbits, slots, nbuckets, nfw, fk, n_alias, hit_words, 5 reserved.
// build_tag changes whenever the meaning of the stored structures does (hash functions, record formats): a stale file is
// refused, not misread.
#include <fcntl.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <thread>
#include <vector>
#include "mlg_internal.h"

namespace {

constexpr uint32_t BUILD_TAG = MLG_BUILD_TAG;
enum : uint32_t { S_DKEY = 1, S_BSTART, S_F, S_ALIAS_Z, S_ALIAS_I, S_ALIAS_BLOOM, S_HOFF, S_HBASE, S_HITS, S_DEN, S_HASEMPTY, S_T1, S_DMULT };
struct Section { uint32_t tag, elem; uint64_t count, offset; };
constexpr size_t CHUNK = (size_t)8 << 20;        // staging granularity.  Page-locking costs ~0.7 ms per MiB on the GPU boxes: 12 x 32 MiB
constexpr int NBUF = 12;                         // took 0.26 s of a 0.65 s load (r4u); 12 x 8 MiB take 0.07 s and keep the copies back to back

inline uint64_t up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

struct Head { uint32_t K = 0, n = 0, nk = 0, ks[8] = {}; uint64_t G = 0, names_bytes = 0, end = 0; int version = 0; };

int read_head(int fd, const char* path, Head& h) {
    unsigned char b[68];
    if (pread(fd, b, 68, 0) != 68) { mlg_set_error("%s: truncated header", path); return MLG_ERR_IO; }
    if (memcmp(b, "MLGDB001", 8) == 0) h.version = 1;
    else if (memcmp(b, "MLGDB002", 8) == 0) h.version = 2;
    else { mlg_set_error("%s: not a .mlgdb file", path); return MLG_ERR_IO; }
    memcpy(&h.K, b + 8, 4); memcpy(&h.n, b + 12, 4); memcpy(&h.G, b + 16, 8); memcpy(&h.nk, b + 24, 4);
    memcpy(h.ks, b + 28, 32); memcpy(&h.names_bytes, b + 60, 8);
    if (h.G == 0 || h.G > 0xFFFFFFFFull || h.nk < 1 || h.nk > 8 || h.n == 0) { mlg_set_error("%s: bad header", path); return MLG_ERR_IO; }
    h.end = up(68 + h.names_bytes, 16);
    return MLG_OK;
}

// pinned staging buffers of one load: allocated once (page-locking memory costs milliseconds per buffer), used by every section
struct Stager {
    void* buf[NBUF] = {};
    cudaEvent_t ev[NBUF] = {};
    int n = 0;
    int init() {
        for (n = 0; n < NBUF; ++n)
            if (cudaMallocHost(&buf[n], CHUNK) != cudaSuccess || cudaEventCreateWithFlags(&ev[n], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                if (buf[n]) { cudaFreeHost(buf[n]); buf[n] = nullptr; }
                break;
            }
        if (n < 2) { mlg_set_error("pinned staging allocation failed"); return MLG_ERR_NOMEM; }
        return MLG_OK;
    }
    ~Stager() { for (int i = 0; i < NBUF; ++i) { if (buf[i]) cudaFreeHost(buf[i]); if (ev[i]) cudaEventDestroy(ev[i]); } }
};

// file range -> device memory.  Chunk c goes through pinned buffer c % nb: reader threads pread() chunks in order, each
// waiting until the copy of the chunk that used its buffer before has completed; the calling thread issues the copies
// in order and retires them (`freed` = chunks whose copy is known to be complete), keeping a few in flight.
int file_to_device(Stager& sg, int fd, const char* path, uint64_t off, void* dst, uint64_t bytes, cudaStream_t st) {
    if (!bytes) return MLG_OK;
    const uint64_t nchunks = (bytes + CHUNK - 1) / CHUNK;
    const int nb = (int)std::min<uint64_t>((uint64_t)sg.n, nchunks);
    int rc = MLG_OK;
    {
        std::vector<std::atomic<int>> ready(nchunks);   // 0 = not read yet, 1 = in its buffer, -1 = read error
        for (auto& r : ready) r.store(0);
        std::atomic<uint64_t> next{0}, freed{0};
        std::atomic<bool> stop{false};
        std::vector<std::thread> readers;
        const int nthreads = std::min(nb, 6);
        for (int t = 0; t < nthreads; ++t)
            readers.emplace_back([&] {
                for (;;) {
                    const uint64_t c = next.fetch_add(1);
                    if (c >= nchunks) return;
                    while (c >= freed.load() + (uint64_t)nb) { if (stop.load()) return; std::this_thread::yield(); }
                    if (stop.load()) return;
                    const uint64_t o = c * CHUNK, m = std::min<uint64_t>(CHUNK, bytes - o);
                    uint64_t got = 0;
                    while (got < m) {
                        const ssize_t k = pread(fd, (char*)sg.buf[c % nb] + got, m - got, (off_t)(off + o + got));
                        if (k <= 0) break;
                        got += (uint64_t)k;
                    }
                    ready[c].store(got == m ? 1 : -1);
                }
            });
        uint64_t retired = 0;
        for (uint64_t c = 0; c < nchunks; ++c) {
            int r;
            while ((r = ready[c].load()) == 0) std::this_thread::yield();
            if (r < 0) { mlg_set_error("%s: truncated or unreadable", path); rc = MLG_ERR_IO; break; }
            const uint64_t o = c * CHUNK, m = std::min<uint64_t>(CHUNK, bytes - o);
            if (cudaMemcpyAsync((char*)dst + o, sg.buf[c % nb], m, cudaMemcpyHostToDevice, st) != cudaSuccess ||
                cudaEventRecord(sg.ev[c % nb], st) != cudaSuccess) { mlg_set_error("%s: host->device copy failed", path); rc = MLG_ERR_CUDA; break; }
            while (c + 1 - retired > (uint64_t)std::max(1, nb / 2)) {      // at most half of the buffers wait for their copy
                if (cudaEventSynchronize(sg.ev[retired % nb]) != cudaSuccess) { mlg_set_error("%s: host->device copy failed", path); rc = MLG_ERR_CUDA; break; }
                freed.store(++retired);
            }
            if (rc != MLG_OK) break;
        }
        stop.store(true);
        if (cudaStreamSynchronize(st) != cudaSuccess && rc == MLG_OK) { mlg_set_error("%s: host->device copy failed", path); rc = MLG_ERR_CUDA; }
        freed.store(nchunks + (uint64_t)nb);
        for (auto& th : readers) th.join();
    }
    return rc;
}

int device_to_file(FILE* f, const void* src, uint64_t bytes, void* pinned, cudaStream_t st) {
    for (uint64_t o = 0; o < bytes; o += CHUNK) {
        const uint64_t m = std::min<uint64_t>(CHUNK, bytes - o);
        CUDA_TRY(cudaMemcpyAsync(pinned, (const char*)src + o, m, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (fwrite(pinned, 1, m, f) != m) { mlg_set_error("short write"); return MLG_ERR_IO; }
    }
    return MLG_OK;
}

}  // namespace

int mlg_db_load_file(mlg_ctx* ctx, const char* path, mlg_db** out) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { mlg_set_error("cannot open %s", path); return MLG_ERR_IO; }
    struct Closer { int fd; ~Closer() { close(fd); } } closer{fd};
    Head h;
    MLG_TRY(read_head(fd, path, h));
    cudaStream_t st = ctx->s_comp;
    const bool verbose = getenv("MLG_VERBOSE_BUILD") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count(); };
    Stager sg;
    MLG_TRY(sg.init());
    if (verbose) fprintf(stderr, "[mlg load] %d pinned staging buffers of %zu MiB after %.3f s\n", sg.n, CHUNK >> 20, since());
    if (h.version == 1) {
        const size_t total = (size_t)h.G * h.n;
        DevBuf<key128> d; MLG_TRY(d.alloc(total));
        MLG_TRY(file_to_device(sg, fd, path, h.end, d.p, (uint64_t)total * sizeof(key128), st));
        return mlg_db_build_device(ctx, d.p, (uint32_t)h.G, h.n, h.K, h.ks, h.nk, out);
    }
    cudaEvent_t e0, e1; CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, st));
    uint32_t tag = 0, nsec = 0; uint64_t sc[16];
    if (pread(fd, &tag, 4, (off_t)h.end) != 4 || pread(fd, &nsec, 4, (off_t)h.end + 4) != 4 || pread(fd, sc, 128, (off_t)h.end + 8) != 128) {
        mlg_set_error("%s: truncated", path); return MLG_ERR_IO;
    }
    if (tag != BUILD_TAG) { mlg_set_error("%s was built by another version of this library (tag %08x, expected %08x): rebuild it from its source", path, tag, BUILD_TAG); return MLG_ERR_IO; }
    if (nsec > 64) { mlg_set_error("%s: bad section table", path); return MLG_ERR_IO; }
    std::vector<Section> secs(nsec);
    if (nsec && pread(fd, secs.data(), nsec * sizeof(Section), (off_t)h.end + 136) != (ssize_t)(nsec * sizeof(Section))) { mlg_set_error("%s: truncated", path); return MLG_ERR_IO; }
    struct stat sb;
    if (fstat(fd, &sb) != 0) { mlg_set_error("%s: fstat failed", path); return MLG_ERR_IO; }
    mlg_db* db = new mlg_db();
    struct Guard { mlg_db* d; ~Guard() { if (d) delete d; } } guard{db};
    db->ctx = ctx;
    DbView& v = db->v;
    v.G = (uint32_t)h.G; v.n = h.n; v.K = h.K; v.nk = h.nk;
    for (uint32_t i = 0; i < MLG_MAX_KS; ++i) v.ks[i] = i < h.nk ? h.ks[i] : 0;
    v.np = (uint32_t)sc[0]; v.nd = (uint32_t)sc[1]; v.layout = (uint32_t)sc[2]; v.fbits = (uint32_t)sc[3]; v.bbits = (uint32_t)sc[4];
    v.slots = (uint32_t)sc[5]; v.nbuckets = sc[6]; v.nfw = (uint32_t)sc[7]; v.fk = (uint32_t)sc[8]; v.n_alias = (uint32_t)sc[9];
    db->hit_words = sc[10];
    db->p_dropped = true;
    auto load = [&](const Section& s, auto& buf, size_t pad_elems) -> int {
        typedef typename std::remove_reference<decltype(*buf.p)>::type T;
        if (s.elem != sizeof(T) || s.offset + s.count * s.elem > (uint64_t)sb.st_size) { mlg_set_error("%s: bad section %u", path, s.tag); return MLG_ERR_IO; }
        MLG_TRY(buf.alloc((size_t)s.count + pad_elems));
        if (pad_elems) CUDA_TRY(cudaMemsetAsync(buf.p + s.count, 0, pad_elems * sizeof(T), st));
        return file_to_device(sg, fd, path, s.offset, buf.p, s.count * s.elem, st);
    };
    for (const Section& s : secs) {
        if (verbose) fprintf(stderr, "[mlg load] section %2u: %8.1f MB at %.3f s\n", s.tag, (double)(s.count * s.elem) / 1e6, since());
        switch (s.tag) {
        case S_DKEY: MLG_TRY(load(s, db->D_key, 1)); break;
        case S_BSTART: MLG_TRY(load(s, db->bstart, 0)); break;
        case S_F: MLG_TRY(load(s, db->F, 0)); break;
        case S_ALIAS_Z: MLG_TRY(load(s, db->alias_z, 0)); break;
        case S_ALIAS_I: MLG_TRY(load(s, db->alias_i, 0)); break;
        case S_ALIAS_BLOOM: MLG_TRY(load(s, db->alias_bloom, 0)); break;
        case S_HOFF: MLG_TRY(load(s, db->hoff, 0)); break;
        case S_HBASE: MLG_TRY(load(s, db->hbase, 0)); break;
        case S_HITS: MLG_TRY(load(s, db->hits, 2 + MLG_MAX_KS)); break;
        case S_DEN: MLG_TRY(load(s, db->den_real, 0)); break;
        case S_HASEMPTY: MLG_TRY(load(s, db->has_empty, 0)); break;
        case S_T1: MLG_TRY(load(s, db->T1, 0)); break;
        case S_DMULT: MLG_TRY(load(s, db->D_mult, 0)); break;      // optional: files written before it existed load without
        default: break;       // sections of a later minor version
        }
    }
    if (!db->D_key.p || !db->bstart.p || !db->den_real.p || !db->has_empty.p || !db->hoff.p || !db->hbase.p || !db->hits.p ||
        (v.layout == 2 && (!db->F.p || !db->alias_bloom.p))) { mlg_set_error("%s: a required section is missing", path); return MLG_ERR_IO; }
    if (!db->T1.p) { MLG_TRY(db->T1.alloc(8)); CUDA_TRY(cudaMemsetAsync(db->T1.p, 0, 32, st)); }
    v.D_key = db->D_key.p; v.bstart = db->bstart.p; v.T1 = db->T1.p; v.F = db->F.p;
    v.alias_z = db->alias_z.p; v.alias_i = db->alias_i.p; v.alias_bloom = db->alias_bloom.p;
    v.P_key = nullptr; v.P_slot = nullptr; v.pidx = nullptr; v.rep = nullptr; v.pbits = 0;
    CUDA_TRY(cudaEventRecord(e1, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (verbose) fprintf(stderr, "[mlg load] all sections on the device after %.3f s\n", since());
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1); db->build_ms = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    guard.d = nullptr;
    *out = db;
    return MLG_OK;
}

int mlg_db_save_file(const mlg_db* db, const char* path, const char* names, uint64_t names_bytes) {
    const DbView& v = db->v;
    if (!db->p_dropped || !db->hoff.p) { mlg_set_error("only a database with precomputed hit records can be saved in built form (MLG_PRECOMPUTE_HITS=0, MLG_HIT_CAP_WORDS or MLG_KEEP_P is set)"); return MLG_ERR_STATE; }
    if (v.layout != 2 && v.F) { mlg_set_error("the built form does not carry the L2 prefilter's access-policy window (layout 0 with a prefilter): load the source form instead"); return MLG_ERR_STATE; }
    FILE* f = fopen(path, "wb");
    if (!f) { mlg_set_error("cannot create %s", path); return MLG_ERR_IO; }
    struct Closer { FILE* f; ~Closer() { fclose(f); } } closer{f};
    void* pinned = nullptr;
    CUDA_TRY(cudaMallocHost(&pinned, CHUNK));
    struct HFree { void* p; ~HFree() { cudaFreeHost(p); } } hfree{pinned};
    const uint64_t G = v.G;
    uint32_t ks[8] = {};
    for (uint32_t i = 0; i < v.nk; ++i) ks[i] = v.ks[i];
    bool ok = fwrite("MLGDB002", 1, 8, f) == 8 && fwrite(&v.K, 4, 1, f) == 1 && fwrite(&v.n, 4, 1, f) == 1 && fwrite(&G, 8, 1, f) == 1 &&
              fwrite(&v.nk, 4, 1, f) == 1 && fwrite(ks, 4, 8, f) == 8 && fwrite(&names_bytes, 8, 1, f) == 1 &&
              (names_bytes == 0 || fwrite(names, 1, names_bytes, f) == names_bytes);
    uint64_t pos = 68 + names_bytes;
    static const char zeros[4096] = {};
    const uint64_t head_end = up(pos, 16);
    ok = ok && fwrite(zeros, 1, head_end - pos, f) == head_end - pos;
    const unsigned long long groups = ((unsigned long long)v.nd + (1ull << MLG_HGROUP_SHIFT) - 1) >> MLG_HGROUP_SHIFT;
    struct Src { uint32_t tag, elem; uint64_t count; const void* p; };
    std::vector<Src> src = {
        {S_DKEY, 16, v.nd, db->D_key.p}, {S_BSTART, 4, v.nbuckets + 1, db->bstart.p},
        {S_HOFF, 4, v.nd, db->hoff.p}, {S_HBASE, 8, groups + 1, db->hbase.p}, {S_HITS, 4, db->hit_words, db->hits.p},
        {S_DEN, 8, (uint64_t)v.G * v.nk, db->den_real.p}, {S_HASEMPTY, 1, v.G, db->has_empty.p},
    };
    if (db->D_mult.p) src.push_back({S_DMULT, 1, v.nd, db->D_mult.p});
    if (v.layout == 2) {
        src.push_back({S_F, 4, (uint64_t)v.nfw, db->F.p});
        src.push_back({S_ALIAS_BLOOM, 4, 2048, db->alias_bloom.p});
        if (v.n_alias) { src.push_back({S_ALIAS_Z, 8, v.n_alias, db->alias_z.p}); src.push_back({S_ALIAS_I, 4, v.n_alias, db->alias_i.p}); }
    } else {
        src.push_back({S_T1, 4, v.nbuckets * v.slots + 8, db->T1.p});
    }
    const uint32_t nsec = (uint32_t)src.size();
    uint64_t sc[16] = {v.np, v.nd, v.layout, v.fbits, v.bbits, v.slots, v.nbuckets, v.nfw, v.fk, v.n_alias, db->hit_words};
    std::vector<Section> secs(nsec);
    uint64_t o = up(head_end + 136 + nsec * sizeof(Section), 4096);
    for (uint32_t i = 0; i < nsec; ++i) { secs[i] = Section{src[i].tag, src[i].elem, src[i].count, o}; o = up(o + src[i].count * src[i].elem, 4096); }
    const uint32_t tag = BUILD_TAG;
    ok = ok && fwrite(&tag, 4, 1, f) == 1 && fwrite(&nsec, 4, 1, f) == 1 && fwrite(sc, 8, 16, f) == 16 && fwrite(secs.data(), sizeof(Section), nsec, f) == nsec;
    if (!ok) { mlg_set_error("%s: short write", path); return MLG_ERR_IO; }
    pos = head_end + 136 + nsec * sizeof(Section);
    CUDA_TRY(cudaSetDevice(db->ctx->device));
    for (uint32_t i = 0; i < nsec; ++i) {
        while (pos < secs[i].offset) { const uint64_t m = std::min<uint64_t>(4096, secs[i].offset - pos); if (fwrite(zeros, 1, m, f) != m) { mlg_set_error("%s: short write", path); return MLG_ERR_IO; } pos += m; }
        MLG_TRY(device_to_file(f, src[i].p, src[i].count * src[i].elem, pinned, db->ctx->s_comp));
        pos += src[i].count * src[i].elem;
    }
    if (fflush(f) != 0) { mlg_set_error("%s: short write", path); return MLG_ERR_IO; }
    return MLG_OK;
}
