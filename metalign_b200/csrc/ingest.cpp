// libmlg_ingest.so: reads file (FASTQ / single-line FASTA, optionally gzip) -> packed batches for
// mlg_query_push_packed_nruns().  Declared in include/metalign_b200_ingest.h; replaces the input side of
// `kmc -k60 -fq|-fa` (scripts/select_db.py:46-52 of the reference).  Host code only.
//
//   plain file       mapped (mmap): the scanner and the packers read the page cache directly, nothing is copied
//   gzip file        reader thread: the mapped file through fast_inflate.h (an in-house DEFLATE decoder: 0.45 GB/s of
//                    FASTQ text against zlib's 0.30; the CRC-32 of every member is checked by the scanner thread;
//                    MLGI_ZLIB=1 goes back to gzread) into recycled blocks -- the stream is sequential, one thread;
//                    a BGZF file (bgzip / htslib: independent members with their sizes in the header) is mapped and
//                    its members are inflated by `threads` threads at a time, CRC-checked (1.2 GB/s of text on 8 cores)
//   scanner          cuts the text into lines (AVX2 compare + movemask where the CPU has it, memchr otherwise), keeps the
//                    sequence lines as (offset, length) pairs; for a mapped file `threads` threads do it on views of
//                    `threads` blocks in two passes (count the newlines of every part, prefix sum = the line numbers a
//                    part starts with, then cut), one thread for the gzip stream
//   mlgi_next()      takes sequence lines until the batch is full, prefix-sums their lengths into read offsets and
//                    lets `threads` workers pack disjoint ranges of the output stream: 32 bases at a time with AVX2
//                    (case-folded compare for A/C/G/T, 2-bit codes from bits 1-2 of the ASCII byte, maddubs / madd /
//                    packus to 8 output bytes), 8 at a time with 64-bit SWAR otherwise, one at a time around any
//                    other symbol (N runs) and at read boundaries that are not byte-aligned in the output
// MLGI_PROFILE=1 prints where the consumer and the scanner waited; MLGI_NO_MMAP / MLGI_NO_AVX2 force the other paths.
#include <zlib.h>
#if defined(__x86_64__)
#include <immintrin.h>
#endif
#include <fcntl.h>
#include <unistd.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <errno.h>
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include <chrono>
#include <stdexcept>
#include "../../include/metalign_b200_ingest.h"
#include "fast_inflate.h"
#include "kmcdb.h"

#define MLGI_API __attribute__((visibility("default")))

namespace {

thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

template <typename T>
class BoundedQueue {
public:
    explicit BoundedQueue(size_t cap) : cap_(cap) {}
    // false when the queue was closed for good by the consumer
    bool push(T v) {
        std::unique_lock<std::mutex> g(mu_);
        not_full_.wait(g, [&] { return q_.size() < cap_ || abandoned_; });
        if (abandoned_) return false;
        q_.push_back(std::move(v));
        not_empty_.notify_one();
        return true;
    }
    // false when the producer has finished and nothing is left
    bool pop(T& out) {
        std::unique_lock<std::mutex> g(mu_);
        not_empty_.wait(g, [&] { return !q_.empty() || done_; });
        if (q_.empty()) return false;
        out = std::move(q_.front());
        q_.pop_front();
        not_full_.notify_one();
        return true;
    }
    void finish() { std::lock_guard<std::mutex> g(mu_); done_ = true; not_empty_.notify_all(); }
    void abandon() { std::lock_guard<std::mutex> g(mu_); abandoned_ = true; done_ = true; not_full_.notify_all(); not_empty_.notify_all(); }
private:
    std::mutex mu_;
    std::condition_variable not_full_, not_empty_;
    std::deque<T> q_;
    size_t cap_;
    bool done_ = false, abandoned_ = false;
};

// a block of file text with HEAD spare bytes in front of it, so that the unterminated tail of the previous block can
// be put in front without copying the block (uninitialised storage: no zero-fill pass over every block)
constexpr size_t HEAD = 1u << 16;
// blocks are recycled: a fresh 8 MiB allocation per block costs a page fault (and a zero-fill by the kernel) per 4 KiB
// inside the reader's read(2), which otherwise is the fastest stage
struct BufPool {
    std::mutex mu;
    std::vector<std::unique_ptr<char[]>> free;
    size_t bytes = 0;                          // size of the pooled blocks
    std::unique_ptr<char[]> get() {
        {
            std::lock_guard<std::mutex> g(mu);
            if (!free.empty()) { auto p = std::move(free.back()); free.pop_back(); return p; }
        }
        return std::unique_ptr<char[]>(new char[bytes]);
    }
    void put(std::unique_ptr<char[]> p) {
        std::lock_guard<std::mutex> g(mu);
        if (free.size() < 16) free.push_back(std::move(p));
    }
};
// a plain file is not read at all: it is mapped, and blocks are views of the mapping (no copy of the text; the page cache
// is what the scanner and the packers read)
struct Mapping {
    void* p = nullptr; size_t n = 0;
    ~Mapping() { if (p) munmap(p, n); }
};
struct TextBuf {
    std::unique_ptr<char[]> mem;
    std::shared_ptr<BufPool> pool;            // set when mem came from the pool
    std::shared_ptr<Mapping> map;             // set when the text is a view of a mapped file ...
    const char* ext = nullptr;                // ... starting here
    size_t off = HEAD, n = 0;                 // text = mem[off, off + n)
    const char* data() const { return ext ? ext : mem.get() + off; }
    size_t size() const { return n; }
    ~TextBuf() { if (pool && mem) pool->put(std::move(mem)); }
};
// gzip members that end inside a block (fast_inflate path): the scanner thread checks their CRC-32 / length
struct MemberEnd { size_t end; uint32_t crc, isize; };
struct RawBlock { std::shared_ptr<TextBuf> buf; std::vector<MemberEnd> ends; bool crc_on = false; };
struct Lines {
    std::shared_ptr<TextBuf> text;
    std::vector<uint32_t> start, len;       // sequence lines inside text
};

unsigned char g_code[256];
struct CodeInit {
    CodeInit() {
        memset(g_code, 4, sizeof(g_code));
        const char* s = "ACGT";
        for (int i = 0; i < 4; ++i) { g_code[(unsigned char)s[i]] = (unsigned char)i; g_code[(unsigned char)(s[i] + 32)] = (unsigned char)i; }
    }
} g_code_init;

bool g_have_avx2 = false;
struct CpuInit { CpuInit() {
#if defined(__x86_64__)
    g_have_avx2 = __builtin_cpu_supports("avx2") && !getenv("MLGI_NO_AVX2");
#endif
} } g_cpu_init;
#if defined(__x86_64__)
// calls f(e) for the position e of every '\n' in base[0, n & ~31), in order; returns n & ~31
template <typename F>
__attribute__((target("avx2"))) size_t scan_newlines_avx2(const char* base, size_t n, F f) {
    const __m256i nl = _mm256_set1_epi8('\n');
    size_t i = 0;
    for (; i + 32 <= n; i += 32) {
        uint32_t m = (uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(_mm256_loadu_si256((const __m256i*)(base + i)), nl));
        while (m) { f(i + (size_t)__builtin_ctz(m)); m &= m - 1; }
    }
    return i;
}
__attribute__((target("avx2,popcnt"))) size_t count_newlines_avx2(const char* base, size_t n) {
    const __m256i nl = _mm256_set1_epi8('\n');
    size_t i = 0, c = 0;
    for (; i + 32 <= n; i += 32)
        c += (size_t)__builtin_popcount((uint32_t)_mm256_movemask_epi8(_mm256_cmpeq_epi8(_mm256_loadu_si256((const __m256i*)(base + i)), nl)));
    for (; i < n; ++i) c += base[i] == '\n';
    return c;
}
#endif
size_t count_newlines(const char* base, size_t n) {
#if defined(__x86_64__)
    if (g_have_avx2) return count_newlines_avx2(base, n);
#endif
    size_t c = 0;
    for (const char* q = base; (q = (const char*)memchr(q, '\n', (size_t)(base + n - q))) != nullptr; ++q) ++c;
    return c;
}

}  // namespace

struct mlgi_reader {
    gzFile fh = nullptr;
    int fd = -1;                        // plain (not gzip) files are read with read(2): no inflate layer in the way
    int type = MLGI_FASTQ;
    int threads = 1;
    size_t block_bytes = 8u << 20;
    std::shared_ptr<BufPool> pool = std::make_shared<BufPool>();
    BoundedQueue<RawBlock> q_raw{4};
    BoundedQueue<Lines> q_lines{4};
    std::thread t_read, t_scan;
    std::vector<uint32_t> spill;        // N runs of the last batch when they did not fit the caller's buffer
    std::string io_error;               // set by the reader thread before it finishes the queue
    std::mutex err_mu;
    // consumer state
    Lines cur;
    size_t cur_i = 0;
    bool eof = false;
    uint64_t tot_reads = 0, tot_bases = 0, tot_text = 0;
    // a share of the file (mlgi_open_share): the text [share_lo, share_hi) of a mapped plain file, or the members
    // [bgzf_in0, bgzf_in1) of a BGZF file less bgzf_skip bytes in front and cut after bgzf_take bytes; its first line has
    // number line_no0 (FASTQ phase) and share_first is its offset in the file's text
    size_t share_lo = 0, share_hi = ~(size_t)0, bgzf_in0 = 0, bgzf_in1 = ~(size_t)0, bgzf_skip = 0, bgzf_take = ~(size_t)0;
    uint64_t line_no0 = 0, share_first = 0;
    int share_phase = 0;
    bool tail_open = false;             // the text's last line has no '\n' (scanner thread)
    double t_wait_lines = 0, t_gather = 0, t_pack = 0, t_scan_wait = 0;   // MLGI_PROFILE=1

    // plain gzip (one long deflate stream): fast_inflate.h on the mapped file, one thread -- the stream is sequential.
    // Every block starts HEAD bytes into its buffer; the last 32 KiB of the previous block are copied in front of it (the
    // decoder's match window, and at the same time the bytes the scanner would prepend as the carried-over line).
    void read_loop_gz_fast() {
        auto fail = [&](const char* m) { std::lock_guard<std::mutex> g(err_mu); io_error = m; q_raw.finish(); };
        fastinf::Inflater* z = new fastinf::Inflater();
        std::unique_ptr<fastinf::Inflater> zguard(z);
        z->in = (const uint8_t*)gzmap->p; z->in_end = z->in + gzmap->n;
        std::vector<uint8_t> hist;                       // tail of the previous block
        uint64_t member_bytes = 0;
        pool->bytes = HEAD + block_bytes + fastinf::SLACK + 8;
        for (bool more = true; more;) {
            RawBlock b;
            b.buf = std::make_shared<TextBuf>();
            b.buf->mem = pool->get();
            b.buf->pool = pool;
            uint8_t* start = (uint8_t*)b.buf->mem.get() + HEAD;
            if (!hist.empty()) memcpy(start - hist.size(), hist.data(), hist.size());
            const uint8_t* begin = start - hist.size();
            uint8_t* out = start;
            uint8_t* const limit = start + block_bytes;
            for (;;) {
                uint8_t* const seg = out;
                const int rc = z->run(out, limit, begin);
                if (rc < 0) { fail(z->error ? z->error : "corrupt gzip stream"); return; }
                member_bytes += (uint64_t)(out - seg);
                if (rc == 1) {                           // a member ended (the scanner thread checks its CRC); go on in the same block
                    if ((uint32_t)member_bytes != z->isize_expected) { fail("gzip length mismatch"); return; }
                    b.ends.push_back(MemberEnd{(size_t)(out - start), z->crc_expected, z->isize_expected});
                    member_bytes = 0;
                    if (out < limit) continue;
                    break;
                }
                if (rc == 2) { more = false; if (member_bytes) { fail("gzip stream ends inside a member"); return; } }
                break;                                   // rc == 0: the block is full
            }
            b.buf->n = (size_t)(out - start);
            b.crc_on = true;
            const size_t keep = std::min<size_t>((size_t)(out - begin), fastinf::WINDOW);
            hist.assign(out - keep, out);
            if (b.buf->n && !q_raw.push(std::move(b))) return;
        }
        q_raw.finish();
    }

    // BGZF (bgzip / htslib): a gzip file made of independent members of at most 64 KiB, each carrying its compressed size
    // in a 'BC' extra field and its inflated size in its trailer -- so members can be found without inflating anything and
    // inflated in parallel into known places.  Jobs of ~block_bytes of output are inflated `threads` at a time and handed
    // to the scanner in file order.
    std::shared_ptr<Mapping> gzmap;      // the compressed file, mapped (BGZF only)
    static bool bgzf_member(const unsigned char* p, size_t left, size_t* csize, size_t* hdr) {
        if (left < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return false;
        const size_t xlen = p[10] | ((size_t)p[11] << 8);
        if (left < 12 + xlen) return false;
        for (size_t o = 12; o + 4 <= 12 + xlen;) {
            const size_t slen = p[o + 2] | ((size_t)p[o + 3] << 8);
            if (p[o] == 'B' && p[o + 1] == 'C' && slen == 2 && o + 6 <= 12 + xlen) {
                *csize = (size_t)(p[o + 4] | ((size_t)p[o + 5] << 8)) + 1;
                *hdr = 12 + xlen;                                    // (FNAME / FCOMMENT / FHCRC are not used by BGZF writers)
                return *csize >= *hdr + 8 && *csize <= left;
            }
            o += 4 + slen;
        }
        return false;
    }
    // inflates the members in base[in0, in1) (found by bgzf_member) into dst, which has room for the sum of their sizes;
    // false on a member that does not inflate to its stated size and CRC-32
    static bool bgzf_inflate(const unsigned char* base, size_t n, size_t in0, size_t in1, char* dst, size_t* out_n) {
        size_t o = 0;
        for (size_t q = in0; q < in1;) {
            size_t cs = 0, hd = 0;
            bgzf_member(base + q, n - q, &cs, &hd);
            const unsigned char* t = base + q + cs - 4;
            const size_t isz = (size_t)t[0] | ((size_t)t[1] << 8) | ((size_t)t[2] << 16) | ((size_t)t[3] << 24);
            z_stream zs;
            memset(&zs, 0, sizeof(zs));
            if (inflateInit2(&zs, -15) != Z_OK) return false;
            zs.next_in = const_cast<unsigned char*>(base + q + hd); zs.avail_in = (uInt)(cs - hd - 8);
            zs.next_out = (unsigned char*)dst + o; zs.avail_out = (uInt)isz;
            const int rc = inflate(&zs, Z_FINISH);
            bool good = rc == Z_STREAM_END && zs.total_out == isz;
            inflateEnd(&zs);
            if (good) {
                const unsigned char* c = t - 4;
                const unsigned long want = (unsigned long)c[0] | ((unsigned long)c[1] << 8) | ((unsigned long)c[2] << 16) | ((unsigned long)c[3] << 24);
                good = crc32(crc32(0L, Z_NULL, 0), (const Bytef*)dst + o, (uInt)isz) == want;
            }
            if (!good) return false;
            o += isz; q += cs;
        }
        *out_n = o;
        return true;
    }
    void read_loop_bgzf() {
        const unsigned char* base = (const unsigned char*)gzmap->p;
        const size_t n = std::min(gzmap->n, bgzf_in1);
        struct Job { size_t in0, in1, out; std::shared_ptr<TextBuf> buf; bool ok = true; };
        const size_t P = (size_t)std::max(1, std::min(threads, 32));
        size_t pos = bgzf_in0;
        uint64_t upos = 0;                                           // text offset of the next job (share trimming)
        auto fail = [&](const char* m) { std::lock_guard<std::mutex> g(err_mu); io_error = m; q_raw.finish(); };
        while (pos < n) {
            std::vector<Job> jobs;
            while (jobs.size() < P && pos < n) {                     // cut the next jobs: whole members, ~block_bytes of output each
                Job j; j.in0 = pos; j.out = 0;
                while (pos < n && j.out < block_bytes) {
                    size_t cs = 0, hd = 0;
                    if (!bgzf_member(base + pos, n - pos, &cs, &hd)) { fail("not a BGZF member where one was expected"); return; }
                    const unsigned char* t = base + pos + cs - 4;
                    j.out += (size_t)t[0] | ((size_t)t[1] << 8) | ((size_t)t[2] << 16) | ((size_t)t[3] << 24);
                    pos += cs;
                }
                j.in1 = pos;
                jobs.push_back(std::move(j));
            }
            auto inflate_job = [&](Job& j) {
                j.buf = std::make_shared<TextBuf>();
                j.buf->mem.reset(new char[HEAD + j.out + 1]);
                j.ok = bgzf_inflate(base, n, j.in0, j.in1, j.buf->mem.get() + HEAD, &j.buf->n);
            };
            std::vector<std::thread> th;
            for (size_t i = 1; i < jobs.size(); ++i) th.emplace_back([&, i] { inflate_job(jobs[i]); });
            inflate_job(jobs[0]);
            for (auto& x : th) x.join();
            for (auto& j : jobs) {
                if (!j.ok) { fail("corrupt BGZF member"); return; }
                const size_t jn = j.buf->n;                          // keep [bgzf_skip, bgzf_skip + bgzf_take) of the text
                const size_t lo = (size_t)std::min<uint64_t>(jn, bgzf_skip > upos ? bgzf_skip - upos : 0);
                const uint64_t stop = bgzf_take > ~(size_t)0 - bgzf_skip ? ~(uint64_t)0 : (uint64_t)(bgzf_skip + bgzf_take);
                const size_t hi = (size_t)std::max<uint64_t>(lo, std::min<uint64_t>(jn, stop > upos ? stop - upos : 0));
                upos += jn;
                j.buf->off = HEAD + lo; j.buf->n = hi - lo;
                RawBlock b; b.buf = j.buf;
                if (j.buf->n && !q_raw.push(std::move(b))) return;
            }
        }
        q_raw.finish();
    }

    void read_loop() {
        for (;;) {
            RawBlock b;
            b.buf = std::make_shared<TextBuf>();
            pool->bytes = HEAD + block_bytes;
            b.buf->mem = pool->get();
            b.buf->pool = pool;
            char* dst = b.buf->mem.get() + HEAD;
            size_t got = 0;
            while (got < block_bytes) {
                int want = (int)std::min<size_t>(block_bytes - got, 1u << 30);
                long n = fd >= 0 ? (long)read(fd, dst + got, (size_t)want) : (long)gzread(fh, dst + got, (unsigned)want);
                if (n < 0) {
                    int errnum = 0;
                    const char* m = fd >= 0 ? strerror(errno) : gzerror(fh, &errnum);
                    std::lock_guard<std::mutex> g(err_mu);
                    io_error = m ? m : "read failed";
                    q_raw.finish();
                    return;
                }
                if (n == 0) break;
                got += (size_t)n;
            }
            b.buf->n = got;
            const bool last = got < block_bytes;
            if (got && !q_raw.push(std::move(b))) return;
            if (last) { q_raw.finish(); return; }
        }
    }

    uint64_t line_no = 0;                // lines completed so far (FASTQ: record = 4 lines); scanner thread only
    std::shared_ptr<Mapping> map;        // plain files
    // cuts text into lines, appends the sequence lines to out; returns the bytes consumed (an incomplete last line is not)
    size_t emit_lines(const std::shared_ptr<TextBuf>& text, bool final_block, Lines& out) {
        const char* base = text->data();
        const size_t n = text->size();
        size_t p = 0;                                     // start of the current line
        out.start.reserve(n / 128); out.len.reserve(n / 128);
        auto line_ends_at = [&](size_t e) {               // the line [p, e) is complete (e = its '\n', or the end of the file)
            size_t le = e;
            if (le > p && base[le - 1] == '\r') --le;
            bool is_seq;
            if (type == MLGI_FASTQ) is_seq = (line_no & 3u) == 1u;
            else is_seq = le > p && base[p] != '>' && base[p] != ';';
            if (is_seq) { out.start.push_back((uint32_t)p); out.len.push_back((uint32_t)(le - p)); }
            ++line_no;
        };
        size_t q = 0;                                     // bytes [0, q) have been searched for '\n'
#if defined(__x86_64__)
        if (g_have_avx2) q = scan_newlines_avx2(base, n, [&](size_t e) { line_ends_at(e); p = e + 1; });
#endif
        while (q < n) {
            const char* nl = (const char*)memchr(base + q, '\n', n - q);
            if (!nl) break;
            const size_t e = (size_t)(nl - base);
            line_ends_at(e);
            p = e + 1; q = e + 1;
        }
        if (p < n && final_block) { line_ends_at(n); p = n; tail_open = true; }   // the file's last line has no '\n'
        return p;                                         // bytes consumed; an incomplete line is carried into the next block
    }

    // One part of a parallel scan of the view vbase[0, vend): the lines that START in [b0, b1).  nl_before = lines
    // completed before b0 (= '\n' seen so far), so every part knows its lines' numbers without waiting for the others.
    // A line may end beyond b1; one that does not end before vend is complete only in the file's last view, otherwise
    // *open_line is set to its start.  Sequence lines go to out (offsets relative to vbase).
    void scan_part(const char* vbase, size_t b0, size_t b1, size_t vend, bool final_view, bool starts_line, uint64_t nl_before,
                   Lines& out, size_t* open_line) const {
        size_t p = b0;
        uint64_t idx = nl_before;
        if (!starts_line) {                                   // b0 is inside a line that belongs to an earlier part
            const char* nl = (const char*)memchr(vbase + b0, '\n', b1 - b0);
            if (!nl) return;                                  // no line starts in this part
            p = (size_t)(nl - vbase) + 1; ++idx;
        }
        out.start.reserve((b1 - b0) / 128 + 4); out.len.reserve((b1 - b0) / 128 + 4);
        auto line = [&](size_t e) {                           // the line [p, e) is complete
            size_t le = e;
            if (le > p && vbase[le - 1] == '\r') --le;
            bool is_seq;
            if (type == MLGI_FASTQ) is_seq = (idx & 3u) == 1u;
            else is_seq = le > p && vbase[p] != '>' && vbase[p] != ';';
            if (is_seq) { out.start.push_back((uint32_t)p); out.len.push_back((uint32_t)(le - p)); }
            ++idx;
            p = e + 1;
        };
        size_t q = p;                                         // bytes [p, q) hold no '\n'
#if defined(__x86_64__)
        if (g_have_avx2 && b1 > p) {
            const size_t from = p;
            q = from + scan_newlines_avx2(vbase + from, b1 - from, [&](size_t e) { line(from + e); });
        }
#endif
        while (p < b1) {                                      // (also finishes the last line that starts before b1)
            if (q < p) q = p;
            const char* nl = (const char*)memchr(vbase + q, '\n', vend - q);
            if (!nl) {
                if (final_view && p < vend) line(vend);
                else if (p < vend) *open_line = p;
                return;
            }
            q = (size_t)(nl - vbase) + 1;
            line(q - 1);
        }
    }

    // plain file: walk the mapping in views of `threads` blocks, scanned by that many threads (pass 1 counts the '\n' of
    // every part, pass 2 cuts the lines); a view's unterminated last line simply starts the next view
    void scan_loop_mapped() {
        const char* base = (const char*)map->p + share_lo;
        const size_t n = std::min(map->n, share_hi) - share_lo;
        const size_t P = (size_t)std::max(1, std::min(threads, 16));
        size_t pos = 0, span = block_bytes * P;
        while (pos < n) {
            const size_t end = std::min(n, pos + span);
            const size_t vn = end - pos;
            if (vn >= 0xFFFFFFF0ull) { std::lock_guard<std::mutex> g(err_mu); io_error = "a single line exceeds 4 GiB"; break; }
            auto text = std::make_shared<TextBuf>();
            text->map = map; text->ext = base + pos; text->n = vn;
            const char* vb = base + pos;
            const size_t parts = (P > 1 && vn >= 64 * P) ? P : 1;
            std::vector<size_t> bnd(parts + 1), cnt(parts, 0), open(parts, (size_t)-1);
            for (size_t i = 0; i <= parts; ++i) bnd[i] = vn * i / parts;
            std::vector<Lines> outs(parts);
            auto run = [&](auto&& fn) {
                std::vector<std::thread> th;
                for (size_t i = 1; i < parts; ++i) th.emplace_back([&fn, i] { fn(i); });
                fn(0);
                for (auto& x : th) x.join();
            };
            if (parts > 1) run([&](size_t i) { cnt[i] = count_newlines(vb + bnd[i], bnd[i + 1] - bnd[i]); });
            std::vector<uint64_t> before(parts + 1, line_no);
            for (size_t i = 0; i < parts; ++i) before[i + 1] = before[i] + cnt[i];
            run([&](size_t i) {
                outs[i].text = text;
                scan_part(vb, bnd[i], bnd[i + 1], vn, end == n, i == 0 || vb[bnd[i] - 1] == '\n', before[i], outs[i], &open[i]);
            });
            size_t used = vn;                                 // everything, unless some line is still open at the end of the view
            for (size_t i = 0; i < parts; ++i) if (open[i] != (size_t)-1) { used = open[i]; break; }
            if (used == 0 && end < n) { span += block_bytes * P; continue; }      // one line longer than the view: widen it
            // lines completed in this view: its '\n' up to `used`, plus the file's unterminated last line
            if (end == n && vn && vb[vn - 1] != '\n') tail_open = true;
            line_no += (parts > 1 ? before[parts] - line_no : (uint64_t)count_newlines(vb, vn)) + (tail_open ? 1u : 0u);
            pos += used; span = block_bytes * P;
            for (size_t i = 0; i < parts; ++i)
                if (!outs[i].start.empty() && !q_lines.push(std::move(outs[i]))) return;
        }
        q_lines.finish();
    }

    void scan_loop() {
        unsigned long run_crc = crc32(0L, Z_NULL, 0);
        std::string carry;               // the unterminated tail of the previous block
        RawBlock b;
        bool more = true;
        while (more) {
            const auto ts0 = std::chrono::steady_clock::now();
            more = q_raw.pop(b);
            t_scan_wait += std::chrono::duration<double>(std::chrono::steady_clock::now() - ts0).count();
            if (more && b.crc_on) {                           // gzip members decoded by fast_inflate: CRC-32 of their bytes
                const unsigned char* d = (const unsigned char*)b.buf->data();
                size_t p = 0;
                bool bad = false;
                for (const MemberEnd& m : b.ends) {
                    run_crc = crc32(run_crc, d + p, (uInt)(m.end - p));
                    if ((uint32_t)run_crc != m.crc) bad = true;
                    run_crc = crc32(0L, Z_NULL, 0);
                    p = m.end;
                }
                run_crc = crc32(run_crc, d + p, (uInt)(b.buf->size() - p));
                if (bad) { std::lock_guard<std::mutex> g(err_mu); io_error = "gzip CRC mismatch"; break; }
            }
            std::shared_ptr<TextBuf> text;
            if (more && carry.size() <= b.buf->off) {          // the usual case: the carried tail fits in front of the block
                text = b.buf;
                memcpy(text->mem.get() + text->off - carry.size(), carry.data(), carry.size());
                text->off -= carry.size(); text->n += carry.size();
            } else {
                text = std::make_shared<TextBuf>();
                const size_t bn = more ? b.buf->n : 0;
                text->mem.reset(new char[carry.size() + bn + 1]);
                text->off = 0; text->n = carry.size() + bn;
                if (!carry.empty()) memcpy(text->mem.get(), carry.data(), carry.size());
                if (bn) memcpy(text->mem.get() + carry.size(), b.buf->data(), bn);   // (or, at the end, just the last unterminated line)
            }
            if (text->size() >= 0xFFFFFFF0ull) { std::lock_guard<std::mutex> g(err_mu); io_error = "a single line exceeds 4 GiB"; break; }
            Lines out;
            out.text = text;
            const size_t used = emit_lines(text, !more, out);
            carry.assign(text->data() + used, text->size() - used);
            if (!out.start.empty() && !q_lines.push(std::move(out))) return;
        }
        q_lines.finish();
    }
};

namespace {

// pack reads [a, b) of the batch; the worker owns stream bases [off[a], off[b])
struct PackJob {
    const char* const* ptr; const uint32_t* len; const uint64_t* off;
    size_t a, b;
    uint8_t* bases;
    std::vector<uint32_t> runs;      // (start, length) pairs found in this range
};

// ---- packing: ASCII -> 2 bits per base, first base in the top bits of each byte ---------------------------------------
// code of a base from its ASCII byte, either case: (c >> 1) & 3 gives A=0 C=1 G=3 T=2; x ^ (x >> 1) swaps the last two
inline uint32_t codes4(uint32_t w) {
    uint32_t x = (w >> 1) & 0x03030303u;
    return x ^ ((x >> 1) & 0x01010101u);
}
// four codes (one per byte, first base in the low byte) -> one packed byte: the multiplier lines the 2-bit codes up in
// bits 24..31 of the product
inline uint8_t pack4(uint32_t codes) { return (uint8_t)((codes * 0x40100401u) >> 24); }
// 0x80 in every byte of x that is NOT one of a/c/g/t (x already has bit 5 set in every byte)
inline uint64_t not_acgt8(uint64_t x) {
    const uint64_t L7 = 0x7F7F7F7F7F7F7F7Full;
    auto nz = [&](uint64_t z) { return (((z & L7) + L7) | z); };          // bit 7 of every non-zero byte
    return nz(x ^ 0x6161616161616161ull) & nz(x ^ 0x6363636363636363ull) & nz(x ^ 0x6767676767676767ull) &
           nz(x ^ 0x7474747474747474ull) & 0x8080808080808080ull;
}
// n bases (n % 4 == 0), all of them A/C/G/T in either case, to n / 4 output bytes; returns false (nothing written that
// matters) at the first 8-byte group that holds another symbol
#if defined(__x86_64__)
__attribute__((target("avx2"))) size_t pack_clean_avx2(const unsigned char* s, size_t n, uint8_t* out) {
    const __m256i lo5 = _mm256_set1_epi8((char)0xDF);
    const __m256i cA = _mm256_set1_epi8('A'), cC = _mm256_set1_epi8('C'), cG = _mm256_set1_epi8('G'), cT = _mm256_set1_epi8('T');
    const __m256i three = _mm256_set1_epi8(3), one = _mm256_set1_epi8(1);
    const __m256i m41 = _mm256_set1_epi16(0x0104);          // bytes (4, 1): first base of a pair times 4 plus the second
    const __m256i m161 = _mm256_set1_epi32(0x00010010);     // words (16, 1)
    size_t i = 0;
    for (; i + 32 <= n; i += 32) {
        const __m256i v = _mm256_loadu_si256((const __m256i*)(s + i));
        const __m256i u = _mm256_and_si256(v, lo5);
        const __m256i ok = _mm256_or_si256(_mm256_or_si256(_mm256_cmpeq_epi8(u, cA), _mm256_cmpeq_epi8(u, cC)),
                                           _mm256_or_si256(_mm256_cmpeq_epi8(u, cG), _mm256_cmpeq_epi8(u, cT)));
        if (_mm256_movemask_epi8(ok) != -1) break;
        __m256i x = _mm256_and_si256(_mm256_srli_epi16(v, 1), three);
        x = _mm256_xor_si256(x, _mm256_and_si256(_mm256_srli_epi16(x, 1), one));
        const __m256i p2 = _mm256_maddubs_epi16(x, m41);      // 16-bit: c0 * 4 + c1
        const __m256i p4 = _mm256_madd_epi16(p2, m161);       // 32-bit: (c0 * 4 + c1) * 16 + (c2 * 4 + c3)
        const __m256i w16 = _mm256_packus_epi32(p4, p4);      // per 128-bit lane: 4 values as 16-bit, twice
        const __m256i w8 = _mm256_packus_epi16(w16, w16);     // per lane: 4 bytes, four times
        const uint32_t a = (uint32_t)_mm256_extract_epi32(w8, 0), b = (uint32_t)_mm256_extract_epi32(w8, 4);
        memcpy(out + i / 4, &a, 4);
        memcpy(out + i / 4 + 4, &b, 4);
    }
    return i;
}
#endif
size_t pack_clean_swar(const unsigned char* s, size_t n, uint8_t* out) {
    size_t i = 0;
    for (; i + 8 <= n; i += 8) {
        uint64_t v;
        memcpy(&v, s + i, 8);
        if (not_acgt8(v | 0x2020202020202020ull)) break;
        out[i / 4] = pack4(codes4((uint32_t)v));
        out[i / 4 + 1] = pack4(codes4((uint32_t)(v >> 32)));
    }
    return i;
}
inline size_t pack_clean(const unsigned char* s, size_t n, uint8_t* out) {
#if defined(__x86_64__)
    if (g_have_avx2) { const size_t d = pack_clean_avx2(s, n, out); return d + pack_clean_swar(s + d, n - d, out + d / 4); }
#endif
    return pack_clean_swar(s, n, out);
}

void pack_range(PackJob& j) {
    if (j.a >= j.b) return;
    uint64_t pos = j.off[j.a];
    uint8_t* out = j.bases + (pos >> 2);
    unsigned fill = (unsigned)(pos & 3u);      // bases already present in the current output byte (owned by a neighbour)
    unsigned acc = 0;
    bool first_partial = fill != 0;
    uint64_t run_start = 0; uint32_t run_len = 0;
    auto one = [&](unsigned char ch) {         // the general path: one base, N bookkeeping, byte assembly
        unsigned c = g_code[ch];
        if (c > 3u) {
            if (run_len && run_start + run_len == pos) ++run_len;
            else { if (run_len) { j.runs.push_back((uint32_t)run_start); j.runs.push_back(run_len); } run_start = pos; run_len = 1; }
            c = 0;
        }
        acc = (acc << 2) | c;
        ++pos;
        if (++fill == 4) {
            if (first_partial) { __atomic_fetch_or(out, (uint8_t)acc, __ATOMIC_RELAXED); first_partial = false; }
            else *out = (uint8_t)acc;
            ++out; fill = 0; acc = 0;
        }
    };
    for (size_t i = j.a; i < j.b; ++i) {
        const unsigned char* s = (const unsigned char*)j.ptr[i];
        const uint32_t L = j.len[i];
        uint32_t k = 0;
        while (k < L) {
            // whole output bytes of clean bases go through the vector / SWAR path; everything else one base at a time
            if (fill == 0 && L - k >= 8) {
                const size_t d = pack_clean(s + k, (size_t)((L - k) & ~3u), out);
                out += d / 4; pos += d; k += (uint32_t)d;
                if (k >= L) break;
                // an unclean group (or the read's tail) follows: take up to 8 bases the slow way, then try again
                const uint32_t lim = std::min<uint32_t>(L, k + 8);
                while (k < lim) one(s[k++]);
            } else {
                one(s[k++]);
            }
        }
    }
    if (run_len) { j.runs.push_back((uint32_t)run_start); j.runs.push_back(run_len); }
    if (fill) {     // trailing partial byte: shared with the next worker (or zero padding)
        const uint8_t v = (uint8_t)(acc << (2 * (4 - fill)));
        __atomic_fetch_or(out, v, __ATOMIC_RELAXED);
    }
}

// ---- whole files (mlgi_files_*): genome files for the sketch builder ----------------------------------------------------
// One file, inflated whole into a fresh buffer: BGZF members through bgzf_inflate, any other gzip through fast_inflate.h
// (every member's CRC-32 and length checked), a plain file through read(2).  Returns "" or what went wrong.
std::string inflate_whole_file(const char* path, std::unique_ptr<char[]>& out, size_t* out_n) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return std::string("cannot open: ") + strerror(errno);
    struct Closer { int fd; ~Closer() { close(fd); } } closer{fd};
    struct stat sb;
    if (fstat(fd, &sb) != 0) return std::string("fstat failed: ") + strerror(errno);
    const size_t size = (size_t)sb.st_size;
    unsigned char magic[2] = {0, 0};
    if (size < 2 || pread(fd, magic, 2, 0) != 2 || magic[0] != 0x1f || magic[1] != 0x8b) {
        out.reset(new char[size + 1]);
        size_t got = 0;
        while (got < size) {
            const ssize_t k = read(fd, out.get() + got, size - got);
            if (k < 0) return std::string("read failed: ") + strerror(errno);
            if (k == 0) return "file shrank while it was read";
            got += (size_t)k;
        }
        *out_n = size;
        return "";
    }
    Mapping m;
    m.p = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (m.p == MAP_FAILED) { m.p = nullptr; return std::string("mmap failed: ") + strerror(errno); }
    m.n = size;
    const unsigned char* base = (const unsigned char*)m.p;
    size_t cs = 0, hd = 0;
    if (mlgi_reader::bgzf_member(base, size, &cs, &hd)) {
        size_t total = 0;
        for (size_t q = 0; q < size; q += cs) {
            if (!mlgi_reader::bgzf_member(base + q, size - q, &cs, &hd)) return "truncated or corrupt BGZF file";
            const unsigned char* t = base + q + cs - 4;
            total += (size_t)t[0] | ((size_t)t[1] << 8) | ((size_t)t[2] << 16) | ((size_t)t[3] << 24);
        }
        out.reset(new char[total + 1]);
        if (!mlgi_reader::bgzf_inflate(base, size, 0, size, out.get(), out_n)) return "corrupt BGZF member (CRC or length mismatch)";
        return "";
    }
    // the output buffer grows as needed; the trailer's ISIZE (the last member's length mod 2^32) is the first guess
    const uint32_t isize_hint = size < 4 ? 0u : (uint32_t)base[size - 4] | ((uint32_t)base[size - 3] << 8) | ((uint32_t)base[size - 2] << 16) |
                                                ((uint32_t)base[size - 1] << 24);
    size_t cap = std::max<size_t>({(size_t)isize_hint + 64, size * 4, (size_t)1 << 16});
    std::unique_ptr<uint8_t[]> buf(new uint8_t[cap + fastinf::SLACK]);
    std::unique_ptr<fastinf::Inflater> z(new fastinf::Inflater());
    z->in = base; z->in_end = base + size;
    size_t produced = 0, member = 0;
    for (;;) {
        uint8_t* o = buf.get() + produced;
        const int rc = z->run(o, buf.get() + cap, buf.get());
        produced = (size_t)(o - buf.get());
        if (rc < 0) return std::string("corrupt or truncated gzip stream: ") + (z->error ? z->error : "?");
        if (rc == 2) break;
        if (rc == 1) {
            if ((uint32_t)(produced - member) != z->isize_expected) return "gzip length mismatch";
            if ((uint32_t)crc32(crc32(0L, Z_NULL, 0), buf.get() + member, (uInt)(produced - member)) != z->crc_expected) return "gzip CRC mismatch";
            member = produced;
            continue;
        }
        cap *= 2;                                        // rc == 0: the buffer is full
        std::unique_ptr<uint8_t[]> bigger(new uint8_t[cap + fastinf::SLACK]);
        memcpy(bigger.get(), buf.get(), produced);
        buf.swap(bigger);
    }
    out.reset(reinterpret_cast<char*>(buf.release()));
    *out_n = produced;
    return "";
}

}  // namespace

// Workers take the files in order, one file each, and run at most `ahead` files past the one the consumer waits for;
// mlgi_files_next hands them over strictly in order, so a batch does not depend on the number of workers or their timing.
struct mlgi_files {
    struct Slot { std::unique_ptr<char[]> buf; size_t n = 0; std::string err; bool ready = false; };
    std::vector<std::string> paths;
    std::vector<Slot> slots;
    std::mutex mu;
    std::condition_variable cv_ready, cv_room;
    size_t next_job = 0, consumed = 0, ahead = 4;
    bool stop = false;
    std::vector<std::thread> workers;

    void work() {
        for (;;) {
            size_t i;
            {
                std::unique_lock<std::mutex> g(mu);
                cv_room.wait(g, [&] { return stop || next_job >= paths.size() || next_job < consumed + ahead; });
                if (stop || next_job >= paths.size()) return;
                i = next_job++;
            }
            Slot s;
            s.err = inflate_whole_file(paths[i].c_str(), s.buf, &s.n);
            if (!s.err.empty()) s.buf.reset();
            s.ready = true;
            std::lock_guard<std::mutex> g(mu);
            slots[i] = std::move(s);
            cv_ready.notify_all();
        }
    }
};

extern "C" {

MLGI_API const char* mlgi_last_error(void) { return g_err; }

MLGI_API int mlgi_files_open(const char* const* paths, uint32_t nfiles, int threads, mlgi_files** out) {
    if ((!paths && nfiles) || !out) { set_error("null argument"); return -2; }
    for (uint32_t i = 0; i < nfiles; ++i) if (!paths[i]) { set_error("null path %u", i); return -2; }
    std::unique_ptr<mlgi_files> r(new mlgi_files());
    r->paths.assign(paths, paths + nfiles);
    r->slots.resize(nfiles);
    int hw = (int)std::thread::hardware_concurrency();
    if (hw < 1) hw = 1;
    const int T = std::max(1, std::min<int>(threads > 0 ? threads : hw, (int)std::max<uint32_t>(nfiles, 1u)));
    r->ahead = (size_t)std::max(4, 4 * T);
    for (int t = 0; t < T; ++t) r->workers.emplace_back([p = r.get()] { p->work(); });
    *out = r.release();
    return 0;
}

MLGI_API int mlgi_files_next(mlgi_files* r, uint8_t* buf, uint64_t cap, uint64_t* file_off, uint32_t max_files, uint32_t* n_files,
                             uint64_t* need) {
    if (!r || !buf || !file_off || !n_files || max_files == 0) { set_error("null argument or max_files = 0"); return -2; }
    *n_files = 0;
    if (need) *need = 0;
    file_off[0] = 0;
    uint64_t pos = 0;
    uint32_t k = 0;
    while (k < max_files) {
        std::unique_lock<std::mutex> g(r->mu);
        if (r->consumed >= r->paths.size()) break;
        mlgi_files::Slot& s = r->slots[r->consumed];
        r->cv_ready.wait(g, [&] { return s.ready; });
        if (!s.err.empty()) { set_error("%s: %s", r->paths[r->consumed].c_str(), s.err.c_str()); return -3; }
        if (pos + s.n > cap) {
            if (k) break;
            if (need) *need = s.n;           // a file larger than the buffer comes alone, in a buffer of its size
            set_error("%s: %llu bytes do not fit a buffer of %llu", r->paths[r->consumed].c_str(), (unsigned long long)s.n, (unsigned long long)cap);
            return 2;
        }
        std::unique_ptr<char[]> mem = std::move(s.buf);
        const size_t m = s.n;
        ++r->consumed;
        r->cv_room.notify_all();
        g.unlock();
        if (m) memcpy(buf + pos, mem.get(), m);
        pos += m;
        file_off[++k] = pos;
    }
    *n_files = k;
    return k ? 1 : 0;
}

MLGI_API void mlgi_files_close(mlgi_files* r) {
    if (!r) return;
    {
        std::lock_guard<std::mutex> g(r->mu);
        r->stop = true;
    }
    r->cv_room.notify_all();
    for (auto& t : r->workers) t.join();
    delete r;
}

MLGI_API int mlgi_open(const char* path, int input_type, int threads, mlgi_reader** out) {
    if (!path || !out) { set_error("null argument"); return -2; }
    if (input_type != MLGI_FASTQ && input_type != MLGI_FASTA) { set_error("input_type must be MLGI_FASTQ or MLGI_FASTA"); return -2; }
    int fd = open(path, O_RDONLY);
    if (fd < 0) { set_error("cannot open %s", path); return -3; }
    unsigned char magic[2] = {0, 0};
    const bool gz = pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    gzFile fh = nullptr;
    std::shared_ptr<Mapping> gzmap;
    if (gz && !getenv("MLGI_NO_BGZF")) {           // BGZF? then the members are inflated in parallel from a mapping of the file
        unsigned char h[64];
        const ssize_t got = pread(fd, h, sizeof(h), 0);
        size_t cs = 0, hd = 0;
        struct stat sb;
        if (got >= 18 && fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size >= 28) {
            // (the member may be longer than the 64 bytes peeked at: only its header has to be inside them)
            const size_t xlen = h[10] | ((size_t)h[11] << 8);
            if (12 + xlen <= (size_t)got && mlgi_reader::bgzf_member(h, (size_t)sb.st_size, &cs, &hd)) {
                void* p = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
                if (p != MAP_FAILED) { gzmap = std::make_shared<Mapping>(); gzmap->p = p; gzmap->n = (size_t)sb.st_size; }
            }
        }
    }
    bool fast_gz = false;
    if (gz && !gzmap && !getenv("MLGI_ZLIB")) {        // plain gzip: map it for the in-house decoder
        struct stat sb;
        if (fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size >= 20) {
            void* p = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
            if (p != MAP_FAILED) { gzmap = std::make_shared<Mapping>(); gzmap->p = p; gzmap->n = (size_t)sb.st_size; fast_gz = true; }
        }
    }
    if (gz && !gzmap) {
        fh = gzdopen(fd, "rb");
        if (!fh) { close(fd); set_error("cannot open %s", path); return -3; }
        gzbuffer(fh, 1u << 20);
        fd = -1;
    }
#if defined(__x86_64__)
    g_have_avx2 = __builtin_cpu_supports("avx2") && !getenv("MLGI_NO_AVX2");     // (the switch is for tests)
#endif
    mlgi_reader* r = new mlgi_reader();
    r->fh = fh; r->fd = fd; r->type = input_type; r->gzmap = gzmap;
    int hw = (int)std::thread::hardware_concurrency();
    if (hw < 1) hw = 1;
    r->threads = threads > 0 ? threads : hw;
    if (const char* s = getenv("MLGI_BLOCK_BYTES")) { long v = atol(s); if (v >= 16) r->block_bytes = (size_t)v; }
    if (fd >= 0 && !gz && !getenv("MLGI_NO_MMAP")) {
        struct stat sb;
        if (fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode) && sb.st_size > 0) {
            void* p = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
            if (p != MAP_FAILED) {
                // (no MADV_SEQUENTIAL: it lets the kernel drop the pages right behind the scan, and a file that is read
                // again -- paired runs, several k ranges -- would come from the disk instead of the page cache)
                r->map = std::make_shared<Mapping>();
                r->map->p = p; r->map->n = (size_t)sb.st_size;
            }
        }
    }
    if (r->map) r->t_scan = std::thread([r] { r->scan_loop_mapped(); });
    else {
        if (r->gzmap && fast_gz) r->t_read = std::thread([r] { r->read_loop_gz_fast(); });
        else if (r->gzmap) r->t_read = std::thread([r] { r->read_loop_bgzf(); });
        else r->t_read = std::thread([r] { r->read_loop(); });
        r->t_scan = std::thread([r] { r->scan_loop(); });
    }
    *out = r;
    return 0;
}

}  // extern "C"

namespace {

// Random access to the text of a file, for the share geometry: a mapped plain file, or the members of a BGZF file
// inflated on demand (a share looks at a few lines around its two ends only).
struct TextAccess {
    size_t total = 0;
    virtual ~TextAccess() {}
    virtual int at(size_t u) = 0;                       // the byte at u < total
    virtual size_t find_nl(size_t u) = 0;               // the first '\n' at or after u, or total
    size_t line_from(size_t u) {                        // the first line start at or after u
        if (u == 0) return 0;
        if (u >= total) return total;
        if (at(u - 1) == '\n') return u;
        const size_t e = find_nl(u);
        return e >= total ? total : e + 1;
    }
    size_t next_line(size_t p) { const size_t e = find_nl(p); return e >= total ? total : e + 1; }
    size_t prev_line(size_t p) {                        // the start of the line before the one starting at p > 0
        size_t u = p - 1;
        while (u > 0 && at(u - 1) != '\n') --u;
        return u;
    }
    // a FASTQ header: the line starts with '@' and the line two after it with '+'
    bool header_at(size_t p) {
        if (p >= total || at(p) != '@') return false;
        const size_t q = next_line(p);
        if (q >= total) return false;
        const size_t q2 = next_line(q);
        return q2 < total && at(q2) == '+';
    }
    // FASTQ line number mod 4 of the line starting at s: from the first header among it and the next three lines, or,
    // near the end of the file, among the four lines before it; -2 when there is none
    int phase(size_t s) {
        size_t p = s;
        for (int k = 0; k < 4 && p < total; ++k, p = next_line(p))
            if (header_at(p)) return (4 - k) & 3;
        p = s;
        for (int k = 1; k <= 4 && p > 0; ++k) {
            p = prev_line(p);
            if (header_at(p)) return k & 3;
        }
        return -2;
    }
};
struct MappedText : TextAccess {
    const char* b;
    MappedText(const char* base, size_t n) : b(base) { total = n; }
    int at(size_t u) override { return (unsigned char)b[u]; }
    size_t find_nl(size_t u) override {
        if (u >= total) return total;
        const char* q = (const char*)memchr(b + u, '\n', total - u);
        return q ? (size_t)(q - b) : total;
    }
};
struct BgzfText : TextAccess {
    const unsigned char* base; size_t n;
    std::vector<size_t> cstart, ustart;                 // per member, plus one entry past the last
    std::vector<std::string> cache;
    BgzfText(const unsigned char* b, size_t nn) : base(b), n(nn) {}
    std::string index() {
        size_t u = 0;
        for (size_t q = 0; q < n;) {
            size_t cs = 0, hd = 0;
            if (!mlgi_reader::bgzf_member(base + q, n - q, &cs, &hd)) return "not a BGZF member at byte " + std::to_string(q);
            cstart.push_back(q); ustart.push_back(u);
            const unsigned char* t = base + q + cs - 4;
            u += (size_t)t[0] | ((size_t)t[1] << 8) | ((size_t)t[2] << 16) | ((size_t)t[3] << 24);
            q += cs;
        }
        cstart.push_back(n); ustart.push_back(u);
        total = u;
        cache.resize(cstart.size());
        return "";
    }
    size_t member_of(size_t u) const { return (size_t)(std::upper_bound(ustart.begin(), ustart.end() - 1, u) - ustart.begin()) - 1; }
    const std::string& text(size_t m) {
        std::string& c = cache[m];
        const size_t want = ustart[m + 1] - ustart[m];
        if (c.size() != want) {
            c.assign(want + 1, '\0');
            size_t got = 0;
            if (!mlgi_reader::bgzf_inflate(base, n, cstart[m], cstart[m + 1], &c[0], &got) || got != want) throw std::runtime_error("corrupt BGZF member");
            c.resize(want);
        }
        return c;
    }
    int at(size_t u) override { const size_t m = member_of(u); return (unsigned char)text(m)[u - ustart[m]]; }
    size_t find_nl(size_t u) override {
        for (size_t m = u < total ? member_of(u) : cstart.size() - 1; u < total; ++m) {
            const std::string& t = text(m);
            const size_t o = u - ustart[m];
            const char* q = (const char*)memchr(t.data() + o, '\n', t.size() - o);
            if (q) return ustart[m] + (size_t)(q - t.data());
            u = ustart[m + 1];
        }
        return total;
    }
};

}  // namespace

extern "C" {

// A share [begin, end) of a reads file: the lines whose first byte is in it (plain file), or in the text of the BGZF members
// whose compressed start is in it.  A plain gzip stream cannot be split: the share that starts at byte 0 reads it all.
MLGI_API int mlgi_open_share(const char* path, int input_type, int threads, uint64_t begin, uint64_t end, mlgi_reader** out) {
    if (!path || !out) { set_error("null argument"); return -2; }
    if (input_type != MLGI_FASTQ && input_type != MLGI_FASTA) { set_error("input_type must be MLGI_FASTQ or MLGI_FASTA"); return -2; }
    if (begin > end) { set_error("share begins at %llu, after its end %llu", (unsigned long long)begin, (unsigned long long)end); return -2; }
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { set_error("cannot open %s", path); return -3; }
    struct Closer { int fd; ~Closer() { close(fd); } } closer{fd};
    struct stat sb;
    if (fstat(fd, &sb) != 0 || !S_ISREG(sb.st_mode)) { set_error("%s: a share needs a regular file", path); return -3; }
    const size_t size = (size_t)sb.st_size;
    if (end > size) end = size;
    if (begin > end) begin = end;
    std::shared_ptr<Mapping> map;
    if (size) {
        void* p = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (p == MAP_FAILED) { set_error("%s: mmap failed: %s", path, strerror(errno)); return -3; }
        map = std::make_shared<Mapping>(); map->p = p; map->n = size;
    }
    const unsigned char* base = map ? (const unsigned char*)map->p : nullptr;
    const bool gz = size >= 2 && base[0] == 0x1f && base[1] == 0x8b;
    size_t cs = 0, hd = 0;
    const bool bgzf = gz && mlgi_reader::bgzf_member(base, size, &cs, &hd);
    std::unique_ptr<mlgi_reader> r;
    if (gz && !bgzf) {                                   // one DEFLATE stream: all of it or nothing
        if (begin == 0) {
            if (end < size)
                fprintf(stderr, "mlgi: %s is one gzip stream and cannot be split: one share reads all of it, the others none "
                                "(recompress it with bgzip to read it in parallel)\n", path);
            mlgi_reader* whole = nullptr;
            const int rc = mlgi_open(path, input_type, threads, &whole);
            if (rc) return rc;
            *out = whole;
            return 0;
        }
        r.reset(new mlgi_reader());
        r->share_phase = -1;
        r->q_lines.finish();
        *out = r.release();
        return 0;
    }
    r.reset(new mlgi_reader());
    r->type = input_type;
    int hw = (int)std::thread::hardware_concurrency();
    if (hw < 1) hw = 1;
    r->threads = threads > 0 ? threads : hw;
    if (const char* s = getenv("MLGI_BLOCK_BYTES")) { long v = atol(s); if (v >= 16) r->block_bytes = (size_t)v; }
    size_t S = 0, E = 0;
    try {
        std::unique_ptr<TextAccess> t;
        size_t u0 = 0, u1 = 0;
        BgzfText* bt = nullptr;
        if (bgzf) {
            bt = new BgzfText(base, size);
            t.reset(bt);
            const std::string e = bt->index();
            if (!e.empty()) { set_error("%s: %s", path, e.c_str()); return -3; }
            const size_t m0 = (size_t)(std::lower_bound(bt->cstart.begin(), bt->cstart.end(), (size_t)begin) - bt->cstart.begin());
            const size_t m1 = (size_t)(std::lower_bound(bt->cstart.begin(), bt->cstart.end(), (size_t)end) - bt->cstart.begin());
            u0 = bt->ustart[m0]; u1 = bt->ustart[m1];
        } else {
            t.reset(new MappedText((const char*)base, size));
            u0 = begin; u1 = end;
        }
        S = t->line_from(u0);
        E = std::max(S, t->line_from(u1));
        r->share_first = S;
        r->share_phase = S < E ? (input_type == MLGI_FASTQ ? t->phase(S) : 0) : -1;
        if (bt && S < E) {                               // the members that hold [S, E)
            const size_t a = bt->member_of(S), b = bt->member_of(E - 1) + 1;
            r->bgzf_in0 = bt->cstart[a]; r->bgzf_in1 = bt->cstart[b];
            r->bgzf_skip = S - bt->ustart[a]; r->bgzf_take = E - S;
        }
    } catch (const std::exception& e) {
        set_error("%s: %s", path, e.what());
        return -3;
    }
    r->line_no = r->line_no0 = r->share_phase > 0 ? (uint64_t)r->share_phase : 0;
    if (S >= E) r->q_lines.finish();
    else if (bgzf) {
        r->gzmap = map;
        r->t_read = std::thread([p = r.get()] { p->read_loop_bgzf(); });
        r->t_scan = std::thread([p = r.get()] { p->scan_loop(); });
    } else {
        r->map = map;
        r->share_lo = S; r->share_hi = E;
        r->t_scan = std::thread([p = r.get()] { p->scan_loop_mapped(); });
    }
    *out = r.release();
    return 0;
}

// What the phase check of a split FASTQ file needs from a share, once mlgi_next has returned 0: the text offset of its
// first line, its number of '\n', and the FASTQ line number mod 4 it took for its first line (-1: the share is empty, -2:
// no record start was found near it).
MLGI_API int mlgi_share_info(mlgi_reader* r, uint64_t* first, uint64_t* newlines, int* phase) {
    if (!r) { set_error("null reader"); return -2; }
    if (!r->eof) { set_error("the share has not been read to its end"); return -4; }
    if (first) *first = r->share_first;
    if (newlines) *newlines = r->line_no - r->line_no0 - (r->tail_open ? 1u : 0u);
    if (phase) *phase = r->share_phase;
    return 0;
}

MLGI_API int mlgi_next(mlgi_reader* r, uint8_t* bases, uint64_t cap_bases_bytes, uint32_t* nruns, uint64_t cap_runs, uint64_t* off,
                       uint64_t max_reads, uint64_t max_bases, uint64_t* n_reads, uint64_t* n_runs) {
    if (!r || !bases || !off || !n_reads || !n_runs) { set_error("null argument"); return -2; }
    if (max_reads == 0 || max_bases == 0 || max_bases >= 0xFFFFFFFFull) { set_error("max_reads must be > 0 and 0 < max_bases < 2^32"); return -2; }
    if (cap_bases_bytes < max_bases / 4 + 32) { set_error("bases buffer too small for max_bases"); return -2; }
    *n_reads = 0; *n_runs = 0;
    std::vector<const char*> ptr;
    std::vector<uint32_t> len;
    std::vector<std::shared_ptr<TextBuf>> keep;
    uint64_t nb = 0;
    while (ptr.size() < max_reads) {
        if (r->cur_i >= r->cur.start.size()) {
            if (r->eof) break;
            Lines nx;
            const auto tw0 = std::chrono::steady_clock::now();
            const bool got_lines = r->q_lines.pop(nx);
            r->t_wait_lines += std::chrono::duration<double>(std::chrono::steady_clock::now() - tw0).count();
            if (!got_lines) { r->eof = true; break; }
            r->tot_text += nx.text->size();
            r->cur = std::move(nx); r->cur_i = 0;
        }
        if (keep.empty() || keep.back() != r->cur.text) keep.push_back(r->cur.text);
        bool full = false;
        while (r->cur_i < r->cur.start.size() && ptr.size() < max_reads) {
            const uint32_t L = r->cur.len[r->cur_i];
            if (L > max_bases) { set_error("a read of %u bases does not fit a batch of %llu bases", L, (unsigned long long)max_bases); return -2; }
            if (nb + L > max_bases) { full = true; break; }
            ptr.push_back(r->cur.text->data() + r->cur.start[r->cur_i]);
            len.push_back(L);
            nb += L;
            ++r->cur_i;
        }
        if (full) break;
    }
    {
        std::lock_guard<std::mutex> g(r->err_mu);
        if (!r->io_error.empty()) { set_error("read error: %s", r->io_error.c_str()); return -3; }
    }
    const size_t n = ptr.size();
    if (n == 0) return 0;
    const auto tg0 = std::chrono::steady_clock::now();
    off[0] = 0;
    for (size_t i = 0; i < n; ++i) off[i + 1] = off[i] + len[i];
    // worker ranges: equal shares of the bases
    const int T = (int)std::min<size_t>((size_t)r->threads, std::max<size_t>(1, nb / 65536));
    std::vector<PackJob> jobs((size_t)T);
    size_t a = 0;
    for (int t = 0; t < T; ++t) {
        const uint64_t target = nb * (uint64_t)(t + 1) / (uint64_t)T;
        size_t b = (t == T - 1) ? n : (size_t)(std::upper_bound(off, off + n + 1, target) - off) - 1;
        if (b < a) b = a;
        jobs[(size_t)t] = PackJob{ptr.data(), len.data(), off, a, b, bases, {}};
        a = b;
    }
    // bytes two workers may both touch (and the padding) start out zero
    for (int t = 0; t < T; ++t) {
        const PackJob& j = jobs[(size_t)t];
        bases[off[j.a] >> 2] = 0;
        bases[off[j.b] >> 2] = 0;
    }
    const uint64_t used = (nb + 3) / 4, padded = (used + 15) / 16 * 16 + 16;
    memset(bases + used, 0, (size_t)std::min<uint64_t>(padded, cap_bases_bytes) - used);
    const auto tp0 = std::chrono::steady_clock::now();
    r->t_gather += std::chrono::duration<double>(tp0 - tg0).count();
    if (T == 1) pack_range(jobs[0]);
    else {
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back([&jobs, t] { pack_range(jobs[(size_t)t]); });
        pack_range(jobs[0]);
        for (auto& x : th) x.join();
    }
    r->t_pack += std::chrono::duration<double>(std::chrono::steady_clock::now() - tp0).count();
    // N runs of the workers, in stream order; runs that touch across a worker boundary are merged
    // A batch with more runs than the caller's buffer holds (very low-quality reads: KMC in the reference just skips N,
    // select_db.py:50) is still delivered: its runs stay with the reader and are fetched with mlgi_spilled_runs().
    uint64_t nr = 0, upper = 0;
    for (int t = 0; t < T; ++t) upper += jobs[(size_t)t].runs.size() / 2;
    const bool spill = upper > cap_runs || !nruns;
    if (spill) r->spill.assign((size_t)(2 * upper + 2), 0u);
    uint32_t* dst = spill ? r->spill.data() : nruns;
    for (int t = 0; t < T; ++t) {
        const std::vector<uint32_t>& v = jobs[(size_t)t].runs;
        for (size_t i = 0; i + 1 < v.size(); i += 2) {
            if (nr && (uint64_t)dst[2 * (nr - 1)] + dst[2 * (nr - 1) + 1] == v[i]) { dst[2 * (nr - 1) + 1] += v[i + 1]; continue; }
            dst[2 * nr] = v[i]; dst[2 * nr + 1] = v[i + 1];
            ++nr;
        }
    }
    if (spill) r->spill.resize((size_t)(2 * nr));
    *n_reads = n; *n_runs = nr;
    r->tot_reads += n; r->tot_bases += nb;
    return spill && nr ? 2 : 1;
}

MLGI_API int mlgi_spilled_runs(mlgi_reader* r, uint32_t* nruns, uint64_t cap_runs) {
    if (!r || !nruns) { set_error("null argument"); return -2; }
    if (cap_runs * 2 < r->spill.size()) { set_error("buffer holds %llu runs, %llu are waiting", (unsigned long long)cap_runs, (unsigned long long)(r->spill.size() / 2)); return -2; }
    if (!r->spill.empty()) memcpy(nruns, r->spill.data(), r->spill.size() * sizeof(uint32_t));
    r->spill.clear();
    return 0;
}

MLGI_API int mlgi_stats(mlgi_reader* r, uint64_t* reads, uint64_t* bases, uint64_t* text_bytes) {
    if (!r) { set_error("null reader"); return -2; }
    if (reads) *reads = r->tot_reads;
    if (bases) *bases = r->tot_bases;
    if (text_bytes) *text_bytes = r->tot_text;
    return 0;
}

// test hook (not in the header): gzip-decode in[0, n) with fast_inflate.h into out[0, cap), stopping and resuming every
// `step` output bytes.  Returns 0 and *out_n on success, -1 on a decoding error, -2 if cap is too small, -3 on a CRC /
// length mismatch.
MLGI_API int mlgi_test_inflate(const uint8_t* in, uint64_t n, uint8_t* out, uint64_t cap, uint64_t step, uint64_t* out_n) {
    std::unique_ptr<fastinf::Inflater> z(new fastinf::Inflater());
    z->in = in; z->in_end = in + n;
    uint8_t* o = out;
    uint8_t* member = out;
    for (;;) {
        if ((uint64_t)(o - out) + step + fastinf::SLACK > cap) return -2;
        const int rc = z->run(o, o + step, out);
        if (rc < 0) { set_error("%s", z->error ? z->error : "?"); return -1; }
        if (rc == 1) {
            if ((uint32_t)crc32(crc32(0L, Z_NULL, 0), member, (uInt)(o - member)) != z->crc_expected || (uint32_t)(o - member) != z->isize_expected) return -3;
            member = o;
        }
        if (rc == 2) break;
    }
    *out_n = (uint64_t)(o - out);
    return 0;
}

// ---- KMC database reader (kmcdb.h) ----
struct mlgi_kmcdb { kmcdb::Reader r; };
MLGI_API int mlgi_kmc_open(const char* prefix, mlgi_kmcdb** out) {
    if (!prefix || !out) { set_error("null argument"); return -2; }
    std::unique_ptr<mlgi_kmcdb> d(new mlgi_kmcdb());
    if (!d->r.open(prefix)) { set_error("%s", d->r.error.c_str()); return -3; }
    *out = d.release();
    return 0;
}
MLGI_API int mlgi_kmc_info(mlgi_kmcdb* d, uint32_t* k, uint64_t* total, uint32_t* counter_size, uint32_t* min_count, uint64_t* max_count,
                           int* canonical, uint32_t* version) {
    if (!d) { set_error("null database"); return -2; }
    const kmcdb::Info& i = d->r.info;
    if (k) *k = i.k;
    if (total) *total = i.total;
    if (counter_size) *counter_size = i.counter_size;
    if (min_count) *min_count = i.min_count;
    if (max_count) *max_count = i.max_count;
    if (canonical) *canonical = i.canonical ? 1 : 0;
    if (version) *version = i.version;
    return 0;
}
MLGI_API int mlgi_kmc_read(mlgi_kmcdb* d, uint64_t* keys, uint32_t* counts_or_null) {
    if (!d || !keys) { set_error("null argument"); return -2; }
    if (!d->r.read_all(keys, counts_or_null)) { set_error("%s", d->r.error.c_str()); return -3; }
    return 0;
}
MLGI_API void mlgi_kmc_close(mlgi_kmcdb* d) { delete d; }

MLGI_API void mlgi_close(mlgi_reader* r) {
    if (!r) return;
    if (getenv("MLGI_PROFILE"))
        fprintf(stderr, "mlgi: consumer waited %.3f s for lines, prepared %.3f s, packed %.3f s; scanner waited %.3f s for blocks\n",
                r->t_wait_lines, r->t_gather, r->t_pack, r->t_scan_wait);
    r->q_lines.abandon();
    r->q_raw.abandon();
    if (r->t_scan.joinable()) r->t_scan.join();
    if (r->t_read.joinable()) r->t_read.join();
    if (r->fh) gzclose(r->fh);
    if (r->fd >= 0) close(r->fd);
    delete r;
}

}  // extern "C"
