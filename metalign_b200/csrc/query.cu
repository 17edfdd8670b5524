// K2 / K3: from the set I of present database k-mers to the per-genome, per-k containment table.
// Replaces the per-record loop of CMash's StreamingQueryDNADatabase.py as Metalign calls it
// (scripts/select_db.py:73-76: `... 30-60-10 -c 0 -r 1000000 -v -f <bf> --sensitive`) up to the
// DataFrame tail: SURVEY.md 3.3 steps R4 (prefix matching, forward first / reverse complement only if
// the forward lookup is empty, smallest-k prefilter gate) and R5 (distinct hit prefixes per genome, k).
//
//   k_expand_hits   one warp per present k-mer x, one lane per offset: the ks[0]-mer at every offset is
//                   looked up forward and reverse-complemented in the sorted array P (bucketed binary
//                   search on the top key bits; a k-prefix is a key range, so every k is served by the
//                   same array); longer k's refine those ranges.  A hit ORs one bit: (k, class
//                   representative slot) -- set semantics, never a sum.
//                   The lane that sets a bit FIRST (atomicOr returned it clear) also adds 1 to num[genome][k]:
//                   the per-genome table is complete when this kernel ends.  (A separate popcount pass
//                   over the whole G*n-bit bitmap cost 0.17 ms at 2e5 genomes for ~2e5 set bits.)
//   k_finalize      containment = num / den in IEEE double where num > 0.
#include "mlg_internal.h"

namespace {

constexpr int WARPS_PER_CTA = 4;
constexpr int MAX_OFF = 64;

// entries of P whose leading k bases equal v: first index and count
__device__ __forceinline__ void prefix_range(const DbView& db, const key128& v, unsigned k, uint32_t& lo_out, uint32_t& cnt_out) {
    const unsigned K = db.K;
    const key128 lo_key = key_shl(v, 2 * (K - k));
    const uint32_t b = (uint32_t)key_shr(lo_key, 2 * K - db.pbits).lo;
    uint32_t lo = db.pidx[b], hi = db.pidx[b + 1];
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (key_lt(db.P_key[mid], lo_key)) lo = mid + 1; else hi = mid;
    }
    uint32_t e = lo;
    while (e < db.np && key_eq(key_prefix(db.P_key[e], K, k), v)) ++e;
    lo_out = lo; cnt_out = e - lo;
}

// ---- where a hit goes -----------------------------------------------------------------------------------------
// (a) query time, on the fly: straight into the hit bitmap (set semantics) and, on the first set, the count table
struct HitSink {
    uint32_t* hitbits;
    unsigned long long words_per_k;
    unsigned long long* num;      // G * nk
    __device__ __forceinline__ void set(const DbView& db, uint32_t ki, uint32_t r) const {
        const uint32_t bit = 1u << (r & 31u);
        const uint32_t old = atomicOr(&hitbits[(unsigned long long)ki * words_per_k + (r >> 5)], bit);
        if (!(old & bit)) atomicAdd(&num[(unsigned long long)(r / db.n) * db.nk + ki], 1ull);
    }
    __device__ __forceinline__ void mark(const DbView& db, uint32_t ki, uint32_t e, bool /*also_under_exact_gate*/) const {
        const unsigned long long total = (unsigned long long)db.G * db.n;
        set(db, ki, db.rep[(unsigned long long)ki * total + db.P_slot[e]]);
    }
};
// (b) database build: the hits of a database k-mer are a static function of the database, so they are expanded
//     ONCE for every k-mer of D (gate = none, each hit flagged with whether the exact gate would also let it
//     through) and kept as a record per k-mer; a query then only replays the records of the k-mers it found.
//     Record formats (word 0 = header; a hit word = representative slot | HIT_EXACT):
//       short      (header & 15) != 15: one 4-bit count per k (<= 14 each), then the hits grouped by k
//       same slot  header = 0xF | 1 << 4 | present-k mask << 8 | exact-k mask << 16, word 1 = the slot every hit names
//                  (the usual case: a k-mer of one genome whose prefixes are their own class representatives)
//       long       header = 0xF | 2 << 4, words 1..nk = count per k, then the hits grouped by k (k-mers shared by many genomes)
constexpr unsigned HCAP = 112;         // hits a short record can hold: 8 k values x 14
constexpr uint32_t HIT_EXACT = 0x80000000u;
constexpr uint32_t HREC_ESC = 15u, HREC_SAME = 1u, HREC_LONG = 2u;
constexpr unsigned HGROUP_SHIFT = MLG_HGROUP_SHIFT;  // record offsets are 32-bit words relative to a 64-bit base per 2^16 k-mers
// pass-1 summary word of a k-mer -> size of its record in words
__device__ __forceinline__ uint32_t hrec_size(uint32_t su) { return (su >> 30) == 1u ? 2u : (su & 0x3FFFFFFFu); }
// pass-1 sink: per-k counts, OR of the exact flags per k, smallest / largest slot named (all per warp, shared memory)
struct TallySink {
    uint32_t* cnt;                // [MLG_MAX_KS]
    uint32_t* ex;                 // bit k: some hit at k passes the exact gate
    uint32_t* rmin; uint32_t* rmax;
    __device__ __forceinline__ void mark(const DbView& db, uint32_t ki, uint32_t e, bool also_under_exact_gate) const {
        const unsigned long long total = (unsigned long long)db.G * db.n;
        const uint32_t r = db.rep[(unsigned long long)ki * total + db.P_slot[e]];
        atomicAdd(&cnt[ki], 1u);
        if (also_under_exact_gate) atomicOr(ex, 1u << ki);
        atomicMin(rmin, r); atomicMax(rmax, r);
    }
};
// pass-2 sinks: a short record is collected in shared memory, a long one is scattered straight into its place
struct CollectSink {
    uint32_t* val;                // [HCAP] per warp, shared memory: representative slot | HIT_EXACT
    unsigned char* kis;           // [HCAP]
    unsigned* n;                  // per warp
    __device__ __forceinline__ void mark(const DbView& db, uint32_t ki, uint32_t e, bool also_under_exact_gate) const {
        const unsigned long long total = (unsigned long long)db.G * db.n;
        const uint32_t r = db.rep[(unsigned long long)ki * total + db.P_slot[e]];
        const unsigned i = atomicAdd(n, 1u);
        if (i < HCAP) { val[i] = r | (also_under_exact_gate ? HIT_EXACT : 0u); kis[i] = (unsigned char)ki; }
    }
};
struct ScatterSink {
    uint32_t* dst;                // first hit word of the record
    uint32_t* cursor;             // [MLG_MAX_KS] per warp, shared memory: next free position per k
    __device__ __forceinline__ void mark(const DbView& db, uint32_t ki, uint32_t e, bool also_under_exact_gate) const {
        const unsigned long long total = (unsigned long long)db.G * db.n;
        const uint32_t r = db.rep[(unsigned long long)ki * total + db.P_slot[e]];
        dst[atomicAdd(&cursor[ki], 1u)] = r | (also_under_exact_gate ? HIT_EXACT : 0u);
    }
};

// all lanes of a warp: expand database k-mer x (SURVEY.md 3.3 R4).  gate_none = 0 applies the exact smallest-k gate.
template <class Sink>
__device__ __forceinline__ void expand_one(const DbView& db, const key128& x, int gate_none, const Sink& sink, unsigned lane,
                                           uint32_t* s_flo, uint32_t* s_fcnt, uint32_t* s_rlo, uint32_t* s_rcnt) {
    const unsigned K = db.K, k0 = db.ks[0], noff = K - k0 + 1;
    for (unsigned o = lane; o < noff; o += 32) {
        const key128 w = key_sub(x, K, o, k0);
        uint32_t lo, cnt;
        prefix_range(db, w, k0, lo, cnt);
        s_flo[o] = lo; s_fcnt[o] = cnt;
        prefix_range(db, key_rc(w, k0), k0, lo, cnt);
        s_rlo[o] = lo; s_rcnt[o] = cnt;
    }
    __syncwarp();
    for (unsigned o = lane; o < noff; o += 32) {
        const uint32_t fl = s_flo[o], fc = s_fcnt[o];
        const uint32_t rl = s_rlo[o], rc = s_rcnt[o];
        // smallest k: forward first, reverse complement only if forward is empty (no gate on this lookup)
        if (fc) { for (uint32_t e = fl; e < fl + fc; ++e) sink.mark(db, 0, e, true); }
        else    { for (uint32_t e = rl; e < rl + rc; ++e) sink.mark(db, 0, e, true); }
        const bool exact_ok = fc || rc;
        if (!(gate_none || exact_ok)) continue;
        for (uint32_t ki = 1; ki < db.nk; ++ki) {
            const unsigned k = db.ks[ki];
            if (o + k > K) continue;
            const key128 wk = key_sub(x, K, o, k);
            bool any = false;
            for (uint32_t e = fl; e < fl + fc; ++e)
                if (key_eq(key_prefix(db.P_key[e], K, k), wk)) { sink.mark(db, ki, e, exact_ok); any = true; }
            if (!any) {
                // rc(wk) starts with the reverse complement of the LAST k0 bases of wk: offset o + k - k0
                const unsigned o2 = o + k - k0;
                const uint32_t rl2 = s_rlo[o2], rc2 = s_rcnt[o2];
                const key128 rk = key_rc(wk, k);
                for (uint32_t e = rl2; e < rl2 + rc2; ++e)
                    if (key_eq(key_prefix(db.P_key[e], K, k), rk)) sink.mark(db, ki, e, exact_ok);
            }
        }
    }
    __syncwarp();
}

// on-the-fly expansion of the listed k-mers (all present ones, or those without a precomputed list)
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) k_expand_hits(DbView db, const uint32_t* __restrict__ present,
                                                                    const unsigned long long* __restrict__ d_n_present,
                                                                    int gate_none, HitSink hs) {
    __shared__ uint32_t s_flo[WARPS_PER_CTA][MAX_OFF], s_fcnt[WARPS_PER_CTA][MAX_OFF];
    __shared__ uint32_t s_rlo[WARPS_PER_CTA][MAX_OFF], s_rcnt[WARPS_PER_CTA][MAX_OFF];
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const unsigned long long n_present = *d_n_present;
    for (unsigned long long xi = (unsigned long long)blockIdx.x * WARPS_PER_CTA + warp; xi < n_present;
         xi += (unsigned long long)gridDim.x * WARPS_PER_CTA)
        expand_one(db, db.D_key[present[xi]], gate_none, hs, lane, s_flo[warp], s_fcnt[warp], s_rlo[warp], s_rcnt[warp]);
}

// database build, pass 1: tally the hits of every k-mer of D.  summary[2e] = kind << 30 | the record's size in words
// (kind 0 short, 2 long), or for kind 1 (same slot: always 2 words) 1 << 30 | the record's finished header with
// summary[2e + 1] = its slot -- such a record is complete after this pass.
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) k_tally_hits(DbView db, uint32_t* summary) {
    __shared__ uint32_t s_flo[WARPS_PER_CTA][MAX_OFF], s_fcnt[WARPS_PER_CTA][MAX_OFF];
    __shared__ uint32_t s_rlo[WARPS_PER_CTA][MAX_OFF], s_rcnt[WARPS_PER_CTA][MAX_OFF];
    __shared__ uint32_t s_cnt[WARPS_PER_CTA][MLG_MAX_KS], s_ex[WARPS_PER_CTA], s_min[WARPS_PER_CTA], s_max[WARPS_PER_CTA];
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    for (unsigned long long e = (unsigned long long)blockIdx.x * WARPS_PER_CTA + warp; e < db.nd;
         e += (unsigned long long)gridDim.x * WARPS_PER_CTA) {
        if (lane < MLG_MAX_KS) s_cnt[warp][lane] = 0;
        if (lane == 0) { s_ex[warp] = 0; s_min[warp] = 0xFFFFFFFFu; s_max[warp] = 0; }
        __syncwarp();
        TallySink sink{s_cnt[warp], &s_ex[warp], &s_min[warp], &s_max[warp]};
        expand_one(db, db.D_key[e], 1, sink, lane, s_flo[warp], s_fcnt[warp], s_rlo[warp], s_rcnt[warp]);
        if (lane == 0) {
            uint32_t n = 0, present = 0; bool fits = true;
            for (unsigned k = 0; k < MLG_MAX_KS; ++k) { const uint32_t c = s_cnt[warp][k]; n += c; if (c) present |= 1u << k; if (c > 14u) fits = false; }
            static_assert(MLG_MAX_KS <= 8, "the same-slot header has 8 bits per mask");
            if (n && s_min[warp] == s_max[warp]) {
                summary[2 * e] = (HREC_SAME << 30) | HREC_ESC | (HREC_SAME << 4) | (present << 8) | (s_ex[warp] << 16);
                summary[2 * e + 1] = s_min[warp];
            } else {
                summary[2 * e] = fits ? (1u + n) : ((HREC_LONG << 30) | (1u + db.nk + n));
                summary[2 * e + 1] = 0;
            }
        }
        __syncwarp();
    }
}
// record sizes -> offsets: sum per group of 2^HGROUP_SHIFT k-mers (one CTA per group), then -- after the group sums have
// been scanned into 64-bit bases -- the exclusive scan inside every group
__global__ void __launch_bounds__(256) k_hit_group_sums(const uint32_t* __restrict__ summary, uint32_t nd, unsigned long long* gsum) {
    __shared__ unsigned long long s_part[256];
    const unsigned long long g0 = (unsigned long long)blockIdx.x << HGROUP_SHIFT;
    unsigned long long acc = 0;
    for (unsigned long long i = g0 + threadIdx.x; i < g0 + (1ull << HGROUP_SHIFT) && i < nd; i += 256) acc += hrec_size(summary[2 * i]);
    s_part[threadIdx.x] = acc;
    __syncthreads();
    for (unsigned o = 128; o; o >>= 1) { if (threadIdx.x < o) s_part[threadIdx.x] += s_part[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) gsum[blockIdx.x] = s_part[0];
}
__global__ void __launch_bounds__(256) k_hit_offsets(const uint32_t* __restrict__ summary, uint32_t nd, uint32_t* hoff) {
    // every thread owns 256 consecutive k-mers of the group: local sums, a scan over the 256 threads, then the offsets
    __shared__ uint32_t s_tot[256];
    const unsigned long long g0 = (unsigned long long)blockIdx.x << HGROUP_SHIFT;
    const unsigned long long a = g0 + (unsigned long long)threadIdx.x * 256ull;
    uint32_t acc = 0;
    for (unsigned long long i = a; i < a + 256ull && i < nd; ++i) acc += hrec_size(summary[2 * i]);
    s_tot[threadIdx.x] = acc;
    __syncthreads();
    for (unsigned o = 1; o < 256; o <<= 1) {
        const uint32_t v = threadIdx.x >= o ? s_tot[threadIdx.x - o] : 0u;
        __syncthreads();
        s_tot[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t off = s_tot[threadIdx.x] - acc;
    for (unsigned long long i = a; i < a + 256ull && i < nd; ++i) { hoff[i] = off; off += hrec_size(summary[2 * i]); }
}
// database build, pass 2: write the records.  Same-slot records come straight from the summary; the others are expanded
// again (short: collected in shared memory; long: tallied for the per-k counts, then scattered into place).  drop_from:
// records that start at or beyond this word are not written and their k-mer is marked HOFF_NONE (tests of the
// on-the-fly path).
__global__ void __launch_bounds__(WARPS_PER_CTA * 32) k_fill_hits(DbView db, const uint32_t* __restrict__ summary, uint32_t* hoff,
                                                                  const unsigned long long* __restrict__ hbase, uint32_t* hits,
                                                                  unsigned long long drop_from) {
    __shared__ uint32_t s_flo[WARPS_PER_CTA][MAX_OFF], s_fcnt[WARPS_PER_CTA][MAX_OFF];
    __shared__ uint32_t s_rlo[WARPS_PER_CTA][MAX_OFF], s_rcnt[WARPS_PER_CTA][MAX_OFF];
    __shared__ uint32_t s_val[WARPS_PER_CTA][HCAP];
    __shared__ unsigned char s_ki[WARPS_PER_CTA][HCAP];
    __shared__ unsigned s_n[WARPS_PER_CTA];
    __shared__ uint32_t s_cnt[WARPS_PER_CTA][MLG_MAX_KS], s_ex[WARPS_PER_CTA], s_min[WARPS_PER_CTA], s_max[WARPS_PER_CTA];
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    for (unsigned long long e = (unsigned long long)blockIdx.x * WARPS_PER_CTA + warp; e < db.nd;
         e += (unsigned long long)gridDim.x * WARPS_PER_CTA) {
        const uint32_t su = summary[2 * e], kind = su >> 30;
        const unsigned long long at = hbase[e >> HGROUP_SHIFT] + hoff[e];
        if (at >= drop_from) { if (lane == 0) hoff[e] = HOFF_NONE; continue; }
        uint32_t* rec = hits + at;
        if (kind == HREC_SAME) {
            if (lane == 0) { rec[0] = su & 0x3FFFFFFFu; rec[1] = summary[2 * e + 1]; }
            continue;
        }
        const key128 x = db.D_key[e];
        if (kind == 0) {
            if (lane == 0) s_n[warp] = 0;
            __syncwarp();
            CollectSink sink{s_val[warp], s_ki[warp], &s_n[warp]};
            expand_one(db, x, 1, sink, lane, s_flo[warp], s_fcnt[warp], s_rlo[warp], s_rcnt[warp]);
            if (lane == 0) {
                const unsigned n = s_n[warp] < HCAP ? s_n[warp] : HCAP;      // == the tally of pass 1
                unsigned cnt[MLG_MAX_KS], start[MLG_MAX_KS], acc = 0;
                for (unsigned k = 0; k < MLG_MAX_KS; ++k) cnt[k] = 0;
                for (unsigned i = 0; i < n; ++i) cnt[s_ki[warp][i]]++;
                uint32_t hdr = 0;
                for (unsigned k = 0; k < MLG_MAX_KS; ++k) { hdr |= cnt[k] << (4 * k); start[k] = acc; acc += cnt[k]; }
                rec[0] = hdr;
                for (unsigned i = 0; i < n; ++i) rec[1 + start[s_ki[warp][i]]++] = s_val[warp][i];
            }
        } else {
            if (lane < MLG_MAX_KS) s_cnt[warp][lane] = 0;
            if (lane == 0) { s_ex[warp] = 0; s_min[warp] = 0xFFFFFFFFu; s_max[warp] = 0; }
            __syncwarp();
            TallySink tally{s_cnt[warp], &s_ex[warp], &s_min[warp], &s_max[warp]};
            expand_one(db, x, 1, tally, lane, s_flo[warp], s_fcnt[warp], s_rlo[warp], s_rcnt[warp]);
            if (lane == 0) {
                rec[0] = HREC_ESC | (HREC_LONG << 4);
                uint32_t acc = 0;
                for (unsigned k = 0; k < db.nk; ++k) { const uint32_t c = s_cnt[warp][k]; rec[1 + k] = c; s_cnt[warp][k] = acc; acc += c; }
            }
            __syncwarp();
            ScatterSink sc{rec + 1 + db.nk, s_cnt[warp]};
            expand_one(db, x, 1, sc, lane, s_flo[warp], s_fcnt[warp], s_rlo[warp], s_rcnt[warp]);
        }
        __syncwarp();
    }
}

// query time: replay the precomputed records of the present k-mers; k-mers without one are queued for the on-the-fly kernel
__global__ void k_apply_hits(DbView db, const uint32_t* __restrict__ present, const unsigned long long* __restrict__ d_n_present,
                             int gate_none, HitSink hs, const uint32_t* __restrict__ hoff, const unsigned long long* __restrict__ hbase,
                             const uint32_t* __restrict__ hits, uint32_t* fallback, unsigned long long* n_fallback) {
    const unsigned long long n_present = *d_n_present;
    for (unsigned long long xi = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; xi < n_present;
         xi += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t e = present[xi];
        const uint32_t off = hoff[e];
        if (off == HOFF_NONE) { fallback[atomicAdd(n_fallback, 1ull)] = e; continue; }
        const uint32_t* hp = hits + hbase[e >> HGROUP_SHIFT] + off;
        uint32_t hdr = *hp++;
        if ((hdr & 15u) != HREC_ESC) {
            for (uint32_t ki = 0; ki < db.nk; ++ki, hdr >>= 4)
                for (uint32_t c = hdr & 15u; c; --c) {
                    const uint32_t v = *hp++;
                    if (gate_none || (v & HIT_EXACT)) hs.set(db, ki, v & ~HIT_EXACT);
                }
        } else if (((hdr >> 4) & 15u) == HREC_SAME) {
            const uint32_t r = *hp;
            const uint32_t take = gate_none ? (hdr >> 8) & 0xFFu : (hdr >> 8) & (hdr >> 16) & 0xFFu;
            for (uint32_t ki = 0; ki < db.nk; ++ki) if ((take >> ki) & 1u) hs.set(db, ki, r);
        } else {
            const uint32_t* cp = hp;
            hp += db.nk;
            for (uint32_t ki = 0; ki < db.nk; ++ki)
                for (uint32_t c = cp[ki]; c; --c) {
                    const uint32_t v = *hp++;
                    if (gate_none || (v & HIT_EXACT)) hs.set(db, ki, v & ~HIT_EXACT);
                }
        }
    }
}

__global__ void k_finalize(const unsigned long long* num, const long long* den_real, const unsigned char* has_empty, uint32_t G,
                           uint32_t nk, int count_empty, long long* out_num, long long* out_den, double* out_ci) {
    unsigned long long c = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (c >= (unsigned long long)G * nk) return;
    uint32_t g = (uint32_t)(c / nk);
    long long nu = (long long)num[c];
    long long de = den_real[c] + ((count_empty && has_empty[g]) ? 1 : 0);
    out_num[c] = nu; out_den[c] = de;
    out_ci[c] = nu > 0 ? (double)nu / (double)de : 0.0;
}

// sparse form of the result: one row per genome with a hit at any k (unordered; the caller sorts the few rows by genome)
__global__ void k_finalize_sparse(const unsigned long long* num, const long long* den_real, const unsigned char* has_empty, uint32_t G,
                                  uint32_t nk, int count_empty, uint32_t* out_g, long long* out_num, long long* out_den, double* out_ci,
                                  unsigned long long cap, unsigned long long* counter) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    unsigned long long any = 0;
    for (uint32_t k = 0; k < nk; ++k) any |= num[(size_t)g * nk + k];
    if (!any) return;
    const unsigned long long r = atomicAdd(counter, 1ull);
    if (r >= cap) return;
    out_g[r] = g;
    const long long extra = (count_empty && has_empty[g]) ? 1 : 0;
    for (uint32_t k = 0; k < nk; ++k) {
        const long long nu = (long long)num[(size_t)g * nk + k], de = den_real[(size_t)g * nk + k] + extra;
        out_num[r * nk + k] = nu; out_den[r * nk + k] = de;
        out_ci[r * nk + k] = nu > 0 ? (double)nu / (double)de : 0.0;
    }
}
// put a query's counter table back to all zeros by visiting only the counters it touched (the table is >99.9 % zeros)
__global__ void k_clear_touched(unsigned char* cnt8, const uint32_t* __restrict__ touched, const unsigned long long* __restrict__ d_n) {
    const unsigned long long n = *d_n;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x)
        cnt8[touched[i]] = 0;
}
// clamp the counters that are non-zero (listed in touched[]) to `clamp` (ci_min unless the query set another level):
// what a rank contributes to the cross-rank sum
__global__ void k_clamp_counts(unsigned char* cnt8, const uint32_t* __restrict__ touched, const unsigned long long* __restrict__ d_n,
                               uint32_t clamp) {
    const unsigned long long n = *d_n;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t e = touched[i];
        if (cnt8[e] > clamp) cnt8[e] = (unsigned char)clamp;
    }
}
// a rank's own counter clamped to `clamp` in place, as its contribution to the cross-rank sum: after a merge the table
// holds sum over ranks of min(count, clamp) on every rank, the same as the dense form (k_clamp_counts) leaves it
__device__ __forceinline__ uint32_t clamp_own(unsigned char* cnt8, uint32_t e, uint32_t clamp) {
    const uint32_t c = cnt8[e];
    if (c <= clamp) return c;
    cnt8[e] = (unsigned char)clamp;
    return clamp;
}
// sparse form of a rank's contribution: one 64-bit entry per non-zero counter = index | min(count, clamp) << 32
__global__ void k_pack_touched(unsigned char* cnt8, const uint32_t* __restrict__ touched,
                               const unsigned long long* __restrict__ d_n, uint32_t clamp, unsigned long long* out) {
    const unsigned long long n = *d_n;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t e = touched[i];
        out[i] = (unsigned long long)e | ((unsigned long long)clamp_own(cnt8, e, clamp) << 32);
    }
}
// add another rank's sparse entries into this rank's counters (saturating); a counter that crosses ci_min joins present[]
__global__ void k_merge_sparse(unsigned char* cnt8, const unsigned long long* __restrict__ entries, unsigned long long n, uint32_t nd,
                               uint32_t ci_min, uint32_t* present, uint32_t* touched, unsigned long long* cursors) {
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long en = entries[i];
        const uint32_t e = (uint32_t)en, c = (uint32_t)(en >> 32);
        if (c == 0u || e >= nd) continue;
        uint32_t* wp = reinterpret_cast<uint32_t*>(cnt8) + (e >> 2);
        const uint32_t sh = (e & 3u) * 8u;
        uint32_t old = *reinterpret_cast<volatile uint32_t*>(wp);
        for (;;) {
            const uint32_t before = (old >> sh) & 0xFFu;
            const uint32_t after = before + c > 255u ? 255u : before + c;
            if (after == before) break;
            const uint32_t assumed = old;
            old = atomicCAS(wp, assumed, (assumed & ~(0xFFu << sh)) | (after << sh));
            if (old == assumed) {
                if (before == 0u) touched[atomicAdd(cursors + 1, 1ull)] = e;
                if (before < ci_min && after >= ci_min) present[atomicAdd(cursors, 1ull)] = e;
                break;
            }
        }
    }
}
// ---- the multi-GPU exchange without a host round trip (mlg_exchange, capi.cu) --------------------------------------
// A rank's contribution travels as one BLOCK of block_words 64-bit words: word 0 = number of non-zero counters n
// (| epoch << 40 on the direct path), word 1 unused, then min(n, cap) entries index | min(count, clamp) << 32.
// Both pack kernels clamp ALL n own counters (not only the first cap) and leave n in *own_count, the count the merge
// judges this rank's block by: the merge itself appends to touched[] and so cannot read n there.
constexpr unsigned long long XCNT_MASK = (1ull << 40) - 1ull;
// fill this rank's block in local memory (the caller all-gathers the blocks, e.g. with NCCL)
__global__ void k_pack_exchange(unsigned char* cnt8, const uint32_t* __restrict__ touched, const unsigned long long* __restrict__ d_n,
                                uint32_t clamp, unsigned long long* out, unsigned long long cap, unsigned long long* own_count) {
    const unsigned long long n = *d_n;
    if (blockIdx.x == 0 && threadIdx.x == 0) { out[0] = n; out[1] = 0; *own_count = n; }
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t e = touched[i];
        const uint32_t c = clamp_own(cnt8, e, clamp);
        if (i < cap) out[2 + i] = (unsigned long long)e | ((unsigned long long)c << 32);
    }
}
// direct path: store the block straight into every peer's mailbox over NVLink (peer-mapped pointers), then -- once every
// CTA's stores are fenced -- publish count | epoch << 40 in word 0 of each copy with a system-scope release
struct PeerBoxes { unsigned long long* box[MLG_MAX_RANKS]; uint32_t n; };
__global__ void k_push_peers(unsigned char* cnt8, const uint32_t* __restrict__ touched, const unsigned long long* __restrict__ d_n,
                             uint32_t clamp, PeerBoxes pb, unsigned long long cap, unsigned long long epoch, unsigned int* done_ctas,
                             unsigned long long* own_count) {
    const unsigned long long n = *d_n;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t e = touched[i];
        const uint32_t c = clamp_own(cnt8, e, clamp);
        if (i >= cap) continue;
        const unsigned long long en = (unsigned long long)e | ((unsigned long long)c << 32);
        for (uint32_t p = 0; p < pb.n; ++p) pb.box[p][2 + i] = en;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(done_ctas, 1u);
        if (t == gridDim.x - 1u) {                       // the last CTA: every other CTA's stores are fenced before its increment
            *done_ctas = 0u;
            *own_count = n;
            __threadfence_system();
            const unsigned long long flag = (n & XCNT_MASK) | (epoch << 40);
            for (uint32_t p = 0; p < pb.n; ++p)
                asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(pb.box[p]), "l"(flag) : "memory");
        }
    }
}
// add every OTHER rank's block into this rank's counters (saturating); a counter that crosses ci_min joins present[].
// recv + w * stride_words = block of rank w.  epoch != 0: the blocks were stored by the peers themselves -- wait for word 0
// of each to carry this epoch (bounded by timeout_ns).  If any rank had more entries than a block holds, NOTHING is merged
// and status[0] = the largest count (the caller repeats the exchange with larger blocks); status[1] = 1 on a timeout.
// The verdict covers all world counts, this rank's own (status[3], left by the pack kernel) included, so that every rank
// reaches the same one: a rank that alone overflowed must repeat the exchange together with its peers.
__global__ void k_merge_exchange(unsigned char* cnt8, const unsigned long long* recv, unsigned long long stride_words, uint32_t world,
                                 uint32_t rank, unsigned long long cap, uint32_t nd, uint32_t ci_min, uint32_t* present, uint32_t* touched,
                                 unsigned long long* cursors, unsigned long long* status, unsigned long long epoch,
                                 unsigned long long timeout_ns) {
    __shared__ unsigned long long s_cnt[MLG_MAX_RANKS];
    __shared__ int s_bad;
    if (threadIdx.x == 0) s_bad = 0;
    __syncthreads();
    if (threadIdx.x < world) {
        const uint32_t w = threadIdx.x;
        unsigned long long v = 0;
        if (w == rank) {
            v = __ldcg(status + 3);
            if (v > cap) atomicMax(&s_bad, 1);
        } else {
            const unsigned long long* fp = recv + (unsigned long long)w * stride_words;
            if (epoch) {
                unsigned long long t0, t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                for (;;) {
                    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(fp) : "memory");
                    if ((v >> 40) == epoch) break;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t1 - t0 > timeout_ns) { s_bad = 2; v = 0; break; }
                    __nanosleep(200);
                }
            } else {
                v = __ldcg(fp);
            }
            v &= XCNT_MASK;
            if (v > cap) atomicMax(&s_bad, 1);
        }
        s_cnt[w] = v;
    }
    __syncthreads();
    if (s_bad) {
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            unsigned long long mx = 0;
            for (uint32_t w = 0; w < world; ++w) mx = s_cnt[w] > mx ? s_cnt[w] : mx;
            if (s_bad == 2) status[1] = 1; else status[0] = mx;
        }
        return;
    }
    const unsigned long long total = (unsigned long long)world * cap;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t w = (uint32_t)(i / cap);
        const unsigned long long k = i - (unsigned long long)w * cap;
        if (w == rank || k >= s_cnt[w]) continue;         // the own counters are in the table already
        const unsigned long long en = __ldcg(recv + (unsigned long long)w * stride_words + 2ull + k);
        const uint32_t e = (uint32_t)en, c = (uint32_t)(en >> 32);
        if (c == 0u || e >= nd) continue;
        uint32_t* wp = reinterpret_cast<uint32_t*>(cnt8) + (e >> 2);
        const uint32_t sh = (e & 3u) * 8u;
        uint32_t old = *reinterpret_cast<volatile uint32_t*>(wp);
        for (;;) {
            const uint32_t before = (old >> sh) & 0xFFu;
            const uint32_t after = before + c > 255u ? 255u : before + c;
            if (after == before) break;
            const uint32_t assumed = old;
            old = atomicCAS(wp, assumed, (assumed & ~(0xFFu << sh)) | (after << sh));
            if (old == assumed) {
                if (before == 0u) touched[atomicAdd(cursors + 1, 1ull)] = e;
                if (before < ci_min && after >= ci_min) present[atomicAdd(cursors, 1ull)] = e;
                break;
            }
        }
    }
}
// present[] = indices of the counters >= ci_min; 16 counters per thread and step (the table is almost all zeros)
__global__ void k_compact_present(const uint4* __restrict__ cnt16, uint32_t nd, uint32_t ci_min, uint32_t* out, unsigned long long* cursor) {
    const unsigned long long nvec = ((unsigned long long)nd + 15ull) / 16ull;       // the table is padded to 16 bytes with zeros
    for (unsigned long long v = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; v < nvec; v += (unsigned long long)gridDim.x * blockDim.x) {
        const uint4 q = cnt16[v];
        if ((q.x | q.y | q.z | q.w) == 0u) continue;
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
        uint32_t hits[16]; unsigned nh = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const unsigned long long idx = v * 16ull + 4 * k + b;
                if (((w[k] >> (8 * b)) & 0xFFu) >= ci_min && idx < nd) hits[nh++] = (uint32_t)idx;
            }
        if (nh) {
            const unsigned long long base = atomicAdd(cursor, (unsigned long long)nh);
            for (unsigned h = 0; h < nh; ++h) out[base + h] = hits[h];
        }
    }
}
// N runs -> N mask.  One thread per (start, length) run; bit i of the mask lives in byte i/8, bit 7-(i%8).
__global__ void k_scatter_nruns(const uint32_t* __restrict__ runs, unsigned long long n_runs, unsigned long long nbases,
                                uint32_t* mask_words) {
    unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    if (t >= n_runs) return;
    unsigned long long a = runs[2 * t], b = a + runs[2 * t + 1];
    if (b > nbases) b = nbases;
    while (a < b) {
        const unsigned long long byte = a >> 3;
        const unsigned first = (unsigned)(a & 7ull);
        unsigned long long stop = (byte + 1) << 3;
        if (stop > b) stop = b;
        const unsigned cnt = (unsigned)(stop - a);                       // bits first .. first+cnt-1, MSB first
        const uint32_t m = ((0xFFu >> first) & (0xFFu << (8u - first - cnt))) & 0xFFu;
        atomicOr(&mask_words[byte >> 2], m << (8u * (unsigned)(byte & 3ull)));
        a = stop;
    }
}
__global__ void k_gather_present_keys(const key128* D_key, const uint32_t* present, uint32_t n_present, key128* out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_present) out[i] = D_key[present[i]];
}
// what `kmc_tools simple <db> <reads> intersect` keeps as a k-mer's counter: the smaller of its two counters, each of
// which saturated at `cap` (-cs) when its database was written
__global__ void k_gather_present_counts(const unsigned char* cnt8, const unsigned char* D_mult, const uint32_t* present, uint32_t n_present,
                                        uint32_t cap, unsigned char* out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_present) return;
    const uint32_t d = present[i];
    uint32_t c = cnt8[d];
    if (D_mult) c = min(c, (uint32_t)D_mult[d]);
    out[i] = (unsigned char)min(c, cap);
}
// hit flags of whole genomes: out[(i * nk + ki) * n + j] = 1 where slot j of genomes[i] is the representative of a
// (genome, k-prefix) class that the query hit at ks[ki]
__global__ void k_gather_hit_flags(const uint32_t* hitbits, unsigned long long words_per_k, const uint32_t* genomes, uint32_t m,
                                   uint32_t n, uint32_t nk, unsigned char* out) {
    const unsigned long long t = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    const unsigned long long cells = (unsigned long long)m * nk * n;
    if (t >= cells) return;
    const uint32_t j = (uint32_t)(t % n), ki = (uint32_t)((t / n) % nk), i = (uint32_t)(t / ((unsigned long long)n * nk));
    const unsigned long long slot = (unsigned long long)genomes[i] * n + j;
    out[t] = (unsigned char)((hitbits[(unsigned long long)ki * words_per_k + (slot >> 5)] >> (slot & 31ull)) & 1u);
}

}  // namespace

int launch_clamp_counts(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp, cudaStream_t st) {
    k_clamp_counts<<<148u * 4u, 256, 0, st>>>(cnt8, touched, d_n_touched, clamp);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_pack_touched(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp,
                        unsigned long long* out, cudaStream_t st) {
    k_pack_touched<<<148u * 4u, 256, 0, st>>>(cnt8, touched, d_n_touched, clamp, out);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_merge_sparse(unsigned char* cnt8, const unsigned long long* entries, unsigned long long n, uint32_t nd, uint32_t ci_min,
                        uint32_t* present, uint32_t* touched, unsigned long long* d_cursors, cudaStream_t st) {
    if (!n) return MLG_OK;
    unsigned long long want = (n + 255) / 256;
    k_merge_sparse<<<(unsigned)(want < 148ull * 8ull ? want : 148ull * 8ull), 256, 0, st>>>(cnt8, entries, n, nd, ci_min, present, touched, d_cursors);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_pack_exchange(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp,
                         unsigned long long* out, unsigned long long cap, unsigned long long* own_count, cudaStream_t st) {
    k_pack_exchange<<<148u * 2u, 256, 0, st>>>(cnt8, touched, d_n_touched, clamp, out, cap, own_count);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_push_peers(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, uint32_t clamp,
                      unsigned long long* const* boxes, uint32_t n_peers, unsigned long long cap, unsigned long long epoch,
                      unsigned int* done_ctas, unsigned long long* own_count, cudaStream_t st) {
    PeerBoxes pb{};
    pb.n = n_peers;
    for (uint32_t p = 0; p < n_peers && p < MLG_MAX_RANKS; ++p) pb.box[p] = boxes[p];
    k_push_peers<<<148u, 256, 0, st>>>(cnt8, touched, d_n_touched, clamp, pb, cap, epoch, done_ctas, own_count);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_merge_exchange(unsigned char* cnt8, const unsigned long long* recv, unsigned long long stride_words, uint32_t world, uint32_t rank,
                          unsigned long long cap, uint32_t nd, uint32_t ci_min, uint32_t* present, uint32_t* touched,
                          unsigned long long* d_cursors, unsigned long long* d_status, unsigned long long epoch,
                          unsigned long long timeout_ns, cudaStream_t st) {
    static_assert(MLG_MAX_RANKS <= 256, "one thread per rank reads the block headers");
    k_merge_exchange<<<148u * 4u, 256, 0, st>>>(cnt8, recv, stride_words, world, rank, cap, nd, ci_min, present, touched, d_cursors,
                                              d_status, epoch, timeout_ns);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_compact_present(const unsigned char* cnt8, uint32_t nd, uint32_t ci_min, uint32_t* out, unsigned long long* d_cursor,
                           cudaStream_t st) {
    CUDA_TRY(cudaMemsetAsync(d_cursor, 0, 8, st));
    if (!nd) return MLG_OK;
    k_compact_present<<<148u * 8u, 256, 0, st>>>(reinterpret_cast<const uint4*>(cnt8), nd, ci_min, out, d_cursor);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_expand_hits(const DbView& db, const uint32_t* present, const unsigned long long* d_n_present, int gate_none,
                       uint32_t* hitbits, unsigned long long words_per_k, unsigned long long* num, cudaStream_t st) {
    // persistent grid: |I| is only known on the device (no host round trip between the probe and this kernel)
    HitSink hs{hitbits, words_per_k, num};
    k_expand_hits<<<148u * 16u, WARPS_PER_CTA * 32, 0, st>>>(db, present, d_n_present, gate_none, hs);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_apply_hits(const DbView& db, const uint32_t* present, const unsigned long long* d_n_present, int gate_none,
                      uint32_t* hitbits, unsigned long long words_per_k, unsigned long long* num, const uint32_t* hoff,
                      const unsigned long long* hbase, const uint32_t* hits, uint32_t* fallback, unsigned long long* d_n_fallback,
                      cudaStream_t st) {
    HitSink hs{hitbits, words_per_k, num};
    CUDA_TRY(cudaMemsetAsync(d_n_fallback, 0, 8, st));
    k_apply_hits<<<148u * 4u, 256, 0, st>>>(db, present, d_n_present, gate_none, hs, hoff, hbase, hits, fallback, d_n_fallback);
    CUDA_TRY(cudaGetLastError());
    // whatever had no record is expanded on the fly (only databases that kept P can have such k-mers)
    if (db.P_key) {
        k_expand_hits<<<148u * 16u, WARPS_PER_CTA * 32, 0, st>>>(db, fallback, d_n_fallback, gate_none, hs);
        CUDA_TRY(cudaGetLastError());
    }
    return MLG_OK;
}
int launch_tally_hits(const DbView& db, uint32_t* summary, cudaStream_t st) {
    if (!db.nd) return MLG_OK;
    k_tally_hits<<<148u * 16u, WARPS_PER_CTA * 32, 0, st>>>(db, summary);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_hit_group_sums(const uint32_t* summary, uint32_t nd, unsigned long long* gsum, cudaStream_t st) {
    const unsigned groups = (unsigned)(((unsigned long long)nd + (1ull << HGROUP_SHIFT) - 1) >> HGROUP_SHIFT);
    if (!groups) return MLG_OK;
    k_hit_group_sums<<<groups, 256, 0, st>>>(summary, nd, gsum);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_hit_offsets(const uint32_t* summary, uint32_t nd, uint32_t* hoff, cudaStream_t st) {
    const unsigned groups = (unsigned)(((unsigned long long)nd + (1ull << HGROUP_SHIFT) - 1) >> HGROUP_SHIFT);
    if (!groups) return MLG_OK;
    static_assert((1u << HGROUP_SHIFT) == 256u * 256u, "k_hit_offsets: 256 threads x 256 k-mers per group");
    k_hit_offsets<<<groups, 256, 0, st>>>(summary, nd, hoff);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_fill_hits(const DbView& db, const uint32_t* summary, uint32_t* hoff, const unsigned long long* hbase,
                     uint32_t* hits, unsigned long long drop_from, cudaStream_t st) {
    if (!db.nd) return MLG_OK;
    k_fill_hits<<<148u * 16u, WARPS_PER_CTA * 32, 0, st>>>(db, summary, hoff, hbase, hits, drop_from);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_scatter_nruns(const uint32_t* d_runs, unsigned long long n_runs, unsigned long long nbases, unsigned char* nmask,
                         cudaStream_t st) {
    if (!n_runs) return MLG_OK;
    k_scatter_nruns<<<(unsigned)((n_runs + 255) / 256), 256, 0, st>>>(d_runs, n_runs, nbases, reinterpret_cast<uint32_t*>(nmask));
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_finalize(const unsigned long long* num, const long long* den_real, const unsigned char* has_empty, uint32_t G,
                    uint32_t nk, int count_empty, long long* out_num, long long* out_den, double* out_ci, cudaStream_t st) {
    unsigned long long cells = (unsigned long long)G * nk;
    k_finalize<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(num, den_real, has_empty, G, nk, count_empty, out_num, out_den, out_ci);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_finalize_sparse(const unsigned long long* num, const long long* den_real, const unsigned char* has_empty, uint32_t G, uint32_t nk,
                           int count_empty, uint32_t* out_g, long long* out_num, long long* out_den, double* out_ci, unsigned long long cap,
                           unsigned long long* d_counter, cudaStream_t st) {
    CUDA_TRY(cudaMemsetAsync(d_counter, 0, 8, st));
    k_finalize_sparse<<<(G + 255) / 256, 256, 0, st>>>(num, den_real, has_empty, G, nk, count_empty, out_g, out_num, out_den, out_ci, cap, d_counter);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_clear_touched(unsigned char* cnt8, const uint32_t* touched, const unsigned long long* d_n_touched, cudaStream_t st) {
    k_clear_touched<<<148u * 2u, 256, 0, st>>>(cnt8, touched, d_n_touched);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_gather_keys(const key128* D_key, const uint32_t* present, uint32_t n_present, key128* out, cudaStream_t st) {
    if (!n_present) return MLG_OK;
    k_gather_present_keys<<<(n_present + 255) / 256, 256, 0, st>>>(D_key, present, n_present, out);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_gather_counts(const unsigned char* cnt8, const unsigned char* D_mult, const uint32_t* present, uint32_t n_present, uint32_t cap,
                         unsigned char* out, cudaStream_t st) {
    if (!n_present) return MLG_OK;
    k_gather_present_counts<<<(n_present + 255) / 256, 256, 0, st>>>(cnt8, D_mult, present, n_present, cap, out);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
int launch_gather_hit_flags(const uint32_t* hitbits, unsigned long long words_per_k, const uint32_t* genomes, uint32_t m, uint32_t n,
                            uint32_t nk, unsigned char* out, cudaStream_t st) {
    const unsigned long long cells = (unsigned long long)m * nk * n;
    if (!cells) return MLG_OK;
    k_gather_hit_flags<<<(unsigned)((cells + 255) / 256), 256, 0, st>>>(hitbits, words_per_k, genomes, m, n, nk, out);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}
