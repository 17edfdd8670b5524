// MZ_RT: threads per CTA of this kernel alone (every warp is its own pipeline, so the CTA size only sets how the
// register file and shared memory are cut up); the other K1 kernels keep 256
#ifdef MZ_RT
#define MLG_RT MZ_RT
#endif
#include "probe_common.cuh"

namespace {

// ======================================================================================================
// K1, minimizer-bitmap layout (db.layout == 2, K == 60; definitions in kmer.cuh).  Same lane-per-read walk and
// per-warp TMA pipelines as the super-k-mer kernel above, but the minimizer is a 32-mer whose (order << 6 | position)
// value is two multiply-adds, level 1 is a bit array over minimizer IDENTITIES, and there is no per-window compare:
//   phase A  sliding minimum over the 29 32-mers under each window (van Herk / Gil-Werman on blocks of 16 positions)
//            and the runs of equal minimizer, block by block; every run start goes to the lane's run list in shared
//            memory (one byte: the minimizer's position relative to the run's first block) and to a 96-bit mask of the
//            segment's run starts in registers;
//   lookup   after the segment's blocks, the warp walks the lists slot by slot up to its longest one: the lane fetches the
//            two halves of its run's minimizer from its copy of the segment in shared memory, mixes their identity and
//            loads the bit-array word (predicated LDG), MZ_LGROUP slots' loads in flight before the first is looked at;
//            a run whose two bits are set becomes ITEMS (stream position of a block's first window, 16-bit mask of the
//            run's valid windows in that block, minimizer position) in a per-warp list in shared memory, one item for
//            each block of 16 windows the run touches (a run covers at most 29 windows: at most 3 items).
// Items are rare (bit density <= 1/32, plus the true hits); the ring is drained 32 at a time, one item per lane: the
// lane rebuilds the canonical key of each window of the item from the staged bases and compares it with the database
// k-mers filed under that identity (bucket index on the identity's high word, plus the alias table).
#ifndef MZ_MINCTAS
#define MZ_MINCTAS 2
#endif
// slots looked up together: their loads are all issued before the first word is looked at.  8 was slower on a B200
// (K1 1.98 against 1.90 ms: ~13 slots per read round up to 16, and twice the unrolled code)
constexpr unsigned MZ_LGROUP = 4;
constexpr unsigned MZ_QDRAIN = 32;            // per-warp item list: drained whenever this many are waiting ...
constexpr unsigned MZ_QCAP = MZ_QDRAIN + 128; // ... and one run adds at most 3 x 32
constexpr unsigned MZ_LIST = 64;              // run list slots per lane (bytes)
constexpr unsigned MZ_CAP = MZ_LIST - 16;     // runs of a segment that are looked up: a block's 16 stores start at slot <= MZ_CAP
                                              // and stay inside the list; later runs go to the drain untested (~7 per segment
                                              // of random sequence, 96 at most)
constexpr uint32_t MZ_M64 = MLG_MZ_ORD_MULT << 6;   // the multiplier carries the << 6 of (order << 6 | position)
// reads per hand-out: one tile counter increment, one TMA issue and one mbarrier wait serve MZ_TILE_READS / 32 warp
// passes.  64 halves the share of the per-tile code (~300 instructions on one lane) but doubles the staging buffers:
// 2 x 108 KB of shared memory per SM leave 28 KB of L1 and the kernel ran 18 % SLOWER (2.56 vs 2.16 ms, r4c); 32 it is.
#ifndef MZ_TILE_READS
#define MZ_TILE_READS 32
#endif
constexpr unsigned MZ_TR = MZ_TILE_READS;
static_assert(MZ_TR % 32 == 0 && MZ_TR >= 32 && MZ_TR <= 128, "tile = whole warp passes");
constexpr unsigned MZ_STAGE_B = MZ_TR * 40 + 64;       // MZ_TR reads x 160 bases fit; longer reads are gathered from global
constexpr unsigned MZ_STAGE_M = MZ_TR * 20 + 64;
struct MzStage {
    __align__(16) unsigned char b[WARPS][2][MZ_STAGE_B];
    __align__(16) unsigned char m[WARPS][2][MZ_STAGE_M];
};
struct MzShared {
    MzStage stg;
    unsigned char rl[MZ_LIST][RT];            // [r][thread]: low byte of the r-th run's minimum of the current segment
                                              //       (its minimizer's position relative to the run's first block)
    uint32_t seq[SEGW + 1][RT];               // [word][thread]: the lane's current segment (160 bases, top-aligned words)
    uint32_t qa[WARPS][MZ_QCAP];              // item: stream position (in bases) of the block's first window, low / high word
    uint32_t qc[WARPS][MZ_QCAP];
    uint32_t qb[WARPS][MZ_QCAP];              // item: windows of the block to compare exactly (bit tt = window tt) | base of the
                                              //       minimizer relative to the block's first window << 16
    uint32_t qoff[WARPS][32];                 // drain: windows before each item of the batch
    uint32_t qn[WARPS];                       // items waiting
};
constexpr uint32_t MZ_ROW = RT * 4;           // byte stride between rows of seq[]

// The L2::64B qualifier matters: without a prefetch-size qualifier a miss on this part moves 128 bytes from HBM for
// every random 4-byte access (3.8 sectors per request, whatever the load's width or cache policy); with it, 64
// (profiles/r3a_ubench_gather.md).  MZ_L2_FETCH=0 builds the kernel without it (A/B measurements).
#ifndef MZ_L2_FETCH
#define MZ_L2_FETCH 64
#endif
#if MZ_L2_FETCH == 64
#define MZ_L2Q ".L2::64B"
#elif MZ_L2_FETCH == 128
#define MZ_L2Q ".L2::128B"
#else
#define MZ_L2Q ""
#endif
__device__ __forceinline__ uint32_t ldg_bitmap_if(bool p, const uint32_t* ptr) {
    uint32_t r;
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.u32 q, %1, 0;\n"
        "mov.u32 %0, 0;\n"
        "@q ld.global.nc.L1::no_allocate" MZ_L2Q ".b32 %0, [%2];\n"
        "}\n" : "=r"(r) : "r"((uint32_t)p), "l"(ptr));
    return r;
}
// the exact path's random reads of database arrays, same fetch size
__device__ __forceinline__ uint32_t ldg_u32(const uint32_t* ptr) {
    uint32_t r;
    asm volatile("ld.global.nc" MZ_L2Q ".b32 %0, [%1];" : "=r"(r) : "l"(ptr));
    return r;
}
__device__ __forceinline__ void sts8(uint32_t addr, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds8(uint32_t addr) {
    uint32_t r;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(r) : "r"(addr));
    return r;
}
__device__ __forceinline__ key128 ldg_key(const key128* ptr) {
    key128 k;
    asm volatile("ld.global.nc" MZ_L2Q ".v2.u64 {%0, %1}, [%2];" : "=l"(k.hi), "=l"(k.lo) : "l"(ptr));
    return k;
}
// The tile's bases and N bits as 32-bit shared loads from this warp's staging buffer (the common case: reads of up to 160
// bases; segment_load in probe_common.cuh is the general form -- 64-bit generic loads with clamped indices -- and cost 220
// of the ~850 instructions a read pays outside its blocks).  brel / mrel: the segment's first base relative to the first
// staged base / mask bit; sb / sk: shared addresses of the staged bytes (or of a zero block for a lane without windows).
template <bool HAS_NMASK>
__device__ __forceinline__ void segment_load_staged(uint32_t (&loc)[SEGW], uint32_t (&nl)[5], uint32_t brel, uint32_t mrel, uint32_t sb, uint32_t sk) {
    const uint32_t ab = sb + (brel >> 4) * 4u;
    const unsigned sh = 2u * (brel & 15u);
    uint32_t W[SEGW + 1];
#pragma unroll
    for (int k = 0; k <= (int)SEGW; ++k) W[k] = __byte_perm(lds32(ab + 4u * (uint32_t)k), 0, 0x0123);
#pragma unroll
    for (int k = 0; k < (int)SEGW; ++k) loc[k] = fsl(W[k], W[k + 1], sh);
#pragma unroll
    for (int k = 0; k < 5; ++k) nl[k] = 0;
    if (HAS_NMASK) {
        const uint32_t am = sk + (mrel >> 5) * 4u;
        const unsigned shn = mrel & 31u;
        uint32_t M[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) M[k] = __byte_perm(lds32(am + 4u * (uint32_t)k), 0, 0x0123);
#pragma unroll
        for (int k = 0; k < 5; ++k) nl[k] = fsl(M[k], M[k + 1], shn);
    }
}
// (order << 6 | position) of the 32-mer at position 16j+i of the current block: first half = bases [16j+i, +16) of
// loc[], reverse complement of the second half = the 16-mer at 16(j+1)+i seen through rcl[] (see sk_mmer)
__device__ __forceinline__ uint32_t mz_val(const uint32_t (&loc)[SEGW], const uint32_t (&rcl)[SEGW], int j, int i) {
    const uint32_t a = fsl(loc[j], loc[j + 1], 2 * i);
    const int ra = i <= 11 ? 7 - j : 6 - j, ro = i <= 11 ? 11 - i : 27 - i;
    const uint32_t b = fsl(rcl[ra], rcl[ra + 1], 2 * ro);
    return b * MZ_M64 + (a * MZ_M64 + (uint32_t)(16 * j + i));
}
// 64 bases of the packed stream starting at base p, top-aligned (hi = the first 32)
__device__ __forceinline__ void mz_bases64(const unsigned long long* bsrc, unsigned long long base_words, unsigned long long p,
                                           unsigned long long& hi, unsigned long long& lo) {
    const unsigned long long q = p >> 5;
    const unsigned sh = 2u * (unsigned)(p & 31ull);
    unsigned long long W[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        unsigned long long idx = q + k;
        if (idx >= base_words) idx = base_words - 1;
        W[k] = bswap64(bsrc[idx]);
    }
    hi = sh ? ((W[0] << sh) | (W[1] >> (64 - sh))) : W[0];
    lo = sh ? ((W[1] << sh) | (W[2] >> (64 - sh))) : W[1];
}
// Exact compare of ONE window of an item (one lane), in two stages.  Stage 1: the window starts at base p, its minimizer
// at base pm of the stream; identity, bucket range and the first two database k-mers of the bucket (both loads in flight
// together).  (Two windows per lane and round were tried: the drain's code doubles and the kernel starts missing in the
// instruction cache, which costs more than the extra memory parallelism gains.)
struct MzWin {
    key128 cn, d0, d1;           // canonical key of the window; first two k-mers of the bucket
    uint32_t s, e, j0, j1;       // bucket range in D, alias range
};
__device__ __forceinline__ void mz_window_begin(MzWin& w, bool on, unsigned long long p, unsigned long long pm,
                                                const unsigned long long* bsrc, unsigned long long base_words, const DbView& db) {
    w.s = w.e = w.j0 = w.j1 = 0;
    w.cn.hi = w.cn.lo = 0; w.d0 = w.cn; w.d1 = w.cn;
    if (!on) return;
    // the window's 64 bases from p hold its minimizer too: it starts at most 28 bases in (pm - p <= K - 32)
    key128 F;
    mz_bases64(bsrc, base_words, p, F.hi, F.lo);
    const unsigned dsh = 2u * (unsigned)(pm - p);
    const unsigned long long mh = dsh ? ((F.hi << dsh) | (F.lo >> (64u - dsh))) : F.hi;
    const uint32_t ha = (uint32_t)(mh >> 32), hb = rev2_32(~(uint32_t)mh);
    const uint32_t zhi = mz_ident_hi(ha, hb), zlo = mz_ident_lo(ha, hb);
    const uint32_t bucket = zhi >> (32u - db.bbits);
    w.s = ldg_u32(db.bstart + bucket); w.e = ldg_u32(db.bstart + bucket + 1);
    // K-mers filed under a second identity (order ties) are rare: a 2^16-bit array says whether to look at all
    if (db.n_alias && ((db.alias_bloom[(zlo & 0xFFFFu) >> 5] >> (zlo & 31u)) & 1u)) {
        const unsigned long long z = ((unsigned long long)zhi << 32) | zlo;
        uint32_t lo = 0, hi = db.n_alias;
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (db.alias_z[mid] < z) lo = mid + 1; else hi = mid; }
        w.j0 = w.j1 = lo;
        while (w.j1 < db.n_alias && db.alias_z[w.j1] == z) ++w.j1;
    }
    F = key_shr(F, 128 - 2 * SK_K);                                 // the 60-mer, bottom-aligned
    const key128 G = key_rc(F, SK_K);
    w.cn = key_lt(G, F) ? G : F;
    if (w.s < w.e) w.d0 = ldg_key(db.D_key + w.s);
    if (w.s + 1u < w.e) w.d1 = ldg_key(db.D_key + w.s + 1u);
}
// stage 2: compare with the database k-mers filed under the identity, count a match
__device__ __forceinline__ void mz_window_end(const MzWin& w, const DbView& db, const CountSink& cs) {
    if (w.s < w.e && w.d0.hi == w.cn.hi && w.d0.lo == w.cn.lo) { bump_counter(cs, w.s); return; }
    if (w.s + 1u < w.e && w.d1.hi == w.cn.hi && w.d1.lo == w.cn.lo) { bump_counter(cs, w.s + 1u); return; }
    for (uint32_t i = w.s + 2u; i < w.e; ++i) {
        const key128 d = ldg_key(db.D_key + i);
        if (d.hi == w.cn.hi && d.lo == w.cn.lo) { bump_counter(cs, i); return; }
    }
    for (uint32_t j = w.j0; j < w.j1; ++j) {
        const uint32_t i = db.alias_i[j];
        const key128 d = db.D_key[i];
        if (d.hi == w.cn.hi && d.lo == w.cn.lo) { bump_counter(cs, i); return; }
    }
}
// exact compare of every window of every waiting item of one warp, one WINDOW per lane (items have 1..16 windows)
// `a` and `db` are the kernel's __grid_constant__ parameters: the references point into parameter space, so nothing is
// copied to the stack for the call (before, every thread kept a 232-byte copy of both structs in local memory and the
// drain read its fields from there: 5.4 M local loads per 10 M reads, 18-27 % of them missing the L1).  Speed is the same
// within run-to-run noise (2.15 ms); what is left on the stack are two values parked around the block loop.
__device__ __noinline__ void mz_drain(uint32_t* qn, const uint32_t* qa, const uint32_t* qc, uint32_t* qb, uint32_t* qoff,
                                      const ProbeArgs& a, const DbView& db) {
    const unsigned long long* const bsrc = a.bases;
    const unsigned long long base_words = a.base_words;
    const CountSink cs{a.cnt8, a.present, a.n_present, a.touched, a.ci_min};
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const unsigned lane = threadIdx.x & 31u;
    __syncwarp();
    const uint32_t n = *qn;
    for (uint32_t base = 0; base < n; base += 32u) {
        const uint32_t i = base + lane;
        uint32_t kb0 = i < n ? qb[i] : 0u;
        // Items of runs beyond the run list's capacity arrive untested (bit 31).  Their level-1 bits are looked at here,
        // once per ITEM and 32 items at a time, before the items are spread over the lanes window by window: 99.6 % of
        // them fail, and used to cost every one of their ~11 windows a lookup of its own.
        if (__any_sync(FULL, (kb0 >> 31) != 0u)) {
            if (kb0 >> 31) {
                const unsigned long long pb = ((unsigned long long)qc[i] << 32) | qa[i];
                unsigned long long mh, ml;
                mz_bases64(bsrc, base_words, pb + ((kb0 >> 16) & 63u), mh, ml);
                const uint32_t ha = (uint32_t)(mh >> 32), hb = rev2_32(~(uint32_t)mh);
                const uint32_t zhi = mz_ident_hi(ha, hb), zlo = mz_ident_lo(ha, hb);
                const unsigned long long idx = mz_bit_index(((unsigned long long)zhi << 32) | zlo, db.fbits);
                const uint32_t f = ldg_u32(db.F + (idx >> 5));
                kb0 = ((f >> (zlo & 31u)) & (f >> mz_bit2(zhi)) & 1u) ? (kb0 & 0x7FFFFFFFu) : 0u;
                qb[i] = kb0;
            }
            __syncwarp();
        }
        const uint32_t cnt = (uint32_t)__popc(kb0 & 0xFFFFu);
        uint32_t inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(FULL, inc, o); if ((int)lane >= o) inc += u; }
        const uint32_t total = __shfl_sync(FULL, inc, 31);
        qoff[lane] = inc - cnt;
        __syncwarp();
        for (uint32_t w = lane; w < total; w += 32u) {
            uint32_t j = 0;                              // the last item of the batch that starts at or before window w
#pragma unroll
            for (uint32_t step = 16; step; step >>= 1) if (qoff[j + step] <= w) j += step;
            const uint32_t kb = qb[base + j];
            const uint32_t tt = __fns(kb & 0xFFFFu, 0u, (int)(w - qoff[j]) + 1);
            const unsigned long long pb = ((unsigned long long)qc[base + j] << 32) | qa[base + j];
            MzWin win;
            mz_window_begin(win, true, pb + tt, pb + ((kb >> 16) & 63u), bsrc, base_words, db);
            mz_window_end(win, db, cs);
        }
        __syncwarp();
    }
    __syncwarp();                 // every lane has read *qn, also when the list was empty and the loop did not run
    if (lane == 0) *qn = 0;
    __syncwarp();
}

template <bool HAS_NMASK>
__global__ void __launch_bounds__(RT, MZ_MINCTAS) k1_minimizer_probe(const __grid_constant__ ProbeArgs a, const __grid_constant__ DbView db) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MzShared& sm = *reinterpret_cast<MzShared*>(smem_raw);
    MzStage& stg = sm.stg;
    __shared__ __align__(8) unsigned long long mbar[WARPS][2];
    __shared__ unsigned long long s_bw0[WARPS][2], s_mw0[WARPS][2];
    __shared__ unsigned s_staged[WARPS][2];
    __shared__ __align__(16) uint32_t s_zero[SEGW + 2];      // what a lane without windows loads instead of staged bytes

    const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
    constexpr unsigned K = SK_K;
    if (tid < SEGW + 2) s_zero[tid] = 0u;
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const unsigned long long nreads = a.r_end - a.r_begin;
    const unsigned long long ntiles = (nreads + MZ_TR - 1) / MZ_TR;       // a tile = MZ_TR reads: MZ_TR / 32 warp passes
    // the hand-out counter: 32 bits are plenty (a tile is >= 32 reads), and the word above it stays zero
    unsigned int* const tile_ctr = reinterpret_cast<unsigned int*>(a.tile_counter);
    auto next_tile = [&]() -> unsigned long long {
        unsigned int t = 0;
        if (lane == 0) t = atomicAdd(tile_ctr, 1u);
        return __shfl_sync(FULL, t, 0);
    };
    // The packed reads go through the L2 with NORMAL priority: the drain reads the bases of its items back from global memory
    // a tile or two later, and with evict_first (the round-1 choice, -DMZ_STREAM_EVICT_FIRST) the level-1 array's random lines
    // had pushed them out by then: 2.139 ms against 2.112 (evict_last: 2.112).
#ifdef MZ_STREAM_EVICT_FIRST
    const unsigned long long pol_stream = policy_evict_first();
#elif defined(MZ_STREAM_EVICT_LAST)
    const unsigned long long pol_stream = policy_evict_last();
#else
    unsigned long long pol_stream;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol_stream));
#endif
    const uint32_t rl_base = smem_u32(&sm.rl[0][tid]), seq_base = smem_u32(&sm.seq[0][tid]);
    const uint32_t* const MB = db.F;
    const uint32_t lt_mask = (1u << lane) - 1u;
    // bit index = identity & (2^fbits - 1): mask of its low word, and of its high word (0 up to 2^32 bits)
    const uint32_t fmask_lo = db.fbits >= 32u ? 0xFFFFFFFFu : ((1u << db.fbits) - 1u);
    const uint32_t fmask_hi = db.fbits > 32u ? ((1u << (db.fbits - 32u)) - 1u) : 0u;

    if (lane == 0) {
        mbar_init(&mbar[warp][0], 1);
        mbar_init(&mbar[warp][1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto issue = [&](unsigned stage, unsigned long long t) {
        const unsigned long long r0 = a.r_begin + t * (unsigned long long)MZ_TR;
        const unsigned long long r1 = (r0 + MZ_TR < a.r_end) ? r0 + MZ_TR : a.r_end;
        const unsigned long long p0 = a.off ? a.off[r0] : r0 * (unsigned long long)a.read_len;
        const unsigned long long p1 = a.off ? a.off[r1] : r1 * (unsigned long long)a.read_len;
        unsigned long long bw0 = (p0 >> 5) & ~1ull;
        unsigned long long bw1 = ((p1 + 31) >> 5) + 6;
        if (bw1 > a.base_words) bw1 = a.base_words;
        bw1 = (bw1 + 1) & ~1ull;
        unsigned long long mw0 = (p0 >> 6) & ~1ull;
        unsigned long long mw1 = ((p1 + 63) >> 6) + 4;
        if (HAS_NMASK) { if (mw1 > a.nmask_words) mw1 = a.nmask_words; mw1 = (mw1 + 1) & ~1ull; }
        const unsigned long long bytes_b = (bw1 - bw0) * 8ull, bytes_m = HAS_NMASK ? (mw1 - mw0) * 8ull : 0ull;
        const bool fits = bw1 > bw0 && bytes_b <= MZ_STAGE_B && bytes_m <= MZ_STAGE_M;
        s_bw0[warp][stage] = bw0; s_mw0[warp][stage] = mw0; s_staged[warp][stage] = fits ? 1u : 0u;
        if (fits) {
            mbar_expect_tx(&mbar[warp][stage], (uint32_t)(bytes_b + bytes_m));
            bulk_g2s(&stg.b[warp][stage][0], a.bases + bw0, (uint32_t)bytes_b, &mbar[warp][stage], pol_stream);
            if (HAS_NMASK && bytes_m) bulk_g2s(&stg.m[warp][stage][0], a.nmask + mw0, (uint32_t)bytes_m, &mbar[warp][stage], pol_stream);
        } else {
            mbar_arrive(&mbar[warp][stage]);
        }
    };

    unsigned my_valid = 0;                    // per lane: a launch would need > 3e14 windows to overflow it
    unsigned my_fetch = 0;
    if (lane == 0) sm.qn[warp] = 0;
    __syncwarp();

    // the two halves (a, b) of the 32-mer at base P of the lane's segment copy (b = reverse complement of the second half)
    auto halves_at = [&](uint32_t P, uint32_t& ha, uint32_t& hb) {
        const uint32_t ad = seq_base + (P >> 4) * MZ_ROW;
        const uint32_t w0 = lds32(ad), w1 = lds32(ad + MZ_ROW), w2 = lds32(ad + 2u * MZ_ROW);
        const unsigned sh = 2u * (P & 15u);
        ha = fsl(w0, w1, sh);
        hb = rev2_32(~fsl(w1, w2, sh));
    };
    auto drain = [&]() {
        // items carry stream positions and the drain reads the bases from global memory (L2: they were just streamed in), so
        // items survive the tile they come from and a drain always has >= MZ_QDRAIN items' windows to spread over the lanes
        mz_drain(&sm.qn[warp], &sm.qa[warp][0], &sm.qc[warp][0], &sm.qb[warp][0], &sm.qoff[warp][0], a, db);
    };
    // lanes with p append one item: windows `ik` of the block whose first window is at stream base `pb`, minimizer at base `rel` of the block
    auto push = [&](bool p, unsigned long long pb, uint32_t ik, uint32_t rel) {
        if (p) {
            const uint32_t i = atomicAdd(&sm.qn[warp], 1u);
            sm.qa[warp][i] = (uint32_t)pb; sm.qc[warp][i] = (uint32_t)(pb >> 32); sm.qb[warp][i] = ik | (rel << 16);
        }
    };
    auto drain_if_full = [&]() {
        __syncwarp();
        if (sm.qn[warp] >= MZ_QDRAIN) drain();
    };

    unsigned it = 0;
    unsigned long long t = next_tile(), t_ahead = next_tile();       // the tile being processed and the one staged behind it
    if (lane == 0) {
        if (t < ntiles) issue(0, t);
        if (t_ahead < ntiles) issue(1, t_ahead);
    }
    for (; t < ntiles; ++it) {
        const unsigned stage = it & 1u, parity = (it >> 1) & 1u;
        __syncwarp();
        mbar_wait(&mbar[warp][stage], parity);

        const bool staged = s_staged[warp][stage] != 0;
        const unsigned long long bw0_32 = s_bw0[warp][stage] * 32ull, mw0_64 = s_mw0[warp][stage] * 64ull;
        const uint32_t sb_stage = smem_u32(&stg.b[warp][stage][0]), sk_stage = smem_u32(&stg.m[warp][stage][0]), s_zero_a = smem_u32(&s_zero[0]);
#pragma unroll 1
        for (unsigned half = 0; half < MZ_TR / 32u; ++half) {
        const unsigned long long r = a.r_begin + t * (unsigned long long)MZ_TR + half * 32u + lane;
        if (half && r - lane >= a.r_end) break;
        const bool active = r < a.r_end;
        unsigned long long R0 = 0, R1 = 0;
        if (active) {
            R0 = a.off ? a.off[r] : r * (unsigned long long)a.read_len;
            R1 = a.off ? a.off[r + 1] : R0 + a.read_len;
        }
        const unsigned long long len = R1 - R0;
        const unsigned long long nw = len >= K ? len - K + 1 : 0ull;
        const unsigned nseg = (unsigned)((nw + WMAX - 1) / WMAX);
        const unsigned max_seg = __reduce_max_sync(FULL, nseg);
        // staged (reads of up to 160 bases): 32-bit positions relative to the staged bytes; otherwise the stream itself
        const uint32_t brel0 = (uint32_t)(R0 - bw0_32), mrel0 = (uint32_t)(R0 - mw0_64);
        __syncwarp();

        for (unsigned seg = 0; seg < max_seg; ++seg) {
            const unsigned c = seg < nseg ? (unsigned)((nw - (unsigned long long)seg * WMAX) < WMAX ? (nw - (unsigned long long)seg * WMAX) : WMAX) : 0u;
            const unsigned long long s = bw0_32 + brel0 + (unsigned long long)seg * WMAX;      // = R0 + seg * WMAX

            uint32_t loc[SEGW];
            uint32_t nl[5];
            if (staged) segment_load_staged<HAS_NMASK>(loc, nl, c ? brel0 + seg * WMAX : 0u, c ? mrel0 + seg * WMAX : 0u, c ? sb_stage : s_zero_a, c ? sk_stage : s_zero_a);
            else segment_load<HAS_NMASK>(loc, nl, c, s, a.bases, a.nmask, a.base_words, a.nmask_words);
            uint32_t v0, v1, v2;
            segment_valid<HAS_NMASK>(nl, c, K, v0, v1, v2);
            my_valid += __popc(v0) + __popc(v1) + __popc(v2);
            if (__all_sync(FULL, (v0 | v1 | v2) == 0u)) continue;

            // the lane's copy of the segment (minimizer halves are fetched from it by position)
#pragma unroll
            for (int k = 0; k < (int)SEGW; ++k) sts32(seq_base + (uint32_t)k * MZ_ROW, loc[k]);
            sts32(seq_base + SEGW * MZ_ROW, 0u);

            // reverse complement of the segment: the complement of base x sits at base 154 - x of rcl[]
            uint32_t rcl[SEGW];
            segment_rc60(loc, rcl);

            // minimizer state carried from block to block: P = prefix minimum of position block 1 up to index 11
            uint32_t P = 0xFFFFFFFFu;
#pragma unroll
            for (int i = 0; i < 12; ++i) P = min(P, mz_val(loc, rcl, 1, i));
            // blocks the warp walks: up to the last one in which some lane has a valid window
            const int lastv = v2 ? 96 - __ffs(v2) : v1 ? 64 - __ffs(v1) : v0 ? 32 - __ffs(v0) : -1;
            const unsigned nblk = __reduce_max_sync(FULL, (unsigned)(lastv + 16) >> 4);
            // Phase A, block by block.  Every run start goes to the run list (the low byte of the window minimum: the
            // minimizer's position relative to the block) and to c0..c2 (bit w = window w, shifted in from the top).  No
            // window is dropped for validity here: a window that is not valid costs at most a wasted lookup; it is masked
            // out of the items.
            uint32_t pw = 0xFFFFFFFFu;                // minimum of the previous window (none before window 0: no value is ~0)
            uint32_t lst = rl_base;                   // where the next run's byte goes
            uint32_t c0 = 0, c1 = 0, c2 = 0;
#pragma unroll 1
            for (unsigned blk = 0; blk < nblk; ++blk) {
                lst = min(lst, rl_base + MZ_CAP * RT);   // a full list: the block's bytes overwrite slots >= MZ_CAP (never read)
                uint32_t Suf[16];
                {
                    uint32_t smn = 0xFFFFFFFFu;
#pragma unroll
                    for (int i = 15; i >= 0; --i) { smn = min(smn, mz_val(loc, rcl, 0, i)); Suf[i] = smn; }
                }
                uint32_t A1 = 0, chg = 0;
#pragma unroll
                for (int tt = 0; tt < 16; ++tt) {
                    uint32_t wm;
                    if (tt < 4) {                              // window tt: positions tt..15, then block 1 up to index tt + 12
                        P = min(P, mz_val(loc, rcl, 1, 12 + tt));
                        wm = min(Suf[tt], P);
                        if (tt == 3) { A1 = P; P = 0xFFFFFFFFu; }
                    } else {                                   // positions tt..15, all of block 1, block 2 up to index tt - 4
                        P = min(P, mz_val(loc, rcl, 2, tt - 4));
                        wm = min(min(Suf[tt], A1), P);
                    }
                    if (wm != pw) {                            // a new run starts at window tt
                        sts8(lst, wm);
                        lst += RT;
                        chg |= 1u << tt;
                    }
                    pw = wm;
                }
                P -= 16u;                                      // block 2 of this block is block 1 of the next one
                pw -= 16u;                                     // (a run going on keeps its value; a position of -1 becomes 63,
                                                               //  which no window minimum has)
                c0 = __funnelshift_r(c0, c1, 16); c1 = __funnelshift_r(c1, c2, 16); c2 = __funnelshift_r(c2, chg, 16);
                // slide the register windows by one word
#pragma unroll
                for (int k = 0; k < (int)SEGW - 1; ++k) loc[k] = loc[k + 1];
#pragma unroll
                for (int k = (int)SEGW - 1; k > 0; --k) rcl[k] = rcl[k - 1];
            }
            for (unsigned blk = nblk; blk < WMAX / 16u; ++blk) { c0 = __funnelshift_r(c0, c1, 16); c1 = __funnelshift_r(c1, c2, 16); c2 >>= 16; }

            // Runs that start after the lane's last valid window have no window to look up.  Window 0 always starts a run.
            {
                const uint32_t lim = (uint32_t)(lastv + 1);
                c0 &= lim >= 32u ? 0xFFFFFFFFu : (1u << lim) - 1u;
                c1 &= lim >= 64u ? 0xFFFFFFFFu : lim > 32u ? (1u << (lim - 32u)) - 1u : 0u;
                c2 &= lim >= 96u ? 0xFFFFFFFFu : lim > 64u ? (1u << (lim - 64u)) - 1u : 0u;
            }
            const uint32_t nr = (uint32_t)(__popc(c0) + __popc(c1) + __popc(c2));
            // fw walks the run starts; c0..c2 hold the starts after it, from window fw + 1 on.  A run covers at most 29
            // windows, so the next start is always in c0.
            uint32_t fw = 0;
            c0 = __funnelshift_r(c0, c1, 1); c1 = __funnelshift_r(c1, c2, 1); c2 >>= 1;
            auto next_start = [&]() -> uint32_t {        // start of the run after the one at fw (96: none)
                const uint32_t d = __ffs(c0);
                c0 = __funnelshift_r(c0, c1, d); c1 = __funnelshift_r(c1, c2, d); c2 >>= d;
                return d ? fw + d : WMAX;
            };
            const uint32_t V0 = __brev(v0), V1 = __brev(v1), V2 = __brev(v2);      // validity, bit w = window w
            // lanes with `on` turn run pk (first window | end << 8 | minimizer position << 16) into items, one for every block
            // of 16 windows the run has valid windows in; `unt`: 0x8000 for runs whose level-1 bits the drain looks at
            auto emit = [&](bool on, uint32_t pk, uint32_t unt) {
                const uint32_t f = pk & 127u, e = (pk >> 8) & 127u, pz = pk >> 16;
                const unsigned long long ia = s_bw0[warp][stage] * 32ull + brel0 + (unsigned long long)seg * WMAX;
#pragma unroll
                for (uint32_t k = 0; k < 3u; ++k) {
                    const uint32_t b0 = (f & ~15u) + 16u * k;                          // the block's first window
                    const uint32_t vb = ((b0 < 32u ? V0 : b0 < 64u ? V1 : V2) >> (b0 & 16u)) & 0xFFFFu;
                    const uint32_t lo = k == 0 ? f - b0 : 0u, hi = e < b0 + 16u ? e - b0 : 16u;
                    const uint32_t mk = e > b0 ? (0xFFFFu << lo) & (0xFFFFu >> (16u - hi)) & vb : 0u;
                    push(on && mk != 0u, ia + b0, mk, (pz - b0) | unt);
                }
            };

            // Lookups: slot i of every lane's list, MZ_LGROUP slots at a time, up to the warp's longest list.
            const uint32_t nrc = min(nr, MZ_CAP);
            const uint32_t nmax = __reduce_max_sync(FULL, nrc);
#pragma unroll 1
            for (uint32_t i0 = 0; i0 < nmax; i0 += MZ_LGROUP) {
                uint32_t Fw[MZ_LGROUP], Bt[MZ_LGROUP], Pk[MZ_LGROUP];      // the word, its two bit positions, the run
#pragma unroll
                for (uint32_t g = 0; g < MZ_LGROUP; ++g) {
                    Fw[g] = 0; Bt[g] = 0; Pk[g] = 0;
                    if (i0 + g < nmax) {
                        const bool on = i0 + g < nrc;
                        const uint32_t nx = next_start();
                        const uint32_t pz = on ? (fw & ~15u) + (lds8(rl_base + (i0 + g) * RT) & 63u) : 0u;
                        uint32_t ha, hb;
                        halves_at(pz, ha, hb);
                        const uint32_t zlo = mz_ident_lo(ha, hb) & fmask_lo, zhi = mz_ident_hi(ha, hb);
                        Bt[g] = (zlo & 31u) | (mz_bit2(zhi) << 8);
                        Fw[g] = ldg_bitmap_if(on, MB + ((zlo >> 5) | ((zhi & fmask_hi) << 27)));
                        Pk[g] = fw | (nx << 8) | (pz << 16);
                        my_fetch += on ? 1u : 0u;
                        fw = nx;
                    }
                }
                uint32_t pm = 0;                         // slots whose run passed (both bits set; 0.4 % by chance, plus the true hits)
#pragma unroll
                for (uint32_t g = 0; g < MZ_LGROUP; ++g) pm |= ((Fw[g] >> (Bt[g] & 31u)) & (Fw[g] >> (Bt[g] >> 8)) & 1u) << g;
                while (__any_sync(FULL, pm != 0u)) {
                    const uint32_t g = __ffs(pm) - 1u;
                    uint32_t pk = Pk[0];
#pragma unroll
                    for (uint32_t h = 1; h < MZ_LGROUP; ++h) if (g == h) pk = Pk[h];
                    emit(pm != 0u, pk, 0u);
                    pm &= pm - 1u;
                    drain_if_full();
                }
            }
            // Runs beyond the list's capacity (only in sequence whose minimizer changes at more than every second window)
            // go to the drain untested.  Their bytes were not kept: the minimizer of the run's first window is found again.
            if (__any_sync(FULL, nr > MZ_CAP)) {
#pragma unroll 1
                for (uint32_t i = MZ_CAP; __any_sync(FULL, i < nr); ++i) {
                    const bool on = i < nr;
                    const uint32_t nx = next_start();
                    uint32_t pk = 0;
                    if (on) {
                        uint32_t best = 0xFFFFFFFFu;
#pragma unroll 1
                        for (uint32_t q = 0; q + MLG_MZ_M <= K; ++q) {
                            uint32_t ha, hb;
                            halves_at(fw + q, ha, hb);
                            best = min(best, (ha + hb) * MZ_M64 + q);
                        }
                        pk = fw | (nx << 8) | ((fw + (best & 63u)) << 16);
                    }
                    emit(on, pk, 0x8000u);
                    drain_if_full();
                    fw = nx;
                }
            }
        }
        }
        __syncwarp();             // every lane is done with this stage's staged bases before it is refilled
        const unsigned long long t_new = next_tile();      // (asking for it at the start of the tile instead changes nothing: 2.164 ms either way, r4h)
        if (lane == 0 && t_new < ntiles) issue(stage, t_new);
        t = t_ahead; t_ahead = t_new;
    }

    drain();                      // the items still waiting
    unsigned long long warp_valid = my_valid;
    for (int o = 16; o > 0; o >>= 1) warp_valid += __shfl_down_sync(FULL, warp_valid, o);
    my_fetch = __reduce_add_sync(FULL, my_fetch);
    if (lane == 0 && warp_valid) atomicAdd(a.n_kmers, warp_valid);
    if (lane == 0 && my_fetch) atomicAdd(a.n_kmers + 1, (unsigned long long)my_fetch);
}

constexpr size_t K1MZ_SMEM = sizeof(MzShared);

template <bool HAS_NMASK>
int launch_mz_t(const DbView& db, const ProbeArgs& a, cudaStream_t st, unsigned grid) {
    auto kern = k1_minimizer_probe<HAS_NMASK>;
    static bool done[64] = {};          // the attribute is per device
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !done[dev]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K1MZ_SMEM));
        // MLG_PROBE_CARVEOUT=<percent of the SM's 228 KB>: shared-memory carve-out (experiments: what is left is the L1)
        if (const char* e = getenv("MLG_PROBE_CARVEOUT")) { int x = atoi(e); if (x >= 0 && x <= 100) CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, x)); }
        if (dev >= 0 && dev < 64) done[dev] = true;
    }
    CUDA_TRY(cudaMemsetAsync(a.tile_counter, 0, 8, st));
    kern<<<grid, RT, K1MZ_SMEM, st>>>(a, db);
    CUDA_TRY(cudaGetLastError());
    return MLG_OK;
}

}  // namespace

int launch_probe_mz(const DbView& db, const ProbeArgs& a, cudaStream_t st, int sm_count) {
    if (db.K != SK_K || !db.F) { mlg_set_error("minimizer-bitmap layout needs K=60 and its bit array"); return MLG_ERR_STATE; }
    // persistent: the CTAs that fit pull 32-read tiles from a global counter
    const unsigned long long wtiles = (a.r_end - a.r_begin + MZ_TR - 1) / MZ_TR;
    const unsigned long long need = (wtiles + WARPS - 1) / WARPS;
    int per_sm = MZ_MINCTAS;
    if (const char* e = getenv("MLG_PROBE_CTAS_PER_SM")) { int x = atoi(e); if (x >= 1 && x <= 64) per_sm = x; }
    const unsigned long long res = (unsigned long long)sm_count * (unsigned)per_sm;
    const unsigned grid = (unsigned)(need < res ? need : res);
    return a.nmask ? launch_mz_t<true>(db, a, st, grid) : launch_mz_t<false>(db, a, st, grid);
}
