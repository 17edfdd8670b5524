"""The run bookkeeping of the minimizer kernel (probe_mz.cu): phase A lists every run of equal window minimum of a
96-window segment, the lookups walk those lists slot by slot up to the warp's longest one, and a passing run becomes one
item per block of 16 windows it touches; runs beyond the list's capacity go to the drain untested.

Every test here follows test_every_window_is_a_database_kmer: the database holds every N-free 60-mer of the reads, so a
window lost or compared twice changes the counters.  The reads are independent random sequence, so their k-mers occur
once each and ci_min = 1 and 2 see a lost and a doubled window; the homopolymer k-mers of the overflow reads occur many
times and are checked at ci_min = their count and one more.  Where a read is built for a run shape, the shape is checked
first against the host restatement of the window minima (_mz_order)."""
import random

import pytest

from metalign_b200 import codec
from metalign_b200.api import Database
from oracle import oracle_py

from helpers import oracle_c_run
from test_gpu_parity import _check, _mz_order

pytestmark = pytest.mark.gpu
K = 60
KS = (30, 40, 50, 60)
SEG = 96                   # window starts per segment
LIST_CAP = 48              # runs of a segment that the kernel looks up itself
ORD_MULT = 0x9E3779B1
ORD_INV = pow(ORD_MULT, -1, 1 << 26)


def _rnd(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def _kmer16(v):
    return "".join("ACGT"[(v >> (2 * (15 - i))) & 3] for i in range(16))


def _low_order_32mer(rng, order):
    """a random 32-mer whose mz_order is `order`: the order is (a + b) * ORD_MULT mod 2^26, so b follows from a"""
    a = rng.getrandbits(32)
    b = ((order * ORD_INV - a) % (1 << 26)) + (rng.getrandbits(6) << 26)
    s = _kmer16(a) + oracle_py.rc(_kmer16(b))
    assert _mz_order(s) == order
    return s


def _run_starts(read):
    """per 96-window segment: the windows (segment-relative) at which the window minimum, as (order, leftmost position),
    changes; N is packed as A"""
    r = read.replace("N", "A")
    nw = len(r) - K + 1
    o = [_mz_order(r[p:p + 32]) for p in range(len(r) - 31)]
    segs = []
    for s0 in range(0, max(nw, 0), SEG):
        starts, prev = [], None
        for w in range(s0, min(s0 + SEG, nw)):
            m = min(o[w:w + K - 31])
            cur = (m, w + o[w:w + K - 31].index(m))
            if cur != prev:
                starts.append(w - s0)
            prev = cur
        segs.append(starts)
    return segs


def _planted(rng, length, first_window, order=7):
    """a random read whose 32-mer at first_window + 28 has a far lower order than any other: the windows that contain
    it, first_window .. first_window + 28, are one run"""
    while True:
        p = first_window + K - 32
        r = _rnd(rng, p) + _low_order_32mer(rng, order) + _rnd(rng, length - p - 32)
        starts = _run_starts(r)[first_window // SEG]
        w = first_window % SEG
        if w in starts and not any(w < x < w + 29 for x in starts):
            return r


def _homopolymer_read(rng, base):
    """random flanks around 150 copies of one base: every window inside the stretch starts a run of its own, far more
    than the run list holds"""
    r = _rnd(rng, 25) + base * 150 + _rnd(rng, 25)
    assert len(_run_starts(r)[0]) > LIST_CAP + 16
    return r


def _windows(reads):
    """canonical N-free 60-mers of the reads with their counts"""
    cnt = {}
    for r in reads:
        for i in range(len(r) - K + 1):
            w = r[i:i + K]
            if "N" not in w:
                c = min(w, oracle_py.rc(w))
                cnt[c] = cnt.get(c, 0) + 1
    return cnt


def _run(ctx, reads, extra_ci=()):
    rng = random.Random(len(reads))
    cnt = _windows(reads)
    kmers = sorted(cnt)
    n = 500
    G = (len(kmers) + n - 1) // n
    kmers += [_rnd(rng, K) for _ in range(G * n - len(kmers))]
    sketches = [kmers[g * n:(g + 1) * n] for g in range(G)]
    keys = codec.sketches_to_keys(sketches, K)
    db = Database.from_keys(ctx, keys, G, n, K, KS)
    try:
        for ci_min in sorted({1, 2, *extra_ci}):
            ref, I_ref = oracle_c_run(keys, G, n, K, KS, lambda q: q.push_reads(reads), ci_min, "exact", True)
            q = db.query(ci_min, "exact", True)
            q.push_reads(reads)
            res = q.finish()
            _check(res, q.intersection(), ref, I_ref, ci_min)
            assert res["stats"]["layout"] == 2
            q.close()
            if ci_min == 1:
                assert ref["n_intersect"] == len(cnt)
    finally:
        db.close()


def test_runs_starting_at_block_and_segment_edges(ctx):
    """runs whose first window is the last or first of a block of 16 (15, 16, 31, 32) and the last of a segment (95)"""
    rng = random.Random(11)
    reads = []
    for i, s in enumerate([15, 16, 31, 32, 95] * 8):
        reads.append(_planted(rng, rng.choice([170, 200, 251]), s, order=3 + i))
    _run(ctx, reads)


def test_maximal_runs_span_three_blocks(ctx):
    """runs of the maximal 29 windows: 15..43 and 47..75 touch three blocks and become three items each"""
    rng = random.Random(12)
    reads = []
    for i, s in enumerate([15, 47, 3, 31] * 10):
        r = _planted(rng, 160, s, order=5 + i)
        starts = _run_starts(r)[0]
        assert s + 29 in starts and starts[starts.index(s) + 1] == s + 29
        reads.append(r)
    _run(ctx, reads)


def test_reads_at_segment_boundaries(ctx):
    """155 / 156 bases: 96 windows (one segment) and 97 (a second segment of one window); 251 / 252: 192 and 193"""
    rng = random.Random(13)
    reads = [_rnd(rng, L) for L in [155, 156, 251, 252] * 40]
    reads += [_planted(rng, 252, s, order=9 + i) for i, s in enumerate([95, 96, 191, 192])]
    _run(ctx, reads)


def test_n_in_first_or_last_window_of_a_run(ctx):
    """an N at the run's first base (its first window is not valid, the rest are) or 59 bases after its last window
    starts (only its last window is not valid)"""
    rng = random.Random(14)
    reads = []
    for i, s in enumerate([20, 33, 48, 64] * 6):
        for x in (s, s + 28 + K - 1):
            r = list(_planted(rng, 200, s, order=11 + i))
            r[x] = "A"
            if s not in _run_starts("".join(r))[0]:
                continue
            r[x] = "N"
            reads.append("".join(r))
    assert len(reads) >= 30
    _run(ctx, reads)


def test_list_overflow_in_an_uneven_warp(ctx):
    """one homopolymer read among 31 random ones in every warp: its lane has more runs than the list holds (they reach
    the drain untested) while the other lanes have ~7; the warp's lookups run to the longest list"""
    rng = random.Random(15)
    reads = []
    for g, base in enumerate("ACTG"):           # two reads for each canonical homopolymer 60-mer: counts stay below 255
        group = [_rnd(rng, rng.choice([100, 150, 151, 250])) for _ in range(31)]
        group.insert((7 * g + 3) % 32, _homopolymer_read(rng, base))
        reads += group
    cnt = _windows(reads)
    homo = {cnt[b * K] for b in "AC"}
    _run(ctx, reads, extra_ci={c for h in homo for c in (h, h + 1)})
