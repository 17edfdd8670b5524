"""mlg_sketch_genomes (csrc/sketch.cu) at every boundary its kernels and its host loop branch on, against the C oracle
oracle/sketch_oracle.c: a literal, one-window-at-a-time restatement of CountEstimator.add that shares nothing with the
GPU's threshold-and-sort method.  Every GPU case compares mins, counts and kmers of every slot, exactly.

A  the oracle against the Python transcription of CountEstimator (test_sketch.py) at every K branch of MurmurHash3,
   primes from 2 to the largest below 2^44, n around the number of distinct hashes, text holding all 256 byte values
B  every K in 1..64; genome starts and ends at every residue mod 32 of the device text; non-ACGT bytes (all 256 values,
   the case fold's near misses such as 0xC1 and 0xE1 among them) next to valid windows; lower case
C  genomes of TILE +- 1 and 2 TILE +- 1 windows, and non-ACGT bytes at TILE - 1, TILE and TILE + K - 1 from a tile start
D  sketches with n - 1, n and n + 1 distinct k-mers; genomes without a valid window, of length 0, K - 1 and K
E  hash collisions mod small primes, in windows of different tiles (earliest window, summed counts; run twice)
F  the count of the last slot of a full sketch (k_fix_last), composed on purpose, against a closed form
G  repeats that need redo rounds and grow the candidate list
H  more than one 1 GB pass at full size, with a redo round that regroups genomes of different passes
I  MLG_SKETCH_PASS_BYTES: passes of one genome, a genome larger than a pass, the split at every genome boundary; the
   pass count against a restatement of the batching and redo rule
J  the genome count: G up to 2^20 - 1 (the sort key's genome bits)
K  the refusals of the C ABI, and the valid-window count
L  build_database and make_sketch_db.py
Parts A and L's argument checks run without a GPU."""
import ctypes as C
import functools
import gzip
import os
import random
import re
import subprocess
import sys
from collections import defaultdict

import numpy as np
import pytest

import test_sketch
from conftest import ROOT
from oracle import sketch_oracle as so

PRIME = so.PRIME
ERR_ARG = -2
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_VALID = np.zeros(256, dtype=bool)
_VALID[list(b"ACGTacgt")] = True


def _tile():
    src = open(os.path.join(ROOT, "metalign_b200", "csrc", "sketch.cu")).read()
    return int(re.search(r"constexpr\s+uint32_t\s+TILE\s*=\s*(\d+)\s*;", src).group(1))


TILE = _tile()


def _is_prime(p):
    """deterministic Miller-Rabin (these bases decide every p < 3.3e24)"""
    if p < 2:
        return False
    bases = (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37)
    for b in bases:
        if p % b == 0:
            return p == b
    d, s = p - 1, 0
    while d % 2 == 0:
        d, s = d // 2, s + 1
    for b in bases:
        x = pow(b, d, p)
        if x in (1, p - 1):
            continue
        for _ in range(s - 1):
            x = x * x % p
            if x == p - 1:
                break
        else:
            return False
    return True


def _largest_prime_below(x):
    p = x - 1
    while not _is_prime(p):
        p -= 1
    return p


P44 = _largest_prime_below(1 << 44)
PRIMES = (2, 3, 61, 4099, 1000003, PRIME, P44)


# ------------------------------------------------------------------------------------------------ helpers
def _bases(rng, L):
    return ACGT[rng.integers(0, 4, L, dtype=np.uint8)].tobytes()


def _pack(genomes):
    """genomes (bytes) -> (text, genome_off) as mlg_sketch_genomes and the oracle take them"""
    off = np.zeros(len(genomes) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(g) for g in genomes])
    return np.frombuffer(b"".join(genomes) + b"N", dtype=np.uint8), off


def _out(G, n, K, fill=0):
    return (np.full((G, n), fill, dtype=np.uint64), np.full((G, n), fill, dtype=np.uint32),
            np.full((G, n, K), fill & 0xFF, dtype=np.uint8))


def _gpu_raw(ctx_h, text, off, G, n, K, prime, outs, st):
    from metalign_b200 import _lib
    ptr = lambda a: None if a is None else a.ctypes.data
    return _lib.lib().mlg_sketch_genomes(ctx_h, ptr(text), ptr(off), G, n, K, prime, *(ptr(a) for a in outs),
                                         None if st is None else C.addressof(st))


def _gpu(ctx, text, off, n, K, prime=PRIME):
    from metalign_b200 import _lib
    G = len(off) - 1
    outs = _out(G, n, K, 0xA5)
    st = _lib.SketchStats()
    _lib.check(_gpu_raw(ctx._h, text, off, G, n, K, prime, outs, st))
    return outs, {f: getattr(st, f) for f, _ in st._fields_ if f != "reserved"}


def _oracle(text, off, n, K, prime=PRIME):
    G = len(off) - 1
    outs = _out(G, n, K)
    so.lib().sko_sketch_genomes(text.ctypes.data, off.ctypes.data, G, n, K, prime, *(a.ctypes.data for a in outs))
    return outs


def _same(got, want, what=""):
    for name, a, b in zip(("mins", "counts", "kmers"), got, want):
        if not np.array_equal(a, b):
            g, s = np.argwhere(a != b)[0][:2]
            raise AssertionError("%s: %s differ in %d entries, first at genome %d slot %d: got %r, want %r"
                                 % (what, name, int((a != b).sum()), g, s, a[g, s], b[g, s]))


def _check(ctx, text, off, n, K, prime=PRIME, what=""):
    got, st = _gpu(ctx, text, off, n, K, prime)
    want = _oracle(text, off, n, K, prime)
    _same(got, want, what or "n=%d K=%d prime=%d" % (n, K, prime))
    return got, st


def _valid_starts(seq, K):
    """window starts of one genome whose K bytes are all ACGT/acgt"""
    v = _VALID[np.frombuffer(seq, dtype=np.uint8)]
    if len(v) < K:
        return np.zeros(0, dtype=np.int64)
    c = np.concatenate([[0], np.cumsum(~v)])
    return np.nonzero(c[K:] == c[:-K])[0]


def _distinct_hashes(seq, K, prime):
    up = seq.upper()
    return np.unique(np.array([so.murmur3_x64_128(up[p:p + K])[0] % prime for p in _valid_starts(seq, K)], dtype=np.uint64))


def _sprinkle(rng, seq, nbytes, values):
    """seq with nbytes bytes replaced by values (cycled), a tenth of the rest lower-cased"""
    a = np.frombuffer(seq, dtype=np.uint8).copy()
    if len(a):
        low = rng.random(len(a)) < 0.1
        a[low] |= 0x20
        pos = rng.integers(0, len(a), nbytes)
        a[pos] = np.resize(np.asarray(values, dtype=np.uint8), nbytes)
    return a.tobytes()


# ------------------------------------------------------------------------------------------------ A (CPU)
A_K = (1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64)


def _all_bytes_genome(K, seed):
    """records of ACGT/acgt separated by every byte value 0..255 (each at least once), about 2500 windows in all"""
    rng = np.random.default_rng(seed)
    vals = list(range(256))
    random.Random(seed).shuffle(vals)
    parts = []
    for i in range(0, 256, 16):
        parts.append(_sprinkle(rng, _bases(rng, int(rng.integers(K, K + 300))), 0, []))
        parts.append(bytes(vals[i:i + 16]))
    g = b"".join(parts)
    assert set(g) == set(range(256))
    return g


@pytest.mark.parametrize("K", A_K)
def test_oracle_matches_transcription_at_every_hash_branch(K, monkeypatch):
    """sko_sketch_genome against py_count_estimator (the transcription decodes the text as latin-1) for every prime and
    n in {1, 2, distinct - 1, distinct, distinct + 1}; the transcription's hash is memoised, its logic is untouched"""
    assert P44 == 17592186044399 and _is_prime(PRIME) and not _is_prime(P44 + 2) and all(_is_prime(p) for p in PRIMES)
    monkeypatch.setattr(test_sketch, "py_murmur3_x64_128", functools.lru_cache(maxsize=None)(test_sketch.py_murmur3_x64_128))
    seq = _all_bytes_genome(K, 40 + K)
    text, off = _pack([seq])
    nwin = len(_valid_starts(seq, K))
    assert nwin > 1000
    for prime in PRIMES:
        m, _, _ = _oracle(text, off, nwin + 1, K, prime)
        d = int((m < prime).sum())
        for n in sorted({1, 2, d - 1, d, d + 1} - {0}):
            om, oc, ok = _oracle(text, off, n, K, prime)
            pm, pc, pk = test_sketch.py_count_estimator(seq.decode("latin-1"), n, K, prime)
            assert om[0].tolist() == pm and oc[0].tolist() == pc, (prime, n)
            assert [bytes(x).rstrip(b"\0").decode() for x in ok[0]] == pk, (prime, n)


# ------------------------------------------------------------------------------------------------ B
def _residue_set(K, seed):
    """64 genomes whose device starts (one separator after each genome) run through every residue mod 32 twice:
    lengths are 4 mod 32, so start i is 5 i mod 32 and the byte after genome i is 5 i + 4 mod 32.  Every byte value
    appears; some genomes begin or end with a non-ACGT byte."""
    rng = np.random.default_rng(seed)
    high = [0xC1, 0xC3, 0xC7, 0xD4, 0xE1, 0xE3, 0xE7, 0xF4, 0x81, 0xA1]   # A/C/G/T | 0x80 (| 0x20): near misses of the fold
    genomes = []
    for i in range(64):
        L = 32 * int(rng.integers(1, 100)) + 4
        g = bytearray(_sprinkle(rng, _bases(rng, L), max(2, L // 300), high))
        for j in range(4):
            g[(j + 1) * L // 5] = i * 4 + j
        if i % 4 == 1:
            g[0] = (b"N", b"\xc1", b"\x00", b"n")[(i // 4) % 4][0]
        if i % 4 == 2:
            g[-1] = (b"R", b"\xe1", b"\xff", b">")[(i // 4) % 4][0]
        genomes.append(bytes(g))
    starts = np.cumsum([0] + [len(g) + 1 for g in genomes])[:-1]
    ends = starts + np.array([len(g) for g in genomes])
    assert set((starts % 32).tolist()) == set(range(32)) == set((ends % 32).tolist()) == set(((ends - 1) % 32).tolist())
    assert set(b"".join(genomes)) == set(range(256))
    return genomes


@pytest.mark.gpu
@pytest.mark.parametrize("K", range(1, 65))
def test_every_k_every_alignment(ctx, K):
    text, off = _pack(_residue_set(K, 1000 + K))
    for n in (1, 7, 64, 4000):                   # 4000: more slots than any genome has windows, so every window shows
        _check(ctx, text, off, n, K)


# ------------------------------------------------------------------------------------------------ C
@pytest.mark.gpu
@pytest.mark.parametrize("K", (1, 16, 21, 32, 33, 60, 64))
def test_tile_boundaries(ctx, K):
    rng = np.random.default_rng(K)
    genomes = [_bases(rng, w + K - 1) for w in (TILE - 1, TILE, TILE + 1, 2 * TILE - 1, 2 * TILE, 2 * TILE + 1)]
    for offs in ([TILE - 1], [TILE], [TILE + K - 1], [TILE - 1, TILE, TILE + K - 1]):
        g = bytearray(_bases(rng, 5 * TILE + K))
        for t, o in enumerate(offs):
            g[t * TILE + o] = ord("N")           # tile t starts at t * TILE of the genome
        g[2 * TILE - 3:2 * TILE + 3] = g[2 * TILE - 3:2 * TILE + 3].lower()
        genomes.append(bytes(g))
    text, off = _pack(genomes)
    for n in (64, 6 * TILE):                     # 6 TILE: every distinct window of every genome is in its sketch
        _check(ctx, text, off, n, K, what="K=%d n=%d" % (K, n))


# ------------------------------------------------------------------------------------------------ D
def _distinct_kmers(rng, K, count, prime=PRIME):
    """count K-mers with pairwise different hashes mod prime, in random order"""
    seen, out = set(), []
    while len(out) < count:
        km = _bases(rng, K)
        h = so.murmur3_x64_128(km)[0] % prime
        if h not in seen:
            seen.add(h)
            out.append(km)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("where", ("first", "middle", "last"))
@pytest.mark.parametrize("K", (21, 60))
def test_sketch_fill(ctx, K, where):
    n = 50
    rng = np.random.default_rng(K)
    special = []
    for d in (n - 1, n, n + 1):
        kms = _distinct_kmers(rng, K, d)
        pieces = kms + [kms[i] for i in rng.integers(0, d, 2 * d)]
        rng.shuffle(pieces)
        special.append(b"N".join(pieces))
    special += [b"ACGTN" * 200 if K > 4 else b"N" * 300, b"\xc1" * 300 + b"N" * 10, b"", _bases(rng, K - 1), _bases(rng, K)]
    full = [_bases(rng, 5000) for _ in range(3)]
    genomes = {"first": special + full, "middle": full[:2] + special + full[2:], "last": full + special}[where]
    text, off = _pack(genomes)
    (mins, counts, kmers), _ = _check(ctx, text, off, n, K)
    s0 = genomes.index(special[0])
    expect_used = [n - 1, n, n, 0, 0, 0, 0, 1]
    for i, used in enumerate(expect_used):
        g = s0 + i
        assert (mins[g, :used] < PRIME).all() and (mins[g, used:] == PRIME).all(), (i, used)
        assert (counts[g, used:] == 0).all() and (kmers[g, used:] == 0).all() and (counts[g, :used] >= 1).all()


# ------------------------------------------------------------------------------------------------ E
E_CASES = ((2, 1), (3, 2), (61, 40), (4099, 1000), (1000003, 1000), (P44, 1000))


@pytest.mark.gpu
@pytest.mark.parametrize("prime,n", E_CASES)
def test_collisions_across_tiles(ctx, prime, n):
    """windows of different CTAs share a hash value: the stored k-mer is the earliest window, the count sums them, and two
    runs agree although the candidate list's append order differs"""
    rng = np.random.default_rng(prime % 1000)
    K = 21
    unit = _bases(rng, 3000)
    genomes = [_bases(rng, 10_000 + K - 1), _bases(rng, 100_000) + unit + _bases(rng, 5000) + unit, _bases(rng, 1_000_000 + K - 1)]
    text, off = _pack(genomes)
    first, st = _check(ctx, text, off, n, K, prime)
    again, _ = _gpu(ctx, text, off, n, K, prime)
    _same(again, first, "second run, prime %d" % prime)
    mins, counts, _ = first
    assert (mins < prime).all()                  # n stays below the number of distinct values
    if prime <= 61 and n > 1:
        assert counts[:, :n - 1].min() > 100     # every slot merges windows of many tiles
    if st["passes"] == 1:
        assert st["n_windows"] == sum(len(g) - K + 1 for g in genomes)


# ------------------------------------------------------------------------------------------------ F
def _closed_form(pieces, hash_of, n, prime):
    """the sketch of a genome made of one-window pieces (the piece index is the window order): the n smallest distinct
    hashes, each with its earliest k-mer and its occurrences -- but once a full sketch's last value L is the largest of
    the sketch, i.e. once the n - 1 smaller values have all appeared, its repeats are not counted (at least 1)"""
    first, occ = {}, defaultdict(list)
    for i, km in enumerate(pieces):
        h = hash_of[km]
        first.setdefault(h, (i, km))
        occ[h].append(i)
    vals = sorted(first)[:n]
    counts = [len(occ[v]) for v in vals]
    if len(vals) == n:
        full_at = max(first[v][0] for v in vals[:-1]) if n > 1 else -1
        counts[-1] = max(1, sum(1 for i in occ[vals[-1]] if i < full_at))
    pad = n - len(vals)
    return vals + [prime] * pad, counts + [0] * pad, [first[v][1] for v in vals] + [b""] * pad


def _pool(K, prime, count, seed):
    rng = np.random.default_rng(seed)
    by_hash = defaultdict(set)
    for _ in range(count):
        km = _bases(rng, K)
        by_hash[so.murmur3_x64_128(km)[0] % prime].add(km)
    return {h: sorted(v) for h, v in by_hash.items()}


def _run_layouts(ctx, layouts, hash_of, n, K, prime, want_last):
    genomes = [b"N".join(p) for p in layouts]
    text, off = _pack(genomes)
    got, _ = _check(ctx, text, off, n, K, prime)
    for g, pieces in enumerate(layouts):
        m, c, k = _closed_form(pieces, hash_of, n, prime)
        assert got[0][g].tolist() == m and got[1][g].tolist() == c, (g, got[1][g].tolist(), c)
        assert [bytes(x).rstrip(b"\0") for x in got[2][g]] == k
        assert c[n - 1] == want_last[g], (g, c[n - 1], want_last[g])


@pytest.mark.gpu
@pytest.mark.parametrize("n", (2, 5, 40))
def test_last_element_placement(ctx, n):
    """L, the n-th smallest value, before the n - 1 smaller ones have all appeared, between them, only after all of
    them, and in all three places; filler k-mers with larger hashes spread every layout over several tiles"""
    K = 21
    pool = _pool(K, PRIME, 4000, n)
    hs = sorted(pool)
    hash_of = {km: h for h, kms in pool.items() for km in kms}
    S, L, fill = [pool[h][0] for h in hs[:n - 1]], pool[hs[n - 1]][0], [pool[h][0] for h in hs[n:]]
    rng = random.Random(n)
    pad = lambda m=250: [rng.choice(fill) for _ in range(m)]
    h = (n - 1) // 2
    rep = S[:2] * 3                              # repeats of smaller values after they are all in
    layouts = [
        [L] + pad() + [L] + pad() + S + pad() + rep,                               # before: 2
        S[:h] + pad() + [L] + pad() + [L, L] + pad() + S[h:] + rep + pad(),        # between: 3 (n = 2: before all)
        pad() + S + pad() + [L] + pad() + [L, L] + rep,                            # after: 1
        [L] + pad() + S[:h] + [L] + pad() + S[h:] + pad() + [L, L] + rep,          # all three: 2 (n = 2: all before)
    ]
    want = [2, 3, 1, 2]
    _run_layouts(ctx, layouts, hash_of, n, K, PRIME, want)


@pytest.mark.gpu
def test_last_element_small_n_and_collisions(ctx):
    """n = 1 (the count is always 1), n = 2 with repeated minima, and L sharing its value with another k-mer mod 4099"""
    K = 21
    pool = _pool(K, PRIME, 3000, 77)
    hs = sorted(pool)
    hash_of = {km: h for h, kms in pool.items() for km in kms}
    s0, L = pool[hs[0]][0], pool[hs[1]][0]
    rng = random.Random(5)
    fills = [pool[h][0] for h in hs[2:]]
    pad = lambda m=300: [rng.choice(fills) for _ in range(m)]
    _run_layouts(ctx, [[s0] + pad() + [s0, s0] + pad() + [s0], pad() + [s0]], hash_of, 1, K, PRIME, [1, 1])
    layouts = [[L] + pad() + [s0, s0] + pad() + [L, s0, L],          # 1
               [L, L] + pad() + [L, s0] + pad() + [s0, L, s0],       # 3
               [s0, s0, s0] + pad() + [L, L],                        # 1
               pad() + [L, s0, L, L, s0] + pad()]                    # 1
    _run_layouts(ctx, layouts, hash_of, 2, K, PRIME, [1, 3, 1, 1])
    # mod 4099: L1 and L2 share L's value; the stored k-mer is the earlier one, the count covers both
    prime, n = 4099, 5
    pool = _pool(K, prime, 3000, 78)
    hash_of = {km: h for h, kms in pool.items() for km in kms}
    hs = sorted(pool)
    hL = next(h for i, h in enumerate(hs) if i >= n - 1 and len(pool[h]) >= 2)
    L1, L2 = pool[hL][:2]
    smaller = [pool[h][0] for h in hs if h < hL]
    S = smaller[-(n - 1):]
    fills = [km for h in hs if h > hL for km in pool[h]]
    layouts = [[L2] + pad() + [S[0], L1] + pad() + [S[1], S[2], L2, L1] + pad() + [S[3]] + pad() + [L1, L2, S[0]],   # 4
               [L1] + pad() + S + pad() + [L2, L1]]                                                                      # 1
    _run_layouts(ctx, layouts, hash_of, n, K, prime, [4, 1])
    got, _ = _gpu(ctx, *_pack([b"N".join(p) for p in layouts]), n, K, prime)
    assert bytes(got[2][0, n - 1]) == L2 and bytes(got[2][1, n - 1]) == L1


# ------------------------------------------------------------------------------------------------ G
@pytest.mark.gpu
@pytest.mark.parametrize("K", (21, 60))
def test_repeats_redo_and_candidate_growth(ctx, K):
    rng = np.random.default_rng(K)
    unit = _bases(rng, 1500)
    genomes = [_bases(rng, 200_000), b"A" * 2_000_000, _bases(rng, 50_000), b"AC" * 250_000, _bases(rng, 3000),
               b"ACG" * 100_000, unit * 200, _bases(rng, 100_000)]
    text, off = _pack(genomes)
    for n in (1, 5, 200):
        _, st = _check(ctx, text, off, n, K, what="K=%d n=%d" % (K, n))
        if n > 1:
            assert st["passes"] > 1, st          # the whole set is one pass in the first round
        assert st["n_candidates"] > 0


# ------------------------------------------------------------------------------------------------ H
@pytest.mark.gpu
def test_full_size_multi_pass(ctx):
    """1.3 GB of text in 24 genomes of 54 MB: the 1 GB split falls between genomes 18 and 19; two repeat-rich genomes,
    one in each pass, are redone together"""
    G, n, K = 24, 1000, 60
    L = 54_200_000
    rng = np.random.default_rng(24)
    off = np.arange(G + 1, dtype=np.uint64) * np.uint64(L)
    text = np.empty(G * L + 1, dtype=np.uint8)
    for g in range(G):
        text[g * L:(g + 1) * L] = ACGT[rng.integers(0, 4, L, dtype=np.uint8)]
        text[g * L + rng.integers(0, L, 2000)] = ord("N")
    text[-1] = ord("N")
    text[3 * L:4 * L] = np.resize(np.frombuffer(_bases(rng, 1500), dtype=np.uint8), L)
    text[21 * L:22 * L] = np.resize(np.frombuffer(b"AC", dtype=np.uint8), L)
    got, st = _gpu(ctx, text, off, n, K)
    want = _oracle(text, off, n, K)
    _same(got, want, "full size")
    assert st["passes"] >= 3, st


# ------------------------------------------------------------------------------------------------ I
def _threshold(nwin, tmul, n, prime):
    frac = tmul * 4.0 * n / nwin if nwin else 1.0
    return prime if frac >= 1.0 else int(float(prime) * frac) + 1


def _predict_passes(lens, hashes, nwins, n, prime, pass_bytes):
    """mlg_sketch_genomes' host loop: whole genomes in order while their text fits in pass_bytes; a genome whose
    threshold is below the prime and lets fewer than n distinct hashes through is redone with 8 times the threshold"""
    tmul, todo, passes = [1.0] * len(lens), list(range(len(lens))), 0
    while todo:
        redo, i = [], 0
        while i < len(todo):
            batch, nbytes = [], 0
            while i < len(todo) and not (batch and nbytes + lens[todo[i]] > pass_bytes):
                batch.append(todo[i])
                nbytes += lens[todo[i]] + 1
                i += 1
            passes += 1
            for g in batch:
                T = _threshold(nwins[g], tmul[g], n, prime)
                if T < prime and np.searchsorted(hashes[g], T) < n:
                    tmul[g] *= 8.0
                    redo.append(g)
        todo = redo
    return passes


@pytest.mark.gpu
def test_pass_size_sweep(ctx, monkeypatch):
    n, K = 64, 21
    rng = np.random.default_rng(9)
    genomes = [_bases(rng, 8000), _bases(rng, 300) * 50, _bases(rng, 30_000), b"AC" * 7000, _bases(rng, 3000),
               _bases(rng, 12_000), b"T" * 5000 + _bases(rng, 40), _bases(rng, 20_000), _bases(rng, 500) * 30, _bases(rng, 6000)]
    lens = [len(g) for g in genomes]
    hashes = [_distinct_hashes(g, K, PRIME) for g in genomes]
    nwins = [max(0, x - K + 1) for x in lens]
    text, off = _pack(genomes)
    want = _oracle(text, off, n, K)
    ends = np.cumsum([x + 1 for x in lens])           # ends[b - 1] - 1 = P: genomes 0..b-1 fit, genome b does not
    sizes = {"one genome each": 1, "a genome larger than a pass": 25_000}
    sizes.update({"split after %d" % b: int(ends[b - 1]) - 1 for b in range(1, len(genomes))})
    for what, P in sizes.items():
        monkeypatch.setenv("MLG_SKETCH_PASS_BYTES", str(P))
        got, st = _gpu(ctx, text, off, n, K)
        _same(got, want, what)
        expect = _predict_passes(lens, hashes, nwins, n, PRIME, P)
        assert st["passes"] == expect, (what, P, st["passes"], expect)
    monkeypatch.delenv("MLG_SKETCH_PASS_BYTES")
    got, st = _gpu(ctx, text, off, n, K)
    _same(got, want, "default pass size")
    assert st["passes"] == _predict_passes(lens, hashes, nwins, n, PRIME, 1 << 30)


# ------------------------------------------------------------------------------------------------ J
def _many_small(G, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(80, 201, G).astype(np.uint64)
    off = np.zeros(G + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    text = np.empty(int(off[-1]) + 1, dtype=np.uint8)
    text[:-1] = ACGT[rng.integers(0, 4, int(off[-1]), dtype=np.uint8)]
    text[-1] = ord("N")
    return text, off


@pytest.mark.gpu
@pytest.mark.parametrize("G", (2, 3, 4, 5, 1 << 16, (1 << 16) + 1, (1 << 19) + 1, (1 << 20) - 1))
def test_genome_count(ctx, G):
    """the radix sort covers 44 + gbits key bits, gbits = ceil(log2 G) up to 20: at G = 2^20 - 1 all 64 bits"""
    text, off = _many_small(G, G)
    _check(ctx, text, off, 2, 21, what="G=%d" % G)


@pytest.mark.gpu
def test_genome_count_limit(ctx):
    from metalign_b200 import _lib
    G = 1 << 20
    text, off = np.frombuffer(b"ACGT" * 64, dtype=np.uint8), np.zeros(G + 1, dtype=np.uint64)
    outs = _out(G, 1, 1, 0x5A)
    assert _gpu_raw(ctx._h, text, off, G, 1, 1, 0, outs, _lib.SketchStats()) == ERR_ARG
    assert (outs[0] == 0x5A).all() and (outs[1] == 0x5A).all() and (outs[2] == 0x5A).all()


# ------------------------------------------------------------------------------------------------ K
@pytest.mark.gpu
def test_abi_refusals_write_nothing(ctx):
    from metalign_b200 import _lib
    rng = np.random.default_rng(3)
    text, off = _pack([_bases(rng, 500), _bases(rng, 300), _bases(rng, 700)])
    G, n, K = 3, 8, 21
    good = dict(ctx_h=ctx._h, text=text, off=off, G=G, n=n, K=K, prime=0)
    cases = {"K=0": dict(K=0), "K=65": dict(K=65), "n=0": dict(n=0), "G=0": dict(G=0), "prime=1": dict(prime=1),
             "prime=2^44": dict(prime=1 << 44), "null ctx": dict(ctx_h=None), "null text": dict(text=None),
             "null genome_off": dict(off=None),
             "genome_off decreases": dict(off=np.array([0, 500, 400, 1500], dtype=np.uint64)),
             "genome_off decreases at the end": dict(off=np.array([0, 500, 800, 700], dtype=np.uint64)),
             "genome_off decreases at the start": dict(off=np.array([600, 500, 800, 1500], dtype=np.uint64))}
    for null in range(3):
        cases["null output %d" % null] = dict(null=null)
    for what, change in cases.items():
        a = dict(good, **{k: v for k, v in change.items() if k != "null"})
        outs = list(_out(max(G, 1), max(n, 1), max(K, 1), 0x5A))
        if "null" in change:
            outs[change["null"]] = None
        st = _lib.SketchStats(7, 7, 7.0, 7, 7)
        rc = _gpu_raw(a["ctx_h"], a["text"], a["off"], a["G"], a["n"], a["K"], a["prime"], outs, st)
        assert rc == ERR_ARG, (what, rc)
        assert all(o is None or (o == 0x5A).all() for o in outs), what
        assert (st.n_windows, st.n_candidates, st.ms_kernels, st.passes) == (7, 7, 7.0, 7), what
    # a valid call after the refusals, and its window count
    genomes = _residue_set(31, 5)
    text, off = _pack(genomes)
    _, st = _check(ctx, text, off, 64, 31)
    assert st["passes"] == 1 and st["n_windows"] == sum(len(_valid_starts(g, 31)) for g in genomes)


# ------------------------------------------------------------------------------------------------ L
def _genome_files(tmp_path, count, seed):
    rng = random.Random(seed)
    paths = []
    for i in range(count):
        p = tmp_path / ("genome_%02d.fna%s" % (count - i, ".gz" if i % 2 else ""))
        recs = ["".join(rng.choice("ACGT") for _ in range(rng.randint(2000, 6000))) for _ in range(2)]
        data = "".join(">c%d\n%s\n" % (j, "\n".join(r[k:k + 70] for k in range(0, len(r), 70))) for j, r in enumerate(recs))
        with (gzip.open if i % 2 else open)(str(p), "wb") as f:
            f.write(data.encode())
        paths.append(str(p))
    return paths


def test_build_database_caps_genomes_per_call(tmp_path, monkeypatch):
    """batches end at GENOMES_PER_CALL genomes (mlg_sketch_genomes takes fewer than 2^20) as well as at batch_bytes"""
    from metalign_b200 import sketch
    assert sketch.GENOMES_PER_CALL == (1 << 20) - 1
    paths = _genome_files(tmp_path, 7, 2)
    calls = []

    def fake(ctx, genomes, n, K, prime=0):
        calls.append(len(genomes))
        m, c, k = so.sketch_genomes(genomes, n, K)
        return m, c, k, {"n_windows": 0, "n_candidates": 0, "ms_kernels": 0.0, "passes": 1}

    monkeypatch.setattr(sketch, "sketch_genomes", fake)
    monkeypatch.setattr(sketch, "GENOMES_PER_CALL", 2)
    sketch.build_database(None, paths, str(tmp_path / "a.mlgdb"), n=20, K=31, ks=(31,))
    assert calls == [2, 2, 2, 1]
    calls.clear()
    sketch.build_database(None, paths, str(tmp_path / "b.mlgdb"), n=20, K=31, ks=(31,), batch_bytes=15000)
    assert len(calls) >= 4 and max(calls) <= 2 and sum(calls) == 7
    assert open(tmp_path / "a.mlgdb", "rb").read() == open(tmp_path / "b.mlgdb", "rb").read()


@pytest.mark.parametrize("args", (["-k", "21"], ["-k", "64"], ["-k", "0"], ["-k", "31", "--k_range", "1-60-1"],
                                  ["-k", "31", "--k_range", "0-30-10"], ["-k", "31", "--k_range", "10-30-0"],
                                  ["-k", "31", "--k_range", "ten"]))
def test_make_sketch_db_refuses_before_sketching(tmp_path, capsys, args):
    """a database the loader would refuse (K > 63, no prefix length, more than 8, a prefix length 0) is an argument
    error before any genome is read: the genome list names a file that does not exist"""
    from metalign_b200 import sketch
    lst = tmp_path / "genomes.txt"
    lst.write_text(str(tmp_path / "missing.fna") + "\n")
    out = tmp_path / "out.mlgdb"
    with pytest.raises(SystemExit) as e:
        sketch.main(args + [str(lst), str(out)])
    assert e.value.code == 2 and "error:" in capsys.readouterr().err
    assert not out.exists()


def test_make_sketch_db_script_exits_at_once(tmp_path):
    lst = tmp_path / "genomes.txt"
    lst.write_text(str(tmp_path / "missing.fna") + "\n")
    out = tmp_path / "out.mlgdb"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "make_sketch_db.py"), "-k", "21", str(lst), str(out)],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "1 to 8" in r.stderr and not out.exists(), r.stderr


@pytest.mark.gpu
def test_build_database_in_many_calls(ctx, tmp_path, monkeypatch):
    from helpers import oracle_c_run
    from metalign_b200 import codec, dbformat, sketch
    from metalign_b200.api import Database
    paths = _genome_files(tmp_path, 9, 4)
    calls = []
    real = sketch.sketch_genomes

    def counted(*a, **kw):
        calls.append(len(a[1]))
        return real(*a, **kw)

    monkeypatch.setattr(sketch, "sketch_genomes", counted)
    out = str(tmp_path / "db.mlgdb")
    n, K, ks = 150, 60, (30, 40, 50, 60)
    sketch.build_database(ctx, paths, out, n=n, K=K, ks=ks, batch_bytes=4000)       # every genome has more
    assert len(calls) >= 4 and sum(calls) == 9, calls
    order = sorted(paths, key=os.path.basename)
    assert dbformat.read_names(out) == [os.path.basename(p) for p in order]
    _, _, ok = so.sketch_genomes([sketch.read_fasta(p) for p in order], n, K)
    keys = dbformat.read_keys(out)
    assert np.array_equal(keys.reshape(-1, 2), codec.ascii_slots_to_keys(ok.reshape(-1, K), K))
    db = Database.load(ctx, out)
    src = sketch.read_fasta(order[4]).decode()
    reads = [src[a:a + 150] for a in range(0, len(src) - 150, 5)]
    ref, _ = oracle_c_run(keys, 9, n, K, ks, lambda q: q.push_reads(reads), 1, "none", True)
    q = db.query(1, "none", True)
    q.push_reads(reads)
    res = q.finish()
    q.close()
    db.close()
    assert np.array_equal(res["num"], ref["num"]) and np.array_equal(res["den"], ref["den"]) and np.array_equal(res["ci"], ref["ci"])
    assert res["ci"][4, -1] > 0.9


@pytest.mark.gpu
def test_make_sketch_db_short_k(ctx, tmp_path):
    from metalign_b200 import dbformat, sketch
    from metalign_b200.api import Database
    paths = _genome_files(tmp_path, 3, 6)
    lst = tmp_path / "genomes.txt"
    lst.write_text("\n".join(paths) + "\n")
    out = tmp_path / "db.mlgdb"
    sketch.main(["-k", "31", "--k_range", "15-31-8", "-n", "50", str(lst), str(out)])
    h = dbformat.read_header(str(out))
    assert (h["G"], h["n"], h["K"], list(h["ks"])) == (3, 50, 31, [15, 23, 31])
    Database.load(ctx, str(out)).close()
