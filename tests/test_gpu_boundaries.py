"""The GPU path at the K, k-range and read-length boundaries its kernels branch on, against the oracles.

- K = 32 / 33: the key leaves the low word (build sort, sort_keys128, key masks and shifts); K <= 7 and K = 61..63.
- 8 k values (every bit of the hit-record headers) and up to 63 offsets per k-mer (ks[0] = 1, K = 63).
- The three hit-record formats: same slot, short (exactly 14 hits at one k), long (15 or more).
- Reads of 0, K - 1, K, WMAX + K - 1 (one full segment), WMAX + K (two), 160, 161 and a few thousand bases.
- The probe kernels' shared-memory staging of a tile: exactly at the limit, one 16-byte unit over and under it.
- The KMC writer at every prefix length p = 1..7, and the passes planner's partial refinement level (b < 10 bases).

Part 1 (the references at every K) runs without a GPU and pins the two oracles against each other first."""
import ast
import os
import random
import re
from collections import Counter

import numpy as np
import pytest

import kmcdb
from conftest import ROOT
from helpers import oracle_c_run
from metalign_b200 import codec, ingest
from metalign_b200.api import Database, MlgError
from oracle import oracle_py
from oracle.read_kmers import OracleReadKmers
from test_gpu_parity import _check
from test_gpu_read_kmer_passes import _budget, _measure, _pass_bytes
from test_gpu_read_kmers import _expected, _mixed_reads, _push, _records, _small_db

ERR_ARG = -2
CSRC = os.path.join(ROOT, "metalign_b200", "csrc")
SWEEP_K = (1, 2, 3, 4, 5, 7, 8, 15, 16, 17, 31, 32, 33, 34, 47, 48, 49, 59, 61, 62, 63)
MODES = [(gate, ce, ci) for gate in ("exact", "none") for ce in (True, False) for ci in (1, 2, 3)]
FORMS = ("ascii", "packed", "nruns", "device")


def _constants(fname, names, env=None):
    """the integer constants `names` of a CUDA source, evaluated from their definitions (constexpr or #define)"""
    src = open(os.path.join(CSRC, fname)).read()
    env = dict(env or {})
    for m in re.finditer(r"(?:constexpr\s+unsigned\s+(\w+)\s*=\s*([^;]+);|#define\s+(\w+)\s+([^\n/]+))", src):
        name, expr = (m.group(1), m.group(2)) if m.group(1) else (m.group(3), m.group(4))
        if name in env:
            continue
        try:
            env[name] = eval(compile(ast.parse(expr.strip(), mode="eval"), fname, "eval"), {"__builtins__": {}}, dict(env))
        except Exception:
            pass
    return {k: env[k] for k in names}


_COMMON = _constants("probe_common.cuh", ("RT", "WMAX", "WSTAGE_B", "WSTAGE_M"))
WMAX = _COMMON["WMAX"]


def _ks_ranges(K):
    """(id, ks): the single k; 8 k values (with 32 and 33 where K > 33); the largest spread ks[0] = max(1, K - 62)"""
    out = [("k1", (K,))]
    if K >= 8:
        want = {K} | ({32, 33} if K > 33 else set())
        lo = max(1, K - 40)
        for v in np.linspace(lo, K, 24).round().astype(int).tolist():
            if len(want) >= 8:
                break
            want.add(v)
        ks = tuple(sorted(want))
        assert len(ks) == 8
        out.append(("k8-off%d" % (K - ks[0] + 1), ks))
    k0 = max(1, K - 62)
    if k0 < K:
        out.append(("spread-off%d" % (K - k0 + 1), tuple(sorted({k0, (k0 + K) // 2, K}))))
    return out


def _rand(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


def _workload(K, seed):
    """sketches and reads over one random genome.  Hub k-mers give the record formats: x in 14 genomes (14 hits at the
    k values where nothing else matches), y in 15 genomes (long), and a k-mer twice in one genome (same slot)."""
    rng = random.Random(seed)
    genome = _rand(rng, 3000 + 4 * K)
    G, n = 17, 10
    pos = lambda: rng.randint(0, len(genome) - K)
    sk = [[genome[p:p + K] if rng.random() < 0.5 else oracle_py.rc(genome[p:p + K]) for p in (pos() for _ in range(n))] for _ in range(G)]
    x, y = _rand(rng, K), oracle_py.rc(_rand(rng, K))     # apart from the genome: no stray hits at ks[0]
    for g in range(1, 15):
        sk[g][0] = x
    for g in range(1, 16):
        sk[g][1] = y
    sk[0][2] = sk[0][3]                                  # one genome, two slots: one class
    sk[16][4] = ""                                       # empty slots
    sk[5][9] = ""
    reads = []
    for L in (0, K - 1, K, WMAX + K - 1, WMAX + K, 160, 161, 3000, 150, 150, 250):
        a = rng.randint(0, len(genome) - L)
        r = genome[a:a + L]
        reads.append(r)
        reads.append(oracle_py.rc(r))
    for L in (K + 1, 2 * K, WMAX + K):                    # N at the first and the last base of a window
        a = rng.randint(0, len(genome) - L)
        r = genome[a:a + L]
        reads.append("N" + r[1:])
        reads.append(r[:-1] + "N")
        if L > K:
            reads.append(r[:K - 1] + "N" + r[K:])          # the last base of window 0, the first of window K - 1
    for L in (100, K + 5, 400):                           # lower case
        a = rng.randint(0, len(genome) - L)
        r = genome[a:a + L]
        reads.append("".join(c.lower() if rng.random() < 0.3 else c for c in r))
    hub = _rand(rng, 20) + x + _rand(rng, 30)             # the hub k-mers, seen 1 to 3 times
    reads += [hub, _rand(rng, 5) + oracle_py.rc(y) + _rand(rng, 7), hub, hub.lower()]
    reads = [r for r in reads for _ in range(rng.choice((1, 1, 2, 3)))]
    rng.shuffle(reads)
    return sk, reads


def _record_kinds(sk, K, ks):
    """the hit-record format of every distinct database k-mer, restated from k_tally_hits (csrc/query.cu): the marks of
    the expansion with gate none, counted per (offset, P entry); same slot when every mark names one class
    representative, short when no k has more than 14 marks, long otherwise"""
    slots = [(g, j, s) for g, row in enumerate(sk) for j, s in enumerate(row) if s]
    rep = {}
    for ki, k in enumerate(ks):
        first = {}
        for g, j, s in slots:
            rep[(ki, g, j)] = first.setdefault((g, s[:k]), (g, j))
    by0 = {}
    for g, j, s in slots:
        by0.setdefault(s[:ks[0]], []).append((g, j, s))
    kinds = Counter()
    max14 = False
    for x in {oracle_py.canon(s) for _, _, s in slots}:
        cnt = [0] * len(ks)
        reps = set()
        for o in range(K - ks[0] + 1):
            w = x[o:o + ks[0]]
            F, R = by0.get(w, []), by0.get(oracle_py.rc(w), [])
            for g, j, _ in (F or R):
                cnt[0] += 1
                reps.add(rep[(0, g, j)])
            for ki in range(1, len(ks)):
                k = ks[ki]
                if o + k > K:
                    continue
                wk = x[o:o + k]
                m = [(g, j) for g, j, s in F if s[:k] == wk]
                if not m:
                    rk = oracle_py.rc(wk)
                    m = [(g, j) for g, j, s in by0.get(oracle_py.rc(x[o + k - ks[0]:o + k]), []) if s[:k] == rk]
                for g, j in m:
                    cnt[ki] += 1
                    reps.add(rep[(ki, g, j)])
        if len(reps) == 1:
            kinds["same"] += 1
        elif max(cnt) <= 14:
            kinds["short"] += 1
            max14 |= 14 in cnt
        else:
            kinds["long"] += 1
    return kinds, max14


def _dump_expected(sk, reads, K, I_ref, counter_max):
    mult = Counter(oracle_py.canon(s) for row in sk for s in row if s)
    cnt = oracle_py.count_read_kmers(reads, K)
    return {x: min(cnt[x], mult[x], counter_max) for x in (codec.key_to_kmer(int(a), int(b), K) for a, b in I_ref)}


# ------------------------------------------------------------------------------------------------ 1. the references (CPU)
def _adversarial(rng, K):
    """helpers.adversarial_case at any K, with ks[0] = max(1, K - 62) and, from K = 8, eight k values"""
    genome = _rand(rng, max(200, 3 * K))
    lo = max(1, K - 62)
    if K >= 8:
        ks = sorted({lo, K} | set(rng.sample(range(lo + 1, K), 6)))
    else:
        ks = sorted({lo, K})
    G, n = rng.randint(2, 6), rng.randint(2, 7)
    sk = [["" if rng.random() < 0.15 else (lambda p: genome[p:p + K] if rng.random() < 0.5 else oracle_py.rc(genome[p:p + K]))(
        rng.randint(0, len(genome) - K)) for _ in range(n)] for _ in range(G)]
    reads = []
    for _ in range(rng.randint(10, 60)):
        a = rng.randint(0, len(genome) - 1)
        r = list(genome[a:rng.randint(a, len(genome))])
        for i in range(len(r)):
            u = rng.random()
            r[i] = "N" if u < 0.02 else (r[i].lower() if u < 0.04 else r[i])
        reads.append("".join(r))
    return ks, sk, reads


@pytest.mark.parametrize("K", SWEEP_K + (60,), ids=lambda K: "K%d" % K)
def test_oracles_agree_at_every_k(K):
    rng = random.Random(5000 + K)
    for rep in range(3):
        ks, sk, reads = _adversarial(rng, K)
        assert ks[0] == max(1, K - 62) and (len(ks) == 8 or K < 8)
        G, n = len(sk), len(sk[0])
        keys = codec.sketches_to_keys(sk, K)
        for gate, ce, ci in MODES[rep::3]:
            py = oracle_py.run(reads, sk, K=K, ks=ks, ci_min=ci, gate=gate, count_empty_in_den=ce)
            r, I = oracle_c_run(keys, G, n, K, ks, lambda q: q.push_reads(reads), ci, gate, ce)
            assert r["num"].tolist() == py["num"] and r["den"].tolist() == py["den"], (rep, gate, ce, ci)
            assert r["n_kmers"] == py["n_kmers"]
            assert [codec.key_to_kmer(int(a), int(b), K) for a, b in I] == py["I"]
            assert np.array_equal(r["ci"], np.array(py["ci"]).reshape(G, len(ks)))
        if K <= 60:
            o = OracleReadKmers(K)
            o.push_reads(reads)
            cnt = oracle_py.count_read_kmers(reads, K)
            for mc, cm in ((1, 255), (2, 3)):
                assert _records(*o.result(mc, cm), K) == _expected(reads, K, mc, cm, cnt)
            o.close()


def test_record_format_model_sees_all_three_formats():
    """the sweep's databases hold all three hit-record formats, 14 hits at one k included, wherever the k range allows
    them: from K = 15 every range has 15 offsets or none is needed (the hubs are whole k-mers)"""
    for K in (15, 32, 33, 60, 63):
        for name, ks in _ks_ranges(K):
            if ks[0] <= 3:
                continue                                   # 1- to 3-mers match almost every window: long records only
            sk, _ = _workload(K, 7 * K)
            kinds, max14 = _record_kinds(sk, K, ks)
            assert kinds["same"] and kinds["short"] and kinds["long"] and max14, (K, name, kinds)


def test_staging_limits_are_read_from_the_sources():
    probe = _constants("probe.cu", ("STAGE_B", "STAGE_M"))
    mz = _constants("probe_mz.cu", ("MZ_STAGE_B", "MZ_STAGE_M", "MZ_TR"), {"MLG_RT": 256})
    assert probe["STAGE_B"] % 16 == 0 and mz["MZ_STAGE_B"] % 16 == 0 and _COMMON["WSTAGE_B"] % 16 == 0
    assert _COMMON["RT"] >= 32 and mz["MZ_TR"] >= 32


# ------------------------------------------------------------------------------------------------ 2. tables across K (GPU)
def _sweep_params():
    out = []
    for K in SWEEP_K:
        for name, ks in _ks_ranges(K):
            out.append(pytest.param(K, ks, None, id="K%d-%s" % (K, name)))
    for layout in (2, 1, 0):
        for name, ks in _ks_ranges(60):
            out.append(pytest.param(60, ks, layout, id="K60-L%d-%s" % (layout, name)))
    return out


def _push_form(q, reads, how, keep):
    if how != "nruns":
        _push(q, reads, how, keep)
        return
    # N runs in 0.25 MB copy chunks (MLG_CHUNK_MB): 1.1 M bases of N reads put the boundary among the reads
    half = len(reads) // 2
    allr = reads[:half] + ["N" * 1600] * 700 + reads[half:]
    bases, nmask, off = codec.pack_reads(allr)
    runs = codec.nmask_to_runs(nmask, int(off[-1]))
    q.push_packed_nruns(bases, runs if len(runs) else None, off, len(allr))


@pytest.mark.gpu
@pytest.mark.parametrize("K,ks,layout", _sweep_params())
def test_tables_across_k(ctx, monkeypatch, tmp_path, K, ks, layout):
    sk, reads = _workload(K, 7 * K)
    G, n = len(sk), len(sk[0])
    keys = codec.sketches_to_keys(sk, K)
    refs = {m: oracle_c_run(keys, G, n, K, ks, lambda q: q.push_reads(reads), m[2], m[0], m[1]) for m in MODES}
    assert any(refs[m][0]["n_intersect"] for m in MODES)
    if layout is not None:
        monkeypatch.setenv("MLG_LAYOUT", str(layout))
    keep = []
    for precompute in ("1", "0"):
        monkeypatch.setenv("MLG_PRECOMPUTE_HITS", precompute)
        db = Database.from_keys(ctx, keys, G, n, K, ks)
        for i, m in enumerate(MODES):
            how = FORMS[(i + (precompute == "0")) % 4]
            if how == "nruns":
                monkeypatch.setenv("MLG_CHUNK_MB", "0.25")
            q = db.query(m[2], m[0], m[1])
            monkeypatch.delenv("MLG_CHUNK_MB", raising=False)
            _push_form(q, reads, how, keep)
            res = q.finish()
            ref, I_ref = refs[m]
            _check(res, q.intersection(), ref, I_ref, (precompute, m, how))
            if layout is not None:
                assert res["stats"]["layout"] == layout
            cm = (3, 255)[i % 2]
            q.dump_intersection(str(tmp_path / "dump"), None, cm)
            got = {a: int(b) for a, b in (ln.split() for ln in open(tmp_path / "dump"))}
            assert got == _dump_expected(sk, reads, K, I_ref, cm), (precompute, m, cm)
            q.close()
        db.close()



# ------------------------------------------------------------------------------------------------ 3. staging limits (GPU)
def _stage_bytes(p0, p1, base_words, nmask_words):
    """bytes of packed bases and of N mask a probe kernel stages for the tile of stream bases [p0, p1) (the `issue`
    lambda of csrc/probe.cu, probe_sk.cu and probe_mz.cu)"""
    bw0, bw1 = (p0 >> 5) & ~1, min(((p1 + 31) >> 5) + 6, base_words)
    bw1 = (bw1 + 1) & ~1
    mw0, mw1 = (p0 >> 6) & ~1, min(((p1 + 63) >> 6) + 4, nmask_words)
    mw1 = (mw1 + 1) & ~1
    return (bw1 - bw0) * 8, (mw1 - mw0) * 8


def _stage_limits(layout):
    """(reads per tile, staged base bytes, staged mask bytes) of the probe kernel of a layout"""
    if layout == 0:
        c = _constants("probe.cu", ("STAGE_B", "STAGE_M"))
        return _COMMON["RT"], c["STAGE_B"], c["STAGE_M"]
    if layout == 1:
        return 32, _COMMON["WSTAGE_B"], _COMMON["WSTAGE_M"]
    c = _constants("probe_mz.cu", ("MZ_TR", "MZ_STAGE_B", "MZ_STAGE_M"), {"MLG_RT": _COMMON["RT"]})
    return c["MZ_TR"], c["MZ_STAGE_B"], c["MZ_STAGE_M"]


def _staging_batch(rng, TR, SB):
    """read lengths of one batch, TR reads per tile: tiles whose staged base bytes are the limit SB (from base 0 and from
    inside a 64-base word), one 16-byte unit over and under it, a staged tile holding one read of several hundred bases,
    and a last tile of short reads, so that no tile of interest is clipped at the end of the batch"""
    short = (SB * 4 - 192) // TR - 4                     # TR - 1 such reads leave a few hundred bases below the limit
    lens = []
    for spec in (0, 16, -16, 0, "long", 16, 0):
        start = sum(lens)
        if spec == "long":
            tile = [rng.randint(60, 120) for _ in range(TR)]
            tile[rng.randrange(TR)] = rng.randint(500, 900)
            tile[-1] += (start + sum(tile)) % 64 == 0             # the next tile starts inside a word
        else:
            tile = [rng.randint(short - 2, short) for _ in range(TR - 1)]
            body = start + sum(tile)
            fit = [L for L in range(8 * SB) if _stage_bytes(start, body + L, 1 << 40, 1 << 40)[0] == SB + spec
                   and (body + L) % 64]
            tile.append(rng.choice(fit))
        lens += tile
    return lens + [rng.randint(60, 200) for _ in range(TR)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout,K", [pytest.param(L, K, id="L%d-K%d-limit-16-0+16" % (L, K)) for L, K in ((0, 31), (0, 63), (1, 60), (2, 60))])
def test_staging_limit(ctx, monkeypatch, layout, K):
    TR, SB, SM = _stage_limits(layout)
    rng = random.Random(900 + K + layout)
    lens = _staging_batch(rng, TR, SB)
    # the reads tile one genome end to end (each window once) and the sketches hold every K-mer of it: with ci_min = 1 a
    # single wrong base in any window changes the intersection
    G = 4
    n = (sum(lens) + G - 1) // G
    genome = _rand(rng, G * n + K - 1)
    reads, p = [], 0
    for L in lens:
        r = genome[p:p + L]
        p += L
        r = list(r if rng.random() < 0.5 else oracle_py.rc(r))
        for i in range(len(r)):
            u = rng.random()
            r[i] = "N" if u < 0.001 else (r[i].lower() if u < 0.01 else r[i])
        reads.append("".join(r))
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    nb = int(off[-1])
    nw64 = (nb + 63) // 64
    base_words, nmask_words = nw64 * 2, (nw64 + 1) // 2 * 2
    tiles = []
    for t in range(len(lens) // TR + (len(lens) % TR > 0)):
        r0, r1 = t * TR, min(len(lens), (t + 1) * TR)
        b, m = _stage_bytes(int(off[r0]), int(off[r1]), base_words, nmask_words)
        tiles.append((int(off[r0]), b, m, b <= SB and m <= SM, max(lens[r0:r1])))
    assert [b - SB for _, b, _, _, _ in tiles[:4]] + [tiles[5][1] - SB, tiles[6][1] - SB] == [0, 16, -16, 0, 16, 0], tiles
    assert [st for _, _, _, st, _ in tiles[:7]] == [True, False, True, True, True, False, True], tiles    # the mask never decides
    assert tiles[0][0] == 0 and all(p0 % 64 for p0, _, _, _, _ in tiles[1:7]), tiles
    assert tiles[4][4] >= 500
    sk = [[genome[p:p + K] if p % 3 else oracle_py.rc(genome[p:p + K]) for p in range(g * n, (g + 1) * n)] for g in range(G)]
    keys = codec.sketches_to_keys(sk, K)
    monkeypatch.setenv("MLG_LAYOUT", str(layout))
    db = Database.from_keys(ctx, keys, G, n, K, (K - 10, K))
    for ci, gate in ((1, "exact"), (1, "none")):
        ref, I_ref = oracle_c_run(keys, G, n, K, (K - 10, K), lambda q: q.push_reads(reads), ci, gate, True)
        assert ref["n_intersect"] > 0.5 * G * n
        q = db.query(ci, gate, True)
        q.push_reads(reads)
        res = q.finish()
        assert res["stats"]["layout"] == layout
        _check(res, q.intersection(), ref, I_ref, (layout, ci, gate))
        q.close()
    db.close()


# ------------------------------------------------------------------------------------------------ 4. read k-mers and KMC files
KMC_P = {5: 1, 6: 2, 7: 3, 8: 4, 10: 6, 31: 7, 32: 4, 33: 5, 34: 6, 58: 6, 60: 4}     # KMC's lut_prefix_length


@pytest.mark.gpu
@pytest.mark.parametrize("K", sorted(KMC_P), ids=lambda K: "K%d-p%d" % (K, KMC_P[K]))
def test_read_kmers_and_kmc_files_across_k(ctx, tmp_path, K):
    rng = random.Random(300 + K)
    batches = [_mixed_reads(rng, 60, K) for _ in range(2)]
    allreads = [r for b in batches for r in b]
    db = _small_db(ctx, K, allreads, (max(1, K - 20), K))
    cnt = oracle_py.count_read_kmers(allreads, K)
    archive, distinct = _measure(db, lambda q: [q.push_reads(b) for b in batches])
    single = db.query(2, "exact", True, read_kmers=True)
    passes = db.query(2, "exact", True, read_kmers=True, read_kmer_passes=True, read_kmer_budget=_budget(archive, distinct, 4))
    for q in (single, passes):
        for b in batches:
            q.push_reads(b)
    for mc, cm in ((1, 255), (2, 3)):
        want = _expected(allreads, K, mc, cm, cnt)
        for tag, q in (("single", single), ("passes", passes)):
            assert _records(*q.read_kmers(mc, cm), K) == want, (tag, mc, cm)
    assert passes.read_kmer_plan()["passes"] >= 2
    files = {}
    for tag, q in (("single", single), ("passes", passes)):
        prefix = str(tmp_path / tag)
        q.write_reads_kmc(prefix, 2, 3)
        hdr, recs = kmcdb.read(prefix)
        assert hdr["k"] == K and hdr["lut_prefix_length"] == KMC_P[K] and hdr["min_count"] == 2 and hdr["max_count"] == 3
        assert dict(recs) == _expected(allreads, K, 2, 3, cnt), tag
        keys, info, counts = ingest.read_kmc_database(prefix, with_counts=True)
        assert info["k"] == K and _records(keys, counts, K) == dict(recs), tag
        files[tag] = [open(prefix + ext, "rb").read() for ext in (".kmc_pre", ".kmc_suf")]
    assert files["single"] == files["passes"]
    res = single.finish()
    I = single.intersection()
    assert res["n_intersect"] > 0
    single.write_intersection_kmc(str(tmp_path / "inter"), 3)
    hdr, recs = kmcdb.read(str(tmp_path / "inter"))
    assert hdr["lut_prefix_length"] == KMC_P[K] and hdr["min_count"] == 1 and hdr["max_count"] == 3
    sk_mult = Counter(oracle_py.canon(s) for row in _small_db_sketches(K, allreads) for s in row if s)
    want = {x: min(cnt[x], sk_mult[x], 3) for x in (codec.key_to_kmer(int(a), int(b), K) for a, b in I)}
    assert dict(recs) == want
    keys, info, counts = ingest.read_kmc_database(str(tmp_path / "inter"), with_counts=True)
    assert _records(keys, counts, K) == want
    single.close(); passes.close(); db.close()


def _small_db_sketches(K, reads, seed=0):
    """the sketches test_gpu_read_kmers._small_db builds its database from"""
    rng = random.Random(seed)
    pool = [r[i:i + K].upper() for r in reads for i in range(0, max(0, len(r) - K + 1), 7)]
    pool = [s for s in pool if set(s) <= set("ACGT")] or ["A" * K]
    return [[rng.choice(pool) if rng.random() < 0.9 else "" for _ in range(6)] for _ in range(4)]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 2, 3, 4], ids=lambda K: "K%d" % K)
def test_kmc_files_refused_below_k5(ctx, tmp_path, K):
    reads = _mixed_reads(random.Random(K), 30, K)
    db = _small_db(ctx, K, reads, (K,))
    for passes in (False, True):
        q = db.query(1, "exact", True, read_kmers=True, read_kmer_passes=passes)
        q.push_reads(reads)
        assert _records(*q.read_kmers(1, 255), K) == _expected(reads, K, 1, 255)
        calls = [lambda p: q.write_reads_kmc(p, 2, 3)]
        if not passes:
            q.finish()
            calls.append(lambda p: q.write_intersection_kmc(p, 3))
        for i, call in enumerate(calls):
            prefix = str(tmp_path / ("out%d%d" % (passes, i)))
            with pytest.raises(MlgError) as e:
                call(prefix)
            assert e.value.code == ERR_ARG
            assert not os.path.exists(prefix + ".kmc_pre") and not os.path.exists(prefix + ".kmc_suf")
        q.close()
    db.close()


# ------------------------------------------------------------------------------------------------ 5. partial refinement level
@pytest.mark.gpu
@pytest.mark.parametrize("K", [15, 12], ids=lambda K: "K%d-b%d" % (K, K - 10))
def test_partial_refinement_level(ctx, tmp_path, K):
    """K - 10 < 10: a bin of 10 leading bases that must be split again is split by its last K - 10 (< 10) bases"""
    rng = random.Random(60 + K)
    reads = ["A" * 150] * 400 + ["T" * 120] * 100 + [("AC" * 80)[:150]] * 300 + [("GT" * 80)[:141]] * 50
    reads += [_rand(rng, 60) for _ in range(15)] + ["A" * 40 + "N" + "A" * 40]
    rng.shuffle(reads)
    db = _small_db(ctx, K, reads, (K,))
    archive, distinct = _measure(db, lambda q: q.push_reads(reads))
    lo, hi = _pass_bytes(1), _pass_bytes(4 ** (K - 10))
    cap = next(_pass_bytes(b) for b in (64, 8, 4, 2) if lo < _pass_bytes(b) < hi)
    q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=archive + cap)
    q.push_reads(reads)
    single = db.query(read_kmers=True)
    single.push_reads(reads)
    o = OracleReadKmers(K)
    o.push_reads(reads)
    for mc, cm in ((1, 255), (2, 3)):
        keys, counts = q.read_kmers(mc, cm)
        plan = q.read_kmer_plan()
        assert plan["refined_bins"] >= 1 and plan["passes"] >= 2, plan
        want = o.result(mc, cm)
        assert np.array_equal(keys, want[0]) and np.array_equal(counts, want[1]), (mc, cm)
    o.close()
    q.write_reads_kmc(str(tmp_path / "passes"), 2, 3)
    single.write_reads_kmc(str(tmp_path / "single"), 2, 3)
    for ext in (".kmc_pre", ".kmc_suf"):
        assert open(str(tmp_path / ("passes" + ext)), "rb").read() == open(str(tmp_path / ("single" + ext)), "rb").read(), ext
    q.close(); single.close(); db.close()
