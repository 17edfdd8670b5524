"""The read k-mer count across ranks (mlg_query_read_kmer_archive / _add_archive, mlg_kmc_concat), emulated on one GPU.
W ranks live in one process: one passes-mode Query per rank on a shared Database, each pushing its own shard of the
reads.  The test moves every rank's archive blob to every other rank itself, with torch copies on the library's compute
stream.  Rank r then counts share r of the canonical key order over all the reads; the shares in rank order must be the
output of one query over all the reads:

  - read_kmers(1, 255) of the ranks, concatenated in rank order, equals the single passes query's output;
  - the ranks' KMC databases joined by kmc_concat are byte-identical to the single passes query's file and to the
    single table's, and decode to the C oracle's records;
  - every rank finds the same share boundaries, by the rule of DESIGN.md section 10 (restated in _share_bounds below),
    and writes the same part whatever order the peers' archives were added in;
  - each share holds fewer than T / W + (the largest top-level bin) of the T windows, and every rank's `windows` is T,
    which is the sum of the ranks' n_kmers.

World sizes 1 to 16; contiguous, interleaved, one-empty-rank and all-on-one-rank shards; the four push forms rotated
across the ranks; K = 60, 31 and 9 (below 10 bases the top-level histogram has b = K bases); budgets under which a rank
with its fair share of the keys runs at least 4 passes, and poly-A reads whose bin has to be refined."""
import filecmp
import random

import numpy as np
import pytest

import synth  # noqa: F401  (builds the generators the oracle tests share)
from helpers import oracle_c_run
from metalign_b200 import codec, dist, ingest
from metalign_b200.api import Database, Exchange, MlgError, kmc_concat
from oracle import oracle_py
from oracle.read_kmers import OracleReadKmers
from test_gpu_read_kmer_passes import _pass_bytes
from test_gpu_read_kmers import _mixed_reads, _push

pytestmark = pytest.mark.gpu
ERR_ARG, ERR_STATE, ERR_NOMEM = -2, -4, -5
KS = {60: (30, 40, 50, 60), 31: (21, 31), 9: (7, 9)}
WORLDS = (1, 2, 3, 5, 8, 16)
SHARDINGS = ("contiguous", "interleaved", "empty_rank", "one_rank")
FORMS = ("ascii", "packed", "nruns", "device")
CASES = [(W, s) for W in WORLDS for s in SHARDINGS if W > 1 or s == "contiguous"]
POLY_A = 400


def _reads(K):
    rng = random.Random(500 + K)
    reads = _mixed_reads(rng, 150, K) + ["A" * 150] * POLY_A + [("AC" * 80)[:150]] * 50
    rng.shuffle(reads)
    return reads


def _db(ctx, K, reads):
    """a database of K-mers taken from the reads (G = 4, n = 6) and its keys, for the C oracle"""
    rng = random.Random(K)
    pool = [r[i:i + K].upper() for r in reads for i in range(0, max(0, len(r) - K + 1), 7)]
    pool = [s for s in pool if set(s) <= set("ACGT")]
    sk = [[rng.choice(pool) if rng.random() < 0.9 else "" for _ in range(6)] for _ in range(4)]
    keys = codec.sketches_to_keys(sk, K)
    return Database.from_keys(ctx, keys, 4, 6, K, KS[K]), keys


def _files_equal(a, b):
    return all(filecmp.cmp(a + ext, b + ext, shallow=False) for ext in (".kmc_pre", ".kmc_suf"))


class Ref:
    """one query over all the reads, in both modes, and the oracles"""

    def __init__(self, ctx, K, tmp):
        self.K, self.reads = K, _reads(K)
        self.db, self.keys = _db(ctx, K, self.reads)
        q = self.db.query(read_kmers=True, read_kmer_passes=True)
        q.push_reads(self.reads)
        self.all = q.read_kmers(1, 255)
        self.distinct = q.read_kmer_plan()["distinct"]
        self.passes_file = str(tmp / ("passes%d" % K))
        q.write_reads_kmc(self.passes_file, 2, 3)
        self.windows = q.read_kmer_stats()["windows"]
        q.close()
        s = self.db.query(read_kmers=True)
        s.push_reads(self.reads)
        self.single_file = str(tmp / ("single%d" % K))
        s.write_reads_kmc(self.single_file, 2, 3)
        s.close()
        o = OracleReadKmers(K)
        o.push_reads(self.reads)
        self.oracle = o.result(2, 3)
        o.close()
        # windows per top-level bin (the min(K, 10) leading bases of the canonical key), from the Python oracle
        b = min(K, 10)
        self.bins = np.zeros(4 ** b, dtype=np.int64)
        for kmer, c in oracle_py.count_read_kmers(self.reads, K).items():
            hi, lo = codec.kmer_to_key(kmer)
            self.bins[((int(hi) << 64 | int(lo)) >> (2 * (K - b)))] += c
        assert self.bins.sum() == self.windows


@pytest.fixture(scope="module")
def refs(ctx, tmp_path_factory):
    made, tmp = {}, tmp_path_factory.mktemp("refs")

    def get(K):
        if K not in made:
            made[K] = Ref(ctx, K, tmp)
        return made[K]
    yield get
    for r in made.values():
        r.db.close()


def _shards(kind, N, W):
    if kind == "contiguous":
        return [slice(*dist.shard_range(N, r, W)) for r in range(W)]
    if kind == "interleaved":
        return [slice(r, N, W) for r in range(W)]
    if kind == "empty_rank":
        rest = [slice(*dist.shard_range(N, r, W - 1)) for r in range(W - 1)]
        return rest[:W // 2] + [slice(0, 0)] + rest[W // 2:]
    return [slice(0, 0)] * (W - 1) + [slice(0, N)]


def _share_bounds(h, W):
    """DESIGN.md section 10: s_r = the first bin i with W * (windows before bin i) >= r * T; s_W = the number of bins"""
    before = np.concatenate([[0], np.cumsum(h)[:-1]])
    T = int(h.sum())
    s = [int(np.argmax(W * before >= r * T)) if (W * before >= r * T).any() else len(h) for r in range(W)]
    return s + [len(h)]


def _ranks(db, shard_reads, budget, keep, **kw):
    """one passes-mode query per rank; rank r pushes its reads in two batches in form FORMS[r % 4]"""
    qs = []
    for r, reads in enumerate(shard_reads):
        q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=budget, **kw)
        half = len(reads) // 2
        for b in (reads[:half], reads[half:]):
            if b:
                _push(q, b, FORMS[r % len(FORMS)], keep)
        qs.append(q)
    return qs


def _archives(qs):
    W = len(qs)
    return [q.read_kmer_archive(r, W) for r, q in enumerate(qs)]


def _move(db, qs, blobs, rng=None):
    """every rank's blob copied by torch on the compute stream, then added to every other rank (in a shuffled order with
    rng)"""
    import torch
    comp = torch.cuda.ExternalStream(db.ctx.streams()[0])
    with torch.cuda.stream(comp):
        copies = [dist.device_view_u8(p, n).clone() for p, n in blobs]
    for d, q in enumerate(qs):
        order = [r for r in range(len(qs)) if r != d]
        if rng is not None:
            rng.shuffle(order)
        for r in order:
            q.add_read_kmer_archive(copies[r].data_ptr(), copies[r].numel())
    return copies


def _write_parts(qs, prefix):
    parts = ["%s.part%d" % (prefix, r) for r in range(len(qs))]
    for q, p in zip(qs, parts):
        q.write_reads_kmc(p, 2, 3)
    return parts


@pytest.mark.parametrize("K", [60, 31, 9])
@pytest.mark.parametrize("world,sharding", CASES)
def test_shares_join_into_the_single_query_output(refs, tmp_path, K, world, sharding):
    R, W = refs(K), world
    shard_reads = [R.reads[s] for s in _shards(sharding, len(R.reads), W)]
    assert sum(len(x) for x in shard_reads) == len(R.reads)
    keep = []
    # no budget, peers added in rank order
    qs = _ranks(R.db, shard_reads, 0, keep)
    copies = _move(R.db, qs, _archives(qs))
    outs = [q.read_kmers(1, 255) for q in qs]
    assert np.array_equal(np.concatenate([o[0] for o in outs]), R.all[0])
    assert np.array_equal(np.concatenate([o[1] for o in outs]), R.all[1])
    plans = [q.read_kmer_plan() for q in qs]
    s = _share_bounds(R.bins, W)
    T, top = R.windows, int(R.bins.max())
    for r, pl in enumerate(plans):
        assert (pl["rank"], pl["world"], pl["peers_added"]) == (r, W, W - 1)
        assert (pl["share_first_bin"], pl["share_end_bin"]) == (s[r], s[r + 1]), (r, pl)
        assert pl["share_windows"] == int(R.bins[s[r]:s[r + 1]].sum())
        assert W * pl["share_windows"] < T + W * top or pl["share_windows"] == 0
        assert pl["distinct"] == len(outs[r][0])
        assert qs[r].read_kmer_stats()["windows"] == T
    parts = _write_parts(qs, str(tmp_path / "a"))
    joined = str(tmp_path / "joined")
    kmc_concat(joined, parts)
    assert _files_equal(joined, R.passes_file) and _files_equal(joined, R.single_file)
    fk, info, fc = ingest.read_kmc_database(joined, with_counts=True)
    assert np.array_equal(fk, R.oracle[0]) and np.array_equal(fc.astype(np.uint8), R.oracle[1]) and info["min_count"] == 2
    assert sum(q.finish()["n_kmers"] for q in qs) == T
    archive = plans[0]["archive_bytes"]
    assert all(pl["archive_bytes"] == archive for pl in plans)
    for q in qs:
        q.close()
    del copies

    # a budget of about 1 / (8 W) of the keys per pass, peers added in a shuffled order: the same parts
    per_pass = max(1, R.distinct // (8 * W))
    qs = _ranks(R.db, shard_reads, archive + _pass_bytes(per_pass), keep)
    copies = _move(R.db, qs, _archives(qs), random.Random(W * 100 + K))
    parts2 = _write_parts(qs, str(tmp_path / "b"))
    for r, (a, b) in enumerate(zip(parts, parts2)):
        assert _files_equal(a, b), r
    plans2 = [q.read_kmer_plan() for q in qs]
    for r, (pl, pl2) in enumerate(zip(plans, plans2)):
        assert (pl2["share_first_bin"], pl2["share_end_bin"]) == (pl["share_first_bin"], pl["share_end_bin"])
        if pl["distinct"] >= 4 * per_pass:
            assert pl2["passes"] >= 4, (r, pl2)
    assert max(pl2["passes"] for pl2 in plans2) >= 4
    if K >= 31:                                   # the rank whose share holds the poly-A bin (bin 0) splits it
        owner = next(r for r in range(W) if s[r] == 0 and s[r + 1] > 0)
        assert plans2[owner]["refined_bins"] >= 1, plans2[owner]
    for q in qs:
        q.close()
    del copies


def test_pushes_launch_what_they_launched_before(refs):
    """the pushes of a rank launch the kernels of a plain query's pushes; packing the archive launches none"""
    R = refs(60)
    keep = []
    for how in FORMS:
        plain = R.db.query()
        _push(plain, R.reads[:200], how, keep)
        q = R.db.query(read_kmers=True, read_kmer_passes=True)
        _push(q, R.reads[:200], how, keep)
        q.sync(); plain.sync()
        n = plain.stats()["gpu_launches"]
        assert q.stats()["gpu_launches"] == n, how
        q.read_kmer_archive(0, 2)
        assert q.stats()["gpu_launches"] == n, how
        plain.close(); q.close()


def _gather(db, qs, exs):
    import torch
    comp = torch.cuda.ExternalStream(db.ctx.streams()[0])
    for q, ex in zip(qs, exs):
        q.exchange_pack(ex)
    with torch.cuda.stream(comp):
        allsend = torch.cat([dist.device_view_i64(ex.send_ptr, ex.block_words) for ex in exs])
        for ex in exs:
            dist.device_view_i64(ex.recv_ptr, ex.block_words * len(exs)).copy_(allsend)
    for q, ex in zip(qs, exs):
        q.exchange_merge(ex)
    return allsend


@pytest.mark.parametrize("when", ["before", "after"])
def test_with_a_counter_exchange(refs, tmp_path, when):
    """a gather-form counter exchange before the archives move, or after the parts are written: finish() equals the C
    oracle on every rank and the joined file is unchanged"""
    R, W = refs(60), 3
    shard_reads = [R.reads[s] for s in _shards("interleaved", len(R.reads), W)]
    qs = _ranks(R.db, shard_reads, 0, [], ci_min=2)
    exs = [Exchange(R.db.ctx, W, r, R.db.n_distinct) for r in range(W)]
    keep = []
    if when == "before":
        keep.append(_gather(R.db, qs, exs))
    copies = _move(R.db, qs, _archives(qs))
    parts = _write_parts(qs, str(tmp_path / "p"))
    if when == "after":
        keep.append(_gather(R.db, qs, exs))
    results = [q.finish() for q in qs]
    text = "".join(R.reads).encode()
    off = np.concatenate([[0], np.cumsum([len(x) for x in R.reads])]).astype(np.uint64)
    ref, I_ref = oracle_c_run(R.keys, 4, 6, 60, KS[60], lambda o: o.push_ascii(text, off), 2, "exact", True)
    for q, res in zip(qs, results):
        assert np.array_equal(res["num"], ref["num"]) and np.array_equal(res["den"], ref["den"])
        assert np.array_equal(res["ci"], ref["ci"]) and np.array_equal(q.intersection(), I_ref)
    assert sum(res["n_kmers"] for res in results) == ref["n_kmers"]
    joined = str(tmp_path / "joined")
    kmc_concat(joined, parts)
    assert _files_equal(joined, R.passes_file)
    parts2 = _write_parts(qs, str(tmp_path / "again"))      # after finish and the exchange: the same parts
    for a, b in zip(parts, parts2):
        assert _files_equal(a, b)
    for q in qs:
        q.close()
    for ex in exs:
        ex.close()
    del copies, keep


def _code(call):
    with pytest.raises(MlgError) as e:
        call()
    return e.value.code


def _tampered(blob, word, value):
    import torch
    t = dist.device_view_u8(*blob).clone()
    t.view(torch.int64)[word] = value
    torch.cuda.synchronize()
    return t


def test_refusals(refs, tmp_path):
    import torch
    R, W = refs(60), 3
    shard_reads = [R.reads[s] for s in _shards("contiguous", len(R.reads), W)]
    # modes without archives, bad ranks and worlds, a second call, pushes after it, adds before it
    for q in (R.db.query(read_kmers=True), R.db.query()):
        assert _code(lambda: q.read_kmer_archive(0, 2)) == ERR_STATE
        q.close()
    q = R.db.query(read_kmers=True, read_kmer_passes=True)
    q.push_reads(shard_reads[0])
    assert _code(lambda: q.add_read_kmer_archive(1, 8)) == ERR_STATE
    for rank, world in ((0, 0), (0, 17), (3, 3), (16, 16)):
        assert _code(lambda: q.read_kmer_archive(rank, world)) == ERR_ARG
    q.read_kmer_archive(0, 16)
    assert _code(lambda: q.read_kmer_archive(0, 16)) == ERR_STATE
    assert _code(lambda: q.push_reads(shard_reads[0])) == ERR_STATE
    assert _code(lambda: q.read_kmers()) == ERR_STATE                 # 15 peers missing
    q.close()

    qs = _ranks(R.db, shard_reads, 0, [])
    qs[0].finish()                                                     # archives may be packed after finish
    blobs = _archives(qs)
    torch.cuda.synchronize()
    hdr = dist.device_view_i64(blobs[1][0], 6).cpu().tolist()
    nb = hdr[4]
    desc = dist.device_view_i64(blobs[1][0], 6 + 6 * nb).cpu().tolist()[6:]
    # the first batch with offsets: where its offsets start, and how many reads it has
    at, off_word, n_reads = 6 + 6 * nb, None, 0
    for i in range(nb):
        d = desc[6 * i:6 * i + 6]
        if d[5] & 2 and d[0] >= 2:
            off_word, n_reads = at + d[3] + (d[4] if d[5] & 1 else 0), d[0]
            break
        at += d[3] + (d[4] if d[5] & 1 else 0) + ((d[0] + 1) if d[5] & 2 else 0)
    assert off_word is not None
    other_K = Database.from_sketches(R.db.ctx, [["A" * 31] * 2], 31, (31,))
    qk = other_K.query(read_kmers=True, read_kmer_passes=True)
    qk.push_reads(shard_reads[1])
    blob_k = qk.read_kmer_archive(1, W)
    qw = R.db.query(read_kmers=True, read_kmer_passes=True)
    qw.push_reads(shard_reads[1])
    blob_w = qw.read_kmer_archive(1, W + 1)
    bad = {
        "magic": _tampered(blobs[1], 0, 0),
        "tag": _tampered(blobs[1], 1, (hdr[1] >> 32 << 32) | 0x1234),
        "rank past world": _tampered(blobs[1], 2, (W << 32) | W),
        "bytes": _tampered(blobs[1], 5, hdr[5] + 8),
        "descriptor": _tampered(blobs[1], 6 + 1, 1 << 50),
        "offsets descend": _tampered(blobs[1], off_word + n_reads // 2, 1 << 40),
        "first offset": _tampered(blobs[1], off_word, 1),
    }
    for what, t in bad.items():
        assert _code(lambda: qs[0].add_read_kmer_archive(t.data_ptr(), t.numel())) == ERR_ARG, what
    assert _code(lambda: qs[0].add_read_kmer_archive(blobs[1][0], blobs[1][1] - 8)) == ERR_ARG
    assert _code(lambda: qs[0].add_read_kmer_archive(blobs[1][0] + 4, blobs[1][1] - 8)) == ERR_ARG   # misaligned
    assert _code(lambda: qs[0].add_read_kmer_archive(blob_k[0], blob_k[1])) == ERR_ARG        # K
    assert _code(lambda: qs[0].add_read_kmer_archive(blob_w[0], blob_w[1])) == ERR_ARG        # world
    assert _code(lambda: qs[0].add_read_kmer_archive(blobs[0][0], blobs[0][1])) == ERR_ARG    # its own
    # none of that changed anything: the real blobs still make the single query's file
    copies = _move(R.db, qs, blobs)
    assert _code(lambda: qs[0].add_read_kmer_archive(copies[1].data_ptr(), copies[1].numel())) == ERR_ARG   # twice
    parts = _write_parts(qs, str(tmp_path / "p"))
    joined = str(tmp_path / "joined")
    kmc_concat(joined, parts)
    assert _files_equal(joined, R.passes_file)
    for x in qs + [qk, qw]:
        x.close()
    other_K.close()
    del copies, bad

    # a query that never packed its archive still refuses after a counter exchange
    q = R.db.query(read_kmers=True, read_kmer_passes=True)
    q.push_reads(shard_reads[0])
    q.counts_export_sparse()
    assert _code(lambda: q.read_kmers()) == ERR_STATE
    q.close()


def test_overflow_reaches_every_rank(refs, tmp_path):
    """one rank's archive outgrew its budget at push time: its blob is a flagged header, and every rank's output calls
    return MLG_ERR_NOMEM and leave no file.  A rank whose budget holds its own archive but not its peers' overflows on
    import."""
    R, W = refs(31), 3
    shard_reads = [R.reads[s] for s in _shards("contiguous", len(R.reads), W)]
    keep = []
    qs = [R.db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=1024 if r == 1 else 0) for r in range(W)]
    for q, reads in zip(qs, shard_reads):
        _push(q, reads, "ascii", keep)
    blobs = _archives(qs)
    assert blobs[1][1] == 48 and blobs[0][1] > 48
    copies = _move(R.db, qs, blobs)
    for r, q in enumerate(qs):
        assert _code(lambda: q.read_kmers()) == ERR_NOMEM, r
        path = str(tmp_path / ("part%d" % r))
        assert _code(lambda: q.write_reads_kmc(path)) == ERR_NOMEM, r
        assert q.read_kmer_stats()["overflowed"] == 1
        for ext in (".kmc_pre", ".kmc_suf"):
            assert not (tmp_path / ("part%d%s" % (r, ext))).exists()
        q.close()
    del copies

    qs = _ranks(R.db, shard_reads, 0, keep)
    own = _archives(qs)[0][1]
    tight = R.db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=own + 4096)
    _push(tight, shard_reads[0], FORMS[0], keep)
    for q in qs:
        q.close()
    qs = [tight] + _ranks(R.db, shard_reads[1:], 0, keep)
    blobs = [tight.read_kmer_archive(0, W)] + [q.read_kmer_archive(r + 1, W) for r, q in enumerate(qs[1:])]
    copies = _move(R.db, qs, blobs)
    assert _code(lambda: tight.write_reads_kmc(str(tmp_path / "tight"))) == ERR_NOMEM
    assert not (tmp_path / "tight.kmc_suf").exists() and not (tmp_path / "tight.kmc_pre").exists()
    assert tight.read_kmer_stats()["bytes_needed"] > own
    for q in qs:
        q.close()
    del copies
