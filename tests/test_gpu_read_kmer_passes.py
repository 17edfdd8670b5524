"""Read k-mers in key-range passes (mlg_query_enable_read_kmer_passes): the pushes keep a device copy of the reads, and
every output call counts it in passes over contiguous intervals of the canonical key order.  The results must be those
of the single table (tests/test_gpu_read_kmers.py) and of the oracles, whatever the number of passes."""
import ctypes as C
import filecmp
import os
import random
import subprocess

import numpy as np
import pytest

import kmcdb
import synth
from conftest import ROOT
from metalign_b200 import _lib, codec, ingest, select_db
from metalign_b200.api import Database, MlgError
from oracle import oracle_py
from oracle.read_kmers import OracleReadKmers
from test_gpu_read_kmers import CASE, DATA, _expected, _fixture_reads, _mixed_reads, _push, _records, _run_dropin, _small_db

ERR_ARG, ERR_IO, ERR_STATE, ERR_NOMEM = -2, -3, -4, -5
OUT_BYTES_PER_KEY = 104      # RK_OUT_BYTES_PER_KEY of csrc/readkmers.cu


def _pass_bytes(bound):
    """device bytes of one pass whose keys are bounded by `bound` (pass_bytes in csrc/readkmers.cu)"""
    s = 1 << 12
    while s * 0.7 < bound:
        s *= 2
    return s * 16 + bound * OUT_BYTES_PER_KEY


def _budget(archive_bytes, distinct, parts):
    """a budget under which no pass holds more than about distinct / parts * 1.4 keys: the plan's bounds add up to at
    least the distinct keys, so there are more than parts / 1.4 passes"""
    return archive_bytes + _pass_bytes(max(1, distinct // parts))


def _ascending(keys):
    return bool(np.all(np.diff(keys[:, 0].astype(object) * (1 << 64) + keys[:, 1].astype(object)) > 0))


def _measure(db, pushes):
    """archive bytes and distinct keys of a read set, from a passes-mode query without a budget"""
    q = db.query(read_kmers=True, read_kmer_passes=True)
    pushes(q)
    q.read_kmers(1, 255)
    plan = q.read_kmer_plan()
    q.close()
    assert plan["passes"] >= 1 and plan["archive_bytes"] > 0
    return plan["archive_bytes"], plan["distinct"]


# ------------------------------------------------------------------------------------------------------------ CPU
def test_plan_struct_matches_header(tmp_path):
    src = tmp_path / "plan.c"
    fields = [f for f, _ in _lib.ReadKmerPlan._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "metalign_b200.h"\nint main(void) {\n'
                   '    printf("%zu\\n", sizeof(mlg_read_kmer_plan));\n'
                   + "".join('    printf("%%zu\\n", offsetof(mlg_read_kmer_plan, %s));\n' % f for f in fields) + "    return 0;\n}\n")
    exe = tmp_path / "plan"
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got[0] == C.sizeof(_lib.ReadKmerPlan)
    assert got[1:] == [getattr(_lib.ReadKmerPlan, f).offset for f in fields]


def test_select_parseargs_read_kmer_passes():
    assert select_db.select_parseargs(["r.fq", "data"]).read_kmer_passes is False
    assert select_db.select_parseargs(["r.fq", "data", "--read_kmer_passes"]).read_kmer_passes is True


def test_library_exports_the_passes_symbols():
    L = C.CDLL(_lib.build())
    for name in ("mlg_query_enable_read_kmer_passes", "mlg_query_read_kmer_plan"):
        assert hasattr(L, name) and name in _lib.SIGNATURES


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("K,ks", [(60, (30, 40, 50, 60)), (31, (21, 31)), (9, (7, 9))])
def test_passes_match_the_oracle_and_the_single_table(ctx, K, ks):
    rng = random.Random(100 + K)
    batches = [_mixed_reads(rng, 120, K) for _ in range(3)]
    allreads = [r for b in batches for r in b]
    db = _small_db(ctx, K, allreads, ks)
    cnt = oracle_py.count_read_kmers(allreads, K)
    single = db.query(read_kmers=True)
    for b in batches:
        single.push_reads(b)
    single.sync()
    for how in ("ascii", "packed", "nruns", "device"):
        keep = []
        archive, distinct = _measure(db, lambda q: [_push(q, b, how, keep) for b in batches])
        q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=_budget(archive, distinct, 8))
        for b in batches:
            _push(q, b, how, keep)
        q.sync()
        for mc, cm in ((1, 255), (2, 3), (5, 10)):
            keys, counts = q.read_kmers(mc, cm)
            assert q.read_kmer_plan()["passes"] >= 4, (how, q.read_kmer_plan())
            assert _records(keys, counts, K) == _expected(allreads, K, mc, cm, cnt), (how, mc, cm)
            assert _ascending(keys)
            sk, sc = single.read_kmers(mc, cm)
            assert np.array_equal(keys, sk) and np.array_equal(counts, sc), (how, mc, cm)
        plan = q.read_kmer_plan()
        assert plan["distinct"] == single.read_kmer_stats()["distinct"] and plan["ms_count"] > 0
        q.close()
    single.close()
    db.close()


@pytest.mark.gpu
def test_low_complexity_bins_are_refined(ctx):
    K = 31
    rng = random.Random(7)
    reads = ["A" * 150] * 3000 + ["C" * 150] * 1500 + ["G" * 150] * 1500 + [("ACGT" * 40)[:150]] * 2000
    reads += ["".join(rng.choice("ACGT") for _ in range(150)) for _ in range(300)]
    rng.shuffle(reads)
    db = _small_db(ctx, K, reads, (21, 31))
    archive, distinct = _measure(db, lambda q: q.push_reads(reads))
    # one pass holds about 1/50 of the distinct keys; the poly-A bin alone holds 3000 * 120 windows
    q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=_budget(archive, distinct, 50))
    q.push_reads(reads)
    for mc, cm in ((1, 255), (2, 3)):
        keys, counts = q.read_kmers(mc, cm)
        assert _records(keys, counts, K) == _expected(reads, K, mc, cm) and _ascending(keys)
        plan = q.read_kmer_plan()
        assert plan["refined_bins"] >= 1 and plan["passes"] >= 2, plan
    q.close()
    db.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mc,cm", [(2, 3), (1, 255)])
def test_written_files_equal_the_single_table(ctx, tmp_path, mc, cm):
    rng = random.Random(31)
    batches = [_mixed_reads(rng, 150, 60) for _ in range(2)]
    allreads = [r for b in batches for r in b]
    db = _small_db(ctx, 60, allreads, (30, 40, 50, 60))
    archive, distinct = _measure(db, lambda q: [q.push_reads(b) for b in batches])
    single = db.query(read_kmers=True)
    passes = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=_budget(archive, distinct, 8))
    for q in (single, passes):
        for b in batches:
            q.push_reads(b)
    single.write_reads_kmc(str(tmp_path / "single"), mc, cm)
    passes.write_reads_kmc(str(tmp_path / "passes"), mc, cm)
    assert passes.read_kmer_plan()["passes"] >= 4
    for ext in (".kmc_pre", ".kmc_suf"):
        assert filecmp.cmp(str(tmp_path / ("single" + ext)), str(tmp_path / ("passes" + ext)), shallow=False), ext
    st = passes.read_kmer_stats()
    assert st["out_records"] == single.read_kmer_stats()["out_records"] and st["out_bytes"] > 0
    _, recs = kmcdb.read(str(tmp_path / "passes"))
    assert dict(recs) == _expected(allreads, 60, mc, cm)
    single.close(); passes.close(); db.close()


@pytest.mark.gpu
def test_dropin_with_passes(ctx, tmp_path):
    # the budget the drop-in gets, found on the same reads pushed the way the drop-in pushes them
    reads = _fixture_reads()
    db = Database.load(ctx, os.path.join(DATA, "cmash_db_n1000_k60.mlgdb"))
    bases, nmask, off = codec.pack_reads(reads)
    runs = codec.nmask_to_runs(nmask, int(off[-1]))

    def push(q):
        q.push_packed_nruns(bases, runs if len(runs) else None, off, len(reads))
    archive, distinct = _measure(db, push)
    budget = _budget(archive, distinct, 8)
    q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=budget)
    push(q)
    q.write_reads_kmc(str(tmp_path / "probe"), 2, 3)
    assert q.read_kmer_plan()["passes"] >= 4
    q.close()
    db.close()
    plain = _run_dropin(tmp_path / "plain", "reads.fq")
    out = _run_dropin(tmp_path / "passes", "reads.fq", read_kmer_passes=True, read_kmer_budget=budget)
    for ext in (".kmc_pre", ".kmc_suf"):
        assert filecmp.cmp(str(out / ("reads_60mers" + ext)), str(plain / ("reads_60mers" + ext)), shallow=False)
    _, recs = kmcdb.read(str(out / "reads_60mers"))
    _, golden = kmcdb.read(os.path.join(CASE, "expected_default", "reads_60mers"))
    assert dict(recs) == dict(golden) and len(recs) == 13138
    exp = os.path.join(CASE, "expected_default")
    for name in ("cmash_query_results.csv", "cmashed_db.fna", "subset_db_info.txt", "60mers_intersection_dump",
                 "60mers_intersection.kmc_pre", "60mers_intersection.kmc_suf"):
        assert filecmp.cmp(str(out / name), os.path.join(exp, name), shallow=False), name
    # a budget below the copy of the reads: reads_60mers is skipped, everything else is written
    small = _run_dropin(tmp_path / "small", "reads.fq", read_kmer_passes=True, read_kmer_budget=archive // 2)
    for name in ("cmash_query_results.csv", "cmashed_db.fna", "subset_db_info.txt", "60mers_intersection_dump",
                 "60mers_intersection.kmc_pre", "60mers_intersection.kmc_suf"):
        assert filecmp.cmp(str(small / name), os.path.join(exp, name), shallow=False), name
    assert not os.path.exists(small / "reads_60mers.kmc_pre") and not os.path.exists(small / "reads_60mers.kmc_suf")


@pytest.mark.gpu
def test_passes_change_nothing_else(ctx):
    rng = random.Random(5)
    batches = [_mixed_reads(rng, 80, 60) for _ in range(3)]
    db = _small_db(ctx, 60, [r for b in batches for r in b], (30, 40, 50, 60))
    plain, passes = db.query(), db.query(read_kmers=True, read_kmer_passes=True)
    for q in (plain, passes):
        for b in batches:
            q.push_reads(b)
    r_plain, r_passes = plain.finish(), passes.finish()
    for k in ("num", "den", "ci", "n_intersect", "n_kmers"):
        assert np.array_equal(r_plain[k], r_passes[k]), k
    assert np.array_equal(plain.intersection(), passes.intersection())
    # three ASCII pushes (pack + probe each) and the finish stage: the archive copies launch no kernel
    assert r_plain["stats"]["gpu_launches"] == 9 and r_passes["stats"]["gpu_launches"] == 9
    passes.read_kmers()
    assert passes.read_kmer_stats()["windows"] == r_passes["n_kmers"]
    plain.close(); passes.close(); db.close()


@pytest.mark.gpu
def test_edges_and_errors(ctx, tmp_path):
    reads = _mixed_reads(random.Random(9), 40, 60)
    db = _small_db(ctx, 60, reads, (30, 40, 50, 60))
    # no push, and only reads shorter than K: an empty, valid database
    for pushed in ([], ["ACGT" * 10, "A" * 59]):
        q = db.query(read_kmers=True, read_kmer_passes=True)
        if pushed:
            q.push_reads(pushed)
        keys, counts = q.read_kmers()
        assert keys.shape == (0, 2) and counts.shape == (0,)
        q.write_reads_kmc(str(tmp_path / "empty"), 2, 3)
        hdr, recs = kmcdb.read(str(tmp_path / "empty"))
        assert recs == [] and hdr["k"] == 60
        fk, info, _ = ingest.read_kmc_database(str(tmp_path / "empty"), with_counts=True)
        assert len(fk) == 0
        q.close()
    # enabling after a push, or both modes
    q = db.query()
    q.push_reads(reads)
    assert _lib.lib().mlg_query_enable_read_kmer_passes(q._h, 0) == ERR_STATE
    q.close()
    q = db.query(read_kmers=True)
    assert _lib.lib().mlg_query_enable_read_kmer_passes(q._h, 0) == ERR_STATE
    q.close()
    q = db.query(read_kmers=True, read_kmer_passes=True)
    assert _lib.lib().mlg_query_enable_read_kmers(q._h, 0) == ERR_STATE
    with pytest.raises(MlgError) as e:
        db.query().read_kmer_plan()
    assert e.value.code == ERR_STATE
    q.close()
    # K > 60
    reads61 = _mixed_reads(random.Random(9), 40, 61)
    db61 = _small_db(ctx, 61, reads61, (41, 61))
    with pytest.raises(MlgError) as e:
        db61.query(read_kmers=True, read_kmer_passes=True)
    assert e.value.code == ERR_ARG
    db61.close()
    # after a counter exchange
    q = db.query(read_kmers=True, read_kmer_passes=True)
    q.push_reads(reads)
    q.counts_export_sparse()
    for call in (lambda: q.read_kmers(), lambda: q.write_reads_kmc(str(tmp_path / "x"))):
        with pytest.raises(MlgError) as e:
            call()
        assert e.value.code == ERR_STATE
    q.close()
    # an archive over the budget: the query goes on, the output calls do not; bytes_needed covers every batch pushed
    q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=1024)
    plain = db.query()
    for x in (q, plain):
        x.push_reads(reads)
        x.push_reads(reads)
    rq, rp = q.finish(), plain.finish()
    assert np.array_equal(rq["num"], rp["num"]) and np.array_equal(rq["ci"], rp["ci"])
    for call in (lambda: q.read_kmers(), lambda: q.write_reads_kmc(str(tmp_path / "y"))):
        with pytest.raises(MlgError) as e:
            call()
        assert e.value.code == ERR_NOMEM
    assert q.read_kmer_stats()["overflowed"] == 1
    assert q.read_kmer_stats()["bytes_needed"] == _measure(db, lambda x: [x.push_reads(reads), x.push_reads(reads)])[0]
    assert not os.path.exists(str(tmp_path / "y.kmc_suf")) and not os.path.exists(str(tmp_path / "y.kmc_pre"))
    q.close(); plain.close()
    # a budget that holds the archive but not the smallest pass
    archive, _ = _measure(db, lambda q: q.push_reads(reads))
    q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=archive + 1000)
    q.push_reads(reads)
    with pytest.raises(MlgError) as e:
        q.read_kmers()
    assert e.value.code == ERR_NOMEM and q.read_kmer_stats()["overflowed"] == 0
    with pytest.raises(MlgError) as e:
        q.write_reads_kmc(str(tmp_path / "z"))
    assert e.value.code == ERR_NOMEM                                  # and no partial database is left behind
    assert not os.path.exists(str(tmp_path / "z.kmc_suf")) and not os.path.exists(str(tmp_path / "z.kmc_pre"))
    q.close()
    # an unwritable prefix
    q = db.query(read_kmers=True, read_kmer_passes=True)
    q.push_reads(reads)
    with pytest.raises(MlgError) as e:
        q.write_reads_kmc(str(tmp_path / "no" / "such" / "dir"))
    assert e.value.code == ERR_IO
    q.close()
    db.close()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["ascii", "nruns"])
def test_batches_with_offsets_beyond_one_grid_sweep(ctx, how):
    """one batch of reads of varied length (offsets, N runs) far longer than one sweep of the grid (sm_count * 16 CTAs x
    256 bases, ~0.6 M bases on a B200): every CTA walks many tiles, each with the reads it spans"""
    K = 31
    rng = np.random.default_rng(17)
    lens = rng.integers(20, 400, size=16000)
    reads = []
    for L in lens:
        r = np.array(list("ACGT"))[rng.integers(0, 4, size=L)]
        if rng.random() < 0.2:
            a = int(rng.integers(0, L))
            r[a:a + int(rng.integers(1, 6))] = "N"
        reads.append("".join(r))
    assert sum(lens) > 4 * 148 * 16 * 256
    db = _small_db(ctx, K, reads[:200], (21, 31))
    archive, distinct = _measure(db, lambda q: _push(q, reads, how, []))
    q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=_budget(archive, distinct, 4))
    _push(q, reads, how, [])
    got = q.read_kmers(1, 255)
    assert q.read_kmer_plan()["passes"] >= 2
    o = OracleReadKmers(K)
    o.push_reads(reads)
    want = o.result(1, 255)
    o.close()
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    res = q.finish()
    assert q.read_kmer_stats()["windows"] == res["n_kmers"]
    q.close()
    db.close()


@pytest.mark.gpu
def test_scale_two_million_reads_in_passes(ctx, tmp_path):
    """about 2 M reads of the bench's generator with 1/8 of the single table's bytes: every record equals the C oracle's"""
    p = synth.params(G=2000, n=1000, seed=20200529, n_present=500, read_len=150)
    keys = synth.sketch_keys(p)
    db = Database.from_keys(ctx, keys, p.G, p.n, 60)
    packed = [synth.reads_packed(p, r0, n) + (n,) for r0, n in ((0, 1_000_000), (1_000_000, 1_000_000))]
    single = db.query(read_kmers=True)
    for b, m, n in packed:
        single.push_packed(b, m, None, n, p.read_len)
    single.sync()
    budget = single.read_kmer_stats()["bytes"] // 8
    single.close()
    q = db.query(read_kmers=True, read_kmer_passes=True, read_kmer_budget=budget)
    o = OracleReadKmers(60)
    for b, m, n in packed:
        q.push_packed(b, m, None, n, p.read_len)
        o.push_packed(b, m, None, n, p.read_len)
    got, want = q.read_kmers(1, 255), o.result(1, 255)
    plan = q.read_kmer_plan()
    assert plan["passes"] >= 8 and plan["archive_bytes"] + plan["pass_cap_bytes"] == budget, plan
    assert got[0].shape == want[0].shape and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    q.write_reads_kmc(str(tmp_path / "reads"), 2, 3)
    fk, info, fc = ingest.read_kmc_database(str(tmp_path / "reads"), with_counts=True)
    wk, wc = o.result(2, 3)
    assert np.array_equal(fk, wk) and np.array_equal(fc.astype(np.uint8), wc) and info["min_count"] == 2
    res = q.finish()
    st = q.read_kmer_stats()
    assert st["windows"] == res["n_kmers"] and st["distinct"] == len(got[0])
    q.close()
    o.close()
    db.close()
