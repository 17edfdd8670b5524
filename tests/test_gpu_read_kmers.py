"""The read k-mer table (mlg_query_enable_read_kmers and the calls after it): every canonical K-mer of the pushed reads
counted on the GPU, and the two KMC databases the reference keeps with --keep_temp_files (reads_60mers,
60mers_intersection).  Checked against the reference-driven fixture, oracle_py (small inputs) and the C oracle's
all-k-mer counter (larger ones)."""
import argparse
import ctypes as C
import filecmp
import gzip
import os
import random

import numpy as np
import pytest

import kmcdb
import synth
from conftest import ROOT
from helpers import adversarial_case
from metalign_b200 import _lib, codec, ingest, select_db
from metalign_b200.api import Database, MlgError
from oracle import oracle_py
from oracle.read_kmers import OracleReadKmers

CASE = os.path.join(ROOT, "tests", "golden", "ref_e2e_case")
DATA = os.path.join(CASE, "data")
ERR_ARG, ERR_IO, ERR_STATE, ERR_NOMEM = -2, -3, -4, -5


def _records(keys, counts, K):
    return {codec.key_to_kmer(int(a), int(b), K): int(c) for (a, b), c in zip(keys, counts)}


def _expected(reads, K, min_count, counter_max, cnt=None):
    cnt = cnt if cnt is not None else oracle_py.count_read_kmers(reads, K)
    return {x: min(c, counter_max) for x, c in cnt.items() if c >= min_count}


def _fixture_reads(name="reads.fq"):
    if name.endswith(".gz"):
        with gzip.open(os.path.join(CASE, name), "rt") as f:
            lines = f.read().split("\n")
        return [lines[i + 1] for i in range(0, len(lines) - 1, 2)]
    with open(os.path.join(CASE, name)) as f:
        lines = f.read().split("\n")
    return [lines[i + 1] for i in range(0, len(lines) - 1, 4)]


def _run_dropin(tmp_path, rfile, **over):
    d = dict(reads=os.path.join(CASE, rfile), data=DATA, cmash_results="NONE", cutoff=0.01, db="AUTO", db_dir="AUTO",
             dbinfo_in="AUTO", dbinfo_out="AUTO", input_type="AUTO", keep_temp_files=True, strain_level=False,
             temp_dir=str(tmp_path / "out"), threads=4)          # the `default` Namespace of test_ref_e2e.py
    d.update(over)
    select_db.select_main(argparse.Namespace(**d))
    return tmp_path / "out"


def _small_db(ctx, K, reads, ks=None, seed=0):
    """a database of K-mers taken from the reads (so that the query has an intersection), G = 4, n = 6"""
    rng = random.Random(seed)
    pool = [r[i:i + K].upper() for r in reads for i in range(0, max(0, len(r) - K + 1), 7)]
    pool = [s for s in pool if set(s) <= set("ACGT")] or ["A" * K]
    sk = [[rng.choice(pool) if rng.random() < 0.9 else "" for _ in range(6)] for _ in range(4)]
    return Database.from_sketches(ctx, sk, K, tuple(ks or (K,)))


def _mixed_reads(rng, n, K):
    """N runs, lower case, reads shorter than K, exactly K, 150 bp and 161-5000 bp, and one k-mer repeated > 300 times"""
    genome = "".join(rng.choice("ACGT") for _ in range(20000))
    reads = []
    for i in range(n):
        L = rng.choice([1, K - 1, K, K + 1, 150, 150, 161, rng.randint(162, 5000)])
        a = rng.randint(0, len(genome) - L)
        r = list(genome[a:a + L])
        if rng.random() < 0.5:
            r = list(oracle_py.rc("".join(r)))
        for j in range(len(r)):
            x = rng.random()
            if x < 0.01:
                r[j] = "N"
            elif x < 0.03:
                r[j] = r[j].lower()
        if rng.random() < 0.05 and len(r) > 40:
            r[10:10 + rng.randint(1, 30)] = "N" * 5
        reads.append("".join(r))
    reads.append(("ACGT" * 100)[:K + 340])                          # one k-mer family >300 times: counts saturate, never wrap
    reads.append("A" * (K + 400))
    return reads


def _push(q, reads, how, keep):
    if how == "ascii":
        q.push_reads(reads)
        return
    bases, nmask, off = codec.pack_reads(reads)
    if how == "packed":
        q.push_packed(bases, nmask, off, len(reads))
    elif how == "nruns":
        runs = codec.nmask_to_runs(nmask, int(off[-1]))
        q.push_packed_nruns(bases, runs if len(runs) else None, off, len(reads))
    else:                                                           # device buffers
        import torch
        t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (bases, nmask, off.view(np.int64))]
        keep.append(t)
        q.push_packed_ptr(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), len(reads), device=True)


# ------------------------------------------------------------------------------------------------------------ CPU
def test_oracle_c_read_kmers_match_oracle_py():
    rng = random.Random(11)
    for _ in range(150):
        c = adversarial_case(rng)
        o = OracleReadKmers(c["K"])
        o.push_reads(c["reads"])
        for mc, cm in ((1, 255), (2, 3), (5, 10)):
            keys, counts = o.result(mc, cm)
            assert _records(keys, counts, c["K"]) == _expected(c["reads"], c["K"], mc, cm)
            assert [tuple(k) for k in keys.tolist()] == sorted(tuple(k) for k in keys.tolist())
        o.close()
    # packed form with a fixed read length, K = 60, across several pushes
    reads = _mixed_reads(random.Random(3), 300, 60)
    reads150 = [("".join(random.Random(i).choice("ACGTN") for _ in range(150))) for i in range(200)]
    o = OracleReadKmers(60)
    o.push_reads(reads)
    b, m, _ = codec.pack_reads(reads150)
    o.push_packed(b, m, None, len(reads150), 150)
    assert _records(*o.result(1, 255), 60) == _expected(reads + reads150, 60, 1, 255)


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("tag,rfile,over", [("default", "reads.fq", {}), ("fasta_gz", "reads.fa.gz", {"cutoff": 0.0})])
def test_dropin_writes_the_reference_kmc_databases(tmp_path, tag, rfile, over):
    out = _run_dropin(tmp_path, rfile, **over)
    reads = _fixture_reads(rfile)
    hdr, recs = kmcdb.read(str(out / "reads_60mers"))
    assert hdr["k"] == 60 and hdr["min_count"] == 2 and hdr["max_count"] == 3 and hdr["canonical"] and hdr["version"] == 0
    assert dict(recs) == _expected(reads, 60, 2, 3)
    keys, info, counts = ingest.read_kmc_database(str(out / "reads_60mers"), with_counts=True)
    assert _records(keys, counts, 60) == dict(recs) and info["k"] == 60
    if tag == "default":
        exp = os.path.join(CASE, "expected_default")
        for ext in (".kmc_pre", ".kmc_suf"):
            assert filecmp.cmp(str(out / ("60mers_intersection" + ext)), os.path.join(exp, "60mers_intersection" + ext), shallow=False)
        _, golden = kmcdb.read(os.path.join(exp, "reads_60mers"))
        assert dict(recs) == dict(golden) and len(recs) == 13138 and max(c for _, c in recs) <= 3
        assert set(os.listdir(exp)) <= set(os.listdir(out))
    # consistency of the pair: intersection = reads (>= 2) & D, count = min(reads, sketch slots), = the dump's column
    _, dmult = kmcdb.read(os.path.join(DATA, "cmash_db_n1000_k60_dump"))
    dmult = dict(dmult)
    reads_db = dict(recs)
    want = {x: min(c, dmult[x]) for x, c in reads_db.items() if x in dmult}
    hdr_i, inter = kmcdb.read(str(out / "60mers_intersection"))
    assert dict(inter) == want and hdr_i["min_count"] == 1 and hdr_i["max_count"] == 3
    dump = [ln.split() for ln in open(out / "60mers_intersection_dump")]
    assert {a: int(b) for a, b in dump} == want


@pytest.mark.gpu
@pytest.mark.parametrize("K,ks", [(60, (30, 40, 50, 60)), (31, (21, 31))])
def test_read_kmers_match_the_oracle(ctx, K, ks):
    rng = random.Random(K)
    batches = [_mixed_reads(rng, 120, K) for _ in range(3)]
    allreads = [r for b in batches for r in b]
    db = _small_db(ctx, K, allreads, ks)
    cnt = oracle_py.count_read_kmers(allreads, K)
    for how in ("ascii", "packed", "nruns", "device"):
        keep = []
        q = db.query(read_kmers=True)
        for b in batches:                                            # three pushes: both staging sets
            _push(q, b, how, keep)
        q.sync()
        for mc, cm in ((1, 255), (2, 3), (5, 10)):
            keys, counts = q.read_kmers(mc, cm)
            assert _records(keys, counts, K) == _expected(allreads, K, mc, cm, cnt), (how, mc, cm)
            assert np.all(np.diff(keys[:, 0].astype(object) * (1 << 64) + keys[:, 1].astype(object)) > 0)
        keys, counts = q.read_kmers(1, 255)
        assert counts.max() == 255                                   # the repeated k-mers saturated instead of wrapping
        st = q.read_kmer_stats()
        assert st["distinct"] == len(keys) and st["overflowed"] == 0 and st["ms_count"] > 0
        if K == 31:
            assert q.stats()["layout"] == 0
        q.close()
    db.close()


@pytest.mark.gpu
def test_growth_and_budget(ctx, tmp_path):
    p = synth.params(G=40, n=100, seed=4, len_min=20000, len_max=60000, n_present=20)
    keys = synth.sketch_keys(p)
    db = Database.from_keys(ctx, keys, p.G, p.n, 60)
    sizes = [10, 2000, 20000, 60000]
    r0 = 0
    packed = []
    for n in sizes:
        b, m = synth.reads_packed(p, r0, n)
        packed.append((b, m, n))
        r0 += n
    grown = db.query(read_kmers=True)
    for b, m, n in packed:
        grown.push_packed(b, m, None, n, p.read_len)
    res_grown = grown.finish()
    st = grown.read_kmer_stats()
    assert st["grows"] >= 2, st
    allb, allm = synth.reads_packed(p, 0, r0)
    once = db.query(read_kmers=True)
    once.push_packed(allb, allm, None, r0, p.read_len)
    once.sync()
    assert once.read_kmer_stats()["grows"] == 0
    for a, b in zip(grown.read_kmers(1, 255), once.read_kmers(1, 255)):
        assert np.array_equal(a, b)
    o = OracleReadKmers(60)
    o.push_packed(allb, allm, None, r0, p.read_len)
    for a, b in zip(grown.read_kmers(2, 3), o.result(2, 3)):
        assert np.array_equal(a, b)
    # a budget far below what the reads need: the table stops, the query does not
    tight = db.query(read_kmers=True, read_kmer_budget=4096)
    plain = db.query()
    for b, m, n in packed:
        tight.push_packed(b, m, None, n, p.read_len)
        plain.push_packed(b, m, None, n, p.read_len)
    rt, rp = tight.finish(), plain.finish()
    for k in ("num", "den", "ci"):
        assert np.array_equal(rt[k], rp[k])
    assert np.array_equal(tight.intersection(), plain.intersection()) and np.array_equal(rt["num"], res_grown["num"])
    with pytest.raises(MlgError) as e:
        tight.read_kmers()
    assert e.value.code == ERR_NOMEM
    assert tight.read_kmer_stats()["overflowed"] == 1 and tight.read_kmer_stats()["bytes_needed"] > 4096
    for q in (grown, once, tight, plain):
        q.close()
    db.close()
    # the drop-in under that budget: every file but reads_60mers.kmc_*
    out = _run_dropin(tmp_path, "reads.fq", read_kmer_budget=4096)
    exp = os.path.join(CASE, "expected_default")
    for name in ("cmash_query_results.csv", "cmashed_db.fna", "subset_db_info.txt", "60mers_intersection_dump",
                 "60mers_intersection.kmc_pre", "60mers_intersection.kmc_suf"):
        assert filecmp.cmp(str(out / name), os.path.join(exp, name), shallow=False), name
    assert not os.path.exists(out / "reads_60mers.kmc_pre") and not os.path.exists(out / "reads_60mers.kmc_suf")


@pytest.mark.gpu
def test_off_is_off(ctx):
    rng = random.Random(5)
    batches = [_mixed_reads(rng, 80, 60) for _ in range(3)]
    db = _small_db(ctx, 60, [r for b in batches for r in b], (30, 40, 50, 60))
    off, on = db.query(), db.query(read_kmers=True)
    for q in (off, on):
        for b in batches:
            q.push_reads(b)
    for call in (lambda: off.read_kmers(), lambda: off.write_reads_kmc("/tmp/unused"), lambda: off.read_kmer_stats()):
        with pytest.raises(MlgError) as e:
            call()
        assert e.value.code == ERR_STATE
    r_off, r_on = off.finish(), on.finish()
    for k in ("num", "den", "ci", "n_intersect", "n_kmers"):
        assert np.array_equal(r_off[k], r_on[k]), k
    assert np.array_equal(off.intersection(), on.intersection())
    # three ASCII pushes (pack + probe each) and the finish stage (hit-record replay + expand + finalize): the count of the
    # library before the read k-mer table existed
    assert r_off["stats"]["gpu_launches"] == 9
    st = on.read_kmer_stats()
    assert r_on["stats"]["gpu_launches"] == 9 + r_on["stats"]["probe_launches"] + st["grows"]
    off.close(); on.close(); db.close()


@pytest.mark.gpu
def test_errors(ctx, tmp_path):
    reads = _mixed_reads(random.Random(9), 40, 61)
    db61 = _small_db(ctx, 61, reads, (41, 61))
    with pytest.raises(MlgError) as e:
        db61.query(read_kmers=True)
    assert e.value.code == ERR_ARG
    db61.close()
    reads = _mixed_reads(random.Random(9), 40, 60)
    db = _small_db(ctx, 60, reads, (30, 40, 50, 60))
    q = db.query()
    q.push_reads(reads)
    assert _lib.lib().mlg_query_enable_read_kmers(q._h, 0) == ERR_STATE                  # after the first push
    q.close()
    q = db.query(read_kmers=True)
    q.push_reads(reads)
    q.counts_export_sparse()
    for call in (lambda: q.read_kmers(), lambda: q.write_reads_kmc(str(tmp_path / "x"))):
        with pytest.raises(MlgError) as e:
            call()
        assert e.value.code == ERR_STATE
    q.close()
    q = db.query(read_kmers=True)
    q.push_reads(reads)
    q.finish()
    for call in (lambda: q.write_reads_kmc(str(tmp_path / "no" / "such" / "dir")),
                 lambda: q.write_intersection_kmc(str(tmp_path / "no" / "such" / "dir"))):
        with pytest.raises(MlgError) as e:
            call()
        assert e.value.code == ERR_IO
    n = C.c_uint64()
    assert _lib.lib().mlg_query_read_kmers(q._h, 0, 3, None, None, 0, C.byref(n)) == ERR_ARG
    q.close()
    db.close()


@pytest.mark.gpu
def test_scale_two_million_reads(ctx, tmp_path):
    """about 2 M reads of the bench's generator (150 bp), pushed in two batches: every record equals the C oracle's"""
    p = synth.params(G=2000, n=1000, seed=20200529, n_present=500, read_len=150)
    keys = synth.sketch_keys(p)
    db = Database.from_keys(ctx, keys, p.G, p.n, 60)
    q = db.query(read_kmers=True)
    o = OracleReadKmers(60)
    for r0, n in ((0, 1_000_000), (1_000_000, 1_000_000)):
        b, m = synth.reads_packed(p, r0, n)
        q.push_packed(b, m, None, n, p.read_len)
        o.push_packed(b, m, None, n, p.read_len)
        q.sync()
    got, want = q.read_kmers(1, 255), o.result(1, 255)
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
