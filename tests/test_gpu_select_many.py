"""select_many on the GPU: many samples through one context and one loaded database.

* Every sample directory of a batch is byte-identical to a single select_db run with the same flags, and for the
  reference reads (reads.fq, reads.fa.gz) to the reference's own files (expected_*), one batch per flag set, with
  --keep_temp_files, the read k-mer table and --read_kmer_passes.
* A missing reads file and a truncated gzip between good samples fail alone: no files of theirs are left, their neighbours'
  files are those of a batch without them, and the script exits non-zero.
* The library's live device bytes, open descriptors, threads and pooled reader buffers after 2, 11 and 20 samples of
  one session are equal.
* The same reads under two ids give identical files (the counter table handed from query to query is clean), and
  repeated queries on one database -- table, passes, none, one closed half-pushed, one over its read k-mer budget -- each
  give what a query on a fresh database gives.
* Under torchrun at 2 ranks and at every GPU up to 8 the files equal the one-GPU batch (skipped below two GPUs)."""
import argparse
import filecmp
import gzip
import os
import random
import subprocess
import sys
import threading

import numpy as np
import pytest

import kmcdb
from conftest import ROOT

pytestmark = pytest.mark.gpu
CASE = os.path.join(ROOT, "tests", "golden", "ref_e2e_case")
DATA = os.path.join(CASE, "data")
SYN = 4


def _genomes():
    d = os.path.join(DATA, "organism_files")
    out = []
    for name in sorted(os.listdir(d)):
        lines = gzip.open(os.path.join(d, name), "rt").read().splitlines()
        text = "".join(ln.strip() for ln in lines if not ln.startswith(">"))
        if len(text) > 400:
            out.append(text)
    return out


def _write_synthetic(path, seed, n_reads=1500):
    """reads of 100-150 bases from a seeded subset of the fixture's genomes, with substitutions and a few N"""
    rng = random.Random(seed)
    genomes = _genomes()
    pick = rng.sample(range(len(genomes)), rng.randint(2, 6))
    recs = []
    for i in range(n_reads):
        g = genomes[rng.choice(pick)]
        L = rng.randint(100, 150)
        a = rng.randrange(0, len(g) - L)
        s = list(g[a:a + L])
        for _ in range(rng.randint(0, 2)):
            s[rng.randrange(L)] = rng.choice("ACGTN")
        recs.append("".join(s))
    fasta = path.endswith((".fa", ".fa.gz"))
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "wt") as f:
        for i, r in enumerate(recs):
            f.write(">s%d\n%s\n" % (i, r) if fasta else "@s%d\n%s\n+\n%s\n" % (i, r, "F" * len(r)))


@pytest.fixture(scope="module")
def reads(tmp_path_factory):
    d = tmp_path_factory.mktemp("reads")
    out = {"ref_fq": os.path.join(CASE, "reads.fq"), "ref_fagz": os.path.join(CASE, "reads.fa.gz")}
    for i, ext in zip(range(SYN), ("fq", "fq.gz", "fa", "fa.gz")):
        p = str(d / ("syn%d.%s" % (i, ext)))
        _write_synthetic(p, 100 + i)
        out["syn%d" % i] = p
    return out


def _write_sheet(path, rows):
    with open(path, "w") as f:
        f.writelines("%s\t%s\n" % r for r in rows)
    return str(path)


def _flags(over):
    return sum((["--" + k] if v is True else ["--" + k, str(v)] for k, v in over.items()), [])


def _batch(sheet, out, over):
    from metalign_b200 import select_db
    args = select_db.select_many_parseargs([sheet, DATA, "--out_dir", str(out), "--threads", "4"] + _flags(over))
    return select_db.select_many(sheet, args)


def _single(reads_path, out, over):
    from metalign_b200 import select_db
    d = dict(reads=reads_path, data=DATA, cmash_results="NONE", cutoff=0.01, db="AUTO", db_dir="AUTO", dbinfo_in="AUTO",
             dbinfo_out="AUTO", input_type="AUTO", keep_temp_files=False, strain_level=False, temp_dir=str(out), threads=4,
             read_kmer_passes=False, read_kmer_budget=0)
    d.update(over)
    return select_db.select_main(argparse.Namespace(**d))


def _same_dir(a, b):
    assert sorted(os.listdir(a)) == sorted(os.listdir(b)), (a, b)
    for name in os.listdir(b):
        assert filecmp.cmp(os.path.join(a, name), os.path.join(b, name), shallow=False), (a, b, name)


def _summary(out):
    with open(os.path.join(str(out), "samples_summary.tsv")) as f:
        lines = f.read().splitlines()
    assert lines[0] == "sample_id\tstatus\tselected\tseconds\terror"
    return [ln.split("\t") for ln in lines[1:]]


BATCHES = [  # (flags, the reference reads of this flag set, its expected_* directory)
    ({"keep_temp_files": True}, "ref_fq", "expected_default"),
    ({"keep_temp_files": True, "read_kmer_passes": True}, "ref_fq", "expected_default"),
    ({"keep_temp_files": True, "strain_level": True}, "ref_fq", "expected_strain_level"),
    ({"keep_temp_files": True, "cutoff": 0.5}, "ref_fq", "expected_cutoff_0.5"),
    ({"keep_temp_files": True, "cutoff": 0.0}, "ref_fagz", "expected_fasta_gz"),
    ({}, "ref_fq", "expected_default"),
]


@pytest.mark.parametrize("over,ref,expected", BATCHES, ids=["keep", "passes", "strain", "cutoff05", "fagz", "plain"])
def test_batch_equals_single_runs_and_reference(tmp_path, reads, over, ref, expected):
    names = [ref] + ["syn%d" % i for i in range(SYN)]
    sheet = _write_sheet(tmp_path / "s.tsv", [(n, reads[n]) for n in names])
    results = _batch(sheet, tmp_path / "batch", over)
    assert [r.id for r in results] == names and all(r.status == "ok" for r in results), results
    assert [r.split("\t")[:2] for r in open(tmp_path / "batch" / "samples_summary.tsv").read().splitlines()[1:]] == \
        [[n, "ok"] for n in names]
    for r in results:
        chosen = _single(reads[r.id], tmp_path / "single" / r.id, over)
        assert r.organisms == chosen
        _same_dir(str(tmp_path / "batch" / r.id), str(tmp_path / "single" / r.id))
    exp = os.path.join(CASE, expected)
    got = str(tmp_path / "batch" / ref)
    want = sorted(os.listdir(exp)) if over.get("keep_temp_files") else ["cmash_query_results.csv", "cmashed_db.fna",
                                                                         "subset_db_info.txt"]
    for name in want:
        if name.startswith("reads_60mers."):
            continue
        assert filecmp.cmp(os.path.join(got, name), os.path.join(exp, name), shallow=False), (expected, name)
    if "reads_60mers.kmc_pre" in want:
        # the reference's kmc wrote this database in the 0x200 layout (its own record order), the library writes the
        # version-0 layout (INTEGRATION.md §A): the same k-mers and counts
        (h1, r1), (h2, r2) = kmcdb.read(os.path.join(got, "reads_60mers")), kmcdb.read(os.path.join(exp, "reads_60mers"))
        assert dict(r1) == dict(r2) and len(r1) == len(r2) > 0
        assert [h1[k] for k in ("k", "min_count", "max_count", "canonical")] == [h2[k] for k in ("k", "min_count", "max_count", "canonical")]


def test_failed_samples_fail_alone(tmp_path, reads):
    raw = open(reads["syn1"], "rb").read()
    trunc = tmp_path / "truncated.fq.gz"
    trunc.write_bytes(raw[:len(raw) * 2 // 3])
    rows = [("a", reads["syn0"]), ("missing", str(tmp_path / "no_such.fq")), ("b", reads["syn2"]), ("cut", str(trunc)),
            ("c", reads["syn3"])]
    sheet = _write_sheet(tmp_path / "s.tsv", rows)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "select_many.py"), sheet, DATA, "--out_dir", str(out),
                        "--keep_temp_files"], capture_output=True, text=True, timeout=900)
    assert r.returncode != 0, r.stderr[-3000:]
    summary = _summary(out)
    assert [(s[0], s[1]) for s in summary] == [("a", "ok"), ("missing", "failed"), ("b", "ok"), ("cut", "failed"), ("c", "ok")]
    assert "no_such.fq" in summary[1][4] and summary[3][4], summary
    assert not os.path.exists(out / "missing") and not os.path.exists(out / "cut")
    good = _write_sheet(tmp_path / "good.tsv", [x for x in rows if x[0] in ("a", "b", "c")])
    results = _batch(good, tmp_path / "good", {"keep_temp_files": True})
    assert all(x.status == "ok" for x in results)
    for sid in ("a", "b", "c"):
        _same_dir(str(out / sid), str(tmp_path / "good" / sid))


def _fds():
    return len(os.listdir("/proc/self/fd"))


def test_nothing_grows_with_the_number_of_samples(tmp_path, reads):
    """the library's live device bytes (its pool: database, the counter table handed from query to query), the open
    descriptors, the threads and the pooled reader buffers are the same after 2, 11 and 20 samples of one session"""
    from metalign_b200 import select_db
    from metalign_b200.api import device_memory
    args = select_db.select_many_parseargs(["unused", DATA, "--out_dir", str(tmp_path), "--keep_temp_files"])
    select_db.normalise_many(args)
    names = ["syn%d" % (i % SYN) for i in range(20)]
    samples = [select_db.Sample("s%02d" % i, reads[n], "fasta" if ".fa" in reads[n] else "fastq") for i, n in enumerate(names)]
    session = select_db.SelectSession(args)
    results, seen = [], []
    try:
        for a, b in ((0, 2), (2, 11), (11, 20)):
            results += session.run(samples[a:b], str(tmp_path))
            seen.append((device_memory(args.device)["live"], _fds(), threading.active_count(), len(session.pool._free)))
    finally:
        session.close()
    assert all(r.status == "ok" for r in results), [r.error for r in results if r.status != "ok"]
    assert seen[0] == seen[1] == seen[2], seen
    assert seen[0][0] > 0
    for i in range(SYN, 20):
        _same_dir(str(tmp_path / ("s%02d" % i)), str(tmp_path / ("s%02d" % (i % SYN))))


def test_same_reads_under_two_ids(tmp_path, reads):
    rows = [("x", reads["syn0"]), ("ref", reads["ref_fq"]), ("y", reads["syn1"]), ("x_again", reads["syn0"])]
    results = _batch(_write_sheet(tmp_path / "s.tsv", rows), tmp_path / "out", {"keep_temp_files": True})
    assert all(r.status == "ok" for r in results)
    _same_dir(str(tmp_path / "out" / "x"), str(tmp_path / "out" / "x_again"))


def _query_result(q):
    res = q.finish()
    return res["num"], res["den"], res["ci"], q.intersection()


def test_repeated_queries_on_one_database(ctx):
    """one loaded database, queries one after the other in every mode, each equal to a query on a fresh database"""
    from metalign_b200 import select_db
    from metalign_b200._lib import MLG_ERR_NOMEM, MlgError
    from metalign_b200.api import Database
    path = os.path.join(DATA, select_db.DB_BASENAME)
    with open(os.path.join(CASE, "reads.fq")) as f:
        lines = f.read().split("\n")
    ref_reads = [lines[i + 1] for i in range(0, len(lines) - 1, 4)]
    other = [r[::-1] for r in ref_reads[: len(ref_reads) // 2]] + ref_reads[:50]

    def fresh(rd, **kw):
        db = Database.load(ctx, path)
        try:
            q = db.query(**kw)
            q.push_reads(rd)
            out = _query_result(q)
            rk = q.read_kmers(2, 3) if kw.get("read_kmers") else None
            q.close()
            return out, rk
        finally:
            db.close()
    want = {id(rd): fresh(rd, read_kmers=True) for rd in (ref_reads, other)}
    db = Database.load(ctx, path)
    try:
        for rd, kw in [(ref_reads, dict(read_kmers=True, read_kmer_passes=True)), (other, {}),
                       (ref_reads, dict(read_kmers=True)), ("half", {}), (other, dict(read_kmers=True, read_kmer_passes=True)),
                       ("budget", dict(read_kmers=True, read_kmer_budget=1)), (ref_reads, {}), (other, dict(read_kmers=True))]:
            q = db.query(**kw)
            if rd == "half":                      # a query that fails after some pushes: closed without finish
                q.push_reads(ref_reads[:len(ref_reads) // 2])
                q.sync()
                q.close()
                continue
            if rd == "budget":                    # over its read k-mer budget: the counters are still right
                q.push_reads(other)
                assert all(np.array_equal(a, b) for a, b in zip(_query_result(q), want[id(other)][0]))
                with pytest.raises(MlgError) as e:
                    q.read_kmers(2, 3)
                assert e.value.code == MLG_ERR_NOMEM
                q.close()
                continue
            q.push_reads(rd)
            got = _query_result(q)
            assert all(np.array_equal(a, b) for a, b in zip(got, want[id(rd)][0])), kw
            if kw.get("read_kmers"):
                k, c = q.read_kmers(2, 3)
                assert np.array_equal(k, want[id(rd)][1][0]) and np.array_equal(c, want[id(rd)][1][1]), kw
            q.close()
    finally:
        db.close()


def _rank_worker(rank, world, port, sheet, out):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as tdist
    from metalign_b200 import select_db
    args = select_db.select_many_parseargs([sheet, DATA, "--out_dir", out, "--keep_temp_files", "--threads", "2"])
    results = select_db.select_many(sheet, args)
    with open(os.path.join(out, "rank%d.ids" % rank), "w") as f:
        f.write(" ".join("%s:%s" % (r.id, r.status) for r in results))
    tdist.destroy_process_group()


def test_ranks_spread_the_samples(tmp_path, reads):
    import torch
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    worlds = sorted({2, min(n, 8)}) if n >= 2 else []
    if not worlds:
        pytest.skip("needs two GPUs")
    names = ["ref_fq", "ref_fagz"] + ["syn%d" % i for i in range(SYN)] + ["syn0"]
    rows = [("%s_%d" % (nm, i), reads[nm]) for i, nm in enumerate(names)]
    sheet = _write_sheet(tmp_path / "s.tsv", rows)
    one = _batch(sheet, tmp_path / "one", {"keep_temp_files": True})
    assert all(r.status == "ok" for r in one)
    for world in worlds:
        out = str(tmp_path / ("w%d" % world))
        os.makedirs(out)
        mp.spawn(_rank_worker, args=(world, 29800 + os.getpid() % 50 + world, sheet, out), nprocs=world, join=True)
        assert open(tmp_path / "one" / "samples_summary.tsv").read().split("\n")[0] == \
            open(os.path.join(out, "samples_summary.tsv")).read().split("\n")[0]
        assert [s[:3] for s in _summary(out)] == [s[:3] for s in _summary(tmp_path / "one")]
        every = " ".join("%s:ok" % sid for sid, _ in rows)
        for r in range(world):
            assert open(os.path.join(out, "rank%d.ids" % r)).read() == every
        for sid, _ in rows:
            _same_dir(os.path.join(out, sid), str(tmp_path / "one" / sid))
