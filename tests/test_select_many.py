"""select_many without a GPU: the sample sheet (parsing, every refusal named by its line, the type from the extension),
the round-robin assignment of samples to ranks, the summary format, the refusal of a bad sheet before any GPU work, the
reader buffer pool that lets one sample's reader take over the previous one's buffers, a batch rank reading and querying
whole samples under torchrun, and run() returning when a sample's bookkeeping fails."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from metalign_b200 import ingest, select_db
from metalign_b200.select_db import SampleResult, SampleSheetError, format_summary, rank_samples, read_sample_sheet


def _sheet(tmp_path, text, name="samples.tsv"):
    p = tmp_path / name
    p.write_text(text)
    return str(p)


def test_sheet_parsing(tmp_path):
    path = _sheet(tmp_path, "# id\treads\n\nS1\treads/a.fq\nS_2.b-c\t/abs/b.fa.gz\tfasta\n"
                            "s3\tc.txt\tfastq\r\n   \nS4\td.FASTQ.gz\tfastq\n")
    got = read_sample_sheet(path)
    assert got == [select_db.Sample("S1", str(tmp_path / "reads" / "a.fq"), "fastq"),
                   select_db.Sample("S_2.b-c", "/abs/b.fa.gz", "fasta"),
                   select_db.Sample("s3", str(tmp_path / "c.txt"), "fastq"),
                   select_db.Sample("S4", str(tmp_path / "d.FASTQ.gz"), "fastq")]
    assert read_sample_sheet(_sheet(tmp_path, "# nothing\n\n", "empty.tsv")) == []


@pytest.mark.parametrize("ext,kind", [("fq", "fastq"), ("fastq", "fastq"), ("fq.gz", "fastq"), ("fastq.gz", "fastq"),
                                      ("fa", "fasta"), ("fna", "fasta"), ("fasta", "fasta"), ("fa.gz", "fasta"),
                                      ("fna.gz", "fasta"), ("fasta.gz", "fasta")])
def test_type_from_extension(tmp_path, ext, kind):
    assert read_sample_sheet(_sheet(tmp_path, "x\tr.%s\n" % ext))[0].input_type == kind
    assert ingest.input_type_of("dir.v2/r." + ext) == kind


@pytest.mark.parametrize("body,line,words", [
    ("a\tx.fq\nb\n", 2, "column"),
    ("a\tx.fq\tfastq\textra\n", 1, "column"),
    ("a\t\n", 1, "column"),
    ("a\tx.fq\nb\ty.fq\na\tz.fq\n", 3, "duplicate sample id 'a' (first on line 1)"),
    ("../up\tx.fq\n", 1, "safe directory name"),
    ("a/b\tx.fq\n", 1, "safe directory name"),
    (".hidden\tx.fq\n", 1, "safe directory name"),
    ("-opt\tx.fq\n", 1, "safe directory name"),
    ("a b\tx.fq\n", 1, "safe directory name"),
    ("\tx.fq\n", 1, "safe directory name"),
    ("samples_summary.tsv\tx.fq\n", 1, "safe directory name"),
    ("x" * 129 + "\tx.fq\n", 1, "safe directory name"),
    ("a\tx.fq\nb\ty.fq\tbam\n", 2, "unknown reads type 'bam'"),
    ("a\tx.fq\tFASTQ\n", 1, "unknown reads type"),
    ("a\tx.fq\n# c\nb\treads.bam\n", 3, "extension"),
])
def test_sheet_refusals_name_the_line(tmp_path, body, line, words):
    path = _sheet(tmp_path, body)
    with pytest.raises(SampleSheetError) as e:
        read_sample_sheet(path)
    assert ("line %d:" % line) in str(e.value) and words in str(e.value), str(e.value)


def test_missing_reads_file_is_not_a_sheet_error(tmp_path):
    assert read_sample_sheet(_sheet(tmp_path, "a\tno_such_file.fq\n"))[0].id == "a"


@pytest.mark.parametrize("n,world", [(0, 2), (1, 2), (7, 1), (7, 3), (8, 8), (20, 8), (3, 5)])
def test_round_robin_assignment(n, world):
    parts = [rank_samples(n, r, world) for r in range(world)]
    assert sorted(i for p in parts for i in p) == list(range(n))
    for r, p in enumerate(parts):
        assert p == [i for i in range(n) if i % world == r]


def test_summary_format():
    rows = [SampleResult("s1", "ok", ["taxid_1_genomic.fna.gz", "taxid_2_genomic.fna.gz"], 1.23456, "", "/o/s1/", {}),
            SampleResult("s2", "failed", None, 0.5, "IOError: bad\tgzip\nCRC", "/o/s2/", {}),
            SampleResult("s3", "ok", [], 0.0, "", "/o/s3/", {})]
    assert format_summary(rows) == ("sample_id\tstatus\tselected\tseconds\terror\n"
                                    "s1\tok\t2\t1.235\t\n"
                                    "s2\tfailed\t0\t0.500\tIOError: bad gzip CRC\n"
                                    "s3\tok\t0\t0.000\t\n")
    for ln in format_summary(rows).splitlines():
        assert len(ln.split("\t")) == 5


def test_bad_sheet_is_refused_before_any_gpu_work(tmp_path):
    """the script exits non-zero naming the line, with a data directory that does not exist and no device in use"""
    sheet = _sheet(tmp_path, "a\tx.fq\na\ty.fq\n")
    out = tmp_path / "out"
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "select_many.py"), sheet, str(tmp_path / "nodata"),
                        "--out_dir", str(out)], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode != 0 and "line 2" in r.stderr and "duplicate" in r.stderr, r.stderr[-2000:]
    assert not out.exists()
    args = select_db.select_many_parseargs([sheet, str(tmp_path / "nodata"), "--cutoff", "1.5"])
    with pytest.raises(ValueError):
        select_db.select_many(sheet, args)


def test_reader_buffer_pool_hands_buffers_on(tmp_path):
    """a closed reader's buffers go to the next reader of the same batch sizes, which reads its own file exactly as a
    reader with fresh buffers does (stale bytes of the previous file do not leak into the batches)"""
    rng = np.random.default_rng(4)
    paths = []
    for i, n in enumerate((3000, 50)):
        p = tmp_path / ("r%d.fq" % i)
        with open(p, "w") as f:
            for j in range(n):
                seq = "".join(rng.choice(list("ACGTN"), size=int(rng.integers(60, 160))))
                f.write("@r%d\n%s\n+\n%s\n" % (j, seq, "I" * len(seq)))
        paths.append(str(p))
    allocated = []

    def alloc(nbytes):
        a = np.full(nbytes, 0xA5, dtype=np.uint8)          # not zeroed: stale-looking bytes
        allocated.append(a)
        return a
    pool = ingest.BufferPool(alloc)

    def batches(path, alloc):
        r = ingest.PackedBatches(path, "fastq", reads_per_batch=700, threads=2, alloc=alloc)
        out = [(b[:(int(o[-1]) + 3) // 4].copy(), n.copy(), o.copy(), k) for b, n, o, k in r]
        r.close()
        return out
    first = batches(paths[0], pool)
    assert len(allocated) == 6
    second = batches(paths[1], pool)
    assert len(allocated) == 6                              # every buffer came from the pool
    for path, got in zip(paths, (first, second)):
        want = batches(path, None)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert all(np.array_equal(x, y) for x, y in zip(g[:3], w[:3])) and g[3] == w[3]
    pool.clear()


def _fastq(path, n, seed=5):
    rng = np.random.default_rng(seed)
    with open(path, "w") as f:
        for j in range(n):
            seq = "".join(rng.choice(list("ACGT"), size=int(rng.integers(80, 151))))
            f.write("@r%d\n%s\n+\n%s\n" % (j, seq, "I" * len(seq)))
    return str(path)


def test_batch_reader_reads_whole_files_and_a_rank_reads_its_share(tmp_path):
    """a rank of select_many runs whole samples: the batch's reader (world 1, in pooled buffers) yields every record of
    the file, while the one-file multi-rank mode of select_db (here rank 1 of 2) reads this rank's byte range only"""
    import argparse
    path = _fastq(tmp_path / "r.fq", 4000)
    args = argparse.Namespace(reads=path, input_type="fastq", threads=2)
    numpy_alloc = lambda nbytes: np.zeros(nbytes, dtype=np.uint8)      # noqa: E731

    def count(reader):
        n = sum(int(b[3]) for b in reader)
        reader.close()
        return n
    assert count(select_db.open_reader(args, alloc=ingest.BufferPool(numpy_alloc))) == 4000
    assert 0 < count(select_db.open_reader(args, 1, 2, alloc=numpy_alloc)) < 4000


def test_query_takes_read_kmer_passes_when_asked_or_split_over_ranks():
    """under torchrun the one-file mode counts read k-mers in passes (its ranks hand the reads around); a batch sample has
    no exchange, so its query is opened as a single run's is"""
    import argparse
    opened = []

    class FakeQuery:
        def sync(self):
            pass

    class FakeDb:
        def query(self, **kw):
            opened.append(kw)
            return FakeQuery()
    for passes in (False, True):
        args = argparse.Namespace(gate="exact", keep_temp_files=True, read_kmer_budget=123, read_kmer_passes=passes)
        select_db.push_sample(args, FakeDb(), [])                 # a batch sample
        select_db.push_sample(args, FakeDb(), [], world=2)        # a rank of the one-file mode
    assert [(q["read_kmer_passes"], q["read_kmer_budget"], q["read_kmers"]) for q in opened] == \
        [(False, 123, True), (True, 123, True), (True, 123, True), (True, 123, True)]


def test_batch_hands_every_sample_over_when_its_bookkeeping_fails(tmp_path, monkeypatch):
    """an error outside a sample's GPU part (here: the helper that opens the next reader cannot start) fails the samples
    it touches, and run() returns instead of waiting for ever"""
    import argparse
    import threading

    def broken(fn):
        raise RuntimeError("cannot start a thread")
    monkeypatch.setattr(select_db, "_on_helper", broken)
    session = object.__new__(select_db.SelectSession)
    session.args = argparse.Namespace(gate="exact", keep_temp_files=False, read_kmer_budget=0, read_kmer_passes=False,
                                      threads=1)
    session.stopped, session.db, session.taxid2info = None, None, {}
    session.pool = ingest.BufferPool(lambda nbytes: np.zeros(nbytes, dtype=np.uint8))
    samples = [select_db.Sample("s%d" % i, str(tmp_path / "r.fq"), "fastq") for i in range(3)]
    box = {}
    th = threading.Thread(target=lambda: box.setdefault("res", session.run(samples, str(tmp_path / "out"))), daemon=True)
    th.start()
    th.join(120)
    assert "res" in box, "run() did not return"
    assert [(r.id, r.status) for r in box["res"]] == [("s0", "failed"), ("s1", "failed"), ("s2", "failed")]
    assert all("cannot start a thread" in r.error for r in box["res"])
