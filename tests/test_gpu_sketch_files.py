"""Genome files straight into a built database (make_sketch_db.py --built: sketch.build_database_from_files ->
mlgi_files_* -> mlg_db_builder_add_fasta) against the two-step path it replaces (build_database -> Database.load -> save):
the built files must be byte-identical, for FASTA shapes at every edge of read_fasta's rules, for reader batches and sketch
passes split at every file, K = 21, 31 and 60, n above and below the distinct count.  Refusals leave no file."""
import gzip
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_ingest import _write_bgzf

pytestmark = pytest.mark.gpu


def _seq(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(alphabet) for _ in range(n))


def _wrap(rng, s, eol="\n"):
    """s in lines of 1 to 200 bytes"""
    out, i = [], 0
    while i < len(s):
        w = rng.randint(1, 200)
        out.append(s[i:i + w] + eol)
        i += w
    return "".join(out)


def _shapes(rng):
    """(name, text) of FASTA files at the edges of read_fasta's rules"""
    g = lambda n: _seq(rng, n)  # noqa: E731
    return [
        ("crlf", ">a desc\r\n" + _wrap(rng, g(3000), "\r\n") + ">b\r\n" + _wrap(rng, g(900), "\r\n")),
        ("blank", ">a\n\n" + g(80) + "\n   \n\t\n" + g(500) + "\n\n>b\n\n\n>c\n" + g(300) + "\n"),
        ("spaces", ">a\n  " + g(70) + "\t \n\t" + g(333) + "  \n \x0b" + g(91) + "\x0c\r\n" + "  >not a header " + g(40) + "\n"),
        ("gt_inside", ">a\n" + g(100) + ">" + g(100) + "\n" + g(50) + "\n"),
        ("no_final_newline", ">a\n" + _wrap(rng, g(1200)) + ">b\n" + g(333)),
        ("header_only", ">a\n>b\n>c\n" + g(400) + "\n>d\n>e"),
        ("many_records", "".join(">r%d\n%s" % (i, _wrap(rng, g(rng.randint(0, 300)))) for i in range(40))),
        ("no_header", _wrap(rng, g(2500))),
        ("iupac_lower", ">a\n" + _wrap(rng, _seq(rng, 4000, "ACGTacgtNRYKMSWnrykm")) + ">b\n" + _wrap(rng, g(2000).lower())),
        ("one_per_line", ">a\n" + "\n".join(g(2000)) + "\n"),
        ("repeats", ">a\n" + _wrap(rng, "ACGTTGCA" * 700) + ">b\n" + _wrap(rng, "A" * 3000)),
        ("empty", ""),
        ("blank_only", "\n\n  \n"),
        ("large", ">a\n" + _wrap(rng, g(40000)) + ">b\n" + _wrap(rng, g(9000))),
    ]


def _write_files(d, rng, shapes):
    """plain, gzip and BGZF files in turn, listed out of basename order"""
    paths = []
    for i, (name, text) in enumerate(shapes):
        data = text.encode()
        p = os.path.join(d, "%s_%02d.fa" % (name, i) + ("" if i % 3 == 0 else ".gz"))
        if i % 3 == 0:
            with open(p, "wb") as f:
                f.write(data)
        elif i % 3 == 1:
            with gzip.open(p, "wb", compresslevel=6) as f:
                f.write(data)
        else:
            _write_bgzf(p, data, rng, max_block=3000)
        paths.append(p)
    rng.shuffle(paths)
    return paths


def _ks(K):
    return [k for k in (30, 40, 50, 60) if k <= K] if K == 60 else [K - 10, K]


def _old(ctx, paths, out, n, K, tmp):
    from metalign_b200.api import Database
    from metalign_b200.sketch import build_database
    src = os.path.join(tmp, "src_%d_%d.mlgdb" % (n, K))
    build_database(ctx, paths, src, n, K, _ks(K))
    db = Database.load(ctx, src)
    try:
        db.save(out)
    finally:
        db.close()


def _new(ctx, paths, out, n, K, **kw):
    from metalign_b200.sketch import build_database_from_files
    return build_database_from_files(ctx, paths, out, n, K, _ks(K), **kw)


def _bytes(p):
    with open(p, "rb") as f:
        return f.read()


@pytest.fixture
def files(tmp_path):
    rng = random.Random(2026)
    d = tmp_path / "genomes"
    d.mkdir()
    return _write_files(str(d), rng, _shapes(rng))


def test_two_builds_of_one_source_save_the_same_bytes(ctx, files, tmp_path):
    """the comparison below rests on this: the build and save are deterministic"""
    from metalign_b200.api import Database
    from metalign_b200.sketch import build_database
    src = str(tmp_path / "src.mlgdb")
    build_database(ctx, files, src, 200, 60)
    outs = []
    for i in range(2):
        db = Database.load(ctx, src)
        outs.append(str(tmp_path / ("b%d.mlgdb" % i)))
        db.save(outs[-1])
        db.close()
    assert _bytes(outs[0]) == _bytes(outs[1])


@pytest.mark.parametrize("K", [21, 31, 60])
def test_built_file_matches_the_two_step_path(ctx, files, tmp_path, monkeypatch, K):
    # K != 60 databases carry an L2 prefilter, which the built form cannot hold: build them without one
    if K != 60:
        monkeypatch.setenv("MLG_FILTER_MB", "0")
    for n in (7, 5000):               # below and above every genome's distinct count
        a, b = str(tmp_path / ("old%d.mlgdb" % n)), str(tmp_path / ("new%d.mlgdb" % n))
        _old(ctx, files, a, n, K, str(tmp_path))
        st = _new(ctx, files, b, n, K, threads=3)
        assert st["files"] == len(files) and st["passes"] >= 1
        assert _bytes(a) == _bytes(b), (K, n)


def test_batches_and_passes_split_at_every_file(ctx, files, tmp_path, monkeypatch):
    from metalign_b200.sketch import read_fasta
    K, n = 31, 40
    monkeypatch.setenv("MLG_FILTER_MB", "0")
    ref = str(tmp_path / "old.mlgdb")
    _old(ctx, files, ref, n, K, str(tmp_path))
    want = _bytes(ref)
    order = sorted(files, key=os.path.basename)
    raw = [len(gzip.open(p).read()) if p.endswith(".gz") else os.path.getsize(p) for p in order]
    text = [len(read_fasta(p)) for p in order]
    for i in range(1, len(order)):
        out = str(tmp_path / ("b%d.mlgdb" % i))
        _new(ctx, files, out, n, K, threads=1 + i % 4, batch_bytes=max(1, sum(raw[:i])))
        assert _bytes(out) == want, ("batch", i)
    for i in range(1, len(order)):
        monkeypatch.setenv("MLG_SKETCH_PASS_BYTES", str(max(1, sum(t + 1 for t in text[:i]) - 1)))
        out = str(tmp_path / ("p%d.mlgdb" % i))
        _new(ctx, files, out, n, K, threads=2, batch_bytes=1 << 16)
        assert _bytes(out) == want, ("pass", i)
    monkeypatch.setenv("MLG_SKETCH_PASS_BYTES", "1000")     # the large genome alone, and larger than a pass
    out = str(tmp_path / "small_pass.mlgdb")
    st = _new(ctx, files, out, n, K, threads=4, batch_bytes=20000)
    passes, i = 0, 0                                         # the batching rule, restated (batches and redo rounds add more)
    while i < len(text):
        j, pb = i, 0
        while j < len(text) and (j == i or pb + text[j] <= 1000):
            pb += text[j] + 1
            j += 1
        passes, i = passes + 1, j
    assert max(text) > 1000 and _bytes(out) == want and st["passes"] >= passes


def test_kmers_across_line_breaks_count_and_across_records_do_not(ctx, tmp_path, monkeypatch):
    from metalign_b200.sketch import read_fasta, sketch_genomes
    rng = random.Random(5)
    K = 21
    a, b, c = _seq(rng, 10), _seq(rng, 11), _seq(rng, 11)
    p = str(tmp_path / "span.fa")
    with open(p, "w") as f:
        f.write(">r1\n" + a + "\n" + b + "\n>r2\n" + c + "\n")
    text = read_fasta(p)
    assert text == (a + b + "N" + c).encode()
    _, _, kmers, _ = sketch_genomes(ctx, [text], n=100, K=K)
    got = {bytes(k).decode() for k in kmers[0] if k[0]}
    assert (a + b) in got and len(got) == 1          # the k-mer across the line break, nothing across the records
    monkeypatch.setenv("MLG_FILTER_MB", "0")
    old, new = str(tmp_path / "o.mlgdb"), str(tmp_path / "n.mlgdb")
    _old(ctx, [p], old, 100, K, str(tmp_path))
    _new(ctx, [p], new, 100, K)
    assert _bytes(old) == _bytes(new)


def test_queries_agree(ctx, files, tmp_path):
    from metalign_b200.api import Database
    from metalign_b200.sketch import read_fasta
    n, K = 300, 60
    a, b = str(tmp_path / "old.mlgdb"), str(tmp_path / "new.mlgdb")
    _old(ctx, files, a, n, K, str(tmp_path))
    _new(ctx, files, b, n, K)
    rng = random.Random(8)
    texts = [read_fasta(p) for p in files]
    reads = []
    for _ in range(3000):
        t = rng.choice([t for t in texts if len(t) > 150])
        s = rng.randrange(len(t) - 150)
        reads.append(t[s:s + 150].decode())
    res = []
    for path in (a, b):
        db = Database.load(ctx, path)
        q = db.query()
        q.push_reads(reads)
        res.append(q.finish())
        q.close()
        db.close()
    assert res[0]["n_intersect"] > 0
    for key in ("num", "den", "ci"):
        assert np.array_equal(res[0][key], res[1][key]), key


def test_refusals_leave_no_file_and_free_the_builder(ctx, files, tmp_path, monkeypatch):
    import ctypes as C
    import torch
    from metalign_b200 import _lib
    from metalign_b200.api import Context, MlgError
    out = str(tmp_path / "out.mlgdb")
    missing = str(tmp_path / "genomes" / "zz_missing.fa")
    corrupt = str(tmp_path / "genomes" / "zz_corrupt.fa.gz")
    gz = bytearray(gzip.compress(b">a\n" + b"ACGT" * 5000 + b"\n"))
    gz[len(gz) // 2] ^= 0x5A
    with open(corrupt, "wb") as f:
        f.write(bytes(gz))
    torch.cuda.init()
    free0 = torch.cuda.mem_get_info()[0]
    with Context(0) as c2:
        for bad in (missing, corrupt):
            with pytest.raises(IOError, match=os.path.basename(bad)):
                _new(c2, files + [bad], out, 100000, 60, threads=2)
            assert not os.path.exists(out)
        # a database whose hit records do not fit has no built form: mlg_db_save's refusal, and no file
        monkeypatch.setenv("MLG_HIT_CAP_WORDS", "16")
        with pytest.raises(MlgError, match="precomputed hit records"):
            _new(c2, files, out, 2000, 60)
        assert not os.path.exists(out)
        monkeypatch.delenv("MLG_HIT_CAP_WORDS")
        # argument refusals of the ABI change nothing: the builder takes the right batch afterwards
        L = _lib.lib()
        ks = np.asarray([30, 40, 50, 60], dtype=np.uint32)
        bld = C.c_void_p()
        _lib.check(L.mlg_db_builder_create(c2._h, 2, 50, 60, ks.ctypes.data, 4, C.byref(bld)))
        try:
            data = np.frombuffer(b">a\n" + b"ACGTTGCAAC" * 40 + b"\n>b\nGGGCCCATAT" * 30, dtype=np.uint8).copy()
            off = np.array([0, 200, data.size], dtype=np.uint64)
            for args, msg in (((off[::-1].copy(), 2, 0), "decreases"), ((np.array([0, 1, 2, data.size], np.uint64), 3, 0), "builder holds"),
                              ((off, 2, 1 << 44), "prime")):
                rc = L.mlg_db_builder_add_fasta(bld, data.ctypes.data, args[0].ctypes.data, args[1], args[2], None)
                assert rc == -2 and msg in L.mlg_last_error().decode()
            _lib.check(L.mlg_db_builder_add_fasta(bld, data.ctypes.data, off.ctypes.data, 2, 0, None))
            h = C.c_void_p()
            _lib.check(L.mlg_db_builder_finish(bld, C.byref(h)))
            bld = None
            L.mlg_db_free(h)
        finally:
            if bld is not None:
                L.mlg_db_builder_destroy(bld)
    torch.cuda.synchronize()
    # the refused builds' builders (30 MB for the unreadable files) were freed with the context's pool
    assert torch.cuda.mem_get_info()[0] >= free0 - (8 << 20)


def test_make_sketch_db_cli_built(files, tmp_path):
    lst = tmp_path / "genomes.txt"
    lst.write_text("\n".join(files) + "\n")
    src, built, cli = str(tmp_path / "src.mlgdb"), str(tmp_path / "built.mlgdb"), str(tmp_path / "cli.mlgdb")
    script = os.path.join(ROOT, "scripts", "make_sketch_db.py")
    subprocess.check_call([sys.executable, script, str(lst), src, "-n", "100"])
    subprocess.check_call([sys.executable, os.path.join(ROOT, "scripts", "build_db.py"), src, built])
    subprocess.check_call([sys.executable, script, str(lst), cli, "-n", "100", "--built", "--threads", "3"])
    assert _bytes(built) == _bytes(cli)
