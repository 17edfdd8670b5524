"""Shares of a reads file (mlgi_open_share): the reads of consecutive byte ranges, joined in order, must be the reads of
mlgi_open over the whole file -- plain and BGZF, FASTQ and FASTA, LF and CRLF, with and without a final newline, every
two-way split of a small file, random cuts into 3 to 9 shares, more shares than records, quality lines that start with
'@' or '+', and sequence lines that cross a BGZF member and a share boundary.  A plain gzip stream goes whole to the share
at byte 0.  The phase check (ingest.check_share_phases) refuses 3- and 5-line "FASTQ" cut where the phase is wrong, and
accepts every cut of well-formed FASTQ.  No GPU."""
import gzip
import random
import zlib

import pytest

from metalign_b200 import codec, ingest
from test_ingest import _norm, _random_reads, _write_bgzf


def _reads(path, kind, share=None, threads=3):
    """(reads, share_info) of the whole file or of one share"""
    rd = ingest.PackedBatches(str(path), kind, reads_per_batch=500, bases_per_batch=100000, threads=threads, share=share)
    out = []
    try:
        for bases, runs, off, n in rd:
            mask = codec.runs_to_nmask(runs, int(off[-1])) if len(runs) else None
            out += codec.unpack_reads(bases, mask, off)
        info = rd.share_info() if share is not None else None
    finally:
        rd.close()
    return out, info


def _cuts_reads(path, kind, cuts, threads=3):
    """the shares [cuts[i], cuts[i + 1]): their reads joined, their infos"""
    reads, infos = [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        r, info = _reads(path, kind, (a, b), threads)
        reads += r
        infos.append(info)
    return reads, infos


def _fastq(rng, n, eol="\n", trailing=True, qual=None):
    reads = _random_reads(rng, n)
    recs = []
    for i, r in enumerate(reads):
        q = qual(i, r) if qual else "I" * len(r)
        recs.append("@r%d x%s%s%s+%s%s" % (i, eol, r, eol, eol, q))
    text = eol.join(recs) + (eol if trailing else "")
    return text, reads


def _fasta(rng, n, eol="\n", trailing=True):
    reads = [r for r in _random_reads(rng, n) if r]
    text = eol.join(">s%d%s%s" % (i, eol, r) for i, r in enumerate(reads)) + (eol if trailing else "")
    return text, reads


def _write_file(tmp_path, name, text, bgzf, rng, max_block=300):
    p = tmp_path / name
    if bgzf:
        _write_bgzf(p, text.encode(), rng, max_block=max_block)
    else:
        p.write_bytes(text.encode())
    return p


FORMATS = [(kind, eol, trailing, bgzf) for kind in ("fastq", "fasta") for eol in ("\n", "\r\n") for trailing in (True, False)
           for bgzf in (False, True)]


@pytest.mark.parametrize("kind,eol,trailing,bgzf", FORMATS)
def test_random_cuts_join_to_the_whole_file(tmp_path, kind, eol, trailing, bgzf):
    rng = random.Random(zlib.crc32(repr((kind, eol, trailing, bgzf)).encode()))
    text, reads = (_fastq if kind == "fastq" else _fasta)(rng, 300, eol, trailing)
    p = _write_file(tmp_path, "r." + kind + (".gz" if bgzf else ""), text, bgzf, rng, max_block=700)
    whole, _ = _reads(p, kind)
    assert whole == [_norm(r) for r in reads]
    size = p.stat().st_size
    for trial in range(12):
        k = rng.randint(3, 9)
        cuts = [0] + sorted(rng.randint(0, size) for _ in range(k - 1)) + [size]
        got, infos = _cuts_reads(p, kind, cuts, threads=rng.choice([1, 2, 5]))
        assert got == whole, (trial, cuts)
        ingest.check_share_phases(infos, kind)
    # ranges of share_ranges, and a range past the end of the file
    got, infos = _cuts_reads(p, kind, [a for a, _ in ingest.share_ranges(str(p), 4)] + [size + 100])
    assert got == whole
    ingest.check_share_phases(infos, kind)


@pytest.mark.parametrize("kind,bgzf", [("fastq", False), ("fastq", True), ("fasta", False), ("fasta", True)])
def test_every_two_way_split(tmp_path, kind, bgzf):
    """quality lines that start with '@' and '+', CRLF, an empty read, no final newline; every cut point of the file"""
    rng = random.Random(5 + bgzf)
    if kind == "fastq":
        text, reads = _fastq(rng, 9, "\r\n", False, qual=lambda i, r: ("@+"[i % 2] + "I" * len(r))[:len(r)])
    else:
        text, reads = _fasta(rng, 9, "\r\n", False)
    p = _write_file(tmp_path, "s." + kind + (".gz" if bgzf else ""), text, bgzf, rng, max_block=40)
    whole, _ = _reads(p, kind)
    assert whole == [_norm(r) for r in reads]
    size = p.stat().st_size
    for c in range(size + 1):
        got, infos = _cuts_reads(p, kind, [0, c, size], threads=2)
        assert got == whole, c
        ingest.check_share_phases(infos, kind)


@pytest.mark.parametrize("bgzf", [False, True])
def test_more_shares_than_records(tmp_path, bgzf):
    rng = random.Random(11)
    text, reads = _fastq(rng, 3)
    p = _write_file(tmp_path, "few.fq" + (".gz" if bgzf else ""), text, bgzf, rng, max_block=50)
    size = p.stat().st_size
    world = size // 3 + 5
    ranges = [(size * r // world, size * (r + 1) // world) for r in range(world)]
    got, infos = _cuts_reads(p, "fastq", [a for a, _ in ranges] + [size], threads=1)
    assert got == [_norm(r) for r in reads]
    assert sum(i["phase"] == -1 for i in infos) >= world - 12         # most shares hold no line start
    ingest.check_share_phases(infos, "fastq")


def test_long_lines_cross_members_and_shares(tmp_path):
    """reads of 2-20 kb in BGZF members of at most 1000 bytes: every sequence line spans members, and cuts inside a line
    hand it to the share that holds its first byte"""
    rng = random.Random(17)
    reads = ["".join(rng.choice("ACGT") for _ in range(rng.randint(2000, 20000))) for _ in range(20)]
    text = "".join("@r%d\n%s\n+\n%s\n" % (i, r, "@" * len(r)) for i, r in enumerate(reads))
    p = _write_file(tmp_path, "long.fq.gz", text, True, rng, max_block=1000)
    size = p.stat().st_size
    for trial in range(10):
        cuts = [0] + sorted(rng.randint(0, size) for _ in range(rng.randint(2, 8))) + [size]
        got, infos = _cuts_reads(p, "fastq", cuts)
        assert got == reads, cuts
        ingest.check_share_phases(infos, "fastq")


def test_plain_gzip_goes_whole_to_the_first_share(tmp_path, capfd):
    rng = random.Random(3)
    text, reads = _fastq(rng, 200)
    p = tmp_path / "one.fq.gz"
    with gzip.open(p, "wb") as f:
        f.write(text.encode())
    size = p.stat().st_size
    cuts = [a for a, _ in ingest.share_ranges(str(p), 4)] + [size]
    got = []
    for i, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        r, info = _reads(p, "fastq", (a, b))
        assert (len(r) == len(reads)) if i == 0 else (r == [] and info["phase"] == -1), i
        got += r
    assert got == [_norm(r) for r in reads]
    assert "bgzip" in capfd.readouterr().err


def _refused_or_equal(p, whole, cuts):
    got, infos = _cuts_reads(p, "fastq", cuts, threads=1)
    try:
        ingest.check_share_phases(infos, "fastq")
    except ValueError:
        return True
    assert got == whole, cuts
    return False


@pytest.mark.parametrize("lines", [3, 5])
def test_phase_check_refuses_records_of_other_lengths(tmp_path, lines):
    """records of 3 or 5 lines: a cut at a record start whose line number is not a multiple of 4 is refused, and no cut
    at all gives reads that differ from the whole-file parse without a refusal"""
    rng = random.Random(lines)
    recs = []
    for i in range(12):
        r = "".join(rng.choice("ACGT") for _ in range(30))
        recs.append(["@r%d" % i, r, "+", "I" * 30, "I" * 30][:lines])
    text = "".join(l + "\n" for rec in recs for l in rec)
    p = tmp_path / ("l%d.fq" % lines)
    p.write_bytes(text.encode())
    whole, _ = _reads(p, "fastq")
    second = len("".join(l + "\n" for l in recs[0]))            # the second record: line number `lines`, not 0 mod 4
    assert _refused_or_equal(p, whole, [0, second, len(text)])
    with pytest.raises(ValueError, match="not 4-line FASTQ"):
        ingest.check_share_phases(_cuts_reads(p, "fastq", [0, second, len(text)])[1], "fastq")
    refused = sum(_refused_or_equal(p, whole, [0, c, len(text)]) for c in range(len(text) + 1))
    assert refused > 0


def test_phase_check_is_a_prefix_sum():
    ok = [dict(first=0, newlines=6, phase=0), dict(first=9, newlines=0, phase=-1), dict(first=9, newlines=5, phase=2),
          dict(first=30, newlines=3, phase=3)]
    ingest.check_share_phases(ok, "fastq")
    with pytest.raises(ValueError, match="text byte 30"):
        ingest.check_share_phases(ok[:3] + [dict(first=30, newlines=3, phase=1)], "fastq")
    with pytest.raises(ValueError):
        ingest.check_share_phases([dict(first=0, newlines=4, phase=0), dict(first=7, newlines=1, phase=-2)], "fastq")
    ingest.check_share_phases([dict(first=0, newlines=3, phase=0), dict(first=7, newlines=1, phase=2)], "fasta")
