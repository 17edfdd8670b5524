"""The whole-file reader of the sketch builder (mlgi_files_*, csrc/ingest.cpp; metalign_b200.ingest.FileBatches) against
Python's gzip module: every file comes back exactly as gzip.open(p).read() (or its plain bytes), in the order given, for
any number of workers and any batch size, including files larger than the batch and empty files; unreadable files are
refused by name.  No GPU."""
import gzip
import os
import random

import pytest

from metalign_b200 import ingest
from test_ingest import _write_bgzf


def _fasta(rng, nbytes):
    out, n = [], 0
    while n < nbytes:
        line = ">g%d desc\n" % rng.randrange(10 ** 6) if rng.random() < 0.02 else \
            "".join(rng.choice("ACGTacgtNRY \t") for _ in range(rng.randint(0, 120))) + rng.choice(["\n", "\r\n"])
        out.append(line)
        n += len(line)
    return "".join(out).encode()


def _files(tmp_path, seed=3, nfiles=23):
    """a mix of plain, gzip (one and several members, levels 1 and 9) and BGZF files, with empty ones among them"""
    rng = random.Random(seed)
    paths, want = [], []
    for i in range(nfiles):
        data = b"" if i in (4, 11) else _fasta(rng, rng.choice([1, 100, 5000, 70000, 300000]))
        kind = i % 4
        p = str(tmp_path / ("f%02d.fa" % i + ("" if kind == 0 else ".gz")))
        if kind == 0:
            with open(p, "wb") as f:
                f.write(data)
        elif kind == 1:
            with gzip.open(p, "wb", compresslevel=rng.choice([1, 9])) as f:
                f.write(data)
        elif kind == 2:
            cut = len(data) // 3
            with open(p, "wb") as f:               # two gzip members back to back, as `cat a.gz b.gz` makes
                f.write(gzip.compress(data[:cut], 6) + gzip.compress(data[cut:], 6))
        else:
            _write_bgzf(p, data, rng, max_block=20000)
        paths.append(p)
        want.append(data)
    return paths, want


def _read_all(paths, batch_bytes, threads, max_files=1 << 16):
    r = ingest.FileBatches(paths, batch_bytes=batch_bytes, threads=threads, max_files=max_files)
    got, sizes = [], []
    try:
        for buf, off in r:
            assert off[0] == 0 and len(off) >= 2
            sizes.append(int(off[-1]))
            for i in range(len(off) - 1):
                got.append(bytes(buf[int(off[i]):int(off[i + 1])]))
    finally:
        r.close()
    return got, sizes


def test_reference_bytes_for_every_thread_count(tmp_path):
    paths, want = _files(tmp_path)
    for p, w in zip(paths, want):                   # the expectation itself: what gzip.open / open read
        with (gzip.open if p.endswith(".gz") else open)(p, "rb") as f:
            assert f.read() == w
    for threads in (1, 2, 7, 16):
        got, _ = _read_all(paths, 1 << 22, threads)
        assert got == want, threads


def test_batch_boundary_at_every_file(tmp_path):
    """batch sizes equal to every prefix sum of the file sizes, and max_files from 1 up: a split after every file"""
    paths, want = _files(tmp_path, seed=5, nfiles=9)
    sizes = [len(w) for w in want]
    pre = [sum(sizes[:i + 1]) for i in range(len(sizes))]
    for cap in sorted(set(max(1, c) for c in pre)):
        got, batches = _read_all(paths, cap, threads=3)
        assert got == want, cap
        assert all(b <= cap or b == max(sizes) or b in sizes for b in batches)
    for mf in (1, 2, 3):
        got, batches = _read_all(paths, 1 << 24, threads=2, max_files=mf)
        assert got == want and len(batches) >= (len(paths) + mf - 1) // mf


def test_file_larger_than_the_batch_comes_alone(tmp_path):
    rng = random.Random(9)
    small, big = _fasta(rng, 3000), _fasta(rng, 200000)
    paths = []
    for i, d in enumerate([small, big, small, b"", big]):
        p = str(tmp_path / ("x%d.fa.gz" % i))
        with gzip.open(p, "wb") as f:
            f.write(d)
        paths.append(p)
    r = ingest.FileBatches(paths, batch_bytes=10000, threads=4)
    batches = [(bytes(b[:int(o[-1])]), o.tolist()) for b, o in r]
    r.close()
    assert [o for _, o in batches] == [[0, len(small)], [0, len(big)], [0, len(small), len(small)], [0, len(big)]]
    assert b"".join(t for t, _ in batches) == small + big + small + big


def test_empty_list_and_empty_files(tmp_path):
    assert _read_all([], 1 << 10, 2) == ([], [])
    p = str(tmp_path / "e.fa")
    open(p, "wb").close()
    q = str(tmp_path / "e.fa.gz")
    with gzip.open(q, "wb"):
        pass
    got, sizes = _read_all([p, q, p], 1 << 10, 2)
    assert got == [b"", b"", b""] and sizes == [0]


def _refused(paths, bad, threads=2):
    with pytest.raises(IOError) as ei:
        _read_all(paths, 1 << 20, threads)
    assert bad in str(ei.value)
    return str(ei.value)


def test_unreadable_files_are_refused_by_name(tmp_path):
    paths, want = _files(tmp_path, seed=11, nfiles=6)
    data = _fasta(random.Random(1), 50000)
    gz = gzip.compress(data, 6)
    trunc = str(tmp_path / "trunc.fa.gz")
    with open(trunc, "wb") as f:
        f.write(gz[:len(gz) // 2])
    corrupt = str(tmp_path / "corrupt.fa.gz")
    bad = bytearray(gz)
    bad[len(bad) // 2] ^= 0x55
    with open(corrupt, "wb") as f:
        f.write(bytes(bad))
    crc = str(tmp_path / "crc.fa.gz")
    bad = bytearray(gz)
    bad[-8] ^= 1                                    # the trailer's CRC-32
    with open(crc, "wb") as f:
        f.write(bytes(bad))
    bgzf_trunc = str(tmp_path / "trunc_bgzf.fa.gz")
    _write_bgzf(bgzf_trunc, data, random.Random(2), max_block=5000)
    with open(bgzf_trunc, "rb") as f:
        b = f.read()
    with open(bgzf_trunc, "wb") as f:
        f.write(b[:len(b) - 100])
    missing = str(tmp_path / "missing.fa")
    assert "cannot open" in _refused(paths[:3] + [missing] + paths[3:], missing)
    assert "truncated" in _refused(paths + [trunc], trunc, threads=1)
    _refused([corrupt] + paths, corrupt, threads=7)
    assert "CRC" in _refused(paths[:2] + [crc], crc)
    _refused(paths[:1] + [bgzf_trunc], bgzf_trunc)
    # the files before the bad one are delivered first
    r = ingest.FileBatches(paths[:2] + [missing], batch_bytes=1 << 24, threads=2, max_files=1)
    try:
        first = r.next_batch()
        assert bytes(first[0][:int(first[1][-1])]) == want[0]
        r.next_batch()
        with pytest.raises(IOError, match="missing.fa"):
            r.next_batch()
    finally:
        r.close()
