"""mlg_kmc_concat (api.kmc_concat): version-0 KMC databases whose keys ascend from one to the next, joined into the one
database that holds them all -- what the ranks of a multi-GPU read k-mer count write, one share of the key order each.
Parts are written by the independent encoder tests/kmcdb.py; the join must be the file that encoder writes for the
union, byte for byte.  Host only: no GPU is needed."""
import os
import random

import pytest

import kmcdb
from metalign_b200.api import MlgError, kmc_concat

ERR_ARG, ERR_IO = -2, -3


def _kmers(K, n, seed):
    rng = random.Random(seed)
    out = {}
    while len(out) < n:
        out["".join(rng.choice("ACGT") for _ in range(K))] = rng.randint(2, 300)
    return out


def _split(kmers, cuts):
    """the k-mers in key order, cut into consecutive parts of the given sizes (the last part takes the rest)"""
    keys = sorted(kmers)
    parts, at = [], 0
    for c in cuts:
        parts.append({k: kmers[k] for k in keys[at:at + c]})
        at += c
    parts.append({k: kmers[k] for k in keys[at:]})
    return parts


def _write_parts(tmp_path, parts, K, **kw):
    names = []
    for i, p in enumerate(parts):
        name = str(tmp_path / ("part%d" % i))
        kmcdb.write(name, p, K, **kw)
        names.append(name)
    return names


def _bytes(prefix):
    return {ext: open(prefix + ext, "rb").read() for ext in (".kmc_pre", ".kmc_suf")}


def _absent(prefix):
    return not os.path.exists(prefix + ".kmc_pre") and not os.path.exists(prefix + ".kmc_suf")


@pytest.mark.parametrize("K,n", [(60, 2000), (31, 1500), (5, 300)])
def test_concat_is_the_database_of_the_union(tmp_path, K, n):
    kmers = _kmers(K, n, K)
    kw = dict(min_count=2, max_count=3)
    parts = _split(kmers, [n // 3, 0, 1, n // 4])             # an empty part, a one-record part
    names = _write_parts(tmp_path, parts, K, **kw)
    before = [_bytes(x) for x in names]
    out = str(tmp_path / "joined")
    kmc_concat(out, names)
    whole = str(tmp_path / "whole")
    kmcdb.write(whole, kmers, K, **kw)
    assert _bytes(out) == _bytes(whole)
    hdr, recs = kmcdb.read(out)
    assert dict(recs) == {k: min(c, 255) for k, c in kmers.items()}
    assert [r[0] for r in recs] == sorted(kmers)
    assert hdr["k"] == K and hdr["total"] == n and hdr["min_count"] == 2 and hdr["max_count"] == 3 and hdr["version"] == 0
    assert hdr["lut_prefix_length"] == kmcdb.choose_lut_prefix_length(K)
    assert [_bytes(x) for x in names] == before                 # the parts are left as they are


@pytest.mark.parametrize("K", [60, 31, 5])
def test_single_part_comes_out_byte_identical(tmp_path, K):
    name = str(tmp_path / "only")
    kmcdb.write(name, _kmers(K, 200, 7), K, min_count=2, max_count=3)
    kmc_concat(str(tmp_path / "out"), [name])
    assert _bytes(str(tmp_path / "out")) == _bytes(name)


def test_empty_parts_are_accepted(tmp_path):
    names = _write_parts(tmp_path, [{}, {}, {}], 60)
    kmc_concat(str(tmp_path / "out"), names)
    hdr, recs = kmcdb.read(str(tmp_path / "out"))
    assert recs == [] and hdr["total"] == 0 and hdr["k"] == 60
    kmcdb.write(str(tmp_path / "empty"), {}, 60)
    assert _bytes(str(tmp_path / "out")) == _bytes(str(tmp_path / "empty"))


def _files(prefix):
    """what exists of a database's two files"""
    return {ext: open(prefix + ext, "rb").read() for ext in (".kmc_pre", ".kmc_suf") if os.path.exists(prefix + ext)}


def _refused(tmp_path, names, code):
    before = [_files(x) for x in names]
    out = str(tmp_path / "out")
    with pytest.raises(MlgError) as e:
        kmc_concat(out, names)
    assert e.value.code == code, str(e.value)
    assert _absent(out)
    assert [_files(x) for x in names] == before


def test_mismatched_parts_are_refused(tmp_path):
    a, b = _split(_kmers(60, 400, 3), [200])
    cases = {
        "k": (dict(), dict(), 31),
        "min_count": (dict(min_count=2), dict(min_count=1), None),
        "max_count": (dict(max_count=3), dict(max_count=255), None),
        "lut_prefix_length": (dict(), dict(lut_prefix_length=8), None),
        "counter_size": (dict(), dict(counter_size=2), None),
    }
    for what, (kw_a, kw_b, k_b) in cases.items():
        d = tmp_path / what
        d.mkdir()
        kmcdb.write(str(d / "a"), a, 60, **kw_a)
        if k_b:
            kmcdb.write(str(d / "b"), {k[:k_b]: c for k, c in b.items()}, k_b, **kw_b)
        else:
            kmcdb.write(str(d / "b"), b, 60, **kw_b)
        _refused(d, [str(d / "a"), str(d / "b")], ERR_ARG)


def test_overlapping_or_descending_parts_are_refused(tmp_path):
    kmers = _kmers(31, 600, 5)
    a, b, c = _split(kmers, [200, 200])
    keys = sorted(kmers)
    overlap = dict(b)
    overlap[keys[199]] = 9                                     # a's last key again
    for what, parts in (("descending", [b, a]), ("overlap", [a, overlap]), ("skip_empty_then_descend", [c, {}, a])):
        d = tmp_path / what
        d.mkdir()
        _refused(d, _write_parts(d, parts, 31), ERR_ARG)
    # equal first and last key across the boundary (one-record parts)
    d = tmp_path / "same_key"
    d.mkdir()
    _refused(d, _write_parts(d, [{keys[0]: 2}, {keys[0]: 3}], 31), ERR_ARG)


def test_missing_or_foreign_files_are_refused(tmp_path):
    a, b = _split(_kmers(60, 300, 9), [100])
    names = _write_parts(tmp_path, [a, b], 60)
    _refused(tmp_path, names + [str(tmp_path / "nothing")], ERR_IO)
    os.remove(names[1] + ".kmc_suf")
    _refused(tmp_path, names, ERR_IO)
    kmcdb.write(names[1], b, 60)
    with open(names[1] + ".kmc_suf", "ab") as f:                # a suffix file that does not match its total
        f.write(b"\0" * 3)
    _refused(tmp_path, names, ERR_ARG)
    kmcdb.write(names[1], b, 60, version=0x200)                # a KMC2 database: not version 0
    _refused(tmp_path, names, ERR_ARG)
    kmcdb.write(names[1], b, 60)
    before = _bytes(names[0])
    with pytest.raises(MlgError) as e:                        # the output is one of the parts
        kmc_concat(names[0], names)
    assert e.value.code == ERR_ARG and _bytes(names[0]) == before
    with pytest.raises(MlgError) as e:
        kmc_concat(str(tmp_path / "out"), [])
    assert e.value.code == ERR_ARG and _absent(str(tmp_path / "out"))
    with pytest.raises(MlgError) as e:                        # an output directory that does not exist
        kmc_concat(str(tmp_path / "no" / "dir" / "out"), names)
    assert e.value.code == ERR_IO
