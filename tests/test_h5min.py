"""metalign_b200/h5min.py -- the minimal HDF5 reader that lets scripts/make_db_from_h5.py read CMash's training database
(select_db.py:69) without h5py -- pinned on a REAL HDF5 file (written by MATLAB's HDF5 library: tests/golden/testhdf5_7.4_GLNX86.mat,
a copy of scipy's test file scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat, BSD-3-Clause) and on files made by the
independent writer tests/h5write.py in CMash's layout (SURVEY.md A.2)."""
import importlib.util
import os
import random

import numpy as np
import pytest

import h5write
from metalign_b200 import codec, dbformat, h5min

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REAL_HDF5 = os.path.join(ROOT, "tests", "golden", "testhdf5_7.4_GLNX86.mat")


def test_reads_a_real_hdf5_file():
    """a MATLAB v7.3 file = HDF5 behind a 512-byte user block: superblock 0, old-style root group, one float64 dataset with
    an attribute.  scipy's own tests say what the variable holds in the sibling files of other formats: theta = 0, pi/4 .. 2 pi"""
    with h5min.H5File(REAL_HDF5) as f:
        assert f.base == 512 and f.keys() == ["testdouble"]
        d = f["testdouble"]
        assert isinstance(d, h5min.Dataset) and d.shape == (9, 1) and d.dtype == np.dtype("<f8")
        assert np.allclose(d.read().reshape(-1), np.pi / 4 * np.arange(9), rtol=0, atol=1e-15)
        assert d.attrs["MATLAB_class"] == b"double"
        with pytest.raises(KeyError):
            f["nothing"]


def _random_sketches(rng, G, n, K):
    sk = {}
    for g in range(G):
        name = "taxid_%d_genomic.fna.gz" % rng.randrange(10 ** 6) if g else "zzz_last.fna.gz"
        real = n if rng.random() < 0.8 else rng.randint(0, n - 1)
        kmers = ["".join(rng.choice("ACGT") for _ in range(K)).encode() for _ in range(real)] + [b""] * (n - real)
        mins = sorted(rng.randrange(1 << 40) for _ in range(real)) + [9999999999971] * (n - real)
        sk[name] = (mins, [rng.randint(1, 9) if i < real else 0 for i in range(n)], kmers)
    return sk


@pytest.mark.parametrize("G,user_block", [(1, 0), (9, 0), (300, 512), (2100, 0)])
def test_cmash_layout_roundtrip(tmp_path, G, user_block):
    """1 genome; 9 (two symbol-table nodes under one B-tree node); 300 (38 nodes: a two-level B-tree); 2100 (three levels)"""
    rng = random.Random(G)
    K, n = 60, 7
    sk = _random_sketches(rng, G, n, K)
    p = str(tmp_path / "train.h5")
    h5write.write_cmash_h5(p, sk, K, user_block=user_block)
    with h5min.H5File(p) as f:
        grp = f["CountEstimators"]
        assert grp.keys() == sorted(sk)
        for name in rng.sample(sorted(sk), min(G, 40)):
            g = grp[name]
            assert g.keys() == ["counts", "kmers", "mins"] and int(g.attrs["ksize"]) == K and g.attrs["class"] == b"CountEstimator"
            mins, counts, kmers = sk[name]
            assert g["kmers"].dtype == np.dtype("S60") and g["kmers"].shape == (n,)
            assert [bytes(x) for x in g["kmers"].read()] == kmers
            assert g["mins"].read().tolist() == mins and g["counts"].read().tolist() == counts
        assert isinstance(f["CountEstimators/" + sorted(sk)[0] + "/mins"], h5min.Dataset)


def test_make_db_from_h5_without_h5py(tmp_path):
    """scripts/make_db_from_h5.py end to end on a file in CMash's layout: names in sorted order, '' slots empty, the keys
    of every slot -- and the refusals: a truncated file, a file that is not HDF5, sketches of unequal size"""
    spec = importlib.util.spec_from_file_location("make_db_from_h5", os.path.join(ROOT, "scripts", "make_db_from_h5.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rng = random.Random(11)
    K, n = 60, 12
    sk = _random_sketches(rng, 25, n, K)
    p = str(tmp_path / "train.h5")
    h5write.write_cmash_h5(p, sk, K)
    out = str(tmp_path / "db.mlgdb")
    mod.main([p, out])
    assert dbformat.read_names(out) == sorted(sk)
    want = codec.sketches_to_keys([[k.decode() for k in sk[name][2]] for name in sorted(sk)], K)
    assert np.array_equal(dbformat.read_keys(out).reshape(-1), np.asarray(want).reshape(-1))
    h = dbformat.read_header(out)
    assert h["K"] == K and h["n"] == n and list(h["ks"]) == [30, 40, 50, 60]
    raw = open(p, "rb").read()
    open(p, "wb").write(raw[: len(raw) // 3])
    with pytest.raises((h5min.H5Unsupported, SystemExit, KeyError, Exception)):
        mod.main([p, out])
    open(p, "wb").write(b"not an hdf5 file" * 100)
    with pytest.raises(h5min.H5Unsupported):
        h5min.H5File(p)
    bad = dict(list(sk.items())[:2])
    first = next(iter(bad))
    bad[first] = (bad[first][0][:-1], bad[first][1][:-1], bad[first][2][:-1])
    h5write.write_cmash_h5(p, bad, K)
    with pytest.raises(SystemExit):
        mod.main([p, out])


def test_damaged_files_raise_cleanly(tmp_path):
    """random byte damage and truncation of a valid file: every outcome is a parsed value, a KeyError for a name that is gone,
    or H5Unsupported -- never another exception, never a hang (B-tree cycles are detected)"""
    rng = random.Random(5)
    K, n = 60, 6
    sk = _random_sketches(rng, 40, n, K)
    p = str(tmp_path / "ok.h5")
    h5write.write_cmash_h5(p, sk, K)
    good = bytearray(open(p, "rb").read())
    q = str(tmp_path / "bad.h5")
    outcomes = {"ok": 0, "refused": 0}
    for trial in range(300):
        raw = bytearray(good)
        if trial % 5 == 0:
            raw = raw[: rng.randrange(8, len(raw))]
        else:
            for _ in range(rng.randint(1, 6)):
                i = rng.randrange(len(raw))
                raw[i] = rng.randrange(256) if trial % 2 else raw[i] ^ (1 << rng.randrange(8))
        open(q, "wb").write(bytes(raw))
        try:
            with h5min.H5File(q) as f:
                grp = f["CountEstimators"]
                for name in grp.keys()[:12]:
                    g = grp[name]
                    g["kmers"].read()
                    g.attrs
            outcomes["ok"] += 1
        except (h5min.H5Unsupported, KeyError):
            outcomes["refused"] += 1
    assert outcomes["ok"] > 0 and outcomes["refused"] > 0, outcomes
