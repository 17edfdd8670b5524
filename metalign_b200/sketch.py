"""Sketch builder: the GPU replacement of CMash's `MakeStreamingDNADatabase.py <list> <out.h5> -n 1000 -k 60`
(local_tests/retrain_and_test_metalign.sh:49 of the reference) for this repo's database format.

    python scripts/make_sketch_db.py genomes.txt out.mlgdb [-n 1000] [-k 60] [--k_range 30-60-10]

`genomes.txt` lists one FASTA path per line (plain or .gz), as the reference's training list does.  Each genome's
bottom-n MinHash sketch (forward strand, MurmurHash3 mod prime: include/metalign_b200.h, mlg_sketch_genomes) is computed
on the GPU; genomes are stored in sorted-basename order, the order in which CMash's import_multiple_from_single_hdf5
hands them to dump_kmers.py:7-14 and StreamingQueryDNADatabase.py, so genome indices mean the same thing.
No CPU fallback: without the CUDA library and a GPU every call raises.
"""
from __future__ import annotations

import argparse
import ctypes as C
import gzip
import os
import sys
from typing import Iterable, Sequence

import numpy as np

from . import _lib
from ._lib import check

PRIME = 9999999999971      # CMash MinHash.CountEstimator's default max_prime (itself prime)
GENOMES_PER_CALL = (1 << 20) - 1   # mlg_sketch_genomes takes G < 2^20 genomes per call


def read_fasta(path: str) -> bytes:
    """All records of a FASTA file (plain or .gz) as one byte string, records separated by b'N' so that no k-mer spans two
    of them (CMash hashes record by record)."""
    op = gzip.open if path.endswith(".gz") else open
    recs, cur = [], []
    with op(path, "rb") as f:
        for line in f:
            if line.startswith(b">"):
                if cur:
                    recs.append(b"".join(cur))
                    cur = []
            else:
                cur.append(line.strip())
    if cur:
        recs.append(b"".join(cur))
    return b"N".join(recs)


def sketch_genomes(ctx, genomes: Sequence[bytes], n: int = 1000, K: int = 60, prime: int = 0):
    """-> (mins [G, n] uint64, counts [G, n] uint32, kmers [G, n, K] uint8 (NUL where the slot is unused), stats dict)"""
    texts = [g.encode() if isinstance(g, str) else bytes(g) for g in genomes]
    G = len(texts)
    off = np.zeros(G + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(t) for t in texts])
    text = np.frombuffer(b"".join(texts) + b"N", dtype=np.uint8)
    mins = np.empty((G, n), dtype=np.uint64)
    counts = np.empty((G, n), dtype=np.uint32)
    kmers = np.empty((G, n, K), dtype=np.uint8)
    st = _lib.SketchStats()
    check(_lib.lib().mlg_sketch_genomes(ctx._h, text.ctypes.data, off.ctypes.data, G, n, K, prime, mins.ctypes.data,
                                        counts.ctypes.data, kmers.ctypes.data, C.addressof(st)))
    return mins, counts, kmers, {f: getattr(st, f) for f, _ in st._fields_ if f != "reserved"}


def build_database(ctx, paths: Iterable[str], out_path: str, n: int = 1000, K: int = 60, ks: Sequence[int] = (30, 40, 50, 60),
                   batch_bytes: int = 1 << 30, log=None):
    """Sketch every genome file and write the .mlgdb database (metalign_b200/dbformat.py).  Returns the stats.
    Genomes go to the GPU in calls of about batch_bytes of text and at most GENOMES_PER_CALL genomes."""
    from . import codec, dbformat
    paths = sorted(paths, key=os.path.basename)
    names = [os.path.basename(p) for p in paths]
    G = len(paths)
    keys = np.empty((G * n, 2), dtype=np.uint64)
    tot = {"n_windows": 0, "n_candidates": 0, "ms_kernels": 0.0, "passes": 0}
    i = 0
    while i < G:
        batch, nbytes = [], 0
        while i < G and (not batch or nbytes < batch_bytes) and len(batch) < GENOMES_PER_CALL:
            batch.append(read_fasta(paths[i]))
            nbytes += len(batch[-1])
            i += 1
        _, _, kmers, st = sketch_genomes(ctx, batch, n, K)
        g0 = i - len(batch)
        keys[g0 * n:i * n] = codec.ascii_slots_to_keys(kmers.reshape(-1, K), K)
        for k in tot:
            tot[k] += st[k]
        if log:
            log("sketched %d / %d genomes" % (i, G))
    dbformat.write(out_path, keys.reshape(-1), names, G, n, K, list(ks))
    return tot


def main(argv=None):
    ap = argparse.ArgumentParser(description="GPU sketch builder (CMash MakeStreamingDNADatabase.py equivalent) -> .mlgdb")
    ap.add_argument("in_file", help="text file with one genome FASTA path (plain or .gz) per line")
    ap.add_argument("out_file", help=".mlgdb database to write")
    ap.add_argument("-n", "--num_hashes", type=int, default=1000)
    ap.add_argument("-k", "--k_size", type=int, default=60)
    ap.add_argument("--k_range", default="30-60-10", help="prefix lengths the database will be queried at")
    ap.add_argument("--device", type=int, default=0)
    a = ap.parse_args(argv)
    # what the database loader accepts (1 <= K <= 63, 1..8 ascending ks within 1..K), checked before any genome is read
    if not 1 <= a.k_size <= 63:
        ap.error("-k %d: a database needs 1 <= K <= 63" % a.k_size)
    try:
        lo, hi, step = (int(x) for x in a.k_range.split("-"))
    except ValueError:
        ap.error("--k_range %s: expected lo-hi-step" % a.k_range)
    if lo < 1 or step < 1:
        ap.error("--k_range %s: need lo >= 1 and step >= 1" % a.k_range)
    ks = [k for k in range(lo, hi + 1, step) if k <= a.k_size]
    if not 1 <= len(ks) <= 8:
        ap.error("--k_range %s with -k %d gives %d prefix lengths %s; a database needs 1 to 8" % (a.k_range, a.k_size, len(ks), ks))
    with open(a.in_file) as f:
        paths = [ln.strip() for ln in f if ln.strip()]
    from .api import Context
    with Context(a.device) as ctx:
        st = build_database(ctx, paths, a.out_file, a.num_hashes, a.k_size, ks, log=lambda m: print(m, file=sys.stderr))
    print("wrote %s: %d genomes x %d slots, K=%d, ks=%s; %d windows hashed in %.1f ms of kernels"
          % (a.out_file, len(paths), a.num_hashes, a.k_size, ks, st["n_windows"], st["ms_kernels"]))


if __name__ == "__main__":
    main()
