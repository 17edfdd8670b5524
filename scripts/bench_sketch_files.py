#! /usr/bin/env python
"""Genome files -> built .mlgdb: the two-step path (make_sketch_db.py + build_db.py: read_fasta, mlg_sketch_genomes,
source file, Database.load, save) against make_sketch_db.py --built (native reader -> FASTA cut and sketch on the device
-> builder -> save), on seeded synthetic genome files (gzip level 6, 80-column lines) written to a temporary directory.

    python scripts/bench_sketch_files.py [--genomes 2000] [--genome-bp 3000000] [--old-subset 100] [--threads 0]

Prints one JSON line: the card and its power limit, wall time and text GB/s of both paths, the --built path's stage
times, a reader-only pass, and whether the two built files are byte-identical.  The old path reads with one Python
thread (hours for thousands of genomes), so it runs on the first --old-subset genomes only, and the --built path runs on
that subset as well for the byte comparison; `old_subset_genomes` in the output says how many."""
import argparse
import json
import multiprocessing as mp
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _write_genome(args):
    path, seed, bp = args
    rng = np.random.default_rng(seed)
    bases = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, bp)]
    bases[rng.integers(0, bp, bp // 5000)] = ord("N")
    nrec = 1 + int(rng.integers(0, 4))
    cuts = np.sort(rng.integers(0, bp, nrec - 1))
    parts, prev = [], 0
    for r, c in enumerate(list(cuts) + [bp]):
        seq = bases[prev:c]
        lines = [seq[i:i + 80].tobytes() for i in range(0, seq.size, 80)]
        parts.append(b">contig_%d synthetic seed %d\n" % (r, seed) + b"\n".join(lines) + b"\n")
        prev = c
    text = b"".join(parts)
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    with open(path, "wb") as f:
        f.write(co.compress(text) + co.flush())
    return len(text)


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = out.strip().splitlines()[0].split(", ")
        return name, power
    except Exception:  # noqa: BLE001
        return "unknown", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genomes", type=int, default=2000)
    ap.add_argument("--genome-bp", type=int, default=3_000_000)
    ap.add_argument("--old-subset", type=int, default=100)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("-n", type=int, default=1000)
    ap.add_argument("-k", type=int, default=60)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    from metalign_b200.api import Context, Database
    from metalign_b200.ingest import FileBatches
    from metalign_b200.sketch import build_database, build_database_from_files
    ks = [k for k in (30, 40, 50, 60) if k <= a.k]
    tmp = tempfile.mkdtemp(prefix="mlg_sketch_files_")
    try:
        paths = [os.path.join(tmp, "genome_%05d.fna.gz" % i) for i in range(a.genomes)]
        t0 = time.perf_counter()
        with mp.Pool() as pool:
            text_bytes = pool.map(_write_genome, [(p, a.seed * 1000003 + i, a.genome_bp) for i, p in enumerate(paths)])
        s_gen = time.perf_counter() - t0
        gz_bytes = sum(os.path.getsize(p) for p in paths)
        sub = paths[:min(a.old_subset, len(paths))]
        sub_text = sum(text_bytes[:len(sub)])
        total_text = sum(text_bytes)
        name, power = gpu_info()
        res = {"bench": "sketch_files", "gpu": name, "power_limit": power, "genomes": a.genomes, "genome_bp": a.genome_bp,
               "n": a.n, "K": a.k, "text_GB": total_text / 1e9, "gzip_GB": gz_bytes / 1e9, "s_generate": s_gen,
               "host_cpus": os.cpu_count(), "old_subset_genomes": len(sub)}
        # reader alone: what the host delivers when nothing waits for the GPU
        t0 = time.perf_counter()
        r = FileBatches(paths, batch_bytes=64 << 20, threads=a.threads)
        got = sum(int(off[-1]) for _, off in r)
        r.close()
        res["reader_s"] = time.perf_counter() - t0
        res["reader_GBps"] = got / 1e9 / res["reader_s"]
        with Context(0) as ctx:
            # warm-up: module load and pool
            build_database_from_files(ctx, paths[:2], os.path.join(tmp, "warm.mlgdb"), a.n, a.k, ks, threads=a.threads)
            # old two-step path on the subset
            t0 = time.perf_counter()
            src = os.path.join(tmp, "old.src.mlgdb")
            build_database(ctx, sub, src, a.n, a.k, ks)
            t1 = time.perf_counter()
            db = Database.load(ctx, src)
            db.save(os.path.join(tmp, "old.mlgdb"))
            db.close()
            t2 = time.perf_counter()
            res["old_subset_s"] = t2 - t0
            res["old_subset_sketch_s"] = t1 - t0
            res["old_subset_build_save_s"] = t2 - t1
            res["old_subset_text_GBps"] = sub_text / 1e9 / (t2 - t0)
            t0 = time.perf_counter()
            build_database_from_files(ctx, sub, os.path.join(tmp, "new_sub.mlgdb"), a.n, a.k, ks, threads=a.threads)
            res["built_subset_s"] = time.perf_counter() - t0
            with open(os.path.join(tmp, "old.mlgdb"), "rb") as f1, open(os.path.join(tmp, "new_sub.mlgdb"), "rb") as f2:
                res["byte_identical"] = f1.read() == f2.read()
            # --built on every genome
            t0 = time.perf_counter()
            st = build_database_from_files(ctx, paths, os.path.join(tmp, "new.mlgdb"), a.n, a.k, ks, threads=a.threads)
            res["built_s"] = time.perf_counter() - t0
            res["built_text_GBps"] = total_text / 1e9 / res["built_s"]
            res["stages"] = {"read_wait_s": st["s_read_wait"], "h2d_ms": st["ms_h2d"], "cut_ms": st["ms_cut"],
                             "sketch_kernels_ms": st["ms_sketch"], "keys_and_append_ms": st["ms_keys"],
                             "finish_s": st["s_finish"], "save_s": st["s_save"], "passes": st["passes"]}
        line = json.dumps(res)
        print(line)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
