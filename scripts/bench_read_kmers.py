#! /usr/bin/env python
"""Cost of the read k-mer table (Database.query(read_kmers=True)) on bench.py's `weak` workload: 10 M x 150 bp reads
against 2e5 genomes x 1000 sketch slots, one GPU.  Prints one JSON line.

Queries with the table off and on alternate in one process (--reps each); every query pushes the workload's reads from
device buffers and is timed from the first push to the end of mlg_query_sync.  K1 is the CUDA-event time of the probe
launches (mlg_stats.ms_probe), the count kernel that of the table's count launches.  The last query with the table
writes `kmc -k60 -ci2 -cs3` of the reads (reads_60mers) to a temporary directory; with --check the C oracle counts
the same reads on the host and the written database must equal its k-mers seen >= 2 times, counts capped at 3.

    python scripts/bench_read_kmers.py [--reps 5] [--no-check]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-check", action="store_true")
    args = ap.parse_args()
    import torch
    import bench
    import synth
    from metalign_b200 import ingest
    from metalign_b200.api import Context, Database

    name, power = gpu_identity()
    G, paired, batches, total, desc = bench.workload_plan("weak", 1, 0)
    p = bench.synth_params(G, paired)
    ctx = Context(0)
    d_keys = torch.empty(G * p.n * 2, dtype=torch.int64, device="cuda")
    assert synth.cuda_lib().syn_cuda_gen_sketch_keys(C.byref(p), d_keys.data_ptr(), None) == 0
    db = Database.from_device_keys(ctx, d_keys.data_ptr(), G, p.n, bench.K, bench.KS)
    del d_keys
    dev = []
    for r0, n in batches:
        nbb, nmb = synth.packed_sizes(n, bench.READ_LEN)
        d_b = torch.empty(nbb, dtype=torch.uint8, device="cuda")
        d_m = torch.empty(nmb, dtype=torch.uint8, device="cuda")
        assert synth.cuda_lib().syn_cuda_gen_reads_packed(C.byref(p), r0, n, d_b.data_ptr(), d_m.data_ptr(), None) == 0
        dev.append((d_b, d_m, n))
    torch.cuda.synchronize()

    def one(on):
        q = db.query(2, "exact", True, read_kmers=on)
        t0 = time.perf_counter()
        for d_b, d_m, n in dev:
            q.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, bench.READ_LEN, device=True)
        q.sync()
        ms = (time.perf_counter() - t0) * 1e3
        rk = q.read_kmer_stats() if on else None
        q.finish_sparse()
        return q, ms, q.stats(), rk

    one(False)[0].close()                                # warm-up of both shapes
    one(True)[0].close()
    runs = {False: [], True: []}
    last = None
    for i in range(args.reps):
        for on in (False, True):
            q, ms, st, rk = one(on)
            runs[on].append(dict(push_to_sync_ms=ms, k1_ms=st["ms_probe"], rk=rk))
            if on and i == args.reps - 1:
                last = q
            else:
                q.close()
    out = tempfile.mkdtemp(prefix="mlg_rk_")
    prefix = os.path.join(out, "reads_60mers")
    last.write_reads_kmc(prefix, 2, 3)
    rk = last.read_kmer_stats()
    solid = rk["out_records"]
    last.close()

    checked = None
    if not args.no_check:
        from oracle.read_kmers import OracleReadKmers
        bench.all_host_threads()                         # OMP_NUM_THREADS = every host core, before the library loads
        o = OracleReadKmers(60)
        for d_b, d_m, n in dev:
            o.push_packed(d_b.cpu().numpy(), d_m.cpu().numpy(), None, n, bench.READ_LEN)
        wk, wc = o.result(2, 3)
        o.close()
        fk, info, fc = ingest.read_kmc_database(prefix, with_counts=True)
        checked = bool(np.array_equal(fk, wk) and np.array_equal(fc.astype(np.uint8), wc) and info["min_count"] == 2)
    files = sum(os.path.getsize(prefix + e) for e in (".kmc_pre", ".kmc_suf"))
    for e in (".kmc_pre", ".kmc_suf"):
        os.remove(prefix + e)
    os.rmdir(out)

    def med(v):
        return float(np.median(v))
    on, off = runs[True], runs[False]
    count_ms = [r["rk"]["ms_count"] for r in on]
    line = {
        "metric": "read k-mer table cost, weak workload", "gpu": name, "power_limit": power, "workload": desc,
        "reads": total, "reps": args.reps,
        "push_to_sync_ms_off": [r["push_to_sync_ms"] for r in off], "push_to_sync_ms_on": [r["push_to_sync_ms"] for r in on],
        "k1_ms_off": [r["k1_ms"] for r in off], "k1_ms_on": [r["k1_ms"] for r in on],
        "median_push_to_sync_ms_off": med([r["push_to_sync_ms"] for r in off]),
        "median_push_to_sync_ms_on": med([r["push_to_sync_ms"] for r in on]),
        "median_k1_ms_off": med([r["k1_ms"] for r in off]), "median_k1_ms_on": med([r["k1_ms"] for r in on]),
        "count_kernel_ms": count_ms, "windows": on[-1]["rk"]["windows"],
        "windows_per_s": on[-1]["rk"]["windows"] / (med(count_ms) / 1e3),
        "rehashes": rk["grows"], "rehash_ms": rk["ms_rehash"], "table_bytes": rk["bytes"], "distinct": rk["distinct"],
        "solid_ge2": solid, "out_ms_compact": rk["ms_compact"], "out_ms_sort": rk["ms_sort"], "out_ms_encode": rk["ms_encode"],
        "file_write_s": rk["s_write"], "file_bytes": files, "checked": checked,
    }
    print(json.dumps(line))
    db.close()
    ctx.close()


if __name__ == "__main__":
    main()
