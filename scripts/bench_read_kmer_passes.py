#! /usr/bin/env python
"""Read k-mers counted in key-range passes (Database.query(read_kmers=True, read_kmer_passes=True)) against the single
table, on bench.py's `weak` workload: 10 M x 150 bp reads generated on the device, 2e5 genomes x 1000 sketch slots, one
GPU.  Prints one JSON line.

Arms, alternated --reps times in one process: the single table; passes with budget 0 (the free device memory: one pass);
passes with budgets that hold the read archive plus about 1/4 and 1/16 of the one-pass table and output stage.  Every
query pushes the reads from device buffers (timed from the first push to the end of mlg_query_sync) and writes
`kmc -k60 -ci2 -cs3` of them (reads_60mers) to a temporary directory: the output call is split into histogram, ranged
counts, select + sort, encode (CUDA events) and copy-back + write (host clock).  The files of all arms must be
byte-identical; without --no-check they are compared once with the C oracle's count of the same reads.

--reads N (N > 10 M) adds a run beyond one table: N reads pushed in 10 M batches.  The single table is tried first on the
same reads (what it does is recorded); then passes with budget 0 write the file, which is checked internally (both
readers here parse it where that is affordable, keys strictly ascending, records = the sum over the passes, windows =
the K1 query's n_kmers).  The C oracle is not used there (its host hash map would need ~100 GB).  If the temporary
directory has less free space than the file can take (8 bytes per window), the file is skipped and the passes are run
through mlg_query_read_kmers without a host buffer instead.

    python scripts/bench_read_kmer_passes.py [--reps 3] [--no-check] [--reads 60000000]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

BATCH = 10_000_000


def pass_bytes(bound):
    """device bytes of a pass whose keys are bounded by `bound` (pass_bytes in csrc/readkmers.cu)"""
    s = 1 << 12
    while s * 0.7 < bound:
        s *= 2
    return s * 16 + bound * 104


def digest(prefix):
    h = hashlib.sha256()
    for e in (".kmc_pre", ".kmc_suf"):
        with open(prefix + e, "rb") as f:
            for blk in iter(lambda: f.read(1 << 24), b""):
                h.update(blk)
    return h.hexdigest()


def remove(prefix):
    for e in (".kmc_pre", ".kmc_suf"):
        if os.path.exists(prefix + e):
            os.remove(prefix + e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--reads", type=int, default=0, help="also run N reads (> 10 M) beyond one table")
    args = ap.parse_args()
    import torch
    import bench
    import synth
    from bench_read_kmers import gpu_identity
    from metalign_b200 import ingest
    from metalign_b200.api import Context, Database, MlgError

    name, power = gpu_identity()
    G, paired, batches, total, desc = bench.workload_plan("weak", 1, 0)
    p = bench.synth_params(G, paired)
    ctx = Context(0)
    d_keys = torch.empty(G * p.n * 2, dtype=torch.int64, device="cuda")
    assert synth.cuda_lib().syn_cuda_gen_sketch_keys(C.byref(p), d_keys.data_ptr(), None) == 0
    db = Database.from_device_keys(ctx, d_keys.data_ptr(), G, p.n, bench.K, bench.KS)
    del d_keys

    def gen(r0, n):
        nbb, nmb = synth.packed_sizes(n, bench.READ_LEN)
        d_b = torch.empty(nbb, dtype=torch.uint8, device="cuda")
        d_m = torch.empty(nmb, dtype=torch.uint8, device="cuda")
        assert synth.cuda_lib().syn_cuda_gen_reads_packed(C.byref(p), r0, n, d_b.data_ptr(), d_m.data_ptr(), None) == 0
        return d_b, d_m, n
    dev = [gen(r0, n) for r0, n in batches]
    torch.cuda.synchronize()
    out = tempfile.mkdtemp(prefix="mlg_rkp_")

    def one(passes, budget, reads, prefix):
        q = db.query(2, "exact", True, read_kmers=True, read_kmer_budget=budget, read_kmer_passes=passes)
        t0 = time.perf_counter()
        for d_b, d_m, n in reads:
            q.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, bench.READ_LEN, device=True)
        q.sync()
        push_ms = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        q.write_reads_kmc(prefix, 2, 3)
        out_s = time.perf_counter() - t0
        st = q.read_kmer_stats()
        plan = q.read_kmer_plan() if passes else None
        r = dict(push_to_sync_ms=push_ms, output_call_s=out_s,
                 histogram_ms=plan["ms_histogram"] if plan else 0.0, count_ms=st["ms_count"],
                 select_sort_ms=st["ms_compact"] + st["ms_sort"], encode_ms=st["ms_encode"], write_s=st["s_write"],
                 passes=plan["passes"] if plan else 1, refined_bins=plan["refined_bins"] if plan else 0,
                 archive_bytes=plan["archive_bytes"] if plan else 0, max_pass_bound=plan["max_pass_bound"] if plan else 0,
                 table_bytes=st["bytes"], windows=st["windows"], distinct=st["distinct"], records=st["out_records"])
        return q, r

    # the budgets of the 4- and 16-pass arms, from the one-pass plan
    q, r = one(True, 0, dev, os.path.join(out, "warm"))
    q.close()
    remove(os.path.join(out, "warm"))
    q, _ = one(False, 0, dev, os.path.join(out, "warm"))
    q.close()
    remove(os.path.join(out, "warm"))
    arms = [("single", False, 0), ("passes_budget0", True, 0)]
    for parts in (4, 16):
        arms.append(("passes_about_%d" % parts, True, r["archive_bytes"] + pass_bytes(-(-r["windows"] // parts))))
    runs = {a[0]: [] for a in arms}
    digests = {}
    keep = None
    for i in range(args.reps):
        for label, passes, budget in arms:
            prefix = os.path.join(out, "%s_%d" % (label, i))
            q, res = one(passes, budget, dev, prefix)
            q.close()
            res["budget"] = budget
            runs[label].append(res)
            digests.setdefault(label, set()).add(digest(prefix))
            if keep is None:
                keep = prefix
            else:
                remove(prefix)
    identical = len(set().union(*digests.values())) == 1

    checked = None
    if not args.no_check:
        from oracle.read_kmers import OracleReadKmers
        bench.all_host_threads()
        o = OracleReadKmers(60)
        for d_b, d_m, n in dev:
            o.push_packed(d_b.cpu().numpy(), d_m.cpu().numpy(), None, n, bench.READ_LEN)
        wk, wc = o.result(2, 3)
        o.close()
        fk, info, fc = ingest.read_kmc_database(keep, with_counts=True)
        checked = bool(np.array_equal(fk, wk) and np.array_equal(fc.astype(np.uint8), wc) and info["min_count"] == 2)
    file_bytes = sum(os.path.getsize(keep + e) for e in (".kmc_pre", ".kmc_suf"))
    remove(keep)

    def med(label, key):
        return float(np.median([x[key] for x in runs[label]]))
    summary = {label: {k: med(label, k) for k in ("push_to_sync_ms", "output_call_s", "histogram_ms", "count_ms",
                                                   "select_sort_ms", "encode_ms", "write_s")} for label, _, _ in arms}
    for label, _, _ in arms:
        summary[label].update(passes=runs[label][-1]["passes"], archive_bytes=runs[label][-1]["archive_bytes"],
                              budget=runs[label][-1]["budget"])
    line = {"metric": "read k-mer passes vs single table, weak workload", "gpu": name, "power_limit": power, "workload": desc,
            "reads": total, "reps": args.reps, "runs": runs, "median": summary, "files_identical": identical,
            "file_bytes": file_bytes, "checked": checked}

    if args.reads > total:
        del dev
        torch.cuda.empty_cache()
        big = [gen(r0, min(BATCH, args.reads - r0)) for r0 in range(0, args.reads, BATCH)]
        torch.cuda.synchronize()
        beyond = {"reads": args.reads, "batches": len(big)}
        # the single table on the same reads
        q = db.query(2, "exact", True, read_kmers=True)
        single = {}
        t0 = time.perf_counter()
        try:
            for i, (d_b, d_m, n) in enumerate(big):
                single["batches_pushed"] = i
                q.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, bench.READ_LEN, device=True)
            q.sync()
            single["push_to_sync_ms"] = (time.perf_counter() - t0) * 1e3
            n = C.c_uint64()
            from metalign_b200 import _lib
            _lib.check(_lib.lib().mlg_query_read_kmers(q._h, 2, 3, None, None, 0, C.byref(n)))
            single["result"] = "ok"
            single["records"] = n.value
        except MlgError as e:
            single["result"] = "MlgError %d: %s" % (e.code, e)
        try:
            single["stats"] = q.read_kmer_stats()
        except MlgError as e:
            single["stats"] = "MlgError %d: %s" % (e.code, e)
        q.close()
        beyond["single_table"] = single
        # passes, budget 0
        q = db.query(2, "exact", True, read_kmers=True, read_kmer_passes=True)
        t0 = time.perf_counter()
        for d_b, d_m, n in big:
            q.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, bench.READ_LEN, device=True)
        q.sync()
        push_ms = (time.perf_counter() - t0) * 1e3
        k1 = db.query(2, "exact", True)
        for d_b, d_m, n in big:
            k1.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, bench.READ_LEN, device=True)
        n_kmers = k1.finish_sparse()["n_kmers"]
        k1.close()
        windows_pushed = args.reads * (bench.READ_LEN - bench.K + 1)
        free = shutil.disk_usage(out).free
        prefix = os.path.join(out, "beyond")
        t0 = time.perf_counter()
        if free >= 8 * windows_pushed:
            q.write_reads_kmc(prefix, 2, 3)
            file_check = "written"
        else:
            n = C.c_uint64()
            from metalign_b200 import _lib
            _lib.check(_lib.lib().mlg_query_read_kmers(q._h, 2, 3, None, None, 0, C.byref(n)))
            file_check = "skipped: %d bytes free, up to %d needed" % (free, 8 * windows_pushed)
        out_s = time.perf_counter() - t0
        st, plan = q.read_kmer_stats(), q.read_kmer_plan()
        q.close()
        res = {"push_to_sync_ms": push_ms, "output_call_s": out_s, "plan": plan, "stats": st, "file": file_check,
               "windows_equal_k1_n_kmers": st["windows"] == n_kmers}
        if file_check == "written":
            res["file_bytes"] = sum(os.path.getsize(prefix + e) for e in (".kmc_pre", ".kmc_suf"))
            fk, info = ingest.read_kmc_database(prefix)
            hi, lo = fk[:, 0], fk[:, 1]
            asc = bool(np.all((hi[1:] > hi[:-1]) | ((hi[1:] == hi[:-1]) & (lo[1:] > lo[:-1]))))
            res.update(native_reader_records=int(len(fk)), keys_ascending=asc,
                       records_equal_sum_over_passes=int(len(fk)) == st["out_records"] == info["total"],
                       python_reader="not run: it decodes record by record in Python")
            del fk, hi, lo
            remove(prefix)
        beyond["passes"] = res
        line["beyond_one_table"] = beyond
    os.rmdir(out)
    print(json.dumps(line))
    db.close()
    ctx.close()


if __name__ == "__main__":
    main()
