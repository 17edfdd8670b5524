#! /usr/bin/env python
"""reads_60mers of reads sharded over the GPUs (dist.share_read_kmers + dist.write_reads_kmc) against one passes-mode
query of the same reads on one GPU, on bench.py's `weak` workload: 10 M x 150 bp reads per GPU generated on the device,
2e5 genomes x 1000 sketch slots.  Run it under torchrun (one process per GPU; plain python is one rank).  Rank 0 prints
one JSON line.

Per rank, for the sharded run: the archive exchange (share_read_kmers, host clock to a join of the compute stream), the
output call's histogram, ranged counts and select + sort (CUDA events), the part write and, on rank 0, the concatenation
(host clock), and the wall time of dist.write_reads_kmc.  Then rank 0 alone runs one passes-mode query over every rank's
reads (budget 0) and writes the same database.  The two files must be byte-identical; without --no-check, and up to
20 M reads in all, rank 0 compares them once with the C oracle's count of the same reads.  Rank 0's reference runs come
after the process group is gone, so the other ranks never wait on them.

    torchrun --nproc_per_node N scripts/bench_read_kmers_sharded.py [--no-check]
"""
import argparse
import ctypes as C
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


ORACLE_MAX_READS = 20_000_000      # the C oracle's host hash map: ~100 GB at 60 M reads


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--out", default="", help="directory for the databases (default: a temporary one; must be shared by the ranks)")
    args = ap.parse_args()
    import torch
    import torch.distributed as tdist
    import bench
    import synth
    from bench_read_kmer_passes import digest, remove
    from bench_read_kmers import gpu_identity
    from metalign_b200 import dist as mdist
    from metalign_b200 import ingest
    from metalign_b200.api import Context, Database

    rank, world, local = mdist.init_from_env("nccl")
    torch.cuda.set_device(local)
    name, power = gpu_identity()
    G, paired, batches, total, desc = bench.workload_plan("weak", world, rank)
    p = bench.synth_params(G, 0)                         # unpaired reads at every world size: the single run repeats them
    ctx = Context(local)
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

    out = args.out or (tempfile.mkdtemp(prefix="mlg_rks_") if rank == 0 else "")
    if world > 1:
        box = [out]
        tdist.broadcast_object_list(box, src=0)
        out = box[0]
    mine = [gen(r0, n) for r0, n in batches]
    torch.cuda.synchronize()

    q = db.query(2, "exact", True, read_kmers=True, read_kmer_passes=True)
    for d_b, d_m, n in mine:
        q.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, bench.READ_LEN, device=True)
    q.sync()
    del mine
    torch.cuda.synchronize()
    if world > 1:
        tdist.barrier()
    t0 = time.perf_counter()
    mdist.share_read_kmers(q, local)
    q.sync()
    exchange_s = time.perf_counter() - t0
    if world > 1:
        tdist.barrier()
    prefix = os.path.join(out, "sharded")
    t0 = time.perf_counter()
    times = mdist.write_reads_kmc(q, prefix, 2, 3, local)
    write_s = time.perf_counter() - t0
    plan, st = q.read_kmer_plan(), q.read_kmer_stats()
    me = dict(rank=rank, exchange_s=exchange_s, histogram_ms=plan["ms_histogram"], count_ms=plan["ms_count"],
              select_sort_ms=st["ms_compact"] + st["ms_sort"], encode_ms=st["ms_encode"], part_s=times["part_s"],
              concat_s=times["concat_s"], write_reads_kmc_s=write_s, passes=plan["passes"], refined_bins=plan["refined_bins"],
              archive_bytes=plan["archive_bytes"], share_bins=[plan["share_first_bin"], plan["share_end_bin"]],
              share_windows=plan["share_windows"], windows=st["windows"], distinct=plan["distinct"], records=st["out_records"])
    q.close()
    ranks = [me]
    if world > 1:
        ranks = [None] * world
        tdist.all_gather_object(ranks, me)
        tdist.destroy_process_group()           # the other ranks are done: rank 0's reference runs need no collective
    if rank == 0:
        # one passes-mode query over every rank's reads on this GPU
        one = db.query(2, "exact", True, read_kmers=True, read_kmer_passes=True)
        for r in range(world):
            for r0, n in bench.workload_plan("weak", world, r)[2]:
                d_b, d_m, n = gen(r0, n)
                one.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, bench.READ_LEN, device=True)
                one.sync()
                del d_b, d_m
        single = os.path.join(out, "single")
        t0 = time.perf_counter()
        one.write_reads_kmc(single, 2, 3)
        single_s = time.perf_counter() - t0
        plan1, st1 = one.read_kmer_plan(), one.read_kmer_stats()
        one.close()
        identical = digest(prefix) == digest(single)
        checked = None
        if not args.no_check and total <= ORACLE_MAX_READS:
            from oracle.read_kmers import OracleReadKmers
            bench.all_host_threads()
            o = OracleReadKmers(60)
            for r in range(world):
                for r0, n in bench.workload_plan("weak", world, r)[2]:
                    d_b, d_m, n = gen(r0, n)
                    o.push_packed(d_b.cpu().numpy(), d_m.cpu().numpy(), None, n, bench.READ_LEN)
            wk, wc = o.result(2, 3)
            o.close()
            fk, info, fc = ingest.read_kmc_database(prefix, with_counts=True)
            checked = bool(np.array_equal(fk, wk) and np.array_equal(fc.astype(np.uint8), wc) and info["min_count"] == 2)
        file_bytes = sum(os.path.getsize(prefix + e) for e in (".kmc_pre", ".kmc_suf"))
        remove(prefix)
        remove(single)
        if not args.out:
            shutil.rmtree(out, ignore_errors=True)
        line = {"metric": "reads_60mers of reads sharded over the GPUs vs one passes query on one GPU, weak workload",
                "gpu": name, "power_limit": power, "world": world, "workload": desc, "total_reads": total,
                "sharded": dict(ranks=ranks, write_reads_kmc_s=max(x["write_reads_kmc_s"] for x in ranks),
                                exchange_s=max(x["exchange_s"] for x in ranks),
                                exchange_plus_write_s=max(x["exchange_s"] + x["write_reads_kmc_s"] for x in ranks)),
                "single_gpu": dict(write_reads_kmc_s=single_s, histogram_ms=plan1["ms_histogram"], count_ms=plan1["ms_count"],
                                   select_sort_ms=st1["ms_compact"] + st1["ms_sort"], encode_ms=st1["ms_encode"], write_s=st1["s_write"],
                                   passes=plan1["passes"], records=st1["out_records"]),
                "files_identical": identical, "oracle_checked": checked, "file_bytes": file_bytes}
        print(json.dumps(line))
    db.close()
    ctx.close()


if __name__ == "__main__":
    main()
