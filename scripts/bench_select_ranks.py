#! /usr/bin/env python
"""select_db.py on 1, 2, 4 and 8 GPUs of one node (torchrun, one process per GPU), on a deep synthetic sample: 40 M x 150 bp
reads of bench.py's default-scale database (2e5 genomes x 1000 slots), written once as plain FASTQ (12.7 GB of text) and
once as BGZF FASTQ.  Every run reads a file that was read just before it (warm page cache), and every rank reads
cores // world threads.  One JSON line per (format, world): wall time of select_main and the slowest rank's stages --
reader and database open, pushes (the reader's time: reads are probed as they arrive), exchange, finish, and the rest
(selection and files) -- the text rate, the GPU name and power limit, and the host core count.  Each run's CSV must equal
the one-GPU plain run's.

    python scripts/bench_select_ranks.py [--reads 40000000] [--worlds 1,2,4,8] [--dir DIR] [--out results.jsonl]

The child mode (--run) is what torchrun starts.
"""
import argparse
import ctypes as C
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
REC = 317                       # "@r" + 10 digits, '\n', 150 bases, '\n', "+\n", 150 quality bytes, '\n'
CHUNK = 1_000_000


def _fastq_chunk(p, r0, n):
    import synth
    seq = synth.reads_ascii(p, r0, n)
    out = np.empty((n, REC), dtype=np.uint8)
    idx = np.arange(r0, r0 + n, dtype=np.int64)
    out[:, 0], out[:, 1] = ord("@"), ord("r")
    for d in range(10):
        out[:, 2 + d] = 48 + (idx // 10 ** (9 - d)) % 10
    out[:, 12] = out[:, 163] = out[:, 165] = out[:, 316] = 10
    out[:, 13:163] = seq
    out[:, 164] = ord("+")
    out[:, 166:316] = 35 + (seq * 7 + np.arange(150, dtype=np.uint8)) % 40         # quality-like, not all one symbol
    return out.reshape(-1)


def _bgzf_member(chunk):
    import struct
    import zlib
    co = zlib.compressobj(1, zlib.DEFLATED, -15)
    body = co.compress(chunk) + co.flush()
    return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, 12 + 6 + len(body) + 8 - 1)
            + body + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))


def _chunk_job(job):
    """(FASTQ text, the same text as BGZF members) of reads [r0, r0 + n)"""
    import bench
    G, r0, n = job
    text = _fastq_chunk(bench.synth_params(G, 0), r0, n).tobytes()
    return text, b"".join(_bgzf_member(text[i:i + 65280]) for i in range(0, len(text), 65280))


def prepare(d, nreads):
    """reads.fq and reads.fq.gz (by host workers, before this process touches the GPU), then data/ (write_data_dir)"""
    from multiprocessing import Pool
    import bench
    G = bench.workload_plan("weak", 1, 0)[0]
    jobs = [(G, r0, min(CHUNK, nreads - r0)) for r0 in range(0, nreads, CHUNK)]
    with open(os.path.join(d, "reads.fq"), "wb") as fq, open(os.path.join(d, "reads.fq.gz"), "wb") as gz, Pool(os.cpu_count()) as pool:
        for text, members in pool.imap(_chunk_job, jobs):
            fq.write(text)
            gz.write(members)
        gz.write(_bgzf_member(b""))
    write_data_dir(d)


def write_data_dir(d):
    """d/data/: bench.py's default-scale database built to a file, db_info.txt and one tiny organism file per genome"""
    import gzip
    import torch
    import bench
    import synth
    from metalign_b200.api import Context, Database
    from metalign_b200.select_db import DB_BASENAME
    G = bench.workload_plan("weak", 1, 0)[0]
    p = bench.synth_params(G, 0)
    data = os.path.join(d, "data")
    os.makedirs(os.path.join(data, "organism_files"), exist_ok=True)
    names = ["taxid_%d_genomic.fna.gz" % g for g in range(G)]
    with Context(0) as ctx:
        d_keys = torch.empty(G * p.n * 2, dtype=torch.int64, device="cuda")
        assert synth.cuda_lib().syn_cuda_gen_sketch_keys(C.byref(p), d_keys.data_ptr(), None) == 0
        db = Database.from_device_keys(ctx, d_keys.data_ptr(), G, p.n, bench.K, bench.KS, names=names)
        del d_keys
        db.save(os.path.join(data, DB_BASENAME))
        db.close()
    with open(os.path.join(data, "db_info.txt"), "w") as f:
        f.write("Accession\tLength\tTaxID\tLineage\tTaxID_Lineage\n")
        for g in range(G):
            f.write("acc%d\t1000\t%d\t|||||||s%d\t1|2|3|4|5|6|%d|%d\n" % (g, g, g, g // 5, g))
    blob = gzip.compress(b">g\nACGT\n")
    for name in names:
        with open(os.path.join(data, "organism_files", name), "wb") as f:
            f.write(blob)


def _read_through(path):
    t0 = time.perf_counter()
    with open(path, "rb", buffering=0) as f:
        while f.read(1 << 26):
            pass
    return time.perf_counter() - t0


def gpu_identity():
    from bench_read_kmers import gpu_identity as ident
    return ident()


def run(d, fmt, threads):
    """one select_db.py run under torchrun; rank 0 prints the JSON line"""
    from metalign_b200 import select_db
    reads = os.path.join(d, "reads.fq" if fmt == "fq" else "reads.fq.gz")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    out = os.path.join(d, "out_%s_%d" % (fmt, world))
    args = select_db.select_parseargs([reads, os.path.join(d, "data"), "--temp_dir", out, "--threads", str(threads)])
    times = {}
    t0 = time.perf_counter()
    select_db.select_main(args, stages=times)
    wall = time.perf_counter() - t0
    rank, world = select_db.ranks()
    all_times = [times]
    if world > 1:
        import torch.distributed as tdist
        all_times = [None] * world
        tdist.all_gather_object(all_times, times)
        walls = [None] * world
        tdist.all_gather_object(walls, wall)
        wall = max(walls)
        tdist.destroy_process_group()
    if rank != 0:
        return
    stage = {k: max(t.get(k, 0.0) for t in all_times) for k in ("open_s", "push_s", "exchange_s", "finish_s")}
    text = os.path.getsize(os.path.join(d, "reads.fq"))
    name, power = gpu_identity()
    print(json.dumps(dict(format=fmt, world=world, reads_file_bytes=os.path.getsize(reads), text_bytes=text, wall_s=round(wall, 3),
                          **{k: round(v, 3) for k, v in stage.items()}, rest_s=round(wall - sum(stage.values()), 3),
                          text_GBps=round(text / wall / 1e9, 3), push_text_GBps=round(text / max(stage["push_s"], 1e-9) / 1e9, 3),
                          threads_per_rank=threads, host_cores=os.cpu_count(), gpu=name, power_limit=power,
                          page_cache="warm (the file was read through once before the runs)")), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=40_000_000)
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--dir", default="", help="work directory (default: a temporary one, removed at the end)")
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    ap.add_argument("--run", default="", help=argparse.SUPPRESS)
    ap.add_argument("--prepare", default="", help=argparse.SUPPRESS)
    ap.add_argument("--format", default="fq", help=argparse.SUPPRESS)
    ap.add_argument("--threads", type=int, default=0, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.run:
        return run(a.run, a.format, a.threads)
    if a.prepare:
        return prepare(a.prepare, a.reads)
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu == 0:
        sys.exit("bench_select_ranks: no GPU")
    d = a.dir or tempfile.mkdtemp(prefix="mlg_bench_select_")
    try:
        t0 = time.perf_counter()
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--prepare", d, "--reads", str(a.reads)])
        sys.stderr.write("prepared in %.0f s\n" % (time.perf_counter() - t0))
        lines = []
        for fmt in ("fq", "bgzf"):
            path = os.path.join(d, "reads.fq" if fmt == "fq" else "reads.fq.gz")
            for world in [int(w) for w in a.worlds.split(",") if int(w) <= ngpu]:
                _read_through(path)
                cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(world),
                       os.path.abspath(__file__), "--run", d, "--format", fmt, "--threads", str(max(1, os.cpu_count() // world))]
                res = subprocess.run(cmd, capture_output=True, text=True)
                if res.returncode:
                    sys.stderr.write(res.stdout[-4000:] + res.stderr[-4000:])
                    raise SystemExit("run failed: %s %d" % (fmt, world))
                line = json.loads([x for x in res.stdout.splitlines() if x.startswith("{")][-1])
                line["csv_equals_one_gpu"] = filecmp.cmp(os.path.join(d, "out_%s_%d" % (fmt, world), "cmash_query_results.csv"),
                                                         os.path.join(d, "out_fq_1", "cmash_query_results.csv"), shallow=False)
                print(json.dumps(line), flush=True)
                lines.append(line)
        if a.out:
            with open(a.out, "a") as f:
                f.writelines(json.dumps(x) + "\n" for x in lines)
    finally:
        if not a.dir:
            shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
