#! /usr/bin/env python
"""Many samples against one database: S cold select_db.py processes one after the other (the loop) against one
select_many.py run over the same sample sheet (the batch), on bench.py's default-scale database (2e5 genomes x 1000 slots)
built to a file.  Sample s is FASTQ of `--reads` 150 bp reads drawn from the first 25 (s + 1) present genomes of the
synthetic workload (a different genome subset and abundance mix per sample).  Every reads file is read through once
before the arms (warm page cache); both arms use --threads (default: the host's cores per GPU).  The arms alternate
`--reps` times.

Each rep checks that every sample's cmash_query_results.csv and subset_db_info.txt are equal between the arms, and
prints one JSON line: GPU name and power limit, host cores, S, reads per sample, seconds of both arms, samples per minute,
and the batch's stages summed over samples (rank 0's database open; pushes, GPU files and subset files per sample).

    python scripts/bench_select_many.py [--samples 16] [--reads 2000000] [--gpus 1] [--reps 2] [--out results.jsonl]

With --gpus N > 1 the batch runs under torchrun, one process per GPU.  The child mode (--run-many) is what the batch arm
starts: select_many.py's work plus its stage times written to a file.
"""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
CHUNK = 500_000


def _sample_chunk(job):
    import bench
    from bench_select_ranks import _fastq_chunk
    G, s, r0, n = job
    p = bench.synth_params(G, 0)
    p.n_present = 25 * (s + 1)
    return _fastq_chunk(p, r0, n).tobytes()


def prepare(d, samples, nreads):
    """the FASTQ samples and the sheet (host workers, before this process touches the GPU), then data/"""
    from multiprocessing import Pool
    import bench
    from bench_select_ranks import write_data_dir
    G = bench.workload_plan("weak", 1, 0)[0]
    with open(os.path.join(d, "samples.tsv"), "w") as sheet, Pool(os.cpu_count()) as pool:
        for s in range(samples):
            path = os.path.join(d, "sample%02d.fq" % s)
            jobs = [(G, s, r0, min(CHUNK, nreads - r0)) for r0 in range(0, nreads, CHUNK)]
            with open(path, "wb") as f:
                for text in pool.imap(_sample_chunk, jobs):
                    f.write(text)
            sheet.write("sample%02d\t%s\n" % (s, path))
    write_data_dir(d)


def run_many(d, out, threads, stages_path):
    """select_many.py's work; rank 0 writes the stage times (the results of every rank are gathered)"""
    from metalign_b200 import select_db
    sheet = os.path.join(d, "samples.tsv")
    args = select_db.select_many_parseargs([sheet, os.path.join(d, "data"), "--out_dir", out, "--threads", str(threads)])
    st = {"open_s": 0.0}
    results = select_db.select_many(sheet, args, stages=st)
    rank, world = select_db.ranks()
    if rank == 0:
        for k in ("push_s", "gpu_files_s", "subset_s"):
            st[k] = sum(r.stages.get(k, 0.0) for r in results)
        st["failed"] = [r.id for r in results if r.status != "ok"]
        with open(stages_path, "w") as f:
            json.dump(st, f)
    if world > 1:
        import torch.distributed as tdist
        tdist.destroy_process_group()
    sys.exit(1 if any(r.status != "ok" for r in results) else 0)


def _read_through(path):
    with open(path, "rb", buffering=0) as f:
        while f.read(1 << 26):
            pass


def _timed(cmd):
    t0 = time.perf_counter()
    res = subprocess.run(cmd, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    if res.returncode:
        sys.stderr.write(res.stdout[-4000:] + res.stderr[-4000:])
        raise SystemExit("failed: %s" % " ".join(cmd))
    return dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=16)
    ap.add_argument("--reads", type=int, default=2_000_000)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--threads", type=int, default=0, help="reader threads of both arms (default: host cores // gpus)")
    ap.add_argument("--dir", default="", help="work directory (default: a temporary one, removed at the end)")
    ap.add_argument("--out", default="", help="also append the JSON lines to this file")
    ap.add_argument("--run-many", default="", help=argparse.SUPPRESS)
    ap.add_argument("--prepare", default="", help=argparse.SUPPRESS)
    ap.add_argument("--out-dir", default="", help=argparse.SUPPRESS)
    ap.add_argument("--stages", default="", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.run_many:
        return run_many(a.run_many, a.out_dir, a.threads, a.stages)
    if a.prepare:
        return prepare(a.prepare, a.samples, a.reads)
    import torch
    if torch.cuda.device_count() < a.gpus or a.gpus < 1:
        sys.exit("bench_select_many: needs %d GPU(s)" % a.gpus)
    from bench_select_ranks import gpu_identity
    threads = a.threads or max(1, os.cpu_count() // a.gpus)
    d = a.dir or tempfile.mkdtemp(prefix="mlg_bench_many_")
    try:
        t0 = time.perf_counter()
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--prepare", d, "--samples", str(a.samples),
                               "--reads", str(a.reads)])
        sys.stderr.write("prepared in %.0f s\n" % (time.perf_counter() - t0))
        ids = ["sample%02d" % s for s in range(a.samples)]
        for sid in ids:
            _read_through(os.path.join(d, sid + ".fq"))
        name, power = gpu_identity()
        lines = []
        for rep in range(a.reps):
            loop_dir, batch_dir = os.path.join(d, "loop%d" % rep), os.path.join(d, "batch%d" % rep)
            loop_s = 0.0
            for sid in ids:
                loop_s += _timed([sys.executable, os.path.join(ROOT, "scripts", "select_db.py"), os.path.join(d, sid + ".fq"),
                                  os.path.join(d, "data"), "--temp_dir", os.path.join(loop_dir, sid), "--threads", str(threads)])
            stages_path = os.path.join(d, "stages%d.json" % rep)
            child = [os.path.abspath(__file__), "--run-many", d, "--out-dir", batch_dir, "--threads", str(threads),
                     "--stages", stages_path]
            if a.gpus > 1:
                cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(a.gpus)] + child
            else:
                cmd = [sys.executable] + child
            batch_s = _timed(cmd)
            with open(stages_path) as f:
                stages = json.load(f)
            equal = all(filecmp.cmp(os.path.join(loop_dir, sid, fn), os.path.join(batch_dir, sid, fn), shallow=False)
                        for sid in ids for fn in ("cmash_query_results.csv", "subset_db_info.txt"))
            line = dict(rep=rep, gpu=name, power_limit=power, host_cores=os.cpu_count(), gpus=a.gpus, threads=threads,
                        samples=a.samples, reads_per_sample=a.reads, loop_s=round(loop_s, 3), batch_s=round(batch_s, 3),
                        loop_samples_per_min=round(60 * a.samples / loop_s, 2),
                        batch_samples_per_min=round(60 * a.samples / batch_s, 2), speedup=round(loop_s / batch_s, 3),
                        batch_stages={k: (round(v, 3) if isinstance(v, float) else v) for k, v in stages.items()},
                        files_equal=equal, page_cache="warm (every reads file read through once before the arms)")
            print(json.dumps(line), flush=True)
            lines.append(line)
            shutil.rmtree(loop_dir, ignore_errors=True)
            shutil.rmtree(batch_dir, ignore_errors=True)
            if not equal:
                raise SystemExit("bench_select_many: the arms' files differ")
        if a.out:
            with open(a.out, "a") as f:
                f.writelines(json.dumps(x) + "\n" for x in lines)
    finally:
        if not a.dir:
            shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
