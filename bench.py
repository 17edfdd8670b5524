#!/usr/bin/env python
"""bench.py -- the reference's headline metric on B200: read k-mers/s (and Gbases/s) queried against the
CMash-style sketch database, plus the probe kernel's fraction of the HBM roofline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload weak|strong|stream|stress]
                  [--dump-outputs DIR]

A "step" is one whole pass of the hot path over one batch of synthetic reads: canonical 60-mer counting
against the database (K1), intersection, multi-k prefix expansion (K2), per-genome tables (K3), and -- with
more than one GPU -- the single all-reduce of the counter table.  Workload at N=1 = BASELINE.json configs[1]:
10M x 150 bp reads simulated from database genomes, full default-scale database (2e5 genomes x 1000 slots),
k range 30-60-10.  N>1 (default workload): weak scaling, 10M reads per GPU, database replicated.  The other
BASELINE.json configs are --workload strong (configs[2]: 100M reads sharded), stream (configs[3]: 500M reads, every GPU
streaming its share from pinned host memory in 10M-read batches through one query) and stress (configs[4]: 10x database).

After the timed region rank 0 runs the CPU oracle over ALL reads of the job and compares its per-genome tables and
intersection size with the GPU's (`parity_checked`; skipped above 100M reads / 2e5 genomes unless MLG_BENCH_PARITY=1).

--dump-outputs DIR writes what the last timed step of the native arm handed its caller as DIR/<name>.npy (float64), so that
two builds run with the same arguments (the inputs are seeded) can be compared output for output: see dump_outputs().

Environment overrides (for quick runs): MLG_BENCH_G, MLG_BENCH_READS (per GPU), MLG_BENCH_TOTAL_READS,
MLG_BENCH_BATCH_READS, MLG_BENCH_CPU_READS, MLG_BENCH_SKIP_CPU=1, MLG_BENCH_PARITY=0|1, MLG_EXCHANGE=sparse|dense|p2p.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

KS = (30, 40, 50, 60)
K = 60
READ_LEN = 150
SEED = 20200529


def env_int(name, default):
    v = os.environ.get(name)
    return int(float(v)) if v else default


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled through NVML every few ms by a thread, DURING the
    timed region only (start() / stop() bracket it)."""
    BAD = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
           ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, index, period_s=0.004):
        self.index, self.period = index, period_s
        self.sm, self.reasons, self.stop_flag, self.thread, self.err = [], set(), False, None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a list of indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                try:
                    phys = int(vis.split(",")[index])
                except (ValueError, IndexError):
                    phys = index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.nv, self.err = None, str(e)

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for name, attr in self.BAD:
                    if r & getattr(nv, attr):
                        self.reasons.add(name)
            except Exception as e:  # noqa: BLE001
                self.err = str(e)
                return
            time.sleep(self.period)

    def start(self):
        if self.nv:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if not self.nv or not self.thread:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no samples: %s" % self.err]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "sm_mhz_min": float(min(self.sm))}


def measured_traffic():
    """DRAM bytes per k-mer of the probe kernel from the committed `ncu --set full` capture (profiles/k1_traffic.json,
    written by scripts/ncu_summary.py): dram__bytes_read.sum + dram__bytes_write.sum over the k-mers of that launch."""
    try:
        with open(os.path.join(ROOT, "profiles", "k1_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def measured_request_ceiling():
    """What this part sustains in independent random 4-byte reads of a 1 GiB table (scripts/ubench/gather.cu, measured on
    the same pool: profiles/r3a_ubench_gather_rates.jsonl), for the load flavour K1 uses (ld.global.nc .L2::64B)."""
    try:
        best = None
        with open(os.path.join(ROOT, "profiles", "r3a_ubench_gather_rates.jsonl")) as f:
            for ln in f:
                d = json.loads(ln)
                if "L2::64B" in d.get("variant", ""):
                    best = float(d["G_loads_per_s"])
        return best
    except Exception:
        return None


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float64 (counts and genome indices are exact there).  When the arrays exceed
    DUMP_BYTES (the dense tables of a large database), those with one row per row of "ci" keep a seeded sample of their
    rows, the same rows in every run, whose indices go to sampled_rows.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        n = arrays["ci"].shape[0]
        keep = np.sort(np.random.default_rng(SEED).choice(n, n * DUMP_BYTES // (2 * total), replace=False))
        arrays = {k: (a[keep] if a.shape[0] == n else a) for k, a in arrays.items()}
        arrays["sampled_rows"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def synth_params(G, paired):
    import synth
    return synth.params(G=G, n=1000, K=K, seed=SEED, n_present=500, read_len=READ_LEN, paired=paired)


# BASELINE.json configs -> what one step processes.  total == 0: `per_gpu` reads on every rank (weak scaling).
WORKLOADS = {
    "weak":   dict(config=1, G=200_000,   per_gpu=10_000_000, total=0,           paired_multi=1, scaling="weak"),
    "strong": dict(config=2, G=200_000,   per_gpu=0,          total=100_000_000, paired_multi=1, scaling="strong"),
    "stream": dict(config=3, G=200_000,   per_gpu=0,          total=500_000_000, paired_multi=0, scaling="strong"),
    "stress": dict(config=4, G=2_000_000, per_gpu=0,          total=100_000_000, paired_multi=0, scaling="strong"),
}
BATCH_READS = 10_000_000        # reads per push: a longer share is streamed batch by batch through one query


def workload_plan(name, world, rank):
    """(G, paired, [(first read, reads)...] of this rank, total reads of the job, description)"""
    w = WORKLOADS[name]
    G = env_int("MLG_BENCH_G", w["G"])
    if w["total"]:
        total = env_int("MLG_BENCH_TOTAL_READS", w["total"])
        base, rem = divmod(total, world)
        r0 = rank * base + min(rank, rem)
        mine = base + (1 if rank < rem else 0)
    else:
        mine = env_int("MLG_BENCH_READS", w["per_gpu"])
        total, r0 = mine * world, rank * mine
    batch = env_int("MLG_BENCH_BATCH_READS", BATCH_READS)
    batches = [(r0 + o, min(batch, mine - o)) for o in range(0, mine, batch)]
    paired = w["paired_multi"] if (world > 1 or name != "weak") else 0
    cfg = w["config"] if not (name == "weak" and world > 1) else 2
    what = {"weak": "%dM reads per GPU" % (mine // 1_000_000),
            "strong": "%dM reads in all, sharded over the GPUs" % (total // 1_000_000),
            "stream": "%dM reads in all, sharded, each GPU streaming its share from pinned host memory in batches of %dM" % (total // 1_000_000, batch // 1_000_000),
            "stress": "%dM reads in all, sharded, against the 10x database" % (total // 1_000_000)}[name]
    desc = ("configs[%d]%s: synthetic %dbp %sreads simulated from database genomes (%s) vs %d genomes x 1000 sketch slots, k=30-60-10, ci_min=2, gate=exact"
            % (cfg, " shape, weak-scaled" if (name == "weak" and world > 1) else "", READ_LEN, "paired " if paired else "", what, G))
    return G, paired, batches, total, desc


# ------------------------------------------------------------------------------------------ CPU legs (the oracle)
def all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs are rank 0's alone and take every core"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(n)
    return n


def oracle_pass(p, keys, batches, repeats=1, want_tables=False):
    """The CPU restatement of the reference path (oracle/oracle.c) on the host cores: R1 counting of the given read
    batches + R3-R5, `repeats` times.  Database build (the analogue of CMash loading its HDF5/trie) is not timed,
    neither is generating the synthetic reads."""
    import synth
    from oracle.oracle_c import OracleDB, OracleQuery, lib as olib
    olib().orc_set_threads(all_host_threads())
    cores = olib().orc_max_threads()
    t0 = time.perf_counter()
    db = OracleDB(keys, p.G, p.n, K, KS)
    t_build = time.perf_counter() - t0
    times, res = [], None
    for _ in range(repeats):
        q = OracleQuery(db)
        t = 0.0
        for r0, n in batches:
            bases, nmask = synth.reads_packed(p, r0, n)
            t0 = time.perf_counter()
            q.push_packed(bases, nmask, None, n, p.read_len)
            t += time.perf_counter() - t0
            del bases, nmask
        t0 = time.perf_counter()
        res = q.finish()
        t += time.perf_counter() - t0
        times.append(t)
        q.close()
    db.close()
    out = dict(times=times, n_kmers=res["n_kmers"], cores=cores, build_s=t_build, n_intersect=res["n_intersect"])
    if want_tables:
        out.update(num=res["num"], den=res["den"], ci=res["ci"])
    return out


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path -- here its restatement oracle/oracle.c, since
    KMC and CMash are absent -- on every host core, one batch of the native arm's workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import synth
    world = int(os.environ.get("WORLD_SIZE", "1"))
    G, paired, batches, total, desc = workload_plan(args.workload, world, 0)
    sample = min(env_int("MLG_BENCH_CPU_READS", BATCH_READS), batches[0][1])
    p = synth_params(G, paired)
    all_host_threads()
    keys = synth.sketch_keys(p)
    r = oracle_pass(p, keys, [(0, sample)], repeats=args.warmup + args.steps)
    times = r["times"][args.warmup:]
    sec = float(np.mean(times))
    val = r["n_kmers"] / sec
    line = {
        "impl": "reference", "metric": "read k-mers/sec queried vs CMash DB", "value": val, "unit": "k-mers/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": WORKLOADS[args.workload]["scaling"], "vs_baseline": None, "dtype": "u128", "data": "synthetic",
        "gbases_per_s": sample * READ_LEN / sec / 1e9,
        "config": {"workload": desc, "genomes": G, "reads_per_step": sample, "read_len": READ_LEN},
        "cpu_baseline": {"value": val, "unit": "k-mers/s", "cores": r["cores"], "kind": "port",
                         "sample": "%d reads of the workload per step (one GPU's batch), every host core; CPU restatement of the reference "
                                   "path (oracle/oracle.c), not KMC/CMash binaries (absent); database build %.1f s not timed" % (sample, r["build_s"])},
        "e2e": {"value": val, "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ native arm
def run_native(args):
    import torch
    import synth
    from metalign_b200.api import Context, Database
    from metalign_b200 import codec
    from metalign_b200 import dist as mdist

    # rank 0 prints ONE JSON line on stdout: whatever NCCL has to say (its version banner, with NCCL_DEBUG set) goes to stderr.
    # The banner is written to file descriptor 1 by the library itself, so the descriptor is pointed at stderr until the line is due.
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = mdist.init_from_env("nccl")
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    import torch.distributed as tdist
    numa = mdist.bind_to_gpu_numa(local) if not os.environ.get("MLG_BENCH_NO_NUMA_BIND") else {"disabled": True}
    xmode = mdist.exchange_mode()

    G, paired, batches, total_reads, desc = workload_plan(args.workload, world, rank)
    reads_rank = sum(n for _, n in batches)
    p = synth_params(G, paired)
    ctx = Context(local)
    comp_stream = torch.cuda.ExternalStream(ctx.streams()[0], device=local)
    skip_cpu = bool(os.environ.get("MLG_BENCH_SKIP_CPU"))
    # the oracle check of the whole job's table runs on rank 0 where it takes about a minute; beyond that
    # (configs[3]: 500 M reads, configs[4]: 2e6 genomes) only on request (MLG_BENCH_PARITY=1)
    want_parity = (not skip_cpu) and (os.environ.get("MLG_BENCH_PARITY", "") == "1" or
                                      (os.environ.get("MLG_BENCH_PARITY", "") != "0" and total_reads <= 100_000_000 and G <= 200_000))

    # database: generated on the device, built on the device
    t0 = time.perf_counter()
    keys_host = None
    need_host_keys = rank == 0 and not skip_cpu and (world == 1 or want_parity)
    if G * p.n <= 400_000_000 or need_host_keys:
        d_keys = torch.empty(G * p.n * 2, dtype=torch.int64, device="cuda")
        assert synth.cuda_lib().syn_cuda_gen_sketch_keys(C.byref(p), d_keys.data_ptr(), None) == 0
        if need_host_keys:
            keys_host = d_keys.cpu().numpy().view(np.uint64).reshape(-1, 2)
            t0 = time.perf_counter()
        db = Database.from_device_keys(ctx, d_keys.data_ptr(), G, p.n, K, KS)
        del d_keys
    else:
        # the 10x database (2e9 slots, 32 GB of keys): generated and handed to the builder 1e5 genomes at a time
        step = 100_000
        d_chunk = torch.empty(step * p.n * 2, dtype=torch.int64, device="cuda")

        def chunks():
            for g0 in range(0, G, step):
                c = min(step, G - g0)
                assert synth.cuda_lib().syn_cuda_gen_sketch_keys_range(C.byref(p), g0, c, d_chunk.data_ptr(), None) == 0
                yield d_chunk.data_ptr(), g0, c
        db = Database.from_device_chunks(ctx, chunks(), G, p.n, K, KS)
        del d_chunk
    torch.cuda.synchronize()
    t_db = time.perf_counter() - t0
    torch.cuda.empty_cache()

    # this rank's reads, batch by batch: generated on the device; a pinned host copy for the end-to-end leg, which hands
    # N over as (start, length) runs, the compact form of the mask (mlg_query_push_packed_nruns): 0.1 % of the bases are
    # N, so the mask would be a third of the PCIe bytes.  The runs are what the native FASTQ reader (csrc/ingest.cpp)
    # emits; here they are derived from the generator's mask before the timed region.
    dev, host = [], []
    for r0, n in batches:
        nbb, nmb = synth.packed_sizes(n, READ_LEN)
        d_b = torch.empty(nbb, dtype=torch.uint8, device="cuda")
        d_m = torch.empty(nmb, dtype=torch.uint8, device="cuda")
        assert synth.cuda_lib().syn_cuda_gen_reads_packed(C.byref(p), r0, n, d_b.data_ptr(), d_m.data_ptr(), None) == 0
        h_b = torch.empty(nbb, dtype=torch.uint8, pin_memory=True)
        h_b.copy_(d_b)
        h_m = d_m.cpu()
        runs_np = codec.nmask_to_runs(h_m.numpy(), n * READ_LEN)
        h_r = torch.empty(max(1, runs_np.size), dtype=torch.int32, pin_memory=True)
        h_r[:runs_np.size].copy_(torch.from_numpy(runs_np.reshape(-1).view(np.int32)))
        h_mp = None
        if os.environ.get("MLG_BENCH_E2E_MASK"):
            h_mp = torch.empty(nmb, dtype=torch.uint8, pin_memory=True)
            h_mp.copy_(h_m)
        dev.append((d_b, d_m, n))
        host.append((h_b, h_r, runs_np.shape[0], h_mp, n))
    in_bytes = sum(int(b.numel()) + int(m.numel()) for b, m, _ in dev)
    nk = len(KS)
    h_num = torch.empty(G * nk, dtype=torch.int64, pin_memory=True)
    h_den = torch.empty(G * nk, dtype=torch.int64, pin_memory=True)
    h_ci = torch.empty(G * nk, dtype=torch.float64, pin_memory=True)
    ROW_CAP = min(G, 1 << 16)
    h_rows_g = torch.empty(ROW_CAP, dtype=torch.int32, pin_memory=True)
    h_rows_ci = torch.empty(ROW_CAP * nk, dtype=torch.float64, pin_memory=True)
    rows = [0]
    torch.cuda.synchronize()

    def step(host_leg: bool, readback_all: bool = False):
        q = db.query(2, "exact", True)
        if host_leg:
            for h_b, h_r, n_runs, h_mp, n in host:
                if h_mp is not None:
                    q.push_packed_ptr(h_b.data_ptr(), h_mp.data_ptr(), None, n, READ_LEN, device=False)
                else:
                    q.push_packed_nruns_ptr(h_b.data_ptr(), h_r.data_ptr() if n_runs else None, n_runs, None, n, READ_LEN)
        else:
            for d_b, d_m, n in dev:
                q.push_packed_ptr(d_b.data_ptr(), d_m.data_ptr(), None, n, READ_LEN, device=True)
        if world > 1:
            mdist.reduce_query(q, local, mode=xmode)
        # the step's result = the containment table (what select_db.py consumes); the integer numerators and the
        # (static) denominators stay on the device unless asked for
        if readback_all or os.environ.get("MLG_BENCH_READBACK_ALL"):
            ni = q.finish_into(h_num.data_ptr(), h_den.data_ptr(), h_ci.data_ptr())
        elif os.environ.get("MLG_BENCH_DENSE_RESULT"):
            ni = q.finish_into(None, None, h_ci.data_ptr())
        else:
            # rows of the genomes with a hit (mlg_query_finish_sparse): everything CMash's CSV can hold, a few KB instead
            # of the 6.4 MB dense table
            ni, rows[0] = q.finish_sparse_into(h_rows_g.data_ptr(), None, None, h_rows_ci.data_ptr(), ROW_CAP)
        st = q.stats()
        q.close()
        return ni, st

    def step_outputs(ni):
        """copies of what the last step handed its caller: the dense tables, or the rows of the genomes with a hit sorted
        by genome (the library returns them in no particular order); and |I|"""
        if os.environ.get("MLG_BENCH_READBACK_ALL") or os.environ.get("MLG_BENCH_DENSE_RESULT"):
            out = {"ci": h_ci.numpy().reshape(G, nk)}
            if os.environ.get("MLG_BENCH_READBACK_ALL"):
                out.update(num=h_num.numpy().reshape(G, nk), den=h_den.numpy().reshape(G, nk))
        else:
            g = h_rows_g.numpy()[:rows[0]]
            order = np.argsort(g, kind="stable")
            out = {"genomes": g[order], "ci": h_rows_ci.numpy()[:rows[0] * nk].reshape(-1, nk)[order]}
        out["n_intersect"] = np.array([ni])
        return {k: np.array(v, dtype=np.float64) for k, v in out.items()}

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    def timed(host_leg: bool, steps: int, warmup: int, sampler=None):
        for _ in range(warmup):
            step(host_leg)
        barrier()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(comp_stream)
        t0 = time.perf_counter()
        stats = []
        for _ in range(steps):
            ni, st = step(host_leg)
            stats.append(st)
        e1.record(comp_stream)
        barrier()
        wall = time.perf_counter() - t0
        clocks = sampler.stop() if sampler else None
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, wall, stats, ni, clocks

    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev, wall_dev, st_dev, ni, clocks = timed(False, args.steps, args.warmup, sampler)
    outputs = step_outputs(ni) if args.dump_outputs and rank == 0 else None
    ms_e2e, wall_e2e, st_e2e, ni2, _ = timed(True, args.steps, args.warmup)
    assert ni == ni2
    ni3, _ = step(False, readback_all=True)          # untimed: the integer tables for the oracle check below
    assert ni3 == ni

    kmers_rank = st_dev[-1]["n_kmers"]
    ni_same = True
    if world > 1:
        t = torch.tensor([kmers_rank], dtype=torch.int64, device="cuda")
        tdist.all_reduce(t)
        kmers_total = int(t.item())
        t = torch.tensor([ni, -ni], dtype=torch.int64, device="cuda")
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        ni_same = int(t[0].item()) == -int(t[1].item())        # every rank derived the same intersection size
    else:
        kmers_total = kmers_rank
    bases_total = total_reads * READ_LEN
    sec_step = ms_dev / 1e3 / args.steps
    sec_step_e2e = ms_e2e / 1e3 / args.steps
    value = kmers_total / sec_step
    e2e_value = kmers_total / sec_step_e2e

    # roofline of the dominant kernel (K1 probe), from the library's CUDA events on its compute stream
    peak, peak_src = measured_peak()
    probe_ms = float(np.mean([s["ms_probe"] for s in st_dev]))
    nbases = reads_rank * READ_LEN
    bucket_bytes = st_dev[-1]["bucket_bytes"]
    # SURVEY.md 8(d): one 32-byte sector per level-1 bucket fetch + the packed bases and N mask read once.  Layout 0
    # fetches one bucket per k-mer; the super-k-mer layouts one per run of windows sharing a minimizer, and the reduced
    # fetch count is reported next to it.
    layout = int(st_dev[-1]["layout"])
    fetches = int(st_dev[-1]["n_bucket_fetches"])
    alg_bytes = fetches * bucket_bytes + nbases // 4 + nbases // 8
    achieved = alg_bytes / (probe_ms / 1e3) / 1e9
    query_ms = float(np.mean([s["ms_query"] for s in st_dev]))
    tr = measured_traffic()
    same_db = bool(tr) and G == tr.get("genomes") and tr.get("layout", 0) == layout
    # the ncu capture counts DRAM bytes of ONE launch; it stands for this run's launches when it was taken at the same launch
    # size (k-mers per launch within 2 %), otherwise it is scaled per k-mer and says so
    kmers_launch = kmers_rank / max(1, int(st_dev[-1]["probe_launches"]))
    same_launch = same_db and abs(tr.get("kmers_in_capture", 0) / max(1.0, kmers_launch) - 1.0) < 0.02
    traffic = tr["dram_bytes_per_kmer"] * kmers_rank if same_db else None
    traffic_src = ("%s: %.2f DRAM bytes per k-mer (ncu --set full, %s, %s) x k-mers per step"
                   % (tr["source"], tr["dram_bytes_per_kmer"], tr["kernel"],
                      "captured at this launch size" if same_launch else "captured at %.3g k-mers per launch, scaled per k-mer" % tr.get("kmers_in_capture", 0))
                   if traffic is not None else "no ncu capture for this database size")
    launches = int(sum(s["gpu_launches"] for s in st_dev))

    if layout == 2 and tr and tr.get("layout") == 2:
        limiter = ("instruction issue and load latency, not HBM bandwidth: one level-1 access per ~%.0f k-mers (DRAM moves %.0f GB/s under "
                   "ncu), %.0f warp instructions per 32 k-mers at %.0f %% issue-slot utilisation (ncu, %s); see DESIGN.md section 4"
                   % (kmers_rank / max(1, fetches), tr.get("dram_gbs_under_ncu", 0), tr.get("warp_instructions_per_32_kmers", 0),
                      tr.get("issue_active_pct", 0), tr.get("source", "")))
    elif layout == 1 and tr and tr.get("layout") == 1:
        limiter = ("instruction issue, not HBM: the super-k-mer kernel fetches one bucket pair per ~17 k-mers, so DRAM runs at "
                   "%.0f GB/s while the SMs issue %.0f warp instructions per 32 k-mers at %.0f %% issue-slot utilisation with %.0f %% "
                   "of the warp slots occupied (ncu, %s); frac is low by construction, see DESIGN.md section 4"
                   % (tr.get("dram_gbs_under_ncu", 0), tr.get("warp_instructions_per_32_kmers", 0), tr.get("issue_active_pct", 0),
                      tr.get("warps_active_pct", 0), tr.get("source", "")))
    else:
        limiter = "random 32-byte DRAM sectors (one per k-mer behind an L2 prefilter)" if layout == 0 else "see profiles/"
    req_ceiling = measured_request_ceiling()
    xmode_eff = mdist.effective_mode(ctx, xmode)
    line = None
    if rank == 0:
        l1_bytes = st_dev[-1]["filter_words"] * 4 if layout == 2 else st_dev[-1]["n_buckets"] * (32 if layout == 1 else bucket_bytes)
        line = {
            "metric": "read k-mers/sec queried vs CMash DB", "value": value, "unit": "k-mers/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_step * 1e3,
            "higher_is_better": True, "scaling": WORKLOADS[args.workload]["scaling"], "vs_baseline": None, "dtype": "u128", "data": "synthetic",
            "gbases_per_s": bases_total / sec_step / 1e9,
            "config": {
                "workload": desc, "workload_name": args.workload,
                "genomes": G, "sketch_slots": 1000, "reads_total": total_reads, "reads_rank0": reads_rank, "pushes_per_step": len(batches),
                "read_len": READ_LEN, "db_distinct_kmers": st_dev[-1]["n_db_distinct"], "intersect": ni,
                "result": ("dense containment table" if os.environ.get("MLG_BENCH_DENSE_RESULT") or os.environ.get("MLG_BENCH_READBACK_ALL")
                           else "containment rows of the %d genomes with a hit (mlg_query_finish_sparse)" % rows[0]),
                "parallelism": ("reads sharded x%d, DB replicated, ONE exchange per job: %s (MLG_EXCHANGE=%s)" % (world, mdist.describe_exchange(xmode_eff, world), xmode_eff)) if world > 1 else "single GPU",
                "l2_policy": "inputs (%.2f GB packed reads per GPU) and level-1 table (%.2f GB) both exceed the 126 MB L2; no flush needed" % (in_bytes / 1e9, l1_bytes / 1e9),
                "db_build_s": round(t_db, 3),
            },
            "e2e": {"value": e2e_value, "unit": "k-mers/s", "h2d_bytes_per_step": int(st_e2e[-1]["h2d_bytes"]) * world,
                    "d2h_bytes_per_step": int(st_e2e[-1]["d2h_bytes"]) * world, "ms_per_step": sec_step_e2e * 1e3,
                    "gbases_per_s": bases_total / sec_step_e2e / 1e9,
                    "n_runs": "N positions travel as (start, length) runs prepared before the timed region (the form the native FASTQ reader emits)"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": {2: "k1_minimizer_probe", 1: "k1_superkmer_probe"}.get(layout, "k1_decode_canon_probe"), "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         # the same fraction with the bytes the DRAM really moves (ncu)
                         "dram_frac_from_ncu_traffic": (traffic / (probe_ms / 1e3) / 1e9 / peak) if traffic else None,
                         "algorithmic_bytes_per_launch_set": int(alg_bytes), "kernel_ms_per_step": probe_ms, "probe_launches_per_step": int(st_dev[-1]["probe_launches"]),
                         "finish_stage_ms_per_step": query_ms, "kmers_per_s_kernel_only": kmers_rank / (probe_ms / 1e3),
                         "layout": layout, "bucket_fetches_per_step": fetches, "kmers_per_bucket_fetch": kmers_rank / max(1, fetches),
                         "algorithmic_bytes_rule": "level-1 fetches x %d B + packed bases + N mask (SURVEY.md 8d, minimizer bucketing: layout 2 = one 32-byte sector of the minimizer-identity bit array per super-k-mer, layout 1 = one 64-byte fingerprint-bucket pair per super-k-mer, layout 0 = one sector per k-mer)" % bucket_bytes,
                         "sector_per_kmer_equivalent_gbs": (kmers_rank * 32 + nbases // 4 + nbases // 8) / (probe_ms / 1e3) / 1e9,
                         "limiter": limiter,
                         # the bound this kernel actually runs into besides instruction issue: random-read REQUESTS per second
                         "request_rate": ({"achieved_g_per_s": fetches / (probe_ms / 1e3) / 1e9, "ceiling_g_per_s": req_ceiling,
                                           "frac": fetches / (probe_ms / 1e3) / 1e9 / req_ceiling,
                                           "source": "profiles/r3a_ubench_gather.md: independent random 4-byte ld.global.nc.L2::64B reads of a 1 GiB table top out at this rate on this part (DRAM then moves 64 B per read, 3.1 TB/s)"}
                                          if req_ceiling and layout == 2 else None)},
            "clocks": clocks,
            "host_numa_binding_rank0": numa,
            "wall_ms_per_step": wall_dev * 1e3 / args.steps,
            "non_probe_ms_per_step": sec_step * 1e3 - probe_ms,
            "intersect_same_on_every_rank": ni_same,
        }
    gpu_num = h_num.numpy().reshape(G, nk).copy()
    gpu_den = h_den.numpy().reshape(G, nk).copy()
    gpu_ci = h_ci.numpy().reshape(G, nk).copy()
    db.close()
    mdist.close_exchanges()
    ctx.close()
    if world > 1:
        tdist.destroy_process_group()
    if rank != 0:
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    # ---- CPU legs on rank 0, after every collective: cpu_baseline (N = 1) and the oracle check of the job's table
    line["cpu_baseline"] = None
    line["parity_checked"] = False
    if keys_host is not None:
        all_batches = [(o, min(BATCH_READS, total_reads - o)) for o in range(0, total_reads, BATCH_READS)]
        if world == 1:
            sample = min(env_int("MLG_BENCH_CPU_READS", batches[0][1]), batches[0][1])
            full = want_parity and sample == total_reads
            r = oracle_pass(p, keys_host, [(0, sample)], repeats=2, want_tables=full)
            line["cpu_baseline"] = {
                "value": r["n_kmers"] / float(np.mean(r["times"])), "unit": "k-mers/s", "cores": r["cores"], "kind": "port",
                "sample": "%d reads of the same workload, twice (%.1f s of CPU work in all); CPU restatement of the reference path "
                          "(oracle/oracle.c), not KMC/CMash binaries (absent here); its database build (%.1f s) is not timed"
                          % (sample, float(np.sum(r["times"])), r["build_s"])}
            if want_parity and not full:
                r = oracle_pass(p, keys_host, all_batches, repeats=1, want_tables=True)
        elif want_parity:
            r = oracle_pass(p, keys_host, all_batches, repeats=1, want_tables=True)
        if want_parity:
            same = {"intersect": int(r["n_intersect"]) == int(ni), "n_kmers": int(r["n_kmers"]) == int(kmers_total),
                    "num": bool(np.array_equal(r["num"], gpu_num)), "den": bool(np.array_equal(r["den"], gpu_den)),
                    "ci": bool(np.array_equal(r["ci"], gpu_ci))}
            line["parity_checked"] = all(same.values())
            line["parity"] = {"against": "oracle/oracle.c on all %d reads of the job (%d cores)" % (total_reads, r["cores"]),
                              "equal": same, "intersect": [int(ni), int(r["n_intersect"])],
                              "genomes_with_k60_hits": int((gpu_num[:, -1] > 0).sum())}
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    if want_parity and not line["parity_checked"]:
        raise SystemExit("PARITY FAILURE: the GPU table differs from the oracle's: %s" % line["parity"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=os.environ.get("MLG_BENCH_WORKLOAD", "weak"), choices=sorted(WORKLOADS),
                    help="weak: 10M reads per GPU (configs[1] at one GPU); strong: configs[2], 100M reads sharded; "
                         "stream: configs[3], 500M reads streamed in batches; stress: configs[4], 10x database")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float64, at most 64 MB; native arm)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
