"""select_main under a torchrun-style launch, on CPU: 2 and 3 processes over gloo, and one process without a group.  Stand-ins
replace the GPU objects (Context, Database.load, the query, pinned_array) and the collectives of dist that move device
memory (share_read_kmers, reduce_query, write_reads_kmc, close_exchanges); the reader (ingest.PackedBatches, with its byte
shares and FASTQ phase check), the rank orchestration, the CSV and the subset files are the real ones.

On success every rank returns the same selection, rank 0 writes the files of a one-process run, every read is pushed on
exactly one rank and every rank's query counts its read k-mers in passes.  When one rank fails (at the push, writing the
intersection dump, or opening a reads file that does not exist) every rank raises and none of the run's files is left.
In every case, one process included, the context, the database and the query are closed before select_main returns or
raises.  The device side is covered by tests/test_gpu_select_ranks.py."""
import json
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

from conftest import ROOT

CASE_DATA = os.path.join(ROOT, "tests", "golden", "select_case", "data")
NAMES = ["taxid_10239_1_genomic.fna.gz", "taxid_10239_2_genomic.fna.gz", "taxid_1280_1_genomic.fna.gz",
         "taxid_4932_1_genomic.fna.gz", "taxid_562_1_genomic.fna.gz", "taxid_562_2_genomic.fna.gz"]
CI = np.array([[0.5, 0.45, 0.41, 0.4], [0.3, 0.25, 0.21, 0.2], [0.05, 0.03, 0.02, 0.01], [0.02, 0.01, 0.006, 0.004],
               [0.9, 0.85, 0.8, 0.75], [0.93, 0.91, 0.9, 0.88]])
SELECTED = ["taxid_562_2_genomic.fna.gz", "taxid_10239_1_genomic.fna.gz", "taxid_10239_2_genomic.fna.gz",
            "taxid_1280_1_genomic.fna.gz"]
FILES = ("cmash_query_results.csv", "cmashed_db.fna", "subset_db_info.txt", "60mers_intersection_dump",
         "60mers_intersection_dump.fa", "60mers_intersection.kmc_pre", "60mers_intersection.kmc_suf", "reads_60mers.kmc_pre",
         "reads_60mers.kmc_suf")
N_READS = 3001

_STATE = {}       # in a worker: its rank, the failure of the current job, and what the stand-ins saw


def _marker(path, what):
    with open(path, "w") as f:
        f.write("%s %s\n" % (os.path.basename(path), what))


class _Closable:
    def __init__(self, kind):
        self.kind, self.closed = kind, False
        _STATE["opened"].append(self)

    def close(self):
        self.closed = True


class _Context(_Closable):
    def __init__(self, device=0):
        super().__init__("context")


class _Query(_Closable):
    def __init__(self, kw):
        super().__init__("query")
        _STATE["query_kw"].append(kw)

    def push_packed_nruns(self, bases, nruns, off, n_reads):
        if _STATE["fail"] == ("push", _STATE["rank"]):
            raise IOError("reads file truncated")
        _STATE["pushed"] += int(n_reads)

    def sync(self):
        pass

    def finish_sparse(self):
        return {"genomes": np.arange(len(NAMES), dtype=np.uint32), "ci": CI}

    def dump_intersection(self, dump, fasta):
        if _STATE["fail"] == ("dump", _STATE["rank"]):
            raise IOError("no space left for the dump")
        _marker(dump, "dump")
        _marker(fasta, "fasta")

    def write_intersection_kmc(self, prefix, counter_max):
        for ext in (".kmc_pre", ".kmc_suf"):
            _marker(prefix + ext, "max %d" % counter_max)

    def write_reads_kmc(self, prefix, min_count, counter_max):
        for ext in (".kmc_pre", ".kmc_suf"):
            _marker(prefix + ext, "min %d max %d" % (min_count, counter_max))


class _Database(_Closable):
    names, ks = NAMES, (30, 40, 50, 60)

    def __init__(self):
        super().__init__("database")

    def query(self, **kw):
        return _Query(kw)


def _install_stand_ins():
    from metalign_b200 import api
    from metalign_b200 import dist as mdist
    api.Context = _Context
    api.Database.load = staticmethod(lambda ctx, path: _Database())
    api.pinned_array = lambda nbytes: np.zeros(nbytes, dtype=np.uint8)

    def write_reads_kmc(query, prefix, min_count=2, counter_max=3, device=0, group=None):
        if _STATE["rank"] == 0:                      # the file rank 0 joins from the ranks' parts
            query.write_reads_kmc(prefix, min_count, counter_max)
        return {}
    mdist.share_read_kmers = lambda query, device=0, group=None: None
    mdist.reduce_query = lambda query, device=0, group=None, mode=None, clamp=None: None
    mdist.write_reads_kmc = write_reads_kmc
    mdist.close_exchanges = lambda: _STATE.__setitem__("close_exchanges", _STATE["close_exchanges"] + 1)


def _args(reads, out):
    """the Namespace the reference's metalign.py hands over (none of the drop-in's extra flags)"""
    import argparse
    return argparse.Namespace(reads=reads, data=CASE_DATA, cmash_results="NONE", cutoff=0.01, db="AUTO", db_dir="AUTO",
                              dbinfo_in="AUTO", dbinfo_out="AUTO", input_type="AUTO", keep_temp_files=True, strain_level=False,
                              temp_dir=out, threads=2)


def _worker(rank, world, port, root, jobs):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from metalign_b200 import dist as mdist
    from metalign_b200 import select_db
    if world > 1:
        mdist.init_from_env("gloo")
    _install_stand_ins()
    for name, reads, fail in jobs:
        _STATE.update(rank=rank, fail=fail, opened=[], query_kw=[], pushed=0, close_exchanges=0)
        out = {}
        try:
            out["chosen"] = select_db.select_main(_args(reads, os.path.join(root, "%s_w%d" % (name, world))))
            out["raised"] = None
        except Exception as e:  # noqa: BLE001
            out["raised"] = type(e).__name__
        out.update(pushed=_STATE["pushed"], passes=[kw["read_kmer_passes"] for kw in _STATE["query_kw"]],
                   opened=sorted(o.kind for o in _STATE["opened"]),
                   unclosed=sorted(o.kind for o in _STATE["opened"] if not o.closed),
                   close_exchanges=_STATE["close_exchanges"])
        with open(os.path.join(root, "%s_w%d_r%d.json" % (name, world, rank)), "w") as f:
            json.dump(out, f)
    if world > 1:
        import torch.distributed as tdist
        tdist.destroy_process_group()


@pytest.fixture(scope="module")
def run(tmp_path_factory):
    """run(world) -> {job: [the outcome of every rank]}, and the directory of the jobs' temp_dirs; one spawn per world"""
    root = tmp_path_factory.mktemp("select_ranks")
    reads = str(root / "reads.fq")
    rng = np.random.default_rng(8)
    with open(reads, "w") as f:
        for j in range(N_READS):
            seq = "".join(rng.choice(list("ACGTN"), size=int(rng.integers(60, 151))))
            f.write("@r%d\n%s\n+\n%s\n" % (j, seq, "I" * len(seq)))
    done = {}

    def get(world):
        if world not in done:
            jobs = [("ok", reads, None), ("dump", reads, ("dump", 0))]
            if world > 1:
                jobs += [("push", reads, ("push", 1)), ("missing", str(root / "missing.fq"), None)]
            mp.spawn(_worker, args=(world, 30200 + (os.getpid() % 200) * 4 + world, str(root), jobs), nprocs=world,
                     join=True)
            done[world] = {name: [json.load(open(str(root / ("%s_w%d_r%d.json" % (name, world, r))))) for r in range(world)]
                           for name, _, _ in jobs}
        return done[world], root
    return get


def _left(root, name, world):
    return sorted(os.listdir(str(root / ("%s_w%d" % (name, world)))))


@pytest.mark.parametrize("world", [2, 3])
def test_ranks_select_and_write_what_one_process_does(run, world):
    outcomes, root = run(world)
    one = run(1)[0]["ok"][0]
    assert one["raised"] is None and one["chosen"] == SELECTED and one["pushed"] == N_READS
    assert one["passes"] == [False] and one["unclosed"] == [] and one["opened"] == ["context", "database", "query"]
    ranks = outcomes["ok"]
    assert [r["raised"] for r in ranks] == [None] * world
    assert all(r["chosen"] == SELECTED for r in ranks)
    assert sum(r["pushed"] for r in ranks) == N_READS
    assert all(r["passes"] == [True] for r in ranks)
    assert all(r["unclosed"] == [] and r["opened"] == ["context", "database", "query"] for r in ranks)
    assert _left(root, "ok", world) == sorted(FILES) == _left(root, "ok", 1)
    for name in FILES:
        a, b = root / ("ok_w%d" % world) / name, root / "ok_w1" / name
        assert a.read_bytes() == b.read_bytes(), name


def _every_rank_raised(ranks, failing):
    """the failing rank raises its own error, every other rank a RuntimeError"""
    assert ranks[failing]["raised"] == "OSError", ranks
    assert all(r["raised"] == "RuntimeError" for i, r in enumerate(ranks) if i != failing), ranks


@pytest.mark.parametrize("world", [2, 3])
def test_a_rank_failing_at_the_push_fails_every_rank(run, world):
    outcomes, root = run(world)
    ranks = outcomes["push"]
    _every_rank_raised(ranks, 1)
    assert _left(root, "push", world) == []
    assert all(r["close_exchanges"] >= 1 for r in ranks)
    assert all(r["unclosed"] == [] and r["opened"] == ["context", "database", "query"] for r in ranks)


@pytest.mark.parametrize("world", [2, 3])
def test_rank0_failing_at_the_dump_fails_every_rank(run, world):
    outcomes, root = run(world)
    ranks = outcomes["dump"]
    _every_rank_raised(ranks, 0)
    assert _left(root, "dump", world) == []
    assert all(r["unclosed"] == [] and r["opened"] == ["context", "database", "query"] for r in ranks)


@pytest.mark.parametrize("world", [2, 3])
def test_a_missing_reads_file_fails_every_rank(run, world):
    outcomes, root = run(world)
    ranks = outcomes["missing"]
    assert all(r["raised"] is not None for r in ranks), ranks
    assert _left(root, "missing", world) == []
    assert all(r["unclosed"] == [] and r["opened"] == ["context", "database"] for r in ranks)


def test_one_process_closes_the_gpu_objects_when_its_files_fail(run):
    """a single run whose files fail after the pushes gives the query, the database and the context back before it
    raises (a caller looping over samples would otherwise keep GBs of device memory referenced)"""
    one = run(1)[0]["dump"][0]
    assert one["raised"] == "OSError"
    assert one["opened"] == ["context", "database", "query"] and one["unclosed"] == []
