"""select_main under a torchrun-style launch, one process per GPU: each rank reads its byte range of the reads file, the
ranks sum their counters in one exchange (clamp 3) and join reads_60mers, and rank 0 writes the files.  With
--keep_temp_files every file must be byte-identical to the reference's (expected_default / expected_fasta_gz) and to a
one-GPU run: for reads.fq, a BGZF copy of it, and reads.fa.gz (one gzip stream: rank 0 reads it all).  A reads path that
does not exist raises on every rank and leaves no file.  metalign.py --select_only writes the same files.  At 2 ranks and
at every visible GPU up to 8; skipped below two GPUs."""
import argparse
import filecmp
import os
import random
import sys

import pytest

from conftest import ROOT
from metalign_b200.select_db import OUTPUT_NAMES

pytestmark = pytest.mark.gpu
CASE = os.path.join(ROOT, "tests", "golden", "ref_e2e_case")
DATA = os.path.join(CASE, "data")


def _args(reads, out):
    return argparse.Namespace(reads=reads, data=DATA, cmash_results="NONE", cutoff=0.01, db="AUTO", db_dir="AUTO",
                              dbinfo_in="AUTO", dbinfo_out="AUTO", input_type="AUTO", keep_temp_files=True, strain_level=False,
                              temp_dir=out, threads=2)


def _worker(rank, world, port, jobs):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as tdist
    from metalign_b200 import metalign, select_db
    for kind, reads, out in jobs:
        try:
            if kind == "select":
                select_db.select_main(_args(reads, out))
            else:
                metalign.main([reads, DATA, "--select_only", "--keep_temp_files", "--temp_dir", out, "--threads", "2"])
        except Exception as e:  # noqa: BLE001
            with open(os.path.join(os.path.dirname(out.rstrip("/")), "raised_%s_%d" % (os.path.basename(out.rstrip("/")), rank)), "w") as f:
                f.write(repr(e))
    tdist.destroy_process_group()


def _same(a, b, names):
    for name in names:
        assert filecmp.cmp(os.path.join(a, name), os.path.join(b, name), shallow=False), (a, b, name)


@pytest.fixture(scope="module")
def bgzf_reads(tmp_path_factory):
    from test_ingest import _write_bgzf
    p = tmp_path_factory.mktemp("bgzf") / "reads.fq.gz"
    with open(os.path.join(CASE, "reads.fq"), "rb") as f:
        _write_bgzf(p, f.read(), random.Random(7), max_block=9000)
    return str(p)


def _worlds():
    import torch
    n = torch.cuda.device_count()
    return sorted({2, min(n, 8)}) if n >= 2 else []


def test_ranks_write_the_one_gpu_files(tmp_path, bgzf_reads):
    import torch.multiprocessing as mp
    from metalign_b200 import select_db
    worlds = _worlds()
    if not worlds:
        pytest.skip("needs two GPUs")
    inputs = {"fq": (os.path.join(CASE, "reads.fq"), "expected_default"), "bgzf": (bgzf_reads, "expected_default"),
              "fagz": (os.path.join(CASE, "reads.fa.gz"), "expected_fasta_gz")}
    for tag, (reads, _) in inputs.items():
        select_db.select_main(_args(reads, str(tmp_path / ("one_" + tag))))
    for world in worlds:
        jobs = [("select", reads, str(tmp_path / ("w%d_%s" % (world, tag)))) for tag, (reads, _) in inputs.items()]
        jobs.append(("select", str(tmp_path / "missing.fq"), str(tmp_path / ("w%d_missing" % world))))
        jobs.append(("metalign", os.path.join(CASE, "reads.fq"), str(tmp_path / ("w%d_metalign" % world))))
        os.makedirs(jobs[3][2])
        mp.spawn(_worker, args=(world, 29900 + os.getpid() % 50 + world, jobs), nprocs=world, join=True)
        for tag, (reads, exp) in inputs.items():
            out = str(tmp_path / ("w%d_%s" % (world, tag)))
            assert not [f for f in os.listdir(str(tmp_path)) if f.startswith("raised_w%d_%s_" % (world, tag))]
            _same(out, str(tmp_path / ("one_" + tag)), OUTPUT_NAMES)
            _same(out, os.path.join(CASE, exp), sorted(os.listdir(os.path.join(CASE, exp))))
        # a reads file that does not exist: every rank raises, nothing is written
        raised = [f for f in os.listdir(str(tmp_path)) if f.startswith("raised_w%d_missing_" % world)]
        assert len(raised) == world, raised
        assert os.listdir(str(tmp_path / ("w%d_missing" % world))) == []
        _same(str(tmp_path / ("w%d_metalign" % world)), str(tmp_path / "one_fq"), OUTPUT_NAMES)
