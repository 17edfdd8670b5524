"""dist.write_reads_kmc on CPU: its collective outcome logic over gloo, with a stand-in for the query that writes its
share of the key order through tests/kmcdb.py (or fails).  Every rank writes <prefix>.part<r>, rank 0 joins the parts,
and whatever happens the parts are removed; if one rank's part fails, or the join fails, every rank raises and no
database is left.  Also the single-process form (no process group).  The device side is covered by
tests/test_gpu_read_kmers_sharded.py and tests/test_gpu_multi_read_kmers.py."""
import os
import random
import sys

import pytest
import torch.multiprocessing as mp

from conftest import ROOT

K = 31


def _kmers():
    rng = random.Random(4)
    out = {}
    while len(out) < 600:
        out["".join(rng.choice("ACGT") for _ in range(K))] = rng.randint(2, 9)
    return out


def _shares(world):
    """the k-mers in key order, cut into `world` consecutive shares (one of them empty)"""
    keys = sorted(_kmers())
    cuts = [len(keys) * r // world for r in range(world + 1)]
    cuts[1] = 0 if world > 2 else cuts[1]                    # rank 0's share is empty when there are > 2 ranks
    return [{k: _kmers()[k] for k in keys[cuts[r]:cuts[r + 1]]} for r in range(world)]


class _Query:
    """what dist.write_reads_kmc calls on a query: write_reads_kmc(prefix, min_count, counter_max)"""

    def __init__(self, kmers, fail=False):
        self.kmers, self.fail = kmers, fail

    def write_reads_kmc(self, prefix, min_count, counter_max):
        import kmcdb
        from metalign_b200.api import MlgError
        if self.fail:
            raise MlgError(-5, "this rank's archive outgrew its budget")
        kmcdb.write(prefix, self.kmers, K, min_count=min_count, max_count=counter_max)


def _worker(rank, world, port, out_dir, mode):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as tdist
    from metalign_b200 import dist as mdist
    mdist.init_from_env("gloo")
    shares = _shares(world)
    if mode == "overlap" and rank == world - 1:              # the last share repeats a key of the one before: the join fails
        shares[rank][sorted(shares[rank - 1])[-1]] = 2
    q = _Query(shares[rank], fail=(mode == "part_fails" and rank == 1))
    try:
        mdist.write_reads_kmc(q, os.path.join(out_dir, "reads"), 2, 3)
        outcome = "ok"
    except Exception as e:  # noqa: BLE001
        outcome = type(e).__name__
    with open(os.path.join(out_dir, "outcome_%d" % rank), "w") as f:
        f.write(outcome)
    tdist.destroy_process_group()


def _outcomes(tmp_path, world):
    return [open(str(tmp_path / ("outcome_%d" % r))).read() for r in range(world)]


def _left(tmp_path):
    return sorted(p.name for p in tmp_path.iterdir() if p.name.startswith("reads"))


@pytest.mark.parametrize("mode,world", [("ok", 2), ("ok", 3), ("part_fails", 3), ("overlap", 2)])
def test_ranks_agree_and_leave_no_part(tmp_path, mode, world):
    import kmcdb
    port = 29900 + (os.getpid() % 50) * 4 + ["ok", "part_fails", "overlap"].index(mode) + world
    mp.spawn(_worker, args=(world, port, str(tmp_path), mode), nprocs=world, join=True)
    out = _outcomes(tmp_path, world)
    if mode == "ok":
        assert out == ["ok"] * world
        assert _left(tmp_path) == ["reads.kmc_pre", "reads.kmc_suf"]
        kmcdb.write(str(tmp_path / "whole"), _kmers(), K, min_count=2, max_count=3)
        for ext in (".kmc_pre", ".kmc_suf"):
            assert (tmp_path / ("reads" + ext)).read_bytes() == (tmp_path / ("whole" + ext)).read_bytes()
        return
    # every rank raises: the failing rank (or rank 0, whose join failed) its own error, the others a RuntimeError
    failing = 1 if mode == "part_fails" else 0
    assert out[failing] == "MlgError" and all(o == "RuntimeError" for r, o in enumerate(out) if r != failing), out
    assert _left(tmp_path) == []


def test_single_process(tmp_path):
    import kmcdb
    from metalign_b200 import dist as mdist
    from metalign_b200.api import MlgError
    times = mdist.write_reads_kmc(_Query(_kmers()), str(tmp_path / "reads"), 2, 3)
    assert set(times) == {"part_s", "concat_s"}
    kmcdb.write(str(tmp_path / "whole"), _kmers(), K, min_count=2, max_count=3)
    for ext in (".kmc_pre", ".kmc_suf"):
        assert (tmp_path / ("reads" + ext)).read_bytes() == (tmp_path / ("whole" + ext)).read_bytes()
    assert not (tmp_path / "reads.part0.kmc_pre").exists() and not (tmp_path / "reads.part0.kmc_suf").exists()
    with pytest.raises(MlgError):
        mdist.write_reads_kmc(_Query({}, fail=True), str(tmp_path / "failed"), 2, 3)
    assert not any(p.name.startswith("failed") for p in tmp_path.iterdir())
