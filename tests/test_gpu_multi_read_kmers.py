"""Two or more real GPUs, one process each: the reads sharded over the ranks, dist.share_read_kmers (the archives over
NCCL), the counter exchange (dist.reduce_query) and dist.write_reads_kmc.  Rank 0's reads_60mers must be byte-identical to
the file of one passes-mode query over all the reads, and its records must equal the C oracle's.  Even shards, and
uneven ones (rank 0 holds 80 % of the reads).  Skipped when fewer than two GPUs are visible."""
import filecmp
import os
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
NREADS = 60_000


def _params():
    import synth
    return synth.params(G=200, n=200, seed=29, len_min=20000, len_max=60000, n_present=40)


def _range(rank, world, uneven):
    from metalign_b200 import dist as mdist
    if not uneven:
        return mdist.shard_range(NREADS, rank, world)
    big = NREADS * 4 // 5
    if rank == 0:
        return 0, big
    a, b = mdist.shard_range(NREADS - big, rank - 1, world - 1)
    return big + a, big + b


def _worker(rank, world, port, out_dir, uneven):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as tdist
    import synth
    from metalign_b200 import dist as mdist
    from metalign_b200.api import Context, Database
    r, w, local = mdist.init_from_env("nccl")
    p = _params()
    keys = synth.sketch_keys(p)
    a, b = _range(rank, world, uneven)
    bases, nmask = synth.reads_packed(p, a, b - a)
    ctx = Context(local)
    db = Database.from_keys(ctx, keys, p.G, p.n, 60)
    q = db.query(read_kmers=True, read_kmer_passes=True)
    q.push_packed(bases, nmask, None, b - a, p.read_len)
    mdist.share_read_kmers(q, local)
    mdist.reduce_query(q, local, mode="sparse")
    q.finish()
    mdist.write_reads_kmc(q, os.path.join(out_dir, "reads_60mers"), 2, 3, local)
    np.save(os.path.join(out_dir, "plan_%d.npy" % rank), np.array([q.read_kmer_plan()["share_first_bin"],
                                                                   q.read_kmer_plan()["share_end_bin"]]))
    q.close()
    db.close()
    mdist.close_exchanges()
    ctx.close()
    tdist.destroy_process_group()


@pytest.mark.parametrize("uneven", [False, True])
def test_ranks_write_the_single_query_file(tmp_path, uneven):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import synth
    from metalign_b200 import ingest
    from metalign_b200.api import Context, Database
    from oracle.read_kmers import OracleReadKmers
    world = min(torch.cuda.device_count(), 4)
    mp.spawn(_worker, args=(world, 29700 + os.getpid() % 200 + 3 * int(uneven), str(tmp_path), uneven), nprocs=world, join=True)
    p = _params()
    bases, nmask = synth.reads_packed(p, 0, NREADS)
    with Context(0) as ctx:
        db = Database.from_keys(ctx, synth.sketch_keys(p), p.G, p.n, 60)
        q = db.query(read_kmers=True, read_kmer_passes=True)
        q.push_packed(bases, nmask, None, NREADS, p.read_len)
        q.write_reads_kmc(str(tmp_path / "single"), 2, 3)
        q.close()
        db.close()
    for ext in (".kmc_pre", ".kmc_suf"):
        assert filecmp.cmp(str(tmp_path / ("reads_60mers" + ext)), str(tmp_path / ("single" + ext)), shallow=False), ext
        for r in range(world):
            assert not (tmp_path / ("reads_60mers.part%d%s" % (r, ext))).exists()
    o = OracleReadKmers(60)
    o.push_packed(bases, nmask, None, NREADS, p.read_len)
    wk, wc = o.result(2, 3)
    o.close()
    fk, _, fc = ingest.read_kmc_database(str(tmp_path / "reads_60mers"), with_counts=True)
    assert np.array_equal(fk, wk) and np.array_equal(fc.astype(np.uint8), wc)
    bounds = [np.load(str(tmp_path / ("plan_%d.npy" % r))).tolist() for r in range(world)]
    assert bounds[0][0] == 0 and all(bounds[r][1] == bounds[r + 1][0] for r in range(world - 1)) and bounds[-1][1] == 4 ** 10
