"""Two real GPUs, one process each: read-sharded probe + ONE exchange of the per-k-mer counters -- the NCCL all-gather
of the non-zero counters, the dense uint8 all-reduce, and the direct NVLink-store form ("p2p"), each without a host
round trip -- against the single-process CPU oracle.  "tiny" forces blocks too small for the counters, i.e. the
repeat-with-larger-blocks path.  "uneven" gives rank 0 most of the reads and blocks that hold rank 1's non-zero counters
but not rank 0's: both ranks must repeat the exchange, rank 0 because of its own count.  Skipped when fewer than two
GPUs are visible."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
KS = (30, 40, 50, 60)
NREADS = 200_001


def _params():
    import synth
    return synth.params(G=400, n=250, seed=13, len_min=20000, len_max=60000, n_present=50, paired=1)


def _uneven_range(rank):
    """rank 0 gets 80 % of the reads, rank 1 the rest"""
    big = NREADS * 4 // 5
    return (0, big) if rank == 0 else (big, NREADS)


def _touched_counts(p, keys, ranges):
    """per read range: the number of distinct k-mers of D in the reads (a rank's non-zero counters), from the read
    k-mer oracle"""
    import synth
    from metalign_b200 import codec
    from oracle.read_kmers import OracleReadKmers
    full = keys[keys[:, 0] != np.uint64(0xFFFFFFFFFFFFFFFF)]
    D = np.unique(codec.canonical_keys(full, 60), axis=0)
    Dset = set(map(tuple, D.tolist()))
    out = []
    for a, b in ranges:
        bases, nmask = synth.reads_packed(p, a, b - a)
        o = OracleReadKmers(60)
        o.push_packed(bases, nmask, None, b - a, p.read_len)
        k, _ = o.result(1, 255)
        o.close()
        k = k[np.isin(k[:, 1], D[:, 1])]
        out.append(sum(1 for x in map(tuple, k.tolist()) if x in Dset))
    return out


def _worker(rank, world, port, out_dir, mode, cap=0):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as tdist
    import synth
    from metalign_b200 import dist as mdist
    from metalign_b200.api import Context, Database
    uneven = mode.endswith("-uneven")
    if mode.endswith("-tiny"):
        mode = mode[:-5]
        os.environ["MLG_EXCHANGE_CAP"] = "64"
    elif uneven:
        mode = mode[:-7]
        os.environ["MLG_EXCHANGE_CAP"] = str(cap)
    r, w, local = mdist.init_from_env("nccl")
    p = _params()
    keys = synth.sketch_keys(p)
    a, b = _uneven_range(rank) if uneven else mdist.shard_range(NREADS, rank, world)
    bases, nmask = synth.reads_packed(p, a, b - a)
    ctx = Context(local)
    db = Database.from_keys(ctx, keys, p.G, p.n, 60, KS)
    q = db.query()
    q.push_packed(bases, nmask, None, b - a, p.read_len)
    mdist.reduce_query(q, local, mode=mode)
    res = q.finish()
    np.save(os.path.join(out_dir, "num_%d.npy" % rank), res["num"])
    np.save(os.path.join(out_dir, "I_%d.npy" % rank), q.intersection())
    # a second query through the same persistent exchange (epochs / buffer reuse)
    q2 = db.query()
    q2.push_packed(bases, nmask, None, b - a, p.read_len)
    mdist.reduce_query(q2, local, mode=mode)
    res2 = q2.finish()
    assert np.array_equal(res2["num"], res["num"])
    q2.close(); q.close()
    mdist.close_exchanges()
    db.close(); ctx.close()
    tdist.destroy_process_group()


MODES = ["sparse", "dense", "p2p", "sparse-tiny", "p2p-tiny", "sparse-uneven", "p2p-uneven"]


@pytest.mark.parametrize("mode", MODES)
def test_two_gpu_read_sharding_matches_oracle(tmp_path, mode):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import synth
    from helpers import oracle_c_run
    world = 2
    p = _params()
    keys = synth.sketch_keys(p)
    cap = 0
    if mode.endswith("-uneven"):
        n0, n1 = _touched_counts(p, keys, [_uneven_range(r) for r in range(world)])
        assert n1 < n0, (n0, n1)
        cap = (n0 + n1) // 2                   # rank 1's block fits, rank 0's does not
    mp.spawn(_worker, args=(world, 29400 + os.getpid() % 500 + 7 * MODES.index(mode), str(tmp_path), mode, cap), nprocs=world,
             join=True)
    bases, nmask = synth.reads_packed(p, 0, NREADS)
    ref, I_ref = oracle_c_run(keys, p.G, p.n, 60, KS, lambda q: q.push_packed(bases, nmask, None, NREADS, p.read_len))
    assert ref["n_intersect"] > 100
    for r in range(world):
        assert np.array_equal(np.load(tmp_path / ("num_%d.npy" % r)), ref["num"])
        assert np.array_equal(np.load(tmp_path / ("I_%d.npy" % r)), I_ref)
