"""The exchange clamp (mlg_query_set_exchange_clamp), on one GPU with emulated ranks (test_gpu_exchange_emulated's
workload and data movement).  Presence is summed counters >= ci_min whatever the clamp; with the clamp at counter_max (3)
the intersection dump and KMC database of every rank must be byte-identical to those of one query over all the reads, in
the gather, sparse and both dense forms, at world sizes up to 16 and with shards where one rank sees a k-mer 3 or more
times.  The refusals: a clamp below ci_min or above 255, clamp * world past the 8-bit sums, a clamp set after an
exchange."""
import numpy as np
import pytest

from metalign_b200.api import Exchange, MlgError
from test_gpu_exchange_emulated import (ERR_ARG, ERR_STATE, FORMS, _exchange, _expected_dump, _off, _shards,  # noqa: F401
                                        workloads)

pytestmark = pytest.mark.gpu
CASES = [(W, s) for W in (2, 3, 5, 8, 16) for s in ("contiguous", "interleaved", "one_rank")]


def _files(q, tmp_path, tag):
    dump, kmc = tmp_path / ("dump_" + tag), tmp_path / ("kmc_" + tag)
    q.dump_intersection(str(dump), None, 3)
    q.write_intersection_kmc(str(kmc), counter_max=3)
    return dump.read_bytes(), (tmp_path / ("kmc_%s.kmc_pre" % tag)).read_bytes(), (tmp_path / ("kmc_%s.kmc_suf" % tag)).read_bytes()


@pytest.mark.parametrize("world,sharding", CASES)
def test_clamp_3_gives_the_single_query_files(workloads, tmp_path, world, sharding):
    w = workloads(60)
    W, ci_min, gate = world, 2, "exact"
    q = w.db.query(ci_min, gate, True)
    q.push_ascii(w.text.reshape(-1), _off(w.N))
    q.finish()
    single = _files(q, tmp_path, "single")
    q.close()
    texts = [np.ascontiguousarray(w.text[s]) for s in _shards(sharding, w.N, W)]
    counts = [w.shard_counts(t) for t in texts]
    # some k-mer of the intersection is seen 3 or more times by one rank and the clamp at ci_min loses it
    assert max(int(c.max()) for c in counts) >= 3
    exs = [Exchange(w.ctx, W, r, w.db.n_distinct) for r in range(W)]
    differs = False
    for form in FORMS:
        for clamp in (None, 3):
            qs = []
            for t in texts:
                qq = w.db.query(ci_min, gate, True)
                if t.shape[0]:
                    qq.push_ascii(t.reshape(-1), _off(t.shape[0]))
                if clamp is not None:
                    qq.set_exchange_clamp(clamp)
                qs.append(qq)
            keep = _exchange(w, form, qs, exs, ci_min)
            for qq in qs:
                qq.finish()
            del keep
            for r, qq in enumerate(qs):
                got = _files(qq, tmp_path, "%s_%s_%d" % (form, clamp, r))
                if clamp == 3:
                    assert got == single, (form, r)
                else:                                # today's counts: the sum of min(c_r, ci_min)
                    ref_I = qq.intersection()
                    assert got[0].decode() == _expected_dump(w, ref_I, counts, ci_min, 3), (form, r)
                    differs |= got != single
            for qq in qs:
                qq.close()
    for ex in exs:
        ex.close()
    if sharding == "one_rank":    # one rank sees every read: the default clamp loses the counts of 3 and more
        assert differs


def test_clamp_refusals(workloads):
    w = workloads(60)
    q = w.db.query(2)
    for bad in (1, 256, -1):
        with pytest.raises(MlgError) as e:
            q.set_exchange_clamp(bad)
        assert e.value.code == ERR_ARG, bad
    q.push_ascii(w.text[:100].reshape(-1), _off(100))
    q.set_exchange_clamp(128)
    ex = Exchange(w.ctx, 2, 0, 8)                       # 128 * 2 > 255
    with pytest.raises(MlgError) as e:
        q.exchange_pack(ex)
    assert e.value.code == ERR_ARG
    q.set_exchange_clamp(127)                           # 127 * 2 = 254: fits
    q.exchange_pack(ex)
    with pytest.raises(MlgError) as e:                  # after an exchange
        q.set_exchange_clamp(3)
    assert e.value.code == ERR_STATE
    q.close()
    ex.close()
    for call in ("counts_export_sparse", "exchange_dense", "counts_export"):
        q = w.db.query(2)
        q.push_ascii(w.text[:100].reshape(-1), _off(100))
        getattr(q, call)()
        with pytest.raises(MlgError) as e:
            q.set_exchange_clamp(3)
        assert e.value.code == ERR_STATE, call
        q.close()
