"""The exchange of the per-k-mer counters between ranks, emulated on one GPU.  W ranks live in one process: one Context,
one Database, one Query and one Exchange per rank, and the test itself moves the data between the ranks with torch
copies on the library's compute stream (the all-gather of the blocks, the all-gather of the sparse arrays, the uint8
sum of the dense tables).  Every form is checked against the single-process C oracle over all the reads, on every rank:

  gather   exchange_pack -> every rank's send block copied into every rank's recv -> exchange_merge
  sparse   counts_export_sparse -> arrays zero-padded to one length -> counts_merge_sparse of every other rank's array
  dense    counts_export -> uint8 sum written back into every table -> counts_import; and exchange_dense, no host join

at world sizes 1 to 16, with contiguous, interleaved, one-empty-rank and all-on-one-rank shards, ci_min 1, 2 and the
largest one the 8-bit sums allow (255 // W), both gates, K = 60 (minimizer layout) and K = 31 (whole-k-mer hash layout).
The counts that dump_intersection writes after an exchange are checked against an independent reference: per-shard
read k-mer counts from the read k-mer oracle and the sketch multiplicities from the keys.  Then the overflow / retry
protocol of the gather form, with every rank over the cap, with one rank alone over it, at the cap exactly and with
reused exchanges; and the counter table that a query hands on to the next one.  (The p2p form needs CUDA IPC between
processes and stays with test_gpu_multi.py.)"""
import numpy as np
import pytest

import synth
from helpers import oracle_c_run
from metalign_b200 import codec, dist
from metalign_b200._lib import MLG_ERR_RETRY
from metalign_b200.api import Exchange, Database, MlgError
from oracle.read_kmers import OracleReadKmers

pytestmark = pytest.mark.gpu
ERR_ARG, ERR_STATE = -2, -4
EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)
READ_LEN = 150
KS = {60: (30, 40, 50, 60), 31: (15, 21, 31)}
WORLDS = (1, 2, 3, 5, 8, 16)
SHARDINGS = ("contiguous", "interleaved", "empty_rank", "one_rank")
FORMS = ("gather", "sparse", "dense_export", "dense_exchange")


# ---------------------------------------------------------------------------------------------------------- workload
def _workload_arrays(K):
    """one database over two communities: a deep one (two 3 kb genomes, error-free reads, counters saturate at 255 on a
    rank) and a wide one (ten genomes of 2-80 kb with skewed abundances, substitutions and N: counts of 1 to ~100).
    Forty more genomes copy random slots of the first fourteen, so that a k-mer's sketch multiplicity (the count of its
    KMC database) runs from 1 to ~10.  Reads: the deep community's first, then the wide one's."""
    n = 300
    deep = synth.params(G=4, n=n, K=K, seed=41 + K, len_min=3000, len_max=3500, n_present=2, strain_period=0, tiny_pct=0,
                        sub_per_64k=0, n_per_64k=0)
    wide = synth.params(G=10, n=n, K=K, seed=42 + K, len_min=2000, len_max=80000, n_present=10)
    base = np.concatenate([synth.sketch_keys(deep), synth.sketch_keys(wide)]).reshape(-1, n, 2)
    rng = np.random.default_rng(K)
    extra = base[rng.integers(0, base.shape[0], 40)].copy()
    extra[rng.random((40, n)) < 0.4] = EMPTY
    keys = np.ascontiguousarray(np.concatenate([base, extra]).reshape(-1, 2))
    text = np.concatenate([synth.reads_ascii(deep, 0, 30000), synth.reads_ascii(wide, 0, 70000)])
    return keys, keys.shape[0] // n, n, text


def _off(n_reads):
    return np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(READ_LEN)


class Workload:
    def __init__(self, ctx, K):
        import torch
        self.ctx, self.K, self.ks = ctx, K, KS[K]
        self.keys, self.G, self.n, self.text = _workload_arrays(K)
        self.N = self.text.shape[0]
        self.db = Database.from_keys(ctx, self.keys, self.G, self.n, K, self.ks)
        self.comp = torch.cuda.ExternalStream(ctx.streams()[0])
        # D with its multiplicities: canonical keys of the non-empty slots, counted, saturated at 255
        full = self.keys[self.keys[:, 0] != EMPTY]
        self.D, mult = np.unique(codec.canonical_keys(full, K), axis=0, return_counts=True)
        self.D_mult = np.minimum(mult, 255)
        self.D_index = {(int(a), int(b)): i for i, (a, b) in enumerate(self.D)}
        self._refs = {}

    def ref(self, ci_min, gate, rows=None):
        """oracle_c_run over the reads `rows` (all of them by default) in one process"""
        key = (ci_min, gate, None if rows is None else (rows.start, rows.stop))
        if key not in self._refs:
            t = self.text if rows is None else self.text[rows]
            self._refs[key] = oracle_c_run(self.keys, self.G, self.n, self.K, self.ks,
                                           lambda q: q.push_ascii(t.tobytes(), _off(t.shape[0])), ci_min, gate, True)
        return self._refs[key]

    def shard_counts(self, t):
        """c_r over D: the read k-mer oracle's count of every k-mer of D in the reads t"""
        out = np.zeros(len(self.D), dtype=np.int64)
        if t.shape[0] == 0:
            return out
        o = OracleReadKmers(self.K)
        o.push_ascii(t.tobytes(), _off(t.shape[0]))
        keys, counts = o.result(1, 255)
        o.close()
        m = np.isin(keys[:, 1], self.D[:, 1])
        for (a, b), c in zip(keys[m], counts[m]):
            i = self.D_index.get((int(a), int(b)))
            if i is not None:
                out[i] = int(c)
        return out


@pytest.fixture(scope="module")
def workloads(ctx):
    made = {}

    def get(K):
        if K not in made:
            made[K] = Workload(ctx, K)
        return made[K]
    yield get
    for w in made.values():
        w.db.close()


def _shards(kind, N, W):
    """row index ranges / slices of each rank's reads"""
    if kind == "contiguous":
        return [slice(*dist.shard_range(N, r, W)) for r in range(W)]
    if kind == "interleaved":
        return [slice(r, N, W) for r in range(W)]
    if kind == "empty_rank":                      # rank W // 2 has no reads; the others share them contiguously
        rest = [slice(*dist.shard_range(N, r, W - 1)) for r in range(W - 1)]
        return rest[:W // 2] + [slice(0, 0)] + rest[W // 2:]
    assert kind == "one_rank"                     # every read on the last rank
    return [slice(0, 0)] * (W - 1) + [slice(0, N)]


# ---------------------------------------------------------------------------------------------------------- the forms
def _begin(w, texts, ci_min, gate, read_kmers_on_rank0=False):
    qs = []
    for r, t in enumerate(texts):
        q = w.db.query(ci_min, gate, True, read_kmers=read_kmers_on_rank0 and r == 0)
        if t.shape[0]:
            q.push_ascii(t.reshape(-1), _off(t.shape[0]))
        qs.append(q)
    return qs


def _gather(w, qs, exs):
    """pack on every rank, the all-gather as copies on the compute stream (no host join), merge on every rank"""
    import torch
    for q, ex in zip(qs, exs):
        q.exchange_pack(ex)
    with torch.cuda.stream(w.comp):
        allsend = torch.cat([dist.device_view_i64(ex.send_ptr, ex.block_words) for ex in exs])
        for ex in exs:
            dist.device_view_i64(ex.recv_ptr, ex.block_words * len(exs)).copy_(allsend)
    for q, ex in zip(qs, exs):
        q.exchange_merge(ex)
    return [allsend]


def _sparse(w, qs, ci_min):
    """export on every rank, zero-padded arrays plus one entry past |D| (ignored by the merge), merge of every other
    rank's array"""
    import torch
    nd = w.db.n_distinct
    exported = [q.counts_export_sparse() for q in qs]
    m = max(n for _, n in exported) + 1
    padded = []
    with torch.cuda.stream(w.comp):
        for p, n in exported:
            t = torch.zeros(m, dtype=torch.int64, device="cuda")
            if n:
                t[:n] = dist.device_view_i64(p, n)
            t[m - 1] = nd | (ci_min << 32)
            padded.append(t)
    for d, q in enumerate(qs):
        for r, t in enumerate(padded):
            if r != d:
                q.counts_merge_sparse(t.data_ptr(), m)
    return padded


def _dense(w, qs, joined):
    """the uint8 all-reduce: every rank's clamped table summed and written back into every rank's table.  Returns the
    sum in int32 too (the caller checks it after finish: no host join here)"""
    import torch
    views = [dist.device_view_u8(*(q.counts_export() if joined else q.exchange_dense())) for q in qs]
    with torch.cuda.stream(w.comp):
        wide = torch.stack([v.to(torch.int32) for v in views]).sum(0)
        total = torch.stack(views).sum(0, dtype=torch.uint8)
        for v in views:
            v.copy_(total)
    if joined:
        for q in qs:
            q.counts_import()
    return [total, wide]


def _exchange(w, form, qs, exs, ci_min):
    if form == "gather":
        return _gather(w, qs, exs)
    if form == "sparse":
        return _sparse(w, qs, ci_min)
    return _dense(w, qs, joined=form == "dense_export")


# ---------------------------------------------------------------------------------------------------------- checks
def _check_rank(res, I, ref, I_ref, tag):
    """test_gpu_parity._check, less n_kmers (a rank probes its own shard only)"""
    assert res["n_intersect"] == ref["n_intersect"], tag
    assert np.array_equal(I, I_ref), tag
    assert np.array_equal(res["den"], ref["den"]), tag
    assert np.array_equal(res["num"], ref["num"]), tag
    assert np.array_equal(res["ci"], ref["ci"]), tag
    assert np.max(np.abs(res["ci"] - ref["ci"]), initial=0.0) <= 1e-12, tag


def _expected_dump(w, I_ref, shard_counts, ci_min, counter_max):
    """min(sum over ranks of min(c_r, ci_min), sketch multiplicity, counter_max) for every k-mer of I, in key order"""
    idx = np.array([w.D_index[(int(a), int(b))] for a, b in I_ref], dtype=np.int64)
    summed = np.minimum(np.stack(shard_counts), ci_min).sum(axis=0)
    cnt = np.minimum(np.minimum(summed[idx], w.D_mult[idx]), counter_max)
    return "".join("%s\t%d\n" % (codec.key_to_kmer(int(a), int(b), w.K), c) for (a, b), c in zip(I_ref, cnt))


def _finish_all(qs):
    return [q.finish() for q in qs]


def _close(qs, first):
    """close every query, rank `first` first: its table is the one handed on to the next query of the database"""
    for r in range(len(qs)):
        qs[(first + r) % len(qs)].close()


def _check_handed_on_table(w, ci_min, gate, tag):
    """a fresh single-rank query over all the reads on the table the closed queries left behind"""
    ref, I_ref = w.ref(ci_min, gate)
    q = w.db.query(ci_min, gate, True)
    q.push_ascii(w.text.reshape(-1), _off(w.N))
    res = q.finish()
    _check_rank(res, q.intersection(), ref, I_ref, ("handed on",) + tag)
    assert res["n_kmers"] == ref["n_kmers"], tag
    q.close()


CASES = [(W, s) for W in WORLDS for s in SHARDINGS if W > 1 or s == "contiguous"]


@pytest.mark.parametrize("K", [60, 31])
@pytest.mark.parametrize("world,sharding", CASES)
def test_every_form_on_every_rank_matches_the_oracle(workloads, tmp_path, K, world, sharding):
    """all forms, every rank: the oracle's table and I, the same dump on every rank and in every form (counts = the sum
    over ranks of the per-rank counts clamped to ci_min, bounded by the sketch multiplicity and counter_max), and a
    counter table that the next query can use"""
    w = workloads(K)
    assert w.db.n_distinct == len(w.D) and w.db.n_distinct % 16 != 0     # k_compact_present's tail is exercised
    W = world
    slices = _shards(sharding, w.N, W)
    texts = [np.ascontiguousarray(w.text[s]) for s in slices]
    assert sum(t.shape[0] for t in texts) == w.N
    counts = [w.shard_counts(t) for t in texts]
    exs = [Exchange(w.ctx, W, r, w.db.n_distinct) for r in range(W)]
    first = 0
    for ci_min in sorted({1, 2, 255 // W}):
        for gate in ("exact", "none"):
            ref, I_ref = w.ref(ci_min, gate)
            dumps = {cm: _expected_dump(w, I_ref, counts, ci_min, cm) for cm in (3, 255)}
            for form in FORMS:
                tag = (form, ci_min, gate)
                rk = gate == "exact"
                qs = _begin(w, texts, ci_min, gate, read_kmers_on_rank0=rk)
                keep = _exchange(w, form, qs, exs, ci_min)
                results = _finish_all(qs)
                if form.startswith("dense"):             # every rank's counters were clamped to ci_min before the sum
                    assert int(keep[1].max()) <= ci_min * W, tag
                del keep
                assert sum(res["n_kmers"] for res in results) == ref["n_kmers"], tag
                for r, (q, res) in enumerate(zip(qs, results)):
                    assert res["stats"]["layout"] == (2 if K == 60 else 0)
                    _check_rank(res, q.intersection(), ref, I_ref, tag + (r,))
                    for cm, want in dumps.items():
                        path = tmp_path / ("dump_%s_%d_%d" % (form, r, cm))
                        q.dump_intersection(str(path), None, cm)
                        assert path.read_text() == want, tag + (r, cm)
                if rk:
                    with pytest.raises(MlgError) as e:
                        qs[0].read_kmers()
                    assert e.value.code == ERR_STATE, tag
                _close(qs, first)
                first += 1
                if form in ("gather", "sparse"):        # a dense sum writes counters on no list: that table is dropped
                    _check_handed_on_table(w, ci_min, gate, tag)
    for ex in exs:
        ex.close()


# ---------------------------------------------------------------------------------------------------------- overflow
def _n_touched(w, texts):
    """non-zero counters per rank: the k-mers of D that the rank's reads contain"""
    return [int((w.shard_counts(t) > 0).sum()) for t in texts]


def _needed(e):
    return int(str(e.value).split(":")[-1].split()[0])


def _expect_retry_everywhere(qs):
    need = []
    for r, q in enumerate(qs):
        with pytest.raises(MlgError) as e:
            q.finish()
        assert e.value.code == MLG_ERR_RETRY, r
        need.append(_needed(e))
    return need


def _redo_and_check(w, qs, cap, ci_min, gate, rows=None):
    W = len(qs)
    exs = [Exchange(w.ctx, W, r, cap) for r in range(W)]
    keep = _gather(w, qs, exs)
    results = _finish_all(qs)
    del keep
    ref, I_ref = w.ref(ci_min, gate, rows)
    assert sum(res["n_kmers"] for res in results) == ref["n_kmers"]
    for r, (q, res) in enumerate(zip(qs, results)):
        _check_rank(res, q.intersection(), ref, I_ref, ("redo", r))
    for ex in exs:
        ex.close()


def test_overflow_every_rank_over_the_cap(workloads):
    """blocks of one entry: every rank's finish asks for a repeat, all with the same count (the largest one, the rank's
    own included); repeated with blocks that large, nothing is counted twice"""
    w = workloads(60)
    W, ci_min, gate = 3, 2, "exact"
    texts = [np.ascontiguousarray(w.text[s]) for s in _shards("interleaved", w.N, W)]
    n = _n_touched(w, texts)
    qs = _begin(w, texts, ci_min, gate)
    exs = [Exchange(w.ctx, W, r, 1) for r in range(W)]
    keep = _gather(w, qs, exs)
    need = _expect_retry_everywhere(qs)
    del keep
    assert need == [max(n)] * W, (need, n)
    for ex in exs:
        ex.close()
    _redo_and_check(w, qs, max(need), ci_min, gate)
    _close(qs, 0)
    _check_handed_on_table(w, ci_min, gate, ("symmetric overflow",))


def test_overflow_one_rank_alone_over_the_cap(workloads):
    """rank 0 holds most of the reads and is the only rank with more non-zero counters than a block holds: every rank --
    rank 0 too -- must reach the same verdict, or the repeated exchange would be a collective that rank 0 never joins"""
    w = workloads(60)
    W, ci_min, gate = 3, 2, "exact"
    big = int(w.N * 0.8)
    slices = [slice(0, big)] + [slice(*(big + np.array(dist.shard_range(w.N - big, r, W - 1)))) for r in range(W - 1)]
    texts = [np.ascontiguousarray(w.text[s]) for s in slices]
    n = _n_touched(w, texts)
    cap = max(n[1:])
    assert n[0] > cap, n
    qs = _begin(w, texts, ci_min, gate)
    exs = [Exchange(w.ctx, W, r, cap) for r in range(W)]
    keep = _gather(w, qs, exs)
    need = _expect_retry_everywhere(qs)
    del keep
    assert need == [n[0]] * W, (need, n)
    for ex in exs:
        ex.close()
    _redo_and_check(w, qs, n[0], ci_min, gate)
    _close(qs, 0)
    _check_handed_on_table(w, ci_min, gate, ("asymmetric overflow",))


def test_overflow_boundary_and_reused_exchanges(workloads):
    """blocks exactly as large as the largest count: no repeat, and every block header carries its rank's count; then the
    same exchanges for a second round of queries over fewer reads, whose blocks end before the stale entries of the first"""
    import torch
    w = workloads(60)
    W, ci_min, gate = 3, 2, "exact"
    texts = [np.ascontiguousarray(w.text[s]) for s in _shards("contiguous", w.N, W)]
    n = _n_touched(w, texts)
    exs = [Exchange(w.ctx, W, r, max(n)) for r in range(W)]
    qs = _begin(w, texts, ci_min, gate)
    keep = _gather(w, qs, exs)
    torch.cuda.synchronize()
    assert [int(t[0]) for t in keep[0].view(W, -1)] == n
    results = _finish_all(qs)
    ref, I_ref = w.ref(ci_min, gate)
    for r, (q, res) in enumerate(zip(qs, results)):
        _check_rank(res, q.intersection(), ref, I_ref, ("boundary", r))
    _close(qs, 1)
    rows = slice(0, w.N // 3)
    sub = w.text[rows]
    texts2 = [np.ascontiguousarray(sub[s]) for s in _shards("interleaved", sub.shape[0], W)]
    n2 = _n_touched(w, texts2)
    assert all(a < b for a, b in zip(n2, n)), (n2, n)
    qs = _begin(w, texts2, ci_min, gate)
    keep = _gather(w, qs, exs)
    results = _finish_all(qs)
    del keep
    ref, I_ref = w.ref(ci_min, gate, rows)
    assert sum(res["n_kmers"] for res in results) == ref["n_kmers"]
    for r, (q, res) in enumerate(zip(qs, results)):
        _check_rank(res, q.intersection(), ref, I_ref, ("reuse", r))
    _close(qs, 2)
    for ex in exs:
        ex.close()
    _check_handed_on_table(w, ci_min, gate, ("reuse",))


def test_exchange_refusals(workloads):
    """more ranks than MLG_MAX_RANKS, and ci_min * world past the 8-bit counters, are refused"""
    w = workloads(60)
    with pytest.raises(MlgError) as e:
        Exchange(w.ctx, 17, 0, 8)
    assert e.value.code == ERR_ARG
    with pytest.raises(MlgError) as e:
        Exchange(w.ctx, 4, 4, 8)
    assert e.value.code == ERR_ARG
    ex = Exchange(w.ctx, 16, 3, 8)
    q = w.db.query(16)
    q.push_ascii(w.text[:100].reshape(-1), _off(100))
    for call in (q.exchange_pack, q.exchange_merge):
        with pytest.raises(MlgError) as e:
            call(ex)
        assert e.value.code == ERR_ARG
    q.close()
    ex.close()
    ex = Exchange(w.ctx, 15, 3, 8)              # 17 * 15 = 255: the largest sum that fits
    q = w.db.query(17)
    q.exchange_pack(ex)
    q.close()
    ex.close()
