"""bench.py's workload plans (BASELINE.json configs[1..4]): every read of the job belongs to exactly one rank's batches, in
order, whatever the world size; the reference arm takes the native arm's first batch."""
import importlib.util
import os

import numpy as np
import pytest

from conftest import ROOT

spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
bench = importlib.util.module_from_spec(spec)
spec.loader.exec_module(bench)


@pytest.mark.parametrize("name", sorted(bench.WORKLOADS))
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_plans_partition_the_reads(name, world, monkeypatch):
    for k in ("MLG_BENCH_G", "MLG_BENCH_READS", "MLG_BENCH_TOTAL_READS", "MLG_BENCH_BATCH_READS"):
        monkeypatch.delenv(k, raising=False)
    nxt, total_seen = 0, None
    for rank in range(world):
        G, paired, batches, total, desc = bench.workload_plan(name, world, rank)
        total_seen = total if total_seen is None else total_seen
        assert total == total_seen and G == bench.WORKLOADS[name]["G"]
        for r0, n in batches:
            assert r0 == nxt and 0 < n <= bench.BATCH_READS
            nxt += n
        assert "configs[" in desc
    assert nxt == total_seen
    w = bench.WORKLOADS[name]
    assert total_seen == (w["total"] or w["per_gpu"] * world)


def test_env_overrides(monkeypatch):
    monkeypatch.setenv("MLG_BENCH_TOTAL_READS", "1e6")
    monkeypatch.setenv("MLG_BENCH_BATCH_READS", "3e5")
    monkeypatch.setenv("MLG_BENCH_G", "1234")
    G, paired, batches, total, desc = bench.workload_plan("stream", 3, 1)
    assert G == 1234 and total == 1_000_000
    assert batches[0][0] == 333_334 and sum(n for _, n in batches) == 333_333 and max(n for _, n in batches) == 300_000


def test_dump_outputs_within_budget(tmp_path, monkeypatch):
    """--dump-outputs: every array as float64; over the budget, tables keep a seeded sample of rows, the same in every run"""
    G, nk = 10_000, 4
    ci = np.random.default_rng(1).random((G, nk))
    num = np.arange(G * nk, dtype=np.int64).reshape(G, nk)
    arrays = {"ci": ci, "num": num, "n_intersect": np.array([123456789], dtype=np.uint64)}
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    assert np.array_equal(np.load(tmp_path / "whole" / "ci.npy"), ci)
    assert not (tmp_path / "whole" / "sampled_rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {f: np.load(tmp_path / "a" / f) for f in sorted(os.listdir(tmp_path / "a"))}
    assert sorted(got) == ["ci.npy", "n_intersect.npy", "num.npy", "sampled_rows.npy"]
    assert all(a.dtype == np.float64 for a in got.values()) and sum(a.nbytes for a in got.values()) <= 1 << 16
    rows = got["sampled_rows.npy"].astype(np.int64)
    assert rows.size > 0 and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["ci.npy"], ci[rows]) and np.array_equal(got["num.npy"], num[rows])
    assert got["n_intersect.npy"].tolist() == [123456789.0]
    for f, a in got.items():
        assert np.array_equal(np.load(tmp_path / "b" / f), a)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_bad_arguments_are_refused(argv, monkeypatch):
    monkeypatch.setattr(bench.sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
