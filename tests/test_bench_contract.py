"""bench.py's JSON contract, checked on CPU through the reference arm (the oracle port on host threads), and its
--dump-outputs files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, has_cuda

REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "impl"}


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "1", "--scenario", "short_0p3s_4x64"], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["unit"] == "events/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["dtype"] == "f64" and d["data"] == "synthetic" and d["scaling"] == "weak"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_b200_arm_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                         text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def _dumped(d):
    return {n: np.load(os.path.join(d, n + ".npy")) for n in ("summary", "replica_ids", "aggregate")}


def test_dump_outputs_stays_within_budget_with_a_fixed_sample(tmp_path):
    import bench
    from distributed_cluster_gpus_b200 import spec as S
    agg = np.arange(S.AGG_K, dtype=np.float64)
    small = np.random.default_rng(1).random((1000, S.SUMMARY_K))
    bench.dump_outputs(str(tmp_path / "small"), small, 5000, agg)
    got = _dumped(tmp_path / "small")
    assert np.array_equal(got["summary"], small) and np.array_equal(got["replica_ids"], 5000 + np.arange(1000.0))
    assert np.array_equal(got["aggregate"], agg)

    big = np.random.default_rng(2).random((120000, S.SUMMARY_K))             # 84 MB of summaries
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), big, 0, agg)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= bench.DUMP_BYTES
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    ids = a["replica_ids"].astype(np.int64)
    assert len(ids) < len(big) and np.all(np.diff(ids) > 0)
    assert np.array_equal(a["summary"], big[ids])
    assert all(np.array_equal(a[n], b[n]) for n in a)
    assert all(v.dtype == np.float64 for v in a.values())


@pytest.mark.gpu
@pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")
def test_dump_outputs_are_the_last_timed_step(oracle, tmp_path):
    """The dumped summaries are the ones the oracle computes at the seed of the last timed step, which exists only if
    --steps steps ran after --warmup."""
    from distributed_cluster_gpus_b200 import scenarios as SC, sharding, spec as S
    R, warmup, steps, duration = 512, 1, 2, 20.0
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                          "--warmup", str(warmup), "--replicas", str(R), "--duration", str(duration), "--no-e2e",
                          "--no-configs", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    got = _dumped(tmp_path)
    assert np.array_equal(got["replica_ids"], np.arange(float(R)))
    sc = dict(SC.BY_NAME["cfg3_4x64_sinusoid_120s"], duration=duration)
    want, _ = oracle.run_batch(SC.to_spec(sc).to_bytes(), R, 123 + (warmup + steps - 1) * R, 0, oracle.RNG_PHILOX,
                               os.cpu_count() or 1)
    summary = got["summary"]
    assert np.all(summary[:, S.S_STATUS] == 0) and np.all(summary[:, S.S_DONE] == 1)
    for col in (S.S_EVENTS, S.S_JOBS_FINISHED, S.S_JOBS_CREATED, S.S_RNG_WORDS, S.S_SEQ):
        assert np.array_equal(summary[:, col], want[:, col]), col
    for col in (S.S_TOTAL_ENERGY_J, S.S_LAT_SUM):
        assert np.max(np.abs(summary[:, col] - want[:, col]) / np.maximum(np.abs(want[:, col]), 1e-300)) <= 1e-9, col
    assert got["aggregate"][S.A_EVENTS] == summary[:, S.S_EVENTS].sum()
    np.testing.assert_allclose(got["aggregate"], sharding.aggregate_rows(summary), rtol=1e-11)
