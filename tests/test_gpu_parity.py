"""Parity tests proper: the sm_100a kernel through the C-ABI against the oracle and the reference fixtures.

Bar (BASELINE.json north_star): exact event / job / RNG-word counts; per-replica total energy and mean job
latency within 1e-9 relative.  Every float of the summary is held to the same 1e-9.
"""
import os

import numpy as np
import pytest

from conftest import golden_names, has_cuda, load_golden
from distributed_cluster_gpus_b200 import scenarios as SC, sharding, spec as S

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")]

RTOL = 1e-9
COUNT_COLS = (S.S_STATUS, S.S_EVENTS, S.S_JOBS_FINISHED, S.S_JOBS_CREATED, S.S_FIN_INF, S.S_FIN_TRN, S.S_RNG_WORDS,
              S.S_SEQ, S.S_EV_ARRIVAL, S.S_EV_XFER, S.S_EV_FINISH, S.S_EV_LOG, S.S_DONE, S.S_MAX_RUN, S.S_MAX_Q)
FLOAT_COLS = (S.S_TOTAL_ENERGY_J, S.S_LAT_SUM, S.S_LAT_SUM_INF, S.S_LAT_SUM_TRN, S.S_LAST_T)
DEVICE_SUPPORTED = golden_names()


def engine_cls():
    from distributed_cluster_gpus_b200.engine import BatchedEngine
    return BatchedEngine


def assert_rows_match(got, want, n_dc, rtol=RTOL):
    for col in COUNT_COLS:
        assert np.array_equal(got[:, col], want[:, col]), f"count column {col}: {got[:, col]} vs {want[:, col]}"
    worst = 0.0
    cols = list(FLOAT_COLS)
    for d in range(n_dc):
        b = S.S_DC0 + d * S.S_DC_STRIDE
        cols += [b + S.SD_ENERGY_J, b + S.SD_UTIL_GPU_TIME, b + S.SD_ACC_JOB_UNIT, b + S.SD_CURRENT_FREQ]
        for k in (S.SD_BUSY, S.SD_Q_INF, S.SD_Q_TRN, S.SD_RUNNING):
            assert np.array_equal(got[:, b + k], want[:, b + k]), f"dc{d} field {k}"
    for col in cols:
        denom = np.maximum(np.abs(want[:, col]), 1e-300)
        rel = np.max(np.where(want[:, col] == got[:, col], 0.0, np.abs(got[:, col] - want[:, col]) / denom))
        assert rel <= rtol, f"float column {col}: rel err {rel:.3e}"
        worst = max(worst, rel)
    return worst


@pytest.mark.parametrize("name", DEVICE_SUPPORTED)
def test_kernel_matches_oracle(oracle, name):
    sc = SC.BY_NAME[name]
    sp = SC.to_spec(sc)
    n = 8 if sc["duration"] * sc["n_dc"] <= 2400 else 3
    with engine_cls()(sp, n, base_seed=123, first_replica_id=0) as eng:
        total = eng.advance(0)
        got = eng.summary()
    want, want_total = oracle.run_batch(sp.to_bytes(), n, 123, 0, n_threads=os.cpu_count() or 1)
    assert total == want_total
    worst = assert_rows_match(got, want, sc["n_dc"])
    print(f"{name}: {n} replicas, {total} events, worst float rel err {worst:.2e}")


@pytest.mark.parametrize("name", ["cfg1_1x4_poisson_5000s", "cfg2_1x64_poisson_600s", "cfg3_4x64_sinusoid_120s",
                                  "cfg5_8x256_sinusoid_60s", "sweep_joint_nf", "sweep_carbon_cost", "sweep_eco_route",
                                  "sweep_bandit"])
def test_kernel_matches_reference_fixture(name):
    """Straight against the reference's own numbers (fixture = reference + injected Philox), no oracle in between."""
    doc = load_golden(name)
    sc = doc["scenario"]
    runs = {r["seed"]: r for r in doc["runs"] if r["rng"] == "philox"}
    with engine_cls()(SC.to_spec(sc), 2, base_seed=123) as eng:      # replicas 0,1 -> seeds 123,124
        eng.advance(0)
        got = eng.summary()
    for r, seed in enumerate((123, 124)):
        run = runs[seed]
        assert int(got[r, S.S_EVENTS]) == run["events"] and int(got[r, S.S_JOBS_FINISHED]) == run["jobs_finished"]
        assert int(got[r, S.S_RNG_WORDS]) == run["rng_words"] and int(got[r, S.S_SEQ]) == run["seq_pushed"]
        e_ref = float.fromhex(run["total_energy_j"])
        assert abs(got[r, S.S_TOTAL_ENERGY_J] - e_ref) <= RTOL * abs(e_ref)
        if run["jobs_finished"]:
            m_ref = float.fromhex(run["mean_latency_s"])
            assert abs(got[r, S.S_LAT_SUM] / got[r, S.S_JOBS_FINISHED] - m_ref) <= RTOL * abs(m_ref)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 6, 7, 37])
def test_partially_filled_last_warp(oracle, n):
    """Replica counts that are not a multiple of the replicas a warp carries: in the lane-group builds the event loop's
    collectives span the warp, so the lane groups without a replica stay in the loop as ghosts (dcsim_advance_impl.cuh)
    — they must neither hang the warp nor touch anything; also with a per-launch event budget (resume)."""
    sp = SC.to_spec(dict(SC.CFG3, duration=15.0))
    want, want_total = oracle.run_batch(sp.to_bytes(), n, 77, 0, n_threads=os.cpu_count() or 1)
    with engine_cls()(sp, n, base_seed=77) as eng:
        assert eng.advance(0) == want_total
        assert_rows_match(eng.summary(), want, 4)
        lanes = eng.launch_info()["lanes_per_replica"]
    with engine_cls()(sp, n, base_seed=77) as eng:
        guard = 0
        while not eng.all_done():
            eng.advance(257)
            guard += 1
            assert guard < 2000
        assert_rows_match(eng.summary(), want, 4)
    print(f"{n} replicas on {lanes} lanes each")


@pytest.mark.parametrize("chunk", [1, 13, 4096])
def test_resume_is_invariant_on_device(chunk):
    sp = SC.to_spec(dict(SC.CFG3, duration=10.0 if chunk == 1 else 40.0))
    with engine_cls()(sp, 5, base_seed=9) as eng:
        eng.advance(0)
        whole = eng.summary()
    with engine_cls()(sp, 5, base_seed=9) as eng:
        guard = 0
        while not eng.all_done():
            eng.advance(chunk)
            guard += 1
            assert guard < 20000
        parts = eng.summary()
    assert np.array_equal(whole, parts)


def test_trace_and_logs_match_oracle(oracle):
    sp = SC.to_spec(SC.BY_NAME["ragged_3dc_12_5_40"])
    with engine_cls()(sp, 4, base_seed=40) as eng:
        eng.set_trace(2, 6000)
        eng.set_logging(2, 20000, 2000)
        eng.advance(0)
        tr, jobs, cl = eng.trace(), eng.job_log(), eng.cluster_log()
    sim = oracle.OracleSim(sp.to_bytes(), 42, trace_cap=6000, joblog_cap=20000, clog_cap=2000)
    sim.advance(0)
    wt, wj, wc = sim.trace(), sim.job_log(), sim.cluster_log()
    assert len(tr) == len(wt) and np.array_equal(tr["kind"], wt["kind"]) and np.array_equal(tr["seq"], wt["seq"])
    np.testing.assert_allclose(tr["t"], wt["t"], rtol=1e-12, atol=0)
    assert len(jobs) == len(wj) and len(cl) == len(wc)
    for f in ("jid", "ingress", "jtype", "dc", "n_gpus"):
        assert np.array_equal(jobs[f], wj[f]), f
    for f in ("size", "f_used", "start_s", "finish_s"):
        np.testing.assert_allclose(jobs[f], wj[f], rtol=1e-12)
    for f in ("dc", "busy", "run_total", "run_inf", "q_inf", "q_train"):
        assert np.array_equal(cl[f], wc[f]), f
    for f in ("time_s", "freq", "util_gpu_time", "util_begin_ts", "acc_job_unit", "power_w", "energy_j"):
        np.testing.assert_allclose(cl[f], wc[f], rtol=1e-9)


def test_full_size_batch_properties(oracle):
    """BASELINE size (65 536 replicas, 4 DC x 64) on a short horizon: every replica finishes cleanly, the batch is
    deterministic, a random sample agrees with the oracle, results do not depend on the batch a replica is in,
    and the on-device reduction equals the host aggregate."""
    import torch
    sp = SC.to_spec(dict(SC.CFG3, duration=12.0))
    n = 65536
    with engine_cls()(sp, n, base_seed=1000) as eng:
        total = eng.advance(0)
        big = eng.summary()
        agg_t = torch.zeros(S.AGG_K, dtype=torch.float64, device="cuda")
        eng.reduce_into(agg_t.data_ptr())
        torch.cuda.synchronize()
        agg = agg_t.cpu().numpy()
        eng.reset(1000)
        assert eng.advance(0) == total
        assert np.array_equal(eng.summary(), big)                      # deterministic, reset is clean
    assert np.all(big[:, S.S_STATUS] == 0) and np.all(big[:, S.S_DONE] == 1)
    assert big[:, S.S_EVENTS].sum() == total
    host = sharding.aggregate_rows(big)
    assert agg[S.A_REPLICAS] == n and agg[S.A_FAILED] == 0 and agg[S.A_EVENTS] == total
    np.testing.assert_allclose(agg, host, rtol=1e-11)
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(n, 64, replace=False))
    for r in sample[:8]:                                               # sharding invariance: same id, different batch
        with engine_cls()(sp, 3, base_seed=1000, first_replica_id=int(r)) as eng:
            eng.advance(0)
            assert np.array_equal(eng.summary()[0], big[r])
    want = np.stack([oracle.run_batch(sp.to_bytes(), 1, 1000, int(r))[0][0] for r in sample])
    assert_rows_match(big[sample], want, 4)
    words = big[:, S.S_RNG_WORDS]
    assert words.min() > 0 and len(np.unique(big[:, S.S_TOTAL_ENERGY_J])) > n * 0.99   # replicas really differ


def test_capacity_overflow_surfaces_and_engine_retries():
    from distributed_cluster_gpus_b200.engine import run_to_completion
    sc = dict(SC.CFG3, duration=30.0)
    with engine_cls()(SC.to_spec(sc, caps={"cap_run": 4}), 2, base_seed=1) as eng:
        eng.advance(0)
        s = eng.summary()
    assert np.all(s[:, S.S_STATUS].astype(int) & S.ST_RUN_OVERFLOW) and np.all(s[:, S.S_DONE] == 0)
    first = {"n": 0}

    def factory(caps):
        first["n"] += 1
        return SC.to_spec(sc, caps=caps if caps else {"cap_run": 4})
    eng, summ = run_to_completion(factory, 2, 1)
    eng.close()
    assert first["n"] == 2 and np.all(summ[:, S.S_STATUS] == 0) and np.all(summ[:, S.S_DONE] == 1)


def test_drop_in_simulator_and_csvs(tmp_path, oracle):
    import csv
    import logging
    from distributed_cluster_gpus_b200.configs import paper_config as pc
    from distributed_cluster_gpus_b200.simcore.simulator_paper_multi import MultiIngressPaperSimulator
    sc = SC.BY_NAME["ragged_3dc_12_5_40"]
    kw = SC.build_inputs(sc)
    sim = MultiIngressPaperSimulator(router_policy=pc.build_router_policy(), logger=logging.getLogger("t"),
                                     sim_duration=sc["duration"], log_interval=sc["log_interval"], log_path=str(tmp_path),
                                     rng_seed=77, algo=sc["algo"], show_progress=False, replicas=16, **kw)
    sim.run()
    want, _ = oracle.run_batch(SC.to_spec(sc).to_bytes(), 16, 77)
    assert_rows_match(sim.summary, want, sc["n_dc"])
    for d, dc in enumerate(kw["dcs"].values()):                        # DataCenters are the result carriers
        assert abs(dc.energy_joules - want[0, S.S_DC0 + d * 8]) <= RTOL * abs(want[0, S.S_DC0 + d * 8])
        assert dc.busy_gpus == int(want[0, S.S_DC0 + d * 8 + S.SD_BUSY])
    rows = list(csv.reader(open(tmp_path / "job_log.csv")))
    assert rows[0][:4] == ["jid", "ingress", "type", "size"] and len(rows) - 1 == int(want[0, S.S_JOBS_FINISHED])
    crow = list(csv.reader(open(tmp_path / "cluster_log.csv")))
    assert crow[0][0] == "time_s" and len(crow) - 1 == int(want[0, S.S_EV_LOG]) * sc["n_dc"]


def test_unsupported_and_invalid_specs_fail_loudly():
    from distributed_cluster_gpus_b200 import _native
    sp = SC.to_spec(SC.CFG1)
    sp.algo = 99
    with pytest.raises(_native.DcsimError, match="algo"):
        engine_cls()(sp, 1, 0)
    sp = SC.to_spec(SC.CFG1)
    sp.n_dc = 0
    with pytest.raises(_native.DcsimError):
        engine_cls()(sp, 1, 0)


@pytest.mark.parametrize("name", ["cfg1_1x4_poisson_5000s", "cfg2_1x64_poisson_600s", "cfg3_4x64_sinusoid_120s",
                                  "cfg3_4x64_sinusoid_600s", "cfg5_8x256_sinusoid_60s", "sweep_joint_nf"])
def test_baseline_configs_64_replica_sample(oracle, name):
    """SURVEY.md 8(d): >= 64 replicas per BASELINE config, full duration, exact counts + 1e-9 floats."""
    sc = SC.BY_NAME[name]
    sp = SC.to_spec(sc)
    with engine_cls()(sp, 64, base_seed=20260921, first_replica_id=5) as eng:
        total = eng.advance(0)
        got = eng.summary()
    want, want_total = oracle.run_batch(sp.to_bytes(), 64, 20260921, 5, n_threads=os.cpu_count() or 1)
    assert total == want_total
    worst = assert_rows_match(got, want, sc["n_dc"])
    print(f"{name}: 64 replicas, {total} events, worst float rel err {worst:.2e}")


def test_cli_runs_a_batch(tmp_path):
    import json
    from distributed_cluster_gpus_b200.run_sim_paper import main
    out = tmp_path / "stats.json"
    sim = main(["--duration", "30", "--inf-mode", "sinusoid", "--inf-rate", "10", "--inf-period", "3600", "--trn-rate", "1",
                "--n-dc", "4", "--gpus-per-dc", "64", "--replicas", "256", "--log-path", str(tmp_path / "run" / "x"),
                "--summary-json", str(out), "--progress", ""])
    stats = json.load(open(out))
    assert stats["replicas"] == 256 and stats["events_total"] == sim.summary[:, S.S_EVENTS].sum() > 256 * 1000
    assert stats["energy_j_ci95"] > 0 and os.path.exists(sim.job_log_path) and os.path.exists(sim.cluster_log_path)


def test_parked_engine_is_reseeded_correctly(tmp_path, oracle):
    """run() parks its device allocations; the next run of the same shape re-seeds them (dcsim_reset) instead of
    re-allocating.  Results, DataCenter write-back and the CSV rows must be those of a fresh engine."""
    import csv
    import logging
    from distributed_cluster_gpus_b200 import engine as E
    from distributed_cluster_gpus_b200.configs import paper_config as pc
    from distributed_cluster_gpus_b200.simcore.simulator_paper_multi import MultiIngressPaperSimulator
    sc = SC.BY_NAME["ragged_3dc_12_5_40"]
    blob = SC.to_spec(sc).to_bytes()
    E.free_cached_engine()
    logs = {}
    for seed in (5, 900, 5):
        kw = SC.build_inputs(sc)
        sim = MultiIngressPaperSimulator(router_policy=pc.build_router_policy(), logger=logging.getLogger("t"),
                                         sim_duration=sc["duration"], log_interval=sc["log_interval"],
                                         log_path=str(tmp_path / str(seed)), rng_seed=seed, algo=sc["algo"],
                                         show_progress=False, replicas=8, **kw).run()
        want, _ = oracle.run_batch(blob, 8, seed)
        assert_rows_match(sim.summary, want, sc["n_dc"])
        rows = list(csv.reader(open(sim.job_log_path)))
        assert len(rows) - 1 == int(want[0, S.S_JOBS_FINISHED])
        assert E._CACHED["engine"] is not None                      # parked for the next run
        assert E._CACHED_LOGGED["engine"] is not None               # ... and so is the one-replica companion (CSV rows)
        logs[seed] = logs.get(seed, []) + [(open(sim.job_log_path).read(), open(sim.cluster_log_path).read())]
    assert logs[5][0] == logs[5][1]      # same seed on a re-seeded companion: the same CSV bytes as on the fresh one
    assert logs[5][0] != logs[900][0]
    E.free_cached_engine()
    assert E._CACHED["engine"] is None and E._CACHED_LOGGED["engine"] is None


def test_latency_histogram_on_device(oracle):
    """Batch histogram = sum of the oracle's per-replica histograms, up to jobs whose latency sits within the
    device's last-ulp difference of a bin edge (they may land one bin over); totals are exact."""
    from distributed_cluster_gpus_b200.engine import latency_quantiles
    sp = SC.to_spec(SC.BY_NAME["cfg3_4x64_sinusoid_600s"])
    n = 32
    with engine_cls()(sp, n, base_seed=4) as eng:
        eng.enable_latency_histogram()
        eng.advance(0)
        got = eng.latency_histogram()
        summ = eng.summary()
    _, hist = oracle.run_batch_hist(sp.to_bytes(), n, 4, n_threads=os.cpu_count() or 1)
    want = hist.astype(np.uint64).sum(axis=0)
    assert got.sum(axis=1).tolist() == [summ[:, S.S_FIN_INF].sum(), summ[:, S.S_FIN_TRN].sum()] == want.sum(axis=1).tolist()
    assert np.abs(got.astype(np.int64) - want.astype(np.int64)).sum() <= 4
    for jt in (0, 1):
        a, b = latency_quantiles(got[jt]), latency_quantiles(want[jt])
        np.testing.assert_allclose(a, b, rtol=1e-3)


def test_wide_seed_on_device(oracle):
    """base_seed 2**40 + 5 with replicas 0..3: seeds straddle the fixture's 2**40 + 7 (non-zero high key word)."""
    doc = load_golden("cfg3_4x64_sinusoid_120s")
    run = [r for r in doc["runs"] if r["rng"] == "philox" and r["seed"] == 2**40 + 7][0]
    sp = SC.to_spec(doc["scenario"])
    with engine_cls()(sp, 4, base_seed=2**40 + 5) as eng:
        eng.advance(0)
        got = eng.summary()
    assert int(got[2, S.S_EVENTS]) == run["events"] and int(got[2, S.S_RNG_WORDS]) == run["rng_words"]
    e_ref = float.fromhex(run["total_energy_j"])
    assert abs(got[2, S.S_TOTAL_ENERGY_J] - e_ref) <= RTOL * e_ref
    want, _ = oracle.run_batch(sp.to_bytes(), 4, 2**40 + 5)
    assert_rows_match(got, want, 4)


def test_random_scenarios_match_oracle(oracle):
    """Differential fuzz on the device (generator of tools/fuzz_core.py, fixed seed): plain runs (lean records),
    logged + traced runs (full records) and chunked stepping, counts exact and floats within 1e-9."""
    import random as pyrandom
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import fuzz_core
    rnd = pyrandom.Random(20260923)
    worst = 0.0
    for case in range(90):
        sc = fuzz_core.random_scenario(rnd, case)
        seed = rnd.randrange(1, 2 ** 40)
        sp = SC.to_spec(sc)
        want, want_total = oracle.run_batch(sp.to_bytes(), 4, seed, 0, n_threads=4)
        with engine_cls()(sp, 4, base_seed=seed) as eng:
            if case % 3 == 1:
                eng.set_logging(1, 60000, 4000)
                eng.set_trace(1, 4000)
            if case % 3 == 2:
                total = 0
                while not eng.all_done():
                    total += eng.advance(997)
            else:
                total = eng.advance(0)
            got = eng.summary()
        assert total == want_total, (case, sc, seed)
        worst = max(worst, assert_rows_match(got, want, sc["n_dc"]))
    print(f"90 random scenarios, worst float rel err {worst:.2e}")


def test_kernel_matches_reference_on_random_scenarios():
    """The kernels straight against the reference's numbers on the random-scenario fixture
    (tests/golden/fuzz_reference.json: 160 scenarios nobody picked by hand): counts exact, floats within 1e-9."""
    from conftest import load_fuzz_reference
    worst = 0.0
    for c in load_fuzz_reference():
        sc, run = c["scenario"], c["run"]
        with engine_cls()(SC.to_spec(sc), 1, base_seed=run["seed"]) as eng:
            eng.advance(0)
            row = eng.summary()[0]
        assert int(row[S.S_STATUS]) == 0 and int(row[S.S_EVENTS]) == run["events"], sc
        assert int(row[S.S_JOBS_FINISHED]) == run["jobs_finished"] and int(row[S.S_JOBS_CREATED]) == run["jobs_created"], sc
        assert int(row[S.S_RNG_WORDS]) == run["rng_words"] and int(row[S.S_SEQ]) == run["seq_pushed"], sc
        pairs = [(row[S.S_TOTAL_ENERGY_J], run["total_energy_j"]), (row[S.S_LAT_SUM], run["latency_sum_s"])]
        for d in range(sc["n_dc"]):
            b = S.S_DC0 + d * S.S_DC_STRIDE
            pairs += [(row[b + S.SD_ENERGY_J], run["dc"][d]["energy_j"]), (row[b + S.SD_UTIL_GPU_TIME], run["dc"][d]["util_gpu_time"]),
                      (row[b + S.SD_ACC_JOB_UNIT], run["dc"][d]["acc_job_unit"])]
            assert int(row[b + S.SD_BUSY]) == run["dc"][d]["busy"] and int(row[b + S.SD_RUNNING]) == run["dc"][d]["running"], sc
        for got, want_hex in pairs:
            want = float.fromhex(want_hex)
            rel = 0.0 if got == want else abs(got - want) / max(abs(want), 1e-300)
            assert rel <= RTOL, (sc, got, want)
            worst = max(worst, rel)
    print(f"160 random scenarios vs the reference, worst float rel err {worst:.2e}")


@pytest.mark.parametrize("name", DEVICE_SUPPORTED)
def test_mersenne_twister_mode_reproduces_the_stock_reference(name):
    """rng = "mt19937": the kernels against the fixture's "mt" run — the reference exactly as shipped, its own
    process-global Mersenne Twister at random.seed(123) (SIM:71), nothing re-bound."""
    doc = load_golden(name)
    sc = doc["scenario"]
    run = [r for r in doc["runs"] if r["rng"] == "mt"][0]
    with engine_cls()(SC.to_spec(sc), 3, base_seed=run["seed"]) as eng:
        eng.set_rng("mt19937")
        eng.advance(0)
        row = eng.summary()[0]
    assert int(row[S.S_STATUS]) == 0 and int(row[S.S_EVENTS]) == run["events"]
    assert int(row[S.S_JOBS_FINISHED]) == run["jobs_finished"] and int(row[S.S_SEQ]) == run["seq_pushed"]
    for got, want_hex in [(row[S.S_TOTAL_ENERGY_J], run["total_energy_j"]), (row[S.S_LAT_SUM], run["latency_sum_s"])] + \
            [(row[S.S_DC0 + d * S.S_DC_STRIDE + S.SD_ENERGY_J], run["dc"][d]["energy_j"]) for d in range(sc["n_dc"])]:
        want = float.fromhex(want_hex)
        assert got == want or abs(got - want) <= RTOL * abs(want), (got, want)


def test_survey_known_answers_on_device(tmp_path):
    """SURVEY.md App. C through the drop-in simulator: `rng="mt19937", rng_seed=123` gives the event counts and total
    energies the survey recorded from the unmodified reference."""
    import json
    import logging
    from conftest import GOLDEN_DIR
    from distributed_cluster_gpus_b200.configs import paper_config as pc
    from distributed_cluster_gpus_b200.simcore.simulator_paper_multi import MultiIngressPaperSimulator
    with open(os.path.join(GOLDEN_DIR, "kat.json")) as f:
        kat = json.load(f)["survey_known_answers"]
    for name, k in kat.items():
        sc = SC.BY_NAME[name]
        kw = SC.build_inputs(sc)
        sim = MultiIngressPaperSimulator(router_policy=pc.build_router_policy(), logger=logging.getLogger("t"),
                                         sim_duration=sc["duration"], log_interval=sc["log_interval"], log_path=str(tmp_path),
                                         rng_seed=123, algo=sc["algo"], show_progress=False, replicas=2, write_logs=False,
                                         rng="mt19937", **kw).run()
        assert int(sim.summary[0, S.S_EVENTS]) == k["expected"]["events"], name
        if "jobs" in k["expected"]:
            assert int(sim.summary[0, S.S_JOBS_FINISHED]) == k["expected"]["jobs"], name
        total = sum(dc.energy_joules for dc in kw["dcs"].values())      # what the survey printed (builtin sum)
        want = float(k["expected"]["total_energy_repr"])
        assert abs(total - want) <= RTOL * want, (name, total, want)


def test_set_rng_rejects_bad_use():
    from distributed_cluster_gpus_b200 import _native as N
    with engine_cls()(SC.to_spec(dict(SC.CFG3, duration=5.0)), 2, base_seed=1) as eng:
        with pytest.raises(ValueError):
            eng.set_rng("xorshift")
        eng.set_rng("mt19937")
        eng.advance(10)
        with pytest.raises(N.DcsimError):
            eng.set_rng("philox")      # the batch has started


def _full_batch_parity(oracle, name, n, seed):
    sc = SC.BY_NAME[name]
    sp = SC.to_spec(sc)
    with engine_cls()(sp, n, base_seed=seed) as eng:
        total = eng.advance(0)
        got = eng.summary()
        info = eng.launch_info()
    want, want_total = oracle.run_batch(sp.to_bytes(), n, seed, 0, n_threads=os.cpu_count() or 1)
    assert total == want_total
    worst = assert_rows_match(got, want, sc["n_dc"])
    print(f"{name}: ALL {n} replicas, {total} events, worst float rel err {worst:.2e}, "
          f"{info['resident_warps_per_sm']} warps/SM, staging mode {info['staging_mode']}")


def test_bench_batch_matches_oracle_replica_by_replica(oracle):
    """The bench workload at bench size: all 65 536 replicas of 4 DC x 64 / 120 s against the (threaded) oracle — every
    count exact, every float of every replica's summary within 1e-9."""
    _full_batch_parity(oracle, "cfg3_4x64_sinusoid_120s", 65536, 123)


def test_cfg5_batch_matches_oracle_replica_by_replica(oracle):
    """8 DC x 256 (head-staged launch mode: running-job records in HBM/L2), 4096 replicas, full duration."""
    _full_batch_parity(oracle, "cfg5_8x256_sinusoid_60s", 4096, 777)


def test_recorder_overflow_is_reported_not_truncated(tmp_path):
    """A job / cluster log that does not fit its recorder raises (with the row count the device saw) instead of
    handing back a truncated prefix; the drop-in re-runs the logged replica at that size."""
    import csv
    import logging
    from distributed_cluster_gpus_b200.engine import RecorderOverflow
    from distributed_cluster_gpus_b200.configs import paper_config as pc
    from distributed_cluster_gpus_b200.simcore.simulator_paper_multi import MultiIngressPaperSimulator
    sc = SC.BY_NAME["ragged_3dc_12_5_40"]
    sp = SC.to_spec(sc)
    with engine_cls()(sp, 2, base_seed=3) as eng:
        eng.set_logging(1, 50, 9)
        eng.advance(0)
        fin = int(eng.summary()[1, S.S_JOBS_FINISHED])
        with pytest.raises(RecorderOverflow) as ei:
            eng.job_log()
        assert ei.value.needed == fin and ei.value.capacity == 50
        with pytest.raises(RecorderOverflow):
            eng.cluster_log()
    kw = SC.build_inputs(sc)
    sim = MultiIngressPaperSimulator(router_policy=pc.build_router_policy(), logger=logging.getLogger("t"),
                                     sim_duration=sc["duration"], log_interval=sc["log_interval"], log_path=str(tmp_path),
                                     rng_seed=3, algo=sc["algo"], show_progress=False, replicas=4, keep_engine=False, **kw)
    sim._log_one_replica(sim._spec, 40, 7)                            # far too small: must grow, not truncate
    rows = list(csv.reader(open(sim.job_log_path)))
    with engine_cls()(sp, 1, base_seed=3) as eng:
        eng.advance(0)
        assert len(rows) - 1 == int(eng.summary()[0, S.S_JOBS_FINISHED])


def _run_cli(args, env_extra=None, timeout=900):
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, **(env_extra or {}))
    env["PYTHONPATH"] = root + os.pathsep + env.get("PYTHONPATH", "")
    return subprocess.run([sys.executable, "-m", "distributed_cluster_gpus_b200.run_sim_paper"] + args, capture_output=True,
                          text=True, timeout=timeout, cwd=root, env=env)


def test_cli_sharded_over_ranks_is_invariant(tmp_path):
    """`run_sim_paper --gpus 2`: two ranks (one process per GPU; on a one-GPU box both share it and talk over gloo),
    replicas sharded by global id, one all-reduce of the aggregate.  Statistics and replica 0's CSVs must equal the
    single-process run's."""
    import json
    import torch
    common = ["--duration", "20", "--inf-mode", "sinusoid", "--inf-rate", "10", "--inf-period", "3600", "--trn-rate", "1",
              "--n-dc", "4", "--gpus-per-dc", "64", "--replicas", "301", "--seed", "77", "--progress", ""]
    one = _run_cli(common + ["--log-path", str(tmp_path / "one" / "x"), "--summary-json", str(tmp_path / "one.json")])
    assert one.returncode == 0, one.stderr[-2000:]
    extra = {} if torch.cuda.device_count() >= 2 else {"DCSIM_DIST_BACKEND": "gloo"}
    two = _run_cli(common + ["--gpus", "2", "--log-path", str(tmp_path / "two" / "x"), "--summary-json", str(tmp_path / "two.json")], extra)
    assert two.returncode == 0, two.stderr[-3000:]
    a, b = json.load(open(tmp_path / "one.json")), json.load(open(tmp_path / "two.json"))
    assert b["gpus"] == 2 and a["replicas"] == b["replicas"] == 301
    assert a["events_total"] == b["events_total"] and a["jobs_finished_total"] == b["jobs_finished_total"]
    for k in ("energy_j_mean", "mean_latency_s_mean", "energy_j_ci95", "mean_latency_s_ci95"):
        assert abs(a[k] - b[k]) <= 1e-9 * abs(a[k]), k
    for k in ("energy_j_p05_p50_p95", "mean_latency_s_p05_p50_p95"):
        assert np.allclose(a[k], b[k], rtol=1e-12), k
    for f in ("job_log.csv", "cluster_log.csv"):
        assert open(tmp_path / "one" / "x" / f).read() == open(tmp_path / "two" / "x" / f).read(), f
