"""Events at the SAME instant on the device: the cases of test_event_ties.py, run by the CUDA kernels.

A continuous clock all but never produces ties, so the device code that resolves them — the list merge's positions
(window walks with push-order tie-breaking), the pre-pass's stream ranks, the lane-group pop-min over (t, seq) — would
otherwise never meet one on the GPU.  The product library has no hook to provoke them; two TEST-ONLY builds of the same
sources do (__graft_entry__.TEST_HOOK_LIBS, -DDCSIM_DEVICE_TEST_HOOKS): dcsim_test_set_time_quantum(q) rounds every
arrival and xfer_done instant up to a multiple of q, exactly as the oracle's hook does.  The second build also cuts the
list merge's ring to one chunk, so that its HBM fall-back paths meet the ties too.

The package loads its library once per process, so every run of a hook build happens in a child process
(tests/hook_child.py, DCSIM_B200_LIB naming the build); the child writes summaries and recorders as .npy, the parent
checks them against the oracle under the same quantum.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, has_cuda
from hook_child import CLUSTER_CAP, JOBS_CAP, TRACE_CAP
from test_event_ties import CASES
from test_gpu_launch_modes import assert_recorders_match
from test_gpu_parity import assert_rows_match
from distributed_cluster_gpus_b200 import scenarios as SC

CHILD_TIMEOUT_S = 900
QUANTA = [2.0 ** -5, 0.25, 1.0]
LANE_CASES = ["cfg3_4x64_sinusoid_120s", "cap_greedy_4x64"]
FALLBACK_CASES = ["cfg3_4x64_sinusoid_120s", "cfg5_8x256_sinusoid_60s", "ragged_3dc_12_5_40", "sweep_eco_route"]
N_REPLICAS = 7
TIE_SEED, FALLBACK_SEED = 900, 31
INERT_CASE = "ragged_3dc_12_5_40"


def _spec(name, max_duration):
    sc = dict(SC.BY_NAME[name])
    sc["duration"] = min(sc["duration"], max_duration)
    return sc, SC.to_spec(sc, caps={"cap_xfer": 4096})   # coarse clocks pile transfers up: give the seq ring room


def _tie_jobs():
    """(id, name, max_duration, q, seed, lanes, chunk) of every run of the hook build."""
    jobs = [(f"ties_{name}_{q}", name, 60.0, q, TIE_SEED, 0, 0) for name in CASES for q in QUANTA]
    jobs += [(f"lanes{g}_{name}", name, 60.0, 0.25, TIE_SEED, g, 7) for name in LANE_CASES for g in (8, 16, 32)]
    jobs += [("inert", INERT_CASE, 60.0, 0.0, TIE_SEED, 0, 0)]
    return jobs


def _fallback_jobs():
    return [(f"fallback_{name}_{q}", name, 40.0, q, FALLBACK_SEED, 0, 0) for name in FALLBACK_CASES for q in (0.0, 0.25)]


@pytest.fixture(scope="session")
def hook_libs():
    """The TEST-ONLY hook builds, compiled here when missing or stale (a failure fails the tests, never skips them)."""
    import __graft_entry__
    __graft_entry__.build_test_hooks()
    return list(__graft_entry__.TEST_HOOK_LIBS)


def _run_child(lib, jobs, tmp):
    os.makedirs(tmp, exist_ok=True)
    entries = []
    for jid, name, max_duration, q, seed, lanes, chunk in jobs:
        _, sp = _spec(name, max_duration)
        blob = os.path.join(tmp, jid + ".spec")
        with open(blob, "wb") as f:
            f.write(sp.to_bytes())
        entries.append({"id": jid, "blob": blob, "q": q, "seed": seed, "n": N_REPLICAS, "lanes": lanes, "chunk": chunk})
    with open(os.path.join(tmp, "jobs.json"), "w") as f:
        json.dump(entries, f)
    env = dict(os.environ, DCSIM_B200_LIB=lib)
    env.pop("DCSIM_GROUP", None)
    env.pop("DCSIM_RECORDS", None)
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "hook_child.py"), os.path.join(tmp, "jobs.json"), tmp], env=env,
                         capture_output=True, text=True, timeout=CHILD_TIMEOUT_S, cwd=ROOT)
    assert res.returncode == 0, f"child run of {os.path.basename(lib)} failed:\n{res.stdout[-3000:]}\n{res.stderr[-6000:]}"
    out = {}
    for jid, *_ in jobs:
        base = os.path.join(tmp, jid)
        out[jid] = {k: np.load(f"{base}_{k}.npy") for k in ("summary", "trace", "jobs", "cluster")}
        with open(base + ".json") as f:
            out[jid].update(json.load(f))
    return out


@pytest.fixture(scope="module")
def tie_runs(hook_libs, tmp_path_factory):
    return _run_child(hook_libs[0], _tie_jobs(), str(tmp_path_factory.mktemp("ties")))


@pytest.fixture(scope="module")
def fallback_runs(hook_libs, tmp_path_factory):
    return _run_child(hook_libs[1], _fallback_jobs(), str(tmp_path_factory.mktemp("fallback")))


@pytest.fixture
def quantum(oracle):
    yield oracle.set_test_time_quantum
    oracle.set_test_time_quantum(0.0)


def test_only_the_hook_builds_export_the_quantum_hook(hook_libs):
    from distributed_cluster_gpus_b200 import _native
    product = os.path.join(ROOT, "distributed_cluster_gpus_b200", "csrc", "libdcsim_b200.so")
    assert not hasattr(C.CDLL(product), "dcsim_test_set_time_quantum")
    for lib in hook_libs:
        L = C.CDLL(lib)
        assert hasattr(L, "dcsim_test_set_time_quantum"), lib
        assert all(hasattr(L, name) for name in _native.EXPORTS), lib


def _check_against_oracle(oracle, quantum, run, name, max_duration, q, seed):
    """Summaries (counts exact, S_SEQ included; floats 1e-9), the traced replica's trace (kind and seq exact, t 1e-12)
    and its logs (integer fields exact) against the oracle under the same quantum.  Returns the tie count."""
    sc, sp = _spec(name, max_duration)
    blob = sp.to_bytes()
    quantum(q)
    want, want_total = oracle.run_batch(blob, N_REPLICAS, seed, 0, n_threads=os.cpu_count() or 1)
    assert run["events"] == want_total
    assert_rows_match(run["summary"], want, sc["n_dc"])
    sim = oracle.OracleSim(blob, seed + N_REPLICAS - 1, trace_cap=TRACE_CAP, joblog_cap=JOBS_CAP, clog_cap=CLUSTER_CAP)
    sim.advance(0)
    ties = int(np.count_nonzero(np.diff(sim.trace()["t"]) == 0.0))
    assert_recorders_match(run["trace"], run["jobs"], run["cluster"], sim)
    sim.close()
    return ties


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("q", QUANTA)
@pytest.mark.gpu
@pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")
def test_same_instant_events_on_device(oracle, quantum, tie_runs, name, q):
    run = tie_runs[f"ties_{name}_{q}"]
    ties = _check_against_oracle(oracle, quantum, run, name, 60.0, q, TIE_SEED)
    li = run["launch"]
    print(f"{name} q={q}: {ties} tied instants in the traced replica's first {len(run['trace'])} events, "
          f"{run['events']} events, launch ({li['lanes_per_replica']}, mode {li['staging_mode']})")
    assert ties > 50, "the hook is supposed to make ties common"


@pytest.mark.parametrize("lanes", [8, 16, 32])
@pytest.mark.parametrize("name", LANE_CASES)
@pytest.mark.gpu
@pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")
def test_same_instant_events_on_every_lane_count(oracle, quantum, tie_runs, name, lanes):
    """Ties through the lane-group pop-min of each build (8 / 16 lanes: shuffle butterflies over (hi, lo, seq|slot)),
    7 replicas (ghost lane groups next to the traced replica 6), in chunks of 7 events."""
    run = tie_runs[f"lanes{lanes}_{name}"]
    assert run["launch"]["lanes_per_replica"] == lanes
    ties = _check_against_oracle(oracle, quantum, run, name, 60.0, 0.25, TIE_SEED)
    print(f"{name} on {lanes} lanes, chunks of 7: {ties} tied instants, {run['events']} events")
    assert ties > 50


@pytest.mark.parametrize("name", FALLBACK_CASES)
@pytest.mark.parametrize("q", [0.0, 0.25])
@pytest.mark.gpu
@pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")
def test_merge_fallback_paths_on_device(oracle, quantum, fallback_runs, name, q):
    """The list merge built with a ring of one chunk: nearly every scan reads HBM; results must not change."""
    run = fallback_runs[f"fallback_{name}_{q}"]
    ties = _check_against_oracle(oracle, quantum, run, name, 40.0, q, FALLBACK_SEED)
    print(f"small ring, {name} q={q}: {ties} tied instants, {run['events']} events")


@pytest.mark.gpu
@pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")
def test_hook_is_inert_when_off(tie_runs):
    """Quantum 0: the hook build computes bit for bit what the product library does."""
    from distributed_cluster_gpus_b200.engine import BatchedEngine
    run = tie_runs["inert"]
    _, sp = _spec(INERT_CASE, 60.0)
    with BatchedEngine(sp, N_REPLICAS, base_seed=TIE_SEED) as eng:
        eng.set_trace(N_REPLICAS - 1, TRACE_CAP)
        eng.set_logging(N_REPLICAS - 1, JOBS_CAP, CLUSTER_CAP)
        total = eng.advance(0)
        got, tr = eng.summary(), eng.trace()
    assert total == run["events"]
    assert np.array_equal(got, run["summary"])
    assert np.array_equal(tr, run["trace"])
