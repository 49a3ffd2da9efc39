"""Every instantiation of the event-loop kernel against the oracle.

The library ships 18 builds of dcsim_advance_kernel (dcsim_advance_impl.cuh): 32 / 16 / 8 lanes per replica x what is
staged in shared memory (the whole state block, its head only, nothing) x the power-cap controller compiled in or not.
The default pick (dcsim_b200.cu size_launch) reaches only some of them on ordinary scenarios, so each one is forced here:
the lanes with DCSIM_GROUP, the staging with DCSIM_RECORDS, and "nothing staged" with a seq ring too large for any
CTA's shared memory (cap_xfer = 20000: a 256 kB head).  Every cell checks that launch_info() reports the kernel it
asked for, so a quiet fall-back to another build fails instead of passing.

Replica counts leave the last warp part-empty: its lane groups without a replica run the loop as ghosts next to
replica n-1 — with nothing staged, on that replica's own block in HBM.  Replica n-1 is also the one traced and logged.
"""
import os

import numpy as np
import pytest

from conftest import has_cuda
from test_gpu_parity import assert_rows_match
from distributed_cluster_gpus_b200 import scenarios as SC

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")]

INPLACE, STAGED, HEAD = 0, 1, 2          # DCSIM_MODE_* (dcsim_advance_impl.cuh) as launch_info() reports them
MODE_NAMES = {INPLACE: "INPLACE", STAGED: "STAGED", HEAD: "HEAD"}
BIG_XFER = {"cap_xfer": 20000}           # seq ring of 32768 entries: the head no longer fits a CTA's shared memory
SEED = 123
TRACE_CAP, JOBS_CAP, CLUSTER_CAP = 6000, 40000, 4000


def _cases(lanes, cap):
    """(label, scenario, replicas).  Replica counts leave the last warp part-empty: 8 lanes -> 37 or 7 (4 replicas per
    warp), 16 -> 5 (2 per warp), 32 -> 3 (a warp each).  cap_greedy_4x64 runs in full and keeps to replicas 0..7 of seed
    123, the batch the plain parity test runs (the conditioning class of DESIGN.md §6a does not arise there)."""
    n = {8: 7, 16: 5, 32: 3}[lanes]
    if cap:
        return [("cap_greedy_4x64", dict(SC.BY_NAME["cap_greedy_4x64"]), n)]
    return [("cfg3_4x64 / 60 s", dict(SC.CFG3, duration=60.0), 37 if lanes == 8 else n),
            ("cfg5_8x256_sinusoid_60s", dict(SC.BY_NAME["cfg5_8x256_sinusoid_60s"]), n)]


def _force(monkeypatch, lanes, mode):
    monkeypatch.setenv("DCSIM_GROUP", str(lanes))
    if mode == INPLACE:
        monkeypatch.delenv("DCSIM_RECORDS", raising=False)
    else:
        monkeypatch.setenv("DCSIM_RECORDS", "shared" if mode == STAGED else "global")


def _check_launch(info, lanes, mode, cap, what):
    got = (info["lanes_per_replica"], info["staging_mode"])
    assert got == (lanes, mode), f"{what}: asked for ({lanes}, {MODE_NAMES[mode]}), launched {got}"
    print(f"launch ({info['lanes_per_replica']}, {MODE_NAMES[info['staging_mode']]}, cap={int(cap)}) {what}: "
          f"regs={info['regs_per_thread']} warps/SM={info['resident_warps_per_sm']} "
          f"smem/CTA={info['smem_bytes_per_cta']}")


def assert_recorders_match(tr, jobs, cl, sim):
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


@pytest.mark.parametrize("cap", [False, True], ids=["nocap", "cap"])
@pytest.mark.parametrize("mode", [STAGED, HEAD, INPLACE], ids=["staged", "head", "inplace"])
@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_launch_mode_matches_oracle(oracle, monkeypatch, lanes, mode, cap):
    """One shot (lean records), then in chunks of 61 events with replica n-1 traced and logged (full records,
    stage-out / stage-in between launches): every summary against the oracle, the recorders against OracleSim."""
    from distributed_cluster_gpus_b200.engine import BatchedEngine
    _force(monkeypatch, lanes, mode)
    for label, sc, n in _cases(lanes, cap):
        sp = SC.to_spec(sc, caps=BIG_XFER if mode == INPLACE else None)
        assert (sp.cap_stale != 0) == cap
        blob = sp.to_bytes()
        want, want_total = oracle.run_batch(blob, n, SEED, 0, n_threads=os.cpu_count() or 1)
        what = f"{label}, {n} replicas"
        with BatchedEngine(sp, n, base_seed=SEED) as eng:
            total = eng.advance(0)
            got = eng.summary()
            _check_launch(eng.launch_info(), lanes, mode, cap, what + " one-shot")
        assert total == want_total
        assert_rows_match(got, want, sc["n_dc"])
        with BatchedEngine(sp, n, base_seed=SEED) as eng:
            eng.set_trace(n - 1, TRACE_CAP)
            eng.set_logging(n - 1, JOBS_CAP, CLUSTER_CAP)
            total, guard = 0, 0
            while not eng.all_done():
                total += eng.advance(61)
                guard += 1
                assert guard < 5000
            got = eng.summary()
            _check_launch(eng.launch_info(), lanes, mode, cap, what + " chunked+logged")
            tr, jobs, cl = eng.trace(), eng.job_log(), eng.cluster_log()
        assert total == want_total
        assert_rows_match(got, want, sc["n_dc"])
        sim = oracle.OracleSim(blob, SEED + n - 1, trace_cap=TRACE_CAP, joblog_cap=JOBS_CAP, clog_cap=CLUSTER_CAP)
        sim.advance(0)
        assert_recorders_match(tr, jobs, cl, sim)
        sim.close()


def test_transfer_overflow_retry_lands_in_place(oracle, monkeypatch):
    """run_to_completion: a first attempt whose seq ring is too small flags XFER_OVERFLOW; the retry asks for a larger
    cap_xfer, gets 20000 — a head too large for shared memory — and runs with nothing staged.  Its summary must be
    the oracle's."""
    from distributed_cluster_gpus_b200.engine import free_cached_engine, run_to_completion
    monkeypatch.delenv("DCSIM_GROUP", raising=False)
    monkeypatch.delenv("DCSIM_RECORDS", raising=False)
    sc = dict(SC.CFG3, duration=60.0)
    n = 37
    calls = []

    def factory(caps):
        calls.append(dict(caps))
        return SC.to_spec(sc, caps=BIG_XFER if "cap_xfer" in caps else {"cap_xfer": 8})
    free_cached_engine()
    eng, summ = run_to_completion(factory, n, SEED)
    try:
        info = eng.launch_info()
    finally:
        eng.close()
    assert len(calls) == 2 and "cap_xfer" in calls[1], calls
    assert (info["lanes_per_replica"], info["staging_mode"]) == (8, INPLACE), info
    want, _ = oracle.run_batch(SC.to_spec(sc, caps=BIG_XFER).to_bytes(), n, SEED, 0, n_threads=os.cpu_count() or 1)
    assert_rows_match(summ, want, sc["n_dc"])
    print(f"retry after XFER_OVERFLOW: cap_xfer {info['cap_xfer']}, ({info['lanes_per_replica']}, "
          f"{MODE_NAMES[info['staging_mode']]}) regs={info['regs_per_thread']} warps/SM={info['resident_warps_per_sm']}")


def test_parked_engine_is_not_reused_under_another_lane_count(monkeypatch):
    """The parked engine of run_to_completion was sized under one DCSIM_GROUP: a run under another must get a fresh one."""
    from distributed_cluster_gpus_b200 import engine as E
    sp = SC.to_spec(dict(SC.CFG3, duration=5.0))
    monkeypatch.delenv("DCSIM_RECORDS", raising=False)
    E.free_cached_engine()
    lanes = []
    for g in ("8", "32", "32"):
        monkeypatch.setenv("DCSIM_GROUP", g)
        eng, _ = E.run_to_completion(lambda caps: sp, 3, 1)
        lanes.append(eng.launch_info()["lanes_per_replica"])
        E.release_engine(eng, sp)
    E.free_cached_engine()
    assert lanes == [8, 32, 32]
