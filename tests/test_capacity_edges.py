"""Capacities at their exact limit, on the host build of the device core (plain and the lane-group loop skeleton)
against the oracle: the rules tests/test_gpu_capacity_edges.py then holds the kernels to.

  1. replica r is flagged iff its need (oracle) exceeds the effective capacity, and then with exactly that one bit;
  2. unflagged replicas equal the oracle on every summary column but S_MAX_XFER (the device keeps no transfer pool);
  3. a flagged replica stops at its next 16-event poll: k <= S_EVENTS <= 16 * ceil(k / 16), k the oracle's first event
     that needs more (it may reach end_time inside that chunk: DONE = 1 with the bit set);
  4. an arrival-list (or seq-ring) overflow is raised before the first event: 0 events, DONE = 0.
"""
import numpy as np
import pytest

import capacity_cases as CC
from distributed_cluster_gpus_b200 import spec as S


def check_flags_and_stops(case, got, pred, ks, last_event):
    """Rules 1, 3 and 4 on one batch's summaries `got`; `last_event(k)` is the last event a replica flagged at event k
    may have processed."""
    bit = CC.KINDS[case["kind"]][1]
    status = got[:, S.S_STATUS].astype(np.int64)
    assert np.array_equal(status != 0, pred), (case["name"], status, pred)
    assert np.all(status[pred] == bit), (case["name"], status)
    events = got[:, S.S_EVENTS].astype(np.int64)
    for r in np.flatnonzero(pred):
        if case["kind"] in ("arrivals", "xfer"):
            assert events[r] == 0 and got[r, S.S_DONE] == 0, (case["name"], r, events[r])
        else:
            k = ks[r]
            assert k <= events[r] <= last_event(k), (case["name"], r, k, events[r])


def prepare(oracle, hostemu, case):
    """(oracle summaries, spec, effective cap, predicted flags, {flagged replica: k})."""
    want, _ = CC.oracle_batch(oracle, case)
    sp = CC.spec(case, want)
    eff = CC.effective_cap(case, sp)
    host_status = None
    if CC.needs(case, want) is None:
        host_status = hostemu.run_batch(sp.to_bytes(), CC.N, case["seed"])["summary"][:, S.S_STATUS]
    pred = CC.predicted_flags(case, want, eff, host_status)
    ks = {int(r): CC.first_exceeding_event(oracle, case, eff, int(r)) for r in np.flatnonzero(pred)} \
        if case["kind"] not in ("xfer", "stale") else {}
    return want, sp, eff, pred, ks


@pytest.mark.parametrize("uniform", [False, True], ids=["plain", "uniform"])
@pytest.mark.parametrize("name", [c["name"] for c in CC.CASES])
def test_capacity_edge_on_host_build(oracle, hostemu, name, uniform):
    case = CC.BY_NAME[name]
    want, sp, eff, pred, ks = prepare(oracle, hostemu, case)
    got = hostemu.run_batch(sp.to_bytes(), CC.N, case["seed"], uniform=uniform)
    layout = got["layout"]
    if case["kind"] == "run":
        assert layout["cap_run"] == eff
    elif case["kind"] == "queue":
        assert layout["cap_q_inf"] == layout["cap_q_trn"] == eff
    elif case["kind"] == "xfer":
        assert layout["cap_xfer"] == eff
    summ = got["summary"]
    check_flags_and_stops(case, summ, pred, ks, lambda k: 16 * -(-k // 16))
    cols = [c for c in range(want.shape[1]) if c != S.S_MAX_XFER]     # (the device keeps no in-flight-transfer pool)
    ok = ~pred
    assert np.array_equal(summ[ok][:, cols], want[ok][:, cols]), (name, np.argwhere(summ[ok][:, cols] != want[ok][:, cols])[:6])
    if case["mixed"]:
        assert 0 < pred.sum() < CC.N, (name, pred)
    if case["exact"]:
        assert CC.needs(case, want)[CC.N - 1] == eff and not pred[CC.N - 1]
    if name == "fifo_mixed":
        assert pred[CC.N - 1]          # the replica the GPU test traces is one of the flagged
    if case["kind"] == "stale":
        assert eff == 4 and sp.cap_stale == 1
        assert np.any(want[:, S.S_EV_FINISH] > want[:, S.S_JOBS_FINISHED])   # superseded job_finish events did occur
    print(f"{name} ({'uniform' if uniform else 'plain'}): cap {eff}, flagged {np.flatnonzero(pred).tolist()}, k {ks}")


def test_fifo_exact_case_wraps_its_ring(oracle):
    """The FIFO-exact case runs replica n-1's queue at exactly its capacity AND wraps that ring at least three times (the
    tail -= cap / head -> 0 paths of dcsim_enqueue / dcsim_dequeue)."""
    case = CC.BY_NAME["fifo_exact"]
    want, _ = CC.oracle_batch(oracle, case)
    cap = CC.requested_cap(case, want)
    wraps = CC.ring_wraps(oracle, case, CC.N - 1, cap)
    print(f"fifo_exact: replica {CC.N - 1} at {cap} entries, its ring wrapped >= {wraps} times")
    assert wraps >= 3


def test_arrivals_exact_case_fills_the_merged_list(oracle):
    """Replica n-1 of the arrival-exact case has exactly cap_arrivals arrivals, each with its xfer_done inside the run:
    its merged event list uses all 2 * cap_arrivals slots."""
    case = CC.BY_NAME["arrivals_exact"]
    want, _ = CC.oracle_batch(oracle, case)
    row = want[CC.N - 1]
    assert row[S.S_JOBS_CREATED] == CC.requested_cap(case, want) == row[S.S_EV_XFER]
