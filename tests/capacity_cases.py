"""TEST-ONLY: the capacity-edge cases shared by tests/test_capacity_edges.py (host build) and
tests/test_gpu_capacity_edges.py (kernels).

Every per-replica structure of the event loop has a fixed capacity; a replica that would exceed one sets a status bit,
refuses the write and stops at its next 16-event poll (DESIGN.md §3).  Each case sets one capacity so that the batch
sits exactly at it (the cap is replica n-1's need, so the last replica's buffers end at the end of the allocation) or
straddles it (some replicas of a warp flagged, their warp-mates not).  The oracle has no capacities: it says what each
replica needs (S_MAX_Q, S_MAX_RUN, S_JOBS_CREATED) and at which event a replica first needs more than it is given.
The seq ring and the stale pool have no oracle column; their flag sets come from the host build of the device core.
"""
import os

import numpy as np

from distributed_cluster_gpus_b200 import scenarios as SC, spec as S

N = 7   # 8 lanes: two warps of 4 + 3 replicas (one ghost); 16: four warps, the last with one ghost; 32: one per warp

# 1 DC x 8 GPUs, one job at a time, Poisson inference near saturation: the queue forms and drains over and over (short
# queues, thousands of dequeues).  The 20 ms cluster log is what proves it: its queue lengths bound the dequeues.
FIFO_CHURN = SC.scenario("fifo_churn_1x8_poisson32", 1, 8, SC.POI(32.0), SC.OFF, 120.0, SC.FREQ8, log_interval=0.02)
# debug algo, one GPU per job on 4 x 64: running sets of 14..25 jobs, different per replica
DEBUG_N1 = SC.scenario("debug_n1_4x64_sin6", 4, 64, dict(SC.SIN10, rate=6.0), SC.POI(0.2), 60.0, SC.FREQ3, algo="debug",
                       num_fixed_gpus=1)
CFG3_30 = dict(SC.CFG3, duration=30.0)
CFG3_30_SIN7 = dict(SC.CFG3, duration=30.0, inf=dict(SC.SIN10, rate=7.0))   # list distances straddle a 32-entry seq ring

# which need a capacity bounds: the oracle's summary column (None: the host build decides) and the status bit
KINDS = {"queue": (S.S_MAX_Q, S.ST_QUEUE_OVERFLOW), "run": (S.S_MAX_RUN, S.ST_RUN_OVERFLOW),
         "arrivals": (S.S_JOBS_CREATED, S.ST_ARRIVALS_OVERFLOW), "xfer": (None, S.ST_XFER_OVERFLOW),
         "stale": (None, S.ST_STALE_OVERFLOW)}


def _case(name, sc, seed, kind, cap=None, mixed=False, min_wraps=0, exact=False):
    """cap None: replica n-1's need (exact).  mixed: the batch must hold flagged and unflagged replicas."""
    return dict(name=name, sc=sc, seed=seed, kind=kind, cap=cap, mixed=mixed, min_wraps=min_wraps, exact=exact)


CASES = [
    _case("fifo_exact", FIFO_CHURN, 123, "queue", min_wraps=3, exact=True),
    _case("fifo_mixed", CFG3_30, 124, "queue", cap="median", mixed=True),
    _case("run_exact_8", CFG3_30, 123, "run", exact=True),                 # every replica fills its 8 records
    _case("run_below_lanes", CFG3_30, 123, "run", cap=4),                   # 4 records: fewer than any lane group
    _case("run_mixed_20", DEBUG_N1, 123, "run", cap=20, mixed=True),        # 20: not a multiple of 8, 16 or 32
    _case("arrivals_exact", FIFO_CHURN, 125, "arrivals", exact=True),
    _case("arrivals_mixed", CFG3_30, 123, "arrivals", cap="median", mixed=True),
    _case("xfer_mixed", CFG3_30_SIN7, 123, "xfer", cap=16, mixed=True),     # seq ring of 32 entries
    _case("stale_cap_greedy", SC.BY_NAME["cap_greedy_4x64"], 123, "stale", cap=1),   # rounds up to a pool of 4
]
BY_NAME = {c["name"]: c for c in CASES}
CAP_KEYS = {"queue": ("cap_q_inf", "cap_q_trn"), "run": ("cap_run",), "arrivals": ("cap_arrivals",),
            "xfer": ("cap_xfer",), "stale": ("cap_stale",)}


def is_cap_case(case):
    """Runs the power-cap controller's build of the event loop."""
    return case["sc"]["algo"] == "cap_greedy" and case["sc"]["power_cap"] > 0


def oracle_batch(oracle, case):
    """(summaries, total events) of the case's batch on the oracle (capacities play no part there)."""
    sp = SC.to_spec(case["sc"])
    return oracle.run_batch(sp.to_bytes(), N, case["seed"], 0, n_threads=os.cpu_count() or 1)


def needs(case, want):
    """Per-replica need of the case's capacity, from the oracle's summaries (None where the oracle has no column)."""
    col = KINDS[case["kind"]][0]
    return None if col is None else want[:, col].astype(np.int64)


def requested_cap(case, want):
    cap = case["cap"]
    if cap is None:
        return int(needs(case, want)[N - 1])
    if cap == "median":
        return int(np.median(needs(case, want)))
    return int(cap)


def caps_dict(case, want):
    c = requested_cap(case, want)
    assert c >= 1, "0 means the library default"
    return {k: c for k in CAP_KEYS[case["kind"]]}


def spec(case, want, extra=None):
    return SC.to_spec(case["sc"], caps=dict(caps_dict(case, want), **(extra or {})))


def effective_cap(case, sp):
    """What the library makes of the requested capacity (dcsim_make_layout): cap_run and cap_stale round up to a multiple
    of 4, the seq ring is the next power of two >= 2 * cap_xfer (of which cap_xfer reports half), the FIFOs and the
    arrival list are taken as given."""
    kind = case["kind"]
    if kind == "queue":
        assert sp.cap_q_inf == sp.cap_q_trn
        return sp.cap_q_inf
    if kind == "run":
        return (sp.cap_run + 3) & ~3
    if kind == "stale":
        return (sp.cap_stale + 3) & ~3
    if kind == "xfer":
        ring = 8
        while ring < 2 * sp.cap_xfer:
            ring <<= 1
        return ring // 2
    return sp.cap_arrivals


def predicted_flags(case, want, eff, host_status=None):
    """Rule 1: replica r is flagged iff its need exceeds the effective capacity.  Kinds without an oracle column take the
    host build's status (host_status) instead."""
    n = needs(case, want)
    if n is None:
        bit = KINDS[case["kind"]][1]
        return (host_status.astype(np.int64) & bit) != 0
    return n > eff


def first_exceeding_event(oracle, case, eff, replica):
    """k: the 1-based index of the event after which the oracle's need first exceeds `eff` (stepping one event at a
    time).  Arrival-list overflows are raised by the pre-pass, before any event: k = 0."""
    col, _ = KINDS[case["kind"]]
    if case["kind"] == "arrivals":
        return 0
    sim = oracle.OracleSim(SC.to_spec(case["sc"]).to_bytes(), case["seed"] + int(replica))
    try:
        k = 0
        while True:
            done = sim.advance(1)
            k += 1
            if sim.summary()[col] > eff:
                return k
            assert not done, f"{case['name']}: replica {replica} never exceeds {eff}"
    finally:
        sim.close()


def ring_wraps(oracle, case, replica, cap):
    """Lower bound on how often one FIFO ring of `replica` wrapped at capacity `cap`: per (DC, queue), the enqueues are at
    least the drops of its length between consecutive cluster-log ticks plus its final length; the ring wrapped at least
    floor(bound / cap) times.  Returns the largest over the replica's rings."""
    sc = case["sc"]
    rows = int(sc["duration"] / sc["log_interval"] + 2) * sc["n_dc"]
    sim = oracle.OracleSim(SC.to_spec(sc).to_bytes(), case["seed"] + int(replica), clog_cap=rows)
    try:
        sim.advance(0)
        cl, final = sim.cluster_log(), sim.summary()
    finally:
        sim.close()
    assert len(cl) < rows
    best = 0
    for d in range(sc["n_dc"]):
        for field, sd in (("q_inf", S.SD_Q_INF), ("q_train", S.SD_Q_TRN)):
            q = cl[cl["dc"] == d][field].astype(np.int64)
            bound = int(np.maximum(q[:-1] - q[1:], 0).sum()) + int(final[S.S_DC0 + d * S.S_DC_STRIDE + sd])
            best = max(best, bound // cap)
    return best
