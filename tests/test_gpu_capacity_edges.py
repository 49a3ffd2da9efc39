"""Capacities at their exact limit on the kernels: every case of tests/capacity_cases.py in every forced launch cell
(8 / 16 / 32 lanes x whole block / head / nothing staged; the power-cap controller's cells run the stale-pool case).

Per case and cell: the flag set is the one the oracle's needs predict (the host build's for the seq ring and the stale
pool), each flagged row holds exactly the one bit; unflagged rows equal the oracle; a flagged replica stops within its
16-event chunk (one shot) or within 15 events of the first one that needs more (in chunks of 61 and of 7, where
all_done() must still terminate); the traced replica n-1 follows OracleSim up to that event; the on-device reduction
counts the flagged replicas as failed and none as running; run_to_completion retries a mixed batch exactly once and
then equals the oracle on every replica.  The seq-ring case does not run with nothing staged: a seq ring too large for
shared memory is what forces that mode.
"""
import numpy as np
import pytest

import capacity_cases as CC
from conftest import has_cuda
from test_capacity_edges import check_flags_and_stops, prepare
from test_gpu_launch_modes import BIG_XFER, HEAD, INPLACE, STAGED, _check_launch, _force
from test_gpu_parity import assert_rows_match
from distributed_cluster_gpus_b200 import sharding, spec as S

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not has_cuda(), reason="needs a CUDA device")]

TRACE_CAP = 20000
_PREPARED = {}


def _prepared(oracle, hostemu, case):
    if case["name"] not in _PREPARED:
        _PREPARED[case["name"]] = prepare(oracle, hostemu, case)
    return _PREPARED[case["name"]]


def _cell_cases(mode, cap):
    return [c for c in CC.CASES if CC.is_cap_case(c) == cap and not (mode == INPLACE and c["kind"] == "xfer")]


def _check_effective_caps(case, info, eff):
    if case["kind"] == "run":
        assert info["cap_run"] == eff
    elif case["kind"] == "queue":
        assert info["cap_q_inf"] == info["cap_q_trn"] == eff
    elif case["kind"] == "xfer":
        assert info["cap_xfer"] == eff


@pytest.mark.parametrize("cap", [False, True], ids=["nocap", "cap"])
@pytest.mark.parametrize("mode", [STAGED, HEAD, INPLACE], ids=["staged", "head", "inplace"])
@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_capacity_edges_in_launch_cell(oracle, hostemu, monkeypatch, lanes, mode, cap):
    import torch
    from distributed_cluster_gpus_b200.engine import BatchedEngine
    _force(monkeypatch, lanes, mode)
    for case in _cell_cases(mode, cap):
        want, sp0, eff, pred, ks = _prepared(oracle, hostemu, case)
        sp = CC.spec(case, want, BIG_XFER if mode == INPLACE else None)
        seed, n, what = case["seed"], CC.N, f"{case['name']} (cap {eff}, flagged {np.flatnonzero(pred).tolist()})"
        ok = ~pred
        with BatchedEngine(sp, n, base_seed=seed) as eng:
            eng.advance(0)
            one = eng.summary()
            info = eng.launch_info()
            agg_t = torch.zeros(S.AGG_K, dtype=torch.float64, device="cuda")
            eng.reduce_into(agg_t.data_ptr())
            torch.cuda.synchronize()
            agg = agg_t.cpu().numpy()
            assert eng.all_done()
        _check_launch(info, lanes, mode, cap, what + " one-shot")
        _check_effective_caps(case, info, eff)
        check_flags_and_stops(case, one, pred, ks, lambda k: 16 * -(-k // 16))
        if ok.any():
            assert_rows_match(one[ok], want[ok], case["sc"]["n_dc"])
        np.testing.assert_allclose(agg, sharding.aggregate_rows(one), rtol=1e-11)
        assert agg[S.A_FAILED] == pred.sum() and agg[S.A_RUNNING] == 0 and agg[S.A_REPLICAS] == n
        for chunk in (61, 7):
            with BatchedEngine(sp, n, base_seed=seed) as eng:
                if chunk == 61:
                    eng.set_trace(n - 1, TRACE_CAP)
                guard = 0
                while not eng.all_done():
                    eng.advance(chunk)
                    guard += 1
                    assert guard < 20000
                got = eng.summary()
                _check_launch(eng.launch_info(), lanes, mode, cap, f"{what} chunks of {chunk}")
                tr = eng.trace() if chunk == 61 else None
            check_flags_and_stops(case, got, pred, ks, lambda k: k + 15)
            assert np.array_equal(got[ok], one[ok]), (what, chunk)
            if tr is not None:
                k = ks.get(n - 1, 0) if pred[n - 1] else len(tr)
                assert k <= TRACE_CAP and len(tr) >= k
                sim = oracle.OracleSim(sp.to_bytes(), seed + n - 1, trace_cap=TRACE_CAP)
                sim.advance(k if pred[n - 1] else 0)
                wt = sim.trace()[:k]
                sim.close()
                assert np.array_equal(tr["kind"][:k], wt["kind"]) and np.array_equal(tr["seq"][:k], wt["seq"]), what
        if case["name"] == "fifo_mixed":
            assert pred[n - 1] and ks[n - 1] > 0


@pytest.mark.parametrize("name", [c["name"] for c in CC.CASES if c["mixed"]])
def test_mixed_batch_is_retried_once_and_matches_oracle(oracle, hostemu, monkeypatch, name):
    """run_to_completion on a batch where some replicas overflow: one retry with the raised capacity, then every replica
    equals the oracle."""
    from distributed_cluster_gpus_b200 import scenarios as SC
    from distributed_cluster_gpus_b200.engine import free_cached_engine, run_to_completion
    monkeypatch.delenv("DCSIM_GROUP", raising=False)
    monkeypatch.delenv("DCSIM_RECORDS", raising=False)
    case = CC.BY_NAME[name]
    want, sp0, eff, pred, ks = _prepared(oracle, hostemu, case)
    first = CC.caps_dict(case, want)
    calls = []

    def factory(caps):
        calls.append(dict(caps))
        return SC.to_spec(case["sc"], caps=dict(first, **caps))
    free_cached_engine()
    eng, summ = run_to_completion(factory, CC.N, case["seed"])
    eng.close()
    free_cached_engine()
    assert len(calls) == 2 and calls[0] == {} and calls[1], calls
    assert np.all(summ[:, S.S_STATUS] == 0) and np.all(summ[:, S.S_DONE] == 1)
    assert_rows_match(summ, want, case["sc"]["n_dc"])
    print(f"{name}: flagged {np.flatnonzero(pred).tolist()} at cap {eff}, retried with {calls[1]}")
