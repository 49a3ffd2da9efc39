"""BatchedEngine — thin owner of one ``dcsim_t`` handle (one CUDA device, one stream, R replicas)."""
import ctypes as C
import os

import numpy as np

from . import _native as N
from . import spec as S

TRACE_DTYPE = np.dtype([("t", "<f8"), ("seq", "<u4"), ("kind", "<u4")])
JOB_DTYPE = np.dtype([("jid", "<u4"), ("n_gpus", "<u4"), ("ingress", "u1"), ("jtype", "u1"), ("dc", "u1"), ("_pad0", "u1"),
                      ("_pad1", "<u4"), ("size", "<f8"), ("f_used", "<f8"), ("start_s", "<f8"), ("finish_s", "<f8")], align=True)
CLUSTER_DTYPE = np.dtype([("time_s", "<f8"), ("freq", "<f8"), ("util_gpu_time", "<f8"), ("util_begin_ts", "<f8"),
                          ("acc_job_unit", "<f8"), ("power_w", "<f8"), ("energy_j", "<f8"), ("dc", "<i4"),
                          ("busy", "<i4"), ("run_total", "<i4"), ("run_inf", "<i4"), ("q_inf", "<i4"),
                          ("q_train", "<i4")], align=True)
assert TRACE_DTYPE.itemsize == C.sizeof(S.TraceRec) and JOB_DTYPE.itemsize == C.sizeof(S.JobRec)
assert CLUSTER_DTYPE.itemsize == C.sizeof(S.ClusterRec)


LAT_BINS = 128


def latency_bin_edges() -> np.ndarray:
    """Lower edges [s] of the LAT_BINS histogram bins (+ the upper edge of the last): 2^e * (1 + m/4), e from -20."""
    k = np.arange(LAT_BINS + 1)
    return np.ldexp(1.0 + (k % 4) / 4.0, k // 4 - 20)


def latency_quantiles(hist_row, qs=(0.5, 0.9, 0.99)):
    """Quantiles [s] of one histogram row, log-interpolated inside the bin that holds the quantile."""
    h = np.asarray(hist_row, dtype=np.float64)
    total = h.sum()
    if total == 0:
        return [float("nan")] * len(qs)
    edges, cum, out = latency_bin_edges(), np.cumsum(h), []
    for q in qs:
        b = int(np.searchsorted(cum, q * total, side="left"))
        b = min(b, LAT_BINS - 1)
        below = cum[b - 1] if b else 0.0
        frac = (q * total - below) / h[b] if h[b] else 0.0
        out.append(float(edges[b] * (edges[b + 1] / edges[b]) ** frac))
    return out


RNG_KINDS = {"philox": 0, "mt19937": 1}


class RecorderOverflow(RuntimeError):
    """A recorder (0 trace, 1 job log, 2 cluster log) saw more rows than its capacity; `.needed` says how many."""

    def __init__(self, which, needed, capacity):
        super().__init__(f"{('trace', 'job log', 'cluster log')[which]} needs {needed} rows, capacity {capacity}")
        self.which, self.needed, self.capacity = which, needed, capacity


class BatchedEngine:
    """R independent replicas of one scenario on one GPU.

    Replica r uses Philox key ``base_seed + first_replica_id + r`` — the key the reference would be given as
    ``rng_seed`` — so results do not depend on how replicas are sharded over GPUs.
    """

    def __init__(self, spec: S.Spec, n_replicas: int, base_seed: int, first_replica_id: int = 0, device: int = 0,
                 cuda_stream: int = 0):
        self._lib = N.load()
        self._h = C.c_void_p()
        self.n_replicas = int(n_replicas)
        self.spec = spec
        blob = spec.to_bytes()
        self._blob = C.create_string_buffer(blob, len(blob))
        N.check(self._lib.dcsim_create(self._blob, len(blob), self.n_replicas, base_seed & (2**64 - 1),
                                       first_replica_id, device, C.byref(self._h)))
        if cuda_stream:
            self.set_stream(cuda_stream)
        self._trace_cap = self._jobs_cap = self._cluster_cap = 0

    # -- configuration ---------------------------------------------------------------------------
    def set_stream(self, cuda_stream: int):
        N.check(self._lib.dcsim_set_stream(self._h, C.c_void_p(cuda_stream)), self._h)

    def reset(self, base_seed: int, first_replica_id: int = 0):
        """All replicas back to t = 0 with new keys; allocations are kept."""
        N.check(self._lib.dcsim_reset(self._h, base_seed & (2**64 - 1), first_replica_id), self._h)

    def set_rng(self, kind: str = "philox"):
        """Word source of the replicas' random streams: "philox" (default; key = seed) or "mt19937" (CPython's own
        generator seeded like ``random.seed(seed)``: replica r is then the STOCK reference run at rng_seed + r)."""
        if kind not in RNG_KINDS:
            raise ValueError(f"unknown rng {kind!r}; expected one of {sorted(RNG_KINDS)}")
        N.check(self._lib.dcsim_set_rng(self._h, RNG_KINDS[kind]), self._h)

    def set_trace(self, replica: int, capacity: int):
        N.check(self._lib.dcsim_set_trace(self._h, replica, capacity), self._h)
        self._trace_cap = capacity

    def set_logging(self, replica: int, job_capacity: int, cluster_capacity: int):
        N.check(self._lib.dcsim_set_logging(self._h, replica, job_capacity, cluster_capacity), self._h)
        self._jobs_cap, self._cluster_cap = job_capacity, cluster_capacity

    # -- run -------------------------------------------------------------------------------------
    def prepare(self):
        """Launches the arrival pre-pass (optional; advance() does it when needed)."""
        N.check(self._lib.dcsim_prepare(self._h), self._h)

    def advance(self, max_events_per_replica: int = 0, sync: bool = True) -> int:
        """Every replica processes up to ``max_events_per_replica`` more events (0 = to end_time).
        With ``sync`` returns the number of events this call processed; otherwise launches and returns -1."""
        if sync:
            total = C.c_uint64(0)
            N.check(self._lib.dcsim_advance(self._h, max_events_per_replica, C.byref(total)), self._h)
            return int(total.value)
        N.check(self._lib.dcsim_advance(self._h, max_events_per_replica, None), self._h)
        return -1

    def all_done(self) -> bool:
        d = C.c_int(0)
        N.check(self._lib.dcsim_all_done(self._h, C.byref(d)), self._h)
        return bool(d.value)

    def summary(self, out=None) -> np.ndarray:
        """[n_replicas, SUMMARY_K] float64; ``out`` may be a (pinned) preallocated array."""
        if out is None and hasattr(self._lib, "dcsim_fetch_summary_host"):
            # through the library's page-locked mirror (a full-rate DMA), then one host copy: the mirror is reused by
            # the next fetch on this handle, the returned array is the caller's
            p = C.POINTER(C.c_double)()
            N.check(self._lib.dcsim_fetch_summary_host(self._h, C.byref(p)), self._h)
            return _copy_rows(np.ctypeslib.as_array(p, shape=(self.n_replicas, S.SUMMARY_K)))
        if out is None:
            out = np.empty((self.n_replicas, S.SUMMARY_K), dtype=np.float64)
        N.check(self._lib.dcsim_fetch_summary(self._h, C.c_void_p(out.ctypes.data), out.nbytes), self._h)
        return out

    def fetch_summary_into(self, host_ptr: int, nbytes: int):
        N.check(self._lib.dcsim_fetch_summary(self._h, C.c_void_p(host_ptr), nbytes), self._h)

    def summary_device_ptr(self) -> int:
        p = C.c_void_p()
        N.check(self._lib.dcsim_summary_device_ptr(self._h, C.byref(p)), self._h)
        return int(p.value)

    def reduce_into(self, device_ptr: int):
        """Writes the AGG_K-vector (spec.A_*) to device memory; the caller all-reduces it."""
        N.check(self._lib.dcsim_reduce_summary(self._h, C.c_void_p(device_ptr)), self._h)

    def enable_latency_histogram(self):
        """Opt-in, before the first advance of a batch: job-latency histogram of the whole batch (~1 % of kernel time)."""
        N.check(self._lib.dcsim_enable_latency_histogram(self._h), self._h)

    def latency_histogram(self) -> np.ndarray:
        """[2, LAT_BINS] uint64: job-latency counts of the whole batch ([0] inference, [1] training)."""
        out = np.zeros((2, LAT_BINS), dtype=np.uint64)
        N.check(self._lib.dcsim_fetch_latency_histogram(self._h, C.c_void_p(out.ctypes.data), out.nbytes), self._h)
        return out

    # -- recorders -------------------------------------------------------------------------------
    def recorder_counts(self):
        """(trace, job_log, cluster_log) rows the recorders WOULD have written: more than a recorder's capacity means
        its rows are a truncated prefix (the kernels keep counting and stop writing)."""
        out = (C.c_uint32 * 3)()
        N.check(self._lib.dcsim_recorder_counts(self._h, C.byref(out)), self._h)
        return int(out[0]), int(out[1]), int(out[2])

    def _fetch(self, fn, dtype, cap, which):
        arr = np.zeros(max(cap, 1), dtype=dtype)
        n = C.c_uint32(0)
        N.check(fn(self._h, C.c_void_p(arr.ctypes.data), cap, C.byref(n)), self._h)
        if cap and which is not None and self.recorder_counts()[which] > cap:     # never hand a silently truncated log to a caller
            raise RecorderOverflow(which, self.recorder_counts()[which], cap)
        return arr[: n.value]

    def trace(self):
        """The first `capacity` processed events of the traced replica (a debug aid: a prefix by design)."""
        return self._fetch(self._lib.dcsim_fetch_trace, TRACE_DTYPE, self._trace_cap, None)

    def job_log(self):
        return self._fetch(self._lib.dcsim_fetch_job_log, JOB_DTYPE, self._jobs_cap, 1)

    def cluster_log(self):
        return self._fetch(self._lib.dcsim_fetch_cluster_log, CLUSTER_DTYPE, self._cluster_cap, 2)

    def launch_info(self) -> dict:
        li = S.LaunchInfo()
        N.check(self._lib.dcsim_launch_info(self._h, C.byref(li)), self._h)
        return {name: int(getattr(li, name)) for name, _ in S.LaunchInfo._fields_ if not name.startswith("_")}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.dcsim_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_COPY_POOL = None


def _copy_rows(src: np.ndarray) -> np.ndarray:
    """A private copy of a large row-major array, row blocks on a few threads (numpy's copy loops release the GIL):
    the 46 MB of summaries of a 65 536-replica batch take 9 ms on one thread, a third of that on four."""
    global _COPY_POOL
    n = src.shape[0]
    if src.nbytes < (8 << 20):
        return src.copy()
    if _COPY_POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _COPY_POOL = ThreadPoolExecutor(max_workers=4, thread_name_prefix="dcsim-copy")
    dst = np.empty_like(src)
    step = (n + 3) // 4
    list(_COPY_POOL.map(lambda a: np.copyto(dst[a:a + step], src[a:a + step]), range(0, n, step)))
    return dst


STATUS_NAMES = {S.ST_XFER_OVERFLOW: "in-flight transfer pool", S.ST_RUN_OVERFLOW: "running set",
                S.ST_QUEUE_OVERFLOW: "FIFO queue", S.ST_STALE_OVERFLOW: "stale-event pool",
                S.ST_RNG_RUNAWAY: "rejection-sampling runaway", S.ST_ARRIVALS_OVERFLOW: "arrival list",
                S.ST_ARRIVAL_TIE: "two arrivals at the identical instant (unused since ABI 2: ties are resolved in push order)",
                S.ST_SEQ_OVERFLOW: "more than 2^28 event pushes in one replica"}


def describe_status(bits: int) -> str:
    return ", ".join(name for bit, name in STATUS_NAMES.items() if bits & bit) or "ok"


# One idle engine is kept after run_to_completion()/release() so that the next run of the SAME scenario shape (same
# spec blob, replica count, device, stream) re-seeds the existing device allocations (dcsim_reset) instead of
# freeing and re-allocating tens of GB.  free_cached_engine() drops it.
_CACHED = {"key": None, "engine": None}
_CACHED_LOGGED = {"key": None, "engine": None}   # the one-replica companion engine of LoggedReplica


def _cache_key(sp, n_replicas, device, cuda_stream):
    # the launch geometry is fixed when the handle is created: an engine sized under other DCSIM_GROUP / DCSIM_RECORDS
    # settings is not the engine the caller asked for
    return (sp.to_bytes(), int(n_replicas), int(device), int(cuda_stream), os.environ.get("DCSIM_RECORDS", ""),
            os.environ.get("DCSIM_GROUP", ""))


def _drop_parked_batch_engine():
    if _CACHED["engine"] is not None:
        _CACHED["engine"].close()
    _CACHED["engine"], _CACHED["key"] = None, None


def acquire_engine(sp, n_replicas, base_seed, first_replica_id=0, device=0, cuda_stream=0):
    key = _cache_key(sp, n_replicas, device, cuda_stream)
    if _CACHED["engine"] is not None and _CACHED["key"] == key:
        eng, _CACHED["engine"], _CACHED["key"] = _CACHED["engine"], None, None
        eng.reset(base_seed, first_replica_id)   # fresh batch: recorders may be re-targeted again
        eng.set_trace(0, 0)
        eng.set_logging(0, 0, 0)
        eng.set_rng("philox")
        return eng
    _drop_parked_batch_engine()   # (tens of GB: gone before the new batch allocates; the one-replica companion stays)
    return BatchedEngine(sp, n_replicas, base_seed, first_replica_id, device, cuda_stream)


def release_engine(eng, sp, device=0, cuda_stream=0):
    """Parks a finished engine for reuse (see acquire_engine); a previously parked batch engine is destroyed.  The
    parked companion of LoggedReplica is a separate slot and is left alone (closing and re-creating it was 16 ms of
    every run())."""
    _drop_parked_batch_engine()
    _CACHED["engine"], _CACHED["key"] = eng, _cache_key(sp, eng.n_replicas, device, cuda_stream)


def free_cached_engine():
    for slot in (_CACHED, _CACHED_LOGGED):
        if slot["engine"] is not None:
            slot["engine"].close()
        slot["engine"], slot["key"] = None, None


class LoggedReplica:
    """The cluster_log.csv / job_log.csv rows of ONE replica of a batch, produced by a one-replica companion engine
    that runs the same trajectory (same spec, same key) on its own stream WHILE the batch runs.

    Switching the recorders on inside the batch makes every replica carry the job log's fields in its running-job
    records (60 instead of 40 bytes; fewer resident warps: +9 % on the 65 536-replica bench batch); a single warp
    next to the batch's grid costs nothing — it is launched first, is resident before the grid fills the GPU, and
    finishes long before it.  Results are identical by construction (one replica = one deterministic trajectory)."""

    def __init__(self, sp, seed, replica_id, device, job_rows, cluster_rows, rng="philox"):
        key = (sp.to_bytes(), int(device))
        if _CACHED_LOGGED["engine"] is not None and _CACHED_LOGGED["key"] == key:
            self.eng, _CACHED_LOGGED["engine"], _CACHED_LOGGED["key"] = _CACHED_LOGGED["engine"], None, None
            self.eng.reset(seed, replica_id)
        else:
            if _CACHED_LOGGED["engine"] is not None:
                _CACHED_LOGGED["engine"].close()
                _CACHED_LOGGED["engine"], _CACHED_LOGGED["key"] = None, None
            self.eng = BatchedEngine(sp, 1, seed, replica_id, device)    # its own (non-blocking) stream
        self._key = key
        self.eng.set_rng(rng)
        self.eng.set_logging(0, job_rows, cluster_rows)
        self.eng.advance(0, sync=False)                                 # in flight; the caller launches the batch now

    def collect(self):
        """(status bits, job rows, cluster rows); synchronises with the companion's stream."""
        bits = int(self.eng.summary()[0, S.S_STATUS])
        return bits, self.eng.job_log(), self.eng.cluster_log()

    def release(self, keep=True):
        if keep:
            _CACHED_LOGGED["engine"], _CACHED_LOGGED["key"] = self.eng, self._key
        else:
            self.eng.close()
        self.eng = None


def run_to_completion(spec_factory, n_replicas, base_seed, first_replica_id=0, device=0, cuda_stream=0,
                      max_retries=3, configure=None, while_running=None):
    """Runs all replicas to end_time.  A replica that overflowed a capacity is never trusted: the whole batch
    is re-run with that capacity raised (``spec_factory(caps)`` rebuilds the blob).  Returns (engine, summary);
    hand the engine back with release_engine() (reuse) or close().  ``while_running()`` is called once, after the
    kernels of the first attempt were launched and before the host waits for them (host work that can overlap)."""
    caps = {}
    for attempt in range(max_retries + 1):
        sp = spec_factory(dict(caps))
        eng = acquire_engine(sp, n_replicas, base_seed, first_replica_id, device, cuda_stream)
        if configure:
            configure(eng)
        eng.advance(0, sync=False)
        if while_running is not None and attempt == 0:
            try:
                while_running()
            except BaseException:
                eng.close()
                raise
        summ = eng.summary()                     # synchronises with the batch's stream
        bits = int(np.bitwise_or.reduce(summ[:, S.S_STATUS].astype(np.int64)))
        if bits == 0:
            return eng, summ
        eng.close()
        raisable = S.ST_RUN_OVERFLOW | S.ST_XFER_OVERFLOW | S.ST_ARRIVALS_OVERFLOW | S.ST_QUEUE_OVERFLOW | S.ST_STALE_OVERFLOW
        if bits & ~raisable or attempt == max_retries:   # a status no capacity can cure (or out of attempts): fail now
            raise RuntimeError(f"replicas stopped: {describe_status(bits)}")
        g_max = max(sp.dc[d].total_gpus for d in range(sp.n_dc))
        if bits & S.ST_RUN_OVERFLOW:
            caps["cap_run"] = g_max
        if bits & S.ST_XFER_OVERFLOW:
            caps["cap_xfer"] = 2 * sp.cap_xfer
        if bits & S.ST_ARRIVALS_OVERFLOW:
            caps["cap_arrivals"] = 2 * sp.cap_arrivals
        if bits & S.ST_QUEUE_OVERFLOW:
            caps["cap_q_inf"], caps["cap_q_trn"] = 2 * sp.cap_q_inf, 2 * sp.cap_q_trn
        if bits & S.ST_STALE_OVERFLOW:                   # cap_greedy: superseded job_finish events still in the event set
            caps["cap_stale"] = 2 * max(64, sp.cap_stale)
    raise AssertionError("unreachable")
