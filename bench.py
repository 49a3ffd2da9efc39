#!/usr/bin/env python
"""bench.py — simulated events/sec of the batched multi-DC event engine (BASELINE.json metric).

    python bench.py --gpus 1 --steps 3 --warmup 3            # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 3   # the reference algorithm on host cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W               # N>1: one rank per GPU, weak scaling
    python bench.py --gpus 1 --steps 3 --warmup 3 --dump-outputs DIR   # also writes the last timed step's outputs

A "step" = one full pass of the hot path over one batch: every one of the R replicas per GPU is simulated from
t = 0 to end_time (reset -> arrival pre-pass -> list merge -> event loop -> on-device summary reduction
[-> one NCCL all-reduce of 16 doubles]).
Workload (config.workload) = BASELINE.json configs[2]: 4 DC x 64 sim-GPUs, sinusoid inference (rate 10, amp 0.6,
period 3600 s) + Poisson training (rate 1) per ingress, default_policy/energy_aware, 65 536 replicas per GPU,
120 simulated seconds (~17 k events per replica).

JSON keys beyond the base contract:
  roofline        algorithmic HBM bytes (SURVEY.md §8d: 96 + 76*D per event) / event-loop kernel time vs measured HBM peak
                  (frac), the same over the whole step (frac_step), and where the DRAM-traffic figure comes from
  cpu_baseline    the oracle (C restatement of the reference loop) on the box's host cores, bounded sample
  e2e             same metric through the drop-in MultiIngressPaperSimulator(...).run() — host spec in, kernels,
                  summaries + CSV rows back in host memory — timed on the host clock; cold first run reported beside it
  configs         every BASELINE.json config at its per-GPU replica count (one device-timed batch each, after the headline)
  strong_scaling  (N > 1) the headline workload with 65 536 replicas in TOTAL, split over the N GPUs
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from distributed_cluster_gpus_b200 import scenarios as SC, sharding, spec as S  # noqa: E402

METRIC = "simulated events/sec, 4-DC x 64-sim-GPU, 65536 replicas per GPU"
UNIT = "events/s"
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
KERNELS_PER_STEP = 4       # dcsim_arrivals_kernel, dcsim_merge_kernel, dcsim_advance_kernel, dcsim_reduce_kernel

# BASELINE.json configs (SURVEY.md §8d table): (label, scenario, how the replica count scales, count, GPUs the config is quoted on)
#   "per_gpu": `count` replicas on every GPU (cfg2/cfg3: 65 536 on one B200; cfg5: 1 048 576 / 8 = 131 072 per GPU)
#   "total"  : `count` replicas in the whole job, split over the GPUs (cfg4: 32 768 seeds per variant on 4 B200)
CONFIG_TABLE = [
    ("cfg2", "cfg2_1x64_poisson_600s", "per_gpu", 65536, 1),
    ("cfg3_600s", "cfg3_4x64_sinusoid_600s", "per_gpu", 16384, 1),
    ("cfg4/default_energy_aware", "sweep_default_energy_aware", "total", 32768, 4),
    ("cfg4/default_perf_first", "sweep_default_perf_first", "total", 32768, 4),
    ("cfg4/joint_nf", "sweep_joint_nf", "total", 32768, 4),
    ("cfg4/carbon_cost", "sweep_carbon_cost", "total", 32768, 4),
    ("cfg4/eco_route", "sweep_eco_route", "total", 32768, 4),
    ("cfg4/debug_n2", "sweep_debug_n2", "total", 32768, 4),
    ("cfg5", "cfg5_8x256_sinusoid_60s", "per_gpu", 131072, 8),
]


def workload(args):
    sc = dict(SC.BY_NAME[args.scenario]) if args.scenario in SC.BY_NAME else dict(SC.CFG3)
    if args.duration:
        sc["duration"] = float(args.duration)
    return sc


def config_dict(sc, args, world, extra=None):
    cfg = {"workload": f"{sc['n_dc']} DC x {sc['gpus_per_dc']} sim-GPUs, inf {sc['inf']['mode']} rate {sc['inf']['rate']} "
                       f"amp {sc['inf']['amp']} period {sc['inf']['period']}s + trn {sc['trn']['mode']} rate {sc['trn']['rate']} "
                       f"per ingress, algo {sc['algo']}/{sc['policy']}, {sc['duration']:.0f} simulated s",
           "scenario": sc["name"], "replicas_per_gpu": args.replicas, "replicas_total": args.replicas * world,
           "sim_duration_s": sc["duration"], "parallelism": f"replica-sharded x{world} (no data-path collective)",
           "l2": "working set (event lists + FIFO rings + state blocks, tens of GB) is far larger than the 126 MB L2; no flush needed"}
    cfg.update(extra or {})
    return cfg


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes per event-loop launch from the committed ncu capture of this workload (a constant read from
    profiles/roofline_traffic.json — it is NOT measured in this run; the file says which capture it came from)."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc, self.thread = gpu_index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, pw, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2])); pw.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on host cores (the reference is pure Python and cannot travel)
# ---------------------------------------------------------------------------------------------------
def oracle_rate(sc, n_replicas, threads, seed=123):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_lib
    oracle_lib.build()
    blob = SC.to_spec(sc).to_bytes()
    t0 = time.perf_counter()
    _, events = oracle_lib.run_batch(blob, n_replicas, seed, 0, oracle_lib.RNG_PHILOX, threads)
    dt = time.perf_counter() - t0
    return events, dt


def usable_cpus():
    """What the host really offers this process: min(scheduler affinity, cgroup CPU quota), and the parts."""
    info = {"logical_cpus": os.cpu_count() or 1, "affinity_cpus": None, "cgroup_quota_cpus": None}
    try:
        info["affinity_cpus"] = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2: "<quota|max> <period>"
            quota, period = f.read().split()[:2]
            if quota != "max":
                info["cgroup_quota_cpus"] = round(int(quota) / int(period), 2)
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                quota, period = int(f.read()), int(g.read())            # cgroup v1: -1 = no quota
                if quota > 0:
                    info["cgroup_quota_cpus"] = round(quota / period, 2)
        except (OSError, ValueError):
            pass
    n = info["affinity_cpus"] or info["logical_cpus"]
    if info["cgroup_quota_cpus"]:
        n = min(n, max(1, int(info["cgroup_quota_cpus"])))
    return max(1, int(n)), info


def _py_worker(args):
    sc, seed = args
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_harness
    return ref_harness.time_reference_as_shipped(sc, seed)


def python_reference_leg(sc, cores):
    """The reference's own Python loop, unmodified, timed here — only when DCSIM_REFERENCE_ROOT names a checkout of
    it; otherwise the leg is skipped."""
    root = os.environ.get("DCSIM_REFERENCE_ROOT")
    if not root or not os.path.isdir(os.path.join(root, "simcore")):
        return None
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_harness
    ref_harness.REFERENCE_ROOT = root
    import multiprocessing as mp
    import oracle_lib
    procs = max(1, min(cores, 16))
    seeds = [4000 + i for i in range(procs)]
    blob = SC.to_spec(sc).to_bytes()
    events = sum(oracle_lib.run_batch(blob, 1, s, 0, oracle_lib.RNG_MT19937, 1)[1] for s in seeds)   # the stock runs' event counts
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(procs) as pool:
        walls = pool.map(_py_worker, [(sc, s) for s in seeds])
    wall = time.perf_counter() - t0
    return {"kind": "python", "value": events / max(walls), "unit": UNIT, "processes": procs,
            "events_per_s_per_core": events / sum(walls), "reference_root": root,
            "sample": f"{procs} unmodified reference runs side by side (one process each, own Mersenne Twister, CSV logs on "
                      f"tmpfs): {events} events, slowest run() {max(walls):.2f} s (interpreter start-up and imports, "
                      f"{wall - max(walls):.1f} s here, not counted)"}


def cpu_sample(sc, threads, target_s, cap_replicas, seed):
    oracle_rate(sc, threads, threads)                        # load + page in
    ev, dt = oracle_rate(sc, threads, threads)               # calibration: one replica per thread
    n = int(max(threads, min(cap_replicas, threads * max(1.0, target_s / max(dt, 1e-3)))))
    n -= n % threads
    return n


def cpu_baseline(sc, target_s=12.0):
    threads, host = usable_cpus()
    n = cpu_sample(sc, threads, target_s, 16384, 1000)
    ev, dt = oracle_rate(sc, n, threads, seed=1000)
    ev1, dt1 = oracle_rate(sc, 4, 1, seed=77)
    out = {"value": ev / dt, "unit": UNIT, "cores": threads, "kind": "port", "single_thread_events_per_s": ev1 / dt1,
           "events_per_s_per_core": ev / dt / threads, "host": host,
           "sample": f"{n} replicas of the same workload ({ev} events) in {dt:.1f} s on {threads} threads "
                     "(= min(affinity, cgroup quota)); oracle/dcsim_oracle.c = C restatement of the reference's Python "
                     "loop (the Python original measured 7-20 k events/s/core on this scenario, tests/golden/*.json ref_wall_s)"}
    py = python_reference_leg(sc, threads)
    if py:
        out["python_reference"] = py
    return out


def run_reference_arm(args, world, rank):
    if rank != 0:
        return
    sc = workload(args)
    threads, host = usable_cpus()
    n = cpu_sample(sc, threads, 8.0, 8192, 123)                                # ~8 s of CPU work per step
    for _ in range(args.warmup):
        oracle_rate(sc, max(threads, n // 8), threads)
    t0 = time.perf_counter()
    events = 0
    for i in range(args.steps):
        e, _ = oracle_rate(sc, n, threads, seed=123 + i * n)
        events += e
    total = time.perf_counter() - t0
    value = events / total
    ev1, dt1 = oracle_rate(sc, 4, 1, seed=77)
    sample = (f"{n} replicas per step ({events // max(args.steps, 1)} events) on {threads} host threads "
              "(= min(affinity, cgroup quota)), oracle port of the reference loop")
    cpu = {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
           "single_thread_events_per_s": ev1 / dt1, "events_per_s_per_core": value / threads, "host": host}
    py = python_reference_leg(sc, threads)
    if py:
        cpu["python_reference"] = py
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * total / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(sc, args, world, {"sample_replicas_per_step": n}),
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, summary, first_replica, aggregate, sample_seed=0):
    """Writes what one step hands its caller, so that two builds run with the same arguments can be compared file for
    file: summary.npy (float64 [rows, SUMMARY_K], one row per replica), replica_ids.npy (the global id of each row)
    and aggregate.npy (the all-reduced AGG_K-vector).  When every row does not fit in DUMP_BYTES, the rows are a
    fixed, seeded sample in replica order."""
    row_bytes = (summary.shape[1] + 1) * 8
    cap = (DUMP_BYTES - aggregate.nbytes - 3 * 4096) // row_bytes          # 4096: room for each file's .npy header
    rows = np.arange(len(summary))
    if len(rows) > cap:
        rows = np.sort(np.random.default_rng(sample_seed).choice(len(rows), cap, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "summary.npy"), np.ascontiguousarray(summary[rows], dtype=np.float64))
    np.save(os.path.join(out_dir, "replica_ids.npy"), (first_replica + rows).astype(np.float64))
    np.save(os.path.join(out_dir, "aggregate.npy"), np.asarray(aggregate, dtype=np.float64))


def timed_batch(torch, dist, eng, stream, world, seed, first, warm=1):
    """`warm` untimed batches, then one batch timed with CUDA events on the launching stream; returns
    (ms max over ranks, pre-pass ms, event-loop ms) of this rank's timed batch."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for w in range(warm):
        eng.reset(seed + 7919 * (w + 1), first)
        eng.prepare()
        eng.advance(0, sync=False)
    a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    barrier()
    eng.reset(seed, first)
    a.record(stream)
    eng.prepare()
    b.record(stream)
    eng.advance(0, sync=False)
    c.record(stream)
    barrier()
    ms = torch.tensor([a.elapsed_time(c)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), a.elapsed_time(b), b.elapsed_time(c)


def side_config(torch, dist, BatchedEngine, stream, world, rank, local_rank, scenario, total_replicas, base_seed=123):
    """One BASELINE config as a side record: `total_replicas` sharded over the ranks (sharding.shard), one warm-up
    and one device-timed batch, the 16-double aggregate all-reduced like a real run."""
    sc = SC.BY_NAME[scenario]
    sp = SC.to_spec(sc)
    first, count = sharding.shard(total_replicas, rank, world)
    eng = BatchedEngine(sp, max(count, 1), base_seed=base_seed, first_replica_id=first, device=local_rank, cuda_stream=stream.cuda_stream)
    try:
        ms, pre_ms, loop_ms = timed_batch(torch, dist, eng, stream, world, base_seed, first)
        agg = torch.zeros(S.AGG_K, dtype=torch.float64, device="cuda")
        eng.reduce_into(agg.data_ptr())
        torch.cuda.current_stream().synchronize()
        stream.synchronize()
        sharding.allreduce_aggregate(agg)
        a = agg.cpu().numpy()
        info = eng.launch_info()
    finally:
        eng.close()
    return {"scenario": scenario, "replicas_total": int(total_replicas), "replicas_per_gpu": int(-(-total_replicas // world)), "n_gpus": world,
            "events": float(a[S.A_EVENTS]), "ms": ms, "prepass_ms_rank0": pre_ms, "event_loop_ms_rank0": loop_ms,
            "events_per_s": float(a[S.A_EVENTS]) / (ms / 1e3), "failed_replicas": float(a[S.A_FAILED]),
            "warps_per_sm": info["resident_warps_per_sm"], "state_block_bytes": info["state_block_bytes"],
            "staged_bytes_per_replica": info["staged_bytes_per_replica"], "staging_mode": info["staging_mode"],
            "algorithmic_bytes_per_event": 96 + 76 * sc["n_dc"], "sim_duration_s": sc["duration"]}


def run_b200(args, world, rank, local_rank):
    import torch
    import torch.distributed as dist
    from distributed_cluster_gpus_b200.engine import BatchedEngine
    from distributed_cluster_gpus_b200.configs import paper_config as pc
    from distributed_cluster_gpus_b200.simcore.simulator_paper_multi import MultiIngressPaperSimulator
    import logging

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sc = workload(args)
    sp = SC.to_spec(sc)
    R = args.replicas
    first, _count = sharding.shard(R * world, rank, world)   # weak scaling: R replicas on every rank, global ids
    stream = torch.cuda.Stream()              # explicit (non-default) stream: its handle is what the C-ABI launches on,
    torch.cuda.set_stream(stream)             # so torch.cuda.Event timing brackets exactly our kernels
    eng = BatchedEngine(sp, R, base_seed=123, first_replica_id=first, device=local_rank, cuda_stream=stream.cuda_stream)
    info = eng.launch_info()
    agg = torch.zeros((args.steps + args.warmup + 1, S.AGG_K), dtype=torch.float64, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(i, k0=None, k1=None, p0=None):
        eng.reset(123 + i * R * world, first)
        if p0 is not None:
            p0.record(stream)
        eng.prepare()                                               # arrival pre-pass + list merge
        if k0 is not None:
            k0.record(stream)
        eng.advance(0, sync=False)                                  # event loop (dcsim_advance_kernel)
        if k1 is not None:
            k1.record(stream)
        eng.reduce_into(agg[i].data_ptr())
        sharding.allreduce_aggregate(agg[i])                        # the run's only collective: 16 doubles over NVLink

    for i in range(args.warmup):
        one_step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    k0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    k1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    p0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record(stream)
    for j in range(args.steps):
        one_step(args.warmup + j, k0[j], k1[j], p0[j])
    t1.record(stream)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng.summary(), first, agg[args.warmup + args.steps - 1].cpu().numpy())
    elapsed_ms = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
    kernel_ms = [a.elapsed_time(b) for a, b in zip(k0, k1)]
    prepass_ms = sum(a.elapsed_time(b) for a, b in zip(p0, k0)) / args.steps
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    elapsed_s = float(elapsed_ms.item()) / 1000.0
    steps_agg = agg[args.warmup: args.warmup + args.steps].cpu().numpy()       # already summed over ranks
    events_total = float(steps_agg[:, S.A_EVENTS].sum())
    failed = float(steps_agg[:, S.A_FAILED].sum())
    value = events_total / elapsed_s

    # ---- roofline of the dominant kernel (the event loop), this rank -------------------------------
    local_events_per_launch = events_total / args.steps / world
    b_alg = 96 + 76 * sc["n_dc"]
    kms = sum(kernel_ms) / len(kernel_ms)
    achieved = local_events_per_launch * b_alg / (kms / 1000.0) / 1e9
    step_ms = 1000.0 * elapsed_s / args.steps
    peak, peak_src = hbm_peak()
    traffic = measured_traffic()
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
                "traffic_source": ({k: traffic.get(k) for k in ("source", "captured", "build", "note")} if traffic else None),
                "kernel": "dcsim_advance_kernel", "kernel_ms": kms, "arrivals_prepass_kernel_ms": prepass_ms,
                "events_per_launch": local_events_per_launch,
                "achieved_step": local_events_per_launch * b_alg / (step_ms / 1000.0) / 1e9,
                "frac_step": local_events_per_launch * b_alg / (step_ms / 1000.0) / 1e9 / peak,
                "algorithmic_bytes_per_event": b_alg, "peak_source": peak_src,
                "note": "frac = algorithmic bytes / event-loop kernel time; frac_step = the same over the whole step (the 400 B "
                        "per event include the arrival / RNG work the pre-pass kernels do).  The path is warp-serial-latency "
                        "bound, not HBM bound (SURVEY.md §8d): see DESIGN.md §4 for the issue-slot bound and profiles/ for ncu evidence",
                "events_per_s_per_resident_warp": local_events_per_launch / (kms / 1000.0) / max(1, info["resident_warps_per_sm"] * info["sm_count"])}

    if args.no_e2e:                                                            # tuning runs
        eng.close()
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                              "ms_per_step": step_ms, "kernel_ms": kms, "prepass_ms": prepass_ms, "launch": info,
                              "clocks": clocks, "tuning_run": True}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- e2e through the drop-in public API (host buffers in and out) -----------------------------
    log_dir = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp", f"dcsim_bench_{os.getpid()}")
    eng.close()
    e2e_steps = max(1, args.steps)

    def e2e_step(i):
        kw_i = SC.build_inputs(sc)
        sim = MultiIngressPaperSimulator(router_policy=pc.build_router_policy(), logger=logging.getLogger("bench"),
                                         sim_duration=sc["duration"], log_interval=sc["log_interval"], log_path=log_dir,
                                         rng_seed=5000 + i * R * world, algo=sc["algo"], show_progress=False,
                                         replicas=R, device=local_rank, first_replica_id=first,
                                         cuda_stream=stream.cuda_stream, **kw_i)
        sim.run()
        ok = bool(np.all(sim.summary[:, S.S_DONE] == 1) and np.all(sim.summary[:, S.S_STATUS] == 0))
        return float(sim.summary[:, S.S_EVENTS].sum()) if ok else float("nan"), sim   # the host reads the result

    barrier()
    c0 = time.perf_counter()
    e2e_step(-1)                                         # COLD: allocates the device buffers (tens of GB) and pages them in
    cold_ms = 1000.0 * (time.perf_counter() - c0)
    barrier()
    w0 = time.perf_counter()
    e2e_events = 0.0
    for i in range(e2e_steps):
        ev_i, sim = e2e_step(i)
        e2e_events += ev_i
    barrier()
    w = torch.tensor([time.perf_counter() - w0], dtype=torch.float64, device="cuda")
    ev_t = torch.tensor([e2e_events], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(w, op=dist.ReduceOp.MAX)
        dist.all_reduce(ev_t, op=dist.ReduceOp.SUM)
    e2e_value = float(ev_t.item()) / float(w.item())
    csv_bytes = sum(os.path.getsize(p) for p in (sim.cluster_log_path, sim.job_log_path) if os.path.exists(p))
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(len(sp.to_bytes()) + 512),
           "d2h_bytes_per_step": int(R * S.SUMMARY_K * 8 + csv_bytes), "steps": e2e_steps,
           "api": "MultiIngressPaperSimulator(..., replicas=R).run(): flatten -> dcsim_create / dcsim_reset -> dcsim_advance -> "
                  "dcsim_fetch_summary -> DataCenter write-back + cluster_log.csv/job_log.csv of replica 0",
           "ms_per_step": 1000.0 * float(w.item()) / e2e_steps,
           "cold_first_run_ms": cold_ms,
           "note": "warm steps re-seed the device allocations parked by the previous run() of the same shape; the cold first "
                   "run() (cudaMalloc + first touch of the event lists / FIFO rings) is reported separately, outside the rate"}

    import shutil
    from distributed_cluster_gpus_b200.engine import free_cached_engine
    free_cached_engine()
    shutil.rmtree(log_dir, ignore_errors=True)

    # ---- side records: the other BASELINE configs, strong scaling ---------------------------------
    configs, strong = None, None
    if not args.no_configs:
        configs = {}
        for label, name, how, count, quoted_gpus in CONFIG_TABLE:
            reps_total = count * world if how == "per_gpu" else count   # N = quoted_gpus reproduces the config exactly
            try:
                rec = side_config(torch, dist, BatchedEngine, stream, world, rank, local_rank, name, reps_total)
                rec["quoted_on_gpus"] = quoted_gpus
                rec["matches_baseline_size"] = bool(world == quoted_gpus or (how == "per_gpu" and quoted_gpus == 1))
            except Exception as e:                                             # never lose the headline to a side record
                rec = {"scenario": name, "error": f"{type(e).__name__}: {e}"[:300]}
            configs[label] = rec
        if world > 1:
            try:
                strong = side_config(torch, dist, BatchedEngine, stream, world, rank, local_rank, sc["name"], 65536)
                strong["note"] = "the headline workload with 65 536 replicas in TOTAL (strong scaling); compare events_per_s with the N=1 headline"
            except Exception as e:
                strong = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_dict(sc, args, world, {"events_per_step": events_total / args.steps,
                                                        "failed_replicas": failed, "launch": info}),
                "roofline": roofline, "cpu_baseline": cpu_baseline(sc) if world == 1 and not args.no_cpu_baseline else None,
                "e2e": e2e, "gpu_launches": KERNELS_PER_STEP * args.steps, "clocks": clocks, "impl": "b200",
                "comm": {"backend": "nccl" if world > 1 else None, "nranks": world,
                         "collective": "one all_reduce of 16 doubles per step" if world > 1 else None,
                         "nccl_version": ".".join(map(str, torch.cuda.nccl.version())) if world > 1 else None},
                "configs": configs, "strong_scaling": strong}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--replicas", type=int, default=65536, help="replicas per GPU")
    ap.add_argument("--scenario", type=str, default="cfg3_4x64_sinusoid_120s")
    ap.add_argument("--duration", type=float, default=None, help="override the scenario's simulated seconds")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="tuning runs only: skip the end-to-end leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the side records (other BASELINE configs, strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/*.npy (rank 0, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm only")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, world, rank)
        return
    if world > 1:
        # stdout must stay ONE JSON line, whatever the libraries underneath write to file descriptor 1 (NCCL prints its
        # version banner and its INFO lines there): fd 1 is pointed at stderr for the rest of the process and Python's own
        # sys.stdout keeps the real stdout.
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        sys.stdout = os.fdopen(real_stdout, "w", buffering=1)
        # BEFORE torch is imported: the communicator's init lines (nranks, NVLS, ...) are wanted as evidence that N ranks
        # really talk.  An INFO / TRACE level chosen by the caller is respected, a quieter one (images often export
        # NCCL_DEBUG=VERSION or WARN) is raised to INFO for the INIT subsystem; the lines end up on stderr (see above).
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ["NCCL_DEBUG_SUBSYS"] = "INIT"
    run_b200(args, world, rank, local_rank)


if __name__ == "__main__":
    main()
