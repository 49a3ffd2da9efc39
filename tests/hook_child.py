"""TEST-ONLY child process of tests/test_gpu_ties.py: runs a list of jobs with the library DCSIM_B200_LIB names (one
of the hook builds, __graft_entry__.TEST_HOOK_LIBS) and writes what each produced as .npy / .json.

    python tests/hook_child.py JOBS.json OUT_DIR

Each job: {"id", "blob" (a spec file), "q" (time quantum, 0 = off), "seed", "n" (replicas), "lanes" (DCSIM_GROUP, 0 =
the default pick), "chunk" (events per advance, 0 = one shot)}; replica n-1 is traced and logged.
"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRACE_CAP, JOBS_CAP, CLUSTER_CAP = 6000, 40000, 4000


def _child(jobs_path, out_dir):
    """Runs the jobs of `jobs_path` with the library DCSIM_B200_LIB names; writes <out_dir>/<id>_*.npy and .json."""
    from distributed_cluster_gpus_b200 import _native, spec as S
    from distributed_cluster_gpus_b200.engine import BatchedEngine
    assert os.path.samefile(_native.LIB_PATH, os.environ["DCSIM_B200_LIB"])
    lib = _native.load()
    lib.dcsim_test_set_time_quantum.argtypes = [C.c_double]
    lib.dcsim_test_set_time_quantum.restype = None
    with open(jobs_path) as f:
        jobs = json.load(f)
    for job in jobs:
        if job["lanes"]:
            os.environ["DCSIM_GROUP"] = str(job["lanes"])
        else:
            os.environ.pop("DCSIM_GROUP", None)
        lib.dcsim_test_set_time_quantum(job["q"])
        with open(job["blob"], "rb") as f:
            sp = S.Spec.from_buffer_copy(f.read())
        n, rec = job["n"], job["n"] - 1
        with BatchedEngine(sp, n, base_seed=job["seed"]) as eng:
            eng.set_trace(rec, TRACE_CAP)
            eng.set_logging(rec, JOBS_CAP, CLUSTER_CAP)
            total = 0
            if job["chunk"]:
                while not eng.all_done():
                    total += eng.advance(job["chunk"])
            else:
                total = eng.advance(0)
            base = os.path.join(out_dir, job["id"])
            np.save(base + "_summary.npy", eng.summary())
            np.save(base + "_trace.npy", eng.trace())
            np.save(base + "_jobs.npy", eng.job_log())
            np.save(base + "_cluster.npy", eng.cluster_log())
            with open(base + ".json", "w") as f:
                json.dump({"events": total, "launch": eng.launch_info()}, f)
    lib.dcsim_test_set_time_quantum(0.0)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _child(sys.argv[1], sys.argv[2])
