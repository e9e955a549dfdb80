"""RunnerUtils.randomDDMin on the GPU (demi_random_ddmin) against the CPU reference of the same minimization.

Workload: raft5 with bug flag bit 0; a Fuzzer-generated program of 64 and of 128 externals (fixed seed, default
weights: it contains WaitQuiescence, Kill and Partition events); the first violating seed of a fuzz batch and its
recorded trace (max_messages = its length, as randomDDMin's setMaxMessages(trace.size)); random_ddmin at
K = max_executions in {1, 64, 1024}.  One JSON line per run: card name and power limit (read in the same call), wall
ms, launches, tests issued / evaluated, executions issued (sequential) / run, executions/s, MCS size, the CPU
reference's wall time and whether the two MCS are equal.  Needs a CUDA device.

    python tools/bench_random_ddmin.py [--sizes 64 128] [--ks 1 64 1024] [--cpu-max-k 64]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import demi_b200 as D  # noqa: E402
from demi_b200 import _native as N, fuzzer as F  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:      # noqa: BLE001
        return "unknown (%s)" % e


def program(n_events, seed=11):
    prefix = [D.Start(a) for a in range(5)] + [D.Send(a, 1, 0x1F) for a in range(5)]
    return D.pack_externals(F.Fuzzer(n_events - 10, F.FuzzerWeights(), F.ClientCommandGenerator(2), prefix,
                                     seed=seed).generateFuzzTest())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--ks", type=int, nargs="+", default=[1, 64, 1024])
    ap.add_argument("--cpu-max-k", type=int, default=1024, help="skip the CPU reference above this K")
    ap.add_argument("--interval", type=int, default=5)
    a = ap.parse_args()
    gpu = card()
    cfg = D.SchedulerConfig(N.MODEL_RAFT5, model_flags=1)
    for size in a.sizes:
        ext = program(size)
        eng = D.Engine(cfg)
        eng.set_externals(ext)
        res = eng.fuzz_batch(0, 1 << 16, 200, a.interval)
        seed = int(np.nonzero(res["violation"])[0][0])
        ev, _, r = eng.fuzz_trace(seed, 200, a.interval)
        viol, mm = int(r["violation"]), len(ev)
        for K in a.ks:
            eng.random_ddmin(K, mm, a.interval, 0, viol)                    # warm-up: module load, scratch
            t0 = time.perf_counter()
            mcs, sizes, keys, out, vseed = eng.random_ddmin(K, mm, a.interval, 0, viol)
            wall = (time.perf_counter() - t0) * 1e3
            st = eng.stats()
            row = {"gpu": gpu, "n_externals": len(ext), "K": K, "violation": viol, "max_messages": mm,
                   "wall_ms": round(wall, 3), "tests_issued": len(sizes) - 1, "tests_evaluated": out.replays_executed,
                   "batches": out.batches, "executions_issued": out.total_replays,
                   "mcs_size": out.mcs_size, "verified": bool(out.verified)}
            # executions run and launches of the whole call are summed over its batches
            row["executions_run_last_batch"] = int(st.prefixes)
            if K <= a.cpu_max_k:
                import random_ddmin_ref as R
                t0 = time.perf_counter()
                ref = R.ddmin_random(N.MODEL_RAFT5, ext, K, 0, mm, a.interval, looking_for=viol, model_flags=1)
                row["cpu_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
                row["mcs_equal"] = R.indices_of(ref["mcs"], len(ext)) == R.indices_of(mcs, len(ext))
                row["cpu_executions_issued"] = ref["executions"]
            print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
