#!/usr/bin/env python
"""bench.py — schedule prefixes/sec on the BASELINE.json north-star workload, plus the secondary configs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--no-secondary] [--dump-outputs DIR]

Headline (BASELINE.json configs[1]): 5-actor Raft model (seeded double-vote bug), RandomScheduler/FullyRandom fuzz,
maxMessages=50, invariant every 5 deliveries, 10^7 prefixes per step per GPU (weak scaling: rank r, step s explores
its own seed range).  One "step" = one pass of the hot path over one batch of prefixes.

  value : prefixes/s, results stay in HBM (demi_fuzz_batch_dev), CUDA-event timed
  e2e   : prefixes/s through the reference-facing C-ABI call demi_fuzz_batch with HOST buffers
          (external program H2D + all result records D2H per step)
  roofline     : algorithmic HBM bytes of the fuzz kernel vs the measured copy peak; the profile-derived figures
                 (DRAM traffic, issue-slot utilisation) come from profiles/k1_profile.json and are dropped when that
                 capture was taken from another build of the kernels
  cpu_baseline : the CPU oracle (C restatement of the reference's JVM scheduler) on all host cores, bounded sample
  secondary    : configs[2] (one DPORwHeuristics search as a frontier, with the in-library NCCL steal round at N > 1),
                 configs[3] (DDMin / STSSched replays over a 2000-event trace), configs[4] (bcast32 + state-hash
                 dedup) — measured after, and outside, the headline's timed region (tools/secondary.py)

`--dump-outputs DIR` writes what the timed path computed in its last step on rank 0 (see dump_outputs) as
DIR/<name>.npy, so that two builds can be compared output for output: the inputs depend on the arguments alone.
The benchmark itself writes nothing into the tree; an oracle library it has to rebuild goes to a temporary directory.

`--impl reference` times the CPU oracle alone on the SAME batch definition (the reference itself needs a JVM + sbt +
Akka + the akka-raft application, none of which exist here).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL_RAFT5 = 2
MAX_MESSAGES = 50
INTERVAL = 5
MODEL_FLAGS = 1            # Raft5 BUG_DOUBLE_VOTE: gives a non-empty, stable violating set
RESULT_BYTES = 32          # sizeof(demi_fuzz_result): the algorithmic HBM bytes per prefix
PREFIXES_PER_STEP = 10_000_000
METRIC = "schedule prefixes/sec (5-actor Raft, depth 50)"
K1_PROFILE = os.path.join(ROOT, "profiles", "k1_profile.json")


def workload_config(n_per_step, n_gpus):
    return {
        "workload": "raft5 depth-50 random fuzz (BASELINE.json configs[1])",
        "model": "raft5 (5 actors, tick timers, log cap 8, seeded double-vote bug)",
        "scheduler": "RandomScheduler/FullyRandom(seed=base+i)",
        "max_messages": MAX_MESSAGES, "invariant_check_interval": INTERVAL,
        "prefixes_per_step_per_gpu": n_per_step, "sharding": "seed ranges per rank, no data-path collective",
        "l2": "each step writes %d MB of fresh result records (> 126 MB L2); no input is re-read across steps"
              % (n_per_step * RESULT_BYTES // 1_000_000),
        "n_gpus": n_gpus,
    }


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                f = [x.strip() for x in out.stdout.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.samples[0][1]) if self.samples[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


def host_cores():
    """Host threads the CPU arm may really use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return max(1, n)


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def k1_profile(k1_id):
    """Profile-derived figures of the headline kernel (tools/profile_k1.py writes the file from one `ncu --set full`
    capture).  They describe ONE build: if the library was built from other sources they are reported as stale and
    not used — loudly, on stderr and in the JSON line."""
    if not os.path.exists(K1_PROFILE):
        return None, "no profiles/k1_profile.json"
    try:
        p = json.load(open(K1_PROFILE))
    except Exception as e:
        return None, "unreadable profile: %s" % e
    if p.get("k1_id") != k1_id:
        msg = "profiles/k1_profile.json was captured from kernel sources %s, the library was built from %s" % (p.get("k1_id"), k1_id)
        sys.stderr.write("bench.py: STALE PROFILE — %s; its figures are not reported (re-run tools/profile_k1.py)\n" % msg)
        return None, msg
    return p, None


DUMP_RECORDS = 1 << 18     # 11 float64 arrays of this length: 23 MB, well inside 64 MB


def dump_outputs(out_dir, n, take, violations, deliveries):
    """Write the last timed step's output as a caller of the fuzz path receives it: every field of the result records
    of a fixed, seeded sample of DUMP_RECORDS records (all records when the batch is smaller; `take(idx)` returns them
    as RESULT_DTYPE), 64-bit hashes split into exact 32-bit halves, and the step's violation / delivery counts."""
    import numpy as np
    from demi_b200 import _native as N
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(n, DUMP_RECORDS, replace=False)) if n > DUMP_RECORDS else np.arange(n)
    rec = take(idx)
    arrays = {"record_index": idx, "counts": np.array([violations, deliveries])}
    for f in N.RESULT_DTYPE.names:
        v = rec[f].astype(np.uint64)
        if N.RESULT_DTYPE[f].itemsize == 8:
            arrays[f + "_lo"], arrays[f + "_hi"] = v & np.uint64(0xFFFFFFFF), v >> np.uint64(32)
        else:
            arrays[f] = v
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_reference(args):
    """CPU arm: the oracle on all host cores, the same batch definition as the GPU arm (same_config)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from demi_b200 import events
    from oracle import binding as O
    O.lib(private=True)
    ext = events.pack_externals(events.raft5_program())
    cores = host_cores()
    n = args.prefixes
    for w in range(args.warmup):                 # warm-up only touches the caches: a small batch is enough
        O.fuzz_batch(MODEL_RAFT5, ext, 1 + w * 100_000, 100_000, MAX_MESSAGES, INTERVAL, model_flags=MODEL_FLAGS, threads=cores)
    t0 = time.perf_counter()
    for s in range(args.steps):
        out = O.fuzz_batch(MODEL_RAFT5, ext, 1 + (args.warmup + s) * n, n, MAX_MESSAGES, INTERVAL,
                           model_flags=MODEL_FLAGS, threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, n, lambda idx: out[idx], int((out["violation"] != 0).sum()),
                     int(out["steps"].sum(dtype="u8")))
    value = n * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "prefixes/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": workload_config(n, args.gpus),
        "cpu_baseline": {"value": value, "per_core": value / cores, "unit": "prefixes/s", "cores": cores, "kind": "port",
                         "sample": "%d prefixes per step x %d steps (C oracle -O3 -march=native, %d pthreads); the JVM "
                                   "reference cannot run here (no JDK/sbt/Akka/akka-raft)" % (n, args.steps, cores)},
        "e2e": {"value": value, "unit": "prefixes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--prefixes", type=int, default=PREFIXES_PER_STEP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.prefixes < 1:
        ap.error("--steps and --prefixes must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import demi_b200 as D
    n = args.prefixes
    W, K = max(args.warmup, 0), args.steps
    eng = D.Engine(D.SchedulerConfig(MODEL_RAFT5, model_flags=MODEL_FLAGS, device=local_rank))
    prog = D.raft5_program()
    ext = D.pack_externals(prog)
    eng.set_externals(ext)
    results_dev = torch.empty(n * RESULT_BYTES, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    from demi_b200 import sharding

    def seed_of(step):      # disjoint seed ranges per (step, rank)
        return sharding.seed_range(step, rank, world, n)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------ device-resident timing ("value")
    for s in range(W):
        eng.fuzz_batch_dev(seed_of(s), n, MAX_MESSAGES, INTERVAL, results_dev.data_ptr(), stream.cuda_stream)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    launches = 0
    barrier()
    evs[0].record(stream)
    for s in range(K):
        eng.fuzz_batch_dev(seed_of(W + s), n, MAX_MESSAGES, INTERVAL, results_dev.data_ptr(), stream.cuda_stream)
        launches += int(eng.stats().kernel_launches)           # counted by the library per batch call
        evs[s + 1].record(stream)
    barrier()
    total_ms = evs[0].elapsed_time(evs[K])
    kernel_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(K)]
    nv, ss = eng.fuzz_summary_dev(stream.cuda_stream)   # counters of the last step
    if args.dump_outputs and rank == 0:
        records = results_dev.view(n, RESULT_BYTES)
        dump_outputs(args.dump_outputs, n,
                     lambda idx: records[torch.from_numpy(idx).to(dev)].cpu().numpy().reshape(-1).view(D._native.RESULT_DTYPE),
                     nv, ss)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    cnt = torch.tensor([float(nv), float(ss)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    total_ms_max = float(t.item())
    value = n * world * K / (total_ms_max * 1e-3)

    # ------------------------------------------------ end-to-end through the host C ABI ("e2e")
    host_out = torch.empty(n * RESULT_BYTES, dtype=torch.uint8, pin_memory=True)
    host_np = host_out.numpy().view(D._native.RESULT_DTYPE)
    e2e_steps = max(1, min(K, 3))
    for s in range(1):
        eng.set_externals(ext)
        eng.fuzz_batch(seed_of(s), n, MAX_MESSAGES, INTERVAL, out=host_np)
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        eng.set_externals(ext)                                   # H2D: the external-event program
        eng.fuzz_batch(seed_of(W + s), n, MAX_MESSAGES, INTERVAL, out=host_np)   # kernel + D2H of every record
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    te = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = n * world * e2e_steps / float(te.item())
    last_viol = int((host_np["violation"] != 0).sum())
    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=2)

    line = None
    if rank == 0:
        peak, peak_kind = measured_peak_hbm()
        k_ms = sum(kernel_ms) / len(kernel_ms)
        achieved = n * RESULT_BYTES / (k_ms * 1e-3) / 1e9
        ver = D._native.lib().demi_version().decode()
        build_id, k1_id = ver.split("build ")[-1].split(" ")[0], ver.split(" k1 ")[-1]
        prof, stale = k1_profile(k1_id)
        lane = not os.environ.get("DEMI_DISABLE_LANE_ENGINE")
        line = {
            "metric": METRIC, "value": value, "unit": "prefixes/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic", "config": workload_config(n, world),
            "deliveries_per_s": float(cnt[1].item()) * K / (total_ms_max * 1e-3),
            "violations_last_step": int(cnt[0].item()),
            "e2e": {"value": e2e_value, "unit": "prefixes/s", "h2d_bytes_per_step": int(ext.nbytes),
                    "d2h_bytes_per_step": n * RESULT_BYTES + 16, "steps": e2e_steps,
                    "violations_last_step_rank0": last_viol},
            "gpu_launches": launches,
            "build_id": build_id, "k1_id": k1_id,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "peak_kind": peak_kind,
                         "traffic": (prof["dram_bytes_per_prefix"] * n) if prof else None,
                         "kernel": ("fuzz_lane_kernel<Raft5,256,96> (+ fuzz_kernel<Raft5,256,32> for deferred prefixes)"
                                    if lane else "fuzz_kernel<Raft5,256,32> (warp engine; lane engine disabled)"),
                         "algorithmic_bytes_per_prefix": RESULT_BYTES, "kernel_ms": k_ms,
                         "from_profile": ({k: prof[k] for k in ("capture", "k1_id", "dram_bytes_per_prefix",
                                                               "issue_slot_utilisation", "warp_instructions_per_prefix",
                                                               "active_lanes_per_instruction", "prefixes") if k in prof}
                                          if prof else None),
                         "profile_stale": stale,
                         "note": "on-chip-state fuzz regime (SURVEY §8d R1): the only algorithmic HBM traffic is the "
                                 "32 B result record, so the kernel is issue-slot bound, not HBM bound; `traffic` and "
                                 "`from_profile` are per-launch figures scaled from the ncu capture named there"},
            "clocks": sampler.summary(),
        }
        line["cpu_baseline"] = None                 # timed at N=1 only (rank 0)
        if not args.no_cpu_baseline and world == 1:
            from oracle import binding as O
            O.lib(private=True)
            cores = host_cores()
            ncpu = 125_000 * cores
            O.fuzz_batch(MODEL_RAFT5, ext, 1, 50_000, MAX_MESSAGES, INTERVAL, model_flags=MODEL_FLAGS, threads=cores)
            t0 = time.perf_counter()
            reps = 0
            while time.perf_counter() - t0 < 2.5 and reps < 40:
                O.fuzz_batch(MODEL_RAFT5, ext, seed_of(W) + reps * ncpu, ncpu, MAX_MESSAGES, INTERVAL,
                             model_flags=MODEL_FLAGS, threads=cores)
                reps += 1
            cdt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": ncpu * reps / cdt, "per_core": ncpu * reps / cdt / cores, "unit": "prefixes/s",
                                    "cores": cores, "kind": "port",
                                    "sample": "%d prefixes of the same workload (C oracle -O3 -march=native, %d pthreads, "
                                              "%.1f s)" % (ncpu * reps, cores, cdt)}

    # ------------------------------------------------ secondary configs (outside the headline's timed region)
    if not args.no_secondary:
        from tools import secondary
        try:
            sec = secondary.run_all(eng, rank, world, local_rank, results_dev, n, host_cores(), with_cpu=not args.no_cpu_baseline)
        except Exception as e:                      # a failing secondary leg must not take the headline with it
            sec = {"error": "%s: %s" % (type(e).__name__, e)}
        if rank == 0:
            line["secondary"] = sec
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
