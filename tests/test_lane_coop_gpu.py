"""The raft5 lane engine (fuzz_lane_kernel: one thread per prefix) vs the CPU oracle, record by record, over 10^5
prefixes per case, in the corners where applying a delivery's sends and timer flushes is easy to get wrong: sends
that are recorded but not inserted (partitions, killed actors), capacity defers, short and long runs, invariant
intervals, looking_for, external Sends at segment starts, and both Raft variants.  Any rework of how the lane engine
applies those operations (profiles/r3_k1_coop_fanout.md) must keep these green."""
import numpy as np
import pytest

import demi_b200 as D
from demi_b200 import _native as N

pytestmark = pytest.mark.gpu

N_PREFIXES = 100_000
RAFT5_BOOT, RAFT5_CLIENT_CMD = 1, 2


def partitioned_program():
    """Partitions and a Kill injected before the first delivery: sends across them are recorded, never delivered."""
    ev = [D.Start(a) for a in range(5)]
    ev += [D.Partition(0, 1), D.Partition(3, 2), D.Kill(4)]
    ev += [D.Send(a, RAFT5_BOOT, 0x1F) for a in range(5)]
    ev.append(D.WaitQuiescence())
    return ev


def segmented_program():
    """Three quiescent segments (timers ignored, so each one ends), each starting with external Sends."""
    ev = [D.Start(a) for a in range(5)]
    ev += [D.Send(a, RAFT5_BOOT, 0x1F) for a in range(5)]
    ev += [D.WaitQuiescence(), D.Partition(0, 1), D.Kill(2)]
    ev += [D.Send(k % 5, RAFT5_CLIENT_CMD, 1 + k) for k in range(6)]
    ev += [D.WaitQuiescence(), D.UnPartition(0, 1), D.Start(2)]
    ev += [D.Send(k % 5, RAFT5_CLIENT_CMD, 20 + k) for k in range(6)]
    ev.append(D.WaitQuiescence())
    return ev


CASES = [
    # id, program, model_flags, max_messages, interval, looking_for, ignore_timers
    ("partitions-kill", partitioned_program, 1, 50, 5, 0, 0),
    ("max-messages-3", D.raft5_program, 1, 3, 1, 0, 0),
    ("max-messages-200", lambda: D.raft5_program(client_cmds=3), 1, 200, 5, 0, 0),
    ("interval-1", D.raft5_program, 1, 50, 1, 0, 0),
    ("interval-7", D.raft5_program, 1, 50, 7, 0, 0),
    ("looking-for", D.raft5_program, 1, 50, 5, 1, 0),
    ("multi-segment", segmented_program, 1, -1, 0, 0, 1),
    ("no-bug", lambda: D.raft5_program(client_cmds=2), 0, 50, 5, 0, 0),
    ("double-vote-bug", lambda: D.raft5_program(client_cmds=2), 1, 50, 5, 0, 0),
]


def run_both(oracle, prog, flags, maxm, interval, looking_for, ignore, seed=1, n=N_PREFIXES):
    ext = D.pack_externals(prog())
    eng = D.Engine(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=flags, ignoreTimers=bool(ignore)))
    eng.set_externals(ext)
    gpu = eng.fuzz_batch(seed, n, maxm, interval, looking_for=looking_for)
    deferred = eng.stats().deferred
    eng.close()
    cpu = oracle.fuzz_batch(N.MODEL_RAFT5, ext, seed, n, maxm, interval, model_flags=flags, ignore_timers=ignore,
                            looking_for=looking_for)
    return gpu, cpu, deferred


def assert_same(gpu, cpu):
    for f in N.RESULT_DTYPE.names:
        bad = np.nonzero(gpu[f] != cpu[f])[0]
        assert len(bad) == 0, "field %s differs at %d prefixes, first idx %d: gpu=%s cpu=%s" % (
            f, len(bad), bad[0], gpu[bad[0]], cpu[bad[0]])


@pytest.fixture(autouse=True)
def lane_engine(monkeypatch):
    monkeypatch.delenv("DEMI_DISABLE_LANE_ENGINE", raising=False)
    monkeypatch.delenv("DEMI_LANE_PENDING_CAP", raising=False)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_lane_engine_matches_oracle(case, oracle):
    _, prog, flags, maxm, interval, looking_for, ignore = case
    gpu, cpu, _ = run_both(oracle, prog, flags, maxm, interval, looking_for, ignore)
    assert_same(gpu, cpu)
    assert (gpu["status"] == 0).all()


def test_partitioned_sends_are_recorded_but_not_inserted(oracle):
    """The partitioned case really has sends that cross a partition or go to the killed actor."""
    ext = D.pack_externals(partitioned_program())
    ev, _, _ = oracle.fuzz_trace(N.MODEL_RAFT5, ext, 3, 50, 5, model_flags=1)
    dropped = [e for e in ev if e["kind"] == N.EV_MSG_SEND and e["src"] < 5 and
               ((e["src"], e["dst"]) in ((0, 1), (1, 0), (3, 2), (2, 3)) or e["dst"] == 4)]
    assert dropped


def test_capacity_defers_are_exact(oracle, monkeypatch):
    """A pending-set bound low enough that many prefixes defer mid-delivery and are re-run by the warp engine."""
    monkeypatch.setenv("DEMI_LANE_PENDING_CAP", "14")
    gpu, cpu, deferred = run_both(oracle, D.raft5_program, 1, 50, 5, 0, 0)
    assert 0 < deferred < N_PREFIXES
    assert_same(gpu, cpu)


def test_bench_workload_defers_nothing():
    """The headline workload (bench.py: raft5, double-vote bug, depth 50, interval 5, 10^7 prefixes) runs entirely on
    the lane engine."""
    eng = D.Engine(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=1))
    eng.set_externals(D.pack_externals(D.raft5_program()))
    n = 10_000_000
    out = eng.fuzz_batch(1, n, 50, 5)
    assert eng.stats().deferred == 0
    assert (out["status"] == 0).all()
    eng.close()
