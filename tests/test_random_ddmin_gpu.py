"""DDMin with RandomScheduler as the TestOracle on the GPU: demi_fuzz_subseq_batch against the single-test path
(demi_set_externals(program_of(mask)) + demi_fuzz_batch on a second handle), demi_random_ddmin against the CPU
reference (random_ddmin_ref), and random_ddmin's EventTrace."""
import os
import subprocess
import sys

import numpy as np
import pytest

import demi_b200 as D
from demi_b200 import _native as N, fuzzer as F
from demi_b200.schedulers import program_of
import random_ddmin_ref as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fuzzed_raft(n_events, seed):
    prefix = [D.Start(a) for a in range(5)] + [D.Send(a, 1, 0x1F) for a in range(5)]
    return D.pack_externals(F.Fuzzer(n_events, F.FuzzerWeights(), F.ClientCommandGenerator(2), prefix, seed=seed).generateFuzzTest())


def _random_masks(n_ext, n, rng):
    out = np.zeros((n, R.mask_words(n_ext)), dtype=np.uint64)
    for t in range(n):
        sel = np.nonzero(rng.random(n_ext) < rng.uniform(0.2, 0.9))[0]
        if not len(sel):
            sel = [int(rng.integers(n_ext))]
        out[t] = R.mask_from(sel, n_ext)
    return out


def _single(eng, ext, mask, K, seed_base, max_messages, interval, looking_for):
    eng.set_externals(program_of(ext, mask))
    res = eng.fuzz_batch(seed_base, K, max_messages, interval, looking_for)
    ends = np.nonzero((res["violation"] != 0) | (res["status"] != 0))[0]
    if not len(ends):
        return K, K
    i = int(ends[0])
    return (K, i) if res["status"][i] else (i, K)


def _parity(cfg, ext, max_messages, interval, looking_for=0, filt=None, K=512, n=200, seed_base=7, masks=None):
    rng = np.random.default_rng(len(ext) * 131 + cfg.model_flags)
    if masks is None:
        masks = _random_masks(len(ext), n, rng)
    a, b = D.Engine(cfg), D.Engine(cfg)
    if filt:
        a.set_user_filter(filt); b.set_user_filter(filt)
    a.set_externals(ext)
    hit, bad = a.fuzz_subseq_batch(masks, K, max_messages, interval, seed_base, looking_for)
    st = a.stats()
    want = np.array([_single(b, ext, m, K, seed_base, max_messages, interval, looking_for) for m in masks])
    assert (hit == want[:, 0]).all() and (bad == want[:, 1]).all()
    assert st.prefixes <= len(masks) * K
    return hit, bad, st


RAFT_FZ = _fuzzed_raft(40, 11)


@pytest.mark.parametrize("flags", [0, 1, 2])
def test_subseq_batch_raft5_matches_single_tests(flags):
    hit, _, _ = _parity(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=flags), RAFT_FZ, 60, 5)
    if flags == 1:
        assert (hit < 512).any() and (hit == 512).any()


def test_subseq_batch_pingpong3_and_bcast32_match_single_tests():
    _parity(D.SchedulerConfig(N.MODEL_PINGPONG3, model_flags=1), D.pack_externals(D.pingpong3_program(20)), 40, 5)
    _parity(D.SchedulerConfig(N.MODEL_BCAST32), D.pack_externals(D.bcast32_program(2)), 60, 3, n=60)


def test_subseq_batch_blocked_actors_and_user_filter_warp_engine():
    rules = [(1 << 2, 0xFFFFFFFF, 1 << 3, 0)]
    _parity(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=1, blocked_mask=1 << 4), RAFT_FZ, 60, 5, filt=rules)


def test_subseq_batch_src_dst_fifo():
    _parity(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=1, strategy=1), RAFT_FZ, 60, 5)


def test_subseq_batch_capacity_status_before_a_hit():
    # more than ~1008 Sends overflow messagesToSend (demi_tosend_cap clamps at 1024) on the first inject; fewer violate
    ext = D.pack_externals(D.pingpong3_program(1100))
    rng = np.random.default_rng(5)
    masks = np.stack([R.mask_from(np.nonzero(rng.random(len(ext)) < (0.99 if t % 2 else 0.5))[0], len(ext)) for t in range(24)])
    hit, bad, _ = _parity(D.SchedulerConfig(N.MODEL_PINGPONG3, model_flags=1), ext, 40, 5, K=64, masks=masks)
    assert (bad < 64).any() and (hit < 64).any()


def test_subseq_batch_forced_lane_deferral():
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import test_random_ddmin_gpu as T, demi_b200 as D\n"
            "from demi_b200 import _native as N\n"
            "h, b, st = T._parity(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=1), T.RAFT_FZ, 60, 5)\n"
            "assert st.deferred > 0, st.deferred\n"
            "print('ok', st.deferred)\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, DEMI_LANE_PENDING_CAP="4")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


# ---------------------------------------------------------------- demi_random_ddmin
DD_CASES = [(1, ()), (64, ()), (1024, ()), (64, ((5, 20),))]


@pytest.mark.parametrize("K,pairs", DD_CASES, ids=["k1", "k64", "k1024", "k64_conjoined"])
def test_random_ddmin_matches_the_cpu_reference(oracle, K, pairs):
    ext, mm, iv, flags = RAFT_FZ, 60, 5, 1
    eng = D.Engine(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=flags))
    eng.set_externals(ext)
    before = eng.fuzz_batch(3, 4096, mm, iv)
    mcs, sizes, keys, out, vseed = eng.random_ddmin(K, mm, iv, 0, 0, pairs)
    ref = R.ddmin_random(N.MODEL_RAFT5, ext, K, 0, mm, iv, conjoin_pairs=pairs, model_flags=flags)
    assert R.indices_of(mcs, len(ext)) == R.indices_of(ref["mcs"], len(ext))
    assert out.total_replays == ref["executions"]
    assert list(sizes) == ref["sizes"] and list(keys) == ref["keys"]
    assert bool(out.verified) == ref["verified"] and vseed == ref["verify_seed"]
    assert out.replays_executed >= len(set(ref["tests"]))
    # the handle's program is unchanged, and a second call gives the same answer
    assert (eng.fuzz_batch(3, 4096, mm, iv) == before).all()
    again = eng.random_ddmin(K, mm, iv, 0, 0, pairs)
    assert (again[0] == mcs).all() and (again[1] == sizes).all() and (again[2] == keys).all()
    assert again[3].total_replays == out.total_replays and again[4] == vseed


def test_random_ddmin_unmodified_check_error():
    eng = D.Engine(D.SchedulerConfig(N.MODEL_RAFT5, model_flags=0))       # no bug: nothing violates
    eng.set_externals(RAFT_FZ)
    with pytest.raises(D.DemiError) as e:
        eng.random_ddmin(4, 60, 5, check_unmodified=True)
    assert "Unmodified trace does not trigger violation" in str(e.value)


def test_random_ddmin_event_trace_is_the_verification_execution(tmp_path):
    from demi_b200 import experiment as X
    cfg = D.SchedulerConfig(N.MODEL_RAFT5, model_flags=1)
    eng = D.Engine(cfg)
    eng.set_externals(RAFT_FZ)
    res = eng.fuzz_batch(0, 4096, 200, 5)
    seed = int(np.nonzero(res["violation"])[0][0])
    ev, par, r = eng.fuzz_trace(seed, 200, 5)
    X.save_experiment(str(tmp_path), N.MODEL_RAFT5, 1, RAFT_FZ, ev, int(r["violation"]), dep_parent=par)
    exp = X.load_experiment(str(tmp_path))
    mcs, stats, trace, viol = D.random_ddmin(exp, cfg, max_executions=16, interval=5)
    assert viol == int(r["violation"]) and 0 < len(mcs) < len(RAFT_FZ)
    assert trace is not None
    assert stats.total_replays > 0 and len(stats.inner().iterationSize) > 0
    # the trace is demi_fuzz_trace at the verification seed on program_of(mcs)
    mcs_mask, _, _, out, vseed = eng.random_ddmin(16, len(ev), 5, 0, int(r["violation"]))
    assert vseed is not None and D.events_of(D.unpack_externals(RAFT_FZ), mcs_mask) == mcs
    other = D.Engine(cfg)
    other.set_externals(program_of(RAFT_FZ, mcs_mask))
    want = other.fuzz_trace(vseed, len(ev), 5, int(r["violation"]))[0]
    assert (trace == want).all()
