"""DDMin with RandomScheduler as the TestOracle (RunnerUtils.randomDDMin) on the CPU: program_of, and the CPU
reference (random_ddmin_ref) against the independent DDMin of micro_oracle driven by the same tests."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import demi_b200 as D
from demi_b200 import _native as N
from demi_b200.schedulers import program_of
import micro_oracle as M
import random_ddmin_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _mask(n, idx):
    return R.mask_from(idx, n)


# ---------------------------------------------------------------- program_of
def test_program_of_collapses_adjacent_wait_quiescence():
    prog = [D.Start(0), D.WaitQuiescence(), D.Send(0, 1, 7), D.WaitQuiescence(), D.Start(1)]
    out = program_of(prog, _mask(5, [0, 1, 3, 4]))              # dropping the Send makes two WaitQuiescence adjacent
    assert [type(e) for e in out] == [D.Start, D.WaitQuiescence, D.Start]
    assert out[1] is prog[1]
    packed = D.pack_externals(prog)
    outp = program_of(packed, _mask(5, [0, 1, 3, 4]))
    assert list(outp["id"]) == [prog[0]._id, prog[1]._id, prog[4]._id]


def test_program_of_keeps_a_leading_wait_quiescence_and_the_order():
    prog = [D.WaitQuiescence(), D.Start(0), D.WaitQuiescence(), D.Start(2)]
    out = program_of(prog, _mask(4, [0, 1, 2, 3]))
    assert [type(e) for e in out] == [D.WaitQuiescence, D.Start, D.WaitQuiescence, D.Start]
    assert out[0] is prog[0]
    # a leading WaitQuiescence is kept when the next selected event is one as well: only the second goes
    assert [type(e) for e in program_of(prog, _mask(4, [0, 2, 3]))] == [D.WaitQuiescence, D.Start]
    assert program_of(prog, _mask(4, [0, 2]))[0] is prog[0]


def test_program_of_rejects_the_empty_mask():
    with pytest.raises(ValueError):
        program_of([D.Start(0)], np.zeros(1, dtype=np.uint64))


# ---------------------------------------------------------------- DDMin: reference vs micro_oracle.DDMin
def _as_tuples(ext):
    """externals as micro_oracle events, each tagged with its index (atomic_events keys on fields 1 and 2)"""
    names = {N.EXT_START: "Start", N.EXT_KILL: "Kill", N.EXT_SEND: "Send", N.EXT_WAIT_QUIESCENCE: "WaitQuiescence",
             N.EXT_PARTITION: "Partition", N.EXT_UNPARTITION: "UnPartition"}
    out = []
    for i, r in enumerate(ext):
        k = int(r["kind"])
        if k in (N.EXT_PARTITION, N.EXT_UNPARTITION):
            out.append((names[k], int(r["a"]), int(r["b"]), i))
        else:
            out.append((names[k], int(r["a"]), i))
    return out


def _programs():
    raft = D.pack_externals(D.raft5_program())
    pp = D.pack_externals(D.pingpong3_program())
    # Start 0..4, a WaitQuiescence after every Send (removals make them adjacent), a partition pair and a kill
    mixed = [D.Start(a) for a in range(5)] + [D.WaitQuiescence()]
    for a in range(5):
        mixed += [D.Send(a, 1, 0x1F), D.WaitQuiescence()]
    mixed += [D.Partition(0, 1), D.Send(2, 2, 5), D.WaitQuiescence(), D.UnPartition(0, 1), D.Kill(3), D.Send(1, 2, 6)]
    return raft, pp, D.pack_externals(mixed)


RAFT, PP, MIXED = _programs()
CASES = [
    ("raft5_f1_k1", N.MODEL_RAFT5, RAFT, 1, 1, 0),
    ("raft5_f1_k8", N.MODEL_RAFT5, RAFT, 1, 8, 3),
    ("raft5_f2_k1", N.MODEL_RAFT5, RAFT, 2, 1, 0),
    ("raft5_f2_k8", N.MODEL_RAFT5, RAFT, 2, 8, 11),
    ("mixed_f1_k1", N.MODEL_RAFT5, MIXED, 1, 1, 5),
    ("mixed_f1_k8", N.MODEL_RAFT5, MIXED, 1, 8, 0),
    ("mixed_f2_k8", N.MODEL_RAFT5, MIXED, 2, 8, 2),
    ("pingpong3_k1", N.MODEL_PINGPONG3, PP, 1, 1, 0),
    ("pingpong3_k8", N.MODEL_PINGPONG3, PP, 1, 8, 4),
]


@pytest.mark.parametrize("name,model,ext,flags,K,seed_base", CASES, ids=[c[0] for c in CASES])
def test_reference_matches_micro_oracle_ddmin(oracle, name, model, ext, flags, K, seed_base):
    max_messages, interval = 60, 5
    n = len(ext)
    ref = R.ddmin_random(model, ext, K, seed_base, max_messages, interval, model_flags=flags)
    hits = []

    def test(events):
        idx = sorted(e[-1] for e in events)
        hit, bad = R.fuzz_subseq(model, ext, R.mask_from(idx, n), K, seed_base, max_messages, interval, model_flags=flags)
        assert bad == K
        hits.append(hit)
        return hit < K

    mo = M.DDMin(test)
    mcs = mo.minimize(_as_tuples(ext))
    assert sorted(i for i, _ in mcs) == R.indices_of(ref["mcs"], n)
    assert mo.tests == ref["tests"]
    assert hits == ref["hits"]
    assert mo.total_replays == len(ref["tests"])
    assert ref["executions"] == sum(h + 1 if h < K else K for h in hits)
    assert ref["keys"] == sorted(ref["keys"]) and len(ref["keys"]) == len(ref["sizes"]) == len(ref["tests"]) + 1


def test_reference_conjoined_pair_stays_together(oracle):
    n = len(MIXED)
    ref = R.ddmin_random(N.MODEL_RAFT5, MIXED, 4, 0, 60, 0, model_flags=1, conjoin_pairs=[(5, 17)])
    for t in ref["tests"]:
        assert (5 in t) == (17 in t)
    m = R.indices_of(ref["mcs"], n)
    assert (5 in m) == (17 in m)


# ---------------------------------------------------------------- the C++ host header
def test_hpp_compiles_with_the_random_ddmin_member():
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    src = '#include "demi_b200.hpp"\nint main() { return 0; }\n'
    r = subprocess.run([gxx, "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-x", "c++", "-"],
                       input=src.encode(), capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
