"""CPU reference of DDMin with RandomScheduler as the TestOracle (RunnerUtils.randomDDMin, RunnerUtils.scala:601-623),
built on the CPU oracle's fuzz_batch (oracle/binding.py).  Test infrastructure only.

fuzz_subseq runs one test the reference's way: executions i = 0, 1, ... of program_of(mask), one after another,
until the first that ends on a matching violation (a hit) or on a capacity status.  ddmin_random is DDMin
(DeltaDebugging.scala:27-109) over the whole program, WaitQuiescence included, with Kill/Start, Partition/UnPartition
and explicitly conjoined pairs as atoms (UnmodifiedEventDag.get_atomic_events, minification/Util.scala:197-265)."""
import numpy as np

from demi_b200 import _native as N
from demi_b200.schedulers import program_of
from oracle import binding as O


def mask_words(n_ext):
    return max(1, (n_ext + 63) // 64)


def mask_from(indices, n_ext):
    m = np.zeros(mask_words(n_ext), dtype=np.uint64)
    for i in indices:
        m[i // 64] |= np.uint64(1) << np.uint64(i % 64)
    return m


def indices_of(mask, n_ext):
    return [i for i in range(n_ext) if (int(mask[i // 64]) >> (i % 64)) & 1]


def fuzz_subseq(model, ext, mask, K, seed_base, max_messages, interval, looking_for=0, **cfg):
    """(first_hit, first_bad) of one test; the one that did not end the test is K."""
    prog = program_of(ext, mask)
    i = 0
    while i < K:
        n = min(K - i, 1 if i < 4 else 64)          # run ahead in small blocks: each execution is a pure function of its seed
        res = O.fuzz_batch(model, prog, seed_base + i, n, max_messages, interval, looking_for=looking_for, threads=1, **cfg)
        for k in range(n):
            if res["status"][k]:
                return K, i + k
            if res["violation"][k]:
                return i + k, K
        i += n
    return K, K


def atomic_events(ext, idx, conjoined):
    """UnmodifiedEventDag.get_atomic_events over the externals `idx` (sorted); atoms as sorted index tuples."""
    atoms, last_start, last_part = [], {}, {}
    sel = set(idx)
    for i in idx:
        p = conjoined.get(i)
        if p is not None:
            if p not in sel:
                raise ValueError("conjoined atom with one half missing")
            if p > i:
                atoms.append((i, p))
    for i in idx:
        if i in conjoined:
            continue
        k, a, b = int(ext[i]["kind"]), int(ext[i]["a"]), int(ext[i]["b"])
        if k == N.EXT_KILL:
            atoms.append((last_start.pop(a), i))
        elif k == N.EXT_START:
            last_start[a] = i
        elif k == N.EXT_PARTITION:
            last_part[(a, b)] = i
        elif k == N.EXT_UNPARTITION:
            atoms.append((last_part.pop((a, b)), i))
        else:
            atoms.append((i,))
    atoms += [(v,) for v in last_start.values()] + [(v,) for v in last_part.values()]
    return sorted(atoms, key=lambda a: a[0])


def ddmin_random(model, ext, K, seed_base, max_messages, interval, looking_for=0, conjoin_pairs=(),
                 check_unmodified=False, **cfg):
    """Returns a dict: mcs (mask), tests (list of index tuples, in order), hits (first_hit per test), sizes, keys,
    executions (stats.total_replays), verified, verify_seed."""
    n = len(ext)
    conj = {}
    for a, b in conjoin_pairs:
        conj[a], conj[b] = b, a
    log = {"tests": [], "hits": [], "sizes": [], "keys": [], "executions": 0}
    memo = {}

    def test(idx, counted):
        key = tuple(idx)
        if key not in memo:
            memo[key] = fuzz_subseq(model, ext, mask_from(idx, n), K, seed_base, max_messages, interval, looking_for, **cfg)
        hit, bad = memo[key]
        if bad < K:
            raise RuntimeError("capacity status in execution %d" % bad)
        if counted:
            log["tests"].append(key)
            log["hits"].append(hit)
            log["executions"] += hit + 1 if hit < K else K
        return hit

    state = {"pruned": 0}

    def ddmin2(dag, rem):
        atoms = atomic_events(ext, dag, conj)
        if len(atoms) <= 1:
            return dag
        n0 = (len(atoms) + 1) // 2
        halves = [sorted(x for a in atoms[:n0] for x in a), sorted(x for a in atoms[n0:] for x in a)]
        for h in halves:
            union = sorted(set(h) | set(rem))
            hit = test(union, True)
            log["sizes"].append(n - state["pruned"])
            log["keys"].append(log["executions"])
            if hit < K:
                state["pruned"] += len(dag) - len(h)
                return ddmin2(h, rem)
        left = ddmin2(halves[0], sorted(set(halves[1]) | set(rem)))
        right = ddmin2(halves[1], sorted(set(halves[0]) | set(rem)))
        return sorted(set(left) | set(right))

    full = list(range(n))
    if check_unmodified and test(full, False) >= K:
        raise ValueError("Unmodified trace does not trigger violation")
    mcs = ddmin2(full, [])
    log["sizes"].append(n - state["pruned"])
    log["keys"].append(log["executions"])
    hit = test(mcs, False)
    log["mcs"] = mask_from(mcs, n)
    log["verified"] = hit < K
    log["verify_seed"] = seed_base + hit if hit < K else None
    return log
