"""ctypes binding of the CPU oracle (oracle/liboracle.so).

ORACLE — test infrastructure only.  Import this from tests/, from
__graft_entry__.smoke() and from bench.py's cpu_baseline / --impl reference
legs only; never from the demi_b200 package.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liboracle.so")

EXT_DTYPE = np.dtype([("kind", "u1"), ("a", "u1"), ("b", "u1"), ("type", "u1"),
                      ("p0", "<u4"), ("p1", "<u4"), ("id", "<u4")])
EVENT_DTYPE = np.dtype([("kind", "u1"), ("src", "u1"), ("dst", "u1"), ("type", "u1"),
                        ("p0", "<u4"), ("p1", "<u4"), ("uniq", "<u2"), ("node", "<u2")])
RESULT_DTYPE = np.dtype([("violation", "<u4"), ("steps", "<u4"), ("state_hash", "<u8"), ("trace_hash", "<u8"),
                         ("n_nodes", "<u2"), ("n_events", "<u2"), ("max_pending", "<u2"), ("status", "<u2")])


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("model", C.c_int32), ("model_flags", C.c_uint32),
                ("blocked_mask", C.c_uint32), ("ignore_timers", C.c_int32), ("strategy", C.c_int32), ("reserved", C.c_int32 * 2)]


class FuzzParams(C.Structure):
    _fields_ = [("seed_base", C.c_int64), ("n_prefixes", C.c_uint64), ("max_messages", C.c_int32),
                ("invariant_check_interval", C.c_int32), ("looking_for", C.c_uint32), ("flags", C.c_uint32)]


_lib = None


def lib(private=False):
    """Load the oracle once.  private=True: never write into the tree (see build.build_oracle); a library built
    elsewhere is removed as soon as it is loaded."""
    global _lib
    if _lib is None:
        # -march=native build: (re)built on the machine that runs it (demi_b200/build.py keeps a CPU stamp)
        import sys
        sys.path.insert(0, os.path.dirname(_HERE))
        from demi_b200 import build
        path = build.build_oracle(private=private)
        _lib = C.CDLL(path)
        if path != LIB_PATH:
            import shutil
            shutil.rmtree(os.path.dirname(path))
    return _lib


def fuzz_batch(model, ext, seed_base, n, max_messages, interval, model_flags=0, blocked_mask=0,
               ignore_timers=0, looking_for=0, threads=None, flags=0, strategy=0):
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    cfg = Config(0, model, model_flags, blocked_mask, ignore_timers, strategy)
    p = FuzzParams(seed_base, n, max_messages, interval, looking_for, flags)
    out = np.empty(n, dtype=RESULT_DTYPE)
    threads = threads or (os.cpu_count() or 1)
    rc = lib().oracle_fuzz_batch(C.byref(cfg), C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)), C.byref(p),
                                 C.c_void_p(out.ctypes.data), C.c_int(threads))
    if rc != 0:
        raise RuntimeError("oracle_fuzz_batch failed: %d" % rc)
    return out


def fuzz_trace(model, ext, seed, max_messages, interval, model_flags=0, blocked_mask=0, ignore_timers=0,
               looking_for=0, cap_events=65536, cap_nodes=65536, strategy=0):
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    cfg = Config(0, model, model_flags, blocked_mask, ignore_timers, strategy)
    p = FuzzParams(seed, 1, max_messages, interval, looking_for, 0)
    ev = np.zeros(cap_events, dtype=EVENT_DTYPE)
    par = np.zeros(cap_nodes, dtype=np.uint16)
    ne, nn = C.c_uint32(), C.c_uint32()
    res = np.zeros(1, dtype=RESULT_DTYPE)
    lib().oracle_fuzz_trace(C.byref(cfg), C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)), C.byref(p),
                            C.c_int64(seed), C.c_void_p(ev.ctypes.data), C.c_uint32(cap_events), C.byref(ne),
                            C.c_void_p(par.ctypes.data), C.c_uint32(cap_nodes), C.byref(nn),
                            C.c_void_p(res.ctypes.data))
    return ev[:ne.value].copy(), par[:nn.value].copy(), res[0]


def kat_jrandom(seed, bound, n):
    out = (C.c_int32 * n)()
    lib().oracle_kat_jrandom(C.c_int64(seed), C.c_int32(bound), C.c_int32(n), out)
    return list(out)


def kat_hashset(seed, ops, blocked_mask=0):
    ops_a = (C.c_int32 * len(ops))(*ops)
    arr = (C.c_int32 * (len(ops) + 1))()
    removed = (C.c_int32 * (len(ops) + 1))()
    nr = C.c_int32()
    n = lib().oracle_kat_hashset(C.c_int64(seed), C.c_uint32(blocked_mask), ops_a, C.c_int32(len(ops)),
                                 arr, removed, C.byref(nr))
    return list(arr[:n]), list(removed[:nr.value])


# ------------------------------------------------------------ STS replay / DDMin
REPLAY_DTYPE = np.dtype([("violation", "<u2"), ("status", "<u2"), ("delivered", "<u2"), ("ignored", "<u2"),
                         ("state_hash", "<u8")])
RF_FILTER_KNOWN_ABSENTS, RF_STRICT = 1, 2
_EXT_TYPE_MASK = {1: 1 << 1, 2: (1 << 1) | (1 << 2), 3: 1 << 2}


class ReplayInput(C.Structure):
    _fields_ = [("events", C.c_void_p), ("n_events", C.c_uint32), ("externals", C.c_void_p),
                ("n_externals", C.c_uint32), ("external_type_mask", C.c_uint32),
                ("pending_cap", C.c_uint32), ("tosend_cap", C.c_uint32)]


def _pow2_at_least(x, lo, hi):
    c = lo
    while c < x and c < hi:
        c <<= 1
    return c


FILTER_RULE_DTYPE = np.dtype([("src_mask", "<u4"), ("dst_mask", "<u4"), ("type_mask", "<u4"), ("flags", "<u4")])


def set_user_filter(rules):
    """FullyRandom(userDefinedFilter) as rules for the following calls on this thread; [] clears."""
    arr = np.array(list(rules), dtype=FILTER_RULE_DTYPE) if len(rules) else np.zeros(0, dtype=FILTER_RULE_DTYPE)
    lib().oracle_set_user_filter(C.c_void_p(arr.ctypes.data) if len(arr) else None, C.c_uint32(len(arr)))


def load_model(blob):
    """oracle_load_model: the CPU interpreter's copy of a demi_load_model blob (model id 100)."""
    rc = lib().oracle_load_model(bytes(blob), C.c_size_t(len(blob)))
    if rc != 0:
        raise RuntimeError("oracle_load_model: %d" % rc)
    lib().oracle_ir_external_mask.restype = C.c_uint32
    _EXT_TYPE_MASK[100] = int(lib().oracle_ir_external_mask())


def make_replay_input(model, events, ext):
    events = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    n_send_ev = int((events["kind"] == 1).sum())
    n_ext_sends = int((ext["kind"] == 3).sum())
    ri = ReplayInput(events.ctypes.data, len(events), ext.ctypes.data, len(ext), _EXT_TYPE_MASK[model],
                     _pow2_at_least(n_send_ev + 8, 64, 8192), _pow2_at_least(n_ext_sends + 16, 32, 1024))
    ri._keep = (events, ext)
    return ri


def mask_words(n_ext):
    return max(1, (n_ext + 63) // 64)


def full_mask(ext, drop_wait_quiescence=True):
    mw = mask_words(len(ext))
    m = np.zeros(mw, dtype=np.uint64)
    for i, e in enumerate(ext):
        if drop_wait_quiescence and e["kind"] == 4:
            continue
        m[i // 64] |= np.uint64(1) << np.uint64(i % 64)
    return m


def replay_batch(model, events, ext, masks, looking_for=0, flags=0, model_flags=0, blocked_mask=0,
                 ignore_timers=0, threads=None):
    ri = make_replay_input(model, events, ext)
    masks = np.ascontiguousarray(masks, dtype=np.uint64).reshape(-1, mask_words(len(ext)))
    cfg = Config(0, model, model_flags, blocked_mask, ignore_timers)
    out = np.zeros(len(masks), dtype=REPLAY_DTYPE)
    lib().oracle_replay_batch(C.byref(cfg), C.byref(ri), C.c_void_p(masks.ctypes.data), C.c_uint32(len(masks)),
                              C.c_uint32(masks.shape[1]), C.c_uint32(looking_for), C.c_uint32(flags),
                              C.c_void_p(out.ctypes.data), C.c_int(threads or (os.cpu_count() or 1)))
    return out


def project(model, events, ext, mask, filter_known_absents=False):
    ri = make_replay_input(model, events, ext)
    mask = np.ascontiguousarray(mask, dtype=np.uint64)
    keep = np.zeros(len(events), dtype=np.uint8)
    lib().oracle_sts_project(C.byref(ri), C.c_void_p(mask.ctypes.data), C.c_int(1 if filter_known_absents else 0),
                             C.c_void_p(keep.ctypes.data))
    return keep


def set_conjoined(pairs, n_ext):
    """UnmodifiedEventDag.conjoinAtoms for the next minimizations on this thread; pairs = [(i, j), ...]; [] clears."""
    global _conj_keep
    if not pairs:
        lib().oracle_set_conjoined(None, C.c_uint32(0))
        _conj_keep = None
        return
    partner = np.full(n_ext, -1, dtype=np.int32)
    for i, j in pairs:
        partner[i], partner[j] = j, i
    _conj_keep = partner
    lib().oracle_set_conjoined(C.c_void_p(partner.ctypes.data), C.c_uint32(n_ext))


_conj_keep = None


def ddmin_sts(model, events, ext, looking_for, flags=0, model_flags=0, check_unmodified=True, cap_iter=65536):
    ri = make_replay_input(model, events, ext)
    cfg = Config(0, model, model_flags, 0, 0)
    mw = mask_words(len(ext))
    mcs = np.zeros(mw, dtype=np.uint64)
    iters = np.zeros(cap_iter, dtype=np.uint32)
    tr, ni, ver = C.c_uint32(), C.c_uint32(), C.c_int()
    rc = lib().oracle_ddmin_sts(C.byref(cfg), C.byref(ri), C.c_uint32(looking_for), C.c_uint32(flags),
                                C.c_int(1 if check_unmodified else 0), C.c_void_p(mcs.ctypes.data), C.c_uint32(mw),
                                C.byref(tr), C.c_void_p(iters.ctypes.data), C.c_uint32(cap_iter), C.byref(ni),
                                C.byref(ver))
    return rc, mcs, tr.value, iters[:ni.value].copy(), ver.value


def ddmin_superset(ext, K, cap=65536):
    """DDMin over `ext` with the monotone oracle "fails iff mask is a superset of K"; returns the test log too."""
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    mw = mask_words(len(ext))
    K = np.ascontiguousarray(K, dtype=np.uint64)
    mcs = np.zeros(mw, dtype=np.uint64)
    iters = np.zeros(cap, dtype=np.uint32)
    log = np.zeros((cap, mw), dtype=np.uint64)
    tr, ni, nl = C.c_uint32(), C.c_uint32(), C.c_uint32()
    rc = lib().oracle_ddmin_superset(C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)), C.c_void_p(K.ctypes.data),
                                     C.c_uint32(mw), C.c_void_p(mcs.ctypes.data), C.byref(tr),
                                     C.c_void_p(iters.ctypes.data), C.c_uint32(cap), C.byref(ni),
                                     C.c_void_p(log.ctypes.data), C.c_uint32(cap), C.byref(nl))
    return rc, mcs, tr.value, iters[:ni.value].copy(), log[:nl.value].copy()


def split_first_len(n, ways, which):
    lib().oracle_split_first_len.restype = C.c_uint32
    return lib().oracle_split_first_len(C.c_uint32(n), C.c_uint32(ways), C.c_uint32(which))


# ----------------------------------------------------------------------- DPOR
class DporParams(C.Structure):
    _fields_ = [("max_messages", C.c_int32), ("depth_bound", C.c_int32), ("max_interleavings", C.c_uint32),
                ("looking_for", C.c_uint32), ("stop_if_found", C.c_uint32), ("node_cap", C.c_uint32),
                ("explored_slots", C.c_uint32), ("heap_cap", C.c_uint32)]


DPOR_RESULT_DTYPE = np.dtype([("interleavings", "<u4"), ("violations", "<u4"), ("deliveries", "<u8"), ("races", "<u8"),
                              ("n_nodes", "<u4"), ("n_explored", "<u4"), ("heap_left", "<u4"), ("exhausted", "<u4"),
                              ("budget_exhausted", "<u4"), ("status", "<u4")])
DPOR_VIOL_DTYPE = np.dtype([("schedule_hash", "<u8"), ("interleaving", "<u4"), ("length", "<u2"), ("code", "<u2")])


def dpor_search(model, ext, max_messages, max_interleavings, looking_for=0, stop_if_found=0, depth_bound=-1,
                model_flags=0, node_cap=1 << 16, explored_slots=1 << 20, heap_cap=1 << 18, cap_viol=4096):
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    cfg = Config(0, model, model_flags, 0, 0)
    P = DporParams(max_messages, depth_bound, max_interleavings, looking_for, stop_if_found, node_cap,
                   explored_slots, heap_cap)
    res = np.zeros(1, dtype=DPOR_RESULT_DTYPE)
    viol = np.zeros(cap_viol, dtype=DPOR_VIOL_DTYPE)
    hashes = np.zeros(max_interleavings + 1, dtype=np.uint64)
    rc = lib().oracle_dpor_search(C.byref(cfg), C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)), C.byref(P),
                                  C.c_void_p(res.ctypes.data), C.c_void_p(viol.ctypes.data), C.c_uint32(cap_viol),
                                  C.c_void_p(hashes.ctypes.data), C.c_uint32(len(hashes)))
    r = res[0]
    return rc, r, viol[:min(int(r["violations"]), cap_viol)].copy(), hashes[:int(r["interleavings"])].copy()


# ------------------------------------------------ recorded STS replay / internal minimization
def replay_trace(model, events, ext, mask, looking_for=0, flags=0, model_flags=0, skip_event=0xFFFFFFFF, cap=65536):
    ri = make_replay_input(model, events, ext)
    cfg = Config(0, model, model_flags, 0, 0, 0)
    mask = np.ascontiguousarray(mask, dtype=np.uint64)
    out = np.zeros(1, dtype=REPLAY_DTYPE)
    rec = np.zeros(cap, dtype=EVENT_DTYPE)
    n = C.c_uint32()
    lib().oracle_sts_replay_trace(C.byref(cfg), C.byref(ri), C.c_void_p(mask.ctypes.data), C.c_uint32(looking_for),
                                  C.c_uint32(flags), C.c_uint32(skip_event), C.c_void_p(out.ctypes.data),
                                  C.c_void_p(rec.ctypes.data), C.c_uint32(cap), C.byref(n))
    return out[0], rec[:n.value].copy()


def internal_minimize(model, verified, mcs_ext, looking_for, flags=0, model_flags=0, cap=65536):
    verified = np.ascontiguousarray(verified, dtype=EVENT_DTYPE)
    mcs_ext = np.ascontiguousarray(mcs_ext, dtype=EXT_DTYPE)
    cfg = Config(0, model, model_flags, 0, 0, 0)
    out = np.zeros(cap, dtype=EVENT_DTYPE)
    sizes = np.zeros(cap, dtype=np.uint32)
    n_out, total, n_sizes, unig = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
    rc = lib().oracle_internal_minimize(C.byref(cfg), C.c_void_p(verified.ctypes.data), C.c_uint32(len(verified)),
                                        C.c_void_p(mcs_ext.ctypes.data), C.c_uint32(len(mcs_ext)), C.c_uint32(looking_for),
                                        C.c_uint32(flags), C.c_void_p(out.ctypes.data), C.c_uint32(cap), C.byref(n_out),
                                        C.byref(total), C.c_void_p(sizes.ctypes.data), C.c_uint32(cap), C.byref(n_sizes),
                                        C.byref(unig))
    return rc, out[:n_out.value].copy(), total.value, sizes[:n_sizes.value].copy(), unig.value


PROVENANCE_DTYPE = np.dtype([("status", "<u4"), ("violation", "<u4"), ("affected_mask", "<u4"), ("n_trace", "<u4"),
                             ("n_kept", "<u4"), ("reserved", "<u4", (3,))])


def provenance(events, dep_parent, affected_mask, mask_words):
    """ProvenanceTracker.pruneConcurrentEvents, literal restatement (oracle/provenance.c)."""
    ev = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
    par = np.ascontiguousarray(dep_parent, dtype=np.uint16)
    keep = np.zeros(mask_words, dtype=np.uint64)
    out = np.zeros(1, dtype=PROVENANCE_DTYPE)
    lib().oracle_provenance(C.c_void_p(ev.ctypes.data), C.c_uint32(len(ev)), C.c_void_p(par.ctypes.data),
                            C.c_uint32(len(par)), C.c_uint32(affected_mask), C.c_void_p(keep.ctypes.data),
                            C.c_uint32(mask_words), C.c_void_p(out.ctypes.data))
    return keep, out[0]


def fuzz_provenance(model, ext, seed, max_messages, interval, mask_words, model_flags=0, looking_for=0, strategy=0):
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    cfg = Config(0, model, model_flags, 0, 0, strategy)
    p = FuzzParams(seed, 1, max_messages, interval, looking_for, 0)
    keep = np.zeros(mask_words, dtype=np.uint64)
    out = np.zeros(1, dtype=PROVENANCE_DTYPE)
    lib().oracle_fuzz_provenance(C.byref(cfg), C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)), C.byref(p),
                                 C.c_int64(seed), C.c_void_p(keep.ctypes.data), C.c_uint32(mask_words),
                                 C.c_void_p(out.ctypes.data))
    return keep, out[0]


# ------------------------------------------------ resumable, edit-distance bounded DPOR / IncrementalDDMin
class DporOpts(C.Structure):
    _fields_ = [("init_nodes", C.c_void_p), ("n_init_nodes", C.c_uint32), ("init_trace", C.c_void_p),
                ("n_init_trace", C.c_uint32), ("arvind", C.c_uint32), ("prioritize_pending", C.c_uint32)]


def dpor_seed(events, dep_parent):
    """(init_nodes, init_trace) of a recorded execution: the DepTracker graph as {src|dst<<8|type<<16, p0, p1, parent}
    per Unique (timer markers become deadLetters, the sender both trackers use) and DepTracker.initialTrace."""
    ev = np.asarray(events, dtype=EVENT_DTYPE)
    n = len(dep_parent)
    nodes = np.zeros((n, 4), dtype=np.uint32)
    for e in ev[ev["kind"] == 1]:                      # MsgSend: the Unique was allocated here
        src = 255 if e["src"] == 254 else int(e["src"])
        nodes[e["node"]] = (src | (int(e["dst"]) << 8) | (int(e["type"]) << 16), e["p0"], e["p1"], dep_parent[e["node"]])
    trace = np.concatenate([[0], ev["node"][ev["kind"] == 2]]).astype(np.uint32)
    return nodes, trace


class DporInstance:
    """One live DPORwHeuristics (oracle_dpor_open/test/close)."""

    def __init__(self, model, ext, max_messages, max_interleavings, seed=None, arvind=0, prioritize_pending=0,
                 looking_for=0, stop_if_found=1, model_flags=0, node_cap=1 << 12, explored_slots=1 << 16,
                 heap_cap=1 << 17):
        ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
        cfg = Config(0, model, model_flags, 0, 0)
        self.P = DporParams(max_messages, -1, max_interleavings, looking_for, stop_if_found, node_cap, explored_slots,
                            heap_cap)
        self.max_interleavings = max_interleavings
        opts = DporOpts(None, 0, None, 0, arvind, prioritize_pending)
        if seed is not None:
            self._nodes = np.ascontiguousarray(seed[0], dtype=np.uint32)
            self._trace = np.ascontiguousarray(seed[1], dtype=np.uint32)
            opts = DporOpts(self._nodes.ctypes.data, len(self._nodes), self._trace.ctypes.data, len(self._trace),
                            arvind, prioritize_pending)
        lib().oracle_dpor_open.restype = C.c_void_p
        self.h = lib().oracle_dpor_open(C.byref(cfg), C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)),
                                        C.byref(self.P), C.byref(opts))
        if not self.h:
            raise RuntimeError("oracle_dpor_open failed")

    def test(self, max_distance=-1):
        res = np.zeros(1, dtype=DPOR_RESULT_DTYPE)
        hashes = np.zeros(self.max_interleavings + 1, dtype=np.uint64)
        lib().oracle_dpor_test(C.c_void_p(self.h), C.c_int32(max_distance), C.c_void_p(res.ctypes.data), None,
                               C.c_uint32(0), C.c_void_p(hashes.ctypes.data), C.c_uint32(len(hashes)))
        return res[0], hashes[:int(res[0]["interleavings"])].copy()

    def close(self):
        if self.h:
            lib().oracle_dpor_close(C.c_void_p(self.h))
            self.h = None


def incremental_ddmin(model, ext, max_messages, max_interleavings, seed, max_max_distance=8, stop_at_size=6,
                      looking_for=0, model_flags=0, node_cap=1 << 12, explored_slots=1 << 16, heap_cap=1 << 17,
                      cap_instances=4096):
    """RunnerUtils.editDistanceDporDDMin's minimisation (RunnerUtils.scala:822-842)."""
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    cfg = Config(0, model, model_flags, 0, 0)
    P = DporParams(max_messages, -1, max_interleavings, looking_for, 1, node_cap, explored_slots, heap_cap)
    nodes = np.ascontiguousarray(seed[0], dtype=np.uint32)
    trace = np.ascontiguousarray(seed[1], dtype=np.uint32)
    opts = DporOpts(nodes.ctypes.data, len(nodes), trace.ctypes.data, len(trace), 1, 1)
    mw = mask_words(len(ext))
    mcs = np.zeros(mw, dtype=np.uint64)
    total, rounds, ninst = C.c_uint32(), C.c_uint32(), C.c_uint32()
    il = C.c_uint64()
    sizes = np.zeros(64, dtype=np.uint32)
    rc = lib().oracle_incremental_ddmin(C.byref(cfg), C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)), C.byref(P),
                                        C.byref(opts), C.c_int32(max_max_distance), C.c_uint32(stop_at_size),
                                        C.c_uint32(cap_instances), C.c_void_p(mcs.ctypes.data), C.c_uint32(mw),
                                        C.byref(total), C.byref(rounds), C.byref(il), C.byref(ninst),
                                        C.c_void_p(sizes.ctypes.data), C.c_uint32(len(sizes)))
    return rc, mcs, {"total_replays": total.value, "rounds": rounds.value, "interleavings": il.value,
                     "instances": ninst.value, "mcs_sizes": sizes[:rounds.value].copy()}


# ------------------------------------------------ frontier ("wide") DPOR
class FrontierParams(C.Structure):
    _fields_ = [("max_messages", C.c_int32), ("looking_for", C.c_uint32), ("stop_if_found", C.c_uint32),
                ("width", C.c_uint32), ("max_interleavings", C.c_uint64), ("explored_slots", C.c_uint64),
                ("pool_cap", C.c_uint64), ("trace_cap", C.c_uint32), ("rounds_per_exchange", C.c_uint32),
                ("steal_max", C.c_uint32), ("flags", C.c_uint32)]


FRONTIER_RESULT_DTYPE = np.dtype([
    ("interleavings", "<u8"), ("violations", "<u8"), ("deliveries", "<u8"), ("races", "<u8"),
    ("keys_enqueued", "<u8"), ("keys_dropped", "<u8"), ("explored_pairs", "<u8"), ("pool_left", "<u8"),
    ("records_sent", "<u8"), ("records_received", "<u8"), ("bytes_sent", "<u8"),
    ("rounds", "<u4"), ("exchanges", "<u4"), ("exhausted", "<u4"), ("budget_exhausted", "<u4"),
    ("status", "<u4"), ("trace_slots", "<u4"),
    ("exec_ms", "<f8"), ("scan_ms", "<f8"), ("select_ms", "<f8"), ("exchange_ms", "<f8")])
assert FRONTIER_RESULT_DTYPE.itemsize == 144 and C.sizeof(FrontierParams) == 56


def frontier_params(max_messages, max_interleavings, width, looking_for=0, stop_if_found=0, explored_slots=1 << 22,
                    pool_cap=1 << 22, trace_cap=None, rounds_per_exchange=1, steal_max=4096, flags=0):
    if trace_cap is None:
        trace_cap = int(max_interleavings) + 8 * steal_max + 16
    return FrontierParams(max_messages, looking_for, stop_if_found, width, max_interleavings, explored_slots,
                          pool_cap, trace_cap, rounds_per_exchange, steal_max, flags)


def dpor_frontier(model, ext, F, n_ranks=1, model_flags=0, blocked_mask=0, ignore_timers=0, cap_viol=4096):
    """oracle_dpor_frontier: per-rank results, violations and schedule hashes (each in slot order)."""
    ext = np.ascontiguousarray(ext, dtype=EXT_DTYPE)
    cfg = Config(0, model, model_flags, blocked_mask, ignore_timers, 0)
    res = np.zeros(n_ranks, dtype=FRONTIER_RESULT_DTYPE)
    viol = np.zeros((n_ranks, cap_viol), dtype=DPOR_VIOL_DTYPE)
    cap_h = int(F.max_interleavings) + 1
    hashes = np.zeros((n_ranks, cap_h), dtype=np.uint64)
    rc = lib().oracle_dpor_frontier(C.byref(cfg), C.c_void_p(ext.ctypes.data), C.c_uint32(len(ext)), C.byref(F),
                                    C.c_uint32(n_ranks), C.c_void_p(res.ctypes.data), C.c_void_p(viol.ctypes.data),
                                    C.c_uint32(cap_viol), C.c_void_p(hashes.ctypes.data), C.c_uint64(cap_h))
    vs = [viol[r, :min(int(res[r]["violations"]), cap_viol)].copy() for r in range(n_ranks)]
    hs = [hashes[r, :int(res[r]["interleavings"])].copy() for r in range(n_ranks)]
    return rc, res, vs, hs
