"""Host-side mirror of the reference's scheduler plugin surface for the hot path.

Same names, argument meaning and error behaviour as the Scala classes; the work
is done by the CUDA engine behind the C ABI (include/demi_b200.h).  There is no
CPU path here: constructing an engine without a CUDA device raises.

  SchedulerConfig   <- SchedulerConfig.scala:9-37
  RandomScheduler   <- schedulers/RandomScheduler.scala:41 (explore :234, test :597,
                       setMaxMessages :55, setInvariant :521)
"""
import ctypes as C

import numpy as np

from . import _native as N
from .events import pack_externals


class DemiError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "demi_b200 error %d: %s" % (code, msg))
        self.code = code


class SchedulerConfig(object):
    """SchedulerConfig.scala:9-37, restricted to what has meaning without a JVM.
    `model`/`model_flags` stand in for the application under test; `invariant_check`
    is the violation code looked for by the model's built-in invariant (None = any)."""

    def __init__(self, model, model_flags=0, device=0, ignoreTimers=False, blocked_mask=0, strategy=0):
        self.model, self.model_flags, self.device = model, model_flags, device
        self.ignoreTimers, self.blocked_mask = ignoreTimers, blocked_mask
        self.strategy = strategy       # 0 = FullyRandom, 1 = SrcDstFIFO (RandomizationStrategy, RandomScheduler.scala:624-631)


class Engine(object):
    """Owns one demi_handle."""

    def __init__(self, schedulerConfig):
        self.cfg = schedulerConfig
        self._h = C.c_void_p()
        c = N.Config(schedulerConfig.device, schedulerConfig.model, schedulerConfig.model_flags,
                     schedulerConfig.blocked_mask, 1 if schedulerConfig.ignoreTimers else 0, schedulerConfig.strategy)
        rc = N.lib().demi_create(C.byref(c), C.byref(self._h))
        if rc != N.OK:
            raise DemiError(rc, N.lib().demi_last_error(None).decode())
        self._ext = None

    def close(self):
        if self._h:
            N.lib().demi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != N.OK:
            raise DemiError(rc, N.lib().demi_last_error(self._h).decode())

    def load_model(self, blob):
        """demi_load_model: the data-only model of the host's application (demi_b200.model_ir builds the blob)."""
        self._check(N.lib().demi_load_model(self._h, bytes(blob), len(blob)))

    def actor_index(self, name):
        return int(N.lib().demi_actor_index(self._h, name.encode()))

    def actor_name(self, index):
        v = N.lib().demi_actor_name(self._h, index)
        return v.decode() if v is not None else None

    def set_user_filter(self, rules):
        """FullyRandom(userDefinedFilter): rules = [(src_mask, dst_mask, type_mask, flags)], a match REJECTS the draw."""
        arr = np.array(list(rules), dtype=N.FILTER_RULE_DTYPE) if len(rules) else np.zeros(0, dtype=N.FILTER_RULE_DTYPE)
        self._check(N.lib().demi_set_user_filter(self._h, arr.ctypes.data if len(arr) else None, len(arr)))

    def set_externals(self, events):
        arr = events if isinstance(events, np.ndarray) else pack_externals(events)
        arr = np.ascontiguousarray(arr, dtype=N.EXT_DTYPE)
        self._ext = arr
        self._check(N.lib().demi_set_externals(self._h, arr.ctypes.data, len(arr)))

    def fuzz_batch(self, seed_base, n, max_messages, interval, looking_for=0, out=None, flags=0):
        p = N.FuzzParams(seed_base, n, max_messages, interval, looking_for or 0, flags)
        if out is None:
            out = np.empty(n, dtype=N.RESULT_DTYPE)
        elif out.dtype != N.RESULT_DTYPE or len(out) < n or not out.flags["C_CONTIGUOUS"]:
            raise ValueError("out must be a C-contiguous array of >= %d demi_fuzz_result records" % n)   # the C call writes n * 32 bytes
        self._check(N.lib().demi_fuzz_batch(self._h, C.byref(p), out.ctypes.data))
        return out

    def fuzz_batch_dev(self, seed_base, n, max_messages, interval, out_ptr, stream=0, looking_for=0, flags=0):
        p = N.FuzzParams(seed_base, n, max_messages, interval, looking_for or 0, flags)
        self._check(N.lib().demi_fuzz_batch_dev(self._h, C.byref(p), C.c_void_p(out_ptr), C.c_void_p(stream)))

    def fuzz_summary_dev(self, stream=0):
        nv, ss = C.c_uint64(), C.c_uint64()
        self._check(N.lib().demi_fuzz_summary_dev(self._h, None, 0, C.c_void_p(stream), C.byref(nv), C.byref(ss)))
        return nv.value, ss.value

    def fuzz_trace(self, seed, max_messages, interval, looking_for=0, cap_events=65536, cap_nodes=65536):
        p = N.FuzzParams(seed, 1, max_messages, interval, looking_for or 0, 0)
        ev = np.zeros(cap_events, dtype=N.EVENT_DTYPE)
        par = np.zeros(cap_nodes, dtype=np.uint16)
        ne, nn = C.c_uint32(), C.c_uint32()
        res = np.zeros(1, dtype=N.RESULT_DTYPE)
        self._check(N.lib().demi_fuzz_trace(self._h, C.byref(p), seed, ev.ctypes.data, cap_events, C.byref(ne),
                                            par.ctypes.data, cap_nodes, C.byref(nn), res.ctypes.data))
        return ev[:ne.value].copy(), par[:nn.value].copy(), res[0]

    # ---- provenance pruning (ProvenanceTracker, schedulers/Util.scala:267-376)
    def provenance(self, events, dep_parent, affected_mask, mask_words=None):
        """pruneConcurrentEvents on one recorded execution: (keep mask over initialTrace positions, out record)."""
        ev = np.ascontiguousarray(events, dtype=N.EVENT_DTYPE)
        par = np.ascontiguousarray(dep_parent, dtype=np.uint16)
        if mask_words is None:
            mask_words = max(1, (int((ev["kind"] == N.EV_MSG_EVENT).sum()) + 1 + 63) // 64)
        keep = np.zeros(mask_words, dtype=np.uint64)
        out = np.zeros(1, dtype=N.PROVENANCE_DTYPE)
        self._check(N.lib().demi_provenance(self._h, ev.ctypes.data, len(ev), par.ctypes.data, len(par),
                                            int(affected_mask), keep.ctypes.data, mask_words, out.ctypes.data))
        return keep, out[0]

    def fuzz_provenance(self, seed_base, prefix_index, max_messages, interval, looking_for=0, mask_words=None):
        """The post-fuzz pruning step on prefixes seed_base + prefix_index[i] (RunnerUtils.scala:138-163)."""
        idx = np.ascontiguousarray(prefix_index, dtype=np.uint32)
        if mask_words is None:
            mask_words = max(1, (max_messages + 2 + 63) // 64)
        p = N.FuzzParams(seed_base, len(idx), max_messages, interval, looking_for or 0, 0)
        keep = np.zeros((len(idx), mask_words), dtype=np.uint64)
        out = np.zeros(len(idx), dtype=N.PROVENANCE_DTYPE)
        res = np.zeros(len(idx), dtype=N.RESULT_DTYPE)
        self._check(N.lib().demi_fuzz_provenance(self._h, C.byref(p), idx.ctypes.data, len(idx), keep.ctypes.data,
                                                 mask_words, out.ctypes.data, res.ctypes.data))
        return keep, out, res

    # ---- STSSched replay / DDMin
    def set_trace(self, events, externals):
        ev = np.ascontiguousarray(events, dtype=N.EVENT_DTYPE)
        ext = externals if isinstance(externals, np.ndarray) else pack_externals(externals)
        ext = np.ascontiguousarray(ext, dtype=N.EXT_DTYPE)
        self._trace, self._trace_ext = ev, ext
        self._check(N.lib().demi_set_trace(self._h, ev.ctypes.data, len(ev), ext.ctypes.data, len(ext)))

    def mask_words(self):
        return max(1, (len(self._trace_ext) + 63) // 64)

    def replay_batch(self, masks, looking_for=0, flags=0, out=None):
        mw = self.mask_words()
        masks = np.ascontiguousarray(masks, dtype=np.uint64).reshape(-1, mw)
        if out is None:
            out = np.empty(len(masks), dtype=N.REPLAY_DTYPE)
        self._check(N.lib().demi_replay_batch(self._h, masks.ctypes.data, len(masks), mw, looking_for or 0, flags,
                                              out.ctypes.data))
        return out

    def replay_batch_dev(self, masks_ptr, n_masks, out_ptr, looking_for=0, flags=0, stream=0):
        self._check(N.lib().demi_replay_batch_dev(self._h, C.c_void_p(masks_ptr), n_masks, self.mask_words(),
                                                  looking_for or 0, flags, C.c_void_p(out_ptr), C.c_void_p(stream)))

    def replay_batch_ex(self, masks=None, skip_events=None, looking_for=0, flags=0):
        mw = self.mask_words()
        n = len(skip_events) if skip_events is not None else len(masks)
        m = None if masks is None else np.ascontiguousarray(masks, dtype=np.uint64).reshape(-1, mw)
        sk = None if skip_events is None else np.ascontiguousarray(skip_events, dtype=np.uint32)
        out = np.empty(n, dtype=N.REPLAY_DTYPE)
        self._check(N.lib().demi_replay_batch_ex(self._h, None if m is None else m.ctypes.data,
                                                 None if sk is None else sk.ctypes.data, n, mw, looking_for or 0, flags,
                                                 out.ctypes.data))
        return out

    def replay_trace(self, mask=None, skip_event=0xFFFFFFFF, looking_for=0, flags=0, cap_events=65536):
        """The EventTrace STSScheduler.test returns (recording mode)."""
        mw = self.mask_words()
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint64)
        ev = np.zeros(cap_events, dtype=N.EVENT_DTYPE)
        n = C.c_uint32()
        res = np.zeros(1, dtype=N.REPLAY_DTYPE)
        self._check(N.lib().demi_replay_trace(self._h, None if m is None else m.ctypes.data, mw, skip_event,
                                              looking_for or 0, flags, ev.ctypes.data, cap_events, C.byref(n),
                                              res.ctypes.data))
        return res[0], ev[:n.value].copy()

    def internal_minimize(self, looking_for, flags=0, cap_events=65536):
        ev = np.zeros(cap_events, dtype=N.EVENT_DTYPE)
        sizes = np.zeros(cap_events, dtype=np.uint32)
        out = N.IntMinOut()
        self._check(N.lib().demi_internal_minimize(self._h, looking_for or 0, flags, ev.ctypes.data, cap_events,
                                                   sizes.ctypes.data, cap_events, C.byref(out)))
        return ev[:out.n_events].copy(), sizes[:out.n_internal_sizes].copy(), out

    def conjoin_atoms(self, e1, e2):
        """UnmodifiedEventDag.conjoinAtoms: externals e1, e2 (indices into the trace's externals) form one atom."""
        self._check(N.lib().demi_conjoin_atoms(self._h, e1, e2))

    def ddmin(self, looking_for, flags=0, check_unmodified=True, cap_iterations=1 << 16):
        mw = self.mask_words()
        mcs = np.zeros(mw, dtype=np.uint64)
        iters = np.zeros(cap_iterations, dtype=np.uint32)
        out = N.DDMinOut()
        self._check(N.lib().demi_ddmin(self._h, looking_for or 0, flags, 1 if check_unmodified else 0,
                                       mcs.ctypes.data, mw, iters.ctypes.data, cap_iterations, C.byref(out)))
        return mcs, iters[:min(out.n_iterations, cap_iterations)].copy(), out

    def fuzz_subseq_batch(self, masks, max_executions, max_messages, interval, seed_base=0, looking_for=0):
        """RandomScheduler.test(program_of(mask_t)) for every row of `masks` (uint64 [n_tests, mask_words] over the
        program given to set_externals), K = max_executions executions each, in one batch.  Returns (first_hit,
        first_bad): per test the first execution that ends on a matching violation / a capacity status, K if none."""
        masks = np.ascontiguousarray(np.atleast_2d(masks), dtype=np.uint64)
        n = len(masks)
        hit, bad = np.empty(n, dtype=np.uint32), np.empty(n, dtype=np.uint32)
        p = N.FuzzParams(seed_base, max_executions, max_messages, interval, looking_for or 0, 0)
        self._check(N.lib().demi_fuzz_subseq_batch(self._h, C.byref(p), masks.ctypes.data if n else None, n,
                                                   masks.shape[1], hit.ctypes.data, bad.ctypes.data))
        return hit, bad

    def random_ddmin(self, max_executions, max_messages, interval, seed_base=0, looking_for=0, conjoin_pairs=(),
                     check_unmodified=False, cap_iterations=1 << 16):
        """RunnerUtils.randomDDMin's DDMin over the program given to set_externals (demi_random_ddmin).  Returns
        (mcs mask, iteration sizes, iteration keys, demi_ddmin_out, verify seed or None)."""
        n_ext = len(self._ext) if self._ext is not None else 0
        mw = max(1, (n_ext + 63) // 64)
        mcs = np.zeros(mw, dtype=np.uint64)
        sizes = np.zeros(cap_iterations, dtype=np.uint32)
        keys = np.zeros(cap_iterations, dtype=np.uint32)
        pairs = np.ascontiguousarray(np.array(list(conjoin_pairs), dtype=np.uint32).reshape(-1, 2))
        p = N.FuzzParams(seed_base, max_executions, max_messages, interval, looking_for or 0, 0)
        out, vs = N.DDMinOut(), C.c_int64()
        self._check(N.lib().demi_random_ddmin(self._h, C.byref(p), pairs.ctypes.data if len(pairs) else None, len(pairs),
                                              1 if check_unmodified else 0, mcs.ctypes.data, mw, sizes.ctypes.data,
                                              keys.ctypes.data, cap_iterations, C.byref(out), C.byref(vs)))
        k = min(out.n_iterations, cap_iterations)
        return mcs, sizes[:k].copy(), keys[:k].copy(), out, (vs.value if vs.value >= 0 else None)

    # ---- state-hash dedup + compaction (K5 / K4)
    def dedup_compact(self, results, mode=0):
        results = np.ascontiguousarray(results, dtype=N.RESULT_DTYPE)
        out = np.empty(len(results), dtype=N.RESULT_DTYPE)
        idx = np.empty(len(results), dtype=np.uint32)
        cnt = C.c_uint64()
        self._check(N.lib().demi_dedup_compact(self._h, results.ctypes.data, len(results), mode, out.ctypes.data,
                                               idx.ctypes.data, C.byref(cnt)))
        return out[:cnt.value].copy(), idx[:cnt.value].copy()

    def dedup_compact_dev(self, results_ptr, n, mode, out_ptr, out_index_ptr, out_count_ptr, stream=0):
        self._check(N.lib().demi_dedup_compact_dev(self._h, C.c_void_p(results_ptr), n, mode, C.c_void_p(out_ptr),
                                                   C.c_void_p(out_index_ptr), C.c_void_p(out_count_ptr),
                                                   C.c_void_p(stream)))

    # ---- DPOR
    def dpor_batch(self, programs, max_messages, max_interleavings, looking_for=0, stop_if_found=False, depth_bound=-1,
                   node_cap=4096, explored_slots=1 << 16, heap_cap=1 << 15, cap_viol=64, want_hashes=False):
        """`programs`: list of external-event programs (Start/Send only), one independent search each."""
        packed = [p if isinstance(p, np.ndarray) else pack_externals(p) for p in programs]
        offs = np.zeros(len(packed) + 1, dtype=np.uint32)
        offs[1:] = np.cumsum([len(p) for p in packed])
        ext = np.ascontiguousarray(np.concatenate(packed), dtype=N.EXT_DTYPE)
        P = N.DporParams(max_messages, depth_bound, max_interleavings, looking_for or 0, 1 if stop_if_found else 0,
                         node_cap, explored_slots, heap_cap)
        res = np.zeros(len(packed), dtype=N.DPOR_RESULT_DTYPE)
        viol = np.zeros((len(packed), cap_viol), dtype=N.DPOR_VIOL_DTYPE)
        cap_h = max_interleavings + 1 if want_hashes else 0
        hashes = np.zeros((len(packed), max(cap_h, 1)), dtype=np.uint64)
        self._check(N.lib().demi_dpor_batch(self._h, ext.ctypes.data, offs.ctypes.data, len(packed), C.byref(P),
                                            res.ctypes.data, viol.ctypes.data, cap_viol,
                                            hashes.ctypes.data if want_hashes else None, cap_h))
        return res, viol, hashes

    @staticmethod
    def _seed(seed):
        """(events, dep_parent) of a recorded execution -> demi_dpor_seed (keeps the arrays alive)."""
        ev = np.ascontiguousarray(seed[0], dtype=N.EVENT_DTYPE)
        par = np.ascontiguousarray(seed[1], dtype=np.uint16)
        return N.DporSeed(ev.ctypes.data, len(ev), par.ctypes.data, len(par)), (ev, par)

    def dpor_batch_ex(self, programs, max_messages, max_interleavings, seed=None, flags=0, caps=None, looking_for=0,
                      stop_if_found=True, node_cap=4096, explored_slots=1 << 16, heap_cap=1 << 15, want_hashes=False):
        """DPOR instances in RunnerUtils.editDistanceDporDDMin's configuration.  `seed` = (events, dep_parent) of the
        recorded execution; `caps[i]` = the setMaxDistance values instance i is tested with, in order (None: one
        uncapped test)."""
        packed = [p if isinstance(p, np.ndarray) else pack_externals(p) for p in programs]
        offs = np.zeros(len(packed) + 1, dtype=np.uint32)
        offs[1:] = np.cumsum([len(p) for p in packed])
        ext = np.ascontiguousarray(np.concatenate(packed), dtype=N.EXT_DTYPE)
        P = N.DporParams(max_messages, -1, max_interleavings, looking_for or 0, 1 if stop_if_found else 0,
                         node_cap, explored_slots, heap_cap)
        ex = N.DporEx(flags, None, None, None)
        keep = []
        if seed is not None:
            sd, alive = self._seed(seed)
            keep += [sd, alive]
            ex.seed = C.pointer(sd)
        if caps is not None:
            coff = np.zeros(len(packed) + 1, dtype=np.uint32)
            coff[1:] = np.cumsum([len(c) for c in caps])
            cflat = np.ascontiguousarray(np.concatenate([np.asarray(c, dtype=np.int32) for c in caps]), dtype=np.int32)
            keep += [coff, cflat]
            ex.caps, ex.cap_offsets = cflat.ctypes.data, coff.ctypes.data
        res = np.zeros(len(packed), dtype=N.DPOR_RESULT_DTYPE)
        cap_h = max_interleavings + 1 if want_hashes else 0
        hashes = np.zeros((len(packed), max(cap_h, 1)), dtype=np.uint64)
        self._check(N.lib().demi_dpor_batch_ex(self._h, ext.ctypes.data, offs.ctypes.data, len(packed), C.byref(P),
                                               C.byref(ex), res.ctypes.data, None, 0,
                                               hashes.ctypes.data if want_hashes else None, cap_h))
        return res, hashes

    def incremental_ddmin(self, externals, max_messages, max_interleavings, seed, looking_for=0, max_max_distance=8,
                          stop_at_size=6, flags=N.DF_ARVIND_ORDERING | N.DF_PRIORITIZE_PENDING, node_cap=4096,
                          explored_slots=1 << 16, heap_cap=1 << 15):
        ext = externals if isinstance(externals, np.ndarray) else pack_externals(externals)
        ext = np.ascontiguousarray(ext, dtype=N.EXT_DTYPE)
        P = N.DporParams(max_messages, -1, max_interleavings, looking_for or 0, 1, node_cap, explored_slots, heap_cap)
        sd, alive = self._seed(seed)
        mw = max(1, (len(ext) + 63) // 64)
        mcs = np.zeros(mw, dtype=np.uint64)
        out = N.IncDDMinOut()
        self._check(N.lib().demi_incremental_ddmin(self._h, ext.ctypes.data, len(ext), C.byref(P), flags, C.byref(sd),
                                                   max_max_distance, stop_at_size, mcs.ctypes.data, mw, C.byref(out)))
        del alive
        return mcs, out

    # ---- frontier ("wide") DPOR: one DPORwHeuristics.test explored as a frontier of backtrack points
    @staticmethod
    def frontier_params(max_messages, max_interleavings, width, looking_for=0, stop_if_found=False,
                        explored_slots=1 << 22, pool_cap=1 << 22, trace_cap=None, rounds_per_exchange=1, steal_max=4096,
                        flags=0):
        if trace_cap is None:
            trace_cap = int(max_interleavings) + 8 * steal_max + 16
        return N.FrontierParams(max_messages, looking_for or 0, 1 if stop_if_found else 0, width, max_interleavings,
                                explored_slots, pool_cap, trace_cap, rounds_per_exchange, steal_max, flags)

    def comm_init(self, unique_id, rank, world):
        """Join the library's NCCL communicator (demi_comm_init); unique_id = the 128 bytes rank 0 made."""
        buf = (C.c_uint8 * N.COMM_ID_BYTES).from_buffer_copy(bytes(unique_id))
        self._check(N.lib().demi_comm_init(self._h, buf, rank, world))

    @staticmethod
    def comm_unique_id():
        buf = (C.c_uint8 * N.COMM_ID_BYTES)()
        rc = N.lib().demi_comm_unique_id(buf)
        if rc != N.OK:
            raise DemiError(rc, (N.lib().demi_last_error(None) or b"").decode())
        return bytes(buf)

    def dpor_frontier(self, program, F, cap_viol=4096, want_hashes=True):
        """demi_dpor_frontier on this handle's device (collective when the handle has a communicator).
        Returns (result record, violations, schedule hashes of this rank's interleavings in execution order)."""
        ext = program if isinstance(program, np.ndarray) else pack_externals(program)
        ext = np.ascontiguousarray(ext, dtype=N.EXT_DTYPE)
        res = np.zeros(1, dtype=N.FRONTIER_RESULT_DTYPE)
        viol = np.zeros(cap_viol, dtype=N.DPOR_VIOL_DTYPE)
        cap_h = int(F.max_interleavings) + int(F.width) + 1 if want_hashes else 0
        hashes = np.zeros(max(cap_h, 1), dtype=np.uint64)
        rc = N.lib().demi_dpor_frontier(self._h, ext.ctypes.data, len(ext), C.byref(F), res.ctypes.data,
                                        viol.ctypes.data, cap_viol, hashes.ctypes.data if want_hashes else None, cap_h)
        self.last_frontier = res[0]
        self._check(rc)
        r = res[0]
        return r, viol[:min(int(r["violations"]), cap_viol)].copy(), hashes[:min(int(r["interleavings"]), cap_h)].copy()

    def stats(self):
        s = N.Perf()
        self._check(N.lib().demi_stats(self._h, C.byref(s)))
        return s


class RandomScheduler(object):
    """RandomScheduler(schedulerConfig, max_executions, invariant_check_interval,
    randomizationStrategy = FullyRandom(seed)) — RandomScheduler.scala:41-44.

    The reference explores executions one after another; here execution i of
    `max_executions` is prefix `seed + i` of one batched kernel launch, and
    explore() returns the first violating one in that order."""

    def __init__(self, schedulerConfig, max_executions=1, invariant_check_interval=0, seed=0, engine=None):
        self.schedulerConfig = schedulerConfig
        self.max_executions = max_executions
        self.invariant_check_interval = invariant_check_interval
        self.seed = seed
        self.maxMessages = -1            # Int.MaxValue (RandomScheduler.scala:54)
        self.test_invariant = True       # models carry their invariant; None => "Must invoke setInvariant"
        self.engine = engine or Engine(schedulerConfig)
        self.stats = None
        self.last_results = None

    def setMaxMessages(self, n):
        self.maxMessages = n

    def setInvariant(self, invariant):
        self.test_invariant = invariant

    def getName(self):
        return "RandomScheduler"

    def explore(self, trace, lookingFor=None):
        """Returns (EventTrace records, violation code) of the first violating
        execution, else None (RandomScheduler.scala:234-272).

        Deviation, on purpose: execution i runs FullyRandom(seed + i) — the loop of RunnerUtils.fuzz
        (RunnerUtils.scala:75-91: a fresh RandomScheduler + FullyRandom per execution, max_executions = 1), made
        reproducible.  The reference's own `for (i <- 1 to max_executions)` keeps ONE FullyRandom whose java.util.Random
        stream runs on across executions (reset_all_state, :575-595, does not re-seed it), so for max_executions > 1
        the i-th interleaving here is not the one a JVM run with the same seed would produce."""
        if self.test_invariant is None:
            raise ValueError("Must invoke setInvariant before test()")   # :244-246
        self.engine.set_externals(trace)
        res = self.engine.fuzz_batch(self.seed, self.max_executions, self.maxMessages,
                                     self.invariant_check_interval, lookingFor or 0)
        self.last_results = res
        if self.stats is not None:
            self.stats.increment_replays(self.max_executions)
        bad = np.nonzero(res["status"])[0]
        if len(bad):
            raise DemiError(N.ERR_CAPACITY, "prefix %d overflowed (status %d)" % (bad[0], res["status"][bad[0]]))
        hits = np.nonzero(res["violation"])[0]
        if not len(hits):
            return None
        i = int(hits[0])
        ev, _, r = self.engine.fuzz_trace(self.seed + i, self.maxMessages, self.invariant_check_interval,
                                          lookingFor or 0)
        return ev, int(r["violation"])

    def test(self, events, violation_fingerprint, stats=None):
        """TestOracle.test: Some(trace) iff the violation was reproduced (RandomScheduler.scala:597-612)."""
        self.stats = stats
        r = self.explore(events, violation_fingerprint)
        return None if r is None else r[0]


def mask_of(externals, subseq):
    """Seq[ExternalEvent] subsequence -> bitmask over the positions of `externals`."""
    pos = {e._id: i for i, e in enumerate(externals)}
    m = np.zeros(max(1, (len(externals) + 63) // 64), dtype=np.uint64)
    for e in subseq:
        i = pos[e._id]
        m[i // 64] |= np.uint64(1) << np.uint64(i % 64)
    return m


def events_of(externals, mask):
    return [e for i, e in enumerate(externals) if (int(mask[i // 64]) >> (i % 64)) & 1]


def program_of(externals, mask):
    """The program a RandomScheduler test of subsequence `mask` runs (include/demi_b200.h, demi_fuzz_subseq_batch):
    the selected externals in order, except that a selected WaitQuiescence right after another selected
    WaitQuiescence is left out.  `externals`: packed records (EXT_DTYPE) or a list of events; the result has the
    same form."""
    packed = isinstance(externals, np.ndarray)
    kinds = externals["kind"] if packed else pack_externals(list(externals))["kind"]
    keep, prev_wq = [], False
    for i in range(len(kinds)):
        if not (int(mask[i // 64]) >> (i % 64)) & 1:
            continue
        wq = int(kinds[i]) == N.EXT_WAIT_QUIESCENCE
        if wq and prev_wq:
            continue
        prev_wq = wq
        keep.append(i)
    if not keep:
        raise ValueError("program_of: the mask selects no external")
    return externals[np.array(keep, dtype=np.int64)] if packed else [externals[i] for i in keep]


from .minimization_stats import MinimizationStats  # noqa: E402  (minification/Minimizer.scala:30-237)


class STSScheduler(object):
    """STSScheduler(schedulerConfig, original_trace, allowPeek=false) — schedulers/STSScheduler.scala:84-86.
    test() is TestOracle.test (:199-310): Some(trace) iff the violation was reproduced.
    Peek (allowPeek=true) needs JVM actor-system checkpoints and is not offered."""

    def __init__(self, schedulerConfig, original_trace, original_externals, allowPeek=False,
                 filterKnownAbsents=False, engine=None):
        if allowPeek:
            raise NotImplementedError("STSSched with Peek is outside the accelerated path")
        self.schedulerConfig = schedulerConfig
        self.original_trace = original_trace
        self.original_externals = list(original_externals)
        self.flags = N.RF_FILTER_KNOWN_ABSENTS if filterKnownAbsents else 0
        self.engine = engine or Engine(schedulerConfig)
        self.engine.set_trace(original_trace, pack_externals(self.original_externals))
        self.test_invariant = True

    def getName(self):
        return "STSSchedNoPeek"

    def setInvariant(self, invariant):
        self.test_invariant = invariant

    def test(self, subseq, violation_fingerprint, stats=None):
        if self.test_invariant is None:
            raise ValueError("Must invoke setInvariant before test()")      # :208-210
        if stats is not None:
            stats.increment_replays()
        r = self.engine.replay_batch(mask_of(self.original_externals, subseq), violation_fingerprint, self.flags)[0]
        if r["status"]:
            raise DemiError(N.ERR_CAPACITY, "replay status %d" % r["status"])
        return r if r["violation"] else None

    def test_batch(self, subseqs, violation_fingerprint):
        masks = np.stack([mask_of(self.original_externals, s) for s in subseqs])
        return self.engine.replay_batch(masks, violation_fingerprint, self.flags)


class ReplayScheduler(STSScheduler):
    """Strict replay (schedulers/ReplayScheduler.scala:71-140): an expected delivery
    that is not pending raises ReplayException."""

    class ReplayException(RuntimeError):
        pass

    def replay(self, violation_fingerprint=0):
        full = [e for e in self.original_externals]
        r = self.engine.replay_batch(mask_of(self.original_externals, full), violation_fingerprint,
                                     self.flags | N.RF_STRICT)[0]
        if r["status"] == N.RS_DIVERGED:
            raise ReplayScheduler.ReplayException("Expected event not pending after %d deliveries" % r["delivered"])
        if r["status"]:
            raise DemiError(N.ERR_CAPACITY, "replay status %d" % r["status"])
        return r


class DDMin(object):
    """DDMin(oracle, checkUnmodifed) — minification/DeltaDebugging.scala:7-109, with an
    STSScheduler as the TestOracle (RunnerUtils.stsSchedDDMin, RunnerUtils.scala:642-707), or with a
    RandomScheduler (RunnerUtils.randomDDMin, RunnerUtils.scala:601-623).  With a RandomScheduler, minimize()
    takes the externals to minimize (the dag, WaitQuiescence included) and runs demi_random_ddmin on the
    scheduler's engine; the engine's program is left as it was."""

    def __init__(self, oracle, checkUnmodifed=False, stats=None):
        self.oracle = oracle
        self.checkUnmodifed = checkUnmodifed
        self._stats = stats or MinimizationStats()
        self.last = None
        self.verify_seed = None
        self._conjoined = []

    def _random(self):
        return isinstance(self.oracle, RandomScheduler)

    def conjoinAtoms(self, e1, e2):
        """UnmodifiedEventDag.conjoinAtoms (minification/Util.scala:167-178) on the dag DDMin minimizes."""
        if self._random():
            self._conjoined.append((e1, e2))       # resolved against the externals given to minimize()
            return
        ext = self.oracle.original_externals
        for e in (e1, e2):
            if e not in ext:
                raise ValueError("No such external event:%r" % (e,))
        self.oracle.engine.conjoin_atoms(ext.index(e1), ext.index(e2))

    def minimize(self, violation_fingerprint, externals=None):
        """STSScheduler: minimize(violation) returns the MCS as a list of ExternalEvents (WaitQuiescence dropped,
        RunnerUtils.scala:678-684).  RandomScheduler: minimize(violation, externals) returns the MCS of `externals`."""
        if self._random():
            return self._minimize_random(violation_fingerprint, externals)
        mcs, iters, out = self.oracle.engine.ddmin(violation_fingerprint, self.oracle.flags, self.checkUnmodifed)
        self._stats.record_series(iters)
        self._stats.total_replays = out.total_replays
        self.last = out
        return events_of(self.oracle.original_externals, mcs)

    def _minimize_random(self, violation_fingerprint, externals):
        if externals is None:
            raise ValueError("DDMin with a RandomScheduler: minimize(violation, externals)")
        if self.oracle.test_invariant is None:
            raise ValueError("Must invoke setInvariant before test()")
        ext = list(externals)
        ids = [e._id for e in ext]
        pairs = []
        for e1, e2 in self._conjoined:
            for e in (e1, e2):
                if e._id not in ids:
                    raise ValueError("No such external event:%r" % (e,))
            pairs.append((ids.index(e1._id), ids.index(e2._id)))
        eng = self.oracle.engine
        saved = eng._ext
        eng.set_externals(ext)
        try:
            mcs, sizes, keys, out, vseed = eng.random_ddmin(
                self.oracle.max_executions, self.oracle.maxMessages, self.oracle.invariant_check_interval,
                self.oracle.seed, violation_fingerprint, pairs, self.checkUnmodifed)
        finally:
            if saved is not None:
                eng.set_externals(saved)
        inner = self._stats.inner()
        for k, v in zip(keys, sizes):                 # MinimizationStats.iterationSize (Minimizer.scala:183-185)
            inner.iterationSize[int(k)] = int(v)
            inner.iteration_size_log.append(int(v))
        self._stats.total_replays = out.total_replays
        self.last, self.verify_seed = out, vseed
        self.mcs_mask = mcs
        return events_of(ext, mcs)

    def verify_mcs(self, mcs, violation_fingerprint):
        return self.oracle.test(mcs, violation_fingerprint)


def random_ddmin(experiment, schedulerConfig, max_executions=1, seed=0, stats=None, interval=0):
    """RunnerUtils.randomDDMin (RunnerUtils.scala:601-623) over `experiment` (experiment.load_experiment output):
    DDMin of its original externals with RandomScheduler(schedulerConfig, max_executions, interval, FullyRandom(seed + i)
    for execution i) as the TestOracle, setMaxMessages(len(trace)) (:608), checkUnmodifed = false (:610).
    Returns (mcs events, stats, EventTrace | None, violation).  The EventTrace is the recorded execution of the
    MCS's violating verification run (demi_fuzz_trace on program_of(mcs), recorded on an Engine of its own), or the
    experiment's trace when nothing was removed."""
    from .events import unpack_externals
    ext = unpack_externals(experiment["externals"])
    trace = experiment["events"]
    violation = int(experiment["meta"]["violation"])
    sched = RandomScheduler(schedulerConfig, max_executions, interval, seed)
    sched.setMaxMessages(len(trace))
    ddmin = DDMin(sched, checkUnmodifed=False, stats=stats)
    mcs = ddmin.minimize(violation, ext)
    if len(mcs) < len(ext):
        validated = None
        if ddmin.verify_seed is not None:
            rec = Engine(schedulerConfig)
            try:
                rec.set_externals(program_of(ext, ddmin.mcs_mask))
                validated = rec.fuzz_trace(ddmin.verify_seed, sched.maxMessages, interval, violation)[0]
            finally:
                rec.close()
        return mcs, ddmin._stats, validated, violation
    return mcs, ddmin._stats, trace, violation


class ProvenanceTracker:
    """ProvenanceTracker(trace, depGraph) (schedulers/Util.scala:267-376).  `trace` / `dep_parent` are the recorded
    EventTrace and DepTracker tree of one execution (Engine.fuzz_trace)."""

    def __init__(self, engine, trace, dep_parent):
        self.engine, self.trace, self.dep_parent = engine, np.asarray(trace, dtype=N.EVENT_DTYPE), dep_parent
        self.last = None

    def prune_concurrent_events(self, affected_nodes):
        """pruneConcurrentEvents(violation): indices into `trace` of the deliveries that stay.  The root event is
        dropped here, as EventTrace.intersection does afterwards (EventTrace.scala:127-131)."""
        delivery_index = np.nonzero(self.trace["kind"] == N.EV_MSG_EVENT)[0]
        keep, out = self.engine.provenance(self.trace, self.dep_parent, affected_nodes)
        self.last = out
        if out["status"] == N.PV_CYCLE:
            raise RuntimeError("happens-before relation is cyclic")            # Util.topologicalSort, Util.scala:506
        if out["status"]:
            raise RuntimeError("provenance: trace does not fit (status %d)" % out["status"])
        bits = np.unpackbits(keep.view(np.uint8), bitorder="little")[1:len(delivery_index) + 1].astype(bool)
        return delivery_index[bits]


class DPORwHeuristics(object):
    """DPORwHeuristics(schedulerConfig, backtrackHeuristic = DefaultBacktrackOrdering, depth_bound,
    stopIfViolationFound, trackHistory = true) — schedulers/DPORwHeuristics.scala:77-88.
    test() explores interleavings of the external events in the reference's order until a matching
    violation is found or the backtrack set / budget is exhausted."""

    def __init__(self, schedulerConfig, depth_bound=None, stopIfViolationFound=True, max_interleavings=1000,
                 engine=None):
        self.schedulerConfig = schedulerConfig
        self.depth_bound = -1 if depth_bound is None else depth_bound
        self.stopIfViolationFound = stopIfViolationFound
        self.max_interleavings = max_interleavings
        self.max_messages = None
        self.engine = engine or Engine(schedulerConfig)
        self.last = None

    def getName(self):
        return "DPORwHeuristics"

    def setMaxMessagesToSchedule(self, n):
        self.max_messages = n

    def setDepthBound(self, d):
        self.depth_bound = d

    def test(self, events, violation_fingerprint, stats=None):
        """Some(record of the first violating interleaving) or None (DPORwHeuristics.scala:1193-1242)."""
        if self.max_messages is None:
            raise ValueError("setMaxMessagesToSchedule is required (models with repeating timers never quiesce)")
        prog = [e for e in events if e.kind in (N.EXT_START, N.EXT_SEND)]   # convertToDPORTrace (:1279-1303)
        res, viol, _ = self.engine.dpor_batch([prog], self.max_messages, self.max_interleavings,
                                              violation_fingerprint, self.stopIfViolationFound, self.depth_bound)
        self.last = res[0]
        if stats is not None:
            stats.increment_replays(int(res[0]["interleavings"]))
        if res[0]["status"]:
            raise DemiError(N.ERR_CAPACITY, "DPOR search status %d" % res[0]["status"])
        return viol[0][0] if res[0]["violations"] else None


class DefaultBacktrackOrdering(object):
    """Deeper backtrack points first (schedulers/BacktrackOrdering.scala:58-69)."""
    pass


class ArvindDistanceOrdering(object):
    """Backtrack points ordered by their edit distance from the original trace
    (schedulers/BacktrackOrdering.scala:99-173); init() is given the recorded execution."""

    def __init__(self):
        self.original = None

    def init(self, events, dep_parent):
        self.original = (events, dep_parent)


class ResumableDPOR(object):
    """One DPORwHeuristics per external-event subsequence (minification/IncrementalDeltaDebugging.scala:90-122),
    configured as RunnerUtils.editDistanceDporDDMin does (RunnerUtils.scala:822-835): seeded with the recorded
    execution's dependency graph and trace, ArvindDistanceOrdering, prioritizePendingUponDivergence.

    An instance's state is a function of the distance caps it has been tested with, so the engine keeps that list
    per subsequence and replays it — test() is side-effect free on the device."""

    def __init__(self, schedulerConfig, events, dep_parent, max_messages=None, max_interleavings=1000, engine=None,
                 backtrackHeuristic=None, prioritizePendingUponDivergence=True):
        self.engine = engine or Engine(schedulerConfig)
        self.seed = (events, dep_parent)
        self.max_messages = max_messages if max_messages is not None else int((np.asarray(events)["kind"] == N.EV_MSG_EVENT).sum()) + 1
        self.max_interleavings = max_interleavings
        heuristic = backtrackHeuristic if backtrackHeuristic is not None else ArvindDistanceOrdering()
        self.flags = (N.DF_ARVIND_ORDERING if isinstance(heuristic, ArvindDistanceOrdering) else 0) | \
                     (N.DF_PRIORITIZE_PENDING if prioritizePendingUponDivergence else 0)
        self.currentMaxDistance = 0
        self.subseqToDPOR = {}            # ids of the subsequence's events -> caps tested so far

    def getName(self):
        return "DPOR"

    def setMaxDistance(self, dist):
        self.currentMaxDistance = dist

    def test(self, events, violation_fingerprint, stats=None):
        prog = [e for e in events if e.kind in (N.EXT_START, N.EXT_SEND)]
        key = tuple(e._id for e in prog)
        caps = self.subseqToDPOR.setdefault(key, [])
        caps.append(self.currentMaxDistance)
        res, _ = self.engine.dpor_batch_ex([prog], self.max_messages, self.max_interleavings, seed=self.seed,
                                           flags=self.flags, caps=[caps], looking_for=violation_fingerprint)
        if res[0]["status"]:
            raise DemiError(N.ERR_CAPACITY, "DPOR instance status %d" % res[0]["status"])
        if stats is not None:
            stats.increment_replays()
        return bool(res[0]["violations"])


class IncrementalDDMin(object):
    """IncrementalDDMin(oracle: ResumableDPOR, maxMaxDistance, stopAtSize) —
    minification/IncrementalDeltaDebugging.scala:20-88.  minimize() runs DDMin under distance caps 0, 2, 4, ...;
    the DPOR tests a round may need are evaluated speculatively in batches, the decisions are the sequential ones."""

    def __init__(self, oracle, maxMaxDistance=256, stopAtSize=1, stats=None):
        self.oracle, self.maxMaxDistance, self.stopAtSize = oracle, maxMaxDistance, stopAtSize
        self._stats = stats or MinimizationStats()
        self.last = None

    def minimize(self, events, violation_fingerprint):
        prog = [e for e in events if e.kind in (N.EXT_START, N.EXT_SEND)]
        o = self.oracle
        mcs, out = o.engine.incremental_ddmin(prog, o.max_messages, o.max_interleavings, o.seed,
                                              looking_for=violation_fingerprint, max_max_distance=self.maxMaxDistance,
                                              stop_at_size=self.stopAtSize, flags=o.flags)
        self.last = out
        self._stats.increment_replays(out.total_replays)
        return [e for i, e in enumerate(prog) if (int(mcs[i >> 6]) >> (i & 63)) & 1]

    def verify_mcs(self, mcs, violation_fingerprint):
        return self.oracle.test(mcs, violation_fingerprint)


class LeftToRightOneAtATime(object):
    """RemovalStrategy that ignores deliveries one at a time, left to right
    (minification/internal_minimization/OneAtATimeRemoval.scala:131-137)."""
    pass


class SrcDstFIFORemoval(object):
    """RemovalStrategy that keeps per-(src,dst) FIFO delivery and only tries the last message of each pair, timers in
    any order (minification/internal_minimization/OneAtATimeRemoval.scala:139-251)."""
    pass


class STSSchedMinimizer(object):
    """STSSchedMinimizer(mcs, verified_mcs, violation, removalStrategy, schedulerConfig, ...) —
    minification/internal_minimization/ScheduleCheckers.scala:19-107; minimize() returns
    (MinimizationStats, minimized EventTrace) like RunnerUtils.minimizeInternals (RunnerUtils.scala:980-1003)."""

    def __init__(self, mcs, verified_mcs, violation, removalStrategy, schedulerConfig, stats=None, engine=None):
        if not isinstance(removalStrategy, (LeftToRightOneAtATime, SrcDstFIFORemoval)):
            raise NotImplementedError("LeftToRightOneAtATime and SrcDstFIFORemoval are the accelerated strategies")
        self.flags = N.IM_SRC_DST_FIFO if isinstance(removalStrategy, SrcDstFIFORemoval) else 0
        self.mcs, self.verified_mcs, self.violation = list(mcs), verified_mcs, violation
        self.engine = engine or Engine(schedulerConfig)
        self._stats = stats or MinimizationStats()
        self.last = None

    def minimize(self):
        self.engine.set_trace(self.verified_mcs, pack_externals(self.mcs))
        trace, sizes, out = self.engine.internal_minimize(self.violation, flags=self.flags)
        self._stats.record_series(sizes, internal=True)
        self._stats.total_replays += out.total_replays
        self.last = out
        return self._stats, trace
