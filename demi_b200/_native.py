"""ctypes binding of the C ABI declared in include/demi_b200.h.

This is the only way Python reaches the engine; the library must exist
(`python -m demi_b200.build`) — there is no Python or CPU fallback.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdemi_b200.so")

# ---- status codes (include/demi_b200.h)
OK, ERR_INVALID, ERR_STATE, ERR_NO_DEVICE, ERR_CUDA, ERR_CAPACITY, ERR_REPLAY = 0, -1, -2, -3, -4, -5, -6
DEADLETTERS, TIMER_SND = 0xFF, 0xFE
MODEL_PINGPONG3, MODEL_RAFT5, MODEL_BCAST32 = 1, 2, 3
EXT_START, EXT_KILL, EXT_SEND, EXT_WAIT_QUIESCENCE, EXT_PARTITION, EXT_UNPARTITION, EXT_HARD_KILL = 1, 2, 3, 4, 5, 6, 7
EV_MSG_SEND, EV_MSG_EVENT, EV_SPAWN, EV_KILL, EV_PARTITION, EV_UNPARTITION, EV_BEGIN_WAIT_QUIESCENCE, EV_QUIESCENCE = range(1, 9)


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("model", C.c_int32), ("model_flags", C.c_uint32),
                ("blocked_mask", C.c_uint32), ("ignore_timers", C.c_int32), ("strategy", C.c_int32), ("reserved", C.c_int32 * 2)]


class FuzzParams(C.Structure):
    _fields_ = [("seed_base", C.c_int64), ("n_prefixes", C.c_uint64), ("max_messages", C.c_int32),
                ("invariant_check_interval", C.c_int32), ("looking_for", C.c_uint32), ("flags", C.c_uint32)]


class Perf(C.Structure):
    _fields_ = [("prefixes", C.c_uint64), ("deliveries", C.c_uint64), ("violations", C.c_uint64),
                ("kernel_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("kernel_launches", C.c_uint32), ("deferred", C.c_uint32)]


EXT_DTYPE = np.dtype([("kind", "u1"), ("a", "u1"), ("b", "u1"), ("type", "u1"),
                      ("p0", "<u4"), ("p1", "<u4"), ("id", "<u4")])
EVENT_DTYPE = np.dtype([("kind", "u1"), ("src", "u1"), ("dst", "u1"), ("type", "u1"),
                        ("p0", "<u4"), ("p1", "<u4"), ("uniq", "<u2"), ("node", "<u2")])
RESULT_DTYPE = np.dtype([("violation", "<u4"), ("steps", "<u4"), ("state_hash", "<u8"), ("trace_hash", "<u8"),
                         ("n_nodes", "<u2"), ("n_events", "<u2"), ("max_pending", "<u2"), ("status", "<u2")])
REPLAY_DTYPE = np.dtype([("violation", "<u2"), ("status", "<u2"), ("delivered", "<u2"), ("ignored", "<u2"),
                         ("state_hash", "<u8")])
RF_FILTER_KNOWN_ABSENTS, RF_STRICT = 1, 2
RS_DIVERGED, RS_UNSUPPORTED = 16, 17


class DDMinOut(C.Structure):
    _fields_ = [("mcs_size", C.c_uint32), ("total_replays", C.c_uint32), ("n_iterations", C.c_uint32),
                ("replays_executed", C.c_uint32), ("batches", C.c_uint32), ("verified", C.c_uint32),
                ("reserved", C.c_uint32 * 2)]


class IntMinOut(C.Structure):
    _fields_ = [("n_events", C.c_uint32), ("deliveries_before", C.c_uint32), ("deliveries_after", C.c_uint32),
                ("total_replays", C.c_uint32), ("n_internal_sizes", C.c_uint32), ("unignorable", C.c_uint32),
                ("replays_executed", C.c_uint32), ("batches", C.c_uint32)]


class DporParams(C.Structure):
    _fields_ = [("max_messages", C.c_int32), ("depth_bound", C.c_int32), ("max_interleavings", C.c_uint32),
                ("looking_for", C.c_uint32), ("stop_if_found", C.c_uint32), ("node_cap", C.c_uint32),
                ("explored_slots", C.c_uint32), ("heap_cap", C.c_uint32)]


class DporSeed(C.Structure):
    _fields_ = [("events", C.c_void_p), ("n_events", C.c_uint32), ("dep_parent", C.c_void_p), ("n_nodes", C.c_uint32)]


class DporEx(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("seed", C.POINTER(DporSeed)), ("caps", C.c_void_p), ("cap_offsets", C.c_void_p)]


class IncDDMinOut(C.Structure):
    _fields_ = [("mcs_size", C.c_uint32), ("total_replays", C.c_uint32), ("rounds", C.c_uint32), ("instances", C.c_uint32),
                ("tests_executed", C.c_uint32), ("batches", C.c_uint32), ("interleavings_executed", C.c_uint64)]


DF_ARVIND_ORDERING, DF_PRIORITIZE_PENDING = 1, 2
IM_SRC_DST_FIFO = 0x100

DPOR_RESULT_DTYPE = np.dtype([("interleavings", "<u4"), ("violations", "<u4"), ("deliveries", "<u8"), ("races", "<u8"),
                              ("n_nodes", "<u4"), ("n_explored", "<u4"), ("heap_left", "<u4"), ("exhausted", "<u4"),
                              ("budget_exhausted", "<u4"), ("status", "<u4")])
DPOR_VIOL_DTYPE = np.dtype([("schedule_hash", "<u8"), ("interleaving", "<u4"), ("length", "<u2"), ("code", "<u2")])
assert DPOR_RESULT_DTYPE.itemsize == 48 and DPOR_VIOL_DTYPE.itemsize == 16 and C.sizeof(DporParams) == 32
assert REPLAY_DTYPE.itemsize == 16
assert EXT_DTYPE.itemsize == 16 and EVENT_DTYPE.itemsize == 16 and RESULT_DTYPE.itemsize == 32

# every symbol include/demi_b200.h declares
PROVENANCE_DTYPE = np.dtype([("status", "<u4"), ("violation", "<u4"), ("affected_mask", "<u4"), ("n_trace", "<u4"),
                             ("n_kept", "<u4"), ("reserved", "<u4", (3,))])
PV_OK, PV_CYCLE, PV_OVERFLOW, PV_PREFIX_FAILED = 0, 1, 2, 3

EXPORTS = [
    "demi_version", "demi_last_error", "demi_device_count", "demi_create", "demi_destroy",
    "demi_set_externals", "demi_fuzz_batch", "demi_fuzz_batch_dev", "demi_fuzz_summary_dev",
    "demi_fuzz_trace", "demi_stats",
    "demi_set_trace", "demi_replay_batch", "demi_replay_batch_dev", "demi_ddmin", "demi_dpor_batch",
    "demi_dedup_compact_dev", "demi_dedup_compact",
    "demi_replay_batch_ex", "demi_replay_trace", "demi_internal_minimize",
    "demi_provenance", "demi_fuzz_provenance", "demi_dpor_batch_ex", "demi_incremental_ddmin",
    "demi_dpor_frontier", "demi_dpor_frontier_multi", "demi_comm_unique_id", "demi_comm_init", "demi_comm_rank",
    "demi_create_multi", "demi_conjoin_atoms", "demi_fuzzer_generate", "demi_experiment_save", "demi_experiment_load",
    "demi_load_model", "demi_actor_index", "demi_actor_name", "demi_set_user_filter",
    "demi_fuzz_subseq_batch", "demi_random_ddmin",
]
FILTER_RULE_DTYPE = np.dtype([("src_mask", "<u4"), ("dst_mask", "<u4"), ("type_mask", "<u4"), ("flags", "<u4")])
FRULE_DEADLETTERS = 1
MODEL_IR = 100


class FuzzerConfig(C.Structure):
    _fields_ = [("kill", C.c_double), ("send", C.c_double), ("wait_quiescence", C.c_double), ("partition", C.c_double),
                ("unpartition", C.c_double), ("num_events", C.c_uint32), ("send_type", C.c_uint32)]


class Experiment(C.Structure):
    _fields_ = [("model", C.c_int32), ("model_flags", C.c_uint32), ("violation", C.c_uint32), ("reserved", C.c_uint32),
                ("externals", C.c_void_p), ("n_externals", C.c_uint32), ("cap_externals", C.c_uint32),
                ("events", C.c_void_p), ("n_events", C.c_uint32), ("cap_events", C.c_uint32),
                ("dep_parent", C.c_void_p), ("n_nodes", C.c_uint32), ("cap_nodes", C.c_uint32),
                ("mcs_mask", C.c_void_p), ("mask_words", C.c_uint32), ("cap_mask_words", C.c_uint32)]


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
FRONTIER_ENTRY_DTYPE = np.dtype([("id", "<u8"), ("src", "u1"), ("dst", "u1"), ("type", "u1"), ("pad", "u1"),
                                 ("parent_pos", "<u2"), ("pad2", "<u2")])
assert FRONTIER_RESULT_DTYPE.itemsize == 144 and C.sizeof(FrontierParams) == 56 and FRONTIER_ENTRY_DTYPE.itemsize == 16
COMM_ID_BYTES = 128
FR_NO_HISTORY = 1

_lib = None


def lib():
    """Load libdemi_b200.so (fails loudly if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "demi_b200: native library %s is missing; run `python -m demi_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.demi_version.restype = C.c_char_p
    L.demi_last_error.restype = C.c_char_p
    L.demi_last_error.argtypes = [vp]
    L.demi_device_count.restype = C.c_int32
    L.demi_create.restype = C.c_int32
    L.demi_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.demi_destroy.restype = None
    L.demi_destroy.argtypes = [vp]
    L.demi_set_externals.restype = C.c_int32
    L.demi_set_externals.argtypes = [vp, vp, C.c_uint32]
    L.demi_fuzz_batch.restype = C.c_int32
    L.demi_fuzz_batch.argtypes = [vp, C.POINTER(FuzzParams), vp]
    L.demi_fuzz_batch_dev.restype = C.c_int32
    L.demi_fuzz_batch_dev.argtypes = [vp, C.POINTER(FuzzParams), vp, vp]
    L.demi_fuzz_summary_dev.restype = C.c_int32
    L.demi_fuzz_summary_dev.argtypes = [vp, vp, C.c_uint64, vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.demi_fuzz_trace.restype = C.c_int32
    L.demi_fuzz_trace.argtypes = [vp, C.POINTER(FuzzParams), C.c_int64, vp, C.c_uint32, C.POINTER(C.c_uint32),
                                  vp, C.c_uint32, C.POINTER(C.c_uint32), vp]
    L.demi_set_trace.restype = C.c_int32
    L.demi_set_trace.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32]
    L.demi_replay_batch.restype = C.c_int32
    L.demi_replay_batch.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp]
    L.demi_replay_batch_dev.restype = C.c_int32
    L.demi_replay_batch_dev.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp]
    L.demi_ddmin.restype = C.c_int32
    L.demi_ddmin.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_int32, vp, C.c_uint32, vp, C.c_uint32,
                             C.POINTER(DDMinOut)]
    L.demi_dedup_compact_dev.restype = C.c_int32
    L.demi_dedup_compact_dev.argtypes = [vp, vp, C.c_uint64, C.c_int32, vp, vp, vp, vp]
    L.demi_dedup_compact.restype = C.c_int32
    L.demi_dedup_compact.argtypes = [vp, vp, C.c_uint64, C.c_int32, vp, vp, C.POINTER(C.c_uint64)]
    L.demi_replay_batch_ex.restype = C.c_int32
    L.demi_replay_batch_ex.argtypes = [vp, vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp]
    L.demi_replay_trace.restype = C.c_int32
    L.demi_replay_trace.argtypes = [vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, vp, C.c_uint32,
                                    C.POINTER(C.c_uint32), vp]
    L.demi_internal_minimize.restype = C.c_int32
    L.demi_internal_minimize.argtypes = [vp, C.c_uint32, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, C.POINTER(IntMinOut)]
    L.demi_provenance.restype = C.c_int32
    L.demi_provenance.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint32, C.c_uint32, vp, C.c_uint32, vp]
    L.demi_fuzz_provenance.restype = C.c_int32
    L.demi_fuzz_provenance.argtypes = [vp, C.POINTER(FuzzParams), vp, C.c_uint32, vp, C.c_uint32, vp, vp]
    L.demi_dpor_batch.restype = C.c_int32
    L.demi_dpor_batch.argtypes = [vp, vp, vp, C.c_uint32, C.POINTER(DporParams), vp, vp, C.c_uint32, vp, C.c_uint32]
    L.demi_dpor_batch_ex.restype = C.c_int32
    L.demi_dpor_batch_ex.argtypes = [vp, vp, vp, C.c_uint32, C.POINTER(DporParams), C.POINTER(DporEx), vp, vp, C.c_uint32,
                                     vp, C.c_uint32]
    L.demi_incremental_ddmin.restype = C.c_int32
    L.demi_incremental_ddmin.argtypes = [vp, vp, C.c_uint32, C.POINTER(DporParams), C.c_uint32, C.POINTER(DporSeed),
                                         C.c_int32, C.c_uint32, vp, C.c_uint32, C.POINTER(IncDDMinOut)]
    L.demi_dpor_frontier.restype = C.c_int32
    L.demi_dpor_frontier.argtypes = [vp, vp, C.c_uint32, C.POINTER(FrontierParams), vp, vp, C.c_uint32, vp, C.c_uint64]
    L.demi_dpor_frontier_multi.restype = C.c_int32
    L.demi_dpor_frontier_multi.argtypes = [vp, C.c_int32, vp, C.c_uint32, C.POINTER(FrontierParams), vp, vp, C.c_uint32,
                                           vp, C.c_uint64]
    L.demi_comm_unique_id.restype = C.c_int32
    L.demi_comm_unique_id.argtypes = [vp]
    L.demi_comm_init.restype = C.c_int32
    L.demi_comm_init.argtypes = [vp, vp, C.c_int32, C.c_int32]
    L.demi_comm_rank.restype = C.c_int32
    L.demi_comm_rank.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.demi_create_multi.restype = C.c_int32
    L.demi_create_multi.argtypes = [C.POINTER(Config), vp, C.c_int32, vp]
    L.demi_set_user_filter.restype = C.c_int32
    L.demi_set_user_filter.argtypes = [vp, vp, C.c_uint32]
    L.demi_load_model.restype = C.c_int32
    L.demi_load_model.argtypes = [vp, C.c_char_p, C.c_size_t]
    L.demi_actor_index.restype = C.c_int32
    L.demi_actor_index.argtypes = [vp, C.c_char_p]
    L.demi_actor_name.restype = C.c_char_p
    L.demi_actor_name.argtypes = [vp, C.c_uint32]
    L.demi_fuzzer_generate.restype = C.c_int32
    L.demi_fuzzer_generate.argtypes = [C.POINTER(FuzzerConfig), C.c_int64, vp, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32,
                                       C.POINTER(C.c_uint32)]
    L.demi_experiment_save.restype = C.c_int32
    L.demi_experiment_save.argtypes = [C.c_char_p, C.POINTER(Experiment)]
    L.demi_experiment_load.restype = C.c_int32
    L.demi_experiment_load.argtypes = [C.c_char_p, C.POINTER(Experiment)]
    L.demi_conjoin_atoms.restype = C.c_int32
    L.demi_conjoin_atoms.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.demi_fuzz_subseq_batch.restype = C.c_int32
    L.demi_fuzz_subseq_batch.argtypes = [vp, C.POINTER(FuzzParams), vp, C.c_uint32, C.c_uint32, vp, vp]
    L.demi_random_ddmin.restype = C.c_int32
    L.demi_random_ddmin.argtypes = [vp, C.POINTER(FuzzParams), vp, C.c_uint32, C.c_int32, vp, C.c_uint32, vp, vp,
                                    C.c_uint32, C.POINTER(DDMinOut), C.POINTER(C.c_int64)]
    L.demi_stats.restype = C.c_int32
    L.demi_stats.argtypes = [vp, C.POINTER(Perf)]
    _lib = L
    return L
