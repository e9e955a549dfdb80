/*
 * demi_b200.h — C ABI of the B200 schedule-space exploration engine.
 *
 * This is the drop-in boundary for the hot path of NetSys/demi (DEMi).  The
 * reference has no FFI: the path sits behind two Scala traits,
 *   trait Scheduler   (src/main/scala/verification/schedulers/Scheduler.scala:13-104)
 *   trait TestOracle  (src/main/scala/verification/minification/TestOracle.scala:30-55)
 * and the scheduler-specific driver entry points
 *   RandomScheduler.explore/test        (schedulers/RandomScheduler.scala:226-272, :597-612)
 *   STSScheduler.test                   (schedulers/STSScheduler.scala:199-310)
 *   DDMin.minimize                      (minification/DeltaDebugging.scala:27-62)
 *   DPORwHeuristics.test                (schedulers/DPORwHeuristics.scala:1193-1242)
 *   IncrementalDDMin / ResumableDPOR    (minification/IncrementalDeltaDebugging.scala:20-122)
 *   STSSchedMinimizer.minimize          (minification/internal_minimization/ScheduleCheckers.scala:19-107)
 *   ProvenanceTracker.pruneConcurrentEvents (schedulers/Util.scala:267-376)
 * Each entry point below names the reference method it replaces.  A JVM host
 * binds these through a ~150-line JNI shim (jni/DemiNative.c, INTEGRATION.md).
 *
 * Conventions (all entry points):
 *   - return int32 status: 0 = DEMI_OK, <0 = error; text via demi_last_error().
 *   - plain pointers + sizes, little-endian PODs, no C++/torch types.
 *   - blocking, single caller per handle (matches TestOracle.test / explore()).
 *   - host buffers are caller-owned and only borrowed for the call; the
 *     library owns all device memory.  "_dev" variants take device pointers
 *     and a CUDA stream and do not synchronise.
 *   - there is NO CPU fallback: without a CUDA device every compute entry
 *     point returns DEMI_ERR_NO_DEVICE.
 */
#ifndef DEMI_B200_H
#define DEMI_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ status */
#define DEMI_OK                 0
#define DEMI_ERR_INVALID       -1   /* IllegalArgumentException analogue        */
#define DEMI_ERR_STATE         -2   /* IllegalStateException analogue (e.g. no model / no invariant) */
#define DEMI_ERR_NO_DEVICE     -3   /* no CUDA device / extension cannot run     */
#define DEMI_ERR_CUDA          -4   /* CUDA runtime error (text in last_error)   */
#define DEMI_ERR_CAPACITY      -5   /* an on-chip structure overflowed           */
#define DEMI_ERR_REPLAY        -6   /* ReplayException analogue (strict replay diverged) */

/* ------------------------------------------------------------ data model   */

/* Actor index of the "deadLetters" pseudo-sender (externals and timers,
 * RandomScheduler.scala:288-290) and of the "Timer" alias recorded on
 * MsgSend events (RandomScheduler.scala:319). */
#define DEMI_DEADLETTERS 0xFFu
#define DEMI_TIMER_SND   0xFEu
#define DEMI_MAX_ACTORS  32

/* One message: (sender, receiver, fingerprint).  The fingerprint of the
 * reference (MessageFingerprints.scala:9-124) is (type,p0,p1) here, so
 * fingerprint equality is integer equality. 12 bytes. */
typedef struct demi_msg {
  uint8_t  src;     /* actor index or DEMI_DEADLETTERS                       */
  uint8_t  dst;     /* actor index                                           */
  uint8_t  type;    /* model-defined message type                            */
  uint8_t  flags;   /* DEMI_MF_*                                             */
  uint32_t p0, p1;  /* model-defined payload                                 */
} demi_msg;
#define DEMI_MF_EXTERNAL 0x1u  /* enqueued via Send external (ExternalEventInjector.scala:258-268) */
#define DEMI_MF_TIMER    0x2u  /* enqueued via handle_timer (ExternalEventInjector.scala:282-297) */

/* External events (ExternalEvents.scala:62-91).  CodeBlock / WaitCondition /
 * HardKill carry JVM closures or live ActorCells and are out of scope. */
enum {
  DEMI_EXT_START = 1,            /* Start(name)            a = actor          */
  DEMI_EXT_KILL = 2,             /* Kill(name) = isolate   a = actor          */
  DEMI_EXT_SEND = 3,             /* Send(name, msg)        a = dst, type/p0/p1*/
  DEMI_EXT_WAIT_QUIESCENCE = 4,  /* WaitQuiescence()                          */
  DEMI_EXT_PARTITION = 5,        /* Partition(a,b)                            */
  DEMI_EXT_UNPARTITION = 6,      /* UnPartition(a,b)                          */
  DEMI_EXT_HARD_KILL = 7         /* HardKill(name): the actor is stopped for good (EventOrchestrator.scala:243-310).
                                    Model semantics: the scheduler drops every pending message addressed to it
                                    (Scheduler.actorTerminated -> FullyRandom.removeAll, RandomScheduler.scala:536-547,
                                    :686-696), its timers are unregistered (:281-287), it stops being blocked, queued
                                    timers / externals for it are dropped when flushed (ExternalEventInjector.scala:343-346),
                                    it is isolated like a killed actor, and a later Start(name) brings up a fresh instance.
                                    RandomScheduler fuzzing only (the warp engine); replay and DPOR reject it as the
                                    reference's DPOR does ("unsuported external event", DPORwHeuristics.scala:710). */
};
typedef struct demi_ext_event {
  uint8_t  kind, a, b, type;
  uint32_t p0, p1;
  uint32_t id;      /* stable id == UniqueExternalEvent._id (ExternalEvents.scala:14-31) */
} demi_ext_event;   /* 16 bytes */

/* Recorded execution event == one element of EventTrace.events
 * (EventTrace.scala:20, :96-110; AuxilaryTypes.scala:34-73). 16 bytes. */
enum {
  DEMI_EV_MSG_SEND = 1,          /* UniqueMsgSend(MsgSend(snd,rcv,msg), uniq)  */
  DEMI_EV_MSG_EVENT = 2,         /* UniqueMsgEvent(MsgEvent(snd,rcv,msg), uniq)*/
  DEMI_EV_SPAWN = 3,             /* SpawnEvent (from Start)                    */
  DEMI_EV_KILL = 4,              /* KillEvent                                  */
  DEMI_EV_PARTITION = 5,         /* PartitionEvent                             */
  DEMI_EV_UNPARTITION = 6,       /* UnPartitionEvent                           */
  DEMI_EV_BEGIN_WAIT_QUIESCENCE = 7,
  DEMI_EV_QUIESCENCE = 8,
  DEMI_EV_HARD_KILL = 9          /* `events += hardKill` (EventOrchestrator.scala:244)                          */
};
typedef struct demi_event {
  uint8_t  kind, src, dst, type;
  uint32_t p0, p1;
  uint16_t uniq;    /* Uniq id: ties a MsgSend to its MsgEvent (per-execution, from 1) */
  uint16_t node;    /* Unique id in the DepTracker tree (per-execution, root = 0)      */
} demi_event;

/* Built-in actor models ("compiled, data-only" stand-ins for the application's
 * receive(); see DESIGN.md §3).  */
enum {
  DEMI_MODEL_PINGPONG3 = 1,
  DEMI_MODEL_RAFT5 = 2,
  DEMI_MODEL_BCAST32 = 3
  /* 100 = DEMI_MODEL_IR (demi_model_ir.h): the model comes from demi_load_model */
};

/* Engine-wide configuration == SchedulerConfig (SchedulerConfig.scala:9-37)
 * restricted to the fields that are meaningful without a JVM. */
typedef struct demi_config {
  int32_t  device;            /* CUDA device ordinal                           */
  int32_t  model;             /* DEMI_MODEL_*                                   */
  uint32_t model_flags;       /* model-defined (raft5: seeded-bug bits)        */
  uint32_t blocked_mask;      /* Instrumenter.blockedActors as a bitmask       */
  int32_t  ignore_timers;     /* SchedulerConfig.ignoreTimers                  */
  int32_t  strategy;          /* RandomizationStrategy of RandomScheduler: DEMI_RS_FULLY_RANDOM / DEMI_RS_SRC_DST_FIFO */
  int32_t  reserved[2];
} demi_config;
/* FullyRandom (RandomScheduler.scala:635-697) */
#define DEMI_RS_FULLY_RANDOM 0
/* SrcDstFIFO (RandomScheduler.scala:702-909): a random (src,dst) pair, FIFO within the pair; timers and
 * externals in random order.  The reference seeds both of its generators from the wall clock (:705, :712);
 * here both are seeded with the prefix seed (what two constructions in the same millisecond give). */
#define DEMI_RS_SRC_DST_FIFO 1

/* Per-prefix result of one RandomScheduler execution. 32 bytes. */
typedef struct demi_fuzz_result {
  uint32_t violation;     /* ViolationFingerprint code, 0 = none              */
  uint32_t steps;         /* messagesScheduledSoFar at the end                */
  uint64_t state_hash;    /* hash of all actor states at the end              */
  uint64_t trace_hash;    /* order-sensitive hash of the whole EventTrace + dep tree */
  uint16_t n_nodes;       /* DepTracker nodes allocated (incl. root)          */
  uint16_t n_events;      /* EventTrace length                                */
  uint16_t max_pending;   /* high-water mark of the pending set               */
  uint16_t status;        /* 0 ok, else DEMI_PS_*                             */
} demi_fuzz_result;
#define DEMI_PS_OK              0
#define DEMI_PS_PENDING_OVF     1
#define DEMI_PS_QUEUE_OVF       2
#define DEMI_PS_NODE_OVF        3
#define DEMI_PS_EVENT_OVF       4

typedef struct demi_fuzz_params {
  int64_t  seed_base;          /* prefix i runs FullyRandom(seed = seed_base + i) (RandomScheduler.scala:635-639) */
  uint64_t n_prefixes;
  int32_t  max_messages;       /* RandomScheduler.setMaxMessages (RandomScheduler.scala:54-57) */
  int32_t  invariant_check_interval; /* RandomScheduler ctor arg (RandomScheduler.scala:43) */
  uint32_t looking_for;        /* 0 = any violation (explore(_, None)); else only this code */
  uint32_t flags;              /* DEMI_FF_* */
} demi_fuzz_params;
#define DEMI_FF_HASH_PENDING 0x1u  /* state_hash also covers the (canonical, order-free) pending multiset */

typedef struct demi_perf {
  uint64_t prefixes;           /* units processed by the last batch call       */
  uint64_t deliveries;         /* sum of steps                                 */
  uint64_t violations;
  double   kernel_ms;          /* CUDA-event time of the kernel(s)             */
  double   h2d_ms, d2h_ms;
  uint64_t h2d_bytes, d2h_bytes;
  uint32_t kernel_launches;
  uint32_t deferred;           /* random fuzz: prefixes the lane engine handed to the general engine */
} demi_perf;

typedef struct demi_handle demi_handle;

/* ---------------------------------------------------------------- lifecycle */
const char* demi_version(void);
/* Last error text for this handle (or for the failed demi_create if h==NULL). */
const char* demi_last_error(const demi_handle* h);
int32_t demi_device_count(void);

/* new RandomScheduler/STSScheduler/DPORwHeuristics(schedulerConfig, ...) */
int32_t demi_create(const demi_config* cfg, demi_handle** out);
void    demi_destroy(demi_handle* h);

/* A data-only actor model for a handle created with model = DEMI_MODEL_IR (include/demi_model_ir.h): the receive()
 * and invariant programs, initial states, the external-message filter and the actor / message-type name table.  This
 * is what stands in for "the application's receive()" (Instrumenter.scala:913-1017) and `setInvariant`
 * (TestOracle.scala:27) when the host's application is not one of the compiled models.  The blob is copied. */
int32_t demi_load_model(demi_handle* h, const void* model_blob, size_t size);
/* The name table: the reference addresses actors by name (Scheduler.scala:13-104: blockedActors: Set[String], ...),
 * the C ABI by index.  Built-in models name their actors "0", "1", ...; a loaded model brings its own names. */
int32_t demi_actor_index(const demi_handle* h, const char* name);         /* -1 if unknown */
const char* demi_actor_name(const demi_handle* h, uint32_t index);        /* NULL if out of range */

/* The external-event program == the `_trace: Seq[ExternalEvent]` argument of
 * RandomScheduler.explore (RandomScheduler.scala:234) / TestOracle.test. */
int32_t demi_set_externals(demi_handle* h, const demi_ext_event* ev, uint32_t n);

/* FullyRandom(userDefinedFilter = ...) (RandomScheduler.scala:633-684): "userDefinedFilter can throw out entries to
 * be delivered, by returning false".  The closure (src, dst, msg) => Boolean becomes data: a message is REJECTED when
 * it matches any rule (sender in src_mask — or any deadLetters/timer sender when DEMI_FR_DEADLETTERS is set —, receiver
 * in dst_mask, type in type_mask).  As written, a rejected draw is put back after the loop and the loop stops when one
 * element is left (`pendingEvents.size > 1`), so the last remaining message is delivered even if the filter rejects it.
 * n == 0 restores the default filter.  FullyRandom only; at most DEMI_MAX_FILTER_RULES rules. */
typedef struct demi_filter_rule { uint32_t src_mask, dst_mask, type_mask, flags; } demi_filter_rule;
#define DEMI_FRULE_DEADLETTERS 0x1u
#define DEMI_MAX_FILTER_RULES 8
int32_t demi_set_user_filter(demi_handle* h, const demi_filter_rule* rules, uint32_t n);

/* ------------------------------------------------------------- random fuzz */
/* RunnerUtils.fuzz inner loop (RunnerUtils.scala:75-91): n_prefixes independent
 * `new RandomScheduler(cfg, 1, interval, new FullyRandom(seed=seed_base+i)).explore(trace)`
 * executions.  `out` (host) receives n_prefixes records. */
int32_t demi_fuzz_batch(demi_handle* h, const demi_fuzz_params* p,
                        demi_fuzz_result* out_host);
/* Same, results stay in HBM: `out_dev` is a device pointer with room for
 * n_prefixes records; `stream` is a cudaStream_t (0 = default). No sync. */
int32_t demi_fuzz_batch_dev(demi_handle* h, const demi_fuzz_params* p,
                            void* out_dev, void* stream);
/* Device-side summary of a finished batch without copying the records:
 * number of violating prefixes and sum of steps. */
int32_t demi_fuzz_summary_dev(demi_handle* h, const void* results_dev, uint64_t n,
                              void* stream, uint64_t* n_violations, uint64_t* sum_steps);
/* Re-run one seed in recording mode and return its EventTrace
 * (== the EventTrace returned by explore(), RandomScheduler.scala:255-259).
 * `dep_parent[node]` (cap_nodes entries, may be NULL) receives the DepTracker
 * tree (DepTracker.scala:111-116).  n_events and n_nodes receive the counts. */
int32_t demi_fuzz_trace(demi_handle* h, const demi_fuzz_params* p, int64_t seed,
                        demi_event* events, uint32_t cap_events, uint32_t* n_events,
                        uint16_t* dep_parent, uint32_t cap_nodes, uint32_t* n_nodes,
                        demi_fuzz_result* result);

/* ----------------------------------------------- STSSched replay and DDMin */
/* Result of one STSScheduler.test (STSScheduler.scala:199-310). 16 bytes. */
typedef struct demi_replay_result {
  uint16_t violation;    /* matched violation code, 0 = test passes (None)          */
  uint16_t status;       /* 0 ok, DEMI_PS_* overflow, DEMI_RS_DIVERGED (strict mode) */
  uint16_t delivered;    /* expected deliveries that were pending and delivered      */
  uint16_t ignored;      /* expected deliveries skipped ("Ignoring message", :528)   */
  uint64_t state_hash;   /* hash of final actor states + delivered-message sequence  */
} demi_replay_result;
#define DEMI_RS_DIVERGED 16
#define DEMI_RS_UNSUPPORTED 17      /* the test left the regime the batched engine restates exactly */
#define DEMI_RF_FILTER_KNOWN_ABSENTS 0x1u  /* SchedulerConfig.filterKnownAbsents (SchedulerConfig.scala:14) */
#define DEMI_RF_STRICT               0x2u  /* ReplayScheduler semantics: an absent expected delivery diverges */

/* The recorded execution to minimise: STSScheduler.original_trace
 * (STSScheduler.scala:85) and EventTrace.original_externals (EventTrace.scala:20).
 * Usually the output of demi_fuzz_trace for a violating seed. */
int32_t demi_set_trace(demi_handle* h, const demi_event* events, uint32_t n_events,
                       const demi_ext_event* externals, uint32_t n_externals);
/* n_masks independent STSScheduler.test(subseq, fingerprint) calls.  Mask i is
 * `mask_words` uint64 words; bit j selects external event j of the trace's
 * original_externals.  looking_for = the ViolationFingerprint code (0 = any). */
int32_t demi_replay_batch(demi_handle* h, const uint64_t* masks, uint32_t n_masks, uint32_t mask_words,
                          uint32_t looking_for, uint32_t flags, demi_replay_result* out_host);
int32_t demi_replay_batch_dev(demi_handle* h, const void* masks_dev, uint32_t n_masks, uint32_t mask_words,
                              uint32_t looking_for, uint32_t flags, void* out_dev, void* stream);

/* Same as demi_replay_batch with two extensions used by the internal-event minimizers: `masks` may be NULL
 * (every test replays the full external sequence) and `skip_events[i]` (may be NULL; 0xFFFFFFFF = none) names
 * one event of the trace — normally a delivery — that test i leaves out, i.e. the EventTrace that
 * OneAtATimeStrategy.getNextTrace builds (internal_minimization/OneAtATimeRemoval.scala:57-124). */
int32_t demi_replay_batch_ex(demi_handle* h, const uint64_t* masks, const uint32_t* skip_events, uint32_t n_tests,
                             uint32_t mask_words, uint32_t looking_for, uint32_t flags, demi_replay_result* out_host);
/* One STSScheduler.test in recording mode: returns the EventTrace of the replayed execution
 * (`Some(event_orchestrator.events)`, STSScheduler.scala:292-297) with per-execution Uniq ids (node = 0). */
int32_t demi_replay_trace(demi_handle* h, const uint64_t* mask, uint32_t mask_words, uint32_t skip_event,
                          uint32_t looking_for, uint32_t flags,
                          demi_event* events, uint32_t cap_events, uint32_t* n_events, demi_replay_result* result);
/* STSSchedMinimizer + LeftToRightOneAtATime over the trace given to demi_set_trace (which must be a verified
 * MCS trace; its externals are the MCS): RunnerUtils.minimizeInternals (RunnerUtils.scala:980-1003;
 * internal_minimization/ScheduleCheckers.scala:19-107).  Decisions and counters are the sequential ones;
 * candidate removals are evaluated speculatively in batches.  On return the handle's trace is the minimized one. */
#define DEMI_IM_SRC_DST_FIFO 0x100u   /* in `flags`: removalStrategy = SrcDstFIFORemoval (OneAtATimeRemoval.scala:139-251)
                                         instead of LeftToRightOneAtATime (:131-137)                                     */
typedef struct demi_intmin_out {
  uint32_t n_events;            /* length of the minimized EventTrace                       */
  uint32_t deliveries_before, deliveries_after;
  uint32_t total_replays;       /* tests the sequential algorithm issued                    */
  uint32_t n_internal_sizes;    /* record_internal_size entries written                     */
  uint32_t unignorable;         /* RemovalStrategy.unignorable                              */
  uint32_t replays_executed, batches;
} demi_intmin_out;
int32_t demi_internal_minimize(demi_handle* h, uint32_t looking_for, uint32_t flags,
                               demi_event* out_trace, uint32_t cap_events,
                               uint32_t* internal_sizes, uint32_t cap_sizes, demi_intmin_out* out);

/* DDMin.minimize over the trace's externals with STSSched as the TestOracle
 * (RunnerUtils.stsSchedDDMin, RunnerUtils.scala:642-707; DeltaDebugging.scala:27-109).
 * WaitQuiescence externals are dropped first (RunnerUtils.scala:678-684).  The
 * decision sequence, the MCS and the MinimizationStats counters are those of the
 * sequential algorithm; tests are evaluated speculatively in batches. */
typedef struct demi_ddmin_out {
  uint32_t mcs_size;            /* number of external events in the MCS                 */
  uint32_t total_replays;       /* tests the sequential algorithm issued (stats.total_replays) */
  uint32_t n_iterations;        /* entries written to iteration_sizes                   */
  uint32_t replays_executed;    /* tests actually evaluated on the GPU (incl. speculation) */
  uint32_t batches;             /* kernel launches                                      */
  uint32_t verified;            /* verify_mcs: 1 if the MCS still reproduces (DeltaDebugging.scala:64-71) */
  uint32_t reserved[2];
} demi_ddmin_out;
/* UnmodifiedEventDag.conjoinAtoms (minification/Util.scala:167-178; RunnerUtils.scala:321): externals e1 and e2 of
 * the trace given to demi_set_trace (indices into its externals) form one atomic event — DDMin keeps or removes them
 * together.  demi_set_trace starts a new EventDag without conjoined atoms. */
int32_t demi_conjoin_atoms(demi_handle* h, uint32_t e1, uint32_t e2);
int32_t demi_ddmin(demi_handle* h, uint32_t looking_for, uint32_t flags, int32_t check_unmodified,
                   uint64_t* mcs_mask, uint32_t mask_words,
                   uint32_t* iteration_sizes, uint32_t cap_iterations, demi_ddmin_out* out);

/* ------------------------------------------------- DDMin with RandomScheduler */
/* program_of(mask): the externals of the program given to demi_set_externals whose bit is set (bit j selects
 * external j), in their order, except that a selected WaitQuiescence whose previous selected external is also a
 * WaitQuiescence is left out (DDMin can make two of them adjacent; demi_set_externals rejects that, and the second
 * would wait for a quiescence that already holds).  An all-zero mask, or a bit at or beyond n_ext, is
 * DEMI_ERR_INVALID.
 *
 * Test t = RandomScheduler(cfg, max_executions = K = p->n_prefixes, p->invariant_check_interval,
 * FullyRandom(p->seed_base + i) for execution i).test(program_of(mask_t), p->looking_for), run the reference's way:
 * executions i = 0, 1, ... until the first that ends on a matching violation (a hit) or on a capacity status
 * (DEMI_PS_*; the capacities are those of program_of(mask_t) with its own number of Sends, demi_limits.h).
 * first_hit[t] = that execution if it was a hit, else K; first_bad[t] = that execution if it ended on a status,
 * else K.  At most one of the two is below K.  The same numbers come from demi_set_externals(program_of(mask_t)) +
 * demi_fuzz_batch(seed_base, K): the first record with a nonzero violation or status.  Every test runs in one
 * batch: item i*n_tests + t is execution i of test t, and items of a test that already stopped are skipped; no
 * per-execution record is written.  demi_stats: prefixes = executions actually run, deferred as for fuzz.  The
 * handle's program is not changed. */
int32_t demi_fuzz_subseq_batch(demi_handle* h, const demi_fuzz_params* p, const uint64_t* masks, uint32_t n_tests,
                               uint32_t mask_words, uint32_t* first_hit, uint32_t* first_bad);
/* RunnerUtils.randomDDMin (RunnerUtils.scala:601-623): DDMin (DeltaDebugging.scala:27-109) over the whole program
 * given to demi_set_externals, WaitQuiescence included, with the tests above as the TestOracle.  Kill/Start,
 * Partition/UnPartition and the conjoin_pairs (n_pairs (e1, e2) index pairs, UnmodifiedEventDag.conjoinAtoms) are
 * atoms.  Decisions, MCS and iteration_sizes are the sequential ones; tests are evaluated speculatively in batches.
 * out->total_replays = executions the sequential run issues (RandomScheduler counts one per execution it runs,
 * RandomScheduler.scala:248-253: first_hit + 1, or K without a hit); iteration_keys[k] = total_replays when
 * iteration_sizes[k] was recorded (MinimizationStats.iterationSize, Minimizer.scala:183-185).  check_unmodified
 * tests the whole program first and is not counted.  A test that ends on a capacity status, when the sequential
 * walk consumes it, is DEMI_ERR_CAPACITY.  out->verified / *verify_seed: verify_mcs, one more test of the MCS, and
 * the seed of its violating execution (-1 if none), for demi_fuzz_trace on program_of(mcs).  out->replays_executed
 * = tests evaluated (speculation included), out->batches = demi_fuzz_subseq_batch calls.  The handle's program is
 * not changed. */
int32_t demi_random_ddmin(demi_handle* h, const demi_fuzz_params* p, const uint32_t* conjoin_pairs, uint32_t n_pairs,
                          int32_t check_unmodified, uint64_t* mcs_mask, uint32_t mask_words,
                          uint32_t* iteration_sizes, uint32_t* iteration_keys, uint32_t cap_iterations,
                          demi_ddmin_out* out, int64_t* verify_seed);

/* --------------------------------------------------------------------- DPOR */
/* DPORwHeuristics(schedulerConfig, backtrackHeuristic = DefaultBacktrackOrdering,
 * depth_bound, stopIfViolationFound, trackHistory = true) driven like
 * RunnerUtils.boundedDPOR (RunnerUtils.scala:881-978; DPORwHeuristics.scala:77-88,
 * :1193-1242).  Externals must be Start / Send only (DPORwHeuristics.scala:684-721).
 * One *search* explores interleavings strictly in the reference's order; a batch
 * runs independent searches (one per external program) concurrently. */
typedef struct demi_dpor_params {
  int32_t  max_messages;        /* setMaxMessagesToSchedule (:121-126); <0 = unbounded (needs quiescing models) */
  int32_t  depth_bound;         /* setDepthBound (:116-119); <0 = none                       */
  uint32_t max_interleavings;   /* exploration budget per search                             */
  uint32_t looking_for;         /* ViolationFingerprint code, 0 = any                        */
  uint32_t stop_if_found;       /* stopIfViolationFound (:82)                                */
  uint32_t node_cap;            /* capacities of the per-search structures                   */
  uint32_t explored_slots;      /* power of two                                              */
  uint32_t heap_cap;
} demi_dpor_params;
typedef struct demi_dpor_result {
  uint32_t interleavings;       /* executions performed (interleavingCounter)                */
  uint32_t violations;          /* executions that ended in a matching violation             */
  uint64_t deliveries;
  uint64_t races;               /* co-enabled pairs analysed (analyze_dep calls)             */
  uint32_t n_nodes, n_explored, heap_left;
  uint32_t exhausted;           /* backtrack set ran empty ("Tutto finito!", :1148)          */
  uint32_t budget_exhausted;
  uint32_t status;              /* 0 ok, DEMI_DS_*                                           */
} demi_dpor_result;
typedef struct demi_dpor_violation {
  uint64_t schedule_hash;       /* id-independent hash of the delivered (snd,rcv,msg) sequence */
  uint32_t interleaving;        /* index of the execution within its search                  */
  uint16_t length;              /* deliveries                                                */
  uint16_t code;
} demi_dpor_violation;
#define DEMI_DS_NODE_OVF 1
#define DEMI_DS_QUEUE_OVF 2
#define DEMI_DS_EXPLORED_OVF 3
#define DEMI_DS_HEAP_OVF 4
#define DEMI_DS_TRACE_OVF 5
#define DEMI_DS_UNSUPPORTED 6
/* `n_searches` independent searches.  Search s uses externals
 * [ext_offsets[s], ext_offsets[s+1]) of `ext`.  Per search: one result record,
 * up to cap_viol violation records (viol + s*cap_viol), and optionally the
 * schedule hash of every executed interleaving (hashes + s*cap_hashes). */
int32_t demi_dpor_batch(demi_handle* h, const demi_ext_event* ext, const uint32_t* ext_offsets, uint32_t n_searches,
                        const demi_dpor_params* params, demi_dpor_result* results,
                        demi_dpor_violation* viol, uint32_t cap_viol, uint64_t* hashes, uint32_t cap_hashes);

/* Edit-distance bounded, resumable DPOR: the DPOR instances RunnerUtils.editDistanceDporDDMin builds
 * (RunnerUtils.scala:822-835) and ResumableDPOR keeps per external subsequence
 * (minification/IncrementalDeltaDebugging.scala:90-122). */
#define DEMI_DF_ARVIND_ORDERING    0x1u  /* backtrackHeuristic = ArvindDistanceOrdering (BacktrackOrdering.scala:99-173),
                                            initialised with the seed's trace; else DefaultBacktrackOrdering            */
#define DEMI_DF_PRIORITIZE_PENDING 0x2u  /* prioritizePendingUponDivergence (DPORwHeuristics.scala:65-68, :542-555)    */
/* The recorded execution every instance starts from: setInitialDepGraph / setInitialTrace
 * (DPORwHeuristics.scala:210-217) — events + DepTracker tree as returned by demi_fuzz_trace. */
typedef struct demi_dpor_seed {
  const demi_event* events; uint32_t n_events;
  const uint16_t*  dep_parent; uint32_t n_nodes;
} demi_dpor_seed;
typedef struct demi_dpor_ex {
  uint32_t flags;                 /* DEMI_DF_*                                                                   */
  const demi_dpor_seed* seed;     /* may be NULL                                                                 */
  /* search s performs one DPORwHeuristics.test per entry of caps[cap_offsets[s] .. cap_offsets[s+1]) on ONE
   * instance, each after setMaxDistance(cap) (:128-134; cap < 0 = uncapped).  An instance's state is a function of
   * the caps it has been tested with, so "resuming" = passing the longer history.  NULL: one uncapped test.      */
  const int32_t* caps; const uint32_t* cap_offsets;
} demi_dpor_ex;
/* demi_dpor_batch with the options above.  The result record accumulates over the instance's tests; the
 * exhausted / budget_exhausted flags are the last test's; violations > 0 <=> the last test returned Some(trace). */
int32_t demi_dpor_batch_ex(demi_handle* h, const demi_ext_event* ext, const uint32_t* ext_offsets, uint32_t n_searches,
                           const demi_dpor_params* params, const demi_dpor_ex* ex, demi_dpor_result* results,
                           demi_dpor_violation* viol, uint32_t cap_viol, uint64_t* hashes, uint32_t cap_hashes);
/* IncrementalDDMin(ResumableDPOR) (IncrementalDeltaDebugging.scala:20-88): DDMin over `externals` (Start / Send
 * only) with DPOR as the test oracle, the distance cap doubling 0, 2, 4, ... while it is below max_max_distance
 * and the MCS is larger than stop_at_size.  Decisions and counters are the sequential ones; the DPOR tests a
 * round may need are evaluated speculatively in batches. */
typedef struct demi_incddmin_out {
  uint32_t mcs_size;
  uint32_t total_replays;         /* sequential count (mergeStats, :33-41)                  */
  uint32_t rounds;                /* DDMin runs = distance caps tried                        */
  uint32_t instances;             /* DPOR instances the sequential run creates               */
  uint32_t tests_executed;        /* DPOR tests evaluated on the GPU, speculation included   */
  uint32_t batches;
  uint64_t interleavings_executed;
} demi_incddmin_out;
int32_t demi_incremental_ddmin(demi_handle* h, const demi_ext_event* externals, uint32_t n_externals,
                               const demi_dpor_params* params, uint32_t flags, const demi_dpor_seed* seed,
                               int32_t max_max_distance, uint32_t stop_at_size,
                               uint64_t* mcs_mask, uint32_t mask_words, demi_incddmin_out* out);

/* ---------------------------------------------------- frontier ("wide") DPOR */
/* ONE DPORwHeuristics.test (DPORwHeuristics.scala:1193-1242, dpor() :1020-1185) explored as a frontier of
 * backtrack points instead of one interleaving at a time (BASELINE.json configs[2]).  The algorithmic content is the
 * reference's: the same race test (isCoEnabeled :1091-1110), the same backtrack point (analyze_dep :1043-1077:
 * branchI = trace index of the common ancestor, replayThis = trace(branchI+1..laterI) minus `earlier`), the same
 * explored-pair history (ExploredTacker, AuxilaryTypes.scala:209-246; setExplored at :1071-1073 and :1169-1171,
 * isExplored at :1156-1160) and DefaultBacktrackOrdering (deeper branch first, BacktrackOrdering.scala:58-69).
 * What changes is how many backtrack points leave the queue between two race scans: a ROUND dequeues up to `width`
 * unexplored points in queue order, replays them concurrently, then scans all new traces.  width = 1 is the
 * reference's order (one getNext per dpor(), :1142-1185); for width > 1 the set of visited interleavings is that of
 * the same algorithm under a different — but fully specified, deterministic — dequeue schedule:
 *   - queue order: branch descending, then trace slot, later position, earlier position ascending (the FIFO order
 *     of the reference's enqueue loop, :1122-1139, when width = 1);
 *   - a dequeued point whose pair is explored is dropped (:1156-1160); the others are marked explored (:1169-1171)
 *     in queue order, so of two points with the same pair in one round the first one runs;
 *   - nextTrace = keyTrace.take(branchI+1) ++ replayThis: the prefix comes from the trace the point was computed
 *     on (under depth-first order that is the reference's `trace.take(maxIndex+1)`, :1180);
 *   - after a round every new trace is scanned for laterI beyond its own branch point (the pairs below it were
 *     scanned on the parent trace and would only re-enqueue copies that are dropped when dequeued); all races of the
 *     round are marked explored before any of its points is enqueued (enqueueing an explored point is a no-op).
 * Dependency-graph nodes are content-addressed: id(child) = hash(id(parent), snd, rcv, fingerprint) — the child
 * reuse rule of getMessage (:773-801) without a shared table, so a backtrack record is self-contained and can move
 * to another GPU.  Multi-GPU: every rank owns a queue, an explored set and a trace store; after every
 * `rounds_per_exchange` rounds the ranks all-gather their queue lengths, compute the same transfer plan and move
 * surplus records (shallowest first) with grouped ncclSend/ncclRecv (demi_comm_*).  Results are deterministic for a
 * given (width, ranks, rounds_per_exchange, steal_max). */
typedef struct demi_frontier_params {
  int32_t  max_messages;          /* setMaxMessagesToSchedule (:121-126); 1..1000                        */
  uint32_t looking_for;           /* ViolationFingerprint code, 0 = any                                  */
  uint32_t stop_if_found;         /* stopIfViolationFound (:82), applied at round granularity            */
  uint32_t width;                 /* backtrack points replayed per round per rank                        */
  uint64_t max_interleavings;     /* exploration budget over all ranks                                    */
  uint64_t explored_slots;        /* per rank, power of two                                              */
  uint64_t pool_cap;              /* per rank: queued backtrack points                                   */
  uint32_t trace_cap;             /* per rank: trace slots (executed + imported)                         */
  uint32_t rounds_per_exchange;   /* steal period in rounds (ignored on one rank)                        */
  uint32_t steal_max;             /* most records one rank sends to one other rank per exchange          */
  uint32_t flags;                 /* DEMI_FR_*                                                            */
} demi_frontier_params;
#define DEMI_FR_NO_HISTORY 0x1u   /* trackHistory = false (DPORwHeuristics.scala:86): no ExploredTacker, every backtrack
                                     point is replayed; only a budget ends the search                                 */
typedef struct demi_frontier_result {   /* per rank */
  uint64_t interleavings;         /* executions performed on this rank                                   */
  uint64_t violations;
  uint64_t deliveries;
  uint64_t races;                 /* co-enabled pairs analysed                                           */
  uint64_t keys_enqueued, keys_dropped;   /* backtrack points enqueued / dropped as explored when dequeued */
  uint64_t explored_pairs;
  uint64_t pool_left;
  uint64_t records_sent, records_received, bytes_sent;
  uint32_t rounds, exchanges;
  uint32_t exhausted;             /* every rank's queue ran empty ("Tutto finito!", :1148)               */
  uint32_t budget_exhausted;
  uint32_t status;                /* 0 ok, DEMI_DS_*                                                     */
  uint32_t trace_slots;
  double   exec_ms, scan_ms, select_ms, exchange_ms;
} demi_frontier_result;
/* One self-contained backtrack record as it travels between ranks: 16-byte header + (later_i + 1) trace entries. */
typedef struct demi_frontier_entry {    /* one delivered event of a trace, 16 bytes */
  uint64_t id;                    /* content-addressed node id                                           */
  uint8_t  src, dst, type, pad;
  uint16_t parent_pos;            /* trace position of the delivery that created the message (0 = root)  */
  uint16_t pad2;
} demi_frontier_entry;
/* Runs on this handle's device; with a communicator (demi_comm_init) every rank calls it collectively.
 * hashes (cap_hashes, may be NULL): schedule hash of every interleaving executed on this rank, in slot order;
 * viol (cap_viol): this rank's violating interleavings in execution order (`interleaving` indexes `hashes`); when more
 * than cap_viol violate, result->violations still counts them all and which cap_viol records are returned is unspecified. */
int32_t demi_dpor_frontier(demi_handle* h, const demi_ext_event* ext, uint32_t n_ext,
                           const demi_frontier_params* params, demi_frontier_result* result,
                           demi_dpor_violation* viol, uint32_t cap_viol, uint64_t* hashes, uint64_t cap_hashes);

/* ------------------------------------------------------------ communicator */
/* NCCL inside the library (SURVEY §8b: "NCCL is internal").  Multi-process: rank 0 calls demi_comm_unique_id and
 * the host ships the 128 bytes to the other ranks by any means; every rank then calls demi_comm_init.
 * Single-process hosts (a JVM) use demi_create_multi, which creates one handle per device and wires them up. */
#define DEMI_COMM_ID_BYTES 128
int32_t demi_comm_unique_id(uint8_t id[DEMI_COMM_ID_BYTES]);
int32_t demi_comm_init(demi_handle* h, const uint8_t id[DEMI_COMM_ID_BYTES], int32_t rank, int32_t world);
int32_t demi_comm_rank(const demi_handle* h, int32_t* rank, int32_t* world);
/* n handles on `devices[0..n)` in one process, already connected; cfg->device is ignored. */
int32_t demi_create_multi(const demi_config* cfg, const int32_t* devices, int32_t n, demi_handle** out);
/* demi_dpor_frontier on n connected handles of one process (one host thread per device inside the call);
 * results / viol / hashes are per rank (rank r at index r, r*cap_viol, r*cap_hashes). */
int32_t demi_dpor_frontier_multi(demi_handle** hs, int32_t n, const demi_ext_event* ext, uint32_t n_ext,
                                 const demi_frontier_params* params, demi_frontier_result* results,
                                 demi_dpor_violation* viol, uint32_t cap_viol, uint64_t* hashes, uint64_t cap_hashes);

/* ------------------------------------------- state-hash dedup + compaction */
/* Frontier bookkeeping the north-star adds on top of the reference (the
 * reference has no dedup; RunnerUtils.fuzz simply discards executions):
 * K5 inserts every record's 64-bit state_hash into an open-addressing table
 * and keeps, per distinct hash, the record with the smallest prefix index;
 * K4 writes the kept records (mode DEMI_DM_UNIQUE) or the violating ones
 * (DEMI_DM_VIOLATING) densely, in prefix-index order.  All buffers are device
 * pointers; `*_count_dev` is one uint64.  No sync. */
#define DEMI_DM_UNIQUE    0
#define DEMI_DM_VIOLATING 1
int32_t demi_dedup_compact_dev(demi_handle* h, const void* results_dev, uint64_t n, int32_t mode,
                               void* out_records_dev, void* out_index_dev /* uint32[n], may be NULL */,
                               void* out_count_dev, void* stream);
/* Host convenience wrapper: records in host memory in, kept records out. */
int32_t demi_dedup_compact(demi_handle* h, const demi_fuzz_result* results, uint64_t n, int32_t mode,
                           demi_fuzz_result* out_records, uint32_t* out_index, uint64_t* out_count);

/* ------------------------------------------------------ provenance pruning */
/* ProvenanceTracker.pruneConcurrentEvents (schedulers/Util.scala:267-376; called from RunnerUtils.fuzz,
 * RunnerUtils.scala:138-163): drop the deliveries that are not in the happens-before past of the violation.
 * `initialTrace` is DepTracker.initialTrace (DepTracker.scala:63, :126-129): position 0 is the root event,
 * position t >= 1 the t-th delivered Unique.  Bit t of the keep mask says position t stays in the filtered
 * queue.  happens-before is the reflexive-transitive closure of "earlier delivery on the same receiver" and
 * "delivery -> message created by it" (Util.scala:289-304); position t stays iff it happens before the last
 * delivery on some affected node and that delivery does not happen before it (Util.scala:367-374, as
 * written: a last delivery itself only stays if it precedes another one). 32 bytes. */
typedef struct demi_provenance_out {
  uint32_t status;          /* DEMI_PV_*                                                        */
  uint32_t violation;       /* the violation code of the execution (demi_fuzz_provenance only)  */
  uint32_t affected_mask;   /* ViolationFingerprint.affectedNodes (TestOracle.scala:9-18)       */
  uint32_t n_trace;         /* initialTrace length, root included                               */
  uint32_t n_kept;          /* length of the filtered queue                                     */
  uint32_t reserved[3];
} demi_provenance_out;
#define DEMI_PV_OK 0
#define DEMI_PV_CYCLE 1          /* the relation is cyclic: Util.topologicalSort's sys.error (Util.scala:506) */
#define DEMI_PV_OVERFLOW 2       /* trace longer than the mask, or a node id outside the tree                */
#define DEMI_PV_PREFIX_FAILED 3  /* the execution itself ended with a DEMI_PS_* capacity status             */
/* One recorded execution (events + DepTracker tree as returned by demi_fuzz_trace) and the violation's
 * affected actors. keep_mask: mask_words uint64 words, mask_words*64 >= initialTrace length. */
int32_t demi_provenance(demi_handle* h, const demi_event* events, uint32_t n_events,
                        const uint16_t* dep_parent, uint32_t n_nodes, uint32_t affected_mask,
                        uint64_t* keep_mask, uint32_t mask_words, demi_provenance_out* out);
/* The post-fuzz step on a whole batch: re-execute prefixes seed_base + prefix_index[i] (the violating ones a
 * fuzz batch reported) in recording mode, take affectedNodes from the model's invariant on the final states
 * and prune.  keep_masks: n x mask_words uint64, out: n records; results (may be NULL): the n result records. */
int32_t demi_fuzz_provenance(demi_handle* h, const demi_fuzz_params* p, const uint32_t* prefix_index, uint32_t n,
                             uint64_t* keep_masks, uint32_t mask_words, demi_provenance_out* out,
                             demi_fuzz_result* results);

/* ------------------------------------------------- fuzz-test generation, persistence */
/* Fuzzer(num_events, FuzzerWeights, message_gen, prefix, postfix).generateFuzzTest (fuzzing/Fuzzer.scala:24-194),
 * seeded: the reference seeds the fuzzer and its RandomizedHashSets from the wall clock (:67-68; Util.scala:110), here
 * all of them take `seed`.  message_gen = "Send(random alive actor, send_type, running counter)".  Host-only. */
typedef struct demi_fuzzer_config {
  double   kill, send, wait_quiescence, partition, unpartition;   /* FuzzerWeights (Fuzzer.scala:24-29)        */
  uint32_t num_events;
  uint32_t send_type;
} demi_fuzzer_config;
int32_t demi_fuzzer_generate(const demi_fuzzer_config* cfg, int64_t seed,
                             const demi_ext_event* prefix, uint32_t n_prefix,
                             const demi_ext_event* postfix, uint32_t n_postfix,
                             demi_ext_event* out, uint32_t cap, uint32_t* n_out);
/* The flat experiment directory that replaces ExperimentSerializer's Java object streams (Serialization.scala:57-74,
 * :176-254): externals.bin (demi_ext_event[]), event_trace.bin (demi_event[]), dep_parent.bin (uint16[], optional),
 * mcs.bin (uint64[] mask over the externals, optional), meta.json {model, model_flags, violation}.  Load: the counts
 * are always filled in; DEMI_ERR_CAPACITY when a caller buffer is missing or too small. */
typedef struct demi_experiment {
  int32_t  model; uint32_t model_flags; uint32_t violation; uint32_t reserved;
  demi_ext_event* externals; uint32_t n_externals, cap_externals;
  demi_event*     events;    uint32_t n_events, cap_events;
  uint16_t*       dep_parent; uint32_t n_nodes, cap_nodes;
  uint64_t*       mcs_mask;  uint32_t mask_words, cap_mask_words;
} demi_experiment;
int32_t demi_experiment_save(const char* dir, const demi_experiment* e);
int32_t demi_experiment_load(const char* dir, demi_experiment* e);

/* ------------------------------------------------------------- statistics */
int32_t demi_stats(const demi_handle* h, demi_perf* out);

#ifdef __cplusplus
}
#endif
#endif /* DEMI_B200_H */
