// demi_b200.hpp — C++ host-side mirror of DEMi's scheduler plugin surface over the C ABI
// (include/demi_b200.h).  Header-only; link with -ldemi_b200.
//
// The reference's host is Scala; this image has no JVM toolchain, so the compiled-language host
// layer that sits above the C ABI is C++ here (the JNI/Scala binding a DEMi maintainer would add is
// in jni/).  Class and method names, argument meaning and error behaviour follow the reference:
//
//   SchedulerConfig      src/main/scala/verification/SchedulerConfig.scala:9-37
//   RandomScheduler      schedulers/RandomScheduler.scala:41 (explore :234, test :597, setMaxMessages :55,
//                        setInvariant :521)
//   STSScheduler         schedulers/STSScheduler.scala:84 (test :199)
//   ReplayScheduler      schedulers/ReplayScheduler.scala:71 (replay; ReplayException :128-130)
//   DDMin                minification/DeltaDebugging.scala:7 (minimize :27, verify_mcs :64)
//   STSSchedMinimizer    minification/internal_minimization/ScheduleCheckers.scala:19 (minimize :34)
//   DPORwHeuristics      schedulers/DPORwHeuristics.scala:77 (test :1193, setMaxMessagesToSchedule :123,
//                        setDepthBound :116)
//   MinimizationStats    minification/Minimizer.scala:30-237 (the counters DDMin / the minimizers drive)
//
// Reference exceptions map to C++ ones: IllegalArgumentException -> std::invalid_argument,
// IllegalStateException -> std::logic_error, ReplayException -> demi::ReplayException, anything the
// engine reports -> demi::Error (code + demi_last_error text).  There is no CPU fallback: without a
// CUDA device the constructors throw demi::Error(DEMI_ERR_NO_DEVICE).
#pragma once
#include <algorithm>
#include <cstdint>
#include <map>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>
#include "demi_b200.h"

namespace demi {

struct Error : std::runtime_error {
  int32_t code;
  Error(int32_t c, const std::string& what) : std::runtime_error(what), code(c) {}
};
struct ReplayException : std::runtime_error { using std::runtime_error::runtime_error; };

typedef uint32_t ViolationFingerprint;          // the model's violation code; 0 = "any" where optional
typedef std::vector<demi_ext_event> ExternalEvents;
typedef std::vector<demi_event> EventTrace;

// ---- external events (ExternalEvents.scala:62-91) with stable ids (UniqueExternalEvent._id)
inline uint32_t next_external_id() { static uint32_t id = 0; return ++id; }            // IDGenerator
inline demi_ext_event Start(uint8_t name) { return {DEMI_EXT_START, name, 0, 0, 0, 0, next_external_id()}; }
inline demi_ext_event Kill(uint8_t name) { return {DEMI_EXT_KILL, name, 0, 0, 0, 0, next_external_id()}; }
inline demi_ext_event Send(uint8_t name, uint8_t type, uint32_t p0 = 0, uint32_t p1 = 0) {
  return {DEMI_EXT_SEND, name, 0, type, p0, p1, next_external_id()};
}
inline demi_ext_event WaitQuiescence() { return {DEMI_EXT_WAIT_QUIESCENCE, 0, 0, 0, 0, 0, next_external_id()}; }
inline demi_ext_event Partition(uint8_t a, uint8_t b) { return {DEMI_EXT_PARTITION, a, b, 0, 0, 0, next_external_id()}; }
inline demi_ext_event UnPartition(uint8_t a, uint8_t b) { return {DEMI_EXT_UNPARTITION, a, b, 0, 0, 0, next_external_id()}; }

struct SchedulerConfig {
  int32_t model = DEMI_MODEL_RAFT5;
  uint32_t model_flags = 0;
  int32_t device = 0;
  bool ignoreTimers = false;
  bool filterKnownAbsents = false;
  uint32_t blocked_mask = 0;
  int32_t strategy = DEMI_RS_FULLY_RANDOM;      // RandomizationStrategy: FullyRandom | SrcDstFIFO
};

// MinimizationStats (minification/Minimizer.scala:30-237) with the reference's shape: one InnerStats per
// <strategy, oracle> pair, the maps keyed by the replay number, and toJson() with the keys of minimization_stats.json.
struct MinimizationStats {
  struct InnerStats {
    std::string name;
    uint32_t total_replays = 0;
    std::map<uint32_t, uint32_t> iterationSize, internalIterationSize, maxDistance;
    std::map<std::string, double> stats;
    explicit InnerStats(const std::string& n) : name(n) { reset(); }
    void reset() {                                                       // :125-157 (total_replays is not reset, as written)
      iterationSize.clear(); internalIterationSize.clear(); maxDistance.clear(); stats.clear();
      for (const char* k : {"prune_duration_seconds", "prune_start_epoch", "prune_end_epoch", "replay_duration_seconds",
                            "replay_end_epoch", "replay_start_epoch", "original_duration_seconds"}) stats[k] = -1.0;
      for (const char* k : {"total_inputs", "total_events", "initial_verification_runs_needed", "minimized_deliveries",
                            "minimized_externals", "minimized_timers"}) stats[k] = 0.0;
    }
    static std::string map_json(const std::map<uint32_t, uint32_t>& m) {
      std::string o = "{"; bool first = true;
      for (auto& kv : m) { o += (first ? "\"" : ", \"") + std::to_string(kv.first) + "\": " + std::to_string(kv.second); first = false; }
      return o + "}";
    }
    std::string toJson() const {                                          // :207-217
      std::string o = "{\"name\": \"" + name + "\", \"iteration_size\": " + map_json(iterationSize) +
                      ", \"internal_iteration_size\": " + map_json(internalIterationSize) + ", \"total_replays\": " +
                      std::to_string(total_replays) + ", \"maxDistance\": " + map_json(maxDistance);
      for (auto& kv : stats) o += ", \"" + kv.first + "\": " + std::to_string(kv.second);
      return o + "}";
    }
  };
  std::string minimization_strategy, test_oracle;
  std::vector<InnerStats> stats;
  void updateStrategy(const std::string& strategy, const std::string& oracle) {   // :41-47
    minimization_strategy = strategy; test_oracle = oracle;
    stats.emplace_back("(" + strategy + "," + oracle + ")");
  }
  InnerStats& inner() { if (stats.empty()) updateStrategy(minimization_strategy, test_oracle); return stats.back(); }
  void reset() { inner().reset(); }
  void increment_replays(uint32_t n = 1) { inner().total_replays += n; }
  void record_iteration_size(uint32_t n) { inner().iterationSize[inner().total_replays] = n; iteration_size.push_back(n); }
  void record_internal_size(uint32_t n) { inner().internalIterationSize[inner().total_replays] = n; internal_size.push_back(n); }
  void record_distance_increase(uint32_t d) { inner().maxDistance[d] = inner().total_replays; }
  void recordDeliveryStats(uint32_t deliveries, uint32_t externals, uint32_t timers) {
    inner().stats["minimized_deliveries"] = deliveries; inner().stats["minimized_externals"] = externals; inner().stats["minimized_timers"] = timers;
  }
  std::string toJson() const {                                            // :98-100
    std::string o = "["; bool first = true;
    for (auto& s : stats) { o += (first ? "" : ", ") + s.toJson(); first = false; }
    return o + "]";
  }
  // the engine returns a minimization's whole record_*_size series; kept in recording order beside the maps
  std::vector<uint32_t> iteration_size, internal_size;
  uint32_t& total_replays_ref() { return inner().total_replays; }
  // one record per test keyed by the replay number, the fencepost record on the last replay number again
  void record_series(const uint32_t* sizes, size_t n, bool internal) {
    InnerStats& in = inner();
    const uint32_t base = in.total_replays;
    for (size_t i = 0; i < n; i++) {
      const uint32_t key = base + (uint32_t)std::min(i + 1, n > 1 ? n - 1 : (size_t)1);
      (internal ? in.internalIterationSize : in.iterationSize)[key] = sizes[i];
      (internal ? internal_size : iteration_size).push_back(sizes[i]);
    }
  }
};

// One demi_handle.
class Engine {
 public:
  explicit Engine(const SchedulerConfig& c) : cfg(c) {
    demi_config dc{};
    dc.device = c.device; dc.model = c.model; dc.model_flags = c.model_flags; dc.blocked_mask = c.blocked_mask;
    dc.ignore_timers = c.ignoreTimers ? 1 : 0; dc.strategy = c.strategy;
    int32_t rc = demi_create(&dc, &h);
    if (rc != DEMI_OK) throw Error(rc, demi_last_error(nullptr));
  }
  ~Engine() { demi_destroy(h); }
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;
  void check(int32_t rc) const {
    if (rc == DEMI_OK) return;
    std::string msg = demi_last_error(h);
    if (rc == DEMI_ERR_INVALID) throw std::invalid_argument(msg);
    if (rc == DEMI_ERR_STATE) throw std::logic_error(msg);
    throw Error(rc, msg);
  }
  demi_handle* handle() const { return h; }
  // an application model as data (demi_model_ir.h) for SchedulerConfig.model == 100; actor / message names as in the blob
  void load_model(const std::vector<uint32_t>& blob) { check(demi_load_model(h, blob.data(), blob.size() * sizeof(uint32_t))); }
  int32_t actor_index(const std::string& name) const { return demi_actor_index(h, name.c_str()); }
  std::string actor_name(int32_t idx) const { const char* n = demi_actor_name(h, idx); return n ? n : ""; }
  // FullyRandom's userDefinedFilter (RandomScheduler.scala:666-684) as rules; an empty list removes it
  void set_user_filter(const std::vector<demi_filter_rule>& rules) { check(demi_set_user_filter(h, rules.data(), (uint32_t)rules.size())); }
  // UnmodifiedEventDag.conjoinAtoms (minification/Util.scala:167-178): DDMin treats the two externals as one atom
  void conjoin_atoms(uint32_t i1, uint32_t i2) { check(demi_conjoin_atoms(h, i1, i2)); }      // indices into the trace's externals
  demi_perf stats() const { demi_perf p{}; demi_stats(h, &p); return p; }
  const SchedulerConfig cfg;
 private:
  demi_handle* h = nullptr;
};

inline std::vector<uint64_t> mask_of(const ExternalEvents& all, const ExternalEvents& subseq) {
  std::vector<uint64_t> m((all.size() + 63) / 64 ? (all.size() + 63) / 64 : 1, 0);
  for (const demi_ext_event& s : subseq)
    for (size_t i = 0; i < all.size(); i++)
      if (all[i].id == s.id) { m[i >> 6] |= 1ull << (i & 63); break; }
  return m;
}
inline ExternalEvents events_of(const ExternalEvents& all, const std::vector<uint64_t>& mask) {
  ExternalEvents out;
  for (size_t i = 0; i < all.size(); i++) if ((mask[i >> 6] >> (i & 63)) & 1ull) out.push_back(all[i]);
  return out;
}

class RandomScheduler {
 public:
  RandomScheduler(const SchedulerConfig& cfg, uint32_t max_executions = 1, int32_t invariant_check_interval = 0,
                  int64_t seed = 0, std::shared_ptr<Engine> e = nullptr)
      : engine(e ? e : std::make_shared<Engine>(cfg)), max_executions(max_executions),
        invariant_check_interval(invariant_check_interval), seed(seed) {}
  std::string getName() const { return "RandomScheduler"; }
  void setMaxMessages(int32_t n) { maxMessages = n; }
  void setInvariant(bool have) { have_invariant = have; }          // models carry their invariant
  // Some((trace, fingerprint)) of the first violating execution, else nullopt (RandomScheduler.scala:234-272)
  std::optional<std::pair<EventTrace, ViolationFingerprint>> explore(const ExternalEvents& trace,
                                                                     ViolationFingerprint lookingFor = 0) {
    if (!have_invariant) throw std::invalid_argument("Must invoke setInvariant before test()");   // :244-246
    engine->check(demi_set_externals(engine->handle(), trace.data(), (uint32_t)trace.size()));
    demi_fuzz_params p{seed, max_executions, maxMessages, invariant_check_interval, lookingFor, 0};
    results.assign(max_executions, demi_fuzz_result{});
    engine->check(demi_fuzz_batch(engine->handle(), &p, results.data()));
    if (stats) stats->increment_replays(max_executions);
    for (uint32_t i = 0; i < max_executions; i++) {
      if (results[i].status) throw Error(DEMI_ERR_CAPACITY, "a prefix overflowed an engine structure");
      if (!results[i].violation) continue;
      EventTrace ev(65536);
      uint32_t n_ev = 0, n_nodes = 0;
      demi_fuzz_result r{};
      depGraph.assign(65536, 0);
      engine->check(demi_fuzz_trace(engine->handle(), &p, seed + i, ev.data(), (uint32_t)ev.size(), &n_ev,
                                    depGraph.data(), (uint32_t)depGraph.size(), &n_nodes, &r));
      ev.resize(n_ev); depGraph.resize(n_nodes);
      // ViolationFingerprint.affectedNodes of the execution found (TestOracle.scala:9-18)
      uint32_t which = i; uint64_t keep[32]; demi_provenance_out po{};
      if (maxMessages >= 0 && maxMessages + 2 <= 32 * 64) {
        engine->check(demi_fuzz_provenance(engine->handle(), &p, &which, 1, keep, 32, &po, nullptr));
        affectedNodes = po.affected_mask;
      }
      return std::make_pair(ev, r.violation);
    }
    return std::nullopt;
  }
  // TestOracle.test: Some(trace) iff the violation was reproduced (RandomScheduler.scala:597-612)
  std::optional<EventTrace> test(const ExternalEvents& events, ViolationFingerprint fp, MinimizationStats* s = nullptr) {
    stats = s;
    auto r = explore(events, fp);
    if (!r) return std::nullopt;
    return r->first;
  }
  // the parameters of one test (DDMin with this scheduler as its oracle runs many at once)
  demi_fuzz_params params(ViolationFingerprint lookingFor) const {
    return demi_fuzz_params{seed, max_executions, maxMessages, invariant_check_interval, lookingFor, 0};
  }
  bool invariant_set() const { return have_invariant; }
  std::shared_ptr<Engine> engine;
  std::vector<demi_fuzz_result> results;
  std::vector<uint16_t> depGraph;      // depTracker.getGraph of the violating execution, as parent pointers
  uint32_t affectedNodes = 0;          // ... and its fingerprint's affectedNodes
 private:
  uint32_t max_executions; int32_t invariant_check_interval; int64_t seed;
  int32_t maxMessages = -1;                                           // Int.MaxValue (:54)
  bool have_invariant = true;
  MinimizationStats* stats = nullptr;
};

class STSScheduler {
 public:
  STSScheduler(const SchedulerConfig& cfg, const EventTrace& original_trace, const ExternalEvents& original_externals,
               bool allowPeek = false, std::shared_ptr<Engine> e = nullptr)
      : engine(e ? e : std::make_shared<Engine>(cfg)), original_trace(original_trace), original_externals(original_externals),
        flags(cfg.filterKnownAbsents ? DEMI_RF_FILTER_KNOWN_ABSENTS : 0) {
    if (allowPeek) throw std::invalid_argument("STSSched with Peek is outside the accelerated path");
    if (original_trace.empty()) throw std::invalid_argument("original_trace must not be empty");     // assume(:203)
    engine->check(demi_set_trace(engine->handle(), original_trace.data(), (uint32_t)original_trace.size(),
                                 original_externals.data(), (uint32_t)original_externals.size()));
  }
  std::string getName() const { return "STSSchedNoPeek"; }
  uint32_t mask_words() const { return (uint32_t)((original_externals.size() + 63) / 64 ? (original_externals.size() + 63) / 64 : 1); }
  // Some(recorded trace) iff the violation was reproduced (STSScheduler.scala:199-310)
  std::optional<EventTrace> test(const ExternalEvents& subseq, ViolationFingerprint fp, MinimizationStats* stats = nullptr) {
    if (stats) stats->increment_replays();
    std::vector<uint64_t> m = mask_of(original_externals, subseq);
    EventTrace ev(65536);
    uint32_t n = 0; demi_replay_result r{};
    engine->check(demi_replay_trace(engine->handle(), m.data(), mask_words(), 0xFFFFFFFFu, fp, flags, ev.data(),
                                    (uint32_t)ev.size(), &n, &r));
    if (r.status) throw Error(DEMI_ERR_CAPACITY, "replay reported a capacity status");
    if (!r.violation) return std::nullopt;
    ev.resize(n);
    return ev;
  }
  std::vector<demi_replay_result> test_batch(const std::vector<std::vector<uint64_t>>& masks, ViolationFingerprint fp) {
    std::vector<uint64_t> flat;
    for (auto& m : masks) flat.insert(flat.end(), m.begin(), m.end());
    std::vector<demi_replay_result> out(masks.size());
    engine->check(demi_replay_batch(engine->handle(), flat.data(), (uint32_t)masks.size(), mask_words(), fp, flags, out.data()));
    return out;
  }
  std::shared_ptr<Engine> engine;
  const EventTrace original_trace;
  const ExternalEvents original_externals;
  const uint32_t flags;
};

class ReplayScheduler : public STSScheduler {
 public:
  using STSScheduler::STSScheduler;
  // strict replay of the recorded trace; throws ReplayException on divergence (ReplayScheduler.scala:71-140)
  demi_replay_result replay(ViolationFingerprint fp = 0) {
    std::vector<uint64_t> m = mask_of(original_externals, original_externals);
    demi_replay_result r{};
    engine->check(demi_replay_batch(engine->handle(), m.data(), 1, mask_words(), fp, flags | DEMI_RF_STRICT, &r));
    if (r.status == DEMI_RS_DIVERGED) throw ReplayException("Expected event not pending after " + std::to_string(r.delivered) + " deliveries");
    if (r.status) throw Error(DEMI_ERR_CAPACITY, "replay reported a capacity status");
    return r;
  }
};

class DDMin {
 public:
  DDMin(STSScheduler& oracle, bool checkUnmodifed = false, MinimizationStats* stats = nullptr)
      : _stats(stats ? stats : &own), oracle(&oracle), checkUnmodifed(checkUnmodifed) {}
  // RunnerUtils.randomDDMin (RunnerUtils.scala:601-623): RandomScheduler as the TestOracle (demi_random_ddmin)
  DDMin(RandomScheduler& oracle, bool checkUnmodifed = false, MinimizationStats* stats = nullptr)
      : _stats(stats ? stats : &own), random(&oracle), checkUnmodifed(checkUnmodifed) {}
  // the MCS (WaitQuiescence dropped, RunnerUtils.scala:678-684); throws std::invalid_argument
  // ("Unmodified trace does not trigger violation") like DeltaDebugging.scala:41-47
  ExternalEvents minimize(ViolationFingerprint fp) {
    if (!oracle) throw std::invalid_argument("DDMin with a RandomScheduler: minimize(fp, externals)");
    std::vector<uint64_t> mcs(oracle->mask_words(), 0);
    std::vector<uint32_t> iters(1 << 16);
    oracle->engine->check(demi_ddmin(oracle->engine->handle(), fp, oracle->flags, checkUnmodifed ? 1 : 0, mcs.data(),
                                     oracle->mask_words(), iters.data(), (uint32_t)iters.size(), &last));
    _stats->iteration_size.clear();
    _stats->record_series(iters.data(), last.n_iterations, false);
    _stats->total_replays_ref() = last.total_replays;
    return events_of(oracle->original_externals, mcs);
  }
  // RandomScheduler oracle: the MCS of `externals` (WaitQuiescence included, RunnerUtils.scala:607-611).  The
  // scheduler's engine runs `externals` for the call and gets its previous program back (`restore`) afterwards.
  ExternalEvents minimize(ViolationFingerprint fp, const ExternalEvents& externals, const ExternalEvents& restore = {}) {
    if (!random) return minimize(fp);
    if (!random->invariant_set()) throw std::invalid_argument("Must invoke setInvariant before test()");
    Engine& e = *random->engine;
    const uint32_t mw = (uint32_t)((externals.size() + 63) / 64 ? (externals.size() + 63) / 64 : 1);
    std::vector<uint64_t> mcs(mw, 0);
    std::vector<uint32_t> sizes(1 << 16), keys(1 << 16);
    const demi_fuzz_params p = random->params(fp);
    e.check(demi_set_externals(e.handle(), externals.data(), (uint32_t)externals.size()));
    const int32_t rc = demi_random_ddmin(e.handle(), &p, conjoined.data(), (uint32_t)(conjoined.size() / 2), checkUnmodifed ? 1 : 0,
                                         mcs.data(), mw, sizes.data(), keys.data(), (uint32_t)sizes.size(), &last, &verify_seed);
    if (!restore.empty()) demi_set_externals(e.handle(), restore.data(), (uint32_t)restore.size());
    e.check(rc);
    _stats->iteration_size.clear();
    for (uint32_t i = 0; i < last.n_iterations && i < sizes.size(); i++) {    // MinimizationStats.iterationSize (Minimizer.scala:183-185)
      _stats->inner().iterationSize[keys[i]] = sizes[i];
      _stats->iteration_size.push_back(sizes[i]);
    }
    _stats->total_replays_ref() = last.total_replays;
    return events_of(externals, mcs);
  }
  // UnmodifiedEventDag.conjoinAtoms for the RandomScheduler form: indices into the externals given to minimize()
  void conjoinAtoms(uint32_t i1, uint32_t i2) { conjoined.push_back(i1); conjoined.push_back(i2); }
  std::optional<EventTrace> verify_mcs(const ExternalEvents& mcs, ViolationFingerprint fp) {
    return oracle ? oracle->test(mcs, fp) : random->test(mcs, fp);
  }
  demi_ddmin_out last{};
  int64_t verify_seed = -1;            // RandomScheduler oracle: seed of the MCS's violating verification execution
  MinimizationStats* _stats;
 private:
  STSScheduler* oracle = nullptr; RandomScheduler* random = nullptr; bool checkUnmodifed; MinimizationStats own;
  std::vector<uint32_t> conjoined;
};

struct LeftToRightOneAtATime {};       // RemovalStrategy (OneAtATimeRemoval.scala:131-137)
struct SrcDstFIFORemoval {};           // RemovalStrategy (OneAtATimeRemoval.scala:139-251)

class STSSchedMinimizer {
 public:
  STSSchedMinimizer(const ExternalEvents& mcs, const EventTrace& verified_mcs, ViolationFingerprint violation,
                    LeftToRightOneAtATime, const SchedulerConfig& cfg, std::shared_ptr<Engine> e = nullptr)
      : engine(e ? e : std::make_shared<Engine>(cfg)), mcs(mcs), verified_mcs(verified_mcs), violation(violation),
        flags(cfg.filterKnownAbsents ? DEMI_RF_FILTER_KNOWN_ABSENTS : 0) {}
  STSSchedMinimizer(const ExternalEvents& mcs, const EventTrace& verified_mcs, ViolationFingerprint violation,
                    SrcDstFIFORemoval, const SchedulerConfig& cfg, std::shared_ptr<Engine> e = nullptr)
      : engine(e ? e : std::make_shared<Engine>(cfg)), mcs(mcs), verified_mcs(verified_mcs), violation(violation),
        flags((cfg.filterKnownAbsents ? DEMI_RF_FILTER_KNOWN_ABSENTS : 0) | DEMI_IM_SRC_DST_FIFO) {}
  std::pair<MinimizationStats, EventTrace> minimize() {
    engine->check(demi_set_trace(engine->handle(), verified_mcs.data(), (uint32_t)verified_mcs.size(), mcs.data(), (uint32_t)mcs.size()));
    EventTrace out(65536); std::vector<uint32_t> sizes(65536);
    engine->check(demi_internal_minimize(engine->handle(), violation, flags, out.data(), (uint32_t)out.size(), sizes.data(),
                                         (uint32_t)sizes.size(), &last));
    out.resize(last.n_events);
    MinimizationStats s;
    s.total_replays_ref() = last.total_replays;
    s.internal_size.clear();
    s.record_series(sizes.data(), last.n_internal_sizes, true);
    return {s, out};
  }
  demi_intmin_out last{};
 private:
  std::shared_ptr<Engine> engine; ExternalEvents mcs; EventTrace verified_mcs; ViolationFingerprint violation; uint32_t flags;
};

// ProvenanceTracker(trace, depGraph) (schedulers/Util.scala:267-376): `trace` is the recorded EventTrace of an
// execution, `dep_parent` its DepTracker tree, both as returned by demi_fuzz_trace.
class ProvenanceTracker {
 public:
  ProvenanceTracker(std::shared_ptr<Engine> e, EventTrace trace, std::vector<uint16_t> dep_parent)
      : engine(std::move(e)), trace(std::move(trace)), dep_parent(std::move(dep_parent)) {}
  // pruneConcurrentEvents(violation): the deliveries of `trace` (by index into it) that stay; the root event,
  // which the reference filters out afterwards (EventTrace.intersection, EventTrace.scala:127-131), is not listed
  std::vector<uint32_t> pruneConcurrentEvents(uint32_t affectedNodes) {
    std::vector<uint32_t> delivery_index;
    for (uint32_t i = 0; i < trace.size(); i++) if (trace[i].kind == DEMI_EV_MSG_EVENT) delivery_index.push_back(i);
    const uint32_t words = (uint32_t)((delivery_index.size() + 1 + 63) / 64);
    std::vector<uint64_t> keep(words, 0);
    engine->check(demi_provenance(engine->handle(), trace.data(), (uint32_t)trace.size(), dep_parent.data(),
                                  (uint32_t)dep_parent.size(), affectedNodes, keep.data(), words, &last));
    if (last.status == DEMI_PV_CYCLE) throw std::runtime_error("happens-before relation is cyclic");   // Util.scala:506
    if (last.status) throw Error(DEMI_ERR_CAPACITY, "provenance: trace does not fit");
    std::vector<uint32_t> kept;
    for (uint32_t t = 1; t <= delivery_index.size(); t++)
      if ((keep[t >> 6] >> (t & 63)) & 1ull) kept.push_back(delivery_index[t - 1]);
    return kept;
  }
  demi_provenance_out last{};
 private:
  std::shared_ptr<Engine> engine;
  EventTrace trace;
  std::vector<uint16_t> dep_parent;
};

class DPORwHeuristics {
 public:
  DPORwHeuristics(const SchedulerConfig& cfg, int32_t depth_bound = -1, bool stopIfViolationFound = true,
                  uint32_t max_interleavings = 1000, std::shared_ptr<Engine> e = nullptr)
      : engine(e ? e : std::make_shared<Engine>(cfg)), depth_bound(depth_bound), stop(stopIfViolationFound), budget(max_interleavings) {}
  std::string getName() const { return "DPORwHeuristics"; }
  void setMaxMessagesToSchedule(int32_t n) { max_messages = n; }
  void setDepthBound(int32_t d) { depth_bound = d; }
  // the first violating interleaving, or nullopt (DPORwHeuristics.scala:1193-1242)
  std::optional<demi_dpor_violation> test(const ExternalEvents& events, ViolationFingerprint fp, MinimizationStats* stats = nullptr) {
    if (max_messages < 0) throw std::invalid_argument("setMaxMessagesToSchedule is required");
    ExternalEvents prog;                                              // convertToDPORTrace (:1279-1303)
    for (const demi_ext_event& e : events) if (e.kind == DEMI_EXT_START || e.kind == DEMI_EXT_SEND) prog.push_back(e);
    uint32_t offs[2] = {0, (uint32_t)prog.size()};
    demi_dpor_params P{max_messages, depth_bound, budget, fp, stop ? 1u : 0u, 4096, 1u << 16, 1u << 15};
    demi_dpor_violation v[8]{};
    engine->check(demi_dpor_batch(engine->handle(), prog.data(), offs, 1, &P, &last, v, 8, nullptr, 0));
    if (stats) stats->increment_replays(last.interleavings);
    if (last.status) throw Error(DEMI_ERR_CAPACITY, "DPOR search reported a capacity status");
    if (!last.violations) return std::nullopt;
    return v[0];
  }
  demi_dpor_result last{};
 private:
  std::shared_ptr<Engine> engine; int32_t depth_bound; bool stop; uint32_t budget; int32_t max_messages = -1;
};

// ResumableDPOR (minification/IncrementalDeltaDebugging.scala:90-122) in RunnerUtils.editDistanceDporDDMin's
// configuration (RunnerUtils.scala:822-835): every instance starts from the recorded execution's dependency graph
// and trace, orders backtrack points by ArvindDistanceOrdering and prioritises pending messages on divergence.
// An instance's state is a function of the caps it has been tested with; that list is what is kept per subsequence.
class ResumableDPOR {
 public:
  ResumableDPOR(const SchedulerConfig& cfg, EventTrace trace, std::vector<uint16_t> depGraph, int32_t max_messages,
                uint32_t max_interleavings = 1000, std::shared_ptr<Engine> e = nullptr,
                uint32_t flags = DEMI_DF_ARVIND_ORDERING | DEMI_DF_PRIORITIZE_PENDING)
      : engine(e ? e : std::make_shared<Engine>(cfg)), trace(std::move(trace)), depGraph(std::move(depGraph)),
        max_messages(max_messages), budget(max_interleavings), flags(flags) {}
  std::string getName() const { return "DPOR"; }
  void setMaxDistance(int32_t d) { currentMaxDistance = d; }
  demi_dpor_seed seed() const { return demi_dpor_seed{trace.data(), (uint32_t)trace.size(), depGraph.data(), (uint32_t)depGraph.size()}; }
  demi_dpor_params params(ViolationFingerprint fp) const { return demi_dpor_params{max_messages, -1, budget, fp, 1u, 4096, 1u << 16, 1u << 16}; }
  // Some(trace) <=> true (:102-121)
  bool test(const ExternalEvents& events, ViolationFingerprint fp, MinimizationStats* stats = nullptr) {
    ExternalEvents prog; std::vector<uint32_t> key;
    for (const demi_ext_event& e : events) if (e.kind == DEMI_EXT_START || e.kind == DEMI_EXT_SEND) { prog.push_back(e); key.push_back(e.id); }
    std::vector<int32_t>& caps = subseqToDPOR[key];
    caps.push_back(currentMaxDistance);
    const uint32_t offs[2] = {0, (uint32_t)prog.size()}, coffs[2] = {0, (uint32_t)caps.size()};
    const demi_dpor_seed sd = seed();
    const demi_dpor_params P = params(fp);
    const demi_dpor_ex ex{flags, &sd, caps.data(), coffs};
    engine->check(demi_dpor_batch_ex(engine->handle(), prog.data(), offs, 1, &P, &ex, &last, nullptr, 0, nullptr, 0));
    if (last.status) throw Error(DEMI_ERR_CAPACITY, "DPOR instance reported a capacity status");
    if (stats) stats->increment_replays();
    return last.violations != 0;
  }
  std::shared_ptr<Engine> engine;
  demi_dpor_result last{};
  uint32_t flags_value() const { return flags; }
 private:
  EventTrace trace; std::vector<uint16_t> depGraph; int32_t max_messages; uint32_t budget, flags;
  int32_t currentMaxDistance = 0;
  std::map<std::vector<uint32_t>, std::vector<int32_t>> subseqToDPOR;
};

// IncrementalDDMin(oracle, maxMaxDistance, stopAtSize) (minification/IncrementalDeltaDebugging.scala:20-88)
class IncrementalDDMin {
 public:
  IncrementalDDMin(ResumableDPOR& oracle, int32_t maxMaxDistance = 256, uint32_t stopAtSize = 1, MinimizationStats* stats = nullptr)
      : oracle(oracle), maxMaxDistance(maxMaxDistance), stopAtSize(stopAtSize), stats(stats) {}
  ExternalEvents minimize(const ExternalEvents& events, ViolationFingerprint fp) {
    ExternalEvents prog;
    for (const demi_ext_event& e : events) if (e.kind == DEMI_EXT_START || e.kind == DEMI_EXT_SEND) prog.push_back(e);
    std::vector<uint64_t> mcs((prog.size() + 63) / 64 ? (prog.size() + 63) / 64 : 1, 0);
    const demi_dpor_seed sd = oracle.seed();
    const demi_dpor_params P = oracle.params(fp);
    oracle.engine->check(demi_incremental_ddmin(oracle.engine->handle(), prog.data(), (uint32_t)prog.size(), &P, oracle.flags_value(),
                                                &sd, maxMaxDistance, stopAtSize, mcs.data(), (uint32_t)mcs.size(), &last));
    if (stats) stats->increment_replays(last.total_replays);
    return events_of(prog, mcs);
  }
  bool verify_mcs(const ExternalEvents& mcs, ViolationFingerprint fp) { return oracle.test(mcs, fp); }
  demi_incddmin_out last{};
 private:
  ResumableDPOR& oracle; int32_t maxMaxDistance; uint32_t stopAtSize; MinimizationStats* stats;
};

// Fuzzer (Fuzzer.scala:24-194): seeded generation of external-event programs.
struct FuzzerWeights { double kill = 0.01, send = 0.3, wait_quiescence = 0.1, partition = 0.1, unpartition = 0.1; };
class Fuzzer {
 public:
  Fuzzer(uint32_t num_events, FuzzerWeights w, uint32_t send_type, ExternalEvents prefix = {}, ExternalEvents postfix = {})
      : num_events(num_events), weights(w), send_type(send_type), prefix(std::move(prefix)), postfix(std::move(postfix)) {}
  ExternalEvents generateFuzzTest(int64_t seed) const {
    demi_fuzzer_config c{weights.kill, weights.send, weights.wait_quiescence, weights.partition, weights.unpartition, num_events, send_type};
    ExternalEvents out(prefix.size() + postfix.size() + 2 * (size_t)num_events + 8);
    uint32_t n = 0;
    int32_t rc = demi_fuzzer_generate(&c, seed, prefix.data(), (uint32_t)prefix.size(), postfix.data(), (uint32_t)postfix.size(),
                                      out.data(), (uint32_t)out.size(), &n);
    if (rc != DEMI_OK) throw Error(rc, demi_last_error(nullptr));
    out.resize(n);
    return out;
  }
 private:
  uint32_t num_events; FuzzerWeights weights; uint32_t send_type; ExternalEvents prefix, postfix;
};

// The flat experiment directory that replaces ExperimentSerializer / ExperimentDeserializer (Serialization.scala:57-254).
struct Experiment {
  int32_t model = 0; uint32_t model_flags = 0; ViolationFingerprint violation = 0;
  ExternalEvents externals; EventTrace trace; std::vector<uint16_t> dep_parent; std::vector<uint64_t> mcs_mask;
  void save(const std::string& dir) const {
    demi_experiment e{};
    e.model = model; e.model_flags = model_flags; e.violation = violation;
    e.externals = const_cast<demi_ext_event*>(externals.data()); e.n_externals = (uint32_t)externals.size();
    e.events = const_cast<demi_event*>(trace.data()); e.n_events = (uint32_t)trace.size();
    e.dep_parent = const_cast<uint16_t*>(dep_parent.data()); e.n_nodes = (uint32_t)dep_parent.size();
    e.mcs_mask = const_cast<uint64_t*>(mcs_mask.data()); e.mask_words = (uint32_t)mcs_mask.size();
    int32_t rc = demi_experiment_save(dir.c_str(), &e);
    if (rc != DEMI_OK) throw Error(rc, demi_last_error(nullptr));
  }
  static Experiment load(const std::string& dir) {
    Experiment x;
    demi_experiment e{};
    int32_t rc = demi_experiment_load(dir.c_str(), &e);                 // counts first
    if (rc != DEMI_OK && rc != DEMI_ERR_CAPACITY) throw Error(rc, demi_last_error(nullptr));
    x.externals.resize(e.n_externals); x.trace.resize(e.n_events); x.dep_parent.resize(e.n_nodes); x.mcs_mask.resize(e.mask_words);
    e.externals = x.externals.data(); e.cap_externals = e.n_externals; e.events = x.trace.data(); e.cap_events = e.n_events;
    e.dep_parent = x.dep_parent.data(); e.cap_nodes = e.n_nodes; e.mcs_mask = x.mcs_mask.data(); e.cap_mask_words = e.mask_words;
    rc = demi_experiment_load(dir.c_str(), &e);
    if (rc != DEMI_OK) throw Error(rc, demi_last_error(nullptr));
    x.model = e.model; x.model_flags = e.model_flags; x.violation = e.violation;
    return x;
  }
};

// ONE DPORwHeuristics.test as a frontier of backtrack points (demi_dpor_frontier); with several devices the frontier is
// sharded and rebalanced by the library's NCCL steal rounds (demi_create_multi + demi_dpor_frontier_multi).
class FrontierDPOR {
 public:
  explicit FrontierDPOR(const SchedulerConfig& cfg, std::vector<int32_t> devices = {}) {
    if (devices.empty()) devices.push_back(cfg.device);
    demi_config dc{};
    dc.device = devices[0]; dc.model = cfg.model; dc.model_flags = cfg.model_flags; dc.blocked_mask = cfg.blocked_mask;
    dc.ignore_timers = cfg.ignoreTimers ? 1 : 0; dc.strategy = cfg.strategy;
    hs.resize(devices.size(), nullptr);
    int32_t rc = devices.size() == 1 ? demi_create(&dc, &hs[0]) : demi_create_multi(&dc, devices.data(), (int32_t)devices.size(), hs.data());
    if (rc != DEMI_OK) throw Error(rc, demi_last_error(nullptr));
  }
  ~FrontierDPOR() { for (demi_handle* h : hs) demi_destroy(h); }
  FrontierDPOR(const FrontierDPOR&) = delete;
  FrontierDPOR& operator=(const FrontierDPOR&) = delete;
  demi_frontier_params params{/*max_messages*/100, 0, 0, /*width*/16384, /*max_interleavings*/1u << 20, /*explored_slots*/1u << 22,
                              /*pool_cap*/1u << 22, /*trace_cap (0: max_interleavings + slack)*/0, /*rounds_per_exchange*/4, /*steal_max*/4096, 0};
  void setMaxMessagesToSchedule(int32_t n) { params.max_messages = n; }
  void trackHistory(bool on) { params.flags = on ? (params.flags & ~DEMI_FR_NO_HISTORY) : (params.flags | DEMI_FR_NO_HISTORY); }
  // returns the violating interleavings found (all ranks); `results[r]` holds rank r's counters
  std::vector<demi_dpor_violation> test(const ExternalEvents& events, ViolationFingerprint fp, uint32_t cap_viol = 4096) {
    params.looking_for = fp;
    if (!params.trace_cap) params.trace_cap = (uint32_t)std::min<uint64_t>(params.max_interleavings + 8ull * params.steal_max + 16, (1u << 28) - 1);
    const size_t n = hs.size();
    results.assign(n, demi_frontier_result{});
    std::vector<demi_dpor_violation> viol(n * cap_viol);
    int32_t rc = n == 1 ? demi_dpor_frontier(hs[0], events.data(), (uint32_t)events.size(), &params, &results[0], viol.data(), cap_viol, nullptr, 0)
                        : demi_dpor_frontier_multi(hs.data(), (int32_t)n, events.data(), (uint32_t)events.size(), &params, results.data(),
                                                   viol.data(), cap_viol, nullptr, 0);
    if (rc != DEMI_OK) { std::string msg = demi_last_error(hs[0]); if (rc == DEMI_ERR_INVALID) throw std::invalid_argument(msg); throw Error(rc, msg); }
    std::vector<demi_dpor_violation> out;
    for (size_t r = 0; r < n; r++) {
      const uint64_t k = std::min<uint64_t>(results[r].violations, cap_viol);
      out.insert(out.end(), viol.begin() + r * cap_viol, viol.begin() + r * cap_viol + k);
    }
    return out;
  }
  uint64_t interleavings() const { uint64_t t = 0; for (auto& r : results) t += r.interleavings; return t; }
  std::vector<demi_frontier_result> results;
 private:
  std::vector<demi_handle*> hs;
};

}  // namespace demi
