// C++ host mirror (include/demi_b200.hpp) end to end.  With a CUDA device: fuzz -> DDMin -> verify ->
// internal minimization -> strict replay -> DPOR.  Without: the no-CPU-fallback contract.
// argv[1]: a directory the experiment round trip may create (the test passes a private temporary one).
#include <cstdio>
#include <cstdlib>
#include "demi_b200.hpp"

using namespace demi;

#define CHECK(c) do { if (!(c)) { std::printf("CHECK failed: %s (line %d)\n", #c, __LINE__); return 1; } } while (0)

int main(int argc, char** argv) {
  SchedulerConfig cfg;
  cfg.model = DEMI_MODEL_RAFT5;
  cfg.model_flags = 1;
  if (demi_device_count() == 0) {
    try { RandomScheduler r(cfg); std::printf("expected an exception\n"); return 1; }
    catch (const Error& e) { CHECK(e.code == DEMI_ERR_NO_DEVICE); std::printf("no device: %s\nOK (no-fallback contract)\n", e.what()); return 0; }
  }
  ExternalEvents prog;
  for (int a = 0; a < 5; a++) prog.push_back(Start((uint8_t)a));
  for (int a = 0; a < 5; a++) prog.push_back(Send((uint8_t)a, 1, 0x1F));
  for (int k = 0; k < 6; k++) prog.push_back(Send((uint8_t)(k % 5), 2, 1 + k));
  prog.push_back(WaitQuiescence());

  RandomScheduler sched(cfg, /*max_executions=*/4000, /*invariant_check_interval=*/5, /*seed=*/1);
  sched.setMaxMessages(50);
  auto found = sched.explore(prog);
  CHECK(found.has_value());
  EventTrace trace = found->first;
  ViolationFingerprint fp = found->second;
  std::printf("violation %u, trace of %zu events\n", fp, trace.size());
  CHECK(!sched.test(prog, 99).has_value());                       // a fingerprint that never occurs

  // RunnerUtils.pruneConcurrentEvents (RunnerUtils.scala:149-163)
  CHECK(sched.affectedNodes != 0);
  ProvenanceTracker prov(sched.engine, trace, sched.depGraph);
  std::vector<uint32_t> kept = prov.pruneConcurrentEvents(sched.affectedNodes);
  std::printf("provenance: %u of %u deliveries precede the violation on nodes %#x\n", (unsigned)kept.size(),
              prov.last.n_trace - 1, sched.affectedNodes);
  CHECK(!kept.empty() && kept.size() + 1 == prov.last.n_kept && prov.last.n_kept < prov.last.n_trace);
  for (uint32_t i : kept) CHECK(trace[i].kind == DEMI_EV_MSG_EVENT);

  // RunnerUtils.editDistanceDporDDMin (RunnerUtils.scala:812-842)
  {
    int32_t deliveries = 0;
    for (const demi_event& e : trace) deliveries += e.kind == DEMI_EV_MSG_EVENT;
    ResumableDPOR rdpor(cfg, trace, sched.depGraph, deliveries, 2000, sched.engine);
    IncrementalDDMin inc(rdpor, /*maxMaxDistance=*/8, /*stopAtSize=*/1);
    ExternalEvents dmcs = inc.minimize(prog, fp);
    std::printf("IncrementalDDMin(DPOR): %u rounds, %u sequential tests, %u DPOR instances -> %zu externals\n",
                inc.last.rounds, inc.last.total_replays, inc.last.instances, dmcs.size());
    CHECK(inc.last.rounds >= 1 && dmcs.size() <= prog.size() - 1 && inc.last.mcs_size == dmcs.size());
  }

  ReplayScheduler replayer(cfg, trace, prog);
  demi_replay_result rr = replayer.replay(fp);                     // validate_replay (RunnerUtils.scala:101-128)
  CHECK(rr.violation == fp && rr.ignored == 0);

  STSScheduler sts(cfg, trace, prog);
  MinimizationStats stats;
  DDMin ddmin(sts, /*checkUnmodifed=*/true, &stats);
  ExternalEvents mcs = ddmin.minimize(fp);
  std::printf("DDMin: %zu -> %zu externals in %u sequential tests (%u executed)\n", prog.size() - 1, mcs.size(),
              stats.total_replays_ref(), ddmin.last.replays_executed);
  CHECK(mcs.size() < prog.size());
  auto verified = ddmin.verify_mcs(mcs, fp);
  if (!verified) { mcs.assign(prog.begin(), prog.end() - 1); verified = sts.test(mcs, fp); }
  CHECK(verified.has_value());
  bool threw = false;
  try { DDMin(sts, true).minimize(77); } catch (const std::invalid_argument&) { threw = true; }   // "Unmodified trace does not trigger violation"
  CHECK(threw);

  STSSchedMinimizer im(mcs, *verified, fp, LeftToRightOneAtATime(), cfg);
  auto res = im.minimize();
  std::printf("internal minimization: %u -> %u deliveries in %u replays\n", im.last.deliveries_before,
              im.last.deliveries_after, res.first.total_replays_ref());
  CHECK(im.last.deliveries_after <= im.last.deliveries_before);
  STSSchedMinimizer fifo_min(mcs, *verified, fp, SrcDstFIFORemoval(), cfg);
  auto fres = fifo_min.minimize();
  std::printf("internal minimization (SrcDstFIFORemoval): %u -> %u deliveries in %u replays\n", fifo_min.last.deliveries_before,
              fifo_min.last.deliveries_after, fres.first.total_replays_ref());
  CHECK(fifo_min.last.deliveries_after <= fifo_min.last.deliveries_before);
  ReplayScheduler final_check(cfg, res.second, mcs);
  CHECK(final_check.replay(fp).violation == fp);

  SchedulerConfig pp; pp.model = DEMI_MODEL_PINGPONG3; pp.model_flags = 1 | (2 << 8);
  DPORwHeuristics dpor(pp, -1, true, 300);
  threw = false;
  try { dpor.test({Start(0)}, 7); } catch (const std::invalid_argument&) { threw = true; }
  CHECK(threw);
  dpor.setMaxMessagesToSchedule(40);
  ExternalEvents pprog = {Start(0), Start(1), Start(2), Send(2, 1, 0), Send(2, 1, 1), Send(2, 1, 2)};
  auto hit = dpor.test(pprog, 7);
  CHECK(hit.has_value() && hit->code == 7);
  std::printf("DPOR: violation after %u interleavings\n", dpor.last.interleavings);

  // one search as a frontier of backtrack points: exhaustive, history on; the same search at width 1 is the reference's order
  {
    FrontierDPOR wide(cfg), narrow(cfg);
    ExternalEvents fprog;
    for (int a = 0; a < 5; a++) fprog.push_back(Start((uint8_t)a));
    for (int a = 0; a < 5; a++) fprog.push_back(Send((uint8_t)a, 1, 0x1F));
    wide.setMaxMessagesToSchedule(36); narrow.setMaxMessagesToSchedule(36);
    wide.params.width = 4096; narrow.params.width = 1;
    wide.params.max_interleavings = narrow.params.max_interleavings = 100000;
    auto vw = wide.test(fprog, 0), vn = narrow.test(fprog, 0);
    std::printf("frontier DPOR: %llu interleavings in %u rounds (width 4096), %llu in %u rounds (width 1); %zu / %zu violations\n",
                (unsigned long long)wide.interleavings(), wide.results[0].rounds, (unsigned long long)narrow.interleavings(),
                narrow.results[0].rounds, vw.size(), vn.size());
    CHECK(wide.results[0].exhausted && narrow.results[0].exhausted);
    CHECK(wide.interleavings() == narrow.interleavings() && vw.size() == vn.size());
  }

  // seeded Fuzzer + the flat experiment directory
  {
    ExternalEvents pre;
    for (int a = 0; a < 5; a++) pre.push_back(Start((uint8_t)a));
    Fuzzer fz(20, FuzzerWeights(), /*send_type=*/2, pre, {WaitQuiescence()});
    ExternalEvents a = fz.generateFuzzTest(7), b = fz.generateFuzzTest(7), c = fz.generateFuzzTest(8);
    CHECK(a.size() == b.size() && a.size() >= pre.size() + 1);
    bool same = true, differs = a.size() != c.size();
    for (size_t i = 0; i < a.size(); i++) same = same && a[i].kind == b[i].kind && a[i].a == b[i].a && a[i].p0 == b[i].p0;
    for (size_t i = 0; i < a.size() && i < c.size(); i++) differs = differs || a[i].kind != c[i].kind || a[i].a != c[i].a || a[i].p0 != c[i].p0;
    CHECK(same && differs);
    Experiment x; x.model = cfg.model; x.model_flags = cfg.model_flags; x.violation = fp; x.externals = prog; x.trace = trace;
    x.dep_parent = sched.depGraph; x.mcs_mask = mask_of(prog, mcs);
    CHECK(argc > 1);
    const std::string dir = argv[1];
    x.save(dir);
    Experiment y = Experiment::load(dir);
    CHECK(y.model == x.model && y.violation == fp && y.externals.size() == prog.size() && y.trace.size() == trace.size());
    CHECK(y.dep_parent == x.dep_parent && y.mcs_mask == x.mcs_mask && y.trace.back().uniq == trace.back().uniq);
    std::printf("Fuzzer: %zu externals (seeded, reproducible); experiment directory round trip ok\n", a.size());
  }
  std::printf("OK\n");
  return 0;
}
