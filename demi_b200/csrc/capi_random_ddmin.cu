// capi_random_ddmin.cu — RunnerUtils.randomDDMin (RunnerUtils.scala:601-623): DDMin over the handle's external
// program with RandomScheduler as the TestOracle.  The speculative commit loop is ddmin_driver.hpp's; one arena
// slice of candidate subsequences is one demi_fuzz_subseq_batch (K1 in subsequence mode, capi.cu).
#include <cstdlib>
#include <vector>
#include "engine.hpp"
#include "ddmin_driver.hpp"

using namespace demi;

namespace {

struct RandomDDMinDriver : DDMinDriver {
  demi_fuzz_params prm{};
  uint32_t K = 0;
  std::vector<uint32_t> hit, bad;          // per arena entry: first_hit / first_bad of its test
  uint64_t executions = 0;                 // stats.total_replays: executions the sequential run issues
  bool counting = false;                   // only the tests of ddmin2 are counted (DeltaDebugging.scala:48)
  uint32_t last_hit = 0;                   // first_hit of the last consumed test

  int32_t evaluate_flat(const uint64_t* masks, size_t n, signed char* out) override {
    const size_t first = (size_t)(masks - wt.arena.data()) / mw;
    hit.resize(first + n); bad.resize(first + n);
    int32_t rc = demi_fuzz_subseq_batch(h, &prm, masks, (uint32_t)n, mw, &hit[first], &bad[first]);
    if (rc != DEMI_OK) return rc;
    for (size_t i = 0; i < n; i++) out[i] = hit[first + i] < K;
    return DEMI_OK;
  }
  int32_t evaluate_batch(const std::vector<Mask>&, std::vector<char>&) override {
    return fail(h, DEMI_ERR_STATE, "demi_random_ddmin: tests are evaluated through the speculation arena only");
  }
  void consumed(const Mask& m) override {
    const int32_t i = wt.find(m.data());
    if (i < 0 || (size_t)i >= hit.size()) { error = fail(h, DEMI_ERR_STATE, "demi_random_ddmin: a consumed test was never evaluated"); return; }
    // the reference stops at the first execution that ends on a violation or a status; a status first is an error
    if (bad[i] < K) { error = fail(h, DEMI_ERR_CAPACITY, "demi_random_ddmin: execution %u of a test overflowed a capacity (demi_limits.h)", bad[i]); return; }
    last_hit = hit[i];
    if (counting) executions += hit[i] < K ? (uint64_t)hit[i] + 1 : K;      // RandomScheduler.scala:248-253
  }
  uint32_t replay_count() const override { return (uint32_t)std::min<uint64_t>(executions, 0xFFFFFFFFull); }
};

}  // namespace

extern "C" int32_t demi_random_ddmin(demi_handle* h, const demi_fuzz_params* p, const uint32_t* conjoin_pairs, uint32_t n_pairs,
                                     int32_t check_unmodified, uint64_t* mcs_mask, uint32_t mask_words,
                                     uint32_t* iteration_sizes, uint32_t* iteration_keys, uint32_t cap_iterations,
                                     demi_ddmin_out* out, int64_t* verify_seed) {
  if (!h) return DEMI_ERR_INVALID;
  if (!p) return fail(h, DEMI_ERR_INVALID, "null params");
  if (!mcs_mask || !out) return fail(h, DEMI_ERR_INVALID, "demi_random_ddmin: null output");
  if (h->ext_host.empty()) return fail(h, DEMI_ERR_STATE, "demi_set_externals has not been called");
  if (p->n_prefixes == 0 || p->n_prefixes > 0xFFFFFFFFull) return fail(h, DEMI_ERR_INVALID, "demi_random_ddmin: max_executions must be in [1, 2^32-1]");
  const uint32_t n_ext = (uint32_t)h->ext_host.size();
  if ((uint64_t)mask_words * 64 < n_ext) return fail(h, DEMI_ERR_INVALID, "mask_words too small");
  if (n_pairs && !conjoin_pairs) return fail(h, DEMI_ERR_INVALID, "demi_random_ddmin: null conjoin_pairs");
  // UnmodifiedEventDag.conjoinAtoms (minification/Util.scala:167-178) over this program; the handle keeps none
  std::vector<int32_t> conjoined(n_ext, -1);
  for (uint32_t k = 0; k < n_pairs; k++) {
    const uint32_t e1 = conjoin_pairs[2 * k], e2 = conjoin_pairs[2 * k + 1];
    if (e1 >= n_ext || e2 >= n_ext) return fail(h, DEMI_ERR_INVALID, "No such external event: %u", e1 >= n_ext ? e1 : e2);
    if (e1 == e2) return fail(h, DEMI_ERR_INVALID, "demi_random_ddmin: an event cannot be conjoined with itself");
    if (conjoined[e1] >= 0 || conjoined[e2] >= 0)
      return fail(h, DEMI_ERR_STATE, "demi_random_ddmin: external %u is already conjoined", conjoined[e1] >= 0 ? e1 : e2);
    conjoined[e1] = (int32_t)e2; conjoined[e2] = (int32_t)e1;
  }
  memset(out, 0, sizeof(*out));
  if (verify_seed) *verify_seed = -1;
  RandomDDMinDriver d;
  d.h = h; d.looking_for = p->looking_for; d.flags = 0; d.mw = mask_words; d.n_ext = n_ext;
  d.ext = h->ext_host.data();
  d.conjoined = &conjoined;
  d.prm = *p; d.K = (uint32_t)p->n_prefixes;
  // tests per speculative batch: about 2^20 executions (K per test) — several waves of the lane engine, since items of
  // a test that already hit are skipped — and no more than 6000 tests, the host's batch-building budget of demi_ddmin
  const uint64_t items = getenv("DEMI_RANDOM_DDMIN_ITEMS") ? (uint64_t)atoll(getenv("DEMI_RANDOM_DDMIN_ITEMS")) : (1ull << 20);
  d.wide_cap = (size_t)std::max<uint64_t>(2, std::min<uint64_t>(6000, items / d.K));
  // randomDDMin passes trace.original_externals as is: WaitQuiescence events are atoms (RunnerUtils.scala:607-611)
  Mask dag(mask_words, 0), zero(mask_words, 0);
  for (uint32_t i = 0; i < n_ext; i++) DDMinDriver::setbit(dag, i);
  if (check_unmodified) {                                                 // DeltaDebugging.scala:41-47
    bool v = d.test(dag, dag, zero);
    if (d.error != DEMI_OK) return d.error;
    if (!v) return fail(h, DEMI_ERR_INVALID, "Unmodified trace does not trigger violation");
  }
  d.original_num_events = DDMinDriver::popcount(dag);
  d.counting = true;
  Mask mcs = d.ddmin2(dag, zero);
  if (d.error != DEMI_OK) return d.error;
  d.iteration_sizes.push_back(d.original_num_events - d.total_inputs_pruned);     // fencepost :60
  d.iteration_keys.push_back(d.replay_count());
  d.counting = false;
  if (d.original_num_events - d.total_inputs_pruned != DDMinDriver::popcount(mcs))
    return fail(h, DEMI_ERR_STATE, "demi_random_ddmin: bookkeeping assertion failed (DeltaDebugging.scala:58)");
  std::copy(mcs.begin(), mcs.end(), mcs_mask);
  // verify_mcs (DeltaDebugging.scala:64-71): one more test of the MCS, with NOP stats
  const bool verified = d.test(mcs, mcs, zero);
  if (d.error != DEMI_OK) return d.error;
  if (verified && verify_seed) *verify_seed = p->seed_base + (int64_t)d.last_hit;
  out->mcs_size = DDMinDriver::popcount(mcs);
  out->reserved[0] = (uint32_t)d.spec_us; out->reserved[1] = (uint32_t)d.eval_us;
  out->total_replays = d.replay_count();
  out->n_iterations = (uint32_t)d.iteration_sizes.size();
  out->replays_executed = d.replays_executed;
  out->batches = d.batches;
  out->verified = verified ? 1u : 0u;
  for (uint32_t i = 0; i < cap_iterations && i < out->n_iterations; i++) {
    if (iteration_sizes) iteration_sizes[i] = d.iteration_sizes[i];
    if (iteration_keys) iteration_keys[i] = d.iteration_keys[i];
  }
  return DEMI_OK;
}
