// ddmin_driver.hpp — DDMin (minification/DeltaDebugging.scala:27-109) as a sequential commit loop over a
// memo of test results that is filled speculatively in batches.  The decisions, the MCS and the counters are
// the sequential ones; what changes is how many tests are evaluated and when.  The test oracle is a hook:
// STSSched replays (capi_replay.cu) or resumable DPOR instances (capi_dpor.cu).
#pragma once
#include <algorithm>
#include <chrono>
#include <cstring>
#include <map>
#include <vector>
#include "engine.hpp"

namespace demi {

typedef std::vector<uint64_t> Mask;

struct Atom { uint32_t first, second; };

struct DDMinDriver {
  demi_handle* h;
  uint32_t looking_for, flags, mw, n_ext;
  const demi_ext_event* ext;
  std::map<Mask, bool> memo;           // mask -> violation reproduced?
  uint32_t original_num_events = 0, total_inputs_pruned = 0, total_replays = 0;
  std::vector<uint32_t> iteration_sizes;
  std::vector<uint32_t> iteration_keys;   // stats.total_replays when each iteration size was recorded (replay_count())
  uint32_t replays_executed = 0, batches = 0;
  int32_t error = DEMI_OK;
  bool malformed = false;
  // interference siblings waiting on the recursion stack: (dag, remainder)
  std::vector<std::pair<Mask, Mask>> pending_siblings;
  static constexpr size_t BATCH_TARGET = 4096;
  // ---- wide speculation.  STSSched replays are cheap and a test's latency, not its cost, is what a minimisation
  // waits for: on a miss, the closure of the decision tree below the current frame is evaluated level by level up to
  // `wide_cap` tests — about one full wave of the replay kernel — so a whole DDMin run is one or two launches.  The
  // host side must then not cost more than the launch: masks live in one flat arena (a batch is a contiguous slice of
  // it, handed to the kernel as is), the memo is an open-addressing table over that arena with exact comparison, and
  // halves() is cached per dag (it depends on the dag alone; a run meets ~2n distinct dags).
  size_t wide_cap = 0;
  struct WideTable {
    uint32_t mw = 0;
    std::vector<uint64_t> arena; std::vector<signed char> res; std::vector<int32_t> slots;
    void init(uint32_t w) { mw = w; arena.clear(); res.clear(); slots.assign(1u << 15, -1); arena.reserve((size_t)w << 15); res.reserve(1u << 15); }
    size_t size() const { return res.size(); }
    static uint64_t hash(const uint64_t* m, uint32_t w) {
      uint64_t h = 0x9E3779B97F4A7C15ull;
      for (uint32_t i = 0; i < w; i++) { h ^= m[i] + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2); h *= 0xD6E8FEB86659FD93ull; }
      return h ^ (h >> 32);
    }
    int32_t find(const uint64_t* m) const {
      const size_t mask = slots.size() - 1;
      for (size_t s = hash(m, mw) & mask;; s = (s + 1) & mask) {
        const int32_t i = slots[s];
        if (i < 0) return -1;
        if (!memcmp(&arena[(size_t)i * mw], m, mw * 8)) return i;
      }
    }
    int32_t insert(const uint64_t* m) {                       // index of m; a new entry has res = -1 (not evaluated)
      int32_t i = find(m);
      if (i >= 0) return i;
      if ((res.size() + 1) * 2 > slots.size()) {
        std::vector<int32_t> ns(slots.size() * 2, -1);
        const size_t mask = ns.size() - 1;
        for (size_t k = 0; k < res.size(); k++) { size_t s = hash(&arena[k * mw], mw) & mask; while (ns[s] >= 0) s = (s + 1) & mask; ns[s] = (int32_t)k; }
        slots.swap(ns);
      }
      i = (int32_t)res.size();
      arena.insert(arena.end(), m, m + mw); res.push_back(-1);
      const size_t mask = slots.size() - 1;
      size_t s = hash(m, mw) & mask; while (slots[s] >= 0) s = (s + 1) & mask; slots[s] = i;
      return i;
    }
  } wt;
  struct DagNode { Mask dag, hv[2]; int32_t child[2]; size_t na; bool ok; };
  std::vector<DagNode> dag_nodes; std::map<Mask, int32_t> dag_index;
  int32_t dag_of(const Mask& dag) {
    auto it = dag_index.find(dag);
    if (it != dag_index.end()) return it->second;
    DagNode n; n.dag = dag; n.child[0] = n.child[1] = -1; n.ok = halves(dag, n.hv, n.na);
    dag_nodes.push_back(std::move(n));
    return dag_index[dag] = (int32_t)dag_nodes.size() - 1;
  }
  int32_t child_of(int32_t d, int k) {
    if (dag_nodes[d].child[k] < 0) { const int32_t c = dag_of(dag_nodes[d].hv[k]); dag_nodes[d].child[k] = c; }
    return dag_nodes[d].child[k];
  }
  // the oracle over a flat slice of masks (default: through evaluate_batch)
  virtual int32_t evaluate_flat(const uint64_t* masks, size_t n, signed char* out) {
    std::vector<Mask> want(n, Mask(mw)); std::vector<char> r(n, 0);
    for (size_t i = 0; i < n; i++) std::copy(masks + i * mw, masks + (i + 1) * mw, want[i].begin());
    int32_t rc = evaluate_batch(want, r);
    for (size_t i = 0; i < n; i++) out[i] = r[i];
    return rc;
  }
  struct Frame { int32_t dag; uint32_t rem; };                  // rem: index into rem_arena
  std::vector<uint64_t> rem_arena;
  // evaluates m and, level by level, the tests the recursion below (dag, rem) — and the waiting siblings — can ask for
  uint64_t spec_us = 0, eval_us = 0;                            // host time building batches / waiting for them
  void speculate_wide(const Mask& m, const Mask& cur_dag, const Mask& cur_rem) {
    const auto tq0 = std::chrono::steady_clock::now();
    const size_t first_new = wt.size();
    wt.insert(m.data());
    rem_arena.clear();
    std::vector<Frame> cur, next;
    auto add_root = [&](const Mask& dag, const Mask& rem) {
      cur.push_back(Frame{dag_of(dag), (uint32_t)(rem_arena.size() / mw)});
      rem_arena.insert(rem_arena.end(), rem.begin(), rem.end());
    };
    add_root(cur_dag, cur_rem);
    for (auto it = pending_siblings.rbegin(); it != pending_siblings.rend(); ++it) add_root(it->first, it->second);
    std::vector<uint64_t> t0(mw), t1(mw);
    while (!cur.empty() && wt.size() - first_new < wide_cap) {
      next.clear();
      for (const Frame f : cur) {
        const DagNode& n = dag_nodes[f.dag];
        if (!n.ok || n.na <= 1) continue;
        for (uint32_t w = 0; w < mw; w++) { const uint64_t r = rem_arena[(size_t)f.rem * mw + w]; t0[w] = n.hv[0][w] | r; t1[w] = n.hv[1][w] | r; }
        wt.insert(t0.data()); wt.insert(t1.data());
        const int32_t c0 = child_of(f.dag, 0), c1 = child_of(f.dag, 1);
        const uint32_t r0 = (uint32_t)(rem_arena.size() / mw);
        rem_arena.insert(rem_arena.end(), t1.begin(), t1.end());      // interference: the remainder grows by the sibling half
        rem_arena.insert(rem_arena.end(), t0.begin(), t0.end());
        next.push_back(Frame{c0, f.rem}); next.push_back(Frame{c1, f.rem});   // a half violates
        next.push_back(Frame{c0, r0}); next.push_back(Frame{c1, r0 + 1});
      }
      if (wt.size() - first_new + 2 * next.size() > 2 * wide_cap) break;     // the next level would not fit a wave
      cur.swap(next);
    }
    // entries inserted earlier but never evaluated cannot exist: every insert above is evaluated right here
    const size_t n_new = wt.size() - first_new;
    if (!n_new) return;
    const auto tq1 = std::chrono::steady_clock::now();
    int32_t rc = evaluate_flat(&wt.arena[first_new * mw], n_new, &wt.res[first_new]);
    const auto tq2 = std::chrono::steady_clock::now();
    spec_us += (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(tq1 - tq0).count();
    eval_us += (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(tq2 - tq1).count();
    if (rc != DEMI_OK) { error = rc; return; }
    replays_executed += (uint32_t)n_new;
    batches++;
  }

  static bool bit(const Mask& m, uint32_t i) { return (m[i >> 6] >> (i & 63)) & 1ull; }
  static void setbit(Mask& m, uint32_t i) { m[i >> 6] |= 1ull << (i & 63); }
  static uint32_t popcount(const Mask& m) { uint32_t c = 0; for (uint64_t w : m) c += (uint32_t)__builtin_popcountll(w); return c; }
  static Mask unite(const Mask& a, const Mask& b) { Mask r(a.size()); for (size_t i = 0; i < a.size(); i++) r[i] = a[i] | b[i]; return r; }

  // UnmodifiedEventDag.get_atomic_events (minification/Util.scala:197-265)
  // UnmodifiedEventDag.conjoinAtoms (minification/Util.scala:167-178): partner index per external, -1 = none
  const std::vector<int32_t>* conjoined = nullptr;
  bool is_conjoined(uint32_t i) const { return conjoined && i < conjoined->size() && (*conjoined)[i] >= 0; }
  bool atomic_events(const Mask& dag, std::vector<Atom>& atoms) const {
    std::vector<int32_t> last_start(DEMI_MAX_ACTORS, -1);
    std::map<std::pair<int, int>, int32_t> last_part;
    atoms.clear();
    // "First deal with explicitly conjoined atoms" (:210-219); both halves must be present (:211).  The reference
    // takes HashSet.head as the atom's first element; canonically the lower original index.
    for (uint32_t i = 0; i < n_ext; i++) {
      if (!bit(dag, i) || !is_conjoined(i)) continue;
      const uint32_t p = (uint32_t)(*conjoined)[i];
      if (p >= n_ext || !bit(dag, p)) return false;
      if (p > i) atoms.push_back({i, p});
    }
    for (uint32_t i = 0; i < n_ext; i++) {
      if (!bit(dag, i)) continue;
      if (is_conjoined(i)) continue;                              // filterNot(_conjoinedAtoms contains ...) :222
      const demi_ext_event& e = ext[i];
      switch (e.kind) {
        case DEMI_EXT_KILL:
          if (last_start[e.a] < 0) return false;                  // "Kill without preceding Start"
          atoms.push_back({(uint32_t)last_start[e.a], i}); last_start[e.a] = -1; break;
        case DEMI_EXT_START: last_start[e.a] = (int32_t)i; break;
        case DEMI_EXT_PARTITION: last_part[{e.a, e.b}] = (int32_t)i; break;
        case DEMI_EXT_UNPARTITION: {
          auto it = last_part.find({e.a, e.b});
          if (it == last_part.end() || it->second < 0) return false;   // "UnPartition without preceding Partition"
          atoms.push_back({(uint32_t)it->second, i}); it->second = -1; break;
        }
        default: atoms.push_back({i, 0xFFFFFFFFu}); break;
      }
    }
    for (int a = 0; a < DEMI_MAX_ACTORS; a++) if (last_start[a] >= 0) atoms.push_back({(uint32_t)last_start[a], 0xFFFFFFFFu});
    for (auto& kv : last_part) if (kv.second >= 0) atoms.push_back({(uint32_t)kv.second, 0xFFFFFFFFu});
    std::stable_sort(atoms.begin(), atoms.end(), [](const Atom& x, const Atom& y) { return x.first < y.first; });
    return true;
  }
  // MinificationUtil.split_list(atoms, 2) (minification/Util.scala:9-37) + remove_events:
  // halves[0] = events of the first chunk, halves[1] = events of the second.
  bool halves(const Mask& dag, Mask out[2], size_t& n_atoms) const {
    std::vector<Atom> atoms;
    if (!atomic_events(dag, atoms)) return false;
    n_atoms = atoms.size();
    size_t n0 = atoms.size() / 2 + (atoms.size() % 2 ? 1 : 0);
    out[0].assign(mw, 0); out[1].assign(mw, 0);
    for (size_t i = 0; i < atoms.size(); i++) {
      Mask& s = out[i < n0 ? 0 : 1];
      setbit(s, atoms[i].first);
      if (atoms[i].second != 0xFFFFFFFFu) setbit(s, atoms[i].second);
    }
    return true;
  }

  // speculative closure of the tests ddmin2(dag, rem) may issue, `depth` levels deep
  void expand(const Mask& dag, const Mask& rem, int depth, std::vector<Mask>& want) {
    if (want.size() >= 4 * BATCH_TARGET) return;
    Mask hv[2]; size_t na;
    if (!halves(dag, hv, na) || na <= 1) return;
    for (int k = 0; k < 2; k++) {
      Mask t = unite(hv[k], rem);
      if (!memo.count(t)) want.push_back(t);
    }
    if (depth <= 0) return;
    expand(hv[0], rem, depth - 1, want);                       // left half violates
    expand(hv[1], rem, depth - 1, want);                       // right half violates
    expand(hv[0], unite(hv[1], rem), depth - 1, want);         // interference
    expand(hv[1], unite(hv[0], rem), depth - 1, want);
  }

  // the oracle: fill `out[i]` = "test(want[i]) reproduces the violation" for the whole batch
  virtual int32_t evaluate_batch(const std::vector<Mask>& want, std::vector<char>& out) = 0;
  // the sequential walk consumed the result of test(m)
  virtual void consumed(const Mask&) {}
  // MinimizationStats.total_replays as the oracle counts it (one per test here; RandomScheduler: one per execution)
  virtual uint32_t replay_count() const { return total_replays; }
  virtual ~DDMinDriver() {}

  void evaluate(std::vector<Mask>& want) {
    std::sort(want.begin(), want.end());
    want.erase(std::unique(want.begin(), want.end()), want.end());
    if (want.empty()) return;
    std::vector<char> res(want.size(), 0);
    int32_t rc = evaluate_batch(want, res);
    if (rc != DEMI_OK) { error = rc; return; }
    for (size_t i = 0; i < want.size(); i++) memo[want[i]] = res[i] != 0;
    replays_executed += (uint32_t)want.size();
    batches++;
  }

  // TestOracle.test for the sequential walk
  bool test(const Mask& m, const Mask& cur_dag, const Mask& cur_rem) {
    if (wide_cap) {
      if (wt.mw != mw) wt.init(mw);
      int32_t i = wt.find(m.data());
      if (i < 0) { speculate_wide(m, cur_dag, cur_rem); if (error != DEMI_OK) return false; i = wt.find(m.data()); }
      consumed(m);
      return wt.res[i] > 0;
    }
    auto it = memo.find(m);
    if (it == memo.end()) {
      std::vector<Mask> want;
      want.push_back(m);
      // depth: 4^d frames * 2 tests; stay near BATCH_TARGET
      int depth = 5;
      expand(cur_dag, cur_rem, depth, want);
      for (auto it2 = pending_siblings.rbegin(); it2 != pending_siblings.rend() && want.size() < BATCH_TARGET; ++it2)
        expand(it2->first, it2->second, 3, want);
      evaluate(want);
      if (error != DEMI_OK) return false;
      it = memo.find(m);
    }
    const bool r = it->second;
    consumed(m);
    return r;
  }

  // DDMin.ddmin2 (DeltaDebugging.scala:73-109)
  Mask ddmin2(const Mask& dag, const Mask& rem) {
    if (error != DEMI_OK) return dag;
    Mask hv[2]; size_t na;
    if (!halves(dag, hv, na)) { malformed = true; error = fail(h, DEMI_ERR_INVALID, "demi_ddmin: Kill/UnPartition without preceding Start/Partition"); return dag; }
    if (na <= 1) return dag;                                             // base case :74-77
    const uint32_t dag_len = popcount(dag);
    for (int k = 0; k < 2; k++) {                                        // :88-102
      Mask t = unite(hv[k], rem);
      bool violates = test(t, dag, rem);
      if (error != DEMI_OK) return dag;
      total_replays++;
      iteration_sizes.push_back(original_num_events - total_inputs_pruned);
      iteration_keys.push_back(replay_count());
      if (violates) {
        total_inputs_pruned += dag_len - popcount(hv[k]);
        return ddmin2(hv[k], rem);
      }
    }
    // interference :104-108 — the right-hand recursion does not depend on the left-hand result
    Mask rem_l = unite(hv[1], rem), rem_r = unite(hv[0], rem);
    pending_siblings.push_back({hv[1], rem_r});
    Mask left = ddmin2(hv[0], rem_l);
    pending_siblings.pop_back();
    Mask right = ddmin2(hv[1], rem_r);
    return unite(left, right);
  }
};


}  // namespace demi
