// engine.hpp — the handle behind the C ABI, shared by capi.cu and capi_replay.cu.
#pragma once
#include <climits>
#include <cstdlib>
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include <string>
#include <vector>
#include <map>
#include <algorithm>
#include <cuda_runtime.h>
#include "../../include/demi_b200.h"
#include "../../include/demi_limits.h"
#include "../../include/demi_model_ir.h"

extern thread_local std::string g_create_error;

struct DedupScratch { void* keys = nullptr; size_t keys_b = 0; void* vals = nullptr; size_t vals_b = 0;
                      void* keep = nullptr; size_t keep_b = 0; void* counts = nullptr; size_t counts_b = 0; };

struct demi_handle {
  DedupScratch dedup;
  demi_config cfg{};
  std::string err;
  int sm_count = 0;
  // external program
  std::vector<demi_ext_event> ext_host;
  demi_ext_event* ext_dev = nullptr;
  uint32_t n_ext_sends = 0;
  // device buffers
  demi_fuzz_result* results_dev = nullptr; size_t results_cap = 0;
  uint4* node_scratch = nullptr; size_t node_scratch_bytes = 0;
  uint4* pend_scratch = nullptr; size_t pend_scratch_bytes = 0;
  unsigned long long* counters_dev = nullptr;      // [0]=sum_steps [1]=n_violations
  // lane engine
  uint4* ext_sends_dev = nullptr;
  bool has_partitions = false, ext_sends_distinct = true;
  uint4* lane_pend = nullptr; size_t lane_pend_bytes = 0;
  uint32_t* ovf_list = nullptr; size_t ovf_list_bytes = 0;
  uint32_t* ovf_count = nullptr;
  uint16_t* fifo_scratch = nullptr; size_t fifo_scratch_bytes = 0;
  int use_lane_engine = 1;
  uint32_t lane_pending_cap = 0;      // DEMI_LANE_PENDING_CAP (tests): the lane engine defers beyond this many pending messages
  uint32_t* rec_counts_dev = nullptr;
  void* prov_scratch = nullptr; size_t prov_scratch_bytes = 0;
  void* dpor_buf[24] = {}; size_t dpor_buf_bytes[24] = {};     // K3 per-search structures (capi_dpor.cu)
  // pinned staging for host transfers
  void* pinned = nullptr; size_t pinned_bytes = 0;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  demi_perf perf{};
  // ---- STSSched replay / DDMin (capi_replay.cu)
  std::vector<demi_event> trace_host;
  std::vector<demi_ext_event> trace_ext_host;
  std::vector<uint16_t> send_ext_index_host;
  std::vector<int32_t> conjoined;          // UnmodifiedEventDag._conjoinedAtoms over trace_ext_host (demi_conjoin_atoms)
  void* trace_dev = nullptr; void* trace_ext_dev = nullptr;
  uint16_t* ev_ordinal_dev = nullptr; uint16_t* send_ext_index_dev = nullptr;
  uint32_t trace_n_uniq = 0, trace_n_send_events = 0, trace_n_ext_sends = 0;
  void* rp_table = nullptr; size_t rp_table_bytes = 0; uint32_t rp_gen_next = 0; uint64_t rp_table_geometry = 0;
  void* rp_tosend = nullptr; size_t rp_tosend_bytes = 0;
  void* rp_pruned = nullptr; size_t rp_pruned_bytes = 0;
  void* rp_masks = nullptr; size_t rp_masks_bytes = 0;
  void* rp_results = nullptr; size_t rp_results_bytes = 0;
  unsigned long long* rp_counters = nullptr;
  // ---- communicator (capi_frontier.cu): NCCL inside the library
  void* comm = nullptr;
  void* frontier = nullptr;      // cached K3F buffers
  // ---- a model loaded with demi_load_model (model == DEMI_MODEL_IR)
  bool ir_loaded = false;
  uint32_t* ir_blob_dev = nullptr;
  demi_ir_device ir_dev{};
  uint32_t ir_ext_mask = 0, ir_fanout = 0, ir_n_actors = 0, ir_n_types = 0;
  std::vector<std::string> names;      // actor names, then message-type names
  // ---- FullyRandom's userDefinedFilter as rules (demi_set_user_filter); HardKill in the external program
  std::vector<demi_filter_rule> filter;
  bool has_hard_kill = false;
  // ---- launch bookkeeping
  std::map<const void*, int> occupancy;          // kernel -> resident blocks per SM (asked once per handle)
  void* trace_rec = nullptr; size_t trace_rec_bytes = 0;   // demi_fuzz_trace's recording buffer
  void* subseq_buf = nullptr; size_t subseq_buf_bytes = 0; // demi_fuzz_subseq_batch: per-test side tables + verdicts
};
void demi_replay_free(demi_handle* h);
void demi_comm_free(demi_handle* h);
void demi_frontier_free(demi_handle* h);

inline int32_t ensure_bytes(demi_handle* h, void** p, size_t* cap, size_t need);

inline int32_t fail(demi_handle* h, int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}
#define CUDA_TRY(h, expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) \
  return fail((h), DEMI_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)


// ---- validation of caller-supplied records (JNI hands over JVM buffers): every actor index, node id and parent
// pointer is range-checked before any host table or kernel indexes with it.
inline int demi_model_actors(const demi_handle* h) {
  const int model = h->cfg.model;
  if (model == DEMI_MODEL_IR) return (int)h->ir_n_actors;
  return model == DEMI_MODEL_PINGPONG3 ? 3 : model == DEMI_MODEL_RAFT5 ? 5 : 32;
}
// the `model` argument of the capacity rules in demi_limits.h (a loaded model carries its fan-out in the key)
inline int demi_model_key(const demi_handle* h) { return h->cfg.model == DEMI_MODEL_IR ? (DEMI_MODEL_IR | (int)(h->ir_fanout << 8)) : h->cfg.model; }
inline uint32_t demi_ext_type_mask(const demi_handle* h) { return h->cfg.model == DEMI_MODEL_IR ? h->ir_ext_mask : demi_external_type_mask(h->cfg.model); }
inline int32_t demi_need_model(demi_handle* h) {
  if (h->cfg.model == DEMI_MODEL_IR && !h->ir_loaded) return fail(h, DEMI_ERR_STATE, "demi_load_model has not been called");
  return DEMI_OK;
}
inline int32_t demi_check_externals(demi_handle* h, const char* who, const demi_ext_event* ev, uint32_t n) {
  const uint32_t na = (uint32_t)demi_model_actors(h);
  for (uint32_t i = 0; i < n; i++) {
    const demi_ext_event& e = ev[i];
    if (e.kind < DEMI_EXT_START || e.kind > DEMI_EXT_UNPARTITION)      // HardKill: RandomScheduler fuzzing only
      return fail(h, DEMI_ERR_INVALID, "%s: external %u has kind %u, which this entry point does not accept", who, i, (unsigned)e.kind);
    const bool needs_a = e.kind != DEMI_EXT_WAIT_QUIESCENCE;
    const bool needs_b = e.kind == DEMI_EXT_PARTITION || e.kind == DEMI_EXT_UNPARTITION;
    if ((needs_a && e.a >= na) || (needs_b && e.b >= na)) return fail(h, DEMI_ERR_INVALID, "%s: external %u names an unknown actor", who, i);
  }
  return DEMI_OK;
}
// n_nodes == 0: node ids are not checked (traces recorded by STSScheduler carry node = 0)
// max_actors == 0: the handle's model decides; else an explicit bound (provenance pruning works on any <= 32 actors)
inline int32_t demi_check_events(demi_handle* h, const char* who, const demi_event* ev, uint32_t n, uint32_t n_nodes,
                                 uint32_t max_actors = 0) {
  const uint32_t na = max_actors ? max_actors : (uint32_t)demi_model_actors(h);
  for (uint32_t i = 0; i < n; i++) {
    const demi_event& e = ev[i];
    bool ok = true;
    switch (e.kind) {
      case DEMI_EV_MSG_SEND:  ok = (e.src < na || e.src == DEMI_DEADLETTERS || e.src == DEMI_TIMER_SND) && e.dst < na; break;
      case DEMI_EV_MSG_EVENT: ok = (e.src < na || e.src == DEMI_DEADLETTERS || e.src == DEMI_TIMER_SND) && e.dst < na; break;
      case DEMI_EV_SPAWN: case DEMI_EV_KILL: ok = e.dst < na; break;
      case DEMI_EV_PARTITION: case DEMI_EV_UNPARTITION: ok = e.src < na && e.dst < na; break;
      case DEMI_EV_BEGIN_WAIT_QUIESCENCE: case DEMI_EV_QUIESCENCE: break;
      default: return fail(h, DEMI_ERR_INVALID, "%s: event %u has unknown kind %u", who, i, (unsigned)e.kind);
    }
    if (!ok) return fail(h, DEMI_ERR_INVALID, "%s: event %u names an unknown actor (src %u, dst %u)", who, i, (unsigned)e.src, (unsigned)e.dst);
    if (n_nodes && (e.kind == DEMI_EV_MSG_SEND || e.kind == DEMI_EV_MSG_EVENT) && e.node >= n_nodes)
      return fail(h, DEMI_ERR_INVALID, "%s: event %u names node %u outside the tree of %u", who, i, (unsigned)e.node, n_nodes);
  }
  return DEMI_OK;
}
inline int32_t demi_check_parents(demi_handle* h, const char* who, const uint16_t* dep_parent, uint32_t n_nodes) {
  for (uint32_t v = 1; v < n_nodes; v++)
    if (dep_parent[v] >= v) return fail(h, DEMI_ERR_INVALID, "%s: node %u has parent %u (a parent is created before its children)", who, v, (unsigned)dep_parent[v]);
  return DEMI_OK;
}

inline int32_t ensure_bytes(demi_handle* h, void** p, size_t* cap, size_t need) {
  if (*cap >= need) return DEMI_OK;
  cudaFree(*p); *p = nullptr; *cap = 0;
  CUDA_TRY(h, cudaMalloc(p, need));
  *cap = need;
  return DEMI_OK;
}
