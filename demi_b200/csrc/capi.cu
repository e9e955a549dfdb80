// capi.cu — the C ABI (include/demi_b200.h) over the CUDA engine.
// No CPU fallback: every compute entry point needs a CUDA device.
#include <climits>
#include <cstdlib>
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include <cuda_runtime.h>
#include "fuzz_kernel.cuh"
#include "provenance_kernel.cuh"
#include "lane_kernel.cuh"
#include "subseq_kernel.cuh"
#include "models/model_ir.cuh"

using namespace demi;

#include "engine.hpp"

thread_local std::string g_create_error;

// ------------------------------------------------------------ kernel table
constexpr int WARPS = 4;
typedef void (*kernel_fn)(const KernelArgs);
typedef void (*subseq_fn)(const SubseqArgs);
struct Variant {
  int model; uint32_t pcap, tcap; bool pend_global, record;
  kernel_fn fn; size_t smem_per_warp;
  subseq_fn sub;             // the same machine in subsequence mode (non-recording variants)
};
template <class MODEL, int PCAP, int TCAP, bool PG, bool REC>
static Variant make_variant() {
  using M = Machine<MODEL, PCAP, TCAP, PG, REC>;
  subseq_fn sub = nullptr;
  if constexpr (!REC) sub = fuzz_subseq_kernel<MODEL, PCAP, TCAP, PG, WARPS>;
  return Variant{MODEL::ID, (uint32_t)PCAP, (uint32_t)TCAP, PG, REC,
                 fuzz_kernel<MODEL, PCAP, TCAP, PG, REC, WARPS>, sizeof(typename M::Smem), sub};
}
static const std::vector<Variant>& variants() {
  static const std::vector<Variant> v = {
    make_variant<PingPong3, 128, 128, false, false>(),
    make_variant<PingPong3, 16384, 1024, true, false>(),
    make_variant<PingPong3, 16384, 1024, true, true>(),
    make_variant<Raft5, 256, 32, false, false>(),
    make_variant<Raft5, 512, 32, false, false>(),
    make_variant<Raft5, 256, 32, false, true>(),          // recording, shared-memory pending set (provenance batches)
    make_variant<Raft5, 16384, 1024, true, false>(),
    make_variant<Raft5, 16384, 1024, true, true>(),
    make_variant<Bcast32, 16384, 32, true, false>(),
    make_variant<Bcast32, 16384, 1024, true, false>(),
    make_variant<Bcast32, 16384, 1024, true, true>(),
    make_variant<IrModel, 128, 128, false, false>(),      // a model loaded with demi_load_model
    make_variant<IrModel, 16384, 1024, true, false>(),
    make_variant<IrModel, 16384, 1024, true, true>(),
  };
  return v;
}
static const Variant* pick_variant(int model, uint32_t pcap, uint32_t tcap, bool record, bool need_global) {
  for (const Variant& v : variants())
    if (v.model == model && v.record == record && v.pcap >= pcap && v.tcap >= tcap && (v.pend_global || !need_global)) return &v;
  return nullptr;
}

// lane-engine table
struct LaneVariant { int model; int bd; uint32_t lpcap; kernel_fn fn; kernel_fn fn_rec; size_t smem_per_block; subseq_fn fn_sub; };
template <class MODEL, int BD, int LPCAP>
static LaneVariant make_lane_variant() {
  using M = LaneMachine<MODEL, BD, LPCAP>;
  return LaneVariant{MODEL::ID, BD, (uint32_t)LPCAP, fuzz_lane_kernel<MODEL, BD, LPCAP>, fuzz_lane_kernel<MODEL, BD, LPCAP, true>,
                     (size_t)M::WORDS * BD * sizeof(uint32_t), fuzz_lane_subseq_kernel<MODEL, BD, LPCAP>};
}
static const LaneVariant* pick_lane_variant(const demi_handle* h);

// ---------------------------------------------------------------- lifecycle
#ifndef DEMI_BUILD_ID
#define DEMI_BUILD_ID "unknown"
#endif
#ifndef DEMI_K1_ID
#define DEMI_K1_ID "unknown"
#endif
extern "C" const char* demi_version(void) { return "demi_b200 0.2 (sm_100a) build " DEMI_BUILD_ID " k1 " DEMI_K1_ID; }

extern "C" const char* demi_last_error(const demi_handle* h) {
  return h ? h->err.c_str() : g_create_error.c_str();
}

extern "C" int32_t demi_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

extern "C" int32_t demi_create(const demi_config* cfg, demi_handle** out) {
  if (!cfg || !out) return fail(nullptr, DEMI_ERR_INVALID, "demi_create: null argument");
  *out = nullptr;
  if (cfg->model != DEMI_MODEL_PINGPONG3 && cfg->model != DEMI_MODEL_RAFT5 && cfg->model != DEMI_MODEL_BCAST32 &&
      cfg->model != DEMI_MODEL_IR)
    return fail(nullptr, DEMI_ERR_INVALID, "demi_create: unknown model %d", cfg->model);
  if (cfg->strategy != DEMI_RS_FULLY_RANDOM && cfg->strategy != DEMI_RS_SRC_DST_FIFO)
    return fail(nullptr, DEMI_ERR_INVALID, "demi_create: unknown randomization strategy %d", cfg->strategy);
  int n = demi_device_count();
  if (n <= 0) return fail(nullptr, DEMI_ERR_NO_DEVICE, "demi_create: no CUDA device (this engine has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= n)
    return fail(nullptr, DEMI_ERR_INVALID, "demi_create: device %d out of range (%d devices)", cfg->device, n);
  demi_handle* h = new demi_handle();
  h->cfg = *cfg;
  cudaError_t e = cudaSetDevice(cfg->device);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, cfg->device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
  if (e == cudaSuccess) e = cudaMalloc(&h->counters_dev, 4 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&h->rec_counts_dev, 4 * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc(&h->ovf_count, sizeof(uint32_t));
  if (getenv("DEMI_DISABLE_LANE_ENGINE")) h->use_lane_engine = 0;
  if (const char* e = getenv("DEMI_LANE_PENDING_CAP")) h->lane_pending_cap = (uint32_t)atoi(e);   // tests: make the lane engine defer early
  if (e != cudaSuccess) {
    fail(nullptr, DEMI_ERR_CUDA, "demi_create: %s", cudaGetErrorString(e));
    demi_destroy(h);                       // frees whatever was created before the failure
    return DEMI_ERR_CUDA;
  }
  *out = h;
  return DEMI_OK;
}

extern "C" void demi_destroy(demi_handle* h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  cudaFree(h->ext_dev); cudaFree(h->results_dev); cudaFree(h->node_scratch); cudaFree(h->pend_scratch);
  cudaFree(h->counters_dev); cudaFree(h->rec_counts_dev); cudaFree(h->prov_scratch);
  for (void* b : h->dpor_buf) cudaFree(b);
  cudaFree(h->ext_sends_dev); cudaFree(h->lane_pend); cudaFree(h->ovf_list); cudaFree(h->ovf_count); cudaFree(h->fifo_scratch);
  demi_replay_free(h);
  demi_frontier_free(h);
  demi_comm_free(h);
  cudaFree(h->ir_blob_dev); cudaFree(h->trace_rec); cudaFree(h->subseq_buf);
  cudaFree(h->dedup.keys); cudaFree(h->dedup.vals); cudaFree(h->dedup.keep); cudaFree(h->dedup.counts);
  if (h->pinned) cudaFreeHost(h->pinned);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  delete h;
}

// demi_load_model: validate, keep the name table on the host, put programs + initial states on the device
extern "C" int32_t demi_load_model(demi_handle* h, const void* model_blob, size_t size) {
  if (!h) return DEMI_ERR_INVALID;
  if (h->cfg.model != DEMI_MODEL_IR) return fail(h, DEMI_ERR_STATE, "demi_load_model: the handle was created for built-in model %d", h->cfg.model);
  const uint32_t* w = (const uint32_t*)model_blob;
  if (!w || size < DEMI_IR_HEADER_WORDS * 4 || w[0] != DEMI_IR_MAGIC) return fail(h, DEMI_ERR_INVALID, "demi_load_model: not a model blob");
  if (w[1] != DEMI_IR_VERSION) return fail(h, DEMI_ERR_INVALID, "demi_load_model: version %u, this library reads %u", w[1], DEMI_IR_VERSION);
  const uint32_t na = w[2], sw = w[3], nt = w[4], rl = w[5], il = w[6], nb = w[9];
  if (na < 1 || na > DEMI_IR_ACTORS || sw < 1 || sw > DEMI_IR_STATE_WORDS || rl > DEMI_IR_MAX_CODE || il > DEMI_IR_MAX_CODE || w[8] > DEMI_IR_OUTBOX || nt > 256)
    return fail(h, DEMI_ERR_INVALID, "demi_load_model: %u actors x %u words, %u + %u instructions, fan-out %u exceed the limits of demi_model_ir.h", na, sw, rl, il, w[8]);
  const size_t words = (size_t)DEMI_IR_HEADER_WORDS + rl + il + (size_t)na * sw;
  if (size < words * 4 + nb) return fail(h, DEMI_ERR_INVALID, "demi_load_model: blob truncated (%zu of %zu bytes)", size, words * 4 + nb);
  // every operand is a register number < 16 by construction; jump targets and opcodes are checked here
  for (int prog = 0; prog < 2; prog++) {
    const uint32_t* code = w + DEMI_IR_HEADER_WORDS + (prog ? rl : 0); const uint32_t len = prog ? il : rl;
    for (uint32_t pc = 0; pc < len; pc++) {
      const uint32_t op = code[pc] & 0xFF;
      if (op > DEMI_IR_RET) return fail(h, DEMI_ERR_INVALID, "demi_load_model: unknown opcode %u at %u", op, pc);
      if (op == DEMI_IR_LDI || (op >= DEMI_IR_JMP && op <= DEMI_IR_JGE)) {
        if (pc + 1 >= len) return fail(h, DEMI_ERR_INVALID, "demi_load_model: instruction at %u lacks its immediate", pc);
        if (op != DEMI_IR_LDI && code[pc + 1] > len) return fail(h, DEMI_ERR_INVALID, "demi_load_model: jump at %u leaves the program", pc);
        pc++;
      }
    }
  }
  std::vector<std::string> names;
  const char* nm = (const char*)(w + words); size_t off = 0;
  while (off < nb && names.size() < (size_t)na + nt) { const size_t l = strnlen(nm + off, nb - off); names.emplace_back(nm + off, l); off += l + 1; }
  if (names.size() != (size_t)na + nt) return fail(h, DEMI_ERR_INVALID, "demi_load_model: %zu names for %u actors + %u message types", names.size(), na, nt);
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  cudaFree(h->ir_blob_dev); h->ir_blob_dev = nullptr; h->ir_loaded = false;
  CUDA_TRY(h, cudaMalloc(&h->ir_blob_dev, words * 4));
  CUDA_TRY(h, cudaMemcpy(h->ir_blob_dev, w, words * 4, cudaMemcpyHostToDevice));
  h->ir_dev.recv = h->ir_blob_dev + DEMI_IR_HEADER_WORDS; h->ir_dev.inv = h->ir_dev.recv + rl; h->ir_dev.init = h->ir_dev.inv + il;
  h->ir_dev.recv_len = rl; h->ir_dev.inv_len = il; h->ir_dev.n_actors = na; h->ir_dev.state_words = sw;
  h->ir_ext_mask = w[7]; h->ir_fanout = w[8]; h->ir_n_actors = na; h->ir_n_types = nt;
  h->names = names;
  h->ir_loaded = true;
  return DEMI_OK;
}
extern "C" int32_t demi_actor_index(const demi_handle* h, const char* name) {
  if (!h || !name) return -1;
  const int na = demi_model_actors(h);
  if (h->cfg.model == DEMI_MODEL_IR) { for (int i = 0; i < na; i++) if (h->names[i] == name) return i; return -1; }
  char* end = nullptr; const long v = strtol(name, &end, 10);
  return (*name && !*end && v >= 0 && v < na) ? (int32_t)v : -1;
}
extern "C" const char* demi_actor_name(const demi_handle* h, uint32_t index) {
  if (!h || (int)index >= demi_model_actors(h)) return nullptr;
  if (h->cfg.model == DEMI_MODEL_IR) return h->names[index].c_str();
  static const char* digits[32] = {"0","1","2","3","4","5","6","7","8","9","10","11","12","13","14","15","16","17","18","19","20",
                                   "21","22","23","24","25","26","27","28","29","30","31"};
  return digits[index];
}

extern "C" int32_t demi_set_externals(demi_handle* h, const demi_ext_event* ev, uint32_t n) {
  if (!h) return DEMI_ERR_INVALID;
  if (!ev && n) return fail(h, DEMI_ERR_INVALID, "demi_set_externals: null events");
  { int32_t mrc = demi_need_model(h); if (mrc != DEMI_OK) return mrc; }
  const int n_actors = demi_model_actors(h);
  uint32_t sends = 0;
  for (uint32_t i = 0; i < n; i++) {
    const demi_ext_event& e = ev[i];
    if (e.kind < DEMI_EXT_START || e.kind > DEMI_EXT_HARD_KILL)
      return fail(h, DEMI_ERR_INVALID, "demi_set_externals: event %u has unknown kind %u", i, e.kind);
    bool needs_a = e.kind != DEMI_EXT_WAIT_QUIESCENCE;
    bool needs_b = e.kind == DEMI_EXT_PARTITION || e.kind == DEMI_EXT_UNPARTITION;
    if ((needs_a && e.a >= n_actors) || (needs_b && e.b >= n_actors))
      return fail(h, DEMI_ERR_INVALID, "demi_set_externals: event %u names an unknown actor", i);
    // MessageTypes.sanityCheckTrace (ExternalEvents.scala:138-149): no two consecutive WaitQuiescence
    if (e.kind == DEMI_EXT_WAIT_QUIESCENCE && i > 0 && ev[i - 1].kind == DEMI_EXT_WAIT_QUIESCENCE)
      return fail(h, DEMI_ERR_INVALID, "demi_set_externals: consecutive WaitQuiescence at %u", i);
    if (e.kind == DEMI_EXT_SEND) sends++;
  }
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  cudaFree(h->ext_dev); h->ext_dev = nullptr;
  h->ext_host.assign(ev, ev + n);
  h->n_ext_sends = sends;
  if (n) {
    CUDA_TRY(h, cudaMalloc(&h->ext_dev, n * sizeof(demi_ext_event)));
    CUDA_TRY(h, cudaMemcpy(h->ext_dev, ev, n * sizeof(demi_ext_event), cudaMemcpyHostToDevice));
  }
  // lane-engine side tables: the Send events in order; whether two Sends are
  // identical (they would share a DepTracker Unique under the root)
  std::vector<uint4> sv;
  h->has_partitions = false; h->ext_sends_distinct = true; h->has_hard_kill = false;
  for (uint32_t i = 0; i < n; i++) {
    const demi_ext_event& e = ev[i];
    if (e.kind == DEMI_EXT_PARTITION || e.kind == DEMI_EXT_UNPARTITION) h->has_partitions = true;
    if (e.kind == DEMI_EXT_HARD_KILL) h->has_hard_kill = true;
    if (e.kind != DEMI_EXT_SEND) continue;
    uint4 m = make_uint4(DEMI_DEADLETTERS | ((uint32_t)e.a << 8) | ((uint32_t)e.type << 16) |
                         ((uint32_t)DEMI_MF_EXTERNAL << 24), e.p0, e.p1, 0u);
    for (const uint4& o : sv) if (o.x == m.x && o.y == m.y && o.z == m.z) h->ext_sends_distinct = false;
    sv.push_back(m);
  }
  cudaFree(h->ext_sends_dev); h->ext_sends_dev = nullptr;
  if (!sv.empty()) {
    CUDA_TRY(h, cudaMalloc(&h->ext_sends_dev, sv.size() * sizeof(uint4)));
    CUDA_TRY(h, cudaMemcpy(h->ext_sends_dev, sv.data(), sv.size() * sizeof(uint4), cudaMemcpyHostToDevice));
  }
  return DEMI_OK;
}

extern "C" int32_t demi_set_user_filter(demi_handle* h, const demi_filter_rule* rules, uint32_t n) {
  if (!h) return DEMI_ERR_INVALID;
  if (n > DEMI_MAX_FILTER_RULES || (!rules && n)) return fail(h, DEMI_ERR_INVALID, "demi_set_user_filter: at most %d rules", DEMI_MAX_FILTER_RULES);
  h->filter.assign(rules, rules + n);
  return DEMI_OK;
}

static const LaneVariant* pick_lane_variant(const demi_handle* h) {
  static const std::vector<LaneVariant> v = {
#ifndef DEMI_K1_BD_RAFT5
#define DEMI_K1_BD_RAFT5 256
#endif
    make_lane_variant<Raft5, DEMI_K1_BD_RAFT5, DEMI_K1_LPCAP_RAFT5>(),
    make_lane_variant<PingPong3, 256, 128>(),
    make_lane_variant<Bcast32, 128, 8192>(),
  };
  if (!h->use_lane_engine || h->cfg.blocked_mask || !h->ext_sends_distinct || h->cfg.strategy != DEMI_RS_FULLY_RANDOM ||
      h->has_hard_kill || !h->filter.empty()) return nullptr;          // actor termination and user filters: the general engine
  for (const LaneVariant& lv : v) if (lv.model == h->cfg.model) return &lv;
  return nullptr;
}

// ------------------------------------------------------------------- launch
struct LaunchPlan { const Variant* v; int grid; size_t smem; KernelArgs args; };

static int32_t ensure(demi_handle* h, void** p, size_t* cap, size_t need) {
  if (*cap >= need) return DEMI_OK;
  cudaFree(*p); *p = nullptr; *cap = 0;
  CUDA_TRY(h, cudaMalloc(p, need));
  *cap = need;
  return DEMI_OK;
}

static int32_t plan_launch(demi_handle* h, const demi_fuzz_params* p, bool record, LaunchPlan* plan) {
  if (!p) return fail(h, DEMI_ERR_INVALID, "null params");
  if (h->ext_host.empty()) return fail(h, DEMI_ERR_STATE, "demi_set_externals has not been called");
  if (p->n_prefixes > 0xFFFFFFFFull) return fail(h, DEMI_ERR_INVALID, "n_prefixes > 2^32-1 per call");
  { int32_t mrc = demi_need_model(h); if (mrc != DEMI_OK) return mrc; }
  const uint32_t pcap = demi_pending_cap(demi_model_key(h), p->max_messages, h->n_ext_sends);
  const uint32_t tcap = demi_tosend_cap(h->n_ext_sends);
  const bool fifo = h->cfg.strategy == DEMI_RS_SRC_DST_FIFO;          // SrcDstFIFO lives in the HBM-pending variants
  const Variant* v = pick_variant(h->cfg.model, pcap, tcap, record, fifo);
  if (!v) return fail(h, DEMI_ERR_CAPACITY, "no kernel variant for pending_cap=%u tosend_cap=%u", pcap, tcap);
  const size_t smem = v->smem_per_warp * WARPS;
  // the attribute and the occupancy of a variant are fixed per device: asked once, not on every launch
  int blocks_per_sm = 0;
  {
    auto it = h->occupancy.find((const void*)v->fn);
    if (it == h->occupancy.end()) {
      CUDA_TRY(h, cudaFuncSetAttribute(v->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, v->fn, WARPS * 32, smem));
      h->occupancy[(const void*)v->fn] = blocks_per_sm;
    } else blocks_per_sm = it->second;
  }
  if (blocks_per_sm < 1) return fail(h, DEMI_ERR_CAPACITY, "kernel variant does not fit on an SM (smem %zu)", smem);
  uint64_t want = (p->n_prefixes + WARPS - 1) / WARPS;
  uint64_t full = (uint64_t)h->sm_count * (uint64_t)blocks_per_sm;
  int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>(want, full));
  const uint64_t total_warps = (uint64_t)grid * WARPS;
  const uint32_t node_cap = demi_node_cap(pcap);

  int32_t rc;
  if ((rc = ensure(h, (void**)&h->node_scratch, &h->node_scratch_bytes,
                   total_warps * node_cap * sizeof(uint4))) != DEMI_OK) return rc;
  if (v->pend_global)
    if ((rc = ensure(h, (void**)&h->pend_scratch, &h->pend_scratch_bytes,
                     total_warps * (uint64_t)v->pcap * sizeof(uint4))) != DEMI_OK) return rc;

  KernelArgs a{};
  a.model_flags = h->cfg.model_flags;
  a.blocked_mask = h->cfg.blocked_mask;
  a.ignore_timers = h->cfg.ignore_timers;
  a.max_messages = p->max_messages < 0 ? INT_MAX : p->max_messages;   // maxMessages = Int.MaxValue (RandomScheduler.scala:54)
  a.interval = p->invariant_check_interval;
  a.looking_for = p->looking_for;
  a.seed_base = p->seed_base;
  a.n_prefixes = p->n_prefixes;
  a.fuzz_flags = p->flags;
  a.strategy = h->cfg.strategy;
  if (fifo) {
    if ((rc = ensure(h, (void**)&h->fifo_scratch, &h->fifo_scratch_bytes,
                     total_warps * (uint64_t)(v->pcap / 2 + 3 * FIFO_PAIRS) * sizeof(uint16_t))) != DEMI_OK) return rc;
    a.fifo_scratch = h->fifo_scratch;
  }
  if (fifo && (h->has_hard_kill || !h->filter.empty()))
    return fail(h, DEMI_ERR_INVALID, "HardKill and userDefinedFilter are offered for FullyRandom only");
  a.n_filter = (uint32_t)h->filter.size();
  for (uint32_t i = 0; i < a.n_filter; i++) a.filter[i] = make_uint4(h->filter[i].src_mask, h->filter[i].dst_mask, h->filter[i].type_mask, h->filter[i].flags);
  a.ext = h->ext_dev;
  a.n_ext = (uint32_t)h->ext_host.size();
  a.node_cap = node_cap;
  a.pending_cap = pcap;
  a.tosend_cap = tcap;
  a.node_scratch = h->node_scratch;
  a.pend_scratch = h->pend_scratch;
  a.sum_steps = h->counters_dev;
  a.n_violations = h->counters_dev + 1;
  plan->v = v; plan->grid = grid; plan->smem = smem; plan->args = a;
  return DEMI_OK;
}

static int32_t launch_fuzz(demi_handle* h, const demi_fuzz_params* p, void* out_dev, void* stream, bool reset_counters);

extern "C" int32_t demi_fuzz_batch_dev(demi_handle* h, const demi_fuzz_params* p, void* out_dev, void* stream) {
  return launch_fuzz(h, p, out_dev, stream, true);
}

// One launch of the lane engine over `n_items` work items; what it defers is appended to h->ovf_list / h->ovf_count.
static int32_t launch_lane(demi_handle* h, const LaneVariant* lv, kernel_fn lfn, const KernelArgs& base, uint64_t n_items, cudaStream_t s) {
  const size_t lsmem = lv->smem_per_block;
  int bps = 0;
  {
    auto it = h->occupancy.find((const void*)lfn);
    if (it == h->occupancy.end()) {
      CUDA_TRY(h, cudaFuncSetAttribute(lfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsmem));
      CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, lfn, lv->bd, lsmem));
      h->occupancy[(const void*)lfn] = bps;
    } else bps = it->second;
  }
  if (bps < 1) return fail(h, DEMI_ERR_CAPACITY, "lane kernel does not fit on an SM");
  uint64_t want = (n_items + lv->bd - 1) / lv->bd;
  int lgrid = (int)std::max<uint64_t>(1, std::min<uint64_t>(want, (uint64_t)h->sm_count * bps));
  const uint64_t lwarps = (uint64_t)lgrid * (lv->bd / 32);
  int32_t rc2;
  if ((rc2 = ensure(h, (void**)&h->lane_pend, &h->lane_pend_bytes, lwarps * lv->lpcap * 32 * sizeof(uint4))) != DEMI_OK) return rc2;
  if ((rc2 = ensure(h, (void**)&h->ovf_list, &h->ovf_list_bytes, std::max<size_t>(n_items * sizeof(uint32_t), 64))) != DEMI_OK) return rc2;
  CUDA_TRY(h, cudaMemsetAsync(h->ovf_count, 0, sizeof(uint32_t), s));
  KernelArgs la = base;
  la.lane_pend = h->lane_pend;
  la.ext_sends = h->ext_sends_dev;
  la.has_partitions = h->has_partitions ? 1u : 0u;
  la.ovf_list = h->ovf_list; la.ovf_count = h->ovf_count;
  if (h->lane_pending_cap) la.pending_cap = std::min(la.pending_cap, h->lane_pending_cap);     // deferring is always exact
  lfn<<<lgrid, lv->bd, lsmem, s>>>(la);
  CUDA_TRY(h, cudaGetLastError());
  h->perf.kernel_launches++;
  return DEMI_OK;
}

static int32_t launch_fuzz(demi_handle* h, const demi_fuzz_params* p, void* out_dev, void* stream, bool reset_counters) {
  if (!h) return DEMI_ERR_INVALID;
  if (!out_dev) return fail(h, DEMI_ERR_INVALID, "demi_fuzz_batch_dev: null output");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  LaunchPlan plan;
  int32_t rc = plan_launch(h, p, false, &plan);
  if (rc != DEMI_OK) return rc;
  if (p->n_prefixes == 0) return DEMI_OK;
  cudaStream_t s = (cudaStream_t)stream;
  plan.args.results = (demi_fuzz_result*)out_dev;
  if (reset_counters) {
    CUDA_TRY(h, cudaMemsetAsync(h->counters_dev, 0, 4 * sizeof(unsigned long long), s));
    h->perf.kernel_launches = 0;
    h->perf.prefixes = 0;
  }
  const LaneVariant* lv = pick_lane_variant(h);
  if (lv) {
    // K1-lane handles every prefix it can prove exact; the rest are deferred to the warp engine
    int32_t rc2 = launch_lane(h, lv, lv->fn, plan.args, p->n_prefixes, s);
    if (rc2 != DEMI_OK) return rc2;
    plan.args.index_list = h->ovf_list;
    plan.args.index_count = h->ovf_count;
  }
  if (h->cfg.model == DEMI_MODEL_IR) CUDA_TRY(h, ir_bind(h->ir_dev, s));
  plan.v->fn<<<plan.grid, WARPS * 32, plan.smem, s>>>(plan.args);
  CUDA_TRY(h, cudaGetLastError());
  h->perf.kernel_launches++;
  h->perf.prefixes += p->n_prefixes;
  return DEMI_OK;
}

extern "C" int32_t demi_fuzz_batch(demi_handle* h, const demi_fuzz_params* p, demi_fuzz_result* out_host) {
  if (!h) return DEMI_ERR_INVALID;
  if (!out_host) return fail(h, DEMI_ERR_INVALID, "demi_fuzz_batch: null output");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  if (!p) return fail(h, DEMI_ERR_INVALID, "null params");
  const size_t bytes = (size_t)p->n_prefixes * sizeof(demi_fuzz_result);
  int32_t rc = ensure(h, (void**)&h->results_dev, &h->results_cap, std::max<size_t>(bytes, 32));
  if (rc != DEMI_OK) return rc;
  // Pipeline: the batch is cut into chunks; chunk i's records travel to the host on the copy
  // stream while chunk i+1 is being explored.
  const uint64_t CHUNK = 2u << 20;
  const uint64_t n = p->n_prefixes;
  const uint64_t n_chunks = n <= 2 * CHUNK ? 1 : (n + CHUNK - 1) / CHUNK;
  const uint64_t per = n_chunks ? (n + n_chunks - 1) / n_chunks : 0;
  CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream));
  if (n == 0) { rc = launch_fuzz(h, p, h->results_dev, h->stream, true); if (rc != DEMI_OK) return rc; }
  std::vector<cudaEvent_t> evs;
  for (uint64_t c = 0, off = 0; off < n; c++, off += per) {
    demi_fuzz_params q = *p;
    q.seed_base = p->seed_base + (int64_t)off;
    q.n_prefixes = std::min<uint64_t>(per, n - off);
    rc = launch_fuzz(h, &q, h->results_dev + off, h->stream, c == 0);
    if (rc != DEMI_OK) break;
    cudaEvent_t ev;
    cudaError_t ce = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (ce == cudaSuccess) {
      evs.push_back(ev);
      ce = cudaEventRecord(ev, h->stream);
      if (ce == cudaSuccess) ce = cudaStreamWaitEvent(h->copy_stream, ev, 0);
      if (ce == cudaSuccess) ce = cudaMemcpyAsync(out_host + off, h->results_dev + off, q.n_prefixes * sizeof(demi_fuzz_result),
                                                  cudaMemcpyDeviceToHost, h->copy_stream);
    }
    if (ce != cudaSuccess) { rc = fail(h, DEMI_ERR_CUDA, "demi_fuzz_batch: %s", cudaGetErrorString(ce)); break; }   // events freed below
  }
  cudaError_t e = cudaEventRecord(h->ev1, h->stream);
  unsigned long long cnt[3] = {0, 0, 0};
  if (e == cudaSuccess) e = cudaMemcpyAsync(cnt, h->counters_dev, sizeof(cnt), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->copy_stream);
  for (cudaEvent_t ev : evs) cudaEventDestroy(ev);
  if (rc != DEMI_OK) return rc;
  if (e != cudaSuccess) return fail(h, DEMI_ERR_CUDA, "demi_fuzz_batch: %s", cudaGetErrorString(e));
  float ms = 0;
  CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->perf.kernel_ms = ms;
  h->perf.deliveries = cnt[0];
  h->perf.violations = cnt[1];
  h->perf.deferred = (uint32_t)std::min<unsigned long long>(cnt[2], 0xFFFFFFFFull);      // deferred to the general engine
  h->perf.d2h_bytes = bytes + sizeof(cnt);
  h->perf.h2d_bytes = 0;
  return DEMI_OK;
}

// Counts from the last *_dev batch launched on `stream` (waits for it).
extern "C" int32_t demi_fuzz_summary_dev(demi_handle* h, const void* /*results_dev*/, uint64_t /*n*/,
                                         void* stream, uint64_t* n_violations, uint64_t* sum_steps) {
  if (!h) return DEMI_ERR_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  unsigned long long c[3] = {0, 0, 0};
  CUDA_TRY(h, cudaMemcpyAsync(c, h->counters_dev, sizeof(c), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CUDA_TRY(h, cudaStreamSynchronize((cudaStream_t)stream));
  if (sum_steps) *sum_steps = c[0];
  if (n_violations) *n_violations = c[1];
  h->perf.deliveries = c[0];
  h->perf.violations = c[1];
  h->perf.deferred = (uint32_t)std::min<unsigned long long>(c[2], 0xFFFFFFFFull);
  return DEMI_OK;
}

extern "C" int32_t demi_fuzz_trace(demi_handle* h, const demi_fuzz_params* p, int64_t seed,
                                   demi_event* events, uint32_t cap_events, uint32_t* n_events,
                                   uint16_t* dep_parent, uint32_t cap_nodes, uint32_t* n_nodes,
                                   demi_fuzz_result* result) {
  if (!h) return DEMI_ERR_INVALID;
  if (!p) return fail(h, DEMI_ERR_INVALID, "null params");
  if (!events || !cap_events) return fail(h, DEMI_ERR_INVALID, "demi_fuzz_trace: events buffer required");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  demi_fuzz_params q = *p;
  q.seed_base = seed; q.n_prefixes = 1;
  LaunchPlan plan;
  int32_t rc = plan_launch(h, &q, true, &plan);
  if (rc != DEMI_OK) return rc;
  const uint32_t cap_ev = std::max<uint32_t>(cap_events, 1), cap_n = std::max<uint32_t>(cap_nodes, 1);
  // one recording buffer, kept in the handle: events | parents | result
  const size_t o_par = (size_t)cap_ev * sizeof(demi_event), o_res = (o_par + (size_t)cap_n * 2 + 15) & ~(size_t)15;
  if ((rc = ensure(h, &h->trace_rec, &h->trace_rec_bytes, o_res + sizeof(demi_fuzz_result))) != DEMI_OK) return rc;
  demi_event* ev_dev = (demi_event*)h->trace_rec;
  uint16_t* par_dev = (uint16_t*)((unsigned char*)h->trace_rec + o_par);
  demi_fuzz_result* res_dev = (demi_fuzz_result*)((unsigned char*)h->trace_rec + o_res);
  plan.args.results = res_dev;
  plan.args.rec_events = ev_dev; plan.args.rec_cap = cap_events;
  plan.args.rec_counts = h->rec_counts_dev;
  plan.args.rec_parent = dep_parent ? par_dev : nullptr; plan.args.rec_parent_cap = cap_nodes;
  CUDA_TRY(h, cudaMemsetAsync(h->counters_dev, 0, 4 * sizeof(unsigned long long), h->stream));
  if (h->cfg.model == DEMI_MODEL_IR) ir_bind(h->ir_dev, h->stream);
  plan.v->fn<<<1, WARPS * 32, plan.smem, h->stream>>>(plan.args);
  cudaError_t e = cudaGetLastError();
  demi_fuzz_result r{}; uint32_t counts[4] = {0, 0, 0, 0};
  if (e == cudaSuccess) e = cudaMemcpyAsync(&r, res_dev, sizeof(r), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(counts, h->rec_counts_dev, sizeof(counts), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e == cudaSuccess && r.status == 0) {
    e = cudaMemcpy(events, ev_dev, (size_t)std::min(counts[0], cap_events) * sizeof(demi_event), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && dep_parent)
      e = cudaMemcpy(dep_parent, par_dev, (size_t)std::min(counts[1], cap_nodes) * sizeof(uint16_t), cudaMemcpyDeviceToHost);
  }
  if (e != cudaSuccess) return fail(h, DEMI_ERR_CUDA, "demi_fuzz_trace: %s", cudaGetErrorString(e));
  if (n_events) *n_events = counts[0];
  if (n_nodes) *n_nodes = counts[1];
  if (result) *result = r;
  if (r.status) return fail(h, DEMI_ERR_CAPACITY, "demi_fuzz_trace: prefix status %u", (unsigned)r.status);
  return DEMI_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Subsequence batches: RandomScheduler.test of many subsequences of the program in one launch (subseq_kernel.cuh)

// program_of(mask) (include/demi_b200.h) as a mask: adjacent WaitQuiescence collapsed.  Returns n_eff (last selected
// index + 1) and the number of Sends; 0 for an empty selection.
static uint32_t subseq_effective(const std::vector<demi_ext_event>& ext, const uint64_t* m, uint64_t* eff, uint32_t* sends) {
  uint32_t n_eff = 0, ns = 0; bool prev_wq = false;
  for (uint32_t j = 0; j < (uint32_t)ext.size(); j++) {
    if (!((m[j >> 6] >> (j & 63)) & 1ull)) continue;
    const bool wq = ext[j].kind == DEMI_EXT_WAIT_QUIESCENCE;
    if (wq && prev_wq) continue;
    prev_wq = wq;
    eff[j >> 6] |= 1ull << (j & 63);
    if (ext[j].kind == DEMI_EXT_SEND) ns++;
    n_eff = j + 1;
  }
  *sends = ns;
  return n_eff;
}

extern "C" int32_t demi_fuzz_subseq_batch(demi_handle* h, const demi_fuzz_params* p, const uint64_t* masks, uint32_t n_tests,
                                          uint32_t mask_words, uint32_t* first_hit, uint32_t* first_bad) {
  if (!h) return DEMI_ERR_INVALID;
  if (!p) return fail(h, DEMI_ERR_INVALID, "null params");
  if (!n_tests) return DEMI_OK;
  if (!masks || !first_hit || !first_bad) return fail(h, DEMI_ERR_INVALID, "demi_fuzz_subseq_batch: masks, first_hit and first_bad are required");
  if (h->ext_host.empty()) return fail(h, DEMI_ERR_STATE, "demi_set_externals has not been called");
  if (p->n_prefixes > 0xFFFFFFFFull) return fail(h, DEMI_ERR_INVALID, "n_prefixes > 2^32-1 per call");
  { int32_t mrc = demi_need_model(h); if (mrc != DEMI_OK) return mrc; }
  const uint32_t n_ext = (uint32_t)h->ext_host.size(), mw = mask_words, K = (uint32_t)p->n_prefixes;
  if (!mw || (uint64_t)mw * 64 < n_ext) return fail(h, DEMI_ERR_INVALID, "demi_fuzz_subseq_batch: %u mask words cannot hold %u externals", mw, n_ext);
  // the per-test side table: effective mask, n_eff, capacities of program_of(mask)
  std::vector<uint64_t> eff((size_t)n_tests * mw, 0);
  std::vector<uint32_t> n_eff(n_tests), sends(n_tests);
  for (uint32_t t = 0; t < n_tests; t++) {
    const uint64_t* m = masks + (size_t)t * mw;
    for (uint32_t w = 0; w < mw; w++) {
      const uint64_t valid = (uint64_t)w * 64 + 64 <= n_ext ? ~0ull : (uint64_t)w * 64 >= n_ext ? 0ull : ((1ull << (n_ext - w * 64)) - 1);
      if (m[w] & ~valid) return fail(h, DEMI_ERR_INVALID, "demi_fuzz_subseq_batch: test %u selects an external beyond the %u of the program", t, n_ext);
    }
    n_eff[t] = subseq_effective(h->ext_host, m, &eff[(size_t)t * mw], &sends[t]);
    if (!n_eff[t]) return fail(h, DEMI_ERR_INVALID, "demi_fuzz_subseq_batch: test %u selects no external", t);
  }
  if (K == 0) { std::fill(first_hit, first_hit + n_tests, 0u); std::fill(first_bad, first_bad + n_tests, 0u); return DEMI_OK; }
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  // the kernel variant and the scratch are those of the whole program: its capacities bound every subsequence's
  const uint32_t per_chunk = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(n_tests, 0xFFFFFFFFull / K));
  demi_fuzz_params q = *p;
  q.n_prefixes = (uint64_t)per_chunk * K;
  LaunchPlan plan;
  int32_t rc = plan_launch(h, &q, false, &plan);
  if (rc != DEMI_OK) return rc;
  if (!plan.v->sub) return fail(h, DEMI_ERR_STATE, "demi_fuzz_subseq_batch: no subsequence kernel for the variant");
  const LaneVariant* lv = pick_lane_variant(h);
  std::vector<KernelArgs> ta(n_tests), tl(lv ? n_tests : 0);
  for (uint32_t t = 0; t < n_tests; t++) {
    KernelArgs a = plan.args;
    a.n_ext = n_eff[t];
    a.pending_cap = demi_pending_cap(demi_model_key(h), p->max_messages, sends[t]);
    a.tosend_cap = demi_tosend_cap(sends[t]);
    a.node_cap = demi_node_cap(a.pending_cap);
    a.results = nullptr; a.sum_steps = nullptr; a.n_violations = nullptr;
    ta[t] = a;
    if (lv) {
      a.ext_sends = h->ext_sends_dev;
      a.has_partitions = h->has_partitions ? 1u : 0u;       // of the whole program: a fast-path flag only
      if (h->lane_pending_cap) a.pending_cap = std::min(a.pending_cap, h->lane_pending_cap);
      tl[t] = a;
    }
  }
  // one device buffer: warp args | lane args | masks | first_hit | first_bad
  auto al = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t b_ta = al(ta.size() * sizeof(KernelArgs)), b_tl = al(tl.size() * sizeof(KernelArgs)),
               b_m = al(eff.size() * sizeof(uint64_t)), b_v = al((size_t)n_tests * sizeof(uint32_t));
  if ((rc = ensure(h, &h->subseq_buf, &h->subseq_buf_bytes, b_ta + b_tl + b_m + 2 * b_v)) != DEMI_OK) return rc;
  unsigned char* d = (unsigned char*)h->subseq_buf;
  KernelArgs* d_ta = (KernelArgs*)d; KernelArgs* d_tl = (KernelArgs*)(d + b_ta);
  uint64_t* d_m = (uint64_t*)(d + b_ta + b_tl);
  uint32_t* d_fh = (uint32_t*)(d + b_ta + b_tl + b_m); uint32_t* d_fb = (uint32_t*)(d + b_ta + b_tl + b_m + b_v);
  std::vector<unsigned char> stage(b_ta + b_tl + b_m + 2 * b_v, 0);
  memcpy(stage.data(), ta.data(), ta.size() * sizeof(KernelArgs));
  if (lv) memcpy(stage.data() + b_ta, tl.data(), tl.size() * sizeof(KernelArgs));
  memcpy(stage.data() + b_ta + b_tl, eff.data(), eff.size() * sizeof(uint64_t));
  std::fill((uint32_t*)(stage.data() + b_ta + b_tl + b_m), (uint32_t*)(stage.data() + b_ta + b_tl + b_m) + n_tests, K);
  std::fill((uint32_t*)(stage.data() + b_ta + b_tl + b_m + b_v), (uint32_t*)(stage.data() + b_ta + b_tl + b_m + b_v) + n_tests, K);
  cudaStream_t s = h->stream;
  CUDA_TRY(h, cudaMemcpyAsync(d, stage.data(), stage.size(), cudaMemcpyHostToDevice, s));
  CUDA_TRY(h, cudaMemsetAsync(h->counters_dev, 0, 4 * sizeof(unsigned long long), s));
  CUDA_TRY(h, cudaEventRecord(h->ev0, s));
  h->perf.kernel_launches = 0;
  if (h->cfg.model == DEMI_MODEL_IR) CUDA_TRY(h, ir_bind(h->ir_dev, s));
  for (uint32_t t0 = 0; t0 < n_tests; t0 += per_chunk) {
    const uint32_t nt = std::min(per_chunk, n_tests - t0);
    const uint64_t items = (uint64_t)nt * K;
    SubseqArgs sa{};
    sa.targs = d_ta + t0; sa.targs_lane = lv ? d_tl + t0 : nullptr;
    sa.masks = d_m + (size_t)t0 * mw; sa.mask_words = mw; sa.n_tests = nt;
    sa.n_items = items; sa.seed_base = p->seed_base;
    sa.first_hit = d_fh + t0; sa.first_bad = d_fb + t0;
    sa.counters = h->counters_dev;
    sa.node_scratch = h->node_scratch; sa.pend_scratch = h->pend_scratch; sa.fifo_scratch = plan.args.fifo_scratch;
    sa.node_stride = plan.args.node_cap;
    if (lv) {
      // K1-lane runs every item it can prove exact; the rest go to the warp engine, as in demi_fuzz_batch
      int bps = 0;
      auto it = h->occupancy.find((const void*)lv->fn_sub);
      if (it == h->occupancy.end()) {
        CUDA_TRY(h, cudaFuncSetAttribute(lv->fn_sub, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lv->smem_per_block));
        CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, lv->fn_sub, lv->bd, lv->smem_per_block));
        h->occupancy[(const void*)lv->fn_sub] = bps;
      } else bps = it->second;
      if (bps < 1) return fail(h, DEMI_ERR_CAPACITY, "lane kernel does not fit on an SM");
      const int lgrid = (int)std::max<uint64_t>(1, std::min<uint64_t>((items + lv->bd - 1) / lv->bd, (uint64_t)h->sm_count * bps));
      const uint64_t lwarps = (uint64_t)lgrid * (lv->bd / 32);
      if ((rc = ensure(h, (void**)&h->lane_pend, &h->lane_pend_bytes, lwarps * lv->lpcap * 32 * sizeof(uint4))) != DEMI_OK) return rc;
      if ((rc = ensure(h, (void**)&h->ovf_list, &h->ovf_list_bytes, std::max<size_t>(items * sizeof(uint32_t), 64))) != DEMI_OK) return rc;
      CUDA_TRY(h, cudaMemsetAsync(h->ovf_count, 0, sizeof(uint32_t), s));
      sa.lane_pend = h->lane_pend; sa.ovf_list = h->ovf_list; sa.ovf_count = h->ovf_count;
      lv->fn_sub<<<lgrid, lv->bd, lv->smem_per_block, s>>>(sa);
      CUDA_TRY(h, cudaGetLastError());
      h->perf.kernel_launches++;
      sa.index_list = h->ovf_list; sa.index_count = h->ovf_count;
      sa.ovf_list = nullptr; sa.ovf_count = nullptr;
    }
    {
      auto it = h->occupancy.find((const void*)plan.v->sub);
      if (it == h->occupancy.end()) {
        int bps = 0;
        CUDA_TRY(h, cudaFuncSetAttribute(plan.v->sub, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
        CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, plan.v->sub, WARPS * 32, plan.smem));
        if (bps < 1) return fail(h, DEMI_ERR_CAPACITY, "subsequence kernel does not fit on an SM (smem %zu)", plan.smem);
        h->occupancy[(const void*)plan.v->sub] = bps;
      }
    }
    // the warp grid (and the scratch behind it) was planned for per_chunk * K items
    plan.v->sub<<<plan.grid, WARPS * 32, plan.smem, s>>>(sa);
    CUDA_TRY(h, cudaGetLastError());
    h->perf.kernel_launches++;
  }
  CUDA_TRY(h, cudaEventRecord(h->ev1, s));
  unsigned long long cnt[4] = {0, 0, 0, 0};
  CUDA_TRY(h, cudaMemcpyAsync(first_hit, d_fh, (size_t)n_tests * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(h, cudaMemcpyAsync(first_bad, d_fb, (size_t)n_tests * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(h, cudaMemcpyAsync(cnt, h->counters_dev, sizeof(cnt), cudaMemcpyDeviceToHost, s));
  CUDA_TRY(h, cudaStreamSynchronize(s));
  // the test stopped at the lower of the two; the other one is "none"
  for (uint32_t t = 0; t < n_tests; t++) {
    if (first_hit[t] < first_bad[t]) first_bad[t] = K;
    else if (first_bad[t] < first_hit[t]) first_hit[t] = K;
  }
  float ms = 0;
  CUDA_TRY(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->perf.kernel_ms = ms;
  h->perf.prefixes = cnt[3];
  h->perf.deliveries = cnt[0];
  h->perf.violations = cnt[1];
  h->perf.deferred = (uint32_t)std::min<unsigned long long>(cnt[2], 0xFFFFFFFFull);
  h->perf.h2d_bytes = stage.size();
  h->perf.d2h_bytes = (size_t)n_tests * 8 + sizeof(cnt);
  return DEMI_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Provenance pruning (ProvenanceTracker, schedulers/Util.scala:267-376)
static int32_t launch_provenance(demi_handle* h, ProvArgs a, cudaStream_t s) {
  constexpr int PW = 4;
  const uint64_t want = ((uint64_t)a.n + PW - 1) / PW;
  const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>(want, (uint64_t)h->sm_count * 8));
  a.t_cap = a.mask_words * 64;
  a.scratch_stride = a.t_cap + 3 * a.par_stride;
  int32_t rc = ensure(h, (void**)&h->prov_scratch, &h->prov_scratch_bytes,
                      (uint64_t)grid * PW * a.scratch_stride * sizeof(uint32_t));
  if (rc != DEMI_OK) return rc;
  a.scratch = (uint32_t*)h->prov_scratch;
  provenance_kernel<PW><<<grid, PW * 32, 0, s>>>(a);
  CUDA_TRY(h, cudaGetLastError());
  h->perf.kernel_launches++;
  return DEMI_OK;
}

extern "C" int32_t demi_provenance(demi_handle* h, const demi_event* events, uint32_t n_events,
                                   const uint16_t* dep_parent, uint32_t n_nodes, uint32_t affected_mask,
                                   uint64_t* keep_mask, uint32_t mask_words, demi_provenance_out* out) {
  if (!h) return DEMI_ERR_INVALID;
  if (!events || !dep_parent || !keep_mask || !out || !mask_words || !n_nodes)
    return fail(h, DEMI_ERR_INVALID, "demi_provenance: events, dep_parent, keep_mask and out are required");
  if (n_nodes > 65536) return fail(h, DEMI_ERR_INVALID, "demi_provenance: node ids are 16-bit");
  { int32_t vrc = demi_check_events(h, "demi_provenance", events, n_events, n_nodes, DEMI_MAX_ACTORS); if (vrc != DEMI_OK) return vrc;
    vrc = demi_check_parents(h, "demi_provenance", dep_parent, n_nodes); if (vrc != DEMI_OK) return vrc; }
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  const size_t ev_b = (size_t)std::max(n_events, 1u) * sizeof(demi_event), par_b = (size_t)n_nodes * 2;
  const size_t keep_b = (size_t)mask_words * 8;
  unsigned char* buf = nullptr;                      // events | parents | counts | keep | out
  const size_t o_par = (ev_b + 15) & ~(size_t)15, o_cnt = (o_par + par_b + 15) & ~(size_t)15, o_keep = o_cnt + 16,
               o_out = o_keep + ((keep_b + 15) & ~(size_t)15), total = o_out + sizeof(demi_provenance_out);
  CUDA_TRY(h, cudaMalloc(&buf, total));
  const uint32_t counts[4] = {n_events, n_nodes, affected_mask, 0};
  cudaError_t e = cudaMemcpyAsync(buf, events, (size_t)n_events * sizeof(demi_event), cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(buf + o_par, dep_parent, par_b, cudaMemcpyHostToDevice, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(buf + o_cnt, counts, sizeof(counts), cudaMemcpyHostToDevice, h->stream);
  int32_t rc = DEMI_OK;
  if (e == cudaSuccess) {
    ProvArgs a{};
    a.events = (const demi_event*)buf; a.ev_stride = std::max(n_events, 1u);
    a.parent = (const uint16_t*)(buf + o_par); a.par_stride = n_nodes;
    a.counts = (const uint32_t*)(buf + o_cnt); a.results = nullptr;
    a.keep = (uint64_t*)(buf + o_keep); a.mask_words = mask_words;
    a.out = (demi_provenance_out*)(buf + o_out); a.n = 1;
    rc = launch_provenance(h, a, h->stream);
  }
  if (rc == DEMI_OK && e == cudaSuccess) e = cudaMemcpyAsync(keep_mask, buf + o_keep, keep_b, cudaMemcpyDeviceToHost, h->stream);
  if (rc == DEMI_OK && e == cudaSuccess) e = cudaMemcpyAsync(out, buf + o_out, sizeof(*out), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(buf);
  if (rc != DEMI_OK) return rc;
  if (e != cudaSuccess) return fail(h, DEMI_ERR_CUDA, "demi_provenance: %s", cudaGetErrorString(e));
  return DEMI_OK;
}

extern "C" int32_t demi_fuzz_provenance(demi_handle* h, const demi_fuzz_params* p, const uint32_t* prefix_index, uint32_t n,
                                        uint64_t* keep_masks, uint32_t mask_words, demi_provenance_out* out,
                                        demi_fuzz_result* results) {
  if (!h) return DEMI_ERR_INVALID;
  if (!p) return fail(h, DEMI_ERR_INVALID, "null params");
  if (!n) return DEMI_OK;
  if (!prefix_index || !keep_masks || !out || !mask_words)
    return fail(h, DEMI_ERR_INVALID, "demi_fuzz_provenance: prefix_index, keep_masks and out are required");
  if (p->max_messages < 0 || (uint64_t)p->max_messages + 2 > (uint64_t)mask_words * 64)
    return fail(h, DEMI_ERR_INVALID, "demi_fuzz_provenance: mask_words*64 must cover max_messages + 2 positions");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  demi_fuzz_params q = *p;
  q.n_prefixes = n;
  LaunchPlan plan;
  int32_t rc = plan_launch(h, &q, true, &plan);
  if (rc != DEMI_OK) return rc;
  // an execution records at most one MsgSend + one MsgEvent per message, plus the external markers
  const uint32_t node_cap = plan.args.node_cap;
  const uint32_t ev_cap = 2 * node_cap + 2 * plan.args.n_ext + 16;
  {
    // bound the per-slot recording buffers to ~4 GB per launch: larger requests run in chunks
    const size_t per_slot = (size_t)ev_cap * sizeof(demi_event) + (size_t)node_cap * 2 + 64 + (size_t)mask_words * 8;
    const uint32_t chunk = (uint32_t)std::max<size_t>(1, ((size_t)4 << 30) / per_slot);
    if (n > chunk) {
      for (uint32_t off = 0; off < n; off += chunk) {
        const uint32_t m = std::min(chunk, n - off);
        rc = demi_fuzz_provenance(h, p, prefix_index + off, m, keep_masks + (size_t)off * mask_words, mask_words, out + off,
                                  results ? results + off : nullptr);
        if (rc != DEMI_OK) return rc;
      }
      return DEMI_OK;
    }
  }
  const size_t b_ev = (size_t)n * ev_cap * sizeof(demi_event), b_par = (((size_t)n * node_cap * 2) + 15) & ~(size_t)15,
               b_cnt = (size_t)n * 16, b_res = (size_t)n * sizeof(demi_fuzz_result), b_idx = (((size_t)n * 4) + 15) & ~(size_t)15,
               b_keep = (size_t)n * mask_words * 8, b_out = (size_t)n * sizeof(demi_provenance_out);
  unsigned char* buf = nullptr;
  CUDA_TRY(h, cudaMalloc(&buf, b_ev + b_par + b_cnt + b_res + b_idx + 16 + b_keep + b_out));
  unsigned char* d_par = buf + b_ev; unsigned char* d_cnt = d_par + b_par; unsigned char* d_res = d_cnt + b_cnt;
  unsigned char* d_idx = d_res + b_res; unsigned char* d_n = d_idx + b_idx; unsigned char* d_keep = d_n + 16;
  unsigned char* d_out = d_keep + b_keep;
  cudaStream_t s = h->stream;
  cudaError_t e = cudaMemcpyAsync(d_idx, prefix_index, (size_t)n * 4, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_n, &n, 4, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_cnt, 0, b_cnt, s);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_res, 0xFF, b_res, s);
  if (e == cudaSuccess) {
    plan.args.results = (demi_fuzz_result*)d_res;
    plan.args.index_list = (const uint32_t*)d_idx; plan.args.index_count = (const uint32_t*)d_n;
    plan.args.rec_events = (demi_event*)buf; plan.args.rec_cap = ev_cap;
    plan.args.rec_counts = (uint32_t*)d_cnt;
    plan.args.rec_parent = (uint16_t*)d_par; plan.args.rec_parent_cap = node_cap;
    plan.args.sum_steps = nullptr; plan.args.n_violations = nullptr;
    cudaEvent_t t0, t1; cudaEventCreate(&t0); cudaEventCreate(&t1);
    cudaEventRecord(t0, s);
    if (h->cfg.model == DEMI_MODEL_IR) ir_bind(h->ir_dev, s);
    // the lane engine records every execution it can prove exact; the slots it defers go to the general engine
    const LaneVariant* lv = pick_lane_variant(h);
    if (lv) {
      rc = launch_lane(h, lv, lv->fn_rec, plan.args, n, s);
      plan.args.pos_list = h->ovf_list; plan.args.pos_count = h->ovf_count;
    }
    if (rc == DEMI_OK) {
      plan.v->fn<<<plan.grid, WARPS * 32, plan.smem, s>>>(plan.args);
      e = cudaGetLastError();
      h->perf.kernel_launches++;
    }
    if (rc == DEMI_OK && e == cudaSuccess) {
      ProvArgs a{};
      a.events = (const demi_event*)buf; a.ev_stride = ev_cap;
      a.parent = (const uint16_t*)d_par; a.par_stride = node_cap;
      a.counts = (const uint32_t*)d_cnt; a.results = (const demi_fuzz_result*)d_res;
      a.keep = (uint64_t*)d_keep; a.mask_words = mask_words; a.out = (demi_provenance_out*)d_out; a.n = n;
      rc = launch_provenance(h, a, s);
    }
    cudaEventRecord(t1, s);
    if (rc == DEMI_OK && e == cudaSuccess) e = cudaMemcpyAsync(keep_masks, d_keep, b_keep, cudaMemcpyDeviceToHost, s);
    if (rc == DEMI_OK && e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, b_out, cudaMemcpyDeviceToHost, s);
    if (rc == DEMI_OK && e == cudaSuccess && results) e = cudaMemcpyAsync(results, d_res, b_res, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    float ms = 0.f;
    if (e == cudaSuccess && cudaEventElapsedTime(&ms, t0, t1) == cudaSuccess) h->perf.kernel_ms = ms;
    cudaEventDestroy(t0); cudaEventDestroy(t1);
  }
  cudaFree(buf);
  if (rc != DEMI_OK) return rc;
  if (e != cudaSuccess) return fail(h, DEMI_ERR_CUDA, "demi_fuzz_provenance: %s", cudaGetErrorString(e));
  return DEMI_OK;
}

extern "C" int32_t demi_stats(const demi_handle* h, demi_perf* out) {
  if (!h || !out) return DEMI_ERR_INVALID;
  *out = h->perf;
  return DEMI_OK;
}
