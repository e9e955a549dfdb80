// subseq_kernel.cuh — K1 in "subsequence" mode: RandomScheduler.test (RandomScheduler.scala:597-612) of many
// subsequences of one external program in one launch, for DDMin with RandomScheduler as its TestOracle
// (RunnerUtils.randomDDMin, RunnerUtils.scala:601-623).
//
// A work item is one execution of one test: item = i*T + t is execution i (seed seed_base + i) of test t, so the
// early executions of every test run first.  Test t runs program_of(mask_t) (include/demi_b200.h): the machines
// below are the K1 machines with two changes, taken from the test's side-table entry:
//   * the inject loop skips the externals the mask leaves out (the lane engine's Send ordinal still counts them,
//     so it keeps indexing the handle's full `ext_sends` table);
//   * the end-of-program test and the capacities are those of program_of(mask_t): each test has its own KernelArgs
//     copy (`targs[t]`) with n_ext = n_eff and the test's pending / messagesToSend / node capacities.
// No per-execution record is written: an execution that ends on a matching violation lowers first_hit[t], one that
// ends on a capacity status lowers first_bad[t] (atomicMin).  An item whose test already stopped at an earlier
// execution (min(first_hit, first_bad) < i) is skipped: it cannot change that minimum, so the verdict is the same
// whatever the schedule of the launch.
//
// The K1 kernels themselves (lane_kernel.cuh, fuzz_kernel.cuh) are untouched: these machines derive from theirs and
// restate only inject_until_quiescence() and run().
#pragma once
#include "fuzz_kernel.cuh"
#include "lane_kernel.cuh"

namespace demi {

struct SubseqArgs {
  const KernelArgs* targs;        // [n_tests] warp engine: per-test copy of the launch's KernelArgs
  const KernelArgs* targs_lane;   // [n_tests] lane engine: the same with the lane engine's fields
  const uint64_t* masks;          // [n_tests][mask_words], after the WaitQuiescence collapse
  uint32_t mask_words, n_tests;
  uint64_t n_items;               // n_tests * K <= 2^32-1
  int64_t seed_base;
  uint32_t* first_hit; uint32_t* first_bad;          // [n_tests], K when none
  const uint32_t* index_list; const uint32_t* index_count;   // warp engine: the items the lane engine deferred
  uint32_t* ovf_list; uint32_t* ovf_count;           // lane engine: items it defers
  unsigned long long* counters;                      // [0] deliveries [1] violations [2] deferred [3] executions run
  // per-warp scratch, laid out for the variant picked for the whole program
  uint4* lane_pend; uint4* node_scratch; uint4* pend_scratch; uint16_t* fifo_scratch; uint32_t node_stride;
};

__device__ __forceinline__ bool subseq_selected(const uint64_t* mask, uint32_t j) {
  return (__ldg(mask + (j >> 6)) >> (j & 63)) & 1ull;
}
// the execution at which test t stopped so far (first hit or first capacity status)
__device__ __forceinline__ uint32_t subseq_stop(const SubseqArgs& s, uint32_t t) {
  return min(__ldcv(s.first_hit + t), __ldcv(s.first_bad + t));
}

template <class MODEL, int BD, int LPCAP>
struct SubseqLaneMachine : LaneMachine<MODEL, BD, LPCAP> {
  using B = LaneMachine<MODEL, BD, LPCAP>;
  const uint64_t* mask;

  // LaneMachine::inject_until_quiescence over the selected externals
  __device__ __forceinline__ void inject_until_quiescence() {
    bool loop = true;
    while (loop && this->ext_idx < this->A->n_ext && !this->status) {
      const uint4 raw = __ldg(reinterpret_cast<const uint4*>(this->A->ext) + this->ext_idx);
      const uint32_t kind = raw.x & 0xFF, a = (raw.x >> 8) & 0xFF, b = (raw.x >> 16) & 0xFF;
      if (!subseq_selected(mask, this->ext_idx)) {
        if (kind == DEMI_EXT_SEND) this->ext_send_idx++;
        this->ext_idx++;
        continue;
      }
      uint32_t ek = 0, es = DEMI_DEADLETTERS, ed = a;
      switch (kind) {
        case DEMI_EXT_START:
          ek = DEMI_EV_SPAWN;
          this->inaccessible &= ~(1u << a); this->killed &= ~(1u << a);
          break;
        case DEMI_EXT_KILL:
          ek = DEMI_EV_KILL;
          this->killed |= 1u << a; this->inaccessible |= 1u << a;
          break;
        case DEMI_EXT_SEND:
          if (this->tosend.n >= LANE_TOSEND_CAP || this->ext_send_idx >= 0x80u) { this->defer(); break; }
          this->tosend.push(0x80u | this->ext_send_idx);
          this->ext_send_idx++;
          break;
        case DEMI_EXT_PARTITION:
          ek = DEMI_EV_PARTITION; es = a; ed = b;
          this->part_row(a) |= 1u << b;
          break;
        case DEMI_EXT_UNPARTITION:
          ek = DEMI_EV_UNPARTITION; es = a; ed = b;
          this->part_row(a) &= ~(1u << b);
          break;
        case DEMI_EXT_WAIT_QUIESCENCE:
          ek = DEMI_EV_BEGIN_WAIT_QUIESCENCE; ed = DEMI_DEADLETTERS;
          loop = false;
          break;
        default: break;
      }
      if (ek) this->record_event(ek, es, ed, 0, 0, 0, 0, 0, 0);
      this->ext_idx++;
    }
  }

  // LaneMachine::run without the result hashes: only the verdict and the step count are kept
  __device__ __forceinline__ void run(int64_t seed, uint32_t& violation_out, uint32_t& status_out, uint32_t& steps_out) {
    this->reset(seed);
    uint32_t n_ops = 0, self = 0;
    for (;;) {
      inject_until_quiescence();
      for (;;) {
        const bool go = this->may_continue();
        this->drain(n_ops, self, go);
        n_ops = 0;
        uint4 pick;
        if (!go || !this->pick_next(pick)) break;
        self = hdr_dst(pick.x);
        n_ops = this->dispatch_new_message(pick);
        if (this->status) break;
      }
      if (this->status | this->violation) break;
      if (this->ext_idx < this->A->n_ext) {
        this->record_event(DEMI_EV_QUIESCENCE, DEMI_DEADLETTERS, DEMI_DEADLETTERS, 0, 0, 0, 0, 0, 0);
        continue;
      }
      break;
    }
    if (!this->status && this->nsched <= this->A->max_messages && !this->violation) this->violation = this->check_invariant();
    status_out = this->status;
    violation_out = this->status ? 0u : this->violation;
    steps_out = this->status ? 0u : (uint32_t)this->nsched;
  }
};

template <class MODEL, int PCAP, int TCAP, bool PG>
struct SubseqMachine : Machine<MODEL, PCAP, TCAP, PG, false> {
  const uint64_t* mask;

  // Machine::inject_until_quiescence over the selected externals
  __device__ __forceinline__ void inject_until_quiescence() {
    bool loop = true;
    while (loop && this->ext_idx < this->A->n_ext && !this->status) {
      const uint4 raw = __ldg(reinterpret_cast<const uint4*>(this->A->ext) + this->ext_idx);
      const uint32_t kind = raw.x & 0xFF, a = (raw.x >> 8) & 0xFF, b = (raw.x >> 16) & 0xFF, type = raw.x >> 24;
      if (!subseq_selected(mask, this->ext_idx)) { this->ext_idx++; continue; }
      switch (kind) {
        case DEMI_EXT_START:
          this->record_event(DEMI_EV_SPAWN, DEMI_DEADLETTERS, a, 0, 0, 0, 0, 0, 0);
          this->inaccessible &= ~(1u << a); this->killed &= ~(1u << a); this->dead &= ~(1u << a);
          break;
        case DEMI_EXT_HARD_KILL: this->hard_kill(a); break;
        case DEMI_EXT_KILL:
          this->record_event(DEMI_EV_KILL, DEMI_DEADLETTERS, a, 0, 0, 0, 0, 0, 0);
          this->killed |= 1u << a; this->inaccessible |= 1u << a;
          break;
        case DEMI_EXT_SEND:
          this->tosend_push(make_hdr(DEMI_DEADLETTERS, a, type, DEMI_MF_EXTERNAL), raw.y, raw.z);
          break;
        case DEMI_EXT_PARTITION:
          this->record_event(DEMI_EV_PARTITION, a, b, 0, 0, 0, 0, 0, 0);
          if (this->lane == a) this->part_row |= 1u << b;
          break;
        case DEMI_EXT_UNPARTITION:
          this->record_event(DEMI_EV_UNPARTITION, a, b, 0, 0, 0, 0, 0, 0);
          if (this->lane == a) this->part_row &= ~(1u << b);
          break;
        case DEMI_EXT_WAIT_QUIESCENCE:
          this->record_event(DEMI_EV_BEGIN_WAIT_QUIESCENCE, DEMI_DEADLETTERS, DEMI_DEADLETTERS, 0, 0, 0, 0, 0, 0);
          loop = false;
          break;
        default: break;
      }
      this->ext_idx++;
    }
  }

  // Machine::run without the result hashes
  __device__ __forceinline__ void run(int64_t seed, uint32_t& violation_out, uint32_t& status_out, uint32_t& steps_out) {
    this->reset(seed);
    for (;;) {
      inject_until_quiescence();
      uint4 pick;
      while (this->schedule_new_message(pick)) {
        this->dispatch_new_message(pick);
        if (this->status) break;
      }
      if (this->status | this->violation) break;
      if (this->ext_idx < this->A->n_ext) {
        this->record_event(DEMI_EV_QUIESCENCE, DEMI_DEADLETTERS, DEMI_DEADLETTERS, 0, 0, 0, 0, 0, 0);
        continue;
      }
      break;
    }
    if (!this->status && this->nsched <= this->A->max_messages && !this->violation) this->violation = this->check_invariant();
    status_out = this->status;
    violation_out = this->status ? 0u : this->violation;
    steps_out = this->status ? 0u : (uint32_t)this->nsched;
  }
};

// K1-lane over the items of a subsequence batch; deferred items go to `ovf_list` (by item number).
template <class MODEL, int BD, int LPCAP>
__global__ void __launch_bounds__(BD, DEMI_K1_MIN_BLOCKS)
fuzz_lane_subseq_kernel(const __grid_constant__ SubseqArgs s) {
  using M = SubseqLaneMachine<MODEL, BD, LPCAP>;
  extern __shared__ __align__(16) uint32_t lane_smem[];
  const uint32_t tid = threadIdx.x;
  const uint64_t gthread = (uint64_t)blockIdx.x * BD + tid;
  const uint64_t total = (uint64_t)gridDim.x * BD;
  const uint64_t gwarp = gthread >> 5;

  M m;
  m.smw = lane_smem + tid;
  m.pend = s.lane_pend + gwarp * (uint64_t)LPCAP * 32 + (tid & 31);
  m.pol = l2_evict_last_policy();
  m.rec_ev = nullptr; m.rec_par = nullptr;

  unsigned long long my_steps = 0, my_viol = 0, my_defer = 0, my_run = 0;
  for (uint64_t it = gthread; it < s.n_items; it += total) {
    const uint32_t item = (uint32_t)it, t = item % s.n_tests, i = item / s.n_tests;
    if (subseq_stop(s, t) < i) continue;
    m.A = s.targs_lane + t;
    m.mask = s.masks + (uint64_t)t * s.mask_words;
    uint32_t viol, status, steps;
    m.run(s.seed_base + (int64_t)i, viol, status, steps);
    if (status == LANE_DEFER) {
      const uint32_t pos = atomicAdd(s.ovf_count, 1u);
      s.ovf_list[pos] = item;
      my_defer++;
      continue;
    }
    if (viol) atomicMin(s.first_hit + t, i);          // the lane engine ends on no capacity status: it defers instead
    my_steps += steps; my_viol += viol ? 1u : 0u; my_run++;
  }
  for (int o = 16; o > 0; o >>= 1) {
    my_steps += __shfl_xor_sync(FULL_MASK, my_steps, o);
    my_viol += __shfl_xor_sync(FULL_MASK, my_viol, o);
    my_defer += __shfl_xor_sync(FULL_MASK, my_defer, o);
    my_run += __shfl_xor_sync(FULL_MASK, my_run, o);
  }
  if ((tid & 31) == 0 && (my_steps | my_viol | my_defer | my_run)) {
    atomicAdd(s.counters, my_steps);
    atomicAdd(s.counters + 1, my_viol);
    if (my_defer) atomicAdd(s.counters + 2, my_defer);
    atomicAdd(s.counters + 3, my_run);
  }
}

// the warp engine over the items of a subsequence batch (all of them, or the ones the lane engine deferred)
template <class MODEL, int PCAP, int TCAP, bool PG, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
fuzz_subseq_kernel(const __grid_constant__ SubseqArgs s) {
  using M = SubseqMachine<MODEL, PCAP, TCAP, PG>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t gw = (uint64_t)blockIdx.x * WARPS + warp;
  const uint64_t total_warps = (uint64_t)gridDim.x * WARPS;

  M m;
  m.sm = reinterpret_cast<typename M::Smem*>(smem_raw + (size_t)warp * sizeof(typename M::Smem));
  m.A = s.targs;
  m.lane = lane;
  m.rec_ev = nullptr;
  m.nodes_g = s.node_scratch + gw * s.node_stride;
  m.pend_g = PG ? (s.pend_scratch + gw * (uint64_t)PCAP) : nullptr;
  if (PG && s.fifo_scratch) {
    uint16_t* f = s.fifo_scratch + gw * (uint64_t)(M::HALF + 3 * FIFO_PAIRS);
    m.f_next = f; m.f_head = f + M::HALF; m.f_tail = m.f_head + FIFO_PAIRS; m.f_pairs = m.f_tail + FIFO_PAIRS;
  } else {
    m.f_next = m.f_head = m.f_tail = m.f_pairs = nullptr;
  }

  const uint64_t count = s.index_list ? (uint64_t)(*s.index_count) : s.n_items;
  unsigned long long my_steps = 0, my_viol = 0, my_run = 0;
  for (uint64_t k = gw; k < count; k += total_warps) {
    const uint32_t item = s.index_list ? s.index_list[k] : (uint32_t)k;
    const uint32_t t = item % s.n_tests, i = item / s.n_tests;
    uint32_t stop = 0;
    if (lane == 0) stop = subseq_stop(s, t);
    stop = __shfl_sync(FULL_MASK, stop, 0);              // one warp-uniform decision
    if (stop < i) continue;
    m.A = s.targs + t;
    m.mask = s.masks + (uint64_t)t * s.mask_words;
    uint32_t viol, status, steps;
    m.run(s.seed_base + (int64_t)i, viol, status, steps);
    if (lane == 0) {
      if (status) atomicMin(s.first_bad + t, i);
      else if (viol) atomicMin(s.first_hit + t, i);
    }
    my_steps += steps; my_viol += viol ? 1u : 0u; my_run++;
  }
  if (lane == 0 && (my_steps | my_viol | my_run)) {
    atomicAdd(s.counters, my_steps);
    atomicAdd(s.counters + 1, my_viol);
    atomicAdd(s.counters + 3, my_run);
  }
}

}  // namespace demi
