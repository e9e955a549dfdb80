// lane_kernel.cuh — K1-lane: the high-throughput random-fuzz kernel.  One
// THREAD owns one schedule prefix (one RandomScheduler execution, reference:
// schedulers/RandomScheduler.scala:234-272, :352-485); a warp advances 32
// prefixes in lock-step.  Same semantics as machine.cuh, restated for a scalar
// owner:
//
//   registers      java.util.Random state, counters, network masks, and the
//                  timer sets as BITMASKS over the model's finite timer universe
//                  (justScheduledTimers / timerToCancellable / timersCancelled-
//                  ThisStep), messagesToSend and timersToResend as byte queues
//   shared memory  actor states, the receive() outbox and partition rows,
//                  thread-interleaved (word w of thread t at [w*BD + t]: every
//                  access is bank-conflict free whatever each lane indexes)
//   HBM / L1 / L2  the pending-message array (RandomizedHashSet.arr), 16-byte
//                  entries interleaved per warp (entry i of lane l at
//                  [(i*32 + l)])
//
// Exactness: every structure here is a bounded, duplicate-free restatement.
// Whenever an execution could leave that regime (a capacity would overflow, or
// the DepTracker child-reuse rule (DepTracker.scala:94-108) could fire) the
// thread stops and appends the prefix index to the defer list; the general
// warp engine (fuzz_kernel.cuh) then re-runs exactly those prefixes.  A
// prefix that completes here has, by construction, the same result as in the
// general engine.
#pragma once
#include <type_traits>
#include "machine.cuh"
#include "models/models.cuh"

namespace demi {

// Does the model split receive() into lane_decide() + plan_item() (`static constexpr bool LANE_PLAN = true`, see
// Raft5)?  Then the lane engine produces receive()'s sends itself (LaneMachine::plan_sends_produced).
template <class M, class = void>
struct lane_plan_model { static constexpr bool value = false; };
template <class M>
struct lane_plan_model<M, std::void_t<decltype(M::LANE_PLAN)>> { static constexpr bool value = M::LANE_PLAN; };

#ifndef DEMI_K1_PEND_HINT
#define DEMI_K1_PEND_HINT 1      // pending array accessed with an L2 evict_last policy
#endif
#ifndef DEMI_K1_RESULT_CS
#define DEMI_K1_RESULT_CS 1      // result records written with streaming (evict-first) stores
#endif
#ifndef DEMI_K1_DIRECT_OUTBOX
#define DEMI_K1_DIRECT_OUTBOX 1  // models with LANE_SENDS_DISTINCT: receive()'s operations are applied as they are issued
#endif
#ifndef DEMI_K1_LPCAP_RAFT5
#define DEMI_K1_LPCAP_RAFT5 96
#endif

constexpr uint32_t LANE_DEFER = 0xFFFFu;      // internal status: hand over to the warp engine

// The pending arrays are the only data this kernel re-reads from global memory; the result records are written once.
// An L2 evict_last policy on the former (and evict-first stores for the latter) keeps the arrays cache-resident:
// measured 533 -> 121 B of DRAM traffic per prefix (profiles/r2_k1_l2_policy.md).  Every access to the arrays goes
// through these two volatile asm statements (which keep their program order), and nothing else aliases the arrays,
// so no "memory" clobber is needed.
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint4 ld_l2_hint(const uint4* p, uint64_t pol) {
#if DEMI_K1_PEND_HINT
  uint4 v;
  asm volatile("ld.global.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
  return v;
#else
  (void)pol; return *p;
#endif
}
__device__ __forceinline__ void st_l2_hint(uint4* p, uint4 v, uint64_t pol) {
#if DEMI_K1_PEND_HINT
  asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1,%2,%3,%4}, %5;"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol));
#else
  (void)pol; *p = v;
#endif
}
constexpr int LANE_TOSEND_CAP = 16;
constexpr int LANE_RESEND_CAP = 8;

// One actor's state, thread-interleaved in shared memory.
struct LaneState {
  uint32_t* base;      // &smem[word0 * BD + tid]
  uint32_t bd;
  __device__ __forceinline__ uint8_t& operator[](uint32_t i) const {
    return reinterpret_cast<uint8_t*>(base + (i >> 2) * bd)[i & 3];
  }
  __device__ __forceinline__ uint8_t& b(uint32_t i) const { return (*this)[i]; }
  __device__ __forceinline__ uint32_t& w(uint32_t i) const { return base[i * bd]; }
};
template <int SW>
struct LaneAll {
  uint32_t* base; uint32_t bd;
  __device__ __forceinline__ LaneState actor(uint32_t a) const { return LaneState{base + a * SW * bd, bd}; }
};

// receive()'s outbox, thread-interleaved in shared memory (3 words per op).
template <int CAP>
struct LaneOutbox {
  uint32_t* base; uint32_t bd;
  uint32_t n, self;
  bool overflow;
  __device__ __forceinline__ void push(uint32_t op, uint32_t dst, uint32_t type, uint32_t p0, uint32_t p1) {
    if (n >= CAP) { overflow = true; return; }
    base[(n * 3 + 0) * bd] = op | (dst << 8) | (type << 16);
    base[(n * 3 + 1) * bd] = p0;
    base[(n * 3 + 2) * bd] = p1;
    n++;
  }
  __device__ __forceinline__ void send(uint32_t dst, uint32_t type, uint32_t p0, uint32_t p1) { push(OP_SEND, dst, type, p0, p1); }
  __device__ __forceinline__ void schedule_once(uint32_t type, uint32_t p0, uint32_t p1) { push(OP_SCHED_ONCE, self, type, p0, p1); }
  __device__ __forceinline__ void schedule_repeating(uint32_t type, uint32_t p0, uint32_t p1) { push(OP_SCHED_REPEAT, self, type, p0, p1); }
  __device__ __forceinline__ void cancel_timer(uint32_t type, uint32_t p0, uint32_t p1) { push(OP_CANCEL, self, type, p0, p1); }
};

// small FIFO of bytes in two 64-bit registers
struct ByteQueue16 {
  uint64_t lo, hi; uint32_t n;
  __device__ __forceinline__ void clear() { lo = hi = 0; n = 0; }
  __device__ __forceinline__ uint32_t get(uint32_t i) const {
    uint64_t v = i < 8 ? lo : hi;
    return (uint32_t)(v >> ((i & 7) * 8)) & 0xFFu;
  }
  __device__ __forceinline__ void push(uint32_t b) {      // caller checks n < 16
    uint64_t v = (uint64_t)b << ((n & 7) * 8);
    if (n < 8) lo |= v; else hi |= v;
    n++;
  }
  __device__ __forceinline__ void remove_at(uint32_t i) { // order preserving
    ByteQueue16 q; q.clear();
    for (uint32_t k = 0; k < n; k++) if (k != i) q.push(get(k));
    *this = q;
  }
};

// receive()'s view when its operations are applied as they are issued (`dst ! msg` is synchronous in the reference,
// Instrumenter.scala:1098-1108): no staging in shared memory.  Only for models whose receive() cannot produce two equal
// sends (MODEL::LANE_SENDS_DISTINCT), because the duplicate-send screen needs the whole outbox.
template <class M>
struct LaneDirectOutbox {
  M* m; uint32_t self;
  __device__ __forceinline__ void send(uint32_t dst, uint32_t type, uint32_t p0, uint32_t p1) { m->actor_send_produced(self, dst, type, p0, p1); }
  __device__ __forceinline__ void schedule_once(uint32_t type, uint32_t p0, uint32_t p1) { m->schedule_timer(OP_SCHED_ONCE, self, type, p0, p1); }
  __device__ __forceinline__ void schedule_repeating(uint32_t type, uint32_t p0, uint32_t p1) { m->schedule_timer(OP_SCHED_REPEAT, self, type, p0, p1); }
  __device__ __forceinline__ void cancel_timer(uint32_t type, uint32_t p0, uint32_t p1) { m->cancel_timer(self, type, p0, p1); }
};

// REC: the execution's EventTrace and DepTracker parents are written out (provenance batches, demi_fuzz_provenance)
template <class MODEL, int BD, int LPCAP, bool REC = false>
struct LaneMachine {
  static constexpr int N = MODEL::N_ACTORS;
  static constexpr int SW = MODEL::STATE_WORDS;
  static constexpr int OB = MODEL::LANE_OUTBOX;
  // the outbox is staged in shared memory only when receive()'s operations are not applied as they are issued
  static constexpr bool DIRECT = DEMI_K1_DIRECT_OUTBOX && MODEL::LANE_SENDS_DISTINCT;
  static constexpr int OBW = DIRECT ? 0 : OB * 3;
  static constexpr int WORDS = N * SW + OBW + N;       // states + outbox + partition rows
  // receive()'s sends produced from the model's plan (recording runs keep receive()'s own send loop, whose
  // record_event() also writes the EventTrace)
  static constexpr bool PLAN = DIRECT && lane_plan_model<MODEL>::value && !REC;

  uint32_t* smw;             // &smem[tid]; word w at smw[w*BD]
  uint4* pend;               // entry i at pend[i*32]
  uint4* rec_ev; uint16_t* rec_par;   // REC: this execution's EventTrace slot and parent array
  uint64_t pol;              // L2 cache policy of the pending array
  const KernelArgs* A;

  JRandom rng;
  uint32_t n_pending, max_pending;
  ByteQueue16 tosend;        // byte: timer slot, or 0x80|k for the k-th external Send
  uint64_t resend; uint32_t n_resend;
  uint32_t just, registry, cancelled;            // bit per timer slot
  uint32_t root_timers, window_timers;           // duplicate guards for the child-reuse rule
  uint32_t n_nodes, parent_event, n_events, n_uniq;
  int32_t nsched, nmod;
  uint32_t ext_idx, ext_send_idx;
  uint32_t violation, status;
  uint32_t inaccessible, killed;
  uint64_t thash;

  __device__ __forceinline__ uint32_t& part_row(uint32_t a) { return smw[(N * SW + OBW + a) * BD]; }
  __device__ __forceinline__ LaneState actor(uint32_t a) { return LaneState{smw + a * SW * BD, BD}; }

  __device__ __forceinline__ void defer() { status = LANE_DEFER; }

  // EventTrace.+= (EventTrace.scala:88-110)
  __device__ __forceinline__ void record_event(uint32_t kind, uint32_t src, uint32_t dst, uint32_t type,
                                               uint32_t p0, uint32_t p1, uint32_t uniq, uint32_t node, uint32_t parent) {
    uint32_t w0 = kind | (src << 8) | (dst << 16) | (type << 24);
    thash += demi_event_term(w0, p0, p1, uniq | (node << 16), n_events, parent);
    if (REC) {
      if (n_events >= A->rec_cap) { defer(); return; }
      rec_ev[n_events] = make_uint4(w0, p0, p1, uniq | (node << 16));
      if (kind == DEMI_EV_MSG_SEND && node < A->rec_parent_cap) rec_par[node] = (uint16_t)parent;   // DepTracker edge
    }
    n_events++;
  }

  // RandomizedHashSet.insert (schedulers/Util.scala:126-136)
  __device__ __forceinline__ void pending_insert(uint4 e) {
    if (n_pending >= A->pending_cap || n_pending >= LPCAP) { defer(); return; }
    st_l2_hint(pend + n_pending * 32, e, pol);
    n_pending++;
    if (n_pending > max_pending) max_pending = n_pending;
  }
  // RandomizedHashSet.remove (schedulers/Util.scala:146-163)
  __device__ __forceinline__ uint4 pending_remove_at(uint32_t i) {
    uint4 v = ld_l2_hint(pend + i * 32, pol);
    uint4 last = ld_l2_hint(pend + (n_pending - 1) * 32, pol);
    st_l2_hint(pend + i * 32, last, pol);
    n_pending--;
    return v;
  }

  // EventOrchestrator.crosses_partition (EventOrchestrator.scala:345-351)
  __device__ __forceinline__ bool crosses_partition(uint32_t snd, uint32_t rcv) {
    if (!(inaccessible | killed) && !A->has_partitions) return false;      // everyone started, no one isolated
    bool snd_actor = snd < DEMI_MAX_ACTORS;
    if (snd == rcv && !((killed >> snd) & 1u)) return false;
    if (A->has_partitions && snd_actor) {
      if ((part_row(snd) >> rcv) & 1u) return true;
      if ((part_row(rcv) >> snd) & 1u) return true;
    }
    if ((inaccessible >> rcv) & 1u) return true;
    if (snd_actor && ((inaccessible >> snd) & 1u)) return true;
    return false;
  }

  // RandomScheduler.event_produced (RandomScheduler.scala:274-321) after
  // Instrumenter.aroundDispatch's cancelled-timer drop (Instrumenter.scala:1090-1096).
  // DepTracker.getMessage (DepTracker.scala:82-109): in the regime this engine
  // accepts no child is ever reused, so the Unique id is simply the next one.
  // The sends of receive() itself (sender an actor, no flags): the external / timer branches do not apply.
  __device__ __forceinline__ void actor_send_produced(uint32_t self, uint32_t dst, uint32_t type, uint32_t p0, uint32_t p1) {
    if (status) return;
    if (cancelled) {
      const int slot = MODEL::timer_slot(dst, type, p0, p1);
      if (slot >= 0 && ((cancelled >> slot) & 1u)) { cancelled &= ~(1u << slot); return; }
    }
    if (n_nodes >= A->node_cap) { defer(); return; }
    const uint32_t uniq = ++n_uniq, node = n_nodes++;
    if (!crosses_partition(self, dst)) {
      pending_insert(make_uint4(make_hdr(self, dst, type, 0), p0, p1, uniq | (node << 16)));
      if (status) return;
    }
    record_event(DEMI_EV_MSG_SEND, self, dst, type, p0, p1, uniq, node, parent_event);
  }
  // A timer message flushed from messagesToSend (sender deadLetters, recorded as "Timer"); `slot` is its key.
  __device__ __forceinline__ void timer_produced(uint32_t slot) {
    const uint32_t bit = 1u << slot;
    if (cancelled & bit) { cancelled &= ~bit; return; }
    if (n_nodes >= A->node_cap) { defer(); return; }
    // two equal timer sends under one parent would share a Unique: defer those
    if (parent_event == 0) { if (root_timers & bit) { defer(); return; } root_timers |= bit; }
    else { if (window_timers & bit) { defer(); return; } window_timers |= bit; }
    const uint32_t uniq = ++n_uniq, node = n_nodes++;
    uint32_t dst, type, p0, p1;
    MODEL::slot_msg(slot, dst, type, p0, p1);
    if (!crosses_partition(DEMI_DEADLETTERS, dst)) {
      pending_insert(make_uint4(make_hdr(DEMI_DEADLETTERS, dst, type, DEMI_MF_TIMER), p0, p1, uniq | (node << 16)));
      if (status) return;
    }
    record_event(DEMI_EV_MSG_SEND, DEMI_TIMER_SND, dst, type, p0, p1, uniq, node, parent_event);
  }
  // An external Send flushed from messagesToSend (`hdr` carries DEMI_MF_EXTERNAL).
  __device__ __forceinline__ void external_produced(uint32_t hdr, uint32_t p0, uint32_t p1) {
    const uint32_t dst = hdr_dst(hdr), type = hdr_type(hdr);
    const int slot = MODEL::timer_slot(dst, type, p0, p1);
    if (slot >= 0) {
      if ((cancelled >> slot) & 1u) { cancelled &= ~(1u << slot); return; }
      defer(); return;                          // an external that equals a timer key could share its Unique
    }
    if (n_nodes >= A->node_cap) { defer(); return; }
    const uint32_t uniq = ++n_uniq;
    parent_event = 0;                           // reportNewlyEnabledExternal (DepTracker.scala:119-122)
    const uint32_t node = n_nodes++;            // (identical external Sends are screened on the host)
    pending_insert(make_uint4(hdr, p0, p1, uniq | (node << 16)));
    if (status) return;
    record_event(DEMI_EV_MSG_SEND, hdr_src(hdr), dst, type, p0, p1, uniq, node, 0u);
  }

  // ExternalEventInjector.handle_timer (ExternalEventInjector.scala:282-297)
  __device__ __forceinline__ void handle_timer(uint32_t slot) {
    if (A->ignore_timers) return;
    if (tosend.n >= LANE_TOSEND_CAP || tosend.n >= A->tosend_cap) { defer(); return; }
    tosend.push(slot);
  }
  // RandomScheduler.enqueue_timer (RandomScheduler.scala:549-559)
  __device__ __forceinline__ void enqueue_timer(uint32_t slot) {
    if ((just >> slot) & 1u) {
      if (n_resend >= LANE_RESEND_CAP) { defer(); return; }
      resend |= (uint64_t)slot << (n_resend * 8);
      n_resend++;
      return;
    }
    handle_timer(slot);
  }
  // scheduler.scheduleOnce / schedule (Instrumenter.scala:1126-1190)
  __device__ __forceinline__ void schedule_timer(uint32_t kind, uint32_t self, uint32_t type, uint32_t p0, uint32_t p1) {
    if (status) return;
    const int s2 = MODEL::timer_slot(self, type, p0, p1);
    if (s2 < 0) { defer(); return; }
    if ((registry >> s2) & 1u) return;                        // "Non-unique timer" (Instrumenter.scala:1154-1157)
    if (kind == OP_SCHED_REPEAT) {
      if (__popc(registry) >= DEMI_TIMERSET_CAP) { defer(); return; }
      registry |= 1u << s2;
    }
    enqueue_timer((uint32_t)s2);
  }
  // First the ops receive() left in the outbox (`n_ops`, sender `self`), in program order; then, if `do_flush`,
  // ExternalEventInjector.send_external_messages (ExternalEventInjector.scala:306-365).  Two loops, so that the
  // lanes of a warp reconverge between the phases and their flush items are processed together.
  __device__ __forceinline__ void drain(uint32_t n_ops, uint32_t self, bool do_flush) {
    if constexpr (!DIRECT) {
      uint32_t* ob = smw + N * SW * BD;
#pragma unroll 1
      for (uint32_t i = 0; i < n_ops && !status; i++) {
        const uint32_t w0 = ob[(i * 3) * BD], p0 = ob[(i * 3 + 1) * BD], p1 = ob[(i * 3 + 2) * BD];
        const uint32_t kind = w0 & 0xFF, odst = (w0 >> 8) & 0xFF, otype = (w0 >> 16) & 0xFF;
        if (kind == OP_SEND) { actor_send_produced(self, odst, otype, p0, p1); continue; }
        if (kind == OP_CANCEL) { cancel_timer(odst, otype, p0, p1); continue; }
        schedule_timer(kind, odst, otype, p0, p1);
      }
    }
    if (status || !do_flush) return;
#pragma unroll 1
    for (uint32_t i = 0; i < tosend.n && !status; i++) {
      const uint32_t b = tosend.get(i);
      if (b & 0x80u) {
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(A->ext_sends) + (b & 0x7Fu));
        external_produced(raw.x, raw.y, raw.z);
      } else {
        timer_produced(b);
      }
    }
    if (!status) tosend.clear();
  }

  // Cancellable.cancel(): Instrumenter.cancelTimer (Instrumenter.scala:159-168) ->
  // RandomScheduler.notify_timer_cancel (RandomScheduler.scala:525-534)
  __device__ __forceinline__ void cancel_timer(uint32_t self, uint32_t type, uint32_t p0, uint32_t p1) {
    if (status) return;
    int slot = MODEL::timer_slot(self, type, p0, p1);
    if (slot < 0) { defer(); return; }
    uint32_t bit = 1u << slot;
    if (!(cancelled & bit) && __popc(cancelled) >= DEMI_TIMERSET_CAP) { defer(); return; }
    cancelled |= bit;
    registry &= ~bit;
    for (uint32_t i = 0; i < tosend.n; i++)           // handle_timer_cancel (ExternalEventInjector.scala:601-610)
      if (tosend.get(i) == (uint32_t)slot) { tosend.remove_at(i); return; }
    // FullyRandom.remove (RandomScheduler.scala:653-664): first match in array order.  Four entries are fetched per
    // step so that their latencies overlap (this scan was 6 % of the kernel's stall samples when it fetched one).
    const uint32_t want = make_hdr(DEMI_DEADLETTERS, self, type, 0);
#pragma unroll 1
    for (uint32_t i = 0; i < n_pending; i += 4) {
      uint4 q[4];
#pragma unroll
      for (uint32_t k = 0; k < 4; k++) q[k] = (i + k < n_pending) ? ld_l2_hint(pend + (i + k) * 32, pol) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (uint32_t k = 0; k < 4; k++)
        if ((q[k].x & 0x00FFFFFFu) == want && q[k].y == p0 && q[k].z == p1) { pending_remove_at(i + k); return; }
    }
  }

  __device__ __forceinline__ uint32_t check_invariant() {
    uint32_t v = MODEL::invariant(LaneAll<SW>{smw, BD}, A->model_flags);
    if (!A->looking_for) return v;                    // violationMatches (RandomScheduler.scala:138-154)
    return (v && v == A->looking_for) ? A->looking_for : 0u;
  }

  // EventOrchestrator.inject_until_quiescence (EventOrchestrator.scala:132-189)
  __device__ __forceinline__ void inject_until_quiescence() {
    bool loop = true;
    while (loop && ext_idx < A->n_ext && !status) {
      uint4 raw = __ldg(reinterpret_cast<const uint4*>(A->ext) + ext_idx);
      uint32_t kind = raw.x & 0xFF, a = (raw.x >> 8) & 0xFF, b = (raw.x >> 16) & 0xFF;
      uint32_t ek = 0, es = DEMI_DEADLETTERS, ed = a;          // the EventTrace element this external leaves
      switch (kind) {
        case DEMI_EXT_START:
          ek = DEMI_EV_SPAWN;
          inaccessible &= ~(1u << a); killed &= ~(1u << a);
          break;
        case DEMI_EXT_KILL:
          ek = DEMI_EV_KILL;
          killed |= 1u << a; inaccessible |= 1u << a;
          break;
        case DEMI_EXT_SEND:
          if (tosend.n >= LANE_TOSEND_CAP || ext_send_idx >= 0x80u) { defer(); break; }
          tosend.push(0x80u | ext_send_idx);
          ext_send_idx++;
          break;
        case DEMI_EXT_PARTITION:
          ek = DEMI_EV_PARTITION; es = a; ed = b;
          part_row(a) |= 1u << b;
          break;
        case DEMI_EXT_UNPARTITION:
          ek = DEMI_EV_UNPARTITION; es = a; ed = b;
          part_row(a) &= ~(1u << b);
          break;
        case DEMI_EXT_WAIT_QUIESCENCE:
          ek = DEMI_EV_BEGIN_WAIT_QUIESCENCE; ed = DEMI_DEADLETTERS;
          loop = false;
          break;
        default: break;
      }
      if (ek) record_event(ek, es, ed, 0, 0, 0, 0, 0, 0);
      ext_idx++;
    }
  }

  // RandomScheduler.schedule_new_message (RandomScheduler.scala:352-485); blockedActors is empty here
  // the stop conditions at the top of schedule_new_message (:354-401); they read
  // only counters and actor states, so they are evaluated before the previous
  // delivery's outbox is drained (drain() then flushes only if we go on)
  __device__ __forceinline__ bool may_continue() {
    if (status | violation) return false;
    if (nsched > A->max_messages) { ext_idx = A->n_ext; return false; }
    if (A->interval > 0 && nmod == 0 && nsched != 0) {
      violation = check_invariant();
      if (violation) return false;
    }
    return true;
  }
  __device__ __forceinline__ bool pick_next(uint4& pick) {
    if (status) return false;
    if (n_pending == 0) return false;
    pick = pending_remove_at(rng.next_int(n_pending));          // Util.scala:171-176
    nsched++;
    if (nsched == 0x7FFFFFFF) nsched = 1;
    if (++nmod == A->interval) nmod = 0;
    uint32_t src = hdr_src(pick.x), dst = hdr_dst(pick.x), type = hdr_type(pick.x);
    record_event(DEMI_EV_MSG_EVENT, src, dst, type, pick.y, pick.z, pick.w & 0xFFFF, pick.w >> 16, 0);
    parent_event = pick.w >> 16;                                // reportNewlyDelivered (DepTracker.scala:132-135)
    window_timers = 0;
    // updateRepeatingTimer :405-421
    int slot = MODEL::timer_slot(dst, type, pick.y, pick.z);
    if (slot >= 0 && ((registry >> slot) & 1u)) {
      just |= 1u << slot;
    } else {
      for (uint32_t i = 0; i < n_resend; i++) handle_timer((uint32_t)(resend >> (i * 8)) & 0xFFu);
      resend = 0; n_resend = 0;
      just = 0;
    }
    return !status;
  }

  // Instrumenter.dispatch_new_message (Instrumenter.scala:913-1017)
  // returns the number of outbox ops receive() produced (applied by drain())
  __device__ __forceinline__ uint32_t dispatch_new_message(const uint4& pick) {
    uint32_t src = hdr_src(pick.x), dst = hdr_dst(pick.x), type = hdr_type(pick.x);
    int slot = MODEL::timer_slot(dst, type, pick.y, pick.z);
    if (slot >= 0 && ((registry >> slot) & 1u)) enqueue_timer((uint32_t)slot);     // re-arm :1008-1016
    if (status) return 0;
    if constexpr (PLAN) {
      dispatch_plan(dst, src, type, pick.y, pick.z);
      return 0;
    } else if constexpr (DIRECT) {
      LaneDirectOutbox<LaneMachine> direct{this, dst};
      MODEL::receive(direct, dst, actor(dst), src, type, pick.y, pick.z, A->model_flags);
      return 0;
    }
    LaneOutbox<OB> ob;
    ob.base = smw + N * SW * BD; ob.bd = BD; ob.n = 0; ob.self = dst; ob.overflow = false;
    MODEL::receive(ob, dst, actor(dst), src, type, pick.y, pick.z, A->model_flags);
    if (ob.overflow) { defer(); return 0; }
    // equal sends out of one receive() would share a Unique (child reuse): defer.  A 64-bit filter over the
    // (op, dst, type) words settles the common case — all headers distinct — in one pass; only a filter hit
    // (a real duplicate, or a 1-in-64 collision) pays for the pairwise comparison.
    if (MODEL::LANE_SENDS_DISTINCT) return ob.n;                    // one send per receiver: nothing can be equal
    uint64_t seen = 0; bool maybe = false;
    for (uint32_t i = 0; i < ob.n; i++) {
      const uint64_t bit = 1ull << ((ob.base[(i * 3) * BD] * 0x9E3779B1u) >> 26);
      maybe |= (seen & bit) != 0;
      seen |= bit;
    }
    if (maybe)
    for (uint32_t i = 1; i < ob.n; i++) {
      const uint32_t wi = ob.base[(i * 3) * BD];
      for (uint32_t j = 0; j < i; j++)
        if (wi == ob.base[(j * 3) * BD] && (wi & 0xFF) == OP_SEND &&
            ob.base[(i * 3 + 1) * BD] == ob.base[(j * 3 + 1) * BD] && ob.base[(i * 3 + 2) * BD] == ob.base[(j * 3 + 2) * BD]) {
          defer(); return 0;
        }
    }
    return ob.n;
  }

  // receive() of a PLAN model, in its order: state update and cancel, then the sends, then the schedule
  template <class MM = MODEL>
  __device__ __forceinline__ void dispatch_plan(uint32_t self, uint32_t src, uint32_t type, uint32_t p0, uint32_t p1) {
    LaneDirectOutbox<LaneMachine> direct{this, self};
    const typename MM::Plan p = MODEL::lane_decide(direct, self, actor(self), src, type, p0, p1, A->model_flags);
    plan_sends_produced<MM>(p, self, src);
    if (p.sched) schedule_timer(OP_SCHED_REPEAT, self, p.sched, 0, 0);
  }
  // actor_send_produced() for each send of plan `p`, in plan order.  While nobody is isolated or partitioned and the
  // node and pending capacities hold all of the sends, every send is inserted and none defers, so the ids, trace
  // positions and pending slots of send k are simply the next ones plus k, and the counters advance once for the
  // whole plan.  (No send of a plan is a timer key, so the cancelled-timer rule never drops one.)  Otherwise each
  // send goes through actor_send_produced().
  template <class MM = MODEL>
  __device__ __forceinline__ void plan_sends_produced(const typename MM::Plan& p, uint32_t self, uint32_t src) {
    const uint32_t n = MODEL::plan_sends(p);
    if (status || n == 0) return;
    LaneState s = actor(self);
    if ((inaccessible | killed) || A->has_partitions || n_nodes + n > A->node_cap ||
        n_pending + n > A->pending_cap || n_pending + n > (uint32_t)LPCAP) {
#pragma unroll 1
      for (uint32_t k = 0; k < n; k++) {
        uint32_t dst, type, q0, q1;
        MODEL::plan_item(p, self, src, k, s, s, dst, type, q0, q1);
        actor_send_produced(self, dst, type, q0, q1);
      }
      return;
    }
#pragma unroll 1
    for (uint32_t k = 0; k < n; k++) {
      uint32_t dst, type, q0, q1;
      MODEL::plan_item(p, self, src, k, s, s, dst, type, q0, q1);
      const uint32_t w3 = (n_uniq + 1u + k) | ((n_nodes + k) << 16);
      st_l2_hint(pend + (n_pending + k) * 32, make_uint4(make_hdr(self, dst, type, 0), q0, q1, w3), pol);
      thash += demi_event_term(DEMI_EV_MSG_SEND | (self << 8) | (dst << 16) | (type << 24), q0, q1, w3,
                               n_events + k, parent_event);
    }
    n_uniq += n; n_nodes += n; n_events += n;
    n_pending += n;
    if (n_pending > max_pending) max_pending = n_pending;       // nothing is removed between the inserts
  }

  __device__ __forceinline__ void reset(int64_t seed) {
    rng.seed(seed);
#pragma unroll 1
    for (uint32_t i = 0; i < N * SW; i++) smw[i * BD] = MODEL::init_word(i, A->model_flags);
    for (uint32_t a = 0; a < N; a++) part_row(a) = 0;
    n_pending = max_pending = 0;
    tosend.clear(); resend = 0; n_resend = 0;
    just = registry = cancelled = root_timers = window_timers = 0;
    n_nodes = 1; parent_event = 0; n_events = n_uniq = 0;
    nsched = 0; nmod = 0; ext_idx = 0; ext_send_idx = 0;
    violation = status = 0;
    inaccessible = (N >= 32) ? 0xFFFFFFFFu : ((1u << N) - 1u);
    killed = 0; thash = 0;
  }

  __device__ __forceinline__ void run(int64_t seed, demi_fuzz_result& out) {
    reset(seed);
    uint32_t n_ops = 0, self = 0;          // outbox of the delivery that has not been drained yet
    for (;;) {
      inject_until_quiescence();
      for (;;) {
        const bool go = may_continue();
        drain(n_ops, self, go);            // previous receive()'s sends, then (if going on) the flush
        n_ops = 0;
        uint4 pick;
        if (!go || !pick_next(pick)) break;
        self = hdr_dst(pick.x);
        n_ops = dispatch_new_message(pick);
        if (status) break;
      }
      if (status | violation) break;
      if (ext_idx < A->n_ext) {
        record_event(DEMI_EV_QUIESCENCE, DEMI_DEADLETTERS, DEMI_DEADLETTERS, 0, 0, 0, 0, 0, 0);
        continue;
      }
      break;
    }
    if (!status && nsched <= A->max_messages && !violation) violation = check_invariant();
    out.status = (uint16_t)status;
    if (!status) {
      uint64_t sh = 0;
#pragma unroll 1
      for (uint32_t i = 0; i < N * SW; i++) sh += demi_state_term(smw[i * BD], i);
      if (A->fuzz_flags & DEMI_FF_HASH_PENDING)
#pragma unroll 1
        for (uint32_t i = 0; i < n_pending; i++) {
          uint4 q = ld_l2_hint(pend + i * 32, pol);
          sh += demi_pending_term(q.x & 0x00FFFFFFu, q.y, q.z);
        }
      out.violation = violation; out.steps = (uint32_t)nsched;
      out.state_hash = sh; out.trace_hash = thash;
      out.n_nodes = (uint16_t)n_nodes;
      out.n_events = (uint16_t)(n_events > 65535u ? 65535u : n_events);
      out.max_pending = (uint16_t)max_pending;
    }
  }
};

#ifndef DEMI_K1_MIN_BLOCKS
#define DEMI_K1_MIN_BLOCKS 3
#endif
// REC launches walk a work list (`index_list`): slot `it` of the list owns rec_events[it*rec_cap ..), rec_parent[it*cap ..),
// rec_counts[it*4 ..) and results[it]; a deferred slot is handed to the general engine by POSITION (ovf_list holds `it`).
template <class MODEL, int BD, int LPCAP, bool REC = false>
__global__ void __launch_bounds__(BD, DEMI_K1_MIN_BLOCKS)
fuzz_lane_kernel(const __grid_constant__ KernelArgs args) {
  using M = LaneMachine<MODEL, BD, LPCAP, REC>;
  extern __shared__ __align__(16) uint32_t lane_smem[];
  const uint32_t tid = threadIdx.x;
  const uint64_t gthread = (uint64_t)blockIdx.x * BD + tid;
  const uint64_t total = (uint64_t)gridDim.x * BD;
  const uint64_t gwarp = gthread >> 5;

  M m;
  m.smw = lane_smem + tid;
  m.pend = args.lane_pend + gwarp * (uint64_t)LPCAP * 32 + (tid & 31);
  m.A = &args;
  m.pol = l2_evict_last_policy();
  m.rec_ev = nullptr; m.rec_par = nullptr;

  const uint64_t count = (REC && args.index_list) ? (uint64_t)(*args.index_count) : args.n_prefixes;
  unsigned long long my_steps = 0, my_viol = 0, my_defer = 0;
  for (uint64_t it = gthread; it < count; it += total) {
    const uint64_t idx = (REC && args.index_list) ? (uint64_t)args.index_list[it] : it;
    if (REC) {
      m.rec_ev = reinterpret_cast<uint4*>(args.rec_events + it * (uint64_t)args.rec_cap);
      m.rec_par = args.rec_parent + it * (uint64_t)args.rec_parent_cap;
      m.rec_par[0] = 0;
    }
    demi_fuzz_result r;
    m.run(args.seed_base + (int64_t)idx, r);
    if (r.status == LANE_DEFER) {
      uint32_t pos = atomicAdd(args.ovf_count, 1u);
      args.ovf_list[pos] = (uint32_t)(REC ? it : idx);
      my_defer++;
    } else {
      // written once, never re-read here: streaming stores, so that the records do not push the pending arrays out of L2
      uint4* dst = reinterpret_cast<uint4*>(args.results + (REC ? it : idx));
      const uint4 r0 = make_uint4(r.violation, r.steps, (uint32_t)r.state_hash, (uint32_t)(r.state_hash >> 32));
      const uint4 r1 = make_uint4((uint32_t)r.trace_hash, (uint32_t)(r.trace_hash >> 32), (uint32_t)r.n_nodes | ((uint32_t)r.n_events << 16),
                                  (uint32_t)r.max_pending | ((uint32_t)r.status << 16));
#if DEMI_K1_RESULT_CS
      __stcs(dst, r0); __stcs(dst + 1, r1);
#else
      dst[0] = r0; dst[1] = r1;
#endif
      if (REC) {
        uint32_t aff = 0;
        if (r.status == 0 && r.violation) {      // ViolationFingerprint.affectedNodes of the violation the execution stopped on
          uint32_t st[M::N * M::SW];
          for (uint32_t i = 0; i < (uint32_t)(M::N * M::SW); i++) st[i] = m.smw[i * BD];
          aff = MODEL::affected(st, args.model_flags, r.violation);
        }
        reinterpret_cast<uint4*>(args.rec_counts)[it] = make_uint4(m.n_events, m.n_nodes, aff, r.violation);
      }
      my_steps += r.steps;
      my_viol += r.violation ? 1u : 0u;
    }
  }
  // warp-aggregate the summary counters
  for (int o = 16; o > 0; o >>= 1) {
    my_steps += __shfl_xor_sync(FULL_MASK, my_steps, o);
    my_viol += __shfl_xor_sync(FULL_MASK, my_viol, o);
    my_defer += __shfl_xor_sync(FULL_MASK, my_defer, o);
  }
  if ((tid & 31) == 0 && args.sum_steps && (my_steps | my_viol | my_defer)) {
    atomicAdd(args.sum_steps, my_steps);
    atomicAdd(args.n_violations, my_viol);
    if (my_defer) atomicAdd(args.sum_steps + 2, my_defer);      // [2]: prefixes handed to the general engine
  }
}

}  // namespace demi
