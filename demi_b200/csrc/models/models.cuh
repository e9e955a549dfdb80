// models.cuh — built-in actor models (the "state-transition functor").
//
// In the reference the transition function is the application's own Akka
// receive(), reached through Instrumenter.dispatch_new_message
// (Instrumenter.scala:913-1017) and ActorCell.receiveMessage
// (WeaveActor.aj:90-108).  The Raft application DEMi was evaluated on
// (akka-raft) is not part of the reference tree (README.md:12,27-28), so these
// are *models of* such applications; their specification is DESIGN.md §3.
//
// Interface a model provides to the engines:
//   N_ACTORS, STATE_WORDS
//   init_word(i, flags)                      initial value of state word i
//   receive<S,O>(out, self, st, src, type, p0, p1, flags)   scalar transition.
//       S = state accessor of ONE actor (st.b(i) byte i, st.w(i) word i), so the
//       same source runs over contiguous shared memory (warp engine, lane 0)
//       and over thread-interleaved shared memory (lane engine, every thread).
//   invariant_lane(states, flags, lane)      warp engine: lane-parallel; the
//                                            engine takes the minimum non-zero code
//   invariant<A>(all, flags)                 lane engine: scalar over all actors;
//                                            all.actor(a) is an S accessor
//   timer_slot / slot_msg                    lane engine: the model's finite timer
//                                            universe (<= 32 (receiver,msg) keys)
//   LANE_OUTBOX                              lane engine: max ops of one receive()
#pragma once
#include "../machine.cuh"

namespace demi {

// ---------------------------------------------------------------- pingpong3
// BASELINE.json configs[0].  Ping(k) to X => X sends Pong(k) to (X+1)%3.
// state: w0 = pings received, w1 = pongs received.
struct PingPong3 {
  static constexpr int N_ACTORS = 3;
  static constexpr int STATE_WORDS = 2;
  static constexpr int ID = DEMI_MODEL_PINGPONG3;
  enum { PING = 1, PONG = 2 };
  __device__ static __forceinline__ uint32_t init_word(uint32_t, uint32_t) { return 0; }
  static constexpr int LANE_OUTBOX = 2;
  static constexpr bool LANE_SENDS_DISTINCT = false;
  static constexpr int REPLAY_OUTBOX = 2;
  template <class S, class O>
  __device__ static __forceinline__ void receive(O& out, uint32_t self, S st, uint32_t /*src*/,
                                                 uint32_t type, uint32_t p0, uint32_t /*p1*/, uint32_t /*flags*/) {
    if (type == PING) {
      st.w(0)++;
      out.send((self + 1) % 3, PONG, p0, 0);
    } else if (type == PONG) {
      st.w(1)++;
    }
  }
  template <class A>
  __device__ static __forceinline__ uint32_t invariant(A all, uint32_t flags) {
    if ((flags & 1u) && all.actor(0).w(1) >= (flags >> 8)) return 7;
    return 0;
  }
  __device__ static __forceinline__ int timer_slot(uint32_t, uint32_t, uint32_t, uint32_t) { return -1; }
  __device__ static __forceinline__ void slot_msg(uint32_t, uint32_t& dst, uint32_t& type, uint32_t& p0, uint32_t& p1) {
    dst = type = p0 = p1 = 0;
  }
  // flags bit0: test hook — code 7 once actor 0 has received >= (flags>>8) pongs
  __device__ static __forceinline__ uint32_t invariant_lane(const uint32_t* states, uint32_t flags, uint32_t lane) {
    if (lane == 0 && (flags & 1u) && states[1] >= (flags >> 8)) return 7;
    return 0;
  }
  // ViolationFingerprint.affectedNodes (TestOracle.scala:9-18) as an actor bitmask
  __device__ static uint32_t affected(const uint32_t*, uint32_t, uint32_t code) { return code == 7 ? 1u : 0u; }
};

// -------------------------------------------------------------------- raft5
// 5-node Raft (Ongaro & Ousterhout, Fig. 2), tick-driven timers, log capacity
// 8, one entry per AppendEntries.  40-byte state, byte layout below.
struct Raft5 {
  static constexpr int N_ACTORS = 5;
  static constexpr int STATE_WORDS = 10;
  static constexpr int ID = DEMI_MODEL_RAFT5;
  enum { ROLE = 0, TERM = 1, VOTED = 2, VOTES = 3, LOGLEN = 4, COMMIT = 5, HEARD = 6,
         LOGTERM = 8, LOGVAL = 16, NEXT = 24, MATCH = 29 };
  enum { INIT = 0, FOLLOWER = 1, CANDIDATE = 2, LEADER = 3 };
  enum { BOOT = 1, CLIENT_CMD = 2, ELECTION_TICK = 3, REQUEST_VOTE = 4, VOTE_REPLY = 5,
         HEARTBEAT_TICK = 6, APPEND_ENTRIES = 7, APPEND_REPLY = 8 };
  static constexpr uint32_t LOG_CAP = 8;
  static constexpr uint32_t NONE = 0xFF;
  static constexpr uint32_t BUG_DOUBLE_VOTE = 1u;
  static constexpr uint32_t BUG_STALE_COMMIT = 2u;

  __device__ static __forceinline__ uint32_t init_word(uint32_t i, uint32_t) {
    return (i % STATE_WORDS == 0) ? (NONE << 16) : 0u;      // byte 2 = votedFor = none
  }

  static constexpr int LANE_OUTBOX = 6;
  // every receive() sends at most one message to each receiver (votes / AppendEntries per peer, one reply), so no two
  // sends of one delivery are equal and the lane engine's duplicate-send screen is skipped
  static constexpr bool LANE_SENDS_DISTINCT = true;
  static constexpr int REPLAY_OUTBOX = 6;
  // timer universe: (actor, ELECTION_TICK) -> 2*actor, (actor, HEARTBEAT_TICK) -> 2*actor+1
  __device__ static __forceinline__ int timer_slot(uint32_t dst, uint32_t type, uint32_t p0, uint32_t p1) {
    if ((type != ELECTION_TICK && type != HEARTBEAT_TICK) || p0 || p1 || dst >= 5) return -1;
    return (int)(dst * 2 + (type == HEARTBEAT_TICK ? 1u : 0u));
  }
  __device__ static __forceinline__ void slot_msg(uint32_t slot, uint32_t& dst, uint32_t& type, uint32_t& p0, uint32_t& p1) {
    dst = slot >> 1; type = (slot & 1u) ? HEARTBEAT_TICK : ELECTION_TICK; p0 = 0; p1 = 0;
  }

  // S is an accessor: s[i] is byte i of this actor's state
  // returns true when the actor was leader: its heartbeat timer is to be cancelled (the caller issues the operation)
  template <class C>
  __device__ static __forceinline__ bool step_down(C& c, uint32_t t) {
    const bool was_leader = c[ROLE] == LEADER;
    if (t > c[TERM]) { c[TERM] = (uint8_t)t; c[VOTED] = (uint8_t)NONE; }
    c[ROLE] = FOLLOWER;
    c[VOTES] = 0;
    return was_leader;
  }
  // The eight scalar bytes of the state (words 0 and 1) are held in two registers for the duration of a receive():
  // a field access is a bit-field extract / insert instead of a byte load or store in (interleaved) shared memory.
  template <class S>
  struct Scalars {
    uint32_t w0, w1;
    struct Ref {
      Scalars* c; uint32_t i;
      __device__ __forceinline__ operator uint32_t() const { return ((i < 4 ? c->w0 : c->w1) >> ((i & 3) * 8)) & 0xFFu; }
      __device__ __forceinline__ Ref& operator=(uint32_t v) {
        const uint32_t sh = (i & 3) * 8;
        uint32_t& w = i < 4 ? c->w0 : c->w1;
        w = (w & ~(0xFFu << sh)) | ((v & 0xFFu) << sh);
        return *this;
      }
      __device__ __forceinline__ Ref& operator=(const Ref& o) { return *this = (uint32_t)o; }
      __device__ __forceinline__ Ref& operator|=(uint32_t v) { return *this = (uint32_t)*this | v; }
      __device__ __forceinline__ Ref& operator++(int) { return *this = (uint32_t)*this + 1u; }
    };
    __device__ __forceinline__ explicit Scalars(const S& s) : w0(s.w(0)), w1(s.w(1)) {}
    __device__ __forceinline__ Ref operator[](uint32_t i) { return Ref{this, i}; }
    __device__ __forceinline__ void flush(const S& s) const { s.w(0) = w0; s.w(1) = w1; }
  };

  template <class S, class O>
  __device__ static __forceinline__ void receive(O& out, uint32_t self, S s, uint32_t src,
                                                 uint32_t type, uint32_t p0, uint32_t p1, uint32_t flags) {
    Scalars<S> c(s);
    const Plan p = decide(out, self, s, c, src, type, p0, p1, flags);
#pragma unroll 1
    for (uint32_t k = 0; k < plan_sends(p); k++) {
      uint32_t dst, qt, q0, q1;
      plan_item(p, self, src, k, s, c, dst, qt, q0, q1);
      out.send(dst, qt, q0, q1);
    }
    if (p.sched) out.schedule_repeating(p.sched, 0, 0);
    c.flush(s);
  }
  // Every handler emits its operations in the order: cancel (step_down), then its sends, then schedule.  The sends
  // are either one reply to the sender or one message per peer, so the handlers only DESCRIBE their operations (a
  // Plan, returned by decide() after the cancel) and these leave through ONE send and ONE schedule site after the
  // switch: engines that apply an operation as it is issued then carry one copy of that code instead of one per
  // handler, and the threads of a warp that handle different message types meet again at those sites.
  //
  // The lane engine (LANE_PLAN) calls lane_decide() and produces the sends itself from plan_item(): send k of a plan,
  // computed from the sender's state after decide().  No type a plan sends is a timer key (timer_slot < 0), so the
  // cancelled-timer rule never drops one of these sends.
  static constexpr bool LANE_PLAN = true;
  enum { PLAN_NONE = 0, PLAN_REPLY = 1, PLAN_REQUEST_VOTES = 2, PLAN_APPEND_ALL = 3 };
  struct Plan { uint32_t kind, type, p0, sched; };
  __device__ static __forceinline__ uint32_t plan_sends(const Plan& p) {
    return p.kind == PLAN_NONE ? 0u : p.kind == PLAN_REPLY ? 1u : 4u;
  }
  // send k of plan p: a reply goes to the sender, the others to every peer in ascending order, skipping `self`
  template <class S, class C>
  __device__ static __forceinline__ void plan_item(const Plan& p, uint32_t self, uint32_t src, uint32_t k, S& s, C& c,
                                                   uint32_t& dst, uint32_t& type, uint32_t& q0, uint32_t& q1) {
    dst = p.kind == PLAN_REPLY ? src : k + (k >= self ? 1u : 0u);
    type = p.kind == PLAN_REPLY ? p.type : (uint32_t)REQUEST_VOTE;
    q0 = p.p0; q1 = 0;
    if (p.kind == PLAN_APPEND_ALL) {
      const uint32_t prev = s[NEXT + dst];
      const uint32_t pt = prev ? s[LOGTERM + prev - 1] : 0u;
      const uint32_t has = prev < c[LOGLEN] ? 1u : 0u;
      const uint32_t et = has ? s[LOGTERM + prev] : 0u, ev = has ? s[LOGVAL + prev] : 0u;
      type = APPEND_ENTRIES;
      q0 = (uint32_t)c[TERM] | (prev << 8) | (pt << 16) | ((uint32_t)c[COMMIT] << 24);
      q1 = has | (et << 8) | (ev << 16);
    }
  }
  // receive() up to and including its cancel; the state is written back, so plan_item() may read it from `s` alone
  template <class S, class O>
  __device__ static __forceinline__ Plan lane_decide(O& out, uint32_t self, S s, uint32_t src,
                                                     uint32_t type, uint32_t p0, uint32_t p1, uint32_t flags) {
    Scalars<S> c(s);
    const Plan p = decide(out, self, s, c, src, type, p0, p1, flags);
    c.flush(s);
    return p;
  }
  template <class S, class C, class O>
  __device__ static __forceinline__ Plan decide(O& out, uint32_t self, S& s, C& c, uint32_t src,
                                                uint32_t type, uint32_t p0, uint32_t p1, uint32_t flags) {
    const uint32_t last_idx = c[LOGLEN];
    const uint32_t last_term = last_idx ? s[LOGTERM + last_idx - 1] : 0u;
    const uint32_t t = p0 & 0xFF;
    if (type != BOOT && type != CLIENT_CMD && c[ROLE] == INIT) return Plan{PLAN_NONE, 0, 0, 0};
    uint32_t plan = PLAN_NONE, plan_type = 0, plan_p0 = 0, sched = 0;
    bool cancel_heartbeat = false;
    switch (type) {
      case BOOT:
        if (c[ROLE] == INIT) { c[ROLE] = FOLLOWER; sched = ELECTION_TICK; }
        break;
      case CLIENT_CMD:
        if (c[ROLE] == LEADER && c[LOGLEN] < LOG_CAP) {
          s[LOGTERM + c[LOGLEN]] = c[TERM];
          s[LOGVAL + c[LOGLEN]] = (uint8_t)(p0 & 0x7F);
          c[LOGLEN]++;
        }
        break;
      case ELECTION_TICK:
        if (c[ROLE] == LEADER) break;
        if (c[HEARD]) { c[HEARD] = 0; break; }
        if (c[TERM] == 255) break;
        c[TERM]++;
        c[ROLE] = CANDIDATE;
        c[VOTED] = (uint8_t)self;
        c[VOTES] = (uint8_t)(1u << self);
        plan = PLAN_REQUEST_VOTES; plan_p0 = (uint32_t)c[TERM] | (last_idx << 8) | (last_term << 16);
        break;
      case REQUEST_VOTE: {
        uint32_t li = (p0 >> 8) & 0xFF, lt = (p0 >> 16) & 0xFF;
        if (t > c[TERM]) cancel_heartbeat = step_down(c, t);
        bool up_to_date = lt > last_term || (lt == last_term && li >= last_idx);
        bool can_vote = (c[VOTED] == NONE || c[VOTED] == src) || (flags & BUG_DOUBLE_VOTE);
        uint32_t grant = (t == c[TERM] && can_vote && up_to_date) ? 1u : 0u;
        if (grant) { c[VOTED] = (uint8_t)src; c[HEARD] = 1; }
        plan = PLAN_REPLY; plan_type = VOTE_REPLY; plan_p0 = (uint32_t)c[TERM] | (grant << 8);
        break;
      }
      case VOTE_REPLY: {
        uint32_t g = (p0 >> 8) & 1u;
        if (t > c[TERM]) { cancel_heartbeat = step_down(c, t); break; }
        if (c[ROLE] == CANDIDATE && t == c[TERM] && g) {
          c[VOTES] |= (uint8_t)(1u << src);
          if (__popc((uint32_t)c[VOTES]) >= 3) {
            c[ROLE] = LEADER;
            for (uint32_t j = 0; j < 5; j++) { s[NEXT + j] = c[LOGLEN]; s[MATCH + j] = 0; }
            if (c[LOGLEN] < LOG_CAP) {                       // leader no-op entry
              s[LOGTERM + c[LOGLEN]] = c[TERM];
              s[LOGVAL + c[LOGLEN]] = (uint8_t)(0x80u | self);
              c[LOGLEN]++;
            }
            plan = PLAN_APPEND_ALL; sched = HEARTBEAT_TICK;   // AppendEntries to every peer, then the heartbeat timer
          }
        }
        break;
      }
      case HEARTBEAT_TICK:
        if (c[ROLE] == LEADER) plan = PLAN_APPEND_ALL;
        break;
      case APPEND_ENTRIES: {
        uint32_t prev = (p0 >> 8) & 0xFF, pt = (p0 >> 16) & 0xFF, lc = (p0 >> 24) & 0xFF;
        uint32_t has = p1 & 1u, et = (p1 >> 8) & 0xFF, ev = (p1 >> 16) & 0xFF;
        plan = PLAN_REPLY; plan_type = APPEND_REPLY;
        if (t < c[TERM]) { plan_p0 = (uint32_t)c[TERM]; break; }
        if (t > c[TERM] || c[ROLE] != FOLLOWER) cancel_heartbeat = step_down(c, t);
        c[HEARD] = 1;
        bool ok = prev <= c[LOGLEN] && (prev == 0 || s[LOGTERM + prev - 1] == pt);
        if (!ok) { plan_p0 = (uint32_t)c[TERM]; break; }
        uint32_t mi = prev;
        if (has) {
          if (c[LOGLEN] > prev && s[LOGTERM + prev] != et) {          // conflict: truncate
            for (uint32_t k = prev; k < LOG_CAP; k++) { s[LOGTERM + k] = 0; s[LOGVAL + k] = 0; }
            c[LOGLEN] = (uint8_t)prev;
          }
          if (c[LOGLEN] == prev && prev < LOG_CAP) {
            s[LOGTERM + prev] = (uint8_t)et; s[LOGVAL + prev] = (uint8_t)ev;
            c[LOGLEN] = (uint8_t)(prev + 1);
          }
          if (c[LOGLEN] > prev) mi = prev + 1;
        }
        uint32_t nc = lc < mi ? lc : mi;
        if (nc > c[COMMIT]) c[COMMIT] = (uint8_t)nc;
        plan_p0 = (uint32_t)c[TERM] | (1u << 8) | (mi << 16);
        break;
      }
      case APPEND_REPLY: {
        uint32_t ok = (p0 >> 8) & 1u, mi = (p0 >> 16) & 0xFF;
        if (t > c[TERM]) { cancel_heartbeat = step_down(c, t); break; }
        if (c[ROLE] != LEADER || t != c[TERM]) break;
        if (ok) {
          if (mi > s[MATCH + src]) s[MATCH + src] = (uint8_t)mi;
          if (mi > s[NEXT + src]) s[NEXT + src] = (uint8_t)mi;
          for (uint32_t idx = c[LOGLEN]; idx > c[COMMIT]; idx--) {
            if (s[LOGTERM + idx - 1] != c[TERM] && !(flags & BUG_STALE_COMMIT)) continue;
            uint32_t cnt = 1;
            for (uint32_t k = 0; k < 5; k++) if (k != self && s[MATCH + k] >= idx) cnt++;
            if (cnt >= 3) { c[COMMIT] = (uint8_t)idx; break; }
          }
        } else if (s[NEXT + src] > 0) {
          s[NEXT + src]--;
        }
        break;
      }
      default: break;
    }
    if (cancel_heartbeat) out.cancel_timer(HEARTBEAT_TICK, 0, 0);
    return Plan{plan, plan_type, plan_p0, sched};
  }

  // lanes 0..9 each own one unordered pair (i<j).  code 1: two leaders in one
  // term; code 2: committed prefixes disagree.
  __device__ static __forceinline__ uint32_t invariant_lane(const uint32_t* states, uint32_t, uint32_t lane) {
    if (lane >= 10) return 0;
    // pair index -> (i,j): (0,1)(0,2)(0,3)(0,4)(1,2)(1,3)(1,4)(2,3)(2,4)(3,4)
    uint32_t i = lane < 4 ? 0u : lane < 7 ? 1u : lane < 9 ? 2u : 3u;
    uint32_t j = lane < 4 ? lane + 1 : lane < 7 ? lane - 2 : lane < 9 ? lane - 4 : 4u;
    const uint8_t* a = reinterpret_cast<const uint8_t*>(states + i * STATE_WORDS);
    const uint8_t* b = reinterpret_cast<const uint8_t*>(states + j * STATE_WORDS);
    if (a[ROLE] == LEADER && b[ROLE] == LEADER && a[TERM] == b[TERM]) return 1;
    uint32_t c = a[COMMIT] < b[COMMIT] ? a[COMMIT] : b[COMMIT];
    for (uint32_t k = 0; k < c; k++)
      if (a[LOGTERM + k] != b[LOGTERM + k] || a[LOGVAL + k] != b[LOGVAL + k]) return 2;
    return 0;
  }
  // affectedNodes: the first pair, in (i, j) order, that witnesses `code`
  __device__ static uint32_t affected(const uint32_t* states, uint32_t, uint32_t code) {
    for (uint32_t i = 0; i < 5; i++)
      for (uint32_t j = i + 1; j < 5; j++) {
        const uint8_t* a = reinterpret_cast<const uint8_t*>(states + i * STATE_WORDS);
        const uint8_t* b = reinterpret_cast<const uint8_t*>(states + j * STATE_WORDS);
        if (code == 1 && a[ROLE] == LEADER && b[ROLE] == LEADER && a[TERM] == b[TERM]) return (1u << i) | (1u << j);
        if (code == 2) {
          uint32_t c = a[COMMIT] < b[COMMIT] ? a[COMMIT] : b[COMMIT];
          for (uint32_t k = 0; k < c; k++)
            if (a[LOGTERM + k] != b[LOGTERM + k] || a[LOGVAL + k] != b[LOGVAL + k]) return (1u << i) | (1u << j);
        }
      }
    return 0;
  }
  template <class A>
  __device__ static __forceinline__ uint32_t invariant(A all, uint32_t) {
    uint32_t code = 0;
#pragma unroll 1
    for (uint32_t i = 0; i < 5; i++)
#pragma unroll 1
      for (uint32_t j = i + 1; j < 5; j++) {
        auto a = all.actor(i);
        auto b = all.actor(j);
        if (a[ROLE] == LEADER && b[ROLE] == LEADER && a[TERM] == b[TERM]) return 1;
        if (code) continue;
        uint32_t c = a[COMMIT] < b[COMMIT] ? a[COMMIT] : b[COMMIT];
#pragma unroll 1
        for (uint32_t k = 0; k < c; k++)
          if (a[LOGTERM + k] != b[LOGTERM + k] || a[LOGVAL + k] != b[LOGVAL + k]) code = 2;
      }
    return code;
  }
};

// ------------------------------------------------------------------ bcast32
// BASELINE.json configs[4]: 32-actor broadcast storm.
// state: w0 = floods received, w1 = max ttl seen + 1.
struct Bcast32 {
  static constexpr int N_ACTORS = 32;
  static constexpr int STATE_WORDS = 2;
  static constexpr int ID = DEMI_MODEL_BCAST32;
  enum { FLOOD = 1, INJECT = 2 };      // INJECT: the external seed message, handled like FLOOD
  __device__ static __forceinline__ uint32_t init_word(uint32_t, uint32_t) { return 0; }
  template <class S, class O>
  __device__ static __forceinline__ void receive(O& out, uint32_t self, S st, uint32_t /*src*/,
                                                 uint32_t type, uint32_t p0, uint32_t /*p1*/, uint32_t /*flags*/) {
    if (type != FLOOD && type != INJECT) return;
    st.w(0)++;
    if (p0 + 1 > st.w(1)) st.w(1) = p0 + 1;
    if (p0 > 0)
      for (uint32_t j = 0; j < 32; j++) if (j != self) out.send(j, FLOOD, p0 - 1, 0);
  }
  static constexpr int REPLAY_OUTBOX = 32;
  static constexpr int LANE_OUTBOX = 32;
  static constexpr bool LANE_SENDS_DISTINCT = false;
  template <class A>
  __device__ static __forceinline__ uint32_t invariant(A all, uint32_t flags) {
    if (!flags) return 0;
    for (uint32_t a = 0; a < 32; a++) if (all.actor(a).w(0) >= flags) return 3;
    return 0;
  }
  __device__ static __forceinline__ int timer_slot(uint32_t, uint32_t, uint32_t, uint32_t) { return -1; }
  __device__ static __forceinline__ void slot_msg(uint32_t, uint32_t& dst, uint32_t& type, uint32_t& p0, uint32_t& p1) {
    dst = type = p0 = p1 = 0;
  }
  // code 3 once some actor has received >= flags floods (flags != 0)
  __device__ static __forceinline__ uint32_t invariant_lane(const uint32_t* states, uint32_t flags, uint32_t lane) {
    if (!flags) return 0;
    return states[lane * 2] >= flags ? 3u : 0u;
  }
  __device__ static uint32_t affected(const uint32_t* states, uint32_t flags, uint32_t code) {
    if (code != 3 || !flags) return 0;
    for (uint32_t a = 0; a < 32; a++) if (states[a * 2] >= flags) return 1u << a;
    return 0;
  }
};

}  // namespace demi
