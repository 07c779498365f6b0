// gs_row.h — one virtual member's lock-step tick: the body of the sm_100a tick kernel.
//
// Reference functions restated here ([U] = hashicorp/memberlist v0.5.2 / serf v0.10.2,
// un-vendored, /root/reference/go.mod:80,85; row numbers = SURVEY.md §8a):
//   a2  schedule/probe/resetNodes       -> probe ring cursor over a keyed permutation
//   a3  probeNode + handleIndirectPing  -> stages IDLE / WAIT_T / WAIT_P, pull-evaluated
//   a4  gossip + kRandomNodes           -> gs_krandom + packet scatter (atomicOr)
//   a5  TransmitLimitedQueue            -> queued mask + tx[r][i] counters, gs_select_packet
//   a6-a9 alive/suspect/dead/refute     -> key transitions of the row owner
//   a7  suspicion (Lifeguard)           -> sus_start/sus_from + timeout table
//   a10 awareness                       -> meta bits 0..2
//   a13 LamportClock.Witness            -> max(clock, v+1) on delivery
//   a14 handleUserEvent                 -> event_min / event_buffer window checks
//
// Determinism: a tick reads only the snapshot written by earlier ticks (key[t&1],
// inbox[t&1]) and its own row; everything a row sends is delivered through commutative
// atomics (atomicOr on inbox[(t+1)&1], atomicMin chain on acc[(t+1)&1]) and consumed by
// the receiving row in tick t+1.  Results do not depend on block scheduling.
#pragma once
#include <string.h>

#include "gs_core.h"
#include "gs_coord.h"

#if defined(__CUDA_ARCH__)
#define GS_DEV __device__ __forceinline__
// Mailbox deliveries may target a row on another GPU (sharded pools).  They are issued as
// system-scope FETCHING atomics: a fire-and-forget reduction over NVLink can still be in flight
// when its kernel retires, a fetching atomic has been performed at the owner once it returns.
__device__ __forceinline__ uint32_t gs_atomic_or_sys(uint32_t* p, uint32_t v) {
  uint32_t old;
  asm volatile("atom.global.sys.or.b32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ uint64_t gs_atomic_min_sys(uint64_t* p, uint64_t v) {
  unsigned long long old;
  asm volatile("atom.global.sys.min.u64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"((unsigned long long)v) : "memory");
  return old;
}
// Mailbox deliveries of a sharded pool are system-scope REDUCTIONS — nobody needs the old value, so none
// travels back over NVLink (half the traffic of a fetching atomic; 2 GPUs: 98 -> 77 us per cascade tick); the
// issuing thread's fence.sys before the inter-tick release is what orders them.  GSIM_FLAG_SHARD_ATOM (128)
// keeps the fetching form for comparison.
__device__ __forceinline__ void gs_red_or_sys(uint32_t* p, uint32_t v) {
  asm volatile("red.global.sys.or.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// (`g` is the GsGlobals in scope at every use: single-GPU pools keep the cheap device-scope forms)
#define GS_ATOMIC_OR32(p, v) (g.world > 1u ? gs_atomic_or_sys((p), (v)) : atomicOr((p), (v)))
#define GS_POST_OR32(p, v)                                                         \
  do {                                                                             \
    if (g.world <= 1u) (void)atomicOr((p), (v));                                   \
    else if (g.flags & 128u) (void)gs_atomic_or_sys((p), (v));                     \
    else gs_red_or_sys((p), (v));                                                  \
  } while (0)
#define GS_ATOMIC_MIN64(p, v)                                                    \
  (g.world > 1u ? gs_atomic_min_sys((uint64_t*)(p), (uint64_t)(v))               \
                : (uint64_t)atomicMin((unsigned long long*)(p), (unsigned long long)(v)))
// Reads of OTHER members' columns go to L2 (ld.global.cg): on a sharded pool the line may live
// on another GPU, and an L1 copy of a peer line is not something to rely on across ticks.
__device__ __forceinline__ uint32_t gs_ld_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint64_t gs_ld_sys64(const uint64_t* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
#define GS_LD_OTHER(p) __ldcg(p)
#define GS_LD_OTHER64(p) gs_ld_sys64(p)
// push-pull mailboxes: requester ids (min chain) and Lamport clocks (max), same scoping rule
__device__ __forceinline__ uint32_t gs_atomic_min32_sys(uint32_t* p, uint32_t v) {
  uint32_t old;
  asm volatile("atom.global.sys.min.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ uint32_t gs_atomic_max32_sys(uint32_t* p, uint32_t v) {
  uint32_t old;
  asm volatile("atom.global.sys.max.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
#define GS_ATOMIC_MIN32(p, v) (g.world > 1u ? gs_atomic_min32_sys((p), (v)) : atomicMin((p), (v)))
#define GS_ATOMIC_MAX32(p, v) (g.world > 1u ? gs_atomic_max32_sys((p), (v)) : atomicMax((p), (v)))
#else
#define GS_DEV inline
#define GS_ATOMIC_OR32(p, v) __atomic_fetch_or((p), (v), __ATOMIC_RELAXED)
#define GS_POST_OR32(p, v) (void)__atomic_fetch_or((p), (v), __ATOMIC_RELAXED)
static inline uint64_t gs_host_atomic_min64(uint64_t* p, uint64_t v) {
  uint64_t old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (old > v && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED,
                                                 __ATOMIC_RELAXED)) {
  }
  return old;
}
#define GS_ATOMIC_MIN64(p, v) gs_host_atomic_min64((uint64_t*)(p), (uint64_t)(v))
static inline uint32_t gs_host_atomic_min32(uint32_t* p, uint32_t v) {
  uint32_t old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (old > v && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return old;
}
static inline uint32_t gs_host_atomic_max32(uint32_t* p, uint32_t v) {
  uint32_t old = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (old < v && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  return old;
}
#define GS_ATOMIC_MIN32(p, v) gs_host_atomic_min32((p), (v))
#define GS_ATOMIC_MAX32(p, v) gs_host_atomic_max32((p), (v))
#define GS_LD_OTHER(p) (*(p))
#define GS_LD_OTHER64(p) (*(p))
#endif

// Stat indices (mirror GSIM_STAT_* in include/gsim.h).
enum {
  GS_ST_PROBES = 0,
  GS_ST_ACKS,
  GS_ST_INDIRECT_PINGS,
  GS_ST_NACKS,
  GS_ST_PROBE_FAILURES,
  GS_ST_SUSPECTS,
  GS_ST_CONFIRMATIONS,
  GS_ST_DEADS,
  GS_ST_REFUTES,
  GS_ST_GOSSIP_PACKETS,
  GS_ST_RUMORS_SENT,
  GS_ST_RUMORS_ACCEPTED,
  GS_ST_RUMORS_DROPPED,
  GS_ST_PACKETS_LOST,
  GS_ST_ACTIVE_ROWS,
  GS_ST_PUSH_PULLS
};

// The key column is the one column every member reads about every other member (probe targets,
// gossip peers, relays).  On a sharded pool each GPU keeps a full replica so those gathers stay
// in local HBM; a key changes rarely (suspect, dead, refute, join), and whoever changes it
// writes all replicas (remote stores over NVLink, ordered by the closing fence.sys).
GS_DEV void gs_key_store(const GsDev& d, const GsGlobals& g, uint32_t buf, uint32_t i, uint32_t k) {
  if (d.kst != nullptr) {  // the member's status byte: only its owner (or the host) ever writes it
    const uint32_t b = d.kst[i], code = gs_kst_code(k);
    d.kst[i] = (uint8_t)(buf ? ((b & 0x0Fu) | (code << 4)) : ((b & 0xF0u) | code));
  }
  if (g.world <= 1u) {
    d.key[buf][i] = k;
    return;
  }
  for (uint32_t r = 0; r < g.world; ++r) d.key_rep[buf][(size_t)r * g.key_stride + i] = k;
}

// What member c looks like to its peers in buffer `cur`.  Peer selection needs truth and rank only,
// so it is answered from the status byte (1 B per member: 64 MB at 64 Mi members, L2-resident, where
// a random 4-byte gather from the 256 MB key column costs a DRAM sector each) — inc reads as 0,
// pending as 0 — unless the member is a pending joiner; a caller that needs the incarnation asks
// for the full key.  Measured (profiles/README.md r2a): 234 -> 188 us/tick at 64 Mi members.
GS_DEV uint32_t gs_peer_key(const GsDev& d, uint32_t cur, uint32_t c, bool need_inc) {
  if (d.kst != nullptr && !need_inc) {
#if defined(__CUDA_ARCH__)
    const uint32_t b = __ldcg(reinterpret_cast<const unsigned char*>(d.kst) + c);
#else
    const uint32_t b = d.kst[c];
#endif
    const uint32_t code = (b >> (cur * 4u)) & 15u;
    if (code != GS_KST_PENDING) return code;
  }
  return GS_LD_OTHER(&d.key[cur][c]);
}

// Deliver `bits` into member j's mailbox word of arrival slot `slot` (commutative).
template <class Sink>
GS_DEV void gs_post(const GsDev& d, const GsGlobals& g, Sink& sink, uint32_t slot, uint32_t j, uint32_t bits) {
  sink.activity();  // a posted word is mail at its arrival tick: the pool is not quiet (DESIGN.md §4.2)
  GS_POST_OR32(&d.inbox[slot][j], bits);
}

// incarnation of peer c whose key-like word k came from gs_peer_key(..., false)
#define GS_PEER_INC(d, cur, c, k) gs_key_inc(gs_peer_key((d), (cur), (c), true))

// WAN latency pools (BASELINE config 5): EXTRA one-way latency in ticks from src to dst on top
// of the one tick every packet takes; 0 everywhere on a pool without datacenters.  An all-zero
// matrix is indistinguishable from n_dcs == 0 (tests/test_latency_cpu.py).
// The pool constants the probe fast path reads, copied out of the device-resident GsGlobals once per
// launch: they are warp-uniform, so they sit in (uniform) registers instead of costing a global load
// each time the 32 members of a group ask for them.  Same field names as GsGlobals: the fast-path
// functions are templates over "something with these fields".
struct GsHot {
  uint32_t n, P, T, seed_lo, seed_hi, perm_bits, loss_thr, graph_n, pp_interval, rot_pp, phase_group, n_dcs;
  const uint8_t* lat;
};
GS_DEV GsHot gs_hot(const GsGlobals& g) {
  GsHot h;
  h.n = g.n; h.P = g.P; h.T = g.T; h.seed_lo = g.seed_lo; h.seed_hi = g.seed_hi;
  h.perm_bits = g.perm_bits; h.loss_thr = g.loss_thr; h.graph_n = g.graph_n;
  h.pp_interval = g.pp_interval; h.rot_pp = g.rot_pp; h.phase_group = g.phase_group; h.n_dcs = g.n_dcs;
  h.lat = g.lat;
  return h;
}

template <class G>
GS_DEV uint32_t gs_extra(const G& g, uint32_t src, uint32_t dst) {
  if (g.n_dcs == 0u) return 0u;
  return g.lat[((src / GS_TILE) % g.n_dcs) * GS_MAX_DCS + (dst / GS_TILE) % g.n_dcs];
}

// Same draw as gs_lost without touching the counters: re-evaluates, at the ProbeTimeout stage,
// whether the direct ping/ack of the probe started at t0 were lost (late acks, latency pools).
GS_DEV bool gs_lost_quiet(const GsGlobals& g, uint32_t src, uint32_t dst, uint32_t t, uint32_t kind,
                          uint32_t idx) {
  if (g.loss_thr == 0u) return false;
  GsU4 r = gs_philox(g.seed_lo, g.seed_hi, src, dst, t, GS_PUR_LOSS | (kind << 8) | (idx << 16));
  return r.x < g.loss_thr;
}

// One simulated UDP packet is lost iff its Philox draw is below the threshold.
template <class Sink>
GS_DEV bool gs_lost(const GsGlobals& g, Sink& sink, uint32_t src, uint32_t dst, uint32_t t,
                    uint32_t kind, uint32_t idx) {
  if (g.loss_thr == 0u) return false;
  GsU4 r = gs_philox(g.seed_lo, g.seed_hi, src, dst, t, GS_PUR_LOSS | (kind << 8) | (idx << 16));
  bool lost = r.x < g.loss_thr;
  if (lost) sink.stat(GS_ST_PACKETS_LOST, 1);
  return lost;
}

// Does member i know member c exists?  Established members are known to everyone; a
// pending joiner is known only to members that have heard its alive rumor.
GS_DEV bool gs_knows(const GsDev& d, const GsGlobals& g, uint32_t i, uint32_t c, uint32_t kc,
                     uint32_t meta_i) {
  if (c == i) return true;
  // a member that has not joined anyone yet knows nobody but itself and what it heard
  if (!gs_key_pending(kc)) return !(meta_i & GS_META_ISOLATED);
  const uint32_t heard_i = d.heard[i];  // rare: only pending joiners reach this point
  uint32_t am = g.class_mask[0] & g.active_mask;
  while (am) {
#if defined(__CUDA_ARCH__)
    uint32_t r = __ffs(am) - 1;
#else
    uint32_t r = (uint32_t)__builtin_ctz(am);
#endif
    am &= am - 1;
    if (g.rumors[r].kind == GS_RUMOR_ALIVE && g.rumors[r].subject == c) return (heard_i >> r) & 1u;
  }
  return false;
}

// The member list of member i as a sequence: the complete graph [0, n) by default, row i of the
// CSR peer graph when one is set.  Same draws, same ring — only the index space changes, so a CSR
// whose rows are all [0, n) reproduces the complete-graph results exactly.
GS_DEV uint32_t gs_peer_count(const GsDev& d, const GsGlobals& g, uint32_t i) {
  if (g.graph_n == 0u) return g.n;
  return i < g.graph_n ? d.row_ptr[i + 1u] - d.row_ptr[i] : 0u;
}
GS_DEV uint32_t gs_peer_at(const GsDev& d, const GsGlobals& g, uint32_t i, uint32_t idx) {
  return g.graph_n == 0u ? idx : d.col_idx[d.row_ptr[i] + idx];
}

// ---- network coordinates: slot selection and the update on a direct ack (gs_coord.h) ---------
GS_DEV uint32_t gs_coord_slot_for_reader(const uint32_t* ctag, size_t cap, uint32_t j, uint32_t t) {
  const uint32_t a = GS_LD_OTHER(&ctag[j]), b = GS_LD_OTHER(&ctag[cap + j]);
  // a slot is readable at tick t if it was written before t (tag = tick + 1 <= t); newer wins
  return (b <= t && (a > t || b > a)) ? 1u : 0u;
}
GS_DEV void gs_coord_load(const double* coord, size_t cap, uint32_t slot, uint32_t j, GsCoord& c) {
  const double* base = coord + ((size_t)slot * GS_COORD_WORDS) * cap + j;
  double w[GS_COORD_WORDS];
  for (uint32_t x = 0; x < GS_COORD_WORDS; ++x) {
    const uint64_t bits = GS_LD_OTHER64(reinterpret_cast<const uint64_t*>(base + (size_t)x * cap));
    memcpy(&w[x], &bits, 8);
  }
  for (uint32_t x = 0; x < GS_COORD_DIM; ++x) c.vec[x] = w[x];
  c.error = w[8];
  c.adjustment = w[9];
  c.height = w[10];
}
// [U] serf/ping_delegate.go NotifyPingComplete -> coordinate.Client.Update: member i got a direct
// ack from j at tick t.
// (out of line on the device: ~150 double-precision operations must not cost the tick kernel's hot
// path a single register)
#if defined(__CUDA_ARCH__)
__device__ __noinline__
#else
inline
#endif
void gs_coord_on_ack(double* coord, uint32_t* ctag, double* adj, uint32_t* adj_idx, const GsGlobals& g, uint32_t i,
                     uint32_t j, uint32_t t) {  // (column pointers by value: taking the address of the
                                                 // kernel's GsDev parameter would copy it to the stack)
  const size_t cap = g.cap;
  const uint32_t ta = ctag[i], tb = ctag[cap + i];
  const uint32_t mine = tb > ta ? 1u : 0u, spare = mine ^ 1u;  // the owner overwrites its OLDER slot
  GsCoord c, other;
  gs_coord_load(coord, cap, mine, i, c);
  gs_coord_load(coord, cap, gs_coord_slot_for_reader(ctag, cap, j, t), j, other);
  const double rtt = g.coord_base_rtt_s + (double)(gs_extra(g, i, j) + gs_extra(g, j, i)) * g.tick_seconds;
  uint32_t idx = adj_idx[i];
  gs_coord_client_update(c, other, rtt, adj + i, cap, &idx, g.seed_lo, g.seed_hi, i, t);
  adj_idx[i] = idx;
  double* out = coord + ((size_t)spare * GS_COORD_WORDS) * cap + i;
  for (uint32_t x = 0; x < GS_COORD_DIM; ++x) out[(size_t)x * cap] = c.vec[x];
  out[(size_t)8 * cap] = c.error;
  out[(size_t)9 * cap] = c.adjustment;
  out[(size_t)10 * cap] = c.height;
  ctag[(size_t)spare * cap + i] = t + 1u;
}

// kRandomNodes ([U] memberlist/util.go): up to min(3n, 32) uniform draws `rand % n`,
// rejecting excluded members and duplicates.  mode 0 = gossip targets (alive, suspect,
// or dead for less than GossipToTheDeadTime), mode 1 = indirect-probe relays (alive only).
GS_DEV uint32_t gs_krandom(const GsDev& d, const GsGlobals& g, uint32_t i, uint32_t t,
                           uint32_t purpose, uint32_t k, uint32_t mode, uint32_t exclude2,
                           uint32_t meta_i, uint32_t* out) {
  const uint32_t n = gs_peer_count(d, g, i);
  if (n == 0u) return 0u;
  uint32_t tries = 3u * n;
  if (tries > GS_KR_MAX_TRIES || n > 0x55555555u) tries = GS_KR_MAX_TRIES;
  uint32_t cnt = 0;
  // One Philox block = four draws.  Their candidates and the candidates' status words are fetched
  // together (four independent gathers in flight instead of a chain of dependent ones); the draws
  // are then judged strictly in order, exactly like the sequential loop — a fetched status that
  // turns out not to be needed (enough peers already) was only read.
  for (uint32_t b4 = 0; b4 * 4u < tries && cnt < k; ++b4) {
    const GsU4 blk = gs_philox(g.seed_lo, g.seed_hi, i, t, purpose, b4);
    uint32_t cc[4], kk[4];
#pragma unroll
    for (uint32_t x = 0; x < 4u; ++x) {
      const uint32_t draw = gs_u4_get(blk, x);
      cc[x] = gs_peer_at(d, g, i, g.graph_n == 0u ? gs_fastmod(draw, n, g.n_magic) : draw % n);
      kk[x] = (b4 * 4u + x < tries && cc[x] != i && cc[x] != exclude2) ? gs_peer_key(d, t & 1u, cc[x], false) : 0u;
    }
#pragma unroll
    for (uint32_t x = 0; x < 4u; ++x) {
      if (!(b4 * 4u + x < tries && cnt < k)) continue;
      const uint32_t c = cc[x], kc = kk[x];
      if (c == i || c == exclude2) continue;
      if (gs_key_truth(kc) == GS_TRUTH_NONE) continue;
      const uint32_t rank = gs_key_rank(kc);
      if (mode == 1u) {
        if (rank != GS_RANK_ALIVE) continue;
      } else {
        if (rank == GS_RANK_LEFT) continue;
        if (rank == GS_RANK_DEAD && (t - GS_LD_OTHER(&d.change_tick[c])) > g.gtd_ticks) continue;
      }
      if (!gs_knows(d, g, i, c, kc, meta_i)) continue;
      bool dup = false;
      for (uint32_t q = 0; q < cnt; ++q) dup = dup || (out[q] == c);
      if (dup) continue;
      out[cnt++] = c;
    }
  }
  return cnt;
}

// TransmitLimitedQueue.GetBroadcasts ([U] memberlist/queue.go) for one packet: walk the
// member's queued rumors by (queue class, transmits asc, size desc, slot desc) and take
// every message that still fits the UDP budget.  Class order = memberlist broadcasts,
// then serf intents, then serf user events ([U] serf/delegate.go GetBroadcasts).
GS_DEV uint32_t gs_select_packet(const GsDev& d, const GsGlobals& g, uint32_t i, uint32_t queued) {
  if (g.active_bytes <= g.udp_avail) return queued;  // every tracked broadcast together fits one packet
  uint32_t total = 0, qm = queued;
  while (qm) {
#if defined(__CUDA_ARCH__)
    uint32_t r = __ffs(qm) - 1;
#else
    uint32_t r = (uint32_t)__builtin_ctz(qm);
#endif
    qm &= qm - 1;
    total += g.rumors[r].size + (g.rumors[r].qclass ? 3u : 2u);
  }
  if (total <= g.udp_avail) return queued;  // everything fits: the common case
  uint32_t used = 0, mask = 0;
  for (uint32_t cls = 0; cls < 3; ++cls) {
    uint32_t cm = queued & g.class_mask[cls];
    const uint32_t ovh = cls ? 3u : 2u;
    while (cm) {
      if (g.udp_avail <= used + ovh) break;
      const uint32_t free_b = g.udp_avail - used - ovh;
      uint32_t best = GS_EMPTY32, best_key = GS_EMPTY32, scan = cm;
      while (scan) {
#if defined(__CUDA_ARCH__)
        uint32_t r = __ffs(scan) - 1;
#else
        uint32_t r = (uint32_t)__builtin_ctz(scan);
#endif
        scan &= scan - 1;
        uint32_t sz = g.rumors[r].size;
        if (sz > free_b) continue;
        uint32_t tx = d.tx[GS_TX(r, g.cap, i)];
        uint32_t key = (tx << 24) | ((0xFFFFu - (sz & 0xFFFFu)) << 8) | (31u - r);
        if (key < best_key) {
          best_key = key;
          best = r;
        }
      }
      if (best == GS_EMPTY32) break;
      mask |= 1u << best;
      cm &= ~(1u << best);
      used += ovh + g.rumors[best].size;
    }
  }
  return mask;
}

template <class Sink>
GS_DEV void gs_log_event(const GsDev& d, const GsGlobals& g, Sink& sink, uint32_t t, uint32_t type,
                         uint32_t subject, uint32_t observer, uint32_t ltime) {
  sink.log_event(d, g, t, type, subject, observer, ltime);
}

// Tile-level gate: can any member of this tile have a probe action due at tick t?  A
// member's `due` is always congruent to its ticker phase or to phase + ProbeTimeout
// (mod ProbeInterval), and phases are uniform per tile, so 1 - 2/P of the tiles never
// need to read the `due` column at all.
// pslot = t % P; pslot_t = (t - T) % P, i.e. the phase whose ProbeTimeout stage is due now.
GS_DEV bool gs_tile_probe_gate(const GsGlobals& g, uint32_t tile, uint32_t pslot, uint32_t pslot_t) {
  if (!g.phase_gate) return true;
  const uint32_t group = tile >> g.phase_shift;  // phase_group = 128 << phase_shift
  const uint32_t pp = gs_probe_phase(g.rot_p, group, g.P);
  return pp == pslot || pp == pslot_t;
}

// The tick of member i, called only for rows that have mail (inb = inbox[t&1][i] != 0,
// which includes the self-posted wake bit) or a probe action due (due[i] == t).
template <class Sink>
GS_DEV void gs_row_step(const GsDev& d, const GsGlobals& g, uint32_t i, uint32_t t, uint32_t gslot,
                        uint32_t inb, Sink& sink) {
  const uint32_t cur = t & 1u, nxt = cur ^ 1u;                            // key / acc buffers
  const uint32_t icur = t & g.ring_mask, inxt = (t + 1u) & g.ring_mask;  // mailbox ring slots
  const uint32_t k0 = d.key[cur][i];
  const uint32_t truth = gs_key_truth(k0);
  if (inb != 0u) sink.activity();
  if (truth == GS_TRUTH_NONE) {
    // no such member (never created, or reaped with packets still in flight): the mail is dropped,
    // otherwise the word would keep its tile in the active set for ever
    if (inb != 0u) d.inbox[icur][i] = 0u;
    return;
  }
  const uint32_t m0 = d.meta[i];
  const uint32_t due0 = d.due[i];
  const bool up = truth == GS_TRUTH_UP;
  const bool gossip_slot = up && gslot == gs_meta_gphase(m0);  // gslot = t % GI
  uint32_t queued = up ? d.queued[i] : 0u;
  if (inb != 0u) d.inbox[icur][i] = 0u;
  sink.stat(GS_ST_ACTIVE_ROWS, 1);  // scheduling diagnostic: rows that left the 4-byte scan
  // periodic push-pull (opt-in): does this member's push-pull ticker fire now?
  const bool pp_now = up && g.pp_interval != 0u && gs_pp_due(g.pp_interval, g.rot_pp, i / g.phase_group, t);

  // ---- nothing to do this tick (a wake that only keeps the row in the active set) ----
  if ((inb & ~GS_WAKE_BIT) == 0u && gs_key_rank(k0) == GS_RANK_ALIVE && !(up && due0 == t) &&
      !(gossip_slot && queued != 0u) && !pp_now) {
    if (m0 & GS_META_DIRTY) {  // bring the other key buffer up to date
      gs_key_store(d, g, nxt, i, k0);
      d.meta[i] = m0 & ~GS_META_DIRTY;
    }
    if (queued != 0u) gs_post(d, g, sink, inxt, i, GS_WAKE_BIT);
    return;
  }

  uint32_t k = k0, m = m0, due = due0;
  const size_t cap = g.cap;
  uint32_t heard = 0;

  // ---- A. consume the mailbox of this arrival tick ------------------------------
  if ((inb & ~GS_WAKE_BIT) != 0u) {
    if ((inb & GS_ACC_BIT) && g.pp_interval != 0u) {
      // [U] serf/delegate.go MergeRemoteState: witness the push-pull partners' clocks first
      // (Witness(remote - 1) == max(local, remote)), then replay what they carried.
      uint32_t* clk = d.pp_clk + (size_t)cur * 2u * cap;
      const uint32_t cm = GS_LD_OTHER(&clk[i]), ce = GS_LD_OTHER(&clk[cap + i]);
      if (cm | ce) {
        clk[i] = 0u;
        clk[cap + i] = 0u;
        if (up) {
          if (cm > d.ltime_member[i]) d.ltime_member[i] = cm;
          if (ce > d.ltime_event[i]) d.ltime_event[i] = ce;
        }
      }
    }
    uint32_t rbits = inb & ~(GS_ACC_BIT | GS_WAKE_BIT) & g.active_mask;
    if (rbits && up) {
      heard = d.heard[i];
      uint32_t fresh = rbits & ~heard;
      uint32_t accepted = 0;
      while (fresh) {
#if defined(__CUDA_ARCH__)
        uint32_t r = __ffs(fresh) - 1;
#else
        uint32_t r = (uint32_t)__builtin_ctz(fresh);
#endif
        fresh &= fresh - 1;
        const GsRumor& ru = g.rumors[r];
        bool accept = true;
        if (ru.kind == GS_RUMOR_USER_EVENT) {
          // [U] serf.handleUserEvent: Witness, then eventMinTime and buffer-window checks.
          uint32_t c = d.ltime_event[i];
          if (ru.ltime >= c) {
            c = ru.ltime + 1u;
            d.ltime_event[i] = c;
          }
          if (ru.ltime < d.event_min[i]) accept = false;
          else if (c > g.event_buffer && ru.ltime < c - g.event_buffer) accept = false;
          if (accept && (m & GS_META_WATCHED))
            gs_log_event(d, g, sink, t, GS_EV_USER, r, i, ru.ltime);
        } else if (ru.kind == GS_RUMOR_JOIN_INTENT || ru.kind == GS_RUMOR_LEAVE_INTENT) {
          // [U] serf.handleNodeJoinIntent / handleNodeLeaveIntent: clock.Witness(LTime).
          uint32_t c = d.ltime_member[i];
          if (ru.ltime >= c) d.ltime_member[i] = ru.ltime + 1u;
        } else if (ru.kind == GS_RUMOR_ALIVE) {
          // [U] memberlist.aliveNode for a new node -> serf.handleNodeJoin -> EventMemberJoin.
          if (m & GS_META_WATCHED) gs_log_event(d, g, sink, t, GS_EV_MEMBER_JOIN, ru.subject, i, 0u);
        } else if (ru.kind == GS_RUMOR_UPDATE) {
          // [U] memberlist.aliveNode with a higher incarnation and new meta -> NotifyUpdate ->
          // serf.handleNodeUpdate -> EventMemberUpdate ((*Serf).SetTags at the subject).
          if (m & GS_META_WATCHED) gs_log_event(d, g, sink, t, GS_EV_MEMBER_UPDATE, ru.subject, i, 0u);
        }
        if (accept) {
          accepted |= 1u << r;
          d.tx[GS_TX(r, cap, i)] = 0;  // queued with transmits = 0
          sink.heard(r);
          sink.stat(GS_ST_RUMORS_ACCEPTED, 1);
        } else {
          sink.stat(GS_ST_RUMORS_DROPPED, 1);
        }
      }
      if (accepted) {
        d.heard[i] = heard | accepted;
        queued |= accepted;
        d.queued[i] = queued;
      }
    }
    if (inb & GS_ACC_BIT) {
      // [U] memberlist.suspectNode, subject side.  Entries are (~inc<<32 | from), sorted.
      uint64_t* acc = d.acc + (size_t)cur * GS_K1MAX * cap;
      for (uint32_t s = 0; s < GS_K1MAX; ++s) {
        uint64_t e = GS_LD_OTHER64(&acc[(size_t)s * cap + i]);  // written by accusers anywhere
        if (e == GS_EMPTY64) break;
        acc[(size_t)s * cap + i] = GS_EMPTY64;
        uint32_t e_inc = ~(uint32_t)(e >> 32), from = (uint32_t)e;
        if (e_inc != gs_key_inc(k)) continue;  // older incarnation: ignored
        uint32_t rank = gs_key_rank(k);
        if (rank == GS_RANK_ALIVE) {
          k = gs_key_with_rank(k, GS_RANK_SUSPECT);
          d.sus_start[i] = t - 1u;  // the accuser started its timer when it sent
          d.sus_from[i] = from;
          for (uint32_t q = 1; q < GS_K1MAX; ++q) d.sus_from[(size_t)q * cap + i] = GS_EMPTY32;
          sink.stat(GS_ST_SUSPECTS, 1);
        } else if (rank == GS_RANK_SUSPECT) {
          // suspicion.Confirm: distinct `from`, at most k confirmations are counted
          for (uint32_t q = 0; q <= g.sus_k && q < GS_K1MAX; ++q) {
            uint32_t f = d.sus_from[(size_t)q * cap + i];
            if (f == from) break;
            if (f == GS_EMPTY32) {
              d.sus_from[(size_t)q * cap + i] = from;
              sink.stat(GS_ST_CONFIRMATIONS, 1);
              break;
            }
          }
        }
      }
    }
    if ((inb & GS_ACC_BIT) && g.pp_interval != 0u) {
      // [U] memberlist/net.go handleConn(pushPullMsg) -> sendLocalState: answer every partner that
      // opened a push-pull with what this member holds now (after merging what they pushed).
      uint32_t* req = d.ppreq + (size_t)cur * GS_PPK * cap;
      for (uint32_t s = 0; s < GS_PPK; ++s) {
        const uint32_t from = GS_LD_OTHER(&req[(size_t)s * cap + i]);
        if (from == GS_EMPTY32) break;
        req[(size_t)s * cap + i] = GS_EMPTY32;
        if (!up) continue;  // a dead process accepts no connection
        uint32_t* clk = d.pp_clk + (size_t)nxt * 2u * cap;
        GS_ATOMIC_MAX32(&clk[from], d.ltime_member[i]);
        GS_ATOMIC_MAX32(&clk[cap + from], d.ltime_event[i]);
        gs_post(d, g, sink, inxt, from, (d.heard[i] & g.active_mask) | GS_ACC_BIT);
      }
    }
  }

  // ---- B. the member's own view transitions -------------------------------------
  {
    uint32_t rank = gs_key_rank(k);
    if (up && !(m & GS_META_LEAVING) && (rank == GS_RANK_SUSPECT || rank == GS_RANK_DEAD)) {
      // [U] memberlist.refute: bump past the accused incarnation, awareness +1,
      // broadcast alive (instantly visible in the shared view).
      uint32_t inc = gs_key_inc(k);
      uint32_t accused = inc;
      inc = inc + 1u;
      if (accused >= inc) inc = accused + 1u;
      k = gs_key_with_rank(gs_key_with_inc(k, inc), GS_RANK_ALIVE);
      uint32_t aw = gs_meta_aw(m) + 1u;
      if (aw > g.awareness_max - 1u) aw = g.awareness_max - 1u;
      m = gs_meta_set_aw(m, aw);
      sink.stat(GS_ST_REFUTES, 1);
    } else if (rank == GS_RANK_SUSPECT) {
      // [U] suspicion timer: fires at start + timeout(confirmations)
      uint32_t c = 0;
      for (uint32_t q = 1; q <= g.sus_k && q < GS_K1MAX; ++q)
        c += d.sus_from[(size_t)q * cap + i] != GS_EMPTY32;
      if (t - d.sus_start[i] >= g.sus_ticks[c]) {
        k = gs_key_with_rank(k, GS_RANK_DEAD);  // [U] memberlist.deadNode
        d.change_tick[i] = t;
        sink.stat(GS_ST_DEADS, 1);
        if (truth == GS_TRUTH_CRASHED) sink.crashed_dead(d, t);
        if (g.flags & 1u) gs_log_event(d, g, sink, t, GS_EV_MEMBER_FAILED, i, GS_EMPTY32, 0u);
      }
    }
  }

  if (up) {
    // ---- C. failure detector: this member as prober ------------------------------
    uint32_t stage = gs_meta_stage(m);
    if (stage == GS_STAGE_WAIT_T && due == t) {
      // ProbeTimeout elapsed without a direct ack: k indirect probes + TCP fallback.
      const uint32_t j = d.probe_tgt[i];
      const uint32_t kj = gs_peer_key(d, cur, j, false);
      const bool j_up = gs_key_truth(kj) == GS_TRUTH_UP;
      uint32_t relays[8];
      uint32_t kk = g.indirect_checks > 8u ? 8u : g.indirect_checks;
      uint32_t nr = gs_krandom(d, g, i, t, GS_PUR_RELAY, kk, 1u, j, m, relays);
      bool success = false;
      uint32_t nacks = 0;
      // Latency pools: whatever comes back must arrive before the probe deadline, i.e. within
      // `budget` ticks of extra latency from now (t0 + P*(awareness+1) - (t0 + T)).
      const uint32_t budget = g.P * (gs_meta_aw(m) + 1u) - g.T;
      for (uint32_t q = 0; q < nr; ++q) {
        const uint32_t r = relays[q];
        const bool r_up = gs_key_truth(gs_peer_key(d, cur, r, false)) == GS_TRUTH_UP;
        sink.stat(GS_ST_INDIRECT_PINGS, 1);
        if (!(r_up && !gs_lost(g, sink, i, r, t, GS_LK_INDREQ, q))) continue;  // no nack either
        const uint32_t via = gs_extra(g, i, r) + gs_extra(g, r, i);
        const uint32_t rtt_rj = gs_extra(g, r, j) + gs_extra(g, j, r);
        // the relay waits ProbeTimeout for the target's ack, then answers with a nack
        bool relay_acked = j_up && !gs_lost(g, sink, r, j, t, GS_LK_INDPING, q) &&
                           !gs_lost(g, sink, j, r, t, GS_LK_INDACK, q) && rtt_rj <= g.T;
        if (relay_acked) {
          if (!gs_lost(g, sink, r, i, t, GS_LK_INDFWD, q) && via + rtt_rj <= budget) success = true;
        } else if (!gs_lost(g, sink, r, i, t, GS_LK_NACK, q) && via <= budget) {
          ++nacks;
          sink.stat(GS_ST_NACKS, 1);
        }
      }
      const uint32_t t0 = t - g.T;
      const uint32_t rtt_ij = gs_extra(g, i, j) + gs_extra(g, j, i);
      if (!g.disable_tcp && j_up && rtt_ij <= budget) success = true;  // TCP fallback ping is reliable
      // a direct ack that was merely slower than ProbeTimeout still counts until the deadline
      if (g.n_dcs != 0u && j_up && rtt_ij > g.T && rtt_ij <= budget + g.T &&
          !gs_lost_quiet(g, i, j, t0, GS_LK_PING, 0) && !gs_lost_quiet(g, j, i, t0, GS_LK_ACK, 0))
        success = true;
      if (success) {
        uint32_t aw = gs_meta_aw(m);
        m = gs_meta_set_aw(m, aw ? aw - 1u : 0u);
        m = gs_meta_set_stage(m, GS_STAGE_IDLE);
        due = t0 + g.P;
        sink.stat(GS_ST_ACKS, 1);
      } else {
        uint32_t miss = nr > 0u ? nr - nacks : 1u;
        if (miss > 7u) miss = 7u;  // 3-bit field; awareness saturates at <= 7, so 8 misses change nothing
        m = gs_meta_set_nmiss(gs_meta_set_stage(m, GS_STAGE_WAIT_P), miss);
        due = t0 + g.P * (gs_meta_aw(m) + 1u);
      }
      stage = gs_meta_stage(m);
    }
    if (stage == GS_STAGE_WAIT_P && due == t) {
      // probe deadline: awareness += missed nacks, then suspectNode(target)
      uint32_t aw = gs_meta_aw(m) + gs_meta_nmiss(m);
      if (aw > g.awareness_max - 1u) aw = g.awareness_max - 1u;
      m = gs_meta_set_stage(gs_meta_set_aw(m, aw), GS_STAGE_IDLE);
      const uint32_t j = d.probe_tgt[i];
      const uint64_t e = ((uint64_t)(~d.probe_inc[i]) << 32) | (uint64_t)i;
      uint64_t* acc = d.acc + (size_t)nxt * GS_K1MAX * cap;
      uint64_t v = e;
      for (uint32_t s = 0; s < GS_K1MAX; ++s) {
        uint64_t old = GS_ATOMIC_MIN64(&acc[(size_t)s * cap + j], v);
        if (old == v || old == GS_EMPTY64) break;
        if (old > v) v = old;  // displaced a larger entry: carry it to the next slot
      }
      gs_post(d, g, sink, inxt, j, GS_ACC_BIT);
      sink.stat(GS_ST_PROBE_FAILURES, 1);
      stage = GS_STAGE_IDLE;  // due == t: the buffered ticker fires immediately
    }
    if (stage == GS_STAGE_IDLE && due == t) {
      // [U] memberlist.probe: next eligible entry of the ring, skipping self, unknown and
      // dead/left members; a wrap re-keys the permutation (resetNodes + shuffle).
      uint32_t cursor = d.cursor[i], pass = d.pass[i];
      const uint32_t n = gs_peer_count(d, g, i);
      const uint32_t hb = g.graph_n == 0u ? g.perm_bits : gs_perm_bits_of(n);
      GsU4 rk = gs_perm_keys(g.seed_lo, g.seed_hi, i, pass);
      uint32_t checked = 0, target = GS_EMPTY32, ktarget = 0;
      const uint32_t limit = n < GS_PROBE_SKIP_CAP ? n : GS_PROBE_SKIP_CAP;
      while (checked < limit) {
        if (cursor >= n) {
          cursor = 0;
          ++pass;
          ++checked;
          rk = gs_perm_keys(g.seed_lo, g.seed_hi, i, pass);
          continue;
        }
        uint32_t c = gs_peer_at(d, g, i, gs_perm(cursor, n, hb, rk));
        ++cursor;
        uint32_t kc = gs_peer_key(d, cur, c, false);
        uint32_t rank = gs_key_rank(kc);
        if (c == i || gs_key_truth(kc) == GS_TRUTH_NONE || rank == GS_RANK_DEAD ||
            rank == GS_RANK_LEFT || !gs_knows(d, g, i, c, kc, m)) {
          ++checked;
          continue;
        }
        target = c;
        ktarget = kc;
        break;
      }
      d.cursor[i] = cursor;
      d.pass[i] = pass;
      if (target != GS_EMPTY32) {
        sink.stat(GS_ST_PROBES, 1);
        bool ok = gs_key_truth(ktarget) == GS_TRUTH_UP && !gs_lost(g, sink, i, target, t, GS_LK_PING, 0) &&
                  !gs_lost(g, sink, target, i, t, GS_LK_ACK, 0) &&
                  gs_extra(g, i, target) + gs_extra(g, target, i) <= g.T;  // ack within ProbeTimeout
        if (ok) {
          uint32_t aw = gs_meta_aw(m);
          m = gs_meta_set_aw(m, aw ? aw - 1u : 0u);
          due = t + g.P;
          sink.stat(GS_ST_ACKS, 1);
          if constexpr (Sink::kCoords) {  // the ack carries the peer's coordinate
            if (d.coord != nullptr) gs_coord_on_ack(d.coord, d.ctag, d.adj, d.adj_idx, g, i, target, t);
          }
        } else {
          m = gs_meta_set_stage(m, GS_STAGE_WAIT_T);
          d.probe_tgt[i] = target;
          d.probe_inc[i] = GS_PEER_INC(d, cur, target, ktarget);  // the incarnation it will accuse
          due = t + g.T;
          sink.horizon(t + g.P);  // the earliest tick this probe can end in an accusation
        }
      } else {
        due = t + g.P;
      }
    }

    // ---- D. gossip: drain the broadcast queue to GossipNodes random peers ----------
    if (gossip_slot && queued != 0u) {
      uint32_t peers[8];
      uint32_t kk = g.gossip_nodes > 8u ? 8u : g.gossip_nodes;
      uint32_t np = gs_krandom(d, g, i, t, GS_PUR_GOSSIP, kk, 0u, GS_EMPTY32, m, peers);
      const uint32_t q0 = queued;
      if (g.active_bytes <= g.udp_avail && np != 0u) {
        // Every packet carries the whole queue (the byte budget cannot bind).  Broadcast r then rides
        // in packets 0 .. sends_r - 1 with sends_r = min(np, max(1, limit - transmits_r)): one read
        // and one write of its counter instead of one per packet, same counters and same packets as
        // the general loop below.
        uint32_t sends[GS_MAX_RUMORS > 8 ? 8 : GS_MAX_RUMORS];
        uint32_t n_pkts = 0, n_q = 0, pm = queued;
        bool few = true;
        while (pm) {
#if defined(__CUDA_ARCH__)
          const uint32_t r = __ffs(pm) - 1;
#else
          const uint32_t r = (uint32_t)__builtin_ctz(pm);
#endif
          pm &= pm - 1;
          if (n_q == 8u) { few = false; break; }
          const uint32_t tx = d.tx[GS_TX(r, cap, i)];
          uint32_t room = g.retransmit_limit > tx ? g.retransmit_limit - tx : 1u;
          if (room == 0u) room = 1u;
          const uint32_t s = room < np ? room : np;
          sends[n_q++] = s;
          if (s > n_pkts) n_pkts = s;
        }
        if (few) {
          pm = queued;
          for (uint32_t x = 0; x < n_q; ++x) {
#if defined(__CUDA_ARCH__)
            const uint32_t r = __ffs(pm) - 1;
#else
            const uint32_t r = (uint32_t)__builtin_ctz(pm);
#endif
            pm &= pm - 1;
            const uint32_t tx = (uint32_t)d.tx[GS_TX(r, cap, i)] + sends[x];
            d.tx[GS_TX(r, cap, i)] = (uint8_t)tx;
            if (tx >= g.retransmit_limit) queued &= ~(1u << r);  // broadcast finished
            sink.stat(GS_ST_RUMORS_SENT, sends[x]);
          }
          sink.stat(GS_ST_GOSSIP_PACKETS, n_pkts);
          for (uint32_t q = 0; q < n_pkts; ++q) {
            uint32_t pkt = 0;
            pm = q0;
            for (uint32_t x = 0; x < n_q; ++x) {
#if defined(__CUDA_ARCH__)
              const uint32_t r = __ffs(pm) - 1;
#else
              const uint32_t r = (uint32_t)__builtin_ctz(pm);
#endif
              pm &= pm - 1;
              if (sends[x] > q) pkt |= 1u << r;
            }
            if (!gs_lost(g, sink, i, peers[q], t, GS_LK_GOSSIP, q))
              gs_post(d, g, sink, (t + 1u + gs_extra(g, i, peers[q])) & g.ring_mask, peers[q], pkt);
          }
          np = 0u;  // done: the general loop below has nothing left to do
        }
      }
      for (uint32_t q = 0; q < np && queued != 0u; ++q) {
        uint32_t pkt = gs_select_packet(d, g, i, queued);
        if (pkt == 0u) break;
        uint32_t pm = pkt;
        while (pm) {
#if defined(__CUDA_ARCH__)
          uint32_t r = __ffs(pm) - 1;
#else
          uint32_t r = (uint32_t)__builtin_ctz(pm);
#endif
          pm &= pm - 1;
          uint32_t tx = (uint32_t)d.tx[GS_TX(r, cap, i)] + 1u;
          d.tx[GS_TX(r, cap, i)] = (uint8_t)tx;
          if (tx >= g.retransmit_limit) queued &= ~(1u << r);  // broadcast finished
          sink.stat(GS_ST_RUMORS_SENT, 1);
        }
        sink.stat(GS_ST_GOSSIP_PACKETS, 1);
        if (!gs_lost(g, sink, i, peers[q], t, GS_LK_GOSSIP, q))
          gs_post(d, g, sink, (t + 1u + gs_extra(g, i, peers[q])) & g.ring_mask, peers[q], pkt);
      }
      if (queued != q0) d.queued[i] = queued;
    }

    // ---- F. periodic push-pull ([U] memberlist/state.go pushPull -> pushPullNode) -------------
    // One random alive peer; the full-state exchange over TCP reduces, in this model, to the
    // tracked-broadcast mask and the Lamport clocks (alive/suspect/dead state is one shared record
    // per subject already).  Push now; the partner's answer arrives two ticks later.
    if (pp_now && !(m & GS_META_ISOLATED)) {
      uint32_t partner[1];
      if (gs_krandom(d, g, i, t, GS_PUR_PUSHPULL, 1u, 1u, GS_EMPTY32, m, partner) != 0u) {
        const uint32_t j = partner[0];
        uint32_t* req = d.ppreq + (size_t)nxt * GS_PPK * cap;
        uint32_t v = i;
        for (uint32_t s = 0; s < GS_PPK; ++s) {
          const uint32_t old = GS_ATOMIC_MIN32(&req[(size_t)s * cap + j], v);
          if (old == v || old == GS_EMPTY32) break;
          if (old > v) v = old;  // displaced a larger id: carry it to the next slot
        }
        uint32_t* clk = d.pp_clk + (size_t)nxt * 2u * cap;
        GS_ATOMIC_MAX32(&clk[j], d.ltime_member[i]);
        GS_ATOMIC_MAX32(&clk[cap + j], d.ltime_event[i]);
        gs_post(d, g, sink, inxt, j, (d.heard[i] & g.active_mask) | GS_ACC_BIT);
        sink.stat(GS_ST_PUSH_PULLS, 1);
      }
    }
  }

  // ---- E. write back ------------------------------------------------------------
  if (k != k0) {
    gs_key_store(d, g, nxt, i, k);
    m |= GS_META_DIRTY;  // the other buffer is stale for one more tick
  } else if (m0 & GS_META_DIRTY) {
    gs_key_store(d, g, nxt, i, k);
    m &= ~GS_META_DIRTY;
  }
  if (m != m0) d.meta[i] = m;
  if (due != due0) d.due[i] = due;
  // stay in the active set while something time-driven is pending: a running suspicion
  // timer, a stale key buffer, or a non-empty broadcast queue
  if (gs_key_rank(k) == GS_RANK_SUSPECT || (m & GS_META_DIRTY) || queued != 0u)
    gs_post(d, g, sink, inxt, i, GS_WAKE_BIT);
}

// ---------------------------------------------------------------------------------------
// Staged fast path for the steady-state case of [U] memberlist.probe/probeNode: a member
// with an empty mailbox whose probe ticker fires, whose ring cursor does not wrap and whose
// next ring entry is an established, non-dead peer.  The three stages let the tick kernel
// batch the memory phases of several members (A: own columns, B: target gather, C: commit)
// so a warp pays two dependent latencies per tile instead of five per member.  Any member
// that does not qualify falls back to gs_row_step, which must produce identical results;
// the fast path performs no write before stage C has accepted the member.
// ---------------------------------------------------------------------------------------
struct GsFastProbe {
  uint32_t k, m, cursor, pass, c, kc;
};

GS_DEV void gs_fast_load(const GsDev& d, uint32_t cur, uint32_t i, GsFastProbe& f) {
  f.k = d.key[cur][i];
  f.m = d.meta[i];
  f.cursor = d.cursor[i];
  f.pass = d.pass[i];
}

template <class G>
GS_DEV bool gs_fast_target(const GsDev& d, const G& g, uint32_t cur, uint32_t i,
                           GsFastProbe& f) {
  if (g.loss_thr != 0u || g.graph_n != 0u || d.coord != nullptr) return false;  // CSR rows, coordinates: generic path
  if (gs_key_truth(f.k) != GS_TRUTH_UP || gs_key_rank(f.k) != GS_RANK_ALIVE) return false;
  if (gs_meta_stage(f.m) != GS_STAGE_IDLE || (f.m & (GS_META_DIRTY | GS_META_ISOLATED))) return false;
  if (f.cursor >= g.n) return false;  // ring wrap: re-key in the generic path
  GsU4 rk = gs_perm_keys(g.seed_lo, g.seed_hi, i, f.pass);
  f.c = gs_perm(f.cursor, g.n, g.perm_bits, rk);
  if (f.c == i) return false;
  f.kc = gs_peer_key(d, cur, f.c, false);
  return true;
}

// Stage C's decision alone (no write): can gs_fast_finish take this member?
template <class G>
GS_DEV bool gs_fast_accept(const G& g, uint32_t i, uint32_t t, const GsFastProbe& f) {
  const uint32_t rank = gs_key_rank(f.kc);
  if (gs_key_truth(f.kc) == GS_TRUTH_NONE || rank == GS_RANK_DEAD || rank == GS_RANK_LEFT ||
      gs_key_pending(f.kc))
    return false;  // ring entry must be skipped or needs the heard mask: generic path
  if (g.pp_interval != 0u && gs_pp_due(g.pp_interval, g.rot_pp, i / g.phase_group, t))
    return false;  // the push-pull ticker fires too: generic path
  return true;
}

// Returns true when the member was fully handled; *acked tells whether the direct probe
// succeeded (stats: PROBES +1, ACKS +acked, ACTIVE_ROWS +1 are added by the caller).
template <class G, class Sink>
GS_DEV bool gs_fast_finish(const GsDev& d, const G& g, Sink& sink, uint32_t i, uint32_t t,
                           const GsFastProbe& f, bool* acked) {
  if (!gs_fast_accept(g, i, t, f)) return false;
  uint32_t m = f.m;
  if (gs_key_truth(f.kc) == GS_TRUTH_UP && gs_extra(g, i, f.c) + gs_extra(g, f.c, i) <= g.T) {
    const uint32_t aw = gs_meta_aw(m);
    m = gs_meta_set_aw(m, aw ? aw - 1u : 0u);
    d.due[i] = t + g.P;
    *acked = true;
  } else {
    m = gs_meta_set_stage(m, GS_STAGE_WAIT_T);
    d.probe_tgt[i] = f.c;
    d.probe_inc[i] = GS_PEER_INC(d, t & 1u, f.c, f.kc);
    d.due[i] = t + g.T;
    sink.horizon(t + g.P);  // the earliest tick this probe can end in an accusation
    *acked = false;
  }
  d.cursor[i] = f.cursor + 1u;
  if (m != f.m) d.meta[i] = m;
  return true;
}

// ---------------------------------------------------------------------------------------
// Staged fast path for the bulk of a join cascade: a member that is up, listed alive,
// established and clean, whose mail only repeats rumors it has heard or brings fresh alive /
// join-intent / leave-intent rumors, and which may have its gossip turn and its probe ticker
// at the same tick.  Same order as gs_row_step — A (accept), C (probe), D (gossip), E (wake) —
// with two rounds of loads instead of about five dependent ones: (A) the member's own columns,
// (B) the status gathers of the four gossip candidates of the first Philox block and of the
// probe target, with the retransmit counters of the queued broadcasts.  Nothing is written
// before every condition has held; a member that does not qualify is left untouched and takes
// gs_row_step.  Declined (generic step): packet loss, CSR graphs, latency pools, push-pull, a
// byte budget that can bind, tracked broadcasts in more than GS_FG_PAIRS counter pairs (GS_TX:
// two slots share one 16-bit element), accusations, user events
// and update rumors (event windows, logging), watched members with fresh mail, a probe action
// other than the ticker of an idle member, gossip candidates that are pending joiners or dead
// (those need the rumor table or change_tick), and a first block short of GossipNodes peers.
// GSIM_FLAG_NO_FAST_GOSSIP (256) turns the tier off; results are identical either way.
// ---------------------------------------------------------------------------------------
#define GS_FG_PAIRS 4u  // retransmit-counter pairs the tier loads at once (up to 8 tracked broadcasts)

GS_DEV uint32_t gs_popc(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __popc(x);
#else
  return (uint32_t)__builtin_popcount(x);
#endif
}
GS_DEV uint32_t gs_lowbit(uint32_t x) {  // index of the lowest set bit of x != 0
#if defined(__CUDA_ARCH__)
  return __ffs(x) - 1;
#else
  return (uint32_t)__builtin_ctz(x);
#endif
}

template <class Sink>
GS_DEV bool gs_fast_gossip(const GsDev& d, const GsGlobals& g, Sink& sink, uint32_t i, uint32_t t, uint32_t gslot,
                           uint32_t inb, bool due_now) {
  const uint32_t am = g.active_mask;
  uint32_t pm = 0;  // counter pairs holding a tracked slot
  for (uint32_t x = am; x != 0u; x &= x - 1u) pm |= 1u << (gs_lowbit(x) >> 1);
  if (inb == 0u || (inb & GS_ACC_BIT) || (g.flags & 256u) || g.loss_thr != 0u || g.graph_n != 0u || g.n_dcs != 0u ||
      g.pp_interval != 0u || g.active_bytes > g.udp_avail || g.n < 2u || g.gossip_nodes == 0u ||
      gs_popc(pm) > GS_FG_PAIRS)
    return false;
  const uint32_t cur = t & 1u;
  const size_t cap = g.cap;

  // ---- stage A: own columns (independent loads) ----
  GsFastProbe f;
  f.k = d.key[cur][i];
  f.m = d.meta[i];
  const uint32_t q0 = d.queued[i], heard0 = d.heard[i];
  const uint32_t rbits = inb & ~(GS_ACC_BIT | GS_WAKE_BIT) & am;
  const uint32_t lt0 = rbits != 0u ? d.ltime_member[i] : 0u;
  if (due_now) {
    f.cursor = d.cursor[i];
    f.pass = d.pass[i];
  }
  const uint32_t m0 = f.m;
  if (gs_key_truth(f.k) != GS_TRUTH_UP || gs_key_rank(f.k) != GS_RANK_ALIVE ||
      (m0 & (GS_META_DIRTY | GS_META_ISOLATED | GS_META_LEAVING)) || (q0 & ~am))
    return false;
  if (due_now && gs_meta_stage(m0) != GS_STAGE_IDLE) return false;  // indirect probes, probe deadline
  // section A: every fresh rumor is accepted (alive and intents have no drop rule)
  const uint32_t fresh = rbits & ~heard0;
  uint32_t lt = lt0;
  if (fresh != 0u) {
    if (m0 & GS_META_WATCHED) return false;  // join events are logged by the generic step
    for (uint32_t fm = fresh; fm != 0u; fm &= fm - 1u) {
      const GsRumor& ru = g.rumors[gs_lowbit(fm)];
      if (ru.kind == GS_RUMOR_JOIN_INTENT || ru.kind == GS_RUMOR_LEAVE_INTENT) {
        if (ru.ltime >= lt) lt = ru.ltime + 1u;  // clock.Witness
      } else if (ru.kind != GS_RUMOR_ALIVE) {
        return false;
      }
    }
  }
  const uint32_t q1 = q0 | fresh;
  const bool gossip = gslot == gs_meta_gphase(m0) && q1 != 0u;

  // ---- stage B: peer status gathers, retransmit counters ----
  if (due_now && !gs_fast_target(d, g, cur, i, f)) return false;
  uint32_t cc[4], kc[4], txw[2] = {0u, 0u};  // txw: the x-th pair of pm in bits 16x .. 16x + 15
  if (gossip) {
    const GsU4 blk = gs_philox(g.seed_lo, g.seed_hi, i, t, GS_PUR_GOSSIP, 0u);
#pragma unroll
    for (uint32_t x = 0; x < 4u; ++x) {
      cc[x] = gs_fastmod(gs_u4_get(blk, x), g.n, g.n_magic);
      kc[x] = cc[x] != i ? gs_peer_key(d, cur, cc[x], false) : 0u;
    }
    uint32_t mm = pm;
#pragma unroll
    for (uint32_t x = 0; x < GS_FG_PAIRS; ++x) {
      if (mm != 0u) {
        const uint32_t p = gs_lowbit(mm);
        mm &= mm - 1u;
        const uint32_t w = *reinterpret_cast<const uint16_t*>(d.tx + GS_TX(2u * p, cap, i));
        txw[x >> 1] |= w << ((x & 1u) * 16u);
      }
    }
  }
  if (due_now && !gs_fast_accept(g, i, t, f)) return false;
  // kRandomNodes (gs_krandom, mode 0) over the first block: tries = min(3n, 32) >= 6 covers all four draws
  const uint32_t want = g.gossip_nodes > 8u ? 8u : g.gossip_nodes;
  uint32_t np = 0, sel = 0;
  if (gossip) {
#pragma unroll
    for (uint32_t x = 0; x < 4u; ++x) {
      if (np < want) {
        const uint32_t c = cc[x], k = kc[x], rank = gs_key_rank(k);
        bool take = c != i && gs_key_truth(k) != GS_TRUTH_NONE && rank != GS_RANK_LEFT;
        if (take && (rank == GS_RANK_DEAD || gs_key_pending(k))) return false;
#pragma unroll
        for (uint32_t y = 0; y < x; ++y) take = take && !(((sel >> y) & 1u) && cc[y] == c);
        if (take) {
          sel |= 1u << x;
          ++np;
        }
      }
    }
    if (np < want) return false;
  }

  // ---- commit: what gs_row_step writes for this member ----
  const uint32_t inxt = (t + 1u) & g.ring_mask;
  sink.activity();
  d.inbox[t & g.ring_mask][i] = 0u;
  sink.stat(GS_ST_ACTIVE_ROWS, 1);
  if (fresh != 0u) {
    for (uint32_t fm = fresh; fm != 0u; fm &= fm - 1u) {
      const uint32_t r = gs_lowbit(fm);
      d.tx[GS_TX(r, cap, i)] = 0;  // queued with transmits = 0
      sink.heard(r);
    }
    sink.stat(GS_ST_RUMORS_ACCEPTED, gs_popc(fresh));
    d.heard[i] = heard0 | fresh;
    if (lt != lt0) d.ltime_member[i] = lt;
  }
  if (due_now) {
    bool acked = false;
    (void)gs_fast_finish(d, g, sink, i, t, f, &acked);  // accepted above
    sink.stat(GS_ST_PROBES, 1);
    if (acked) sink.stat(GS_ST_ACKS, 1);
  }
  uint32_t q = q1;
  if (gossip) {
    // every packet carries the whole queue: broadcast r rides in packets 0 .. sends_r - 1,
    // sends_r = min(np, max(1, limit - transmits_r)) (gs_row_step section D)
    const uint32_t lim = g.retransmit_limit;
    uint32_t pk0 = 0, pk1 = 0, pk2 = 0, pk3 = 0, n_pkts = 0, sent = 0;
    for (uint32_t qm = q1; qm != 0u; qm &= qm - 1u) {
      const uint32_t r = gs_lowbit(qm), x = gs_popc(pm & ((1u << (r >> 1)) - 1u));  // r's pair in txw
      const uint32_t tx = (fresh >> r) & 1u ? 0u : ((x >> 1 ? txw[1] : txw[0]) >> ((x & 1u) * 16u + (r & 1u) * 8u)) & 0xFFu;
      const uint32_t room = lim > tx ? lim - tx : 1u;
      const uint32_t s = room < np ? room : np;
      d.tx[GS_TX(r, cap, i)] = (uint8_t)(tx + s);
      if (tx + s >= lim) q &= ~(1u << r);  // broadcast finished
      sent += s;
      if (s > n_pkts) n_pkts = s;
      pk0 |= 1u << r;
      pk1 |= s > 1u ? 1u << r : 0u;
      pk2 |= s > 2u ? 1u << r : 0u;
      pk3 |= s > 3u ? 1u << r : 0u;
    }
    sink.stat(GS_ST_RUMORS_SENT, sent);
    sink.stat(GS_ST_GOSSIP_PACKETS, n_pkts);
    // packet q goes to the q-th peer taken: the selected candidates in draw order
#pragma unroll
    for (uint32_t x = 0; x < 4u; ++x) {
      if ((sel >> x) & 1u) {
        if (pk0 != 0u) gs_post(d, g, sink, inxt, cc[x], pk0);
        pk0 = pk1;
        pk1 = pk2;
        pk2 = pk3;
        pk3 = 0u;
      }
    }
  }
  if (q != q0) d.queued[i] = q;
  if (q != 0u) gs_post(d, g, sink, inxt, i, GS_WAKE_BIT);
  return true;
}
