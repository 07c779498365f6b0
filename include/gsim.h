/*
 * gsim.h — C ABI of the B200-native SWIM/Serf gossip simulator (libgsim.so).
 *
 * This is the drop-in boundary for Consul's gossip hot path.  The reference has no
 * FFI seam for this path: `agent/consul` calls two Go modules directly
 * (github.com/hashicorp/serf v0.10.2, github.com/hashicorp/memberlist v0.5.2 —
 * /root/reference/go.mod:80,85).  A Go facade package with the upstream import
 * paths (selected by `go.mod replace`) binds the functions below through cgo; see
 * INTEGRATION.md for the stub.  Every entry point cites the reference call site it
 * stands behind.  [U] = upstream module file that is not vendored in the reference.
 *
 * Conventions: opaque handles are owned by the library; every out buffer is caller
 * allocated and passed as (ptr, cap, *n); strings/payloads are copied on entry (cgo
 * pointer rules).  Return value 0 = GSIM_OK, negative = error (gsim_strerror).
 * One pool = one simulated gossip pool (LAN or WAN: agent/consul/server.go:683-709)
 * holding up to `capacity` virtual members on one CUDA device (or one shard of G).
 * Calls on one pool are serialised by an internal mutex; gsim_step is the only long
 * call.  There is no CPU fallback: pool creation fails with GSIM_ERR_NO_DEVICE when
 * no sm_100-class CUDA device is usable.
 */
#ifndef GSIM_H
#define GSIM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSIM_ABI_VERSION 1

/* ---- error codes ------------------------------------------------------- */
#define GSIM_OK 0
#define GSIM_ERR_INVALID (-1)      /* bad argument                                   */
#define GSIM_ERR_NO_DEVICE (-2)    /* no usable CUDA device (no CPU fallback exists) */
#define GSIM_ERR_CUDA (-3)         /* CUDA runtime error, see gsim_last_error        */
#define GSIM_ERR_CAPACITY (-4)     /* member capacity or rumor slots exhausted       */
#define GSIM_ERR_NOT_FOUND (-5)    /* unknown member id / rumor slot                 */
#define GSIM_ERR_STATE (-6)        /* operation illegal in the member's state        */
#define GSIM_ERR_TOO_LARGE (-7)    /* user event exceeds UserEventSizeLimit          */
#define GSIM_ERR_NOMEM (-8)

/* ---- serf.MemberStatus (pinned by /root/reference/api/agent.go:299-303) -- */
#define GSIM_STATUS_NONE 0
#define GSIM_STATUS_ALIVE 1
#define GSIM_STATUS_LEAVING 2
#define GSIM_STATUS_LEFT 3
#define GSIM_STATUS_FAILED 4
#define GSIM_STATUS_REAP (-1) /* agent/consul/server_serf.go:33 StatusReap */

/* ---- memberlist node state as gossiped ([U] memberlist/state.go NodeStateType) */
#define GSIM_RANK_ALIVE 0
#define GSIM_RANK_SUSPECT 1
#define GSIM_RANK_DEAD 2
#define GSIM_RANK_LEFT 3

/* ---- ground truth of a virtual member (simulator-only) ------------------ */
#define GSIM_TRUTH_NONE 0    /* id never created or reaped                  */
#define GSIM_TRUTH_UP 1      /* process running                             */
#define GSIM_TRUTH_CRASHED 2 /* Shutdown() without Leave(): server_test.go:725 */
#define GSIM_TRUTH_GONE 3    /* left gracefully and shut down               */

/* ---- serf.EventType (values follow [U] serf/event.go iota order) --------- */
#define GSIM_EVENT_MEMBER_JOIN 0
#define GSIM_EVENT_MEMBER_LEAVE 1
#define GSIM_EVENT_MEMBER_FAILED 2
#define GSIM_EVENT_MEMBER_UPDATE 3
#define GSIM_EVENT_MEMBER_REAP 4
#define GSIM_EVENT_USER 5
#define GSIM_EVENT_QUERY 6

/* ---- rumor kinds (tracked, exactly disseminated broadcasts) -------------- */
#define GSIM_RUMOR_FREE 0
#define GSIM_RUMOR_ALIVE 1        /* memberlist alive{Node,Incarnation} of a joiner   */
#define GSIM_RUMOR_JOIN_INTENT 2  /* serf messageJoin{LTime,Node}                     */
#define GSIM_RUMOR_LEAVE_INTENT 3 /* serf messageLeave{LTime,Node}                    */
#define GSIM_RUMOR_USER_EVENT 4   /* serf messageUserEvent{LTime,Name,Payload,CC}     */
#define GSIM_RUMOR_UPDATE 5       /* memberlist alive{Incarnation+1, new Meta} (SetTags) */
#define GSIM_MAX_RUMORS 30        /* inbox bits 0..29; bit 30 = wake, bit 31 = accusations */
#define GSIM_MAX_SUSPICION_SLOTS 5 /* k+1 with k = SuspicionMult-2 <= 4               */

typedef struct gsim_pool gsim_pool;

/*
 * Pool configuration.  Field names mirror memberlist.Config / serf.Config; the
 * authoritative list of knobs Consul writes is CloneSerfLANConfig
 * (/root/reference/agent/consul/config.go:661-698) and agent/agent.go:1383-1425.
 * Durations are nanoseconds like time.Duration; the library quantises them to the
 * base tick `tick_ns` (must divide probe_interval, probe_timeout, gossip_interval).
 */
typedef struct gsim_config {
  uint32_t struct_size; /* sizeof(gsim_config), for ABI evolution */
  uint32_t flags;       /* GSIM_FLAG_* */
  uint64_t seed;        /* Philox4x32-10 key */
  uint32_t capacity;    /* max virtual members (rows) in this pool */
  uint32_t n_initial;   /* members created converged (all Alive, inc=1, clocks=1) */
  uint64_t tick_ns;     /* base tick tau; 0 = gcd of the three intervals below */
  /* memberlist.Config ([U] memberlist/config.go; defaults pinned by
     agent/config/runtime.go:1271-1413) */
  uint64_t probe_interval_ns;
  uint64_t probe_timeout_ns;
  uint64_t gossip_interval_ns;
  uint64_t gossip_to_the_dead_ns;
  uint64_t push_pull_interval_ns; /* carried; periodic anti-entropy is SURVEY 8(f) N1 */
  uint32_t gossip_nodes;
  uint32_t indirect_checks;
  uint32_t retransmit_mult;
  uint32_t suspicion_mult;
  uint32_t suspicion_max_timeout_mult;
  uint32_t awareness_max_multiplier;
  uint32_t udp_buffer_size;
  uint32_t disable_tcp_pings;
  uint32_t packet_loss_ppm; /* simulated UDP loss per packet, parts per million */
  /* serf.Config ([U] serf/config.go; Consul overrides libserf/serf.go:19-36) */
  uint32_t event_buffer;          /* 512 */
  uint32_t user_event_size_limit; /* 512 */
  uint64_t leave_propagate_delay_ns;
  uint64_t broadcast_timeout_ns;
  uint64_t reap_interval_ns;
  uint64_t reconnect_timeout_ns;
  uint64_t tombstone_timeout_ns;
  /* sharding (SURVEY 8e): this process simulates rows with owner(i)==rank */
  uint32_t world_size;
  uint32_t rank;
  int32_t device; /* CUDA device ordinal, -1 = current */
  uint32_t event_log_capacity; /* device event ring entries (0 = default 65536) */
  /* Ticker stagger granularity: members [g*phase_group, (g+1)*phase_group) share one random
   * probe/gossip phase ([U] state.go triggerFunc draws it per agent).  0 = default 128, which
   * makes the failure-detector path uniform per 128-thread CTA; 1 = per-member phases (small
   * clusters, no CTA-level gating).  Must be 1 or a multiple of 128. */
  uint32_t phase_group;
  /* Mailbox ring depth: arrival slots per member (power of two, 2..8; 0 = 2).  A pool that will
   * carry a latency matrix (gsim_latency_set) needs depth > the largest one-way latency. */
  uint32_t mailbox_depth;
} gsim_config;

#define GSIM_FLAG_LOG_GLOBAL_EVENTS 1u /* log Failed/Left/Join transitions of every member */
#define GSIM_FLAG_NO_GRAPH 2u          /* launch tick kernels one by one (debug/profiling)  */
#define GSIM_FLAG_SHARD_SYNC_SCAN 4u   /* sharded pools: scan mailboxes with ld.relaxed.sys (debug) */
/* Sharded pools, measurement only: drop the per-thread fence.sys at the end of a tick and rely on
 * the cumulativity of the one fence the releasing thread executes after the CTA barrier.  Not a
 * supported mode until the 2/4/8-GPU digest tests have passed with it. */
#define GSIM_FLAG_SHARD_LEAN_FENCE 8u
/* Periodic push-pull anti-entropy ([U] memberlist/state.go pushPull, serf/delegate.go
 * LocalState/MergeRemoteState; SURVEY 8f N1): every pushPullScale(push_pull_interval, n) each
 * member exchanges its tracked-broadcast mask and Lamport clocks with one random alive peer
 * (push at tick t, the partner's answer arrives at t+2).  Off by default: the headline configs
 * of BASELINE.json run shorter than one push-pull interval at their sizes. */
/* Run every tick as its own launch even while the pool is quiet (no quiet windows, DESIGN.md 4.2):
 * for measurements and for tests that compare the two schedules.  Same results either way. */
#define GSIM_FLAG_NO_WINDOWS 16u
#define GSIM_FLAG_PUSH_PULL 32u
/* Sharded pools deliver mail with system-scope reductions (red.global.sys.or: nothing travels back over
 * NVLink).  This flag selects the fetching form (atom.sys) instead — measurement variant; same results. */
#define GSIM_FLAG_SHARD_ATOM 128u
/* Network coordinates ([U] serf/coordinate: Vivaldi with height, adjustment window and gravity;
 * SURVEY 8f N3).  Every direct probe ack updates the prober's coordinate with the measured round
 * trip (0.5 ms + the latency matrix there and back) and the target's coordinate.  348 B per
 * member; single-GPU pools.  IEEE double arithmetic, bit-identical to the oracle. */
#define GSIM_FLAG_COORDINATES 64u
/* Run every member with mail through the generic row step, without the fast gossip tier (DESIGN.md
 * 4.1): for measurements and for tests that compare the two.  Same results either way.  The
 * environment variable GSIM_NO_FAST_GOSSIP does the same for every pool of the process. */
#define GSIM_FLAG_NO_FAST_GOSSIP 256u

/* Preset defaults.  LAN/WAN: [U] memberlist DefaultLANConfig/DefaultWANConfig as
 * pinned by agent/config/runtime.go:1271-1413 with Consul's overrides
 * (libserf/serf.go:19-36, agent/consul/config.go:622-635, default.go:88-89 WAN
 * gossip_nodes=3).  TEST: agent/consul/server_test.go:221-237. */
void gsim_config_default_lan(gsim_config* cfg);
void gsim_config_default_wan(gsim_config* cfg);
void gsim_config_consul_test(gsim_config* cfg);

/* ---- pure formulas ([U] memberlist/util.go, suspicion.go; SURVEY 8c KATs) -- */
uint32_t gsim_retransmit_limit(uint32_t retransmit_mult, uint32_t n);
uint64_t gsim_suspicion_timeout_ns(uint32_t suspicion_mult, uint32_t n, uint64_t interval_ns);
int64_t gsim_remaining_suspicion_ns(uint32_t n_confirm, uint32_t k, uint64_t elapsed_ns,
                                    uint64_t min_ns, uint64_t max_ns);
uint64_t gsim_push_pull_scale_ns(uint64_t interval_ns, uint32_t n);
uint32_t gsim_lamport_witness(uint32_t clock, uint32_t v); /* [U] serf/lamport.go Witness */
uint32_t gsim_refute_incarnation(uint32_t cur, uint32_t accused); /* [U] state.go refute */
void gsim_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

/* ---- lifecycle ----------------------------------------------------------- */
/* serf.Create for the whole pool: server_serf.go:63, client_serf.go:76 create one
 * *serf.Serf per agent; here one pool holds all virtual agents and member_add
 * creates one of them. */
int gsim_pool_create(const gsim_config* cfg, gsim_pool** out);
void gsim_pool_destroy(gsim_pool* p); /* (*Serf).Shutdown: server.go:1261 */
const char* gsim_strerror(int code);
const char* gsim_last_error(gsim_pool* p);
int gsim_abi_version(void);

typedef struct gsim_member_desc {
  uint32_t alive_msg_size; /* encoded size of this member's alive{} message incl. Meta (tags); 0 = computed
                            * by the encoder (gsim_wire_alive) from name_len and meta_len */
  uint32_t flags;          /* GSIM_MEMBER_* */
  uint32_t name_len;       /* bytes of the node name ("node" / "node.dc"); 0 = the canonical "node-<id>" */
  uint32_t meta_len;       /* bytes of memberlist Meta (serf's encoded tags); used when alive_msg_size == 0 */
} gsim_member_desc;
#define GSIM_MEMBER_WATCHED 1u /* record this observer's serf events (EventCh) */

/* serf.Create of ONE virtual agent ([U] serf.Create -> memberlist.Create -> setAlive):
 * incarnation 1, three Lamport clocks incremented to 1, own alive{} queued. */
int gsim_member_add(gsim_pool* p, const gsim_member_desc* desc, uint32_t* id_out);

/* (*Serf).Join(existing []string, ignoreOld bool) (int, error) — server_ce.go:44,
 * client.go:222, server.go:1445, agent/router/serf_flooder.go:72.  Each reachable
 * seed is one push-pull state exchange ([U] memberlist.Join -> pushPullNode(join=true)),
 * then serf broadcasts a join intent.  n_ok = number of seeds contacted. */
int gsim_join(gsim_pool* p, uint32_t id, const uint32_t* seeds, size_t n_seeds, int ignore_old,
              int* n_ok);
/* (*Serf).Leave() — server.go:1360,1367, client.go:205. */
int gsim_leave(gsim_pool* p, uint32_t id);
/* Shutdown() without Leave() — the reference tests' fault injection
 * (server_test.go:725, agent_endpoint_test.go:2544). */
int gsim_crash(gsim_pool* p, uint32_t id);
int gsim_crash_many(gsim_pool* p, const uint32_t* ids, size_t n);
/* Crash every UP member i with philox(seed; i, salt, CRASH).x < ppm/1e6 * 2^32
 * (BASELINE config 3: 10 % crash injection at tick 0). */
int gsim_crash_fraction(gsim_pool* p, uint32_t ppm, uint32_t salt, uint32_t* n_crashed);
/* (*Serf).RemoveFailedNode / RemoveFailedNodePrune — server.go:1510-1534. */
int gsim_force_leave(gsim_pool* p, uint32_t via, uint32_t target, int prune);
/* (*Serf).UserEvent(name, payload, coalesce) — server_ce.go:125 (callers
 * internal_endpoint.go:862, leader.go:150).  slot_out = tracked rumor slot. */
int gsim_user_event(gsim_pool* p, uint32_t id, const void* name, size_t name_len,
                    const void* payload, size_t payload_len, int coalesce, uint32_t* slot_out);

/* Out-of-band delivery of tracked broadcast `slot` to member `id`, exactly as if a gossip packet
 * carrying it had just arrived (Lamport witness, de-dup, event-window checks, re-queue with
 * transmits = 0).  BASELINE config 5: bridge members re-fire an event they delivered in one WAN
 * pool into the other pool (the ForwardRPC of agent/consul/internal_endpoint.go:839).
 * *accepted = 1 when the member had not heard it and took it. */
int gsim_rumor_inject(gsim_pool* p, uint32_t slot, uint32_t id, int* accepted);

/* (*Serf).SetTags(tags) — internal/gossip/libserf/serf.go:51; [U] memberlist.UpdateNode: the
 * member re-broadcasts alive under its next incarnation; every other member raises
 * EventMemberUpdate when it arrives.  Tags stay host-side; alive_msg_size (0 = 64) is the encoded
 * size of the new alive message for the UDP budget. */
int gsim_member_update(gsim_pool* p, uint32_t id, uint32_t alive_msg_size, uint32_t* slot_out);

/* Peer graph in CSR form (BASELINE north_star: "message-passing kernel over a CSR peer graph").
 * Default: the complete graph — a converged memberlist knows every member.  With a graph, member
 * i's memberlist is col_idx[row_ptr[i] .. row_ptr[i+1]): gossip peers, indirect-probe relays,
 * push-pull partners and the probe ring are all drawn from that row (restricted topologies such
 * as Consul's serf_lan_allowed_cidrs, agent/config/runtime.go:1222-1232, or network segments).
 * n_rows must equal the current member count; rows may contain the member itself (skipped like
 * memberlist skips the local node).  A graph whose every row is 0..n-1 gives exactly the
 * complete-graph results.  The topology is static: gsim_member_add fails while a graph is set;
 * n_rows = 0 removes it.  Not supported on sharded pools.  A snapshot does not carry the graph:
 * set the same graph before gsim_restore. */
int gsim_graph_set(gsim_pool* p, uint32_t n_rows, const uint32_t* row_ptr, const uint32_t* col_idx);

/* serf.Config.ReconnectTimeoutOverride — internal/gossip/libserf/serf.go:68-85 (a member
 * advertises its own reconnect timeout in the "rc_tm" tag; agent/consul/client_test.go:862-894).
 * The override callback is host code; its result for member `id` is stored with the member and
 * used by the reaper instead of the pool's reconnect_timeout_ns.  0 = the pool's value. */
int gsim_member_reconnect_timeout_set(gsim_pool* p, uint32_t id, uint64_t timeout_ns);

/* (*Serf).GetCoordinate() / GetCachedCoordinate(name) — agent/router/router.go:62-67.
 * out = {Vec[0..7], Error, Adjustment, Height} in seconds, as coordinate.Coordinate. */
int gsim_coordinate_get(gsim_pool* p, uint32_t id, double out[11]);

/* Event logging of one member on/off after creation (that agent's EventCh; see
 * gsim_member_desc.flags / GSIM_MEMBER_WATCHED and gsim_poll_events). */
int gsim_member_watch(gsim_pool* p, uint32_t id, int on);

/* WAN latency (BASELINE config 5; Consul's WAN pool wiring: agent/consul/server_serf.go:187-213,
 * agent/consul/wanfed/wanfed.go:36-40).  Members are grouped into n_dcs (<= 64) synthetic
 * datacenters, member i in datacenter (i / 128) % n_dcs.  lat_ticks[a * n_dcs + b] = one-way
 * latency in ticks of a packet from datacenter a to datacenter b, 1 <= latency < mailbox_depth
 * (1 = the tick every packet takes on a pool without a matrix, so an all-ones matrix changes
 * nothing).  Applies to gossip packets and to probe round trips: an ack slower than ProbeTimeout
 * sends the prober into the indirect/TCP stage, where it still counts until the probe deadline.
 * n_dcs = 0 removes the matrix.  Callable between steps; packets in flight keep their slots. */
int gsim_latency_set(gsim_pool* p, uint32_t n_dcs, const uint8_t* lat_ticks);

/* ---- time ---------------------------------------------------------------- */
int gsim_step(gsim_pool* p, uint32_t ticks);
#define GSIM_PRED_RUMOR_CONVERGED 1 /* arg = slot: every UP member heard it          */
#define GSIM_PRED_ALL_RUMORS_CONVERGED 2
#define GSIM_PRED_CRASHED_ALL_DEAD 3 /* every CRASHED member is Dead in the view      */
/* Advance in chunks of `check_every` ticks until the predicate holds or max_ticks
 * elapsed.  *tick_out = exact tick at which the predicate first held (recorded on
 * the device), or UINT32_MAX. */
int gsim_run_until(gsim_pool* p, int predicate, uint32_t arg, uint32_t max_ticks,
                   uint32_t check_every, uint32_t* tick_out);
uint32_t gsim_now(gsim_pool* p); /* current tick */

/* ---- observation --------------------------------------------------------- */
typedef struct gsim_member {
  uint32_t id;
  int32_t status;       /* GSIM_STATUS_* as `observer` reports it from Members() */
  uint32_t incarnation;
  uint32_t rank;        /* GSIM_RANK_* */
} gsim_member;
/* (*Serf).Members() — server.go:1492,1500, server_serf.go:412, router.go:169. */
int gsim_members(gsim_pool* p, uint32_t observer, gsim_member* out, size_t cap, size_t* n);
/* (*Serf).NumNodes() — agent/router/router.go:62-67. */
int gsim_num_nodes(gsim_pool* p, uint32_t observer, uint32_t* n);

typedef struct gsim_event {
  uint32_t tick;
  uint32_t type;     /* GSIM_EVENT_* */
  uint32_t subject;  /* member id (member events) or rumor slot (user events) */
  uint32_t observer; /* watching member, or UINT32_MAX for pool-wide transitions */
  uint32_t ltime;    /* serf.UserEvent.LTime for user events */
  uint32_t reserved;
} gsim_event;
/* EventCh pump (server_serf.go:270-297, client_serf.go:80-110): drains the device
 * event ring, oldest first. */
int gsim_poll_events(gsim_pool* p, gsim_event* out, size_t cap, size_t* n);

typedef struct gsim_rumor_info {
  uint32_t kind, subject, incarnation, ltime, origin, size_bytes, start_tick;
  uint32_t heard_count;    /* UP members that have accepted it */
  uint32_t converged_tick; /* first tick at which heard_count == up_count, else UINT32_MAX */
  uint32_t queued_count;   /* members still retransmitting it */
} gsim_rumor_info;
int gsim_rumor_info_get(gsim_pool* p, uint32_t slot, gsim_rumor_info* out);
/* Fold a finished rumor into the base state and free its slot. */
int gsim_rumor_retire(gsim_pool* p, uint32_t slot);
/* Copy the stored name/payload of a user event slot. */
int gsim_user_event_get(gsim_pool* p, uint32_t slot, void* name, size_t name_cap, size_t* name_len,
                        void* payload, size_t payload_cap, size_t* payload_len);

/* (*Serf).Stats() — server.go:1733,1744 — plus simulator message counters. */
enum {
  GSIM_STAT_PROBES = 0,      /* direct pings sent                         */
  GSIM_STAT_ACKS,            /* direct acks received                      */
  GSIM_STAT_INDIRECT_PINGS,  /* indirectPingReq sent                      */
  GSIM_STAT_NACKS,           /* nackResp received                         */
  GSIM_STAT_PROBE_FAILURES,  /* probes that ended in suspectNode          */
  GSIM_STAT_SUSPECTS,        /* Alive -> Suspect transitions              */
  GSIM_STAT_CONFIRMATIONS,   /* accepted independent confirmations        */
  GSIM_STAT_DEADS,           /* Suspect -> Dead transitions               */
  GSIM_STAT_REFUTES,         /* incarnation bumps                         */
  GSIM_STAT_GOSSIP_PACKETS,  /* compound gossip packets sent              */
  GSIM_STAT_RUMORS_SENT,     /* broadcasts carried by those packets       */
  GSIM_STAT_RUMORS_ACCEPTED, /* first-time deliveries (re-queued)         */
  GSIM_STAT_RUMORS_DROPPED,  /* deliveries rejected (too old, min time)   */
  GSIM_STAT_PACKETS_LOST,    /* simulated UDP loss                        */
  GSIM_STAT_ACTIVE_ROWS,     /* rows that left the idle fast path         */
  GSIM_STAT_PUSH_PULLS,      /* periodic push-pull exchanges started      */
  GSIM_STAT_COUNT = 16
};
typedef struct gsim_stats {
  uint64_t counters[GSIM_STAT_COUNT];
  uint64_t node_ticks; /* sum over executed ticks of created members */
  uint32_t tick;
  uint32_t n_members; /* created ids */
  uint32_t n_up, n_crashed, n_gone;
  uint32_t n_view_alive, n_view_suspect, n_view_dead, n_view_left;
  uint32_t retransmit_limit;
  uint32_t suspicion_k;
  uint32_t suspicion_ticks[GSIM_MAX_SUSPICION_SLOTS]; /* timeout after c confirmations */
  uint32_t probe_interval_ticks, probe_timeout_ticks, gossip_interval_ticks;
  uint32_t events_dropped;
} gsim_stats;
int gsim_stats_get(gsim_pool* p, gsim_stats* out);

/* Order-independent 4x64-bit digest of the complete integer state (SURVEY 8d/8e:
 * equal for GPU and oracle, and for every shard count G). */
int gsim_state_hash(gsim_pool* p, uint64_t out[4]);

/* Raw column access for parity tests (values are copied device -> host). */
enum {
  GSIM_COL_KEY = 0,      /* u32: inc<<5 | pending<<4 | rank<<2 | truth */
  GSIM_COL_META,         /* u32: awareness, probe stage, flags          */
  GSIM_COL_DUE,          /* u32: tick of the next probe action          */
  GSIM_COL_CURSOR,       /* u32: probe ring cursor                      */
  GSIM_COL_PASS,         /* u32: probe ring pass                        */
  GSIM_COL_PROBE_TGT,    /* u32 */
  GSIM_COL_PROBE_INC,    /* u32 */
  GSIM_COL_SUS_START,    /* u32 */
  GSIM_COL_SUS_FROM,     /* u32[GSIM_MAX_SUSPICION_SLOTS][capacity]     */
  GSIM_COL_CHANGE_TICK,  /* u32 */
  GSIM_COL_LTIME_MEMBER, /* u32 */
  GSIM_COL_LTIME_EVENT,  /* u32 */
  GSIM_COL_EVENT_MIN,    /* u32 */
  GSIM_COL_HEARD,        /* u32 mask */
  GSIM_COL_QUEUED,       /* u32 mask */
  GSIM_COL_TX,           /* u8[GSIM_MAX_RUMORS][capacity] */
  GSIM_COL_INBOX,        /* u32: inbox slot that will be consumed at the next tick */
  GSIM_COL_COUNT
};
int gsim_column_read(gsim_pool* p, int column, void* out, size_t cap_bytes, size_t* n_bytes);

/* Checkpoint / resume (SURVEY §5): the blob restores bit-exactly. */
int gsim_snapshot_size(gsim_pool* p, size_t* n_bytes);
int gsim_snapshot(gsim_pool* p, void* out, size_t cap_bytes, size_t* n_bytes);
int gsim_restore(gsim_pool* p, const void* blob, size_t n_bytes);

/* ---- sharded pools: one process per GPU, cfg.world_size > 1 (SURVEY 8e, DESIGN.md §7) ----
 * Every rank creates the pool with the same config except `rank`/`device`, exchanges the file
 * descriptors of its physical column slices with every other rank (SCM_RIGHTS or pidfd_getfd), attaches
 * the peers' descriptors and calls gsim_shard_ready.  After that EVERY rank must issue the same
 * API calls in the same order: rank 0 executes the host-side operation, the others adopt its
 * result; gsim_step runs the tick kernels on all ranks with a device barrier per tick.  Bulk
 * observation (members, column_read, poll_events, snapshot, user_event_get) is served by rank 0. */
int gsim_shard_export_fds(gsim_pool* p, int* fds, size_t cap, size_t* n); /* one per column slice */
int gsim_shard_attach(gsim_pool* p, uint32_t peer_rank, const int* fds, size_t n);
int gsim_shard_ready(gsim_pool* p);

/* ---- measurement hooks (bench.py) ---------------------------------------- */
/* Device time of the tick kernels of the last gsim_step, measured with CUDA events
 * on the launching stream: total ms and number of tick launches. */
int gsim_last_step_timing(gsim_pool* p, double* kernel_ms, uint64_t* launches);
/* Total kernels launched by this pool since creation (bench "gpu_launches"). */
uint64_t gsim_launch_count(gsim_pool* p);
/* ---- wire formats (SURVEY 8f N4; consul_b200/csrc/gs_wire.h) -------------------------------------
 * The encoders behind every message size the byte budget of a gossip packet is checked against:
 * msgpack as hashicorp/go-msgpack v2 writes it for memberlist and serf (codec.MsgpackHandle{}: raw
 * strings, no str8/bin), memberlist's alive / suspect / dead and compound packet, serf's join /
 * leave intents and user event, the WAN-federation frame (agent/consul/wanfed/wanfed.go:112-121) and
 * Consul's UserEvent payload (agent/user_event.go:27-52, msgpackHandleUserEvent: str8 and bin).
 * Each call writes at most `cap` bytes to `out` (which may be NULL) and returns the encoded size. */
size_t gsim_wire_alive(void* out, size_t cap, uint32_t incarnation, const char* node, const void* addr,
                       size_t addr_len, uint16_t port, const void* meta, size_t meta_len, const uint8_t vsn[6]);
size_t gsim_wire_suspect(void* out, size_t cap, uint32_t incarnation, const char* node, const char* from);
size_t gsim_wire_dead(void* out, size_t cap, uint32_t incarnation, const char* node, const char* from);
size_t gsim_wire_join_intent(void* out, size_t cap, uint64_t ltime, const char* node);
size_t gsim_wire_leave_intent(void* out, size_t cap, uint64_t ltime, const char* node, int prune);
size_t gsim_wire_user_event(void* out, size_t cap, uint64_t ltime, const void* name, size_t name_len,
                            const void* payload, size_t payload_len, int coalesce);
/* memberlist compound packet of `count` messages (count <= 255) */
size_t gsim_wire_compound(void* out, size_t cap, const void* const* msgs, const size_t* lens, size_t count);
size_t gsim_wire_wanfed_frame(void* out, size_t cap, const void* packet, size_t len);
size_t gsim_wire_consul_user_event(void* out, size_t cap, const char* id, const char* name, const void* payload,
                                   size_t payload_len, const char* node_filter, const char* service_filter,
                                   const char* tag_filter, int version);

/* Entry `position` of the probe ring of `member` in its pass number `pass` over a member list of n entries:
 * the keyed Feistel permutation of [0, n) that stands in for memberlist's shuffled node slice ([U] state.go
 * resetNodes / shuffleNodes).  Pure function, exported for known-answer tests. */
uint32_t gsim_ring_entry(uint64_t seed, uint32_t n, uint32_t member, uint32_t pass, uint32_t position);
/* ... and the position at which `entry` appears in that ring (the inverse permutation; quiet windows of a
 * pristine pool use it to find a member's own entry without walking the ring). */
uint32_t gsim_ring_position(uint64_t seed, uint32_t n, uint32_t member, uint32_t pass, uint32_t entry);

/* Scheduling counters since creation: out[0] = quiet-window launches, out[1] = ticks advanced inside
 * quiet windows, out[2] = single-tick launches, out[3] = horizon scans, out[4] / out[5] = nanoseconds of
 * CUDA-event time spent in window / single-tick launches, out[6] = those of the window launches that ran
 * in closed form (pristine pool: every probe a prompt ack), out[7] = ticks they advanced. */
int gsim_sched_counts(gsim_pool* p, uint64_t out[8]);

#ifdef __cplusplus
}
#endif
#endif /* GSIM_H */
