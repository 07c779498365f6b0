// gs_api.cpp — host side of libgsim: the C ABI declared in include/gsim.h.
//
// Everything here is control plane: configuration, the N-dependent scalar tables
// (SURVEY §8a row a11, evaluated in double exactly like [U] memberlist/util.go and
// suspicion.go and then quantised to ticks so no floating point runs on the GPU), the
// serf-level operations that happen between ticks (Create/Join/Leave/UserEvent), and the
// rumor-slot bookkeeping.  The data plane is gs_cuda.cu.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <type_traits>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <thread>
#include <vector>

#include "../../include/gsim.h"
#include "gs_backend.h"
#include "gs_wire.h"
#include "gs_coord.h"

#ifndef GS_MAKE_BACKEND
#define GS_MAKE_BACKEND gs_make_cuda_backend
#endif
GsBackend* GS_MAKE_BACKEND(int device, char* err, size_t err_cap);

// ---------------------------------------------------------------------------
// pure formulas
// ---------------------------------------------------------------------------
extern "C" uint32_t gsim_retransmit_limit(uint32_t retransmit_mult, uint32_t n) {
  // [U] memberlist/util.go retransmitLimit: mult * ceil(log10(n+1));
  // doc form pinned by /root/reference/agent/config/runtime.go:1328-1330
  double node_scale = ceil(log10((double)n + 1.0));
  return retransmit_mult * (uint32_t)(int64_t)node_scale;
}

extern "C" uint64_t gsim_suspicion_timeout_ns(uint32_t suspicion_mult, uint32_t n,
                                              uint64_t interval_ns) {
  // [U] memberlist/util.go suspicionTimeout: mult * max(1, log10(max(1,n))) * interval,
  // computed as mult * Duration(nodeScale*1000) * interval / 1000 in int64;
  // doc form pinned by agent/config/runtime.go:1310-1312
  double node_scale = fmax(1.0, log10(fmax(1.0, (double)n)));
  int64_t scaled = (int64_t)(node_scale * 1000.0);
  return (uint64_t)((int64_t)suspicion_mult * scaled * (int64_t)interval_ns / 1000);
}

static uint64_t suspicion_total_ns(uint32_t n_confirm, uint32_t k, uint64_t min_ns,
                                   uint64_t max_ns) {
  // [U] memberlist/suspicion.go remainingSuspicionTime without the elapsed term
  if (k < 1) return min_ns;
  double frac = log((double)n_confirm + 1.0) / log((double)k + 1.0);
  double max_s = (double)max_ns / 1e9, min_s = (double)min_ns / 1e9;
  double raw = max_s - frac * (max_s - min_s);
  int64_t timeout = (int64_t)floor(1000.0 * raw) * 1000000ll;
  if (timeout < (int64_t)min_ns) timeout = (int64_t)min_ns;
  return (uint64_t)timeout;
}

extern "C" int64_t gsim_remaining_suspicion_ns(uint32_t n_confirm, uint32_t k, uint64_t elapsed_ns,
                                               uint64_t min_ns, uint64_t max_ns) {
  return (int64_t)suspicion_total_ns(n_confirm, k, min_ns, max_ns) - (int64_t)elapsed_ns;
}

extern "C" uint64_t gsim_push_pull_scale_ns(uint64_t interval_ns, uint32_t n) {
  // [U] memberlist/util.go pushPullScale, threshold 32
  if (n <= 32) return interval_ns;
  double mult = ceil(log2((double)n) - log2(32.0)) + 1.0;
  return (uint64_t)((int64_t)mult * (int64_t)interval_ns);
}

extern "C" uint32_t gsim_lamport_witness(uint32_t clock, uint32_t v) {
  // [U] serf/lamport.go Witness: if v >= cur, cur = v + 1
  return v < clock ? clock : v + 1u;
}

extern "C" uint32_t gsim_refute_incarnation(uint32_t cur, uint32_t accused) {
  // [U] memberlist/state.go refute: inc = nextIncarnation(); if accused >= inc,
  // inc = skipIncarnation(accused - inc + 1)
  uint32_t inc = cur + 1u;
  if (accused >= inc) inc += accused - inc + 1u;
  return inc;
}

extern "C" uint32_t gsim_ring_entry(uint64_t seed, uint32_t n, uint32_t member, uint32_t pass, uint32_t position) {
  if (n == 0 || position >= n) return GS_EMPTY32;
  const GsU4 rk = gs_perm_keys((uint32_t)seed, (uint32_t)(seed >> 32), member, pass);
  return gs_perm(position, n, gs_perm_bits_of(n), rk);
}

extern "C" uint32_t gsim_ring_position(uint64_t seed, uint32_t n, uint32_t member, uint32_t pass, uint32_t entry) {
  if (n == 0 || entry >= n) return GS_EMPTY32;
  const GsU4 rk = gs_perm_keys((uint32_t)seed, (uint32_t)(seed >> 32), member, pass);
  return gs_perm_inv(entry, n, gs_perm_bits_of(n), rk);
}

extern "C" void gsim_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  GsU4 r = gs_philox(key[0], key[1], ctr[0], ctr[1], ctr[2], ctr[3]);
  out[0] = r.x;
  out[1] = r.y;
  out[2] = r.z;
  out[3] = r.w;
}

// ---------------------------------------------------------------------------
// config presets
// ---------------------------------------------------------------------------
static const uint64_t MS = 1000000ull, SEC = 1000000000ull;

extern "C" void gsim_config_default_lan(gsim_config* c) {
  memset(c, 0, sizeof(*c));
  c->struct_size = sizeof(*c);
  c->seed = 0x5EED0001ull;
  c->capacity = 1024;
  // [U] memberlist DefaultLANConfig, pinned by agent/config/runtime.go:1271-1336
  c->probe_interval_ns = 1 * SEC;
  c->probe_timeout_ns = 500 * MS;
  c->gossip_interval_ns = 200 * MS;
  c->gossip_to_the_dead_ns = 30 * SEC;
  c->push_pull_interval_ns = 30 * SEC;
  c->gossip_nodes = 3;
  c->indirect_checks = 3;
  c->retransmit_mult = 4;
  c->suspicion_mult = 4;
  c->suspicion_max_timeout_mult = 6;
  c->awareness_max_multiplier = 8;
  c->udp_buffer_size = 1400;
  // [U] serf DefaultConfig with Consul's overrides: libserf/serf.go:19-36,
  // agent/consul/config.go:622-623 (ReconnectTimeout 72h)
  c->event_buffer = 512;
  c->user_event_size_limit = 512;
  c->leave_propagate_delay_ns = 3 * SEC;
  c->broadcast_timeout_ns = 5 * SEC;
  c->reap_interval_ns = 15 * SEC;
  c->reconnect_timeout_ns = 72ull * 3600 * SEC;
  c->tombstone_timeout_ns = 24ull * 3600 * SEC;
  c->world_size = 1;
  c->rank = 0;
  c->device = -1;
}

extern "C" void gsim_config_default_wan(gsim_config* c) {
  gsim_config_default_lan(c);
  // [U] memberlist DefaultWANConfig, pinned by agent/config/runtime.go:1348-1413;
  // gossip_nodes stays 3: agent/config/default.go:88-89 seeds gossip_wan from the LAN struct
  c->probe_interval_ns = 5 * SEC;
  c->probe_timeout_ns = 3 * SEC;
  c->gossip_interval_ns = 500 * MS;
  c->gossip_to_the_dead_ns = 60 * SEC;
  c->push_pull_interval_ns = 60 * SEC;
  c->suspicion_mult = 6;
}

extern "C" void gsim_config_consul_test(gsim_config* c) {
  gsim_config_default_lan(c);
  // agent/consul/server_test.go:221-237
  c->probe_interval_ns = 100 * MS;
  c->probe_timeout_ns = 50 * MS;
  c->gossip_interval_ns = 100 * MS;
  c->suspicion_mult = 2;
}

// ---------------------------------------------------------------------------
// pool
// ---------------------------------------------------------------------------
struct RumorHost {
  std::string name, payload;
  int coalesce = 0;
};
struct Sched {
  uint32_t tick, id, action;  // action 1 = shut down after Leave()
};

// A few host threads that stay around between calls (Members() of a large pool splits the id range over
// them): creating threads per call costs more than the work in a process that has a GPU context mapped.
class HostWorkers {
 public:
  explicit HostWorkers(unsigned n) : n_(n) {
    for (unsigned w = 1; w < n_; ++w) th_.emplace_back([this, w] { loop(w); });
  }
  ~HostWorkers() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
    }
    start_.notify_all();
    for (auto& t : th_) t.join();
  }
  unsigned size() const { return n_; }
  // job(w) on every worker w in [0, n); the caller is worker 0; returns when all are done
  void run(const std::function<void(unsigned)>& job) {
    {
      std::lock_guard<std::mutex> lk(m_);
      job_ = &job;
      pending_ = n_ - 1;
      ++gen_;
    }
    start_.notify_all();
    job(0);
    std::unique_lock<std::mutex> lk(m_);
    done_.wait(lk, [this] { return pending_ == 0; });
    job_ = nullptr;
  }

 private:
  void loop(unsigned w) {
    uint64_t seen = 0;
    for (;;) {
      const std::function<void(unsigned)>* job;
      {
        std::unique_lock<std::mutex> lk(m_);
        start_.wait(lk, [&] { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
        job = job_;
      }
      (*job)(w);
      {
        std::lock_guard<std::mutex> lk(m_);
        if (--pending_ == 0) done_.notify_one();
      }
    }
  }
  unsigned n_;
  std::vector<std::thread> th_;
  std::mutex m_;
  std::condition_variable start_, done_;
  const std::function<void(unsigned)>* job_ = nullptr;
  uint64_t gen_ = 0;
  unsigned pending_ = 0;
  bool stop_ = false;
};

struct gsim_pool {
  gsim_config cfg;
  GsBackend* be = nullptr;
  GsDev d;
  GsGlobals g;
  GsGlobals* g_dev = nullptr;
  bool g_dirty = true;
  bool counts_stale = true;
  uint32_t now = 0;
  uint64_t node_ticks = 0;
  std::mutex mu;
  RumorHost rh[GS_MAX_RUMORS];
  std::vector<Sched> sched;
  std::vector<void*> allocs;
  GsRecount rc;
  double last_ms = 0;
  uint64_t last_launches = 0;
  uint32_t events_dropped = 0;
  std::string err;
  uint64_t tick_ns = 0;
  uint32_t n_established = 0;  // members folded into the base set (not pending)
  // sharded (multi-GPU) pools: DESIGN.md §7
  bool sharded = false;
  uint32_t world = 1, rank = 0;
  size_t rows_per_rank = 0;
  uint8_t* pages = nullptr;  // page column: rank r's pool-wide words at pages + r*GS_PAGE_BYTES
  const int* shard_fds = nullptr;  // one exported descriptor per column slice
  size_t n_shard_fds = 0;
  uint32_t attached = 1;     // ranks whose memory is mapped here (including this one)
  bool ready = true;         // false between gsim_pool_create and gsim_shard_ready
  uint32_t call_seq = 0;     // controller calls so far (selects the blob slot)
  // rank-local counting: every rank counts its own rows, rank 0 sums (collective_recount)
  HostWorkers* workers = nullptr;  // created by the first bulk read that wants them
  uint32_t* stage = nullptr;  // pinned host staging for bulk reads (host_stage)
  size_t stage_words = 0;
  uint32_t quiet_fails = 0;  // consecutive looks at a pool that was still busy (try_quiet backs off)
  bool partials_fresh = false;  // (rank 0) the partial counts in its page describe (partials_seq, partials_now)
  uint32_t partials_seq = 0, partials_now = 0;
  // retirement at a step boundary clears the freed slots' bits rank by rank: the controller only collects
  // the mask (defer_and), every rank applies it to its own rows after the call (pending_keep)
  bool defer_and = false;
  uint32_t pending_keep = 0xFFFFFFFFu;
  std::vector<uint32_t> graph_rp, graph_col;  // host copy of the CSR peer graph (gsim_graph_set)
  GsXbar xb;
  std::vector<std::pair<uint32_t, uint32_t>> name_lens;  // (member, bytes of its node name) where not canonical
  // quiet-window scheduling (DESIGN.md §4.2)
  bool quiet = false;        // the pool is known to be quiet at p->now: windows may run
  bool healthy = false;      // ... and no probe can go unanswered: a launch may cover many ProbeIntervals
  bool pristine = false;     // ... and every member is up, listed alive and established: probes have a closed form
  uint32_t dirty_seq = 0;    // bumped by every host-side write to device state (quiet no longer known)
  uint32_t dirty_tick = 0;   // p->now at that write
  uint32_t retry_at = 0;     // do not look for quietness again before this tick
  // window launches, ticks run in windows, single-tick launches, horizon scans, ns of window kernels, ns of tick kernels
  uint64_t sched_counts[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

static void counts_invalidate(gsim_pool* p) {
  p->counts_stale = true;
  p->partials_fresh = false;
}

static void mark_dirty(gsim_pool* p) {
  p->quiet = false;
  p->healthy = false;
  p->pristine = false;
  p->retry_at = 0;  // (the clock may have gone back: restore)
  p->quiet_fails = 0;
  p->dirty_seq++;
  p->dirty_tick = p->now;
}

static uint64_t gcd64(uint64_t a, uint64_t b) {
  while (b) {
    uint64_t t = a % b;
    a = b;
    b = t;
  }
  return a;
}
static uint32_t ceil_ticks(uint64_t ns, uint64_t tick) { return (uint32_t)((ns + tick - 1) / tick); }
static uint32_t clamp_ticks(uint64_t ns, uint64_t tick);

static int fail(gsim_pool* p, int code, const char* msg) {
  p->err = msg ? msg : "";
  if (code == GSIM_ERR_CUDA && p->be) p->err += std::string(": ") + p->be->last_error();
  return code;
}

template <class T>
static bool peek(gsim_pool* p, const T* col, size_t i, T* out) {
  return p->be->d2h(out, col + i, sizeof(T));
}
template <class T>
static bool poke(gsim_pool* p, T* col, size_t i, T v) {
  mark_dirty(p);  // a host write to device state: whatever was known about quietness is void
  return p->be->h2d_word(col + i, &v, sizeof(T));
}

// Host-side write of a member's key word: every replica on a sharded pool.
static bool poke_key(gsim_pool* p, uint32_t buf, uint32_t i, uint32_t k) {
  if (p->d.kst) {  // keep the member's status byte in step (see gs_kst_code)
    uint8_t b;
    if (!peek(p, p->d.kst, i, &b)) return false;
    const uint32_t code = gs_kst_code(k);
    b = (uint8_t)(buf ? ((b & 0x0Fu) | (code << 4)) : ((b & 0xF0u) | code));
    if (!poke(p, p->d.kst, i, b)) return false;
  }
  if (!p->sharded) return poke(p, p->d.key[buf], i, k);
  for (uint32_t r = 0; r < p->world; ++r)
    if (!poke(p, p->d.key_rep[buf], (size_t)r * p->g.key_stride + i, k)) return false;
  return true;
}

// N-dependent scalars, recomputed whenever the member count changes (a11).
static void recompute_tables(gsim_pool* p) {
  GsGlobals& g = p->g;
  const gsim_config& c = p->cfg;
  const uint32_t n = g.n;
  g.retransmit_limit = gsim_retransmit_limit(c.retransmit_mult, n);
  if (g.retransmit_limit > 255u) g.retransmit_limit = 255u;
  // [U] memberlist/state.go suspectNode: k = SuspicionMult - 2, 0 if n-2 < k
  int k = (int)c.suspicion_mult - 2;
  if ((int)n - 2 < k) k = 0;
  if (k < 0) k = 0;
  if (k > GS_K1MAX - 1) k = GS_K1MAX - 1;
  g.sus_k = (uint32_t)k;
  uint64_t min_ns = gsim_suspicion_timeout_ns(c.suspicion_mult, n, c.probe_interval_ns);
  uint64_t max_ns = (uint64_t)c.suspicion_max_timeout_mult * min_ns;
  for (uint32_t q = 0; q < GS_K1MAX; ++q) {
    uint32_t cc = q > g.sus_k ? g.sus_k : q;
    g.sus_ticks[q] = ceil_ticks(suspicion_total_ns(cc, g.sus_k, min_ns, max_ns), p->tick_ns);
  }
  g.perm_bits = gs_perm_bits_of(n);
  g.n_magic = n ? 0xFFFFFFFFFFFFFFFFull / n + 1ull : 0ull;
  // [U] memberlist/state.go schedule: the push-pull ticker runs every pushPullScale(PushPullInterval, n)
  g.pp_interval = 0;
  g.rot_pp = 0;
  if ((c.flags & GSIM_FLAG_PUSH_PULL) && c.push_pull_interval_ns) {
    g.pp_interval = ceil_ticks(gsim_push_pull_scale_ns(c.push_pull_interval_ns, n), p->tick_ns);
    if (g.pp_interval < 2u) g.pp_interval = 2u;  // the exchange itself takes two ticks
    g.rot_pp = (gs_phase_rot(g.seed_lo, g.seed_hi) >> 8) % g.pp_interval;
  }
  p->g_dirty = true;
}

static bool upload_globals(gsim_pool* p) {
  if (!p->g_dirty) return true;
  if (p->sharded) {
    // the controller (rank 0) writes every rank's device copy; only `rank` differs
    for (uint32_t r = 0; r < p->world; ++r) {
      GsGlobals tmp = p->g;
      tmp.rank = r;
      if (!p->be->h2d(p->pages + (size_t)r * GS_PAGE_BYTES + GS_PG_GLOBALS, &tmp, sizeof(GsGlobals))) return false;
    }
  } else if (!p->be->h2d(p->g_dev, &p->g, sizeof(GsGlobals))) {
    return false;
  }
  p->g_dirty = false;
  return true;
}

// ---- sharded pools: the controller protocol ---------------------------------------------------
// Every rank calls every API function in the same order.  Rank 0 (the controller) executes the
// host-side operation — all device pokes go through the unified address space, to whichever GPU
// owns the row — then publishes the resulting host state (GsGlobals incl. the rumor table, clock,
// schedule, return code, small out-parameters) in a blob in its page and enters the device
// barrier; the other ranks enter the barrier, read the blob and adopt the state.
struct BlobHdr {
  int32_t rc;
  uint32_t now, n_established, n_sched, out_bytes, dirty_seq;
  uint64_t node_ticks;
  uint32_t call_seq, want_bytes;  // which call this blob answers: a rank out of step must fail, not adopt
  uint32_t pending_keep;          // bit columns every rank still has to AND on its own rows (~0 = nothing)
};

template <class F>
static int controller_call(gsim_pool* p, void* out, size_t out_bytes, F f) {
  if (!p->sharded) return f();
  const uint32_t seq = p->call_seq++;
  const uint32_t slot = seq & 1u;
  uint8_t* blob_dev = p->pages + GS_PG_BLOB + (size_t)slot * GS_BLOB_BYTES;  // in rank 0's page
  std::vector<uint8_t> blob(GS_BLOB_BYTES, 0);
  BlobHdr h;
  memset(&h, 0, sizeof(h));
  if (p->rank == 0) {
    h.rc = f();
    if (p->g_dirty && !upload_globals(p)) h.rc = h.rc ? h.rc : GSIM_ERR_CUDA;
    h.now = p->now;
    h.n_established = p->n_established;
    h.n_sched = (uint32_t)p->sched.size();
    h.out_bytes = (uint32_t)(out ? out_bytes : 0);
    h.node_ticks = p->node_ticks;
    h.dirty_seq = p->dirty_seq;
    h.call_seq = seq;
    h.want_bytes = (uint32_t)out_bytes;
    h.pending_keep = p->pending_keep;
    uint8_t* w = blob.data();
    if (sizeof(h) + sizeof(GsGlobals) + (size_t)h.n_sched * sizeof(Sched) + h.out_bytes > GS_BLOB_BYTES) {
      // every rank must still leave the barrier: publish the error instead of the state
      fail(p, GSIM_ERR_INVALID, "state blob overflow (too many scheduled shutdowns for a sharded pool)");
      h.rc = GSIM_ERR_INVALID;
      h.n_sched = 0;
      h.out_bytes = 0;
    }
    memcpy(w, &h, sizeof(h)); w += sizeof(h);
    memcpy(w, &p->g, sizeof(GsGlobals)); w += sizeof(GsGlobals);
    if (h.n_sched) memcpy(w, p->sched.data(), h.n_sched * sizeof(Sched));
    w += h.n_sched * sizeof(Sched);
    if (out && h.out_bytes) memcpy(w, out, h.out_bytes);
    w += h.out_bytes;
    if (!p->be->h2d(blob_dev, blob.data(), (size_t)(w - blob.data()))) return fail(p, GSIM_ERR_CUDA, "blob h2d");
    if (!p->be->xbar_host(p->xb)) return fail(p, GSIM_ERR_CUDA, "barrier");
    return h.rc;
  }
  if (!p->be->xbar_host(p->xb)) return fail(p, GSIM_ERR_CUDA, "barrier");
  if (!p->be->d2h(blob.data(), blob_dev, GS_BLOB_BYTES)) return fail(p, GSIM_ERR_CUDA, "blob d2h");
  const uint8_t* r = blob.data();
  memcpy(&h, r, sizeof(h)); r += sizeof(h);
  if (h.call_seq != seq || h.want_bytes != (uint32_t)out_bytes) {
    char msg[160];
    snprintf(msg, sizeof(msg), "controller protocol out of step: call %u (%zu bytes out) met the blob of call %u (%u bytes out)",
             seq, out_bytes, h.call_seq, h.want_bytes);
    if (getenv("GSIM_DEBUG_PROTOCOL")) fprintf(stderr, "libgsim rank %u: %s\n", p->rank, msg);
    return fail(p, GSIM_ERR_STATE, msg);
  }
  memcpy(&p->g, r, sizeof(GsGlobals)); r += sizeof(GsGlobals);
  p->g.rank = p->rank;
  p->sched.resize(h.n_sched);
  if (h.n_sched) memcpy(p->sched.data(), r, h.n_sched * sizeof(Sched));
  r += h.n_sched * sizeof(Sched);
  if (out && h.out_bytes == out_bytes && out_bytes) memcpy(out, r, out_bytes);
  p->now = h.now;
  p->n_established = h.n_established;
  p->node_ticks = h.node_ticks;
  p->pending_keep = h.pending_keep;
  if (h.dirty_seq != p->dirty_seq) {  // the controller wrote device state: same consequence on every rank
    p->dirty_seq = h.dirty_seq;
    p->dirty_tick = p->now;
    p->quiet = false;
    p->healthy = false;
    p->pristine = false;
    p->retry_at = 0;
    p->quiet_fails = 0;
  }
  p->g_dirty = false;
  counts_invalidate(p);
  if (h.rc) p->err = "controller reported an error";
  return h.rc;
}

#define GS_CONTROLLER_ONLY(p)                                                                        \
  if ((p)->sharded && (p)->rank != 0)                                                                \
    return fail((p), GSIM_ERR_STATE, "bulk observation of a sharded pool is served by rank 0 only")

static void rebuild_class_masks(gsim_pool* p) {
  GsGlobals& g = p->g;
  g.class_mask[0] = g.class_mask[1] = g.class_mask[2] = 0;
  g.active_bytes = 0;
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r)
    if ((g.active_mask >> r) & 1u) {
      g.class_mask[g.rumors[r].qclass] |= 1u << r;
      g.active_bytes += g.rumors[r].size + (g.rumors[r].qclass ? 3u : 2u);
    }
  p->g_dirty = true;
}

template <class T>
static bool alloc_col(gsim_pool* p, T** out, size_t count) {
  void* q = p->be->alloc(count * sizeof(T));
  if (!q) return false;
  p->allocs.push_back(q);
  *out = reinterpret_cast<T*>(q);
  return true;
}

// Sharded pools: every rank's progress words say "all ticks < now are done" (controller only).
static bool reset_tick_flags(gsim_pool* p) {
  if (!p->sharded) return true;
  uint32_t words[GS_MAX_WORLD];
  for (uint32_t r = 0; r < GS_MAX_WORLD; ++r) words[r] = p->now;
  const uint32_t zero = 0;
  for (uint32_t r = 0; r < p->world; ++r) {
    uint8_t* page = p->pages + (size_t)r * GS_PAGE_BYTES;
    if (!p->be->h2d(page + GS_PG_TICK_FLAGS, words, sizeof(words))) return false;
    if (!p->be->h2d(page + GS_PG_DONE_CTR, &zero, 4)) return false;
    if (!p->be->h2d(page + GS_PG_TICK_BASE, &p->now, 4)) return false;
  }
  return true;
}

// Quiet-window words of every rank: nothing known (controller only).
static bool reset_qstate(gsim_pool* p) {
  const uint32_t words[GS_Q_WORDS] = {p->now, GS_NEVER, p->now, 0u};  // last-active+1 = now: tick now-1 counts as active
  for (uint32_t r = 0; r < (p->sharded ? p->world : 1u); ++r)
    if (!p->be->h2d(p->d.qstate[r], words, sizeof(words))) return false;
  mark_dirty(p);
  return true;
}

// Device-side initial state: empty columns, zeroed counters, the converged initial members.
// On a sharded pool this runs on rank 0 only and reaches every GPU through the unified columns.
static int init_device_state(gsim_pool* p) {
  GsBackend* be = p->be;
  GsDev& d = p->d;
  GsGlobals& g = p->g;
  const size_t cap = g.cap;
  bool okk = true;
  // key = 0 means truth NONE for rows that were never created
  const size_t key_words = p->sharded ? (size_t)g.key_stride * p->world : cap;
  okk = okk && be->fill32(d.key_rep[0], 0, key_words) && be->fill32(d.key_rep[1], 0, key_words);
  for (uint32_t s = 0; s <= g.ring_mask; ++s) okk = okk && be->fill32(d.inbox[s], 0, cap);
  if (d.kst) okk = okk && be->fill8(d.kst, 0, cap);
  okk = okk && be->fill32(d.due, GS_NEVER, cap);  // rows that do not exist are never due
  okk = okk && be->fill32(d.reap_after, 0, cap);
  // rows that were never created hold the same defaults gs_init_row writes, so that a column
  // nobody has touched is one repeated word (gsim_snapshot stores such planes as a fill)
  okk = okk && be->fill32(d.cursor, 0, cap) && be->fill32(d.pass, 0, cap) && be->fill32(d.probe_tgt, 0, cap) &&
        be->fill32(d.probe_inc, 0, cap) && be->fill32(d.sus_start, 0, cap) && be->fill32(d.change_tick, 0, cap) &&
        be->fill32(d.event_min, 0, cap) && be->fill32(d.heard, 0, cap) && be->fill32(d.queued, 0, cap) &&
        be->fill32(d.ltime_member, 1, cap) && be->fill32(d.ltime_event, 1, cap) && be->fill32(d.meta, 0, cap) &&
        be->fill32(d.sus_from, GS_EMPTY32, cap * GS_K1MAX) &&
        be->fill32(reinterpret_cast<uint32_t*>(d.acc), GS_EMPTY32, cap * GS_K1MAX * 2 * 2);
  okk = okk && be->fill8(d.tx, 0, cap * GS_MAX_RUMORS);
  if (d.ppreq) okk = okk && be->fill32(d.ppreq, GS_EMPTY32, cap * 2 * GS_PPK) && be->fill32(d.pp_clk, 0, cap * 4);
  okk = okk && be->fill32(reinterpret_cast<uint32_t*>(d.stats), 0, GSIM_STAT_COUNT * 2);
  okk = okk && be->fill32(d.heard_cnt, 0, 32) && be->fill32(d.conv_tick, GS_EMPTY32, 32);
  okk = okk && be->fill32(d.view_cnt, 0, 4) && be->fill32(d.crashed_alive, 0, 1);
  okk = okk && be->fill32(d.crashed_dead_tick, GS_EMPTY32, 1);
  okk = okk && be->fill32(d.evlog_cursor, 0, 2) && be->fill32(d.tick_base, 0, 1);
  if (!p->sharded) okk = okk && be->fill32(d.done_ctr, 0, 1);
  okk = okk && reset_qstate(p);

  p->g_dirty = true;
  okk = okk && upload_globals(p);
  okk = okk && reset_tick_flags(p);
  okk = okk && be->init_rows(d, p->g_dev, g, 0, p->cfg.n_initial, 0);
  return okk ? GSIM_OK : GSIM_ERR_CUDA;
}

extern "C" int gsim_abi_version(void) { return GSIM_ABI_VERSION; }

extern "C" const char* gsim_strerror(int code) {
  switch (code) {
    case GSIM_OK: return "ok";
    case GSIM_ERR_INVALID: return "invalid argument";
    case GSIM_ERR_NO_DEVICE: return "no usable sm_100 CUDA device (libgsim has no CPU fallback)";
    case GSIM_ERR_CUDA: return "CUDA error";
    case GSIM_ERR_CAPACITY: return "capacity exhausted";
    case GSIM_ERR_NOT_FOUND: return "not found";
    case GSIM_ERR_STATE: return "illegal state";
    case GSIM_ERR_TOO_LARGE: return "user event too large";
    case GSIM_ERR_NOMEM: return "out of memory";
  }
  return "unknown error";
}

extern "C" const char* gsim_last_error(gsim_pool* p) { return p ? p->err.c_str() : ""; }

static_assert(GS_PG_GLOBALS + sizeof(GsGlobals) <= GS_PG_SCRATCH, "GsGlobals outgrew its page slot");
static_assert(sizeof(BlobHdr) + sizeof(GsGlobals) + 4096 <= GS_BLOB_BYTES, "state blob too small");
static thread_local std::string g_create_err;

extern "C" int gsim_pool_create(const gsim_config* cfg, gsim_pool** out) {
  if (!cfg || !out || cfg->struct_size != sizeof(gsim_config)) return GSIM_ERR_INVALID;
  if (cfg->capacity == 0 || cfg->n_initial > cfg->capacity) return GSIM_ERR_INVALID;
  if (!cfg->probe_interval_ns || !cfg->probe_timeout_ns || !cfg->gossip_interval_ns)
    return GSIM_ERR_INVALID;
  if (cfg->probe_timeout_ns >= cfg->probe_interval_ns) return GSIM_ERR_INVALID;
  if (cfg->world_size < 1 || cfg->world_size > GS_MAX_WORLD || cfg->rank >= cfg->world_size) return GSIM_ERR_INVALID;
  const bool sharded = cfg->world_size > 1;
  uint64_t tick = cfg->tick_ns;
  if (!tick) tick = gcd64(gcd64(cfg->probe_interval_ns, cfg->probe_timeout_ns), cfg->gossip_interval_ns);
  if (cfg->probe_interval_ns % tick || cfg->probe_timeout_ns % tick || cfg->gossip_interval_ns % tick)
    return GSIM_ERR_INVALID;
  if (cfg->gossip_interval_ns / tick > 255 || cfg->awareness_max_multiplier < 1 ||
      cfg->awareness_max_multiplier > 8 || cfg->gossip_nodes > 8 || cfg->indirect_checks > 8)
    return GSIM_ERR_INVALID;
  const uint32_t phase_group = cfg->phase_group ? cfg->phase_group : GS_TILE;
  // 1 (per member) or 128 * 2^k (whole tiles)
  if (phase_group != 1 && (phase_group % GS_TILE != 0 || ((phase_group / GS_TILE) & (phase_group / GS_TILE - 1)) != 0))
    return GSIM_ERR_INVALID;
  // mailbox ring: 2 arrival slots unless the pool is going to carry a latency matrix
  const uint32_t ring_depth = cfg->mailbox_depth ? cfg->mailbox_depth : 2u;
  if (ring_depth < 2 || ring_depth > GS_RING_MAX || (ring_depth & (ring_depth - 1u)) != 0) return GSIM_ERR_INVALID;

  char errbuf[256] = {0};
  GsBackend* be = GS_MAKE_BACKEND(cfg->device, errbuf, sizeof(errbuf));
  if (!be) {
    g_create_err = errbuf;
    fprintf(stderr, "libgsim: %s\n", errbuf);
    return GSIM_ERR_NO_DEVICE;
  }
  gsim_pool* p = new gsim_pool();
  p->cfg = *cfg;
  p->be = be;
  p->tick_ns = tick;
  memset(&p->d, 0, sizeof(p->d));
  memset(&p->g, 0, sizeof(p->g));
  memset(&p->rc, 0, sizeof(p->rc));
  // column stride: padded to whole tiles so the tick kernel never needs a bounds check
  size_t cap = ((size_t)cfg->capacity + GS_TILE - 1) / GS_TILE * GS_TILE;
  GsDev& d = p->d;
  GsGlobals& g = p->g;
  if (sharded) {
    // one virtual address range per column, physically sharded over the GPUs (gs_vmm.h);
    // rows per rank is a multiple of the 2 MB mapping granularity so byte columns align too
    if (!be->shard_begin(cfg->world_size, cfg->rank)) {
      g_create_err = be->last_error();
      fprintf(stderr, "libgsim: sharded pools unavailable: %s\n", be->last_error());
      gsim_pool_destroy(p);
      return GSIM_ERR_CUDA;
    }
    const size_t gran = be->shard_granularity();
    size_t per = ((size_t)cfg->capacity + cfg->world_size - 1) / cfg->world_size;
    const size_t gran_rows = gran / 2;  // the narrowest column has 2-byte elements (GS_TX)
    per = (per + gran_rows - 1) / gran_rows * gran_rows;
    p->sharded = true;
    p->world = cfg->world_size;
    p->rank = cfg->rank;
    p->rows_per_rank = per;
    p->ready = false;
    cap = per * cfg->world_size;
  }
  const size_t per_rank = p->rows_per_rank;
  auto acol = [&](auto** out, size_t planes) -> bool {
    typedef typename std::remove_pointer<typename std::remove_pointer<decltype(out)>::type>::type T;
    if (!sharded) return alloc_col(p, out, cap * planes);
    void* q = be->shard_alloc(per_rank * sizeof(T), planes);
    *out = reinterpret_cast<T*>(q);
    return q != nullptr;
  };
  bool okk = true;
  if (!sharded) {
    okk = okk && alloc_col(p, &d.key[0], cap) && alloc_col(p, &d.key[1], cap);
    d.key_rep[0] = d.key[0];
    d.key_rep[1] = d.key[1];
  } else {
    // one full replica of the key column per rank (gathers stay local; writers update all)
    const size_t gran = be->shard_granularity();
    const size_t rep_bytes = (cap * 4 + gran - 1) / gran * gran;
    g.key_stride = (uint32_t)(rep_bytes / 4);
    for (int b = 0; b < 2 && okk; ++b) {
      d.key_rep[b] = reinterpret_cast<uint32_t*>(be->shard_alloc(rep_bytes, 1));
      okk = d.key_rep[b] != nullptr;
      d.key[b] = okk ? d.key_rep[b] + (size_t)cfg->rank * g.key_stride : nullptr;
    }
  }
  if (!sharded) okk = okk && alloc_col(p, &d.kst, cap);  // performance variant: status replica
  g.ring_mask = ring_depth - 1u;
  for (uint32_t s = 0; s < ring_depth; ++s) okk = okk && acol(&d.inbox[s], 1);
  okk = okk && acol(&d.due, 1) && acol(&d.meta, 1);
  okk = okk && acol(&d.cursor, 1) && acol(&d.pass, 1);
  okk = okk && acol(&d.probe_tgt, 1) && acol(&d.probe_inc, 1);
  okk = okk && acol(&d.sus_start, 1) && acol(&d.sus_from, GS_K1MAX);
  okk = okk && acol(&d.acc, GS_K1MAX * 2);
  okk = okk && acol(&d.change_tick, 1) && acol(&d.reap_after, 1);
  okk = okk && acol(&d.ltime_member, 1) && acol(&d.ltime_event, 1);
  okk = okk && acol(&d.event_min, 1);
  okk = okk && acol(&d.heard, 1) && acol(&d.queued, 1);
  {  // two rumors per 16-bit element (GS_TX): the narrowest sharded slice is 2 bytes per member
    uint16_t* tx16 = nullptr;
    okk = okk && acol(&tx16, GS_MAX_RUMORS / 2);
    d.tx = reinterpret_cast<uint8_t*>(tx16);
  }
  if (cfg->flags & GSIM_FLAG_COORDINATES) {  // Vivaldi state: 348 B per member, only when asked for
    if (sharded) {
      g_create_err = "network coordinates are not supported on sharded pools yet";
      fprintf(stderr, "libgsim: %s\n", g_create_err.c_str());
      gsim_pool_destroy(p);
      return GSIM_ERR_INVALID;
    }
    okk = okk && alloc_col(p, &d.coord, cap * 2 * GS_COORD_WORDS) && alloc_col(p, &d.ctag, cap * 2) &&
          alloc_col(p, &d.adj, cap * GS_ADJ_WINDOW) && alloc_col(p, &d.adj_idx, cap);
  }
  if (cfg->flags & GSIM_FLAG_PUSH_PULL)  // push-pull mailboxes: 48 B per member, only when asked for
    okk = okk && acol(&d.ppreq, 2 * GS_PPK) && acol(&d.pp_clk, 4);
  uint32_t evcap = cfg->event_log_capacity ? cfg->event_log_capacity : 65536u;
  if (!sharded) {
    okk = okk && alloc_col(p, &d.stats, (size_t)GSIM_STAT_COUNT);
    okk = okk && alloc_col(p, &d.heard_cnt, (size_t)32) && alloc_col(p, &d.conv_tick, (size_t)32);
    okk = okk && alloc_col(p, &d.view_cnt, (size_t)4);
    okk = okk && alloc_col(p, &d.crashed_alive, (size_t)1) && alloc_col(p, &d.crashed_dead_tick, (size_t)1);
    okk = okk && alloc_col(p, &d.evlog, (size_t)evcap) && alloc_col(p, &d.evlog_cursor, (size_t)2);
    okk = okk && alloc_col(p, &d.tick_base, (size_t)1);
    okk = okk && alloc_col(p, &d.done_ctr, (size_t)1);  // grid barrier of multi-tick launches
    okk = okk && alloc_col(p, &d.qstate[0], (size_t)GS_Q_WORDS);
    okk = okk && alloc_col(p, &p->g_dev, (size_t)1);
  } else if (okk) {
    // pool-wide words: one 2 MB page per rank; counters and the event log live in rank 0's
    p->pages = reinterpret_cast<uint8_t*>(be->shard_alloc(GS_PAGE_BYTES, 1));
    okk = p->pages != nullptr && be->shard_commit(&p->shard_fds, &p->n_shard_fds);
    if (okk) {
      uint8_t* page0 = p->pages;
      uint8_t* mine = p->pages + (size_t)p->rank * GS_PAGE_BYTES;
      d.stats = reinterpret_cast<unsigned long long*>(mine + GS_PG_STATS);  // per rank, summed on read
      d.heard_cnt = reinterpret_cast<uint32_t*>(page0 + GS_PG_HEARD_CNT);
      d.conv_tick = reinterpret_cast<uint32_t*>(page0 + GS_PG_CONV_TICK);
      d.view_cnt = reinterpret_cast<uint32_t*>(page0 + GS_PG_VIEW_CNT);
      d.crashed_alive = reinterpret_cast<uint32_t*>(page0 + GS_PG_CRASHED_ALIVE);
      d.crashed_dead_tick = reinterpret_cast<uint32_t*>(page0 + GS_PG_CRASHED_DEAD_TICK);
      d.evlog_cursor = reinterpret_cast<uint32_t*>(page0 + GS_PG_EVLOG_CURSOR);
      d.evlog = reinterpret_cast<GsEventRec*>(page0 + GS_PG_EVLOG);
      const uint32_t room = (GS_PAGE_BYTES - GS_PG_EVLOG) / (uint32_t)sizeof(GsEventRec);
      if (evcap > room) evcap = room;
      d.tick_base = reinterpret_cast<uint32_t*>(mine + GS_PG_TICK_BASE);
      p->g_dev = reinterpret_cast<GsGlobals*>(mine + GS_PG_GLOBALS);
      for (uint32_t r = 0; r < GS_MAX_WORLD; ++r)
        p->xb.flags[r] = reinterpret_cast<uint32_t*>(p->pages + (size_t)(r < p->world ? r : 0) * GS_PAGE_BYTES + GS_PG_XBAR_FLAGS);
      for (uint32_t r = 0; r < GS_MAX_WORLD; ++r)
        d.tick_flags[r] = reinterpret_cast<uint32_t*>(p->pages + (size_t)(r < p->world ? r : 0) * GS_PAGE_BYTES + GS_PG_TICK_FLAGS);
      d.done_ctr = reinterpret_cast<uint32_t*>(mine + GS_PG_DONE_CTR);
      for (uint32_t r = 0; r < p->world; ++r)
        d.qstate[r] = reinterpret_cast<uint32_t*>(p->pages + (size_t)r * GS_PAGE_BYTES + GS_PG_QSTATE);
      p->xb.epoch = reinterpret_cast<uint32_t*>(mine + GS_PG_XBAR_EPOCH);
      p->xb.rank = p->rank;
      p->xb.world = p->world;
      // peers write barrier flags into this page as soon as they have mapped it: zero it now
      okk = be->fill8(mine, 0, GS_PAGE_BYTES) && be->sync();
    }
  }
  if (!okk) {
    g_create_err = be->last_error();
    fprintf(stderr, "libgsim: allocation failed: %s\n", be->last_error());
    gsim_pool_destroy(p);
    return GSIM_ERR_NOMEM;
  }

  g.n = cfg->n_initial;
  p->n_established = cfg->n_initial;
  g.cap = (uint32_t)cap;
  g.up_count = cfg->n_initial;
  g.P = (uint32_t)(cfg->probe_interval_ns / tick);
  g.T = (uint32_t)(cfg->probe_timeout_ns / tick);
  g.GI = (uint32_t)(cfg->gossip_interval_ns / tick);
  g.gossip_nodes = cfg->gossip_nodes;
  g.indirect_checks = cfg->indirect_checks;
  g.awareness_max = cfg->awareness_max_multiplier;
  g.gtd_ticks = ceil_ticks(cfg->gossip_to_the_dead_ns, tick);
  // [U] memberlist/state.go gossip(): bytesAvail = UDPBufferSize - compoundHeaderOverhead(2)
  g.udp_avail = cfg->udp_buffer_size > 2 ? cfg->udp_buffer_size - 2 : 0;
  g.disable_tcp = cfg->disable_tcp_pings;
  g.loss_thr = (uint32_t)(((uint64_t)cfg->packet_loss_ppm << 32) / 1000000ull);
  if (cfg->packet_loss_ppm >= 1000000u) g.loss_thr = 0xFFFFFFFFu;
  g.event_buffer = cfg->event_buffer;
  g.seed_lo = (uint32_t)cfg->seed;
  g.seed_hi = (uint32_t)(cfg->seed >> 32);
  g.flags = cfg->flags;
  if (getenv("GSIM_NO_FAST_GOSSIP") != nullptr) g.flags |= GSIM_FLAG_NO_FAST_GOSSIP;  // measurement knob
  g.evlog_cap = evcap;
  g.world = cfg->world_size;
  g.rank = cfg->rank;
  g.phase_group = phase_group;
  g.phase_gate = (phase_group % GS_TILE == 0) ? 1u : 0u;
  g.phase_shift = 0;
  while (g.phase_gate && (GS_TILE << g.phase_shift) < phase_group) g.phase_shift++;
  {
    const uint32_t rot = gs_phase_rot(g.seed_lo, g.seed_hi);
    g.rot_p = rot % g.P;
    g.rot_g = (rot >> 16) % g.GI;
  }
  g.rows_per_rank = (uint32_t)p->rows_per_rank;
  g.tick_seconds = (double)tick / 1.0e9;
  g.coord_base_rtt_s = 0.0005;  // a direct ack inside one tick: half a millisecond on top of the matrix
  recompute_tables(p);
  if (!sharded && init_device_state(p) != GSIM_OK) {  // sharded pools: gsim_shard_ready
    g_create_err = be->last_error();
    fprintf(stderr, "libgsim: pool init failed: %s\n", be->last_error());
    gsim_pool_destroy(p);
    return GSIM_ERR_CUDA;
  }
  *out = p;
  return GSIM_OK;
}

// ---- sharded pools: wiring the ranks together ------------------------------------------------------
extern "C" int gsim_shard_export_fds(gsim_pool* p, int* fds, size_t cap, size_t* n) {
  if (!p || !n || !p->sharded) return GSIM_ERR_INVALID;
  *n = p->n_shard_fds;
  if (fds) {
    if (cap < p->n_shard_fds) return GSIM_ERR_INVALID;
    memcpy(fds, p->shard_fds, p->n_shard_fds * sizeof(int));
  }
  return GSIM_OK;
}

extern "C" int gsim_shard_attach(gsim_pool* p, uint32_t peer_rank, const int* fds, size_t n) {
  if (!p || !p->sharded || p->ready || !fds) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  if (!p->be->shard_attach(peer_rank, fds, n)) return fail(p, GSIM_ERR_CUDA, "shard_attach");
  p->attached += 1;
  return GSIM_OK;
}

extern "C" int gsim_shard_ready(gsim_pool* p) {
  if (!p) return GSIM_ERR_INVALID;
  if (!p->sharded) return GSIM_OK;
  std::lock_guard<std::mutex> lk(p->mu);
  if (p->ready) return GSIM_OK;
  if (p->attached != p->world) return fail(p, GSIM_ERR_STATE, "not every peer rank has been attached");
  if (!p->be->xbar_host(p->xb)) return fail(p, GSIM_ERR_CUDA, "barrier");  // every page is mapped and zeroed
  int rc = controller_call(p, nullptr, 0, [&]() -> int { return init_device_state(p); });
  if (rc) return fail(p, rc, "init");
  p->ready = true;
  return GSIM_OK;
}

extern "C" void gsim_pool_destroy(gsim_pool* p) {
  if (!p) return;
  if (p->be) {
    p->be->sync();
    if (p->stage) p->be->host_free(p->stage);
    delete p->workers;
    p->workers = nullptr;
    for (void* q : p->allocs) p->be->release(q);
    delete p->be;
  }
  delete p;
}

// ---- rumor slots --------------------------------------------------------------
static void shard_rows(const gsim_pool* p, uint32_t* first, uint32_t* count) {
  const uint32_t n = p->g.n;
  *first = 0;
  *count = n;
  if (p->sharded) {
    const uint64_t f = (uint64_t)p->rank * p->rows_per_rank;
    *first = f < n ? (uint32_t)f : n;
    *count = *first + p->rows_per_rank < n ? (uint32_t)p->rows_per_rank : n - *first;
  }
}

// Sharded pools count rank by rank: every rank runs the count over ITS rows (local HBM instead of a
// walk of the whole pool over NVLink from GPU 0) and leaves the partial in rank 0's page; the
// controller sums them in do_recount as long as nothing was written since.  Called by every rank,
// outside controller_call, right before a call whose controller side wants counts.
static int collective_recount(gsim_pool* p) {
  if (!p->sharded || !p->ready) return GSIM_OK;
  static_assert(sizeof(GsRecount) <= 512 && GS_PG_SCRATCH + 512u * GS_MAX_WORLD_ <= GS_PG_BLOB, "partial counts");
  GsRecount part;
  uint32_t first, count;
  shard_rows(p, &first, &count);
  // (the device copy of the globals is current: every controller call ends with the upload)
  const bool usable = !(p->rank == 0 && p->g_dirty);
  if (!p->be->recount(p->d, p->g_dev, p->g, p->now, first, count, &part)) return GSIM_ERR_CUDA;
  if (!p->be->h2d(p->pages + GS_PG_SCRATCH + 512u * p->rank, &part, sizeof(part))) return GSIM_ERR_CUDA;
  if (!p->be->xbar_host(p->xb)) return GSIM_ERR_CUDA;
  if (p->rank == 0) {
    p->partials_fresh = usable;
    p->partials_seq = p->dirty_seq;
    p->partials_now = p->now;
  }
  return GSIM_OK;
}

static bool do_recount(gsim_pool* p) {
  if (!p->counts_stale) return true;
  if (!upload_globals(p)) return false;
  if (p->sharded && p->partials_fresh && p->partials_seq == p->dirty_seq && p->partials_now == p->now) {
    std::vector<uint8_t> raw(512u * p->world);
    if (!p->be->d2h(raw.data(), p->pages + GS_PG_SCRATCH, raw.size())) return false;
    memset(&p->rc, 0, sizeof(p->rc));
    uint32_t* sum = reinterpret_cast<uint32_t*>(&p->rc);
    for (uint32_t r = 0; r < p->world; ++r) {
      GsRecount part;
      memcpy(&part, raw.data() + 512u * r, sizeof(part));
      const uint32_t* w = reinterpret_cast<const uint32_t*>(&part);
      for (size_t x = 0; x < sizeof(GsRecount) / 4; ++x) sum[x] += w[x];
    }
  } else if (!p->be->recount(p->d, p->g_dev, p->g, p->now, 0u, p->g.n, &p->rc)) {
    return false;
  }
  p->counts_stale = false;
  return true;
}

static bool and_bit_columns(gsim_pool* p, uint32_t keep);

static int retire_slot(gsim_pool* p, uint32_t slot) {
  GsGlobals& g = p->g;
  GsRumor& ru = g.rumors[slot];
  if (ru.kind == GSIM_RUMOR_ALIVE) {
    // fold into the base state: the subject becomes known to every non-isolated member
    uint32_t k0, k1;
    if (!peek(p, p->d.key[0], ru.subject, &k0) || !peek(p, p->d.key[1], ru.subject, &k1))
      return GSIM_ERR_CUDA;
    if (gs_key_pending(k0)) p->n_established += 1;
    k0 &= ~(1u << 4);
    k1 &= ~(1u << 4);
    if (!poke_key(p, 0, ru.subject, k0) || !poke_key(p, 1, ru.subject, k1))
      return GSIM_ERR_CUDA;
  }
  g.active_mask &= ~(1u << slot);
  memset(&ru, 0, sizeof(ru));
  p->rh[slot] = RumorHost();
  rebuild_class_masks(p);
  if (!and_bit_columns(p, ~(1u << slot))) return GSIM_ERR_CUDA;
  if (!poke(p, p->d.heard_cnt, slot, 0u) || !poke(p, p->d.conv_tick, slot, GS_EMPTY32))
    return GSIM_ERR_CUDA;
  counts_invalidate(p);
  return GSIM_OK;
}

// heard/queued/inbox bits of a freed slot must be zero before the slot is reused.
static bool and_bit_columns(gsim_pool* p, uint32_t keep) {
  mark_dirty(p);
  if (p->sharded && p->defer_and) {  // step boundary: every rank clears its own rows after the call
    p->pending_keep &= keep;
    return true;
  }
  return p->be->and_columns(p->d, p->g, keep, 0u, p->g.n);
}

// ... which is this, on every rank, right after the controller call that collected the mask.
static int apply_pending_and(gsim_pool* p) {
  if (!p->sharded || p->pending_keep == 0xFFFFFFFFu) return GSIM_OK;
  uint32_t first, count;
  shard_rows(p, &first, &count);
  const bool ok = p->be->and_columns(p->d, p->g, p->pending_keep, first, count) && p->be->sync();
  p->pending_keep = 0xFFFFFFFFu;
  // nobody goes on (to reuse a freed slot, to tick) before every rank's rows are clean
  if (!ok || !p->be->xbar_host(p->xb)) return GSIM_ERR_CUDA;
  return GSIM_OK;
}

// Retire finished membership rumors (alive / intents): every UP member has heard them and
// nobody is retransmitting any more.  Runs at step boundaries only.
static int auto_retire(gsim_pool* p) {
  GsGlobals& g = p->g;
  uint32_t cand = 0;
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r)
    if (((g.active_mask >> r) & 1u) && g.rumors[r].kind != GSIM_RUMOR_USER_EVENT) cand |= 1u << r;
  if (!cand) return GSIM_OK;
  if (!do_recount(p)) return GSIM_ERR_CUDA;
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r) {
    if (!((cand >> r) & 1u)) continue;
    // an alive rumor folds into the base set only when nobody still depends on having
    // heard it individually (members that have not joined the base set yet)
    if (g.rumors[r].kind == GSIM_RUMOR_ALIVE && p->rc.isolated_up != 0) continue;
    if (p->rc.heard_cnt[r] == g.up_count && p->rc.queued_cnt[r] == 0) {
      int rcode = retire_slot(p, r);
      if (rcode) return rcode;
    }
  }
  return GSIM_OK;
}

static int alloc_slot(gsim_pool* p, uint32_t* slot_out) {
  GsGlobals& g = p->g;
  for (int attempt = 0; attempt < 2; ++attempt) {
    for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r)
      if (!((g.active_mask >> r) & 1u)) {
        *slot_out = r;
        return GSIM_OK;
      }
    if (attempt == 0) {
      int rc = auto_retire(p);
      if (rc) return rc;
    }
  }
  return GSIM_ERR_CAPACITY;
}

// A member whose broadcast queue became non-empty between ticks must be looked at by the
// next tick: set the wake bit in the mailbox that tick will read.
static bool post_wake(gsim_pool* p, uint32_t row) {
  uint32_t* col = p->d.inbox[p->now & p->g.ring_mask];
  uint32_t w;
  if (!peek(p, col, row, &w)) return false;
  return poke(p, col, row, w | GS_WAKE_BIT);
}

// ---- message sizes: what the encoder (gs_wire.h) produces for this member ------------------------
// A virtual member is called "node-<id>" unless gsim_member_desc.name_len said otherwise.
static uint32_t member_name_len(const gsim_pool* p, uint32_t id) {
  for (const auto& kv : p->name_lens)
    if (kv.first == id) return kv.second;
  uint32_t digits = 1;
  for (uint32_t v = id; v >= 10u; v /= 10u) ++digits;
  return 5u + digits;
}
static uint32_t alive_size(const gsim_pool* p, uint32_t id, uint32_t inc, uint32_t meta_len) {
  static const uint8_t vsn[6] = {1, 5, 2, 2, 5, 4}, addr[4] = {10, 0, 0, 1};
  static const char none = 0;
  return (uint32_t)gsw::alive(nullptr, 0, inc, nullptr, member_name_len(p, id), addr, 4, 8301, &none, meta_len, vsn);
}
static uint32_t intent_size(const gsim_pool* p, uint32_t id, bool leave, uint32_t ltime) {
  return (uint32_t)gsw::serf_intent(nullptr, 0, leave, ltime, nullptr, member_name_len(p, id), false, false);
}

static int start_rumor(gsim_pool* p, uint32_t slot, uint32_t kind, uint32_t subject, uint32_t inc,
                       uint32_t ltime, uint32_t origin, uint32_t size, uint32_t qclass) {
  GsGlobals& g = p->g;
  GsRumor& ru = g.rumors[slot];
  ru.kind = kind;
  ru.subject = subject;
  ru.inc = inc;
  ru.ltime = ltime;
  ru.origin = origin;
  ru.size = size;
  ru.qclass = qclass;
  ru.start_tick = p->now;
  g.active_mask |= 1u << slot;
  rebuild_class_masks(p);
  // the origin holds it with transmits = 0
  uint32_t h, q;
  if (!peek(p, p->d.heard, origin, &h) || !peek(p, p->d.queued, origin, &q)) return GSIM_ERR_CUDA;
  h |= 1u << slot;
  q |= 1u << slot;
  if (!poke(p, p->d.heard, origin, h) || !poke(p, p->d.queued, origin, q)) return GSIM_ERR_CUDA;
  if (!poke(p, p->d.tx, GS_TX(slot, g.cap, origin), (uint8_t)0)) return GSIM_ERR_CUDA;
  if (!post_wake(p, origin)) return GSIM_ERR_CUDA;
  if (!poke(p, p->d.heard_cnt, slot, 1u)) return GSIM_ERR_CUDA;
  if (!poke(p, p->d.conv_tick, slot, g.up_count == 1u ? p->now : GS_EMPTY32)) return GSIM_ERR_CUDA;
  counts_invalidate(p);
  return GSIM_OK;
}

static void log_host_event(gsim_pool* p, uint32_t type, uint32_t subject, uint32_t observer,
                           uint32_t ltime) {
  uint32_t cur[2];
  if (!p->be->d2h(cur, p->d.evlog_cursor, 8)) return;
  if (cur[0] < p->g.evlog_cap) {
    GsEventRec e = {p->now, type, subject, observer, ltime, 0u};
    p->be->h2d(p->d.evlog + cur[0], &e, sizeof(e));
    cur[0]++;
  } else {
    cur[1]++;
  }
  p->be->h2d(p->d.evlog_cursor, cur, 8);
}

// ---- membership operations -------------------------------------------------------
extern "C" int gsim_member_add(gsim_pool* p, const gsim_member_desc* desc, uint32_t* id_out) {
  if (!p || !id_out) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, id_out, sizeof(uint32_t), [&]() -> int {
  GsGlobals& g = p->g;
  if (g.graph_n) return fail(p, GSIM_ERR_STATE, "the peer graph of this pool is static (gsim_graph_set)");
  if (g.n >= p->cfg.capacity) return fail(p, GSIM_ERR_CAPACITY, "member capacity exhausted");
  uint32_t slot;
  int rc = alloc_slot(p, &slot);
  if (rc) return fail(p, rc, "no free rumor slot for the member's alive broadcast");
  const uint32_t id = g.n;
  if (!upload_globals(p)) return fail(p, GSIM_ERR_CUDA, "upload");
  if (!p->be->init_rows(p->d, p->g_dev, g, id, 1, p->now)) return fail(p, GSIM_ERR_CUDA, "init_rows");
  // [U] memberlist.Create -> setAlive: incarnation 1, alive{} queued on the new member;
  // pending: other members learn of it only through that rumor (aliveNode).
  const uint32_t k = gs_key_make(1u, 1u, GS_RANK_ALIVE, GS_TRUTH_UP);
  uint32_t m;
  if (!peek(p, p->d.meta, id, &m)) return fail(p, GSIM_ERR_CUDA, "peek");
  // it knows nobody yet; with an empty base set there is nothing it could be missing
  if (p->n_established > 0) m |= GS_META_ISOLATED;
  if (desc && (desc->flags & GSIM_MEMBER_WATCHED)) m |= GS_META_WATCHED;
  if (!poke_key(p, 0, id, k) || !poke_key(p, 1, id, k) || !poke(p, p->d.meta, id, m))
    return fail(p, GSIM_ERR_CUDA, "poke");
  g.n += 1;
  g.up_count += 1;
  recompute_tables(p);
  if (desc && desc->name_len) p->name_lens.push_back(std::make_pair(id, desc->name_len));
  uint32_t size = desc && desc->alive_msg_size ? desc->alive_msg_size : alive_size(p, id, 1u, desc ? desc->meta_len : 0u);
  rc = start_rumor(p, slot, GSIM_RUMOR_ALIVE, id, 1u, 0u, id, size, 0u);
  if (rc) return fail(p, rc, "start_rumor");
  *id_out = id;
  return GSIM_OK;
  });
}

// One direction of a join push-pull: `dst` merges what `src` knows
// ([U] memberlist.mergeState -> aliveNode; [U] serf/delegate.go MergeRemoteState).
static int merge_remote(gsim_pool* p, uint32_t dst, uint32_t src, bool ignore_old_events) {
  GsGlobals& g = p->g;
  uint32_t rs[8], rd[8];  // {key0, key1, meta, heard, queued, ltime_member, ltime_event, event_min} of both ends
  if (!p->be->row_read(p->d, src, rs) || !p->be->row_read(p->d, dst, rd)) return GSIM_ERR_CUDA;
  uint32_t hs = rs[3], hd = rd[3], qd = rd[4], lm_s = rs[5], le_s = rs[6], lm_d = rd[5], le_d = rd[6], emin = rd[7], md = rd[2];
  // clocks: Witness(remote - 1)  ==  max(local, remote)
  if (lm_s > lm_d) lm_d = lm_s;
  if (le_s > le_d) le_d = le_s;
  if (ignore_old_events && le_s > emin) emin = le_s;  // eventMinTime = pp.EventLTime
  uint32_t fresh = hs & ~hd & g.active_mask;
  uint32_t accepted = 0;
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r) {
    if (!((fresh >> r) & 1u)) continue;
    const GsRumor& ru = g.rumors[r];
    bool accept = true;
    if (ru.kind == GSIM_RUMOR_USER_EVENT) {
      if (ru.ltime >= le_d) le_d = ru.ltime + 1u;
      if (ru.ltime < emin) accept = false;
      else if (le_d > g.event_buffer && ru.ltime < le_d - g.event_buffer) accept = false;
      if (accept && (md & GS_META_WATCHED)) log_host_event(p, GSIM_EVENT_USER, r, dst, ru.ltime);
    } else if (ru.kind == GSIM_RUMOR_JOIN_INTENT || ru.kind == GSIM_RUMOR_LEAVE_INTENT) {
      if (ru.ltime >= lm_d) lm_d = ru.ltime + 1u;
    } else if (ru.kind == GSIM_RUMOR_ALIVE) {
      if (md & GS_META_WATCHED) log_host_event(p, GSIM_EVENT_MEMBER_JOIN, ru.subject, dst, 0u);
    } else if (ru.kind == GSIM_RUMOR_UPDATE) {
      if (md & GS_META_WATCHED) log_host_event(p, GSIM_EVENT_MEMBER_UPDATE, ru.subject, dst, 0u);
    }
    if (accept) {
      accepted |= 1u << r;
      if (!poke(p, p->d.tx, GS_TX(r, g.cap, dst), (uint8_t)0)) return GSIM_ERR_CUDA;
      uint32_t c;
      if (!peek(p, p->d.heard_cnt, r, &c)) return GSIM_ERR_CUDA;
      c += 1;
      if (!poke(p, p->d.heard_cnt, r, c)) return GSIM_ERR_CUDA;
      if (c == g.up_count) {
        uint32_t ct;
        if (!peek(p, p->d.conv_tick, r, &ct)) return GSIM_ERR_CUDA;
        if (ct == GS_EMPTY32 && !poke(p, p->d.conv_tick, r, p->now)) return GSIM_ERR_CUDA;
      }
    }
  }
  hd |= accepted;
  qd |= accepted;
  if (accepted && !post_wake(p, dst)) return GSIM_ERR_CUDA;
  if (!poke(p, p->d.heard, dst, hd) || !poke(p, p->d.queued, dst, qd) ||
      !poke(p, p->d.ltime_member, dst, lm_d) || !poke(p, p->d.ltime_event, dst, le_d) ||
      !poke(p, p->d.event_min, dst, emin))
    return GSIM_ERR_CUDA;
  counts_invalidate(p);
  return GSIM_OK;
}

extern "C" int gsim_join(gsim_pool* p, uint32_t id, const uint32_t* seeds, size_t n_seeds,
                         int ignore_old, int* n_ok) {
  if (!p || (!seeds && n_seeds)) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  int n_ok_local = 0;
  if (!n_ok) n_ok = &n_ok_local;
  return controller_call(p, n_ok, sizeof(int), [&]() -> int {
  GsGlobals& g = p->g;
  if (id >= g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  uint32_t kid;
  if (!peek(p, p->d.key[p->now & 1u], id, &kid)) return fail(p, GSIM_ERR_CUDA, "peek");
  if (gs_key_truth(kid) != GS_TRUTH_UP) return fail(p, GSIM_ERR_STATE, "member is not running");
  int okc = 0;
  for (size_t s = 0; s < n_seeds; ++s) {
    uint32_t sd = seeds[s];
    if (sd >= g.n || sd == id) continue;
    uint32_t ks;
    if (!peek(p, p->d.key[p->now & 1u], sd, &ks)) return fail(p, GSIM_ERR_CUDA, "peek");
    if (gs_key_truth(ks) != GS_TRUTH_UP) continue;  // unreachable seed: Join skips it
    // push-pull in both directions; eventJoinIgnore applies to the joiner only
    int rc = merge_remote(p, id, sd, ignore_old != 0);
    if (!rc) rc = merge_remote(p, sd, id, false);
    if (rc) return fail(p, rc, "merge");
    uint32_t mi, ms;
    if (!peek(p, p->d.meta, id, &mi) || !peek(p, p->d.meta, sd, &ms)) return fail(p, GSIM_ERR_CUDA, "peek");
    uint32_t iso = mi & ms & GS_META_ISOLATED;
    mi = (mi & ~GS_META_ISOLATED) | iso;
    ms = (ms & ~GS_META_ISOLATED) | iso;
    if (!poke(p, p->d.meta, id, mi) || !poke(p, p->d.meta, sd, ms)) return fail(p, GSIM_ERR_CUDA, "poke");
    ++okc;
  }
  if (okc > 0) {
    // [U] serf.Join -> broadcastJoin(clock.Time()): Witness(ltime), join intent queued
    uint32_t lm;
    if (!peek(p, p->d.ltime_member, id, &lm)) return fail(p, GSIM_ERR_CUDA, "peek");
    uint32_t slot;
    int rc = alloc_slot(p, &slot);
    if (rc == GSIM_OK) {
      rc = start_rumor(p, slot, GSIM_RUMOR_JOIN_INTENT, id, 0u, lm, id, intent_size(p, id, false, lm), 1u);
      if (rc) return fail(p, rc, "start_rumor");
    } else if (rc != GSIM_ERR_CAPACITY) {
      return fail(p, rc, "alloc_slot");
    }
    if (!poke(p, p->d.ltime_member, id, lm + 1u)) return fail(p, GSIM_ERR_CUDA, "poke");
  }
  if (n_ok) *n_ok = okc;
  return GSIM_OK;
  });
}

static int set_truth(gsim_pool* p, uint32_t id, uint32_t truth) {
  for (int b = 0; b < 2; ++b) {
    uint32_t k;
    if (!peek(p, p->d.key[b], id, &k)) return GSIM_ERR_CUDA;
    k = (k & ~3u) | truth;
    if (!poke_key(p, b, id, k)) return GSIM_ERR_CUDA;
  }
  return GSIM_OK;
}

static int refresh_after_truth_change(gsim_pool* p) {
  counts_invalidate(p);
  if (!do_recount(p)) return GSIM_ERR_CUDA;
  GsGlobals& g = p->g;
  g.up_count = p->rc.truth_cnt[GS_TRUTH_UP];
  p->g_dirty = true;
  if (!poke(p, p->d.crashed_alive, 0, p->rc.crashed_alive)) return GSIM_ERR_CUDA;
  uint32_t cdt = GS_EMPTY32;
  if (p->rc.crashed_alive == 0 && p->rc.truth_cnt[GS_TRUTH_CRASHED] > 0) cdt = p->now;
  if (!poke(p, p->d.crashed_dead_tick, 0, cdt)) return GSIM_ERR_CUDA;
  // heard counters are over UP members only
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r) {
    if (!((g.active_mask >> r) & 1u)) continue;
    if (!poke(p, p->d.heard_cnt, r, p->rc.heard_cnt[r])) return GSIM_ERR_CUDA;
    if (p->rc.heard_cnt[r] == g.up_count) {
      uint32_t ct;
      if (!peek(p, p->d.conv_tick, r, &ct)) return GSIM_ERR_CUDA;
      if (ct == GS_EMPTY32 && !poke(p, p->d.conv_tick, r, p->now)) return GSIM_ERR_CUDA;
    }
  }
  return GSIM_OK;
}

extern "C" int gsim_crash_many(gsim_pool* p, const uint32_t* ids, size_t n) {
  if (!p || (!ids && n)) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, nullptr, 0, [&]() -> int {
  for (size_t x = 0; x < n; ++x) {
    if (ids[x] >= p->g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
    uint32_t k;
    if (!peek(p, p->d.key[p->now & 1u], ids[x], &k)) return fail(p, GSIM_ERR_CUDA, "peek");
    if (gs_key_truth(k) != GS_TRUTH_UP) continue;
    int rc = set_truth(p, ids[x], GS_TRUTH_CRASHED);
    if (rc) return fail(p, rc, "set_truth");
  }
  int rc = refresh_after_truth_change(p);
  return rc ? fail(p, rc, "recount") : GSIM_OK;
  });
}

extern "C" int gsim_crash(gsim_pool* p, uint32_t id) { return gsim_crash_many(p, &id, 1); }

extern "C" int gsim_crash_fraction(gsim_pool* p, uint32_t ppm, uint32_t salt, uint32_t* n_crashed) {
  if (!p || ppm > 1000000u) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  uint32_t n_crashed_local = 0;
  if (!n_crashed) n_crashed = &n_crashed_local;
  return controller_call(p, n_crashed, sizeof(uint32_t), [&]() -> int {
  uint32_t thr = ppm >= 1000000u ? 0xFFFFFFFFu : (uint32_t)(((uint64_t)ppm << 32) / 1000000ull);
  uint32_t cnt = 0;
  if (!upload_globals(p)) return fail(p, GSIM_ERR_CUDA, "upload");
  mark_dirty(p);
  if (!p->be->crash_fraction(p->d, p->g_dev, p->g, thr, salt, p->now, &cnt))
    return fail(p, GSIM_ERR_CUDA, "crash_fraction");
  if (n_crashed) *n_crashed = cnt;
  int rc = refresh_after_truth_change(p);
  return rc ? fail(p, rc, "recount") : GSIM_OK;
  });
}

// (*Serf).SetTags -> [U] memberlist.UpdateNode: the member re-announces itself with new meta under
// the next incarnation; every receiver's aliveNode takes the higher incarnation and raises
// NotifyUpdate -> serf EventMemberUpdate.  The tags themselves stay on the host (SURVEY 8b).
extern "C" int gsim_member_update(gsim_pool* p, uint32_t id, uint32_t alive_msg_size, uint32_t* slot_out) {
  if (!p) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  uint32_t slot_local = 0;
  if (!slot_out) slot_out = &slot_local;
  return controller_call(p, slot_out, sizeof(uint32_t), [&]() -> int {
  GsGlobals& g = p->g;
  if (id >= g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  uint32_t k, m;
  if (!peek(p, p->d.key[p->now & 1u], id, &k) || !peek(p, p->d.meta, id, &m))
    return fail(p, GSIM_ERR_CUDA, "peek");
  if (gs_key_truth(k) != GS_TRUTH_UP || (m & GS_META_LEAVING))
    return fail(p, GSIM_ERR_STATE, "member is not running");
  uint32_t slot;
  int rc = alloc_slot(p, &slot);
  if (rc) return fail(p, rc, "no free rumor slot");
  const uint32_t inc = gs_key_inc(k) + 1u;  // nextIncarnation
  for (int b = 0; b < 2; ++b) {
    uint32_t kk;
    if (!peek(p, p->d.key[b], id, &kk)) return fail(p, GSIM_ERR_CUDA, "peek");
    if (!poke_key(p, b, id, gs_key_with_inc(kk, inc))) return fail(p, GSIM_ERR_CUDA, "poke");
  }
  rc = start_rumor(p, slot, GSIM_RUMOR_UPDATE, id, inc, 0u, id, alive_msg_size ? alive_msg_size : alive_size(p, id, inc, 0u), 0u);
  if (rc) return fail(p, rc, "start_rumor");
  *slot_out = slot;
  return GSIM_OK;
  });
}

extern "C" int gsim_leave(gsim_pool* p, uint32_t id) {
  if (!p) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, nullptr, 0, [&]() -> int {
  GsGlobals& g = p->g;
  if (id >= g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  uint32_t k, m;
  if (!peek(p, p->d.key[p->now & 1u], id, &k) || !peek(p, p->d.meta, id, &m))
    return fail(p, GSIM_ERR_CUDA, "peek");
  if (gs_key_truth(k) != GS_TRUTH_UP || (m & GS_META_LEAVING))
    return fail(p, GSIM_ERR_STATE, "member is not running or already leaving");
  // [U] serf.Leave: leave intent with the member clock, then memberlist.Leave broadcasts
  // dead{Node == From} which every receiver records as StateLeft.
  uint32_t lm;
  if (!peek(p, p->d.ltime_member, id, &lm)) return fail(p, GSIM_ERR_CUDA, "peek");
  uint32_t slot;
  int rc = alloc_slot(p, &slot);
  if (rc == GSIM_OK) {
    rc = start_rumor(p, slot, GSIM_RUMOR_LEAVE_INTENT, id, 0u, lm, id, intent_size(p, id, true, lm), 1u);
    if (rc) return fail(p, rc, "start_rumor");
  } else if (rc != GSIM_ERR_CAPACITY) {
    return fail(p, rc, "alloc_slot");
  }
  if (!poke(p, p->d.ltime_member, id, lm + 1u)) return fail(p, GSIM_ERR_CUDA, "poke");
  for (int b = 0; b < 2; ++b) {
    uint32_t kk;
    if (!peek(p, p->d.key[b], id, &kk)) return fail(p, GSIM_ERR_CUDA, "peek");
    kk = gs_key_with_rank(kk, GS_RANK_LEFT);
    if (!poke_key(p, b, id, kk)) return fail(p, GSIM_ERR_CUDA, "poke");
  }
  m |= GS_META_LEAVING;
  if (!poke(p, p->d.meta, id, m) || !poke(p, p->d.change_tick, id, p->now))
    return fail(p, GSIM_ERR_CUDA, "poke");
  if (g.flags & GSIM_FLAG_LOG_GLOBAL_EVENTS) log_host_event(p, GSIM_EVENT_MEMBER_LEAVE, id, GS_EMPTY32, 0);
  // the process lingers while its two broadcasts drain, then LeavePropagateDelay
  uint32_t rounds = g.gossip_nodes ? (g.retransmit_limit + g.gossip_nodes - 1) / g.gossip_nodes : 0;
  uint32_t drain = rounds * g.GI;
  uint32_t bt = ceil_ticks(p->cfg.broadcast_timeout_ns, p->tick_ns);
  if (drain > bt) drain = bt;
  uint32_t linger = 2 * drain + ceil_ticks(p->cfg.leave_propagate_delay_ns, p->tick_ns);
  Sched s = {p->now + linger, id, 1u};
  p->sched.push_back(s);
  counts_invalidate(p);
  return GSIM_OK;
  });
}

extern "C" int gsim_force_leave(gsim_pool* p, uint32_t via, uint32_t target, int prune) {
  if (!p) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, nullptr, 0, [&]() -> int {
  if (via >= p->g.n || target >= p->g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  // [U] serf.RemoveFailedNode: a forged leave intent turns Failed into Left.  The decision is
  // taken on the member's CURRENT record (the buffer the next tick reads); the other buffer may
  // still hold the previous state (DIRTY), so the result is written to both and DIRTY is dropped.
  uint32_t k, m;
  if (!peek(p, p->d.key[p->now & 1u], target, &k) || !peek(p, p->d.meta, target, &m))
    return fail(p, GSIM_ERR_CUDA, "peek");
  const uint32_t k_before = k;
  if (gs_key_rank(k) == GS_RANK_DEAD) k = gs_key_with_rank(k, GS_RANK_LEFT);
  if (prune && gs_key_rank(k) == GS_RANK_LEFT && gs_key_truth(k) != GS_TRUTH_UP && gs_key_truth(k) != GS_TRUTH_NONE) {
    if (!gs_key_pending(k)) p->n_established -= 1;
    k &= ~3u;
  }
  if (k != k_before) {
    if (!poke_key(p, 0, target, k) || !poke_key(p, 1, target, k)) return fail(p, GSIM_ERR_CUDA, "poke");
    if ((m & GS_META_DIRTY) && !poke(p, p->d.meta, target, m & ~GS_META_DIRTY)) return fail(p, GSIM_ERR_CUDA, "poke");
  }
  int rc = refresh_after_truth_change(p);
  return rc ? fail(p, rc, "recount") : GSIM_OK;
  });
}

extern "C" int gsim_user_event(gsim_pool* p, uint32_t id, const void* name, size_t name_len,
                               const void* payload, size_t payload_len, int coalesce,
                               uint32_t* slot_out) {
  if (!p || (!name && name_len) || (!payload && payload_len)) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  uint32_t slot_local = 0;
  if (!slot_out) slot_out = &slot_local;
  return controller_call(p, slot_out, sizeof(uint32_t), [&]() -> int {
  GsGlobals& g = p->g;
  if (id >= g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  // [U] serf.UserEvent: size limit on name+payload (agent side: user_event.go:82-113)
  if (name_len + payload_len > p->cfg.user_event_size_limit)
    return fail(p, GSIM_ERR_TOO_LARGE, "user event exceeds UserEventSizeLimit");
  uint32_t k, m;
  if (!peek(p, p->d.key[p->now & 1u], id, &k) || !peek(p, p->d.meta, id, &m))
    return fail(p, GSIM_ERR_CUDA, "peek");
  if (gs_key_truth(k) != GS_TRUTH_UP) return fail(p, GSIM_ERR_STATE, "member is not running");
  uint32_t le;
  if (!peek(p, p->d.ltime_event, id, &le)) return fail(p, GSIM_ERR_CUDA, "peek");
  std::string nm((const char*)name, name_len), pl((const char*)payload, payload_len);
  // identical (LTime, Name, Payload) is the same event for serf's de-dup ring
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r) {
    if (!((g.active_mask >> r) & 1u) || g.rumors[r].kind != GSIM_RUMOR_USER_EVENT) continue;
    if (g.rumors[r].ltime == le && p->rh[r].name == nm && p->rh[r].payload == pl) {
      // [U] serf.UserEvent -> handleUserEvent on the caller's own buffer, then QueueBroadcast: a
      // member that had not seen this (LTime, Name, Payload) delivers it now; either way its copy
      // is (re)queued with transmits = 0.
      uint32_t h, q;
      if (!peek(p, p->d.heard, id, &h) || !peek(p, p->d.queued, id, &q)) return fail(p, GSIM_ERR_CUDA, "peek");
      if (!((h >> r) & 1u)) {
        uint32_t c, ct;
        if (!poke(p, p->d.heard, id, h | (1u << r)) || !peek(p, p->d.heard_cnt, r, &c) ||
            !poke(p, p->d.heard_cnt, r, c + 1u) || !peek(p, p->d.conv_tick, r, &ct))
          return fail(p, GSIM_ERR_CUDA, "poke");
        if (c + 1u == g.up_count && ct == GS_EMPTY32 && !poke(p, p->d.conv_tick, r, p->now))
          return fail(p, GSIM_ERR_CUDA, "poke");
        if (m & GS_META_WATCHED) log_host_event(p, GSIM_EVENT_USER, r, id, le);
      }
      if (!poke(p, p->d.queued, id, q | (1u << r)) || !poke(p, p->d.tx, GS_TX(r, g.cap, id), (uint8_t)0) ||
          !post_wake(p, id) || !poke(p, p->d.ltime_event, id, le + 1u))
        return fail(p, GSIM_ERR_CUDA, "poke");
      counts_invalidate(p);
      if (slot_out) *slot_out = r;
      return GSIM_OK;
    }
  }
  // the encoded messageUserEvent{LTime,Name,Payload,CC} behind its serf type byte
  static const char some = 0;  // (a non-nil payload slice; sizing reads no bytes)
  uint32_t size = (uint32_t)gsw::serf_user_event(nullptr, 0, le, nullptr, name_len, &some, payload_len, coalesce != 0, false);
  // [U] serf.UserEvent checks the limit a second time on the ENCODED message
  if (size > p->cfg.user_event_size_limit)
    return fail(p, GSIM_ERR_TOO_LARGE, "encoded user event exceeds UserEventSizeLimit");
  uint32_t slot;
  int rc = alloc_slot(p, &slot);
  if (rc) return fail(p, rc, "no free rumor slot");
  rc = start_rumor(p, slot, GSIM_RUMOR_USER_EVENT, id, 0u, le, id, size, 2u);
  if (rc) return fail(p, rc, "start_rumor");
  p->rh[slot].name = nm;
  p->rh[slot].payload = pl;
  p->rh[slot].coalesce = coalesce;
  if (!poke(p, p->d.ltime_event, id, le + 1u)) return fail(p, GSIM_ERR_CUDA, "poke");
  if (m & GS_META_WATCHED) log_host_event(p, GSIM_EVENT_USER, slot, id, le);
  if (slot_out) *slot_out = slot;
  return GSIM_OK;
  });
}

// Out-of-band delivery of a tracked broadcast to one member: what arrival by gossip would do, but
// now and by name.  BASELINE config 5's bridge members use it to re-fire an event they delivered
// in one WAN pool into the other (models ForwardRPC, agent/consul/internal_endpoint.go:839).
extern "C" int gsim_rumor_inject(gsim_pool* p, uint32_t slot, uint32_t id, int* accepted_out) {
  if (!p || slot >= GS_MAX_RUMORS) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  int acc_local = 0;
  if (!accepted_out) accepted_out = &acc_local;
  return controller_call(p, accepted_out, sizeof(int), [&]() -> int {
  GsGlobals& g = p->g;
  *accepted_out = 0;
  if (!((g.active_mask >> slot) & 1u)) return fail(p, GSIM_ERR_NOT_FOUND, "slot is free");
  if (id >= g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  uint32_t k, m, h, q, le, lm, emin;
  if (!peek(p, p->d.key[p->now & 1u], id, &k) || !peek(p, p->d.meta, id, &m) ||
      !peek(p, p->d.heard, id, &h) || !peek(p, p->d.queued, id, &q) ||
      !peek(p, p->d.ltime_event, id, &le) || !peek(p, p->d.ltime_member, id, &lm) ||
      !peek(p, p->d.event_min, id, &emin))
    return fail(p, GSIM_ERR_CUDA, "peek");
  if (gs_key_truth(k) != GS_TRUTH_UP) return fail(p, GSIM_ERR_STATE, "member is not running");
  if ((h >> slot) & 1u) return GSIM_OK;  // already delivered: serf's de-dup ring drops it
  const GsRumor& ru = g.rumors[slot];
  bool accept = true;
  if (ru.kind == GSIM_RUMOR_USER_EVENT) {
    if (ru.ltime >= le) le = ru.ltime + 1u;
    if (ru.ltime < emin) accept = false;
    else if (le > g.event_buffer && ru.ltime < le - g.event_buffer) accept = false;
    if (accept && (m & GS_META_WATCHED)) log_host_event(p, GSIM_EVENT_USER, slot, id, ru.ltime);
    if (!poke(p, p->d.ltime_event, id, le)) return fail(p, GSIM_ERR_CUDA, "poke");
  } else if (ru.kind == GSIM_RUMOR_JOIN_INTENT || ru.kind == GSIM_RUMOR_LEAVE_INTENT) {
    if (ru.ltime >= lm) lm = ru.ltime + 1u;
    if (!poke(p, p->d.ltime_member, id, lm)) return fail(p, GSIM_ERR_CUDA, "poke");
  } else if (ru.kind == GSIM_RUMOR_ALIVE) {
    if (m & GS_META_WATCHED) log_host_event(p, GSIM_EVENT_MEMBER_JOIN, ru.subject, id, 0u);
  } else if (ru.kind == GSIM_RUMOR_UPDATE) {
    if (m & GS_META_WATCHED) log_host_event(p, GSIM_EVENT_MEMBER_UPDATE, ru.subject, id, 0u);
  }
  if (!accept) return GSIM_OK;
  uint32_t c, ct;
  if (!poke(p, p->d.heard, id, h | (1u << slot)) || !poke(p, p->d.queued, id, q | (1u << slot)) ||
      !poke(p, p->d.tx, GS_TX(slot, g.cap, id), (uint8_t)0) || !post_wake(p, id) ||
      !peek(p, p->d.heard_cnt, slot, &c) || !poke(p, p->d.heard_cnt, slot, c + 1u) ||
      !peek(p, p->d.conv_tick, slot, &ct))
    return fail(p, GSIM_ERR_CUDA, "poke");
  if (c + 1u == g.up_count && ct == GS_EMPTY32 && !poke(p, p->d.conv_tick, slot, p->now))
    return fail(p, GSIM_ERR_CUDA, "poke");
  counts_invalidate(p);
  *accepted_out = 1;
  return GSIM_OK;
  });
}

// Peer graph in CSR form (north_star: "message-passing kernel over a CSR peer graph"; SURVEY 7):
// member i's memberlist becomes col_idx[row_ptr[i] .. row_ptr[i+1]) — peer selection for gossip,
// indirect-probe relays, push-pull and the probe ring all draw from that row instead of [0, n).
// A graph whose every row is [0, n) reproduces the complete-graph results bit for bit.  Static
// topology: rows for exactly the current members; gsim_member_add is refused while a graph is set.
extern "C" int gsim_graph_set(gsim_pool* p, uint32_t n_rows, const uint32_t* row_ptr, const uint32_t* col_idx) {
  if (!p || (n_rows && (!row_ptr || !col_idx))) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  if (p->sharded) return fail(p, GSIM_ERR_STATE, "peer graphs are not supported on sharded pools");
  GsGlobals& g = p->g;
  if (n_rows == 0) {
    g.graph_n = 0;
    p->d.row_ptr = p->d.col_idx = nullptr;
    p->graph_rp.clear();
    p->graph_col.clear();
    p->g_dirty = true;
    return GSIM_OK;
  }
  if (n_rows != g.n) return fail(p, GSIM_ERR_INVALID, "the graph must have one row per member");
  if (row_ptr[0] != 0) return fail(p, GSIM_ERR_INVALID, "row_ptr[0] must be 0");
  for (uint32_t i = 0; i < n_rows; ++i)
    if (row_ptr[i + 1] < row_ptr[i]) return fail(p, GSIM_ERR_INVALID, "row_ptr must be non-decreasing");
  const uint32_t nnz = row_ptr[n_rows];
  for (uint32_t e = 0; e < nnz; ++e)
    if (col_idx[e] >= g.n) return fail(p, GSIM_ERR_INVALID, "col_idx out of range");
  uint32_t *rp_dev = nullptr, *col_dev = nullptr;
  if (!alloc_col(p, &rp_dev, (size_t)n_rows + 1) || !alloc_col(p, &col_dev, (size_t)(nnz ? nnz : 1)))
    return fail(p, GSIM_ERR_NOMEM, "graph allocation");
  if (!p->be->h2d(rp_dev, row_ptr, ((size_t)n_rows + 1) * 4) || (nnz && !p->be->h2d(col_dev, col_idx, (size_t)nnz * 4)))
    return fail(p, GSIM_ERR_CUDA, "h2d");
  p->graph_rp.assign(row_ptr, row_ptr + n_rows + 1);
  p->graph_col.assign(col_idx, col_idx + nnz);
  p->d.row_ptr = rp_dev;
  p->d.col_idx = col_dev;
  g.graph_n = n_rows;
  p->g_dirty = true;
  return GSIM_OK;
}

// serf.Config.ReconnectTimeoutOverride (internal/gossip/libserf/serf.go:68-85: a member may
// advertise its own reconnect timeout in a tag; agent/consul/client_test.go:862-894).  The callback
// is host code; its result for one member is stored here and used by the reaper instead of the
// pool's ReconnectTimeout.  0 restores the default.
extern "C" int gsim_member_reconnect_timeout_set(gsim_pool* p, uint32_t id, uint64_t timeout_ns) {
  if (!p) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, nullptr, 0, [&]() -> int {
  if (id >= p->g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  uint32_t ticks = timeout_ns ? clamp_ticks(timeout_ns, p->tick_ns) : 0u;
  if (timeout_ns && ticks == 0u) ticks = 1u;
  if (!poke(p, p->d.reap_after, id, ticks)) return fail(p, GSIM_ERR_CUDA, "poke");
  if (ticks && (p->g.reap_min_override == 0u || ticks < p->g.reap_min_override)) {
    p->g.reap_min_override = ticks;
    p->g_dirty = true;
  }
  return GSIM_OK;
  });
}

// (*Serf).GetCoordinate / GetCachedCoordinate(name) — agent/router/router.go:62-67: the member's
// current network coordinate (vec[8], error, adjustment, height; seconds).
extern "C" int gsim_coordinate_get(gsim_pool* p, uint32_t id, double out[11]) {
  if (!p || !out) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  GS_CONTROLLER_ONLY(p);
  if (!p->d.coord) return fail(p, GSIM_ERR_STATE, "the pool was created without GSIM_FLAG_COORDINATES");
  if (id >= p->g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  const size_t cap = p->g.cap;
  uint32_t ta, tb;
  if (!peek(p, p->d.ctag, id, &ta) || !peek(p, p->d.ctag, cap + id, &tb)) return fail(p, GSIM_ERR_CUDA, "peek");
  const size_t slot = tb > ta ? 1 : 0;
  for (size_t x = 0; x < GS_COORD_WORDS; ++x)
    if (!peek(p, p->d.coord, (slot * GS_COORD_WORDS + x) * cap + id, &out[x])) return fail(p, GSIM_ERR_CUDA, "peek");
  return GSIM_OK;
}

// Turn event logging for one member on or off after creation (gsim_member_desc.flags does it at
// creation): the EventCh of that agent, polled through gsim_poll_events.
extern "C" int gsim_member_watch(gsim_pool* p, uint32_t id, int on) {
  if (!p) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, nullptr, 0, [&]() -> int {
  if (id >= p->g.n) return fail(p, GSIM_ERR_NOT_FOUND, "unknown member");
  uint32_t m;
  if (!peek(p, p->d.meta, id, &m)) return fail(p, GSIM_ERR_CUDA, "peek");
  m = on ? (m | GS_META_WATCHED) : (m & ~GS_META_WATCHED);
  if (!poke(p, p->d.meta, id, m)) return fail(p, GSIM_ERR_CUDA, "poke");
  return GSIM_OK;
  });
}

// WAN latency pools (BASELINE config 5, SURVEY 8d C5): n_dcs synthetic datacenters, member i
// lives in datacenter (i / 128) % n_dcs; a packet from datacenter a to b takes lat[a*n_dcs+b]
// ticks (>= 1; 1 is the latency every packet has on a pool without a matrix).
extern "C" int gsim_latency_set(gsim_pool* p, uint32_t n_dcs, const uint8_t* lat_ticks) {
  if (!p || n_dcs > GS_MAX_DCS || (n_dcs && !lat_ticks)) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, nullptr, 0, [&]() -> int {
  GsGlobals& g = p->g;
  for (uint32_t x = 0; x < n_dcs * n_dcs; ++x)
    if (lat_ticks[x] < 1u || lat_ticks[x] > g.ring_mask)
      return fail(p, GSIM_ERR_INVALID, "latency must be in [1, mailbox_depth - 1] ticks");
  memset(g.lat, 0, sizeof(g.lat));
  for (uint32_t a = 0; a < n_dcs; ++a)
    for (uint32_t b = 0; b < n_dcs; ++b) g.lat[a * GS_MAX_DCS + b] = (uint8_t)(lat_ticks[a * n_dcs + b] - 1u);
  g.n_dcs = n_dcs;
  p->g_dirty = true;
  mark_dirty(p);  // what a probe round trip costs has changed
  return GSIM_OK;
  });
}

// ---- time -----------------------------------------------------------------------
static int apply_sched(gsim_pool* p) {
  bool any = false;
  for (size_t x = 0; x < p->sched.size();) {
    if (p->sched[x].tick <= p->now) {
      if (p->sched[x].action == 1u) {
        uint32_t k;
        if (!peek(p, p->d.key[p->now & 1u], p->sched[x].id, &k)) return GSIM_ERR_CUDA;
        if (gs_key_truth(k) == GS_TRUTH_UP) {
          int rc = set_truth(p, p->sched[x].id, GS_TRUTH_GONE);
          if (rc) return rc;
          any = true;
        }
      }
      p->sched.erase(p->sched.begin() + x);
    } else {
      ++x;
    }
  }
  if (any) return refresh_after_truth_change(p);
  return GSIM_OK;
}

// Advance `ticks` ticks.  On a sharded pool every rank runs this together: the host-side parts
// (scheduled shutdowns, globals upload, rumor retirement) are controller calls, the tick kernels
// run on every rank with a device barrier after each tick.
// [U] serf.handleReap: every ReapInterval, erase members that have been Failed for longer than
// ReconnectTimeout or Left for longer than TombstoneTimeout (SURVEY 8a row a17).  The reaper's
// ticker fires at ticks that are multiples of ReapInterval; with Consul's production values
// (72 h / 24 h, agent/consul/config.go:622-623) nothing can be old enough within any simulated
// horizon and no pass is ever scheduled — only test timings (server_test.go:675-677) reach it.
struct ReapPlan {
  uint32_t every, reconnect, tombstone;
};
static uint32_t clamp_ticks(uint64_t ns, uint64_t tick) {
  const uint64_t t = (ns + tick - 1) / tick;
  return t > 0xFFFFFFF0ull ? 0xFFFFFFF0u : (uint32_t)t;
}
static ReapPlan reap_plan(const gsim_pool* p) {
  ReapPlan r;
  r.every = p->cfg.reap_interval_ns ? clamp_ticks(p->cfg.reap_interval_ns, p->tick_ns) : 0u;
  r.reconnect = clamp_ticks(p->cfg.reconnect_timeout_ns, p->tick_ns);
  r.tombstone = clamp_ticks(p->cfg.tombstone_timeout_ns, p->tick_ns);
  return r;
}
// first tick > now at which a reap pass can possibly find something, or GS_NEVER
static uint32_t next_reap_tick(const gsim_pool* p, uint32_t now) {
  const ReapPlan r = reap_plan(p);
  if (!r.every) return GS_NEVER;
  uint32_t youngest = r.reconnect < r.tombstone ? r.reconnect : r.tombstone;
  if (p->g.reap_min_override && p->g.reap_min_override < youngest) youngest = p->g.reap_min_override;
  uint64_t t = (uint64_t)(now / r.every + 1u) * r.every;
  if (t <= youngest) t = ((uint64_t)youngest / r.every + 1u) * r.every;  // nobody is that old before
  return t >= GS_NEVER ? GS_NEVER : (uint32_t)t;
}
static int reap_pass(gsim_pool* p) {
  const ReapPlan r = reap_plan(p);
  if (!r.every || p->now == 0 || p->now % r.every != 0) return GSIM_OK;
  uint32_t youngest = r.reconnect < r.tombstone ? r.reconnect : r.tombstone;
  if (p->g.reap_min_override && p->g.reap_min_override < youngest) youngest = p->g.reap_min_override;
  if (p->now <= youngest) return GSIM_OK;
  uint32_t counts[2] = {0, 0};
  if (!upload_globals(p)) return GSIM_ERR_CUDA;
  mark_dirty(p);
  if (!p->be->reap_rows(p->d, p->g_dev, p->g, p->now, r.reconnect, r.tombstone,
                        (p->cfg.flags & GSIM_FLAG_LOG_GLOBAL_EVENTS) != 0, counts))
    return GSIM_ERR_CUDA;
  if (!counts[0]) return GSIM_OK;
  p->n_established -= counts[1];
  return refresh_after_truth_change(p);
}

// ---- quiet-window scheduling (DESIGN.md §4.2) --------------------------------------------------
static bool windows_possible(const gsim_pool* p) {
  static const bool env_off = getenv("GSIM_NO_WINDOWS") != nullptr;
  const GsGlobals& g = p->g;
  // per-tile ticker phases (the window kernel derives a tile's due ticks from its phase), no
  // per-member periodic tickers besides the probe (push-pull), no coordinate exchange on acks
  return !env_off && !(p->cfg.flags & GSIM_FLAG_NO_WINDOWS) && g.phase_gate != 0u && g.pp_interval == 0u &&
         p->d.coord == nullptr && g.P >= 2u && g.T < g.P && g.n != 0u;
}

#define GS_LONG_WINDOW 32u  // ProbeIntervals one launch covers on a healthy quiet pool
#define GS_PRISTINE_WINDOW 256u  // ... and on a pristine one (every probe a prompt ack: gs_pristine_probes)
static bool pristine_windows_on() {
  static const bool off = getenv("GSIM_NO_PRISTINE_WINDOWS") != nullptr;
  return !off;
}
static bool long_windows_on() {
  static const bool off = getenv("GSIM_NO_LONG_WINDOWS") != nullptr;
  return !off;
}

// After single ticks: has the pool been quiet long enough, and how far is the horizon?
static int try_quiet(gsim_pool* p) {
  GsBackend* be = p->be;
  const GsGlobals& g = p->g;
  const uint32_t depth = g.ring_mask + 1u;
  uint32_t* qs = p->d.qstate[p->sharded ? p->rank : 0u];
  if (p->sharded && !be->xbar_host(p->xb)) return GSIM_ERR_CUDA;  // every rank's last tick has published
  uint32_t la = 0;
  if (!be->d2h(&la, qs + GS_Q_LAST_ACTIVE, 4)) return GSIM_ERR_CUDA;
  // ... and nobody runs on (and writes this rank's copy from its next tick) before everybody has read
  if (p->sharded && !be->xbar_host(p->xb)) return GSIM_ERR_CUDA;
  if (p->dirty_tick + 1u > la) la = p->dirty_tick + 1u;  // a host write at tick T counts like mail at T
  // every arrival slot has been scanned empty once and nobody posted meanwhile: `depth` quiet ticks
  if (p->now < la + depth) {
    // Still busy.  Looking again after every tick would put a host round trip (on a sharded pool: two
    // barriers) behind each tick of a cascade: back off 1, 2, 4, 8 ticks.  Finding the quiet a few ticks
    // late only means those ticks ran as single launches.
    const uint32_t wait = 1u << (p->quiet_fails < 3u ? p->quiet_fails : 3u);
    if (p->quiet_fails < 3u) p->quiet_fails++;
    p->retry_at = la + depth > p->now + wait ? la + depth : p->now + wait;
    return GSIM_OK;
  }
  p->quiet_fails = 0;
  const uint32_t never = GS_NEVER;
  if (!be->h2d(qs + GS_Q_HORIZON, &never, 4)) return GSIM_ERR_CUDA;
  if (p->sharded && !be->xbar_host(p->xb)) return GSIM_ERR_CUDA;
  uint32_t first = 0, count = g.n;
  if (p->sharded) {
    first = p->rank * (uint32_t)p->rows_per_rank < g.n ? p->rank * (uint32_t)p->rows_per_rank : g.n;
    count = first + (uint32_t)p->rows_per_rank < g.n ? (uint32_t)p->rows_per_rank : g.n - first;
  }
  if (!be->quiet_scan(p->d, p->g_dev, g, p->now, first, count)) return GSIM_ERR_CUDA;
  if (p->sharded && !be->xbar_host(p->xb)) return GSIM_ERR_CUDA;
  p->sched_counts[3]++;
  uint32_t hz = 0;
  if (!be->d2h(&hz, qs + GS_Q_HORIZON, 4)) return GSIM_ERR_CUDA;
  if (p->sharded && !be->xbar_host(p->xb)) return GSIM_ERR_CUDA;  // (same: read before anybody moves on)
  if (hz >= p->now + g.P / 2u + 1u) {
    p->quiet = true;
    // No probe in flight, and can one fail at all?  Not if every member the cluster lists as alive or
    // suspect is actually running, no packet is lost and no link is slower than ProbeTimeout: then the
    // horizon cannot move and one launch may run many ProbeIntervals (the controller counts, every
    // rank adopts the answer).
    uint32_t ok_long = 0;
    bool links_ok = true;  // every round trip of the latency matrix fits ProbeTimeout
    for (uint32_t a = 0; a < g.n_dcs && links_ok; ++a)
      for (uint32_t b = 0; b < g.n_dcs; ++b)
        if ((uint32_t)g.lat[a * GS_MAX_DCS + b] + g.lat[b * GS_MAX_DCS + a] > g.T) links_ok = false;
    if (hz == GS_NEVER && g.loss_thr == 0u && links_ok) {
      counts_invalidate(p);  // (ticks have run since the last count)
      int rc = collective_recount(p);
      if (rc) return rc;
      rc = controller_call(p, &ok_long, sizeof(ok_long), [&]() -> int {
        if (!do_recount(p)) return GSIM_ERR_CUDA;
        ok_long = p->rc.unreachable_live == 0u ? 1u : 0u;
        // everybody running, listed alive by everybody, folded into the established set
        // (members still pending are the subjects of tracked alive rumors: the closed form stops in front
        // of their ring entries as it does in front of a member's own)
        uint32_t spec[GS_MAX_SPECIAL];
        const uint32_t n_spec = gs_special_members(g, spec);
        if (ok_long && p->rc.truth_cnt[GS_TRUTH_UP] == g.n && p->rc.rank_cnt[GS_RANK_ALIVE] == g.n &&
            n_spec <= GS_MAX_SPECIAL && p->rc.pending <= n_spec && p->rc.isolated_up == 0u && pristine_windows_on())
          ok_long |= 2u;
        return GSIM_OK;
      });
      if (rc) return rc;
    }
    p->healthy = (ok_long & 1u) != 0u;
    p->pristine = (ok_long & 2u) != 0u;
  } else {  // a probe deadline is upon us: single ticks until it has passed, then look again
    p->retry_at = (hz > p->now ? hz : p->now) + depth + 1u;
  }
  return GSIM_OK;
}

// `chunk` ticks, as quiet windows where the pool allows it and as single ticks where it does not.
static int advance_ticks(gsim_pool* p, uint32_t chunk, bool use_graph) {
  GsBackend* be = p->be;
  const GsXbar* xb = p->sharded ? &p->xb : nullptr;
  uint32_t left = chunk;
  const bool can_window = windows_possible(p);
  while (left) {
    if (can_window && p->quiet) {
      uint32_t done = 0;
      uint64_t nl = 0;
      double wms = 0;
      // ticks per launch: one ProbeInterval; up to GS_LONG_WINDOW of them on a healthy pool
      const bool lng = p->healthy && long_windows_on();
      const bool prist = lng && p->pristine;  // (the closed form costs the same for any number of probes)
      const uint32_t per_launch = prist ? p->g.P * GS_PRISTINE_WINDOW : lng ? p->g.P * GS_LONG_WINDOW : p->g.P;
      if (!be->run_windows(p->d, p->g_dev, p->g, p->now, left, per_launch, use_graph, &wms, &nl, &done, xb, prist))
        return GSIM_ERR_CUDA;
      p->last_ms += wms;
      p->sched_counts[4] += (uint64_t)(wms * 1e6);
      p->last_launches += nl;
      p->sched_counts[0] += nl;
      p->sched_counts[1] += done;
      if (prist) {
        p->sched_counts[6] += nl;
        p->sched_counts[7] += done;
      }
      p->now += done;
      p->node_ticks += (uint64_t)done * p->g.n;
      left -= done;
      if (left) {  // the chain stopped at the horizon: single ticks from here
        p->quiet = false;
        p->healthy = false;
        p->pristine = false;
        p->retry_at = p->now + 1u;
      }
      continue;
    }
    uint32_t c = left;
    if (can_window && c > 16u) c = 16u;  // look for quietness every few ticks
    if (can_window && p->retry_at > p->now && p->retry_at - p->now < c) c = p->retry_at - p->now;
    double tms = 0;
    if (!be->run_ticks(p->d, p->g_dev, p->g, p->now, c, use_graph, &tms, &p->last_launches, xb))
      return GSIM_ERR_CUDA;
    p->last_ms += tms;
    p->sched_counts[5] += (uint64_t)(tms * 1e6);
    p->sched_counts[2] += c;
    p->now += c;
    p->node_ticks += (uint64_t)c * p->g.n;
    left -= c;
    if (can_window && left && p->now >= p->retry_at) {
      int rc = try_quiet(p);
      if (rc) return rc;
    }
  }
  return GSIM_OK;
}

extern "C" int gsim_sched_counts(gsim_pool* p, uint64_t out[8]) {
  if (!p || !out) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  memcpy(out, p->sched_counts, sizeof(p->sched_counts));
  return GSIM_OK;
}

static int step_locked(gsim_pool* p, uint32_t ticks) {
  if (!p->ready) return GSIM_ERR_STATE;
  p->last_ms = 0;
  p->last_launches = 0;
  uint32_t left = ticks;
  const bool use_graph = !(p->cfg.flags & GSIM_FLAG_NO_GRAPH);
  while (left) {
    int rc = controller_call(p, nullptr, 0, [&]() -> int {
      int r = apply_sched(p);
      if (r) return r;
      r = reap_pass(p);
      if (r) return r;
      return upload_globals(p) ? GSIM_OK : GSIM_ERR_CUDA;
    });
    if (rc) return rc;
    uint32_t chunk = left;
    for (const Sched& s : p->sched)
      if (s.tick > p->now && s.tick - p->now < chunk) chunk = s.tick - p->now;
    const uint32_t reap_at = next_reap_tick(p, p->now);
    if (reap_at != GS_NEVER && reap_at - p->now < chunk) chunk = reap_at - p->now;
    rc = advance_ticks(p, chunk, use_graph);
    if (rc) return rc;
    left -= chunk;
    counts_invalidate(p);
  }
  // (the mask is the same on every rank: the loop's last controller call published it)
  bool cand = false;
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r)
    if (((p->g.active_mask >> r) & 1u) && p->g.rumors[r].kind != GSIM_RUMOR_USER_EVENT) cand = true;
  if (cand) {
    int rc = collective_recount(p);
    if (rc) return rc;
  }
  int rc = controller_call(p, nullptr, 0, [&]() -> int {
    int r = apply_sched(p);
    if (r) return r;
    p->defer_and = true;
    r = auto_retire(p);
    p->defer_and = false;
    return r;
  });
  if (rc) return rc;
  return apply_pending_and(p);
}

extern "C" int gsim_step(gsim_pool* p, uint32_t ticks) {
  if (!p) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  int rc = step_locked(p, ticks);
  return rc ? fail(p, rc, "step") : GSIM_OK;
}

extern "C" uint32_t gsim_now(gsim_pool* p) { return p ? p->now : 0; }

extern "C" int gsim_run_until(gsim_pool* p, int predicate, uint32_t arg, uint32_t max_ticks,
                              uint32_t check_every, uint32_t* tick_out) {
  if (!p || !check_every) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  if (tick_out) *tick_out = GS_EMPTY32;
  uint32_t done = 0;
  double ms = 0;
  uint64_t launches = 0;
  for (;;) {
    uint32_t result = GS_EMPTY32;
    if (predicate == GSIM_PRED_RUMOR_CONVERGED) {
      if (arg >= GS_MAX_RUMORS) return fail(p, GSIM_ERR_INVALID, "bad slot");
      if (!peek(p, p->d.conv_tick, arg, &result)) return fail(p, GSIM_ERR_CUDA, "peek");
    } else if (predicate == GSIM_PRED_ALL_RUMORS_CONVERGED) {
      uint32_t ct[32];
      if (!p->be->d2h(ct, p->d.conv_tick, sizeof(ct))) return fail(p, GSIM_ERR_CUDA, "d2h");
      uint32_t mx = 0;
      bool all = true;
      for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r)
        if ((p->g.active_mask >> r) & 1u) {
          if (ct[r] == GS_EMPTY32) all = false;
          else if (ct[r] > mx) mx = ct[r];
        }
      if (all) result = mx;
    } else if (predicate == GSIM_PRED_CRASHED_ALL_DEAD) {
      if (!peek(p, p->d.crashed_dead_tick, 0, &result)) return fail(p, GSIM_ERR_CUDA, "peek");
    } else {
      return fail(p, GSIM_ERR_INVALID, "unknown predicate");
    }
    if (result != GS_EMPTY32) {
      if (tick_out) *tick_out = result;
      break;
    }
    if (done >= max_ticks) break;
    uint32_t chunk = max_ticks - done < check_every ? max_ticks - done : check_every;
    int rc = step_locked(p, chunk);
    if (rc) return fail(p, rc, "step");
    ms += p->last_ms;
    launches += p->last_launches;
    done += chunk;
  }
  p->last_ms = ms;
  p->last_launches = launches;
  return GSIM_OK;
}

// ---- observation ------------------------------------------------------------------
static bool host_knows(const GsGlobals& g, uint32_t i, uint32_t c, uint32_t kc, uint32_t heard_i,
                       uint32_t meta_i) {
  if (c == i) return true;
  if (!gs_key_pending(kc)) return !(meta_i & GS_META_ISOLATED);
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r)
    if (((g.active_mask >> r) & 1u) && g.rumors[r].kind == GSIM_RUMOR_ALIVE && g.rumors[r].subject == c)
      return (heard_i >> r) & 1u;
  return false;
}

// Pinned staging for bulk reads (Members() pulls one key per member): grown on demand, freed with the pool.
static uint32_t* host_stage(gsim_pool* p, size_t words) {
  if (words > p->stage_words) {
    if (p->stage) p->be->host_free(p->stage);
    p->stage_words = 0;
    p->stage = static_cast<uint32_t*>(p->be->host_alloc(words * 4u));
    if (p->stage) p->stage_words = words;
  }
  return p->stage;
}

static int members_locked(gsim_pool* p, uint32_t observer, gsim_member* out, size_t cap, size_t* n) {
  const GsGlobals& g = p->g;
  if (observer >= g.n) return GSIM_ERR_NOT_FOUND;
  uint32_t* keys = host_stage(p, g.n);
  uint32_t heard, meta;
  if (!keys || !p->be->d2h(keys, p->d.key[p->now & 1u], (size_t)g.n * 4) ||
      !peek(p, p->d.heard, observer, &heard) || !peek(p, p->d.meta, observer, &meta))
    return GSIM_ERR_CUDA;
  // on a CSR peer graph a member's list is itself plus its row
  std::vector<uint8_t> in_row;
  if (g.graph_n) {
    in_row.assign(g.n, 0);
    in_row[observer] = 1;
    for (uint32_t e = p->graph_rp[observer]; e < p->graph_rp[observer + 1]; ++e) in_row[p->graph_col[e]] = 1;
  }
  auto visible = [&](uint32_t c) -> bool {
    const uint32_t kc = keys[c];
    if (gs_key_truth(kc) == GS_TRUTH_NONE) return false;
    if (g.graph_n && !in_row[c]) return false;
    return host_knows(g, observer, c, kc, heard, meta);
  };
  auto emit = [&](uint32_t c, gsim_member& mm) {
    const uint32_t kc = keys[c];
    mm.id = c;
    mm.incarnation = gs_key_inc(kc);
    mm.rank = gs_key_rank(kc);
    // memberlist suspect is still serf alive; dead -> failed; left -> left
    mm.status = mm.rank == GS_RANK_DEAD   ? GSIM_STATUS_FAILED
                : mm.rank == GS_RANK_LEFT ? GSIM_STATUS_LEFT
                                          : GSIM_STATUS_ALIVE;
  };
  // The list is 16 B per member: at a million members the host loop, not the 4 MB copy, is the cost of
  // the call.  Large pools split the id range over a few threads (count, exclusive scan, fill).
  unsigned nt = 1;
  if (g.n >= (1u << 17)) {
    nt = std::thread::hardware_concurrency();
    nt = nt > 8u ? 8u : nt < 1u ? 1u : nt;
    if (const char* e = getenv("GSIM_MEMBERS_THREADS")) nt = (unsigned)atoi(e) ? (unsigned)atoi(e) : 1u;
  }
  if (!out) cap = 0;
  if (nt <= 1) {
    size_t cnt = 0;
    for (uint32_t c = 0; c < g.n; ++c) {
      if (!visible(c)) continue;
      if (cnt < cap) emit(c, out[cnt]);
      ++cnt;
    }
    if (n) *n = cnt;
    return GSIM_OK;
  }
  if (p->workers && p->workers->size() != nt) {
    delete p->workers;
    p->workers = nullptr;
  }
  if (!p->workers) p->workers = new HostWorkers(nt);
  std::vector<size_t> part(nt, 0);
  std::atomic<unsigned> counted{0};
  const uint32_t chunk = (g.n + nt - 1) / nt;
  const std::function<void(unsigned)> work = [&](unsigned w) {
    const uint32_t lo = w * chunk < g.n ? w * chunk : g.n, hi = lo + chunk < g.n ? lo + chunk : g.n;
    size_t mine = 0;
    for (uint32_t c = lo; c < hi; ++c) mine += visible(c) ? 1u : 0u;
    part[w] = mine;
    counted.fetch_add(1, std::memory_order_release);
    while (counted.load(std::memory_order_acquire) < nt) std::this_thread::yield();
    size_t at = 0;
    for (unsigned q = 0; q < w; ++q) at += part[q];
    if (at >= cap) return;
    for (uint32_t c = lo; c < hi && at < cap; ++c)
      if (visible(c)) emit(c, out[at++]);
  };
  p->workers->run(work);
  size_t cnt = 0;
  for (unsigned w = 0; w < nt; ++w) cnt += part[w];
  if (n) *n = cnt;
  return GSIM_OK;
}

extern "C" int gsim_members(gsim_pool* p, uint32_t observer, gsim_member* out, size_t cap, size_t* n) {
  if (!p) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  GS_CONTROLLER_ONLY(p);
  int rc = members_locked(p, observer, out, cap, n);
  return rc ? fail(p, rc, "members") : GSIM_OK;
}

extern "C" int gsim_num_nodes(gsim_pool* p, uint32_t observer, uint32_t* n) {
  if (!p || !n) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, n, sizeof(uint32_t), [&]() -> int {
  size_t cnt = 0;
  int rc = members_locked(p, observer, nullptr, 0, &cnt);
  *n = (uint32_t)cnt;
  return rc ? fail(p, rc, "num_nodes") : GSIM_OK;
  });
}

extern "C" int gsim_poll_events(gsim_pool* p, gsim_event* out, size_t cap, size_t* n) {
  if (!p || !n || (!out && cap)) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  GS_CONTROLLER_ONLY(p);
  uint32_t cur[2];
  if (!p->be->d2h(cur, p->d.evlog_cursor, 8)) return fail(p, GSIM_ERR_CUDA, "d2h");
  uint32_t have = cur[0] < p->g.evlog_cap ? cur[0] : p->g.evlog_cap;
  std::vector<GsEventRec> ev(have);
  if (have && !p->be->d2h(ev.data(), p->d.evlog, (size_t)have * sizeof(GsEventRec)))
    return fail(p, GSIM_ERR_CUDA, "d2h");
  // the device appends in scheduling order; canonical order is (tick, type, subject, observer)
  std::sort(ev.begin(), ev.end(), [](const GsEventRec& a, const GsEventRec& b) {
    if (a.tick != b.tick) return a.tick < b.tick;
    if (a.type != b.type) return a.type < b.type;
    if (a.subject != b.subject) return a.subject < b.subject;
    return a.observer < b.observer;
  });
  size_t take = have < cap ? have : cap;
  for (size_t x = 0; x < take; ++x) {
    out[x].tick = ev[x].tick;
    out[x].type = ev[x].type;
    out[x].subject = ev[x].subject;
    out[x].observer = ev[x].observer;
    out[x].ltime = ev[x].ltime;
    out[x].reserved = 0;
  }
  *n = take;
  // keep what did not fit
  uint32_t rest = have - (uint32_t)take;
  if (rest && !p->be->h2d(p->d.evlog, ev.data() + take, (size_t)rest * sizeof(GsEventRec)))
    return fail(p, GSIM_ERR_CUDA, "h2d");
  p->events_dropped += cur[1];
  uint32_t reset[2] = {rest, 0};
  if (!p->be->h2d(p->d.evlog_cursor, reset, 8)) return fail(p, GSIM_ERR_CUDA, "h2d");
  return GSIM_OK;
}

extern "C" int gsim_rumor_info_get(gsim_pool* p, uint32_t slot, gsim_rumor_info* out) {
  if (!p || !out || slot >= GS_MAX_RUMORS) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  if (int rcc = collective_recount(p)) return fail(p, rcc, "recount");
  return controller_call(p, out, sizeof(gsim_rumor_info), [&]() -> int {
  const GsGlobals& g = p->g;
  if (!((g.active_mask >> slot) & 1u)) return fail(p, GSIM_ERR_NOT_FOUND, "slot is free");
  if (!do_recount(p)) return fail(p, GSIM_ERR_CUDA, "recount");
  const GsRumor& ru = g.rumors[slot];
  out->kind = ru.kind;
  out->subject = ru.subject;
  out->incarnation = ru.inc;
  out->ltime = ru.ltime;
  out->origin = ru.origin;
  out->size_bytes = ru.size;
  out->start_tick = ru.start_tick;
  out->heard_count = p->rc.heard_cnt[slot];
  out->queued_count = p->rc.queued_cnt[slot];
  if (!peek(p, p->d.conv_tick, slot, &out->converged_tick)) return fail(p, GSIM_ERR_CUDA, "peek");
  return GSIM_OK;
  });
}

extern "C" int gsim_rumor_retire(gsim_pool* p, uint32_t slot) {
  if (!p || slot >= GS_MAX_RUMORS) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, nullptr, 0, [&]() -> int {
  if (!((p->g.active_mask >> slot) & 1u)) return fail(p, GSIM_ERR_NOT_FOUND, "slot is free");
  if (p->g.rumors[slot].kind == GSIM_RUMOR_ALIVE) {
    if (!do_recount(p)) return fail(p, GSIM_ERR_CUDA, "recount");
    if (p->rc.heard_cnt[slot] != p->g.up_count || p->rc.isolated_up != 0)
      return fail(p, GSIM_ERR_STATE, "alive rumor has not reached every running member");
  }
  int rc = retire_slot(p, slot);
  return rc ? fail(p, rc, "retire") : GSIM_OK;
  });
}

extern "C" int gsim_user_event_get(gsim_pool* p, uint32_t slot, void* name, size_t name_cap,
                                   size_t* name_len, void* payload, size_t payload_cap,
                                   size_t* payload_len) {
  if (!p || slot >= GS_MAX_RUMORS) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  GS_CONTROLLER_ONLY(p);
  if (!((p->g.active_mask >> slot) & 1u) || p->g.rumors[slot].kind != GSIM_RUMOR_USER_EVENT)
    return fail(p, GSIM_ERR_NOT_FOUND, "not a user event slot");
  const RumorHost& rh = p->rh[slot];
  if (name_len) *name_len = rh.name.size();
  if (payload_len) *payload_len = rh.payload.size();
  if (name && name_cap) memcpy(name, rh.name.data(), std::min(name_cap, rh.name.size()));
  if (payload && payload_cap) memcpy(payload, rh.payload.data(), std::min(payload_cap, rh.payload.size()));
  return GSIM_OK;
}

extern "C" int gsim_stats_get(gsim_pool* p, gsim_stats* out) {
  if (!p || !out) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  if (int rcc = collective_recount(p)) return fail(p, rcc, "recount");
  return controller_call(p, out, sizeof(gsim_stats), [&]() -> int {
  memset(out, 0, sizeof(*out));
  if (!do_recount(p)) return fail(p, GSIM_ERR_CUDA, "recount");
  if (!p->sharded) {
    if (!p->be->d2h(out->counters, p->d.stats, sizeof(out->counters))) return fail(p, GSIM_ERR_CUDA, "d2h");
  } else {
    // message counters are accumulated per rank (no cross-GPU atomics in the tick): sum the pages
    for (uint32_t r = 0; r < p->world; ++r) {
      uint64_t part[GSIM_STAT_COUNT];
      if (!p->be->d2h(part, p->pages + (size_t)r * GS_PAGE_BYTES + GS_PG_STATS, sizeof(part)))
        return fail(p, GSIM_ERR_CUDA, "d2h");
      for (int q = 0; q < GSIM_STAT_COUNT; ++q) out->counters[q] += part[q];
    }
  }
  const GsGlobals& g = p->g;
  out->node_ticks = p->node_ticks;
  out->tick = p->now;
  out->n_members = g.n;
  out->n_up = p->rc.truth_cnt[GS_TRUTH_UP];
  out->n_crashed = p->rc.truth_cnt[GS_TRUTH_CRASHED];
  out->n_gone = p->rc.truth_cnt[GS_TRUTH_GONE];
  out->n_view_alive = p->rc.rank_cnt[GS_RANK_ALIVE];
  out->n_view_suspect = p->rc.rank_cnt[GS_RANK_SUSPECT];
  out->n_view_dead = p->rc.rank_cnt[GS_RANK_DEAD];
  out->n_view_left = p->rc.rank_cnt[GS_RANK_LEFT];
  out->retransmit_limit = g.retransmit_limit;
  out->suspicion_k = g.sus_k;
  for (int q = 0; q < GS_K1MAX; ++q) out->suspicion_ticks[q] = g.sus_ticks[q];
  out->probe_interval_ticks = g.P;
  out->probe_timeout_ticks = g.T;
  out->gossip_interval_ticks = g.GI;
  uint32_t cur[2] = {0, 0};
  p->be->d2h(cur, p->d.evlog_cursor, 8);
  out->events_dropped = p->events_dropped + cur[1];
  return GSIM_OK;
  });
}

extern "C" int gsim_state_hash(gsim_pool* p, uint64_t out[4]) {
  if (!p || !out) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  return controller_call(p, out, 4 * sizeof(uint64_t), [&]() -> int {
  if (!upload_globals(p)) return fail(p, GSIM_ERR_CUDA, "upload");
  if (!p->be->state_hash(p->d, p->g_dev, p->g, p->now, out)) return fail(p, GSIM_ERR_CUDA, "hash");
  // pool-wide scalars
  uint64_t h = gs_mix64(0x243F6A8885A308D3ull, p->now);
  h = gs_mix64(h, p->g.n);
  h = gs_mix64(h, p->g.up_count);
  h = gs_mix64(h, p->g.active_mask);
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r)
    if ((p->g.active_mask >> r) & 1u) {
      const GsRumor& ru = p->g.rumors[r];
      h = gs_mix64(h, ((uint64_t)r << 32) | ru.kind);
      h = gs_mix64(h, ((uint64_t)ru.subject << 32) | ru.ltime);
    }
  uint64_t lanes[4];
  gs_hash_lanes(h, lanes);
  for (int q = 0; q < 4; ++q) out[q] += lanes[q];
  return GSIM_OK;
  });
}

extern "C" int gsim_column_read(gsim_pool* p, int column, void* out, size_t cap_bytes, size_t* n_bytes) {
  if (!p || !out) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  GS_CONTROLLER_ONLY(p);
  const GsDev& d = p->d;
  const size_t cap = p->g.cap;
  const void* src = nullptr;
  size_t bytes = cap * 4;
  switch (column) {
    case GSIM_COL_KEY: src = d.key[p->now & 1u]; break;
    case GSIM_COL_META: src = d.meta; break;
    case GSIM_COL_DUE: src = d.due; break;
    case GSIM_COL_CURSOR: src = d.cursor; break;
    case GSIM_COL_PASS: src = d.pass; break;
    case GSIM_COL_PROBE_TGT: src = d.probe_tgt; break;
    case GSIM_COL_PROBE_INC: src = d.probe_inc; break;
    case GSIM_COL_SUS_START: src = d.sus_start; break;
    case GSIM_COL_SUS_FROM: src = d.sus_from; bytes = cap * 4 * GS_K1MAX; break;
    case GSIM_COL_CHANGE_TICK: src = d.change_tick; break;
    case GSIM_COL_LTIME_MEMBER: src = d.ltime_member; break;
    case GSIM_COL_LTIME_EVENT: src = d.ltime_event; break;
    case GSIM_COL_EVENT_MIN: src = d.event_min; break;
    case GSIM_COL_HEARD: src = d.heard; break;
    case GSIM_COL_QUEUED: src = d.queued; break;
    case GSIM_COL_TX: src = d.tx; bytes = cap * GS_MAX_RUMORS; break;
    case GSIM_COL_INBOX: src = d.inbox[p->now & p->g.ring_mask]; break;
    default: return fail(p, GSIM_ERR_INVALID, "unknown column");
  }
  // the caller sees rows of `capacity` elements; the device stride is padded to whole tiles
  const size_t ucap = p->cfg.capacity;
  const size_t planes = column == GSIM_COL_SUS_FROM ? GS_K1MAX : column == GSIM_COL_TX ? GS_MAX_RUMORS : 1;
  const size_t elem = column == GSIM_COL_TX ? 1 : 4;
  const size_t out_bytes = planes * ucap * elem;
  (void)bytes;
  if (n_bytes) *n_bytes = out_bytes;
  if (cap_bytes < out_bytes) return fail(p, GSIM_ERR_INVALID, "buffer too small");
  if (column == GSIM_COL_TX) {
    // device layout: two rumors per 16-bit element (GS_TX); the caller sees [rumor][capacity] bytes
    std::vector<uint8_t> pair(ucap * 2);
    uint8_t* o = reinterpret_cast<uint8_t*>(out);
    for (size_t q = 0; q < GS_MAX_RUMORS / 2; ++q) {
      if (!p->be->d2h(pair.data(), reinterpret_cast<const uint8_t*>(src) + q * cap * 2, ucap * 2))
        return fail(p, GSIM_ERR_CUDA, "d2h");
      for (size_t i = 0; i < ucap; ++i) {
        o[(2 * q) * ucap + i] = pair[2 * i];
        o[(2 * q + 1) * ucap + i] = pair[2 * i + 1];
      }
    }
    return GSIM_OK;
  }
  for (size_t q = 0; q < planes; ++q)
    if (!p->be->d2h(reinterpret_cast<uint8_t*>(out) + q * ucap * elem,
                    reinterpret_cast<const uint8_t*>(src) + q * cap * elem, ucap * elem))
      return fail(p, GSIM_ERR_CUDA, "d2h");
  if (column == GSIM_COL_META) {
    uint32_t* mm = reinterpret_cast<uint32_t*>(out);
    for (size_t i = 0; i < ucap; ++i) mm[i] &= ~GS_META_DIRTY;  // implementation detail
  }
  if (column == GSIM_COL_INBOX) {
    uint32_t* mm = reinterpret_cast<uint32_t*>(out);
    for (size_t i = 0; i < ucap; ++i) mm[i] &= ~GS_WAKE_BIT;  // implementation detail
  }
  return GSIM_OK;
}

// ---- checkpoint / resume ------------------------------------------------------------
// A snapshot is a header followed by the columns, plane by plane.  Most planes of the cold columns
// hold one repeated 32-bit word (empty accusation slots, untouched retransmit counters, zero
// change ticks ...): such a plane is stored as (tag 1, word) and restored with a device fill
// instead of a host->device copy; everything else is (tag 0, raw bytes).
struct SnapCol {
  void* ptr;
  size_t bytes;      // all planes together
  uint32_t planes;   // equally sized, each a multiple of 4 bytes
  bool may_fill;     // planes may be stored as a repeated word
};
static std::vector<SnapCol> snap_cols(gsim_pool* p) {
  const GsDev& d = p->d;
  const size_t cap = p->g.cap;
  std::vector<SnapCol> v;
  auto add = [&](void* q, size_t b, uint32_t planes = 1, bool may_fill = true) { v.push_back(SnapCol{q, b, planes, may_fill}); };
  add(d.key[0], cap * 4, 1, false); add(d.key[1], cap * 4, 1, false);  // (replicated per rank when sharded)
  for (uint32_t s = 0; s <= p->g.ring_mask; ++s) add(d.inbox[s], cap * 4);
  add(d.due, cap * 4); add(d.meta, cap * 4); add(d.cursor, cap * 4); add(d.pass, cap * 4);
  add(d.probe_tgt, cap * 4); add(d.probe_inc, cap * 4); add(d.sus_start, cap * 4);
  add(d.sus_from, cap * 4 * GS_K1MAX, GS_K1MAX); add(d.acc, cap * 8 * GS_K1MAX * 2, GS_K1MAX * 2); add(d.change_tick, cap * 4);
  add(d.reap_after, cap * 4);
  add(d.ltime_member, cap * 4); add(d.ltime_event, cap * 4); add(d.event_min, cap * 4);
  add(d.heard, cap * 4); add(d.queued, cap * 4); add(d.tx, cap * GS_MAX_RUMORS, GS_MAX_RUMORS / 2);
  if (d.kst) add(d.kst, cap);
  if (d.coord) {
    add(d.coord, cap * 8 * 2 * GS_COORD_WORDS, 2 * GS_COORD_WORDS);
    add(d.ctag, cap * 4 * 2, 2);
    add(d.adj, cap * 8 * GS_ADJ_WINDOW, GS_ADJ_WINDOW);
    add(d.adj_idx, cap * 4);
  }
  if (d.ppreq) {
    add(d.ppreq, cap * 4 * 2 * GS_PPK, 2 * GS_PPK);
    add(d.pp_clk, cap * 4 * 4, 4);
  }
  add(d.stats, GSIM_STAT_COUNT * 8, 1, false); add(d.heard_cnt, 32 * 4, 1, false); add(d.conv_tick, 32 * 4, 1, false);
  add(d.crashed_alive, 4, 1, false); add(d.crashed_dead_tick, 4, 1, false);
  return v;
}
struct SnapHeader {
  uint64_t magic;
  uint32_t version, cap;
  uint32_t now, n_sched;
  uint64_t node_ticks;
  uint32_t n_established;
  uint32_t layout;       // which optional column sets the blob carries (snap_layout)
  uint64_t graph_hash;   // FNV-1a of the CSR peer graph the state was produced on (0: complete graph)
  GsGlobals g;
};
static const uint64_t SNAP_MAGIC = 0x4753494D534E4150ull;  // "GSIMSNAP"
static const uint32_t SNAP_VERSION = 3;

// The optional column sets of a pool, as a bit mask: a blob is only ever parsed by a pool with the
// same set (the planes follow each other without per-plane names).
static uint32_t snap_layout(const gsim_pool* p) {
  uint32_t m = 0;
  if (p->d.coord) m |= 1u;
  if (p->d.ppreq) m |= 2u;
  if (p->d.kst) m |= 4u;
  if (p->sharded) m |= 16u;
  return m;
}
static uint64_t snap_graph_hash(const gsim_pool* p) {
  if (p->g.graph_n == 0u) return 0ull;
  uint64_t h = 0xCBF29CE484222325ull;
  auto mix = [&](const std::vector<uint32_t>& v) {
    for (uint32_t x : v) {
      h ^= x;
      h *= 0x100000001B3ull;
    }
  };
  mix(p->graph_rp);
  mix(p->graph_col);
  return h ? h : 1ull;
}

static size_t snap_size(gsim_pool* p) {
  size_t s = sizeof(SnapHeader) + p->sched.size() * sizeof(Sched);
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r) s += 12 + p->rh[r].name.size() + p->rh[r].payload.size();
  for (const SnapCol& c : snap_cols(p)) s += c.bytes + 4u * c.planes;  // upper bound: every plane raw
  return s;
}

extern "C" int gsim_snapshot_size(gsim_pool* p, size_t* n_bytes) {
  if (!p || !n_bytes) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  GS_CONTROLLER_ONLY(p);
  *n_bytes = snap_size(p);
  return GSIM_OK;
}

extern "C" int gsim_snapshot(gsim_pool* p, void* out, size_t cap_bytes, size_t* n_bytes) {
  if (!p || !out) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  GS_CONTROLLER_ONLY(p);
  size_t need = snap_size(p);
  if (n_bytes) *n_bytes = need;
  if (cap_bytes < need) return fail(p, GSIM_ERR_INVALID, "buffer too small");
  uint8_t* w = reinterpret_cast<uint8_t*>(out);
  uint8_t* const w0 = w;
  SnapHeader h;
  memset(&h, 0, sizeof(h));
  h.magic = SNAP_MAGIC;
  h.version = SNAP_VERSION;
  h.layout = snap_layout(p);
  h.graph_hash = snap_graph_hash(p);
  h.cap = p->g.cap;
  h.now = p->now;
  h.n_sched = (uint32_t)p->sched.size();
  h.node_ticks = p->node_ticks;
  h.n_established = p->n_established;
  h.g = p->g;
  memcpy(w, &h, sizeof(h));
  w += sizeof(h);
  if (!p->sched.empty()) memcpy(w, p->sched.data(), p->sched.size() * sizeof(Sched));
  w += p->sched.size() * sizeof(Sched);
  for (uint32_t r = 0; r < GS_MAX_RUMORS; ++r) {
    uint32_t hdr[3] = {(uint32_t)p->rh[r].name.size(), (uint32_t)p->rh[r].payload.size(),
                       (uint32_t)p->rh[r].coalesce};
    memcpy(w, hdr, 12);
    w += 12;
    memcpy(w, p->rh[r].name.data(), hdr[0]);
    w += hdr[0];
    memcpy(w, p->rh[r].payload.data(), hdr[1]);
    w += hdr[1];
  }
  for (const SnapCol& c : snap_cols(p)) {
    const size_t pb = c.bytes / c.planes;
    for (uint32_t q = 0; q < c.planes; ++q) {
      uint8_t* raw = w + 4;
      if (!p->be->d2h(raw, reinterpret_cast<uint8_t*>(c.ptr) + (size_t)q * pb, pb)) return fail(p, GSIM_ERR_CUDA, "d2h");
      // one repeated word?  (buf[0..n-4) == buf[4..n) iff all 32-bit words are equal)
      const bool uniform = c.may_fill && pb >= 8 && memcmp(raw, raw + 4, pb - 4) == 0;
      const uint32_t tag = uniform ? 1u : 0u;
      memcpy(w, &tag, 4);
      w += 4 + (uniform ? 4 : pb);
    }
  }
  if (n_bytes) *n_bytes = (size_t)(w - w0);  // what was actually written (<= gsim_snapshot_size)
  return GSIM_OK;
}

extern "C" int gsim_restore(gsim_pool* p, const void* blob, size_t n_bytes) {
  if (!p || !blob || n_bytes < sizeof(SnapHeader)) return GSIM_ERR_INVALID;
  std::lock_guard<std::mutex> lk(p->mu);
  const int rc_all = controller_call(p, nullptr, 0, [&]() -> int {
  const uint8_t* r = reinterpret_cast<const uint8_t*>(blob);
  const uint8_t* end = r + n_bytes;
  SnapHeader h;
  memcpy(&h, r, sizeof(h));
  r += sizeof(h);
  if (h.magic != SNAP_MAGIC || h.version != SNAP_VERSION) return fail(p, GSIM_ERR_INVALID, "not a gsim snapshot of this version");
  // The blob is trusted for nothing that selects memory: stride, member count, column set, sharding
  // geometry and peer graph must be this pool's before a single plane is copied.
  if (h.cap != p->g.cap || h.g.cap != p->g.cap || h.g.n > p->cfg.capacity || h.g.n > p->g.cap ||
      h.g.ring_mask != p->g.ring_mask || (h.g.pp_interval != 0u) != (p->g.pp_interval != 0u) ||
      h.layout != snap_layout(p) || h.g.world != p->g.world || h.g.key_stride != p->g.key_stride ||
      h.g.rows_per_rank != p->g.rows_per_rank || h.g.phase_group != p->g.phase_group ||
      h.g.graph_n != p->g.graph_n || h.graph_hash != snap_graph_hash(p) || h.n_established > h.g.n)
    return fail(p, GSIM_ERR_INVALID, "snapshot does not match this pool (capacity, column set, sharding or peer graph)");
  if ((size_t)(end - r) < (size_t)h.n_sched * sizeof(Sched)) return fail(p, GSIM_ERR_INVALID, "truncated");
  p->sched.resize(h.n_sched);
  if (h.n_sched) memcpy(p->sched.data(), r, (size_t)h.n_sched * sizeof(Sched));
  r += (size_t)h.n_sched * sizeof(Sched);
  for (uint32_t x = 0; x < GS_MAX_RUMORS; ++x) {
    if (end - r < 12) return fail(p, GSIM_ERR_INVALID, "truncated");
    uint32_t hdr[3];
    memcpy(hdr, r, 12);
    r += 12;
    if ((size_t)(end - r) < (size_t)hdr[0] + hdr[1]) return fail(p, GSIM_ERR_INVALID, "truncated");
    p->rh[x].name.assign((const char*)r, hdr[0]);
    r += hdr[0];
    p->rh[x].payload.assign((const char*)r, hdr[1]);
    r += hdr[1];
    p->rh[x].coalesce = (int)hdr[2];
  }
  for (const SnapCol& c : snap_cols(p)) {
    if (c.may_fill) {  // plane by plane: a device fill or a copy
      const size_t pb = c.bytes / c.planes;
      for (uint32_t q = 0; q < c.planes; ++q) {
        if (end - r < 8) return fail(p, GSIM_ERR_INVALID, "truncated");
        uint32_t tag, word;
        memcpy(&tag, r, 4);
        memcpy(&word, r + 4, 4);
        uint8_t* dst = reinterpret_cast<uint8_t*>(c.ptr) + (size_t)q * pb;
        if (tag == 1u) {
          if (!p->be->fill32(reinterpret_cast<uint32_t*>(dst), word, pb / 4)) return fail(p, GSIM_ERR_CUDA, "fill");
          r += 8;
        } else if (tag == 0u) {
          if ((size_t)(end - r) < 4 + pb) return fail(p, GSIM_ERR_INVALID, "truncated");
          if (!p->be->h2d_async(dst, r + 4, pb)) return fail(p, GSIM_ERR_CUDA, "h2d");
          r += 4 + pb;
        } else {
          return fail(p, GSIM_ERR_INVALID, "corrupt snapshot");
        }
      }
      continue;
    }
    if ((size_t)(end - r) < 4 + c.bytes) return fail(p, GSIM_ERR_INVALID, "truncated");
    r += 4;  // tag 0 (these columns are always stored raw)
    if (!p->be->h2d_async(c.ptr, r, c.bytes)) return fail(p, GSIM_ERR_CUDA, "h2d");
    if (p->sharded && (c.ptr == p->d.key[0] || c.ptr == p->d.key[1])) {
      // the key column is replicated per rank: restore every replica
      uint32_t* rep0 = c.ptr == p->d.key[0] ? p->d.key_rep[0] : p->d.key_rep[1];
      for (uint32_t q = 0; q < p->world; ++q)
        if (!p->be->h2d_async(rep0 + (size_t)q * p->g.key_stride, r, c.bytes)) return fail(p, GSIM_ERR_CUDA, "h2d");
    }
    if (p->sharded && c.ptr == (void*)p->d.stats) {
      // counters restore into rank 0's page; the other ranks' partial sums restart at zero
      std::vector<uint8_t> zeros(c.bytes, 0);
      for (uint32_t q = 1; q < p->world; ++q)
        if (!p->be->h2d(p->pages + (size_t)q * GS_PAGE_BYTES + GS_PG_STATS, zeros.data(), c.bytes)) return fail(p, GSIM_ERR_CUDA, "h2d");
    }
    r += c.bytes;
  }
  if (!p->be->sync()) return fail(p, GSIM_ERR_CUDA, "sync");  // every plane has left the caller's blob
  {
    // topology fields stay the live pool's (they were checked equal above, except the rank, which is
    // this process's own on a sharded pool)
    const uint32_t world = p->g.world, rank = p->g.rank, stride = p->g.key_stride, rpr = p->g.rows_per_rank;
    p->g = h.g;
    p->g.world = world;
    p->g.rank = rank;
    p->g.key_stride = stride;
    p->g.rows_per_rank = rpr;
  }
  p->now = h.now;
  p->node_ticks = h.node_ticks;
  p->n_established = h.n_established;
  p->g_dirty = true;
  counts_invalidate(p);
  if (!poke(p, p->d.tick_base, 0, p->now) || !reset_tick_flags(p) || !reset_qstate(p)) return fail(p, GSIM_ERR_CUDA, "poke");
  uint32_t zero2[2] = {0, 0};
  if (!p->be->h2d(p->d.evlog_cursor, zero2, 8)) return fail(p, GSIM_ERR_CUDA, "h2d");
  return GSIM_OK;
  });
  p->be->sync();  // whatever happened, no copy out of the caller's blob is still in flight
  return rc_all;
}

// ---- measurement hooks ------------------------------------------------------------
extern "C" int gsim_last_step_timing(gsim_pool* p, double* kernel_ms, uint64_t* launches) {
  if (!p) return GSIM_ERR_INVALID;
  if (kernel_ms) *kernel_ms = p->last_ms;
  if (launches) *launches = p->last_launches;
  return GSIM_OK;
}

extern "C" uint64_t gsim_launch_count(gsim_pool* p) { return p && p->be ? p->be->total_launches() : 0; }

// ---- wire formats (include/gsim.h; encoders in gs_wire.h) ---------------------------------------
static size_t zlen(const char* s) { return s ? strlen(s) : 0; }
extern "C" size_t gsim_wire_alive(void* out, size_t cap, uint32_t incarnation, const char* node, const void* addr,
                                  size_t addr_len, uint16_t port, const void* meta, size_t meta_len, const uint8_t vsn[6]) {
  static const uint8_t vsn0[6] = {0, 0, 0, 0, 0, 0};
  return gsw::alive(out, cap, incarnation, node, zlen(node), addr, addr_len, port, meta, meta_len, vsn ? vsn : vsn0);
}
extern "C" size_t gsim_wire_suspect(void* out, size_t cap, uint32_t incarnation, const char* node, const char* from) {
  return gsw::suspect_or_dead(out, cap, false, incarnation, node, zlen(node), from, zlen(from));
}
extern "C" size_t gsim_wire_dead(void* out, size_t cap, uint32_t incarnation, const char* node, const char* from) {
  return gsw::suspect_or_dead(out, cap, true, incarnation, node, zlen(node), from, zlen(from));
}
extern "C" size_t gsim_wire_join_intent(void* out, size_t cap, uint64_t ltime, const char* node) {
  return gsw::serf_intent(out, cap, false, ltime, node, zlen(node), false, false);
}
extern "C" size_t gsim_wire_leave_intent(void* out, size_t cap, uint64_t ltime, const char* node, int prune) {
  return gsw::serf_intent(out, cap, true, ltime, node, zlen(node), prune != 0, false);
}
extern "C" size_t gsim_wire_user_event(void* out, size_t cap, uint64_t ltime, const void* name, size_t name_len,
                                       const void* payload, size_t payload_len, int coalesce) {
  return gsw::serf_user_event(out, cap, ltime, name, name_len, payload, payload_len, coalesce != 0, false);
}
extern "C" size_t gsim_wire_compound(void* out, size_t cap, const void* const* msgs, const size_t* lens, size_t count) {
  if (count > 255 || (count && (!msgs || !lens))) return 0;
  return gsw::compound(out, cap, msgs, lens, count);
}
extern "C" size_t gsim_wire_wanfed_frame(void* out, size_t cap, const void* packet, size_t len) {
  return gsw::wanfed_frame(out, cap, packet, len);
}
extern "C" size_t gsim_wire_consul_user_event(void* out, size_t cap, const char* id, const char* name,
                                              const void* payload, size_t payload_len, const char* node_filter,
                                              const char* service_filter, const char* tag_filter, int version) {
  return gsw::consul_user_event(out, cap, id ? id : "", name ? name : "", payload, payload_len, node_filter,
                                service_filter, tag_filter, version);
}
