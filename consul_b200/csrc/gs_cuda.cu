// gs_cuda.cu — sm_100a kernels and the CUDA backend of libgsim.
//
// Kernels (all HBM/L2-bound integer work; no tensor cores by design — there is no dense
// contraction anywhere on this path):
//   gs_tick_kernel      one launch = one lock-step tick of every virtual member
//                       (SURVEY §7 K1+K2 fused: emit and apply are separated by the
//                       double-buffered mailbox instead of a grid barrier)
//   gs_advance_kernel   bumps the device tick counter at the end of a CUDA-graph chunk
//   gs_init_kernel, gs_crash_kernel, gs_recount_kernel, gs_hash_kernel   control plane
//
// Launch shape of the tick: a persistent grid (SMs x resident CTAs) of 256-thread CTAs; every warp
// owns a contiguous chunk of 128-member tiles, scans their 4-byte mailbox words through a
// shared-memory ring and works only on tiles with mail or a due probe ticker (DESIGN.md §4).
// Ticks are chained inside a CUDA graph of GS_GRAPH_TICKS launches with programmatic dependent
// launch, so the per-launch host cost is off the critical path.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>

#include "gs_aux.h"
#include "gs_backend.h"
#include "gs_vmm.h"

#define GS_BLOCK 256
#define GS_GRAPH_TICKS 64
#define GS_WIN_GRAPH 8   // quiet windows per CUDA graph

namespace {

// COORDS selects the tick-kernel instantiation that carries the network-coordinate update
// (gs_coord.h, ~150 double-precision operations per direct ack).  The default instantiation
// contains none of that code, so pools without GSIM_FLAG_COORDINATES run exactly the kernel the
// round-1 profiles describe.
template <bool COORDS>
struct DevSinkT {
  static constexpr bool kCoords = COORDS;
  uint32_t* s_stat;
  uint32_t* s_heard;
  uint32_t* s_q;  // [0] this CTA saw mail or posted some, [1] min horizon raised by its members
  __device__ __forceinline__ void activity() { s_q[0] = 1u; }
  __device__ __forceinline__ void horizon(uint32_t h) { atomicMin(&s_q[1], h); }
  // Counters are kept per lane (one shared-memory bank each): the 32 members of a group bump the same
  // counter at the same instruction, and 32 atomics on ONE shared word replay 32 times.
  __device__ __forceinline__ void stat(int idx, uint32_t v) { atomicAdd(&s_stat[idx * 32 + (threadIdx.x & 31u)], v); }
  __device__ __forceinline__ void heard(uint32_t r) { atomicAdd(&s_heard[r * 32u + (threadIdx.x & 31u)], 1u); }
  // Pool-wide words (crashed_alive, the event-log cursor, heard_cnt) live in rank 0's page on a
  // sharded pool and are updated by every GPU: system-scope atomics (device scope is not atomic
  // across GPUs).  They are rare — one per event, not per member — so single-GPU pools pay nothing
  // measurable for the wider scope.
  __device__ __forceinline__ void crashed_dead(const GsDev& d, uint32_t t) {
    uint32_t old = atomicSub_system(d.crashed_alive, 1u);
    if (old == 1u) *d.crashed_dead_tick = t;
  }
  __device__ __forceinline__ void log_event(const GsDev& d, const GsGlobals& g, uint32_t t,
                                            uint32_t type, uint32_t subject, uint32_t observer,
                                            uint32_t ltime) {
    uint32_t pos = atomicAdd_system(&d.evlog_cursor[0], 1u);
    if (pos < g.evlog_cap) {
      GsEventRec e;
      e.tick = t;
      e.type = type;
      e.subject = subject;
      e.observer = observer;
      e.ltime = ltime;
      e.reserved = 0u;
      d.evlog[pos] = e;
    } else {
      atomicAdd_system(&d.evlog_cursor[1], 1u);
    }
  }
};
typedef DevSinkT<false> DevSink;

#ifndef GS_MIN_BLOCKS
#define GS_MIN_BLOCKS 4
#endif
#define GS_WARPS (GS_BLOCK / 32)
#define GS_ROUND 4                   // tiles a warp brings in with one bulk copy and scans between two drains of the CTA's queue

// Bulk asynchronous copies (TMA, 1-D): ONE lane moves a whole run of tiles global -> shared with a single
// instruction (cp.async.bulk: SASS UBLKCP) and the data's arrival is counted in bytes on an mbarrier in
// shared memory (expect_tx / complete_tx: SASS SYNCS), which the warp then waits on.  The round-1 scan
// issued a 16-byte cp.async per lane and tile (LDGSTS.128): ~40 warp instructions per idle tile, most of
// them address arithmetic and commit/wait bookkeeping.
__device__ __forceinline__ uint32_t gs_smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void gs_mbar_init(uint64_t* bar, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(gs_smem_addr(bar)), "r"(arrivals) : "memory");
}
__device__ __forceinline__ void gs_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(gs_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gs_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   gs_smem_addr(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(gs_smem_addr(bar))
               : "memory");
}
// true once the phase with this parity has completed; bounded (a byte-count bug must not hang the device:
// the caller raises the pool's VIOLATION word instead)
__device__ __forceinline__ bool gs_mbar_wait(uint64_t* bar, uint32_t parity) {
  for (uint32_t spin = 0; spin < (1u << 24); ++spin) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(gs_smem_addr(bar)), "r"(parity)
        : "memory");
    if (done) return true;
  }
  return false;
}

// ---- sharded pools: the inter-tick barrier lives inside the kernels ---------------------------
// Acquire side: tick t may start once every rank has published "all ticks < t done" in this rank's
// progress array (written by the peers over NVLink with st.release.sys at the end of their
// previous launch).
__device__ __forceinline__ void gs_ranks_wait(const GsDev& d, const GsGlobals& g, uint32_t t) {
  if (threadIdx.x < g.world) {
    uint32_t v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(d.tick_flags[g.rank] + threadIdx.x) : "memory");
    } while ((int32_t)(v - t) < 0);
  }
  __syncthreads();
}
// Release side.  Every thread that delivered something fenced at system scope, so its mailbox
// clears, key updates and remote deliveries are performed; CTAs count in with a device-scope atomic
// and the last one publishes `t_done` to every rank.  The chain (write -> fence.sys -> bar -> atomic
// ... atomic -> fence.sys -> st.release.sys) does not rely on kernel boundaries, which is what
// makes it safe inside a CUDA graph.
__device__ __forceinline__ void gs_ranks_release(const GsDev& d, const GsGlobals& g, uint32_t t_done) {
  __syncthreads();
  if (threadIdx.x == 0u) {
    __threadfence_system();
    const uint32_t arrived = atomicAdd(d.done_ctr, 1u);
    if (arrived == gridDim.x - 1u) {
      __threadfence_system();
      *d.done_ctr = 0u;
      __threadfence_system();
      for (uint32_t r = 0; r < g.world; ++r)
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(d.tick_flags[r] + g.rank), "r"(t_done) : "memory");
    }
  }
}

// Quiet-window scheduling words (GS_Q_*): every rank keeps a copy, writers update all of them.
__device__ __forceinline__ void gs_q_publish(const GsDev& d, const GsGlobals& g, const uint32_t* s_q, uint32_t t) {
  if (s_q[0] != 0u) {
    if (g.world <= 1u) atomicMax(d.qstate[0] + GS_Q_LAST_ACTIVE, t + 1u);
    else for (uint32_t r = 0; r < g.world; ++r) atomicMax_system(d.qstate[r] + GS_Q_LAST_ACTIVE, t + 1u);
  }
  if (s_q[1] != GS_NEVER) {
    if (g.world <= 1u) atomicMin(d.qstate[0] + GS_Q_HORIZON, s_q[1]);
    else for (uint32_t r = 0; r < g.world; ++r) atomicMin_system(d.qstate[r] + GS_Q_HORIZON, s_q[1]);
  }
}

// The generic row step, out of line.  Inlined into the persistent loops it costs every launch its
// registers (80 -> 3 resident CTAs per SM); as a call it costs the members that take it ~30
// instructions on top of several hundred, and the loops around it fit 64 registers (4 CTAs per SM:
// a quarter more warps to hide the L2 round trips, and at 1 M members two tiles per warp, not three).
template <bool COORDS>
__device__ __noinline__ void gs_row_step_call(const GsDev* dp, const GsGlobals* gp, uint32_t i, uint32_t t,
                                              uint32_t inb, uint32_t* s_stat, uint32_t* s_heard, uint32_t* s_q) {
  DevSinkT<COORDS> sink{s_stat, s_heard, s_q};
  gs_row_step(*dp, *gp, i, t, t % gp->GI, inb, sink);
}

// The fast gossip tier (gs_fast_gossip), out of line for the same reason: its own register budget, and a
// few hundred instructions that stay resident in the instruction cache while a cascade tick drains its
// queue.  Returns false, having written nothing, for a member that needs the generic step.
template <bool COORDS>
__device__ __noinline__ bool gs_fast_gossip_call(const GsDev* dp, const GsGlobals* gp, uint32_t i, uint32_t t,
                                                 uint32_t gslot, uint32_t inb, bool due_now, uint32_t* s_stat,
                                                 uint32_t* s_heard, uint32_t* s_q) {
  DevSinkT<COORDS> sink{s_stat, s_heard, s_q};
  return gs_fast_gossip(*dp, *gp, sink, i, t, gslot, inb, due_now);
}

// Persistent, warp-centric tick.  Every warp owns a CONTIGUOUS chunk of tiles (128 members
// each); because ticker phases are dealt round-robin over tiles, every chunk holds the same
// number of probing tiles (+-1) at every tick, so the static split is balanced.
//   Scan: each lane moves the mailbox words of 4 members (16 B; a tile is one 512-byte
// request) into a per-warp shared-memory ring with cp.async, GS_STAGES-1 tiles ahead; tiles
// whose ticker phase can be due at this tick also bring their `due` words.  An idle tile
// costs ~40 warp instructions and 4 bytes per member.
//   Work: a tile with activity is re-read from shared memory one member per lane (coalesced
// column accesses).  The four 32-member groups of a probing tile go through the staged fast
// path together — own columns, target gathers and commits are each issued for all four
// before the first is consumed — so the tile pays two dependent memory latencies, not eight.
// Every other group with activity is queued for the CTA's drain, where members with mail go through
// the fast gossip tier (gs_fast_gossip) and whatever either fast path declines goes to the generic
// gs_row_step.
template <bool COORDS>
__global__ void __launch_bounds__(GS_BLOCK, GS_MIN_BLOCKS)
    gs_tick_kernel(const __grid_constant__ GsDev d, const GsGlobals* __restrict__ gp, uint32_t k_off) {
  __shared__ uint32_t s_stat[GS_NSTAT * 32];  // [counter][lane]
  __shared__ uint32_t s_heard[32 * 32];       // [broadcast slot][lane]
  __shared__ __align__(128) uint32_t s_inb[GS_WARPS][GS_ROUND][GS_TILE];  // a warp's round of mailbox words ...
  __shared__ __align__(128) uint32_t s_due[GS_WARPS][GS_ROUND][GS_TILE];  // ... and `due` words (gated tiles only)
  __shared__ __align__(8) uint64_t s_bar[GS_WARPS];                       // one transaction barrier per warp
  __shared__ uint32_t s_q[2];
  // groups of 32 members that need the generic step, queued by the scanning warps and taken by
  // whichever warp of the CTA is free (two counters each: rounds alternate, see below)
  __shared__ uint32_t s_work[GS_WARPS * GS_ROUND * 4];
  __shared__ uint32_t s_wn[2], s_wtake[2];
  const uint32_t tid = threadIdx.x;
  for (uint32_t x = tid; x < GS_NSTAT * 32u; x += GS_BLOCK) s_stat[x] = 0u;
  for (uint32_t x = tid; x < 32u * 32u; x += GS_BLOCK) s_heard[x] = 0u;
  if (tid == 64u) s_q[0] = 0u;
  if (tid == 65u) s_q[1] = GS_NEVER;
  if (tid >= 66u && tid < 68u) s_wn[tid - 66u] = 0u;
  if (tid >= 68u && tid < 70u) s_wtake[tid - 68u] = 0u;
  if (tid >= 96u && tid < 96u + GS_WARPS) gs_mbar_init(&s_bar[tid - 96u], 1u);  // one arrival per phase: the issuing lane
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  // Programmatic dependent launch: let the next tick's grid start launching now; it blocks in
  // its own griddepcontrol.wait until this grid has completed and flushed.  Everything above
  // this line touches no global memory.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  __syncthreads();
  const GsGlobals& g = *gp;
  const uint32_t t = *d.tick_base + k_off;
  if (g.world > 1u) gs_ranks_wait(d, g, t);
  const uint32_t cur = t & 1u, P = g.P, pslot = t % P, gslot = t % g.GI;
  const uint32_t pslot_t = (t + P - g.T % P) % P;
  const uint32_t lane = tid & 31u, wib = tid >> 5;
  // this rank's tiles: everything on one GPU, a contiguous range of members when sharded
  uint32_t tile_lo = 0, tile_hi = (g.n + GS_TILE - 1u) / GS_TILE;
  if (g.world > 1u) {
    const uint32_t per = g.rows_per_rank / GS_TILE;
    tile_lo = g.rank * per < tile_hi ? g.rank * per : tile_hi;
    tile_hi = tile_lo + per < tile_hi ? tile_lo + per : tile_hi;
  }
  // contiguous runs of tiles, floor or ceil of tiles / warps each: every warp (and so every SM) gets
  // its share — with ceil-sized chunks the last quarter of the grid had nothing to do at 1 M members
  const uint32_t n_warps = gridDim.x * GS_WARPS, n_tiles = tile_hi - tile_lo;
  const uint32_t wid = blockIdx.x * GS_WARPS + wib;
  const uint32_t t_begin = tile_lo + (uint32_t)(((uint64_t)wid * n_tiles) / n_warps);
  const uint32_t t_end = tile_lo + (uint32_t)(((uint64_t)(wid + 1u) * n_tiles) / n_warps);
  const uint32_t* __restrict__ inbox_cur = d.inbox[t & g.ring_mask];  // this tick's arrival slot
  const bool gated = g.phase_gate != 0u;
  const uint32_t shift = g.phase_shift;
  DevSinkT<COORDS> sink{s_stat, s_heard, s_q};

  // Rounds.  A warp scans up to GS_ROUND of its tiles and runs the staged probe fast path inline;
  // every group that needs the generic step goes into the CTA's queue instead.  Then the whole CTA
  // drains the queue, one group per warp at a time: a warp whose tiles were idle helps the warp whose
  // tiles all gossip (ticker phases come in runs of ProbeInterval tiles, so consecutive tiles are
  // busy together and a static split leaves half the warps waiting at the closing barrier).  Results
  // do not depend on who steps a group: everything a member sends is a commutative atomic.
  const uint32_t max_run = (n_tiles + n_warps - 1u) / n_warps, n_rounds = (max_run + GS_ROUND - 1u) / GS_ROUND;
  bool did_work = false;  // this thread touched global state (needs the closing fence when sharded)
  const bool sys_scan = g.world > 1u && (g.flags & 4u);  // GSIM_FLAG_SHARD_SYNC_SCAN (debug): system-scope loads, no bulk copy
  // Bring round r of this warp's tiles into its shared-memory buffers: ONE bulk copy for the mailbox words of
  // the whole round, one per tile that can have a probe action due at this tick (2 of every P phases) for its
  // `due` words; the other tiles' `due` reads as "never".  Issued for round r + 1 as soon as the warp has
  // scanned round r, so the copy flies while the CTA drains its queue.
  auto bring = [&](uint32_t r) {
    const uint32_t b0 = t_begin + r * GS_ROUND < t_end ? t_begin + r * GS_ROUND : t_end;
    const uint32_t b1 = b0 + GS_ROUND < t_end ? b0 + GS_ROUND : t_end;
    const uint32_t tiles = b1 - b0;
    if (!tiles) return;
    uint32_t gate_mask = 0;
    for (uint32_t x = 0; x < tiles; ++x) {
      bool gate = true;
      if (gated) {
        const uint32_t pp = gs_probe_phase(g.rot_p, (b0 + x) >> shift, P);
        gate = pp == pslot || pp == pslot_t;
      }
      gate_mask |= gate ? 1u << x : 0u;
    }
    const size_t off0 = (size_t)b0 * GS_TILE;  // columns are padded to whole tiles
    if (sys_scan) {
      for (uint32_t x = 0; x < tiles; ++x) {
        uint4 v;
        asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(inbox_cur + off0 + x * GS_TILE + lane * 4u) : "memory");
        *reinterpret_cast<uint4*>(&s_inb[wib][x][lane * 4u]) = v;
        const uint4 dv = (gate_mask >> x) & 1u ? *reinterpret_cast<const uint4*>(d.due + off0 + x * GS_TILE + lane * 4u)
                                               : make_uint4(GS_NEVER, GS_NEVER, GS_NEVER, GS_NEVER);
        *reinterpret_cast<uint4*>(&s_due[wib][x][lane * 4u]) = dv;
      }
      __syncwarp();
      return;
    }
    for (uint32_t x = 0; x < tiles; ++x)
      if (!((gate_mask >> x) & 1u))
        *reinterpret_cast<uint4*>(&s_due[wib][x][lane * 4u]) = make_uint4(GS_NEVER, GS_NEVER, GS_NEVER, GS_NEVER);
    __syncwarp();
    if (lane == 0u) {
      // the buffers were last touched through the generic proxy: order that before the bulk writes
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      gs_mbar_expect_tx(&s_bar[wib], (tiles + __popc(gate_mask)) * GS_TILE * 4u);
      gs_bulk_g2s(&s_inb[wib][0][0], inbox_cur + off0, tiles * GS_TILE * 4u, &s_bar[wib]);
      for (uint32_t x = 0; x < tiles; ++x)
        if ((gate_mask >> x) & 1u) gs_bulk_g2s(&s_due[wib][x][0], d.due + off0 + x * GS_TILE, GS_TILE * 4u, &s_bar[wib]);
    }
  };
  bring(0u);
  for (uint32_t round = 0; round < n_rounds; ++round) {
  const uint32_t par = round & 1u;
  const uint32_t r_begin = t_begin + round * GS_ROUND < t_end ? t_begin + round * GS_ROUND : t_end;
  const uint32_t r_end = r_begin + GS_ROUND < t_end ? r_begin + GS_ROUND : t_end;
  if (r_end > r_begin && !sys_scan && !gs_mbar_wait(&s_bar[wib], round & 1u)) {  // (every lane waits: the data is then visible to it)
    if (lane == 0u) atomicExch(d.qstate[g.rank] + GS_Q_VIOLATION, t + 1u);
  }
  for (uint32_t tile = r_begin; tile < r_end; ++tile) {
    const uint32_t st = tile - r_begin;
    const uint4 i4 = *reinterpret_cast<const uint4*>(&s_inb[wib][st][lane * 4u]);
    const uint4 d4 = *reinterpret_cast<const uint4*>(&s_due[wib][st][lane * 4u]);
    bool mine = (i4.x | i4.y | i4.z | i4.w) != 0u || d4.x == t || d4.y == t || d4.z == t || d4.w == t;
    // periodic push-pull (opt-in): the ticker of this tile's phase group (or, with per-member
    // phases, of one of its members) fires at this tick
    bool pp_tile = false;
    if (g.pp_interval != 0u) {
      if (gated) {
        pp_tile = gs_pp_due(g.pp_interval, g.rot_pp, tile >> shift, t);
      } else {
#pragma unroll
        for (uint32_t u = 0; u < 4u; ++u)
          pp_tile |= gs_pp_due(g.pp_interval, g.rot_pp, (tile * GS_TILE + lane * 4u + u) / g.phase_group, t);
      }
      mine |= pp_tile;
    }
    if (__any_sync(0xFFFFFFFFu, mine)) {
      did_work = true;
      __syncwarp();  // other lanes' copies are now visible: re-read one member per lane
      const uint32_t base = tile * GS_TILE + lane;
      bool act[4], cand[4];
      bool any_cand = false;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t w = s_inb[wib][st][u * 32 + lane];
        const bool due_now = s_due[wib][st][u * 32 + lane] == t;
        act[u] = w != 0u || due_now ||
                 (g.pp_interval != 0u && gs_pp_due(g.pp_interval, g.rot_pp, (base + 32u * u) / g.phase_group, t));
        cand[u] = w == 0u && due_now;  // empty mailbox + ticker fired
        any_cand |= cand[u];
      }
      if (__any_sync(0xFFFFFFFFu, any_cand)) {
        GsFastProbe f[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (cand[u]) gs_fast_load(d, cur, base + 32u * u, f[u]);               // A: own columns
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (cand[u]) cand[u] = gs_fast_target(d, g, cur, base + 32u * u, f[u]);  // B: gathers
        uint32_t n_probe = 0, n_ack = 0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          bool acked = false;
          const bool done = cand[u] && gs_fast_finish(d, g, sink, base + 32u * u, t, f[u], &acked);  // C
          if (done) act[u] = false;
          n_probe += __popc(__ballot_sync(0xFFFFFFFFu, done));
          n_ack += __popc(__ballot_sync(0xFFFFFFFFu, done && acked));
        }
        if (lane == 0u && n_probe) {
          atomicAdd(&s_stat[GS_ST_PROBES * 32], n_probe);
          atomicAdd(&s_stat[GS_ST_ACTIVE_ROWS * 32], n_probe);
          if (n_ack) atomicAdd(&s_stat[GS_ST_ACKS * 32], n_ack);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (__any_sync(0xFFFFFFFFu, act[u]) && lane == 0u) s_work[atomicAdd(&s_wn[par], 1u)] = tile * 4u + (uint32_t)u;
      }
    }
  }
  __syncwarp();                              // this warp is done with its round buffers:
  if (round + 1u < n_rounds) bring(round + 1u);  // the next round's copy flies while the CTA drains its queue
  __syncthreads();  // the queue of this round is complete
  if (tid == 0u) s_wn[par ^ 1u] = s_wtake[par ^ 1u] = 0u;  // the next round's counters (nobody uses them now)
  const uint32_t n_work = s_wn[par];
  for (;;) {
    uint32_t idx = 0;
    if (lane == 0u) idx = atomicAdd(&s_wtake[par], 1u);
    idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
    if (idx >= n_work) break;
    did_work = true;
    const uint32_t i = s_work[idx] * 32u + lane;
    // which members of the group: mail, a probe action due (members the fast path finished have moved
    // their `due` on), or the push-pull ticker
    const uint32_t w = __ldcg(inbox_cur + i);
    const bool due_now = __ldcg(d.due + i) == t;
    const bool a = w != 0u || due_now ||
                   (g.pp_interval != 0u && gs_pp_due(g.pp_interval, g.rot_pp, i / g.phase_group, t));
    // members with mail try the fast gossip tier first; whatever it declines takes the generic step
    const bool fast = w != 0u && gs_fast_gossip_call<COORDS>(&d, gp, i, t, gslot, w, due_now, s_stat, s_heard, s_q);
    if (a && !fast) gs_row_step_call<COORDS>(&d, gp, i, t, w, s_stat, s_heard, s_q);
  }
  __syncthreads();  // the queue is drained (and its counters may be reused two rounds from now)
  }  // rounds
  // Sharded pools: mailbox deliveries to other GPUs are fire-and-forget reductions over NVLink;
  // a system-scope fence by the issuing thread is what guarantees they have been performed at
  // the owner before this rank can signal the inter-tick barrier.
  if (g.world > 1u && did_work && !(g.flags & 8u)) __threadfence_system();  // 8: GSIM_FLAG_SHARD_LEAN_FENCE
  __syncthreads();
  // one global atomic per counter per CTA, and only for CTAs that saw activity
  if (tid < GS_NSTAT) {
    uint32_t v = 0;
    for (uint32_t x = 0; x < 32u; ++x) v += s_stat[tid * 32u + ((x + tid) & 31u)];
    if (v) atomicAdd(&d.stats[tid], (unsigned long long)v);
  } else if (tid >= 32u && tid < 32u + GS_MAX_RUMORS) {
    uint32_t r = tid - 32u, c = 0;
    for (uint32_t x = 0; x < 32u; ++x) c += s_heard[r * 32u + ((x + r) & 31u)];
    if (c) {
      uint32_t old = atomicAdd_system(&d.heard_cnt[r], c);  // rank 0's page on a sharded pool
      if (old + c == g.up_count) d.conv_tick[r] = t;  // every UP member has heard rumor r
    }
  }
  if (tid == 0u) gs_q_publish(d, g, s_q, t);  // (after the CTA barrier above: every warp's flags are in)
  if (g.world > 1u) gs_ranks_release(d, g, t + 1u);
}

// ---------------------------------------------------------------------------------------------
// Quiet window: up to ProbeInterval ticks in ONE launch (DESIGN.md §4.2).
//
// On a quiet pool (every mailbox slot empty, nothing time-driven pending but probe tickers) a tick
// changes only the members whose ticker fires, and those write only their own row: the probe is
// pull-evaluated from the target's published key, which nobody changes.  The first tick at which a
// member can touch another one again is the deadline of an unanswered probe, at least
// ProbeInterval after it started; the minimum over all members is the HORIZON word.  Up to the
// horizon the ticks of a tile are independent of every other tile, so a warp runs all the ticks of
// the window for its tiles back to back: no mailbox scan (the words are known to be zero), no
// grid-wide synchronisation, and on a sharded pool one inter-rank barrier per window instead of one
// per tick.  Results are bit-identical to running the ticks one by one — the per-row code is the
// same gs_fast_* / gs_row_step — which tests/test_windows_cpu.py and the GPU parity tests check.
//
// A tile's members are due only at ticks congruent to its ticker phase (probe start, probe
// deadline) or to phase + ProbeTimeout (indirect stage): at most two ticks of a window.
// The generic path of a window for one batch of four groups: one ProbeInterval after the other (rows are
// independent inside a quiet window, so a warp finishes all the ticks of its groups before it looks at
// the next ones), staged probe fast path first, then the generic row step for whatever it declines.
template <bool COORDS>
__device__ __noinline__ void gs_window_generic(const GsDev* dp, const GsGlobals* gp, uint32_t gb, uint32_t g_end,
                                               uint32_t tf00, uint32_t tf01, uint32_t tf02, uint32_t tf03,
                                               uint32_t tx00, uint32_t tx01, uint32_t tx02, uint32_t tx03,
                                               uint32_t t0, uint32_t w1, uint32_t* s_stat, uint32_t* s_heard,
                                               uint32_t* s_q, uint32_t* counts) {
  const GsDev& d = *dp;
  const GsGlobals& g = *gp;
  const GsHot h = gs_hot(g);
  const uint32_t P = h.P, T = h.T, lane = threadIdx.x & 31u;
  const uint32_t tf0[4] = {tf00, tf01, tf02, tf03}, tx0[4] = {tx00, tx01, tx02, tx03};
  const bool fast_ok = h.loss_thr == 0u && h.graph_n == 0u && d.coord == nullptr && h.pp_interval == 0u;
  DevSinkT<COORDS> sink{s_stat, s_heard, s_q};
  uint32_t n_probe = 0, n_ack = 0;
  bool did_work = false;
  (void)did_work;
#pragma unroll 1
    for (uint32_t s0 = t0; s0 < w1; s0 += P) {
    const uint32_t off = s0 - t0;
    uint32_t tf[4], tx[4], due[4];
    bool cand[4], slow[4];
    bool any_slow = false;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (gb + u < g_end) {
        tf[u] = tf0[u] + off;
        tx[u] = tx0[u] + off;
        due[u] = __ldcg(d.due + (gb + u) * 32u + lane);
      } else {
        tf[u] = tx[u] = GS_NEVER;
        due[u] = GS_NEVER - 1u;
      }
      cand[u] = fast_ok && due[u] == tf[u] && tf[u] < w1;
      // anything else that is due inside the window takes the generic step below
      slow[u] = (due[u] == tf[u] && tf[u] < w1 && !fast_ok) || (due[u] == tx[u] && tx[u] < w1);
    }
    // ---- A. own columns of every candidate (independent loads, issued together) ----
    GsFastProbe f[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (cand[u]) gs_fast_load(d, tf[u] & 1u, (gb + u) * 32u + lane, f[u]);
    // ---- B. ring entry -> target, status gathers ----
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (cand[u]) {
        const bool okk = gs_fast_target(d, h, tf[u] & 1u, (gb + u) * 32u + lane, f[u]);
        if (!okk) { cand[u] = false; slow[u] = true; }
      }
    // ---- C. commit ----
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      bool acked = false, done = false;
      if (cand[u]) {
        done = gs_fast_finish(d, h, sink, (gb + u) * 32u + lane, tf[u], f[u], &acked);
        if (!done) slow[u] = true;
        // an unanswered probe reaches its indirect stage at tf + T: inside this window it is stepped below
        else if (!acked && tf[u] + T < w1) slow[u] = true;
      }
      n_probe += done ? 1u : 0u;  // (per lane; summed over the warp at the end)
      n_ack += done && acked ? 1u : 0u;
      any_slow |= slow[u];
    }
    // ---- D. whatever is left: the generic step, tick by tick in ascending order ----
    if (__any_sync(0xFFFFFFFFu, any_slow)) {
      did_work = true;
#pragma unroll 1
      for (int u = 0; u < 4; ++u) {
        const bool sl = u == 0 ? slow[0] : u == 1 ? slow[1] : u == 2 ? slow[2] : slow[3];
        if (!__any_sync(0xFFFFFFFFu, sl)) continue;
        const uint32_t a = u == 0 ? tf[0] : u == 1 ? tf[1] : u == 2 ? tf[2] : tf[3];
        const uint32_t b = u == 0 ? tx[0] : u == 1 ? tx[1] : u == 2 ? tx[2] : tx[3];
        const uint32_t i = (gb + u) * 32u + lane;
#pragma unroll 1
        for (int which = 0; which < 2; ++which) {
          const uint32_t t = which == 0 ? (a < b ? a : b) : (a < b ? b : a);
          if (t >= w1) break;
          // (a member the fast path finished at `a` has moved its `due` on: it is not stepped twice)
          if (sl && __ldcg(d.due + i) == t) gs_row_step_call<COORDS>(&d, gp, i, t, 0u, s_stat, s_heard, s_q);
        }
      }
    }
    }  // ProbeIntervals of this launch
  counts[0] = n_probe;
  counts[1] = n_ack;
}

#ifndef GS_WIN_BLOCKS
#define GS_WIN_BLOCKS 4
#endif
// (resident CTAs per SM the window kernel is compiled for: 4 = 64 registers per thread)
#ifndef GS_WIN_BLOCKS_CLOSED
#define GS_WIN_BLOCKS_CLOSED 4
#endif

// PRISTINE = the instantiation for pools whose probes have a closed form (its own register allocation: it
// contains neither the per-probe loop nor that loop's arrays).
template <bool COORDS, bool PRISTINE>
__global__ void __launch_bounds__(GS_BLOCK, PRISTINE ? GS_WIN_BLOCKS_CLOSED : GS_WIN_BLOCKS)
    gs_window_kernel(const __grid_constant__ GsDev d, const GsGlobals* __restrict__ gp, uint32_t k_off, uint32_t n_ticks,
                     uint32_t mode) {
  __shared__ uint32_t s_stat[GS_NSTAT * 32];  // [counter][lane]
  __shared__ uint32_t s_heard[32 * 32];       // [broadcast slot][lane]
  __shared__ uint32_t s_q[2];
  __shared__ uint32_t s_spec[GS_MAX_SPECIAL + 1];  // [GS_MAX_SPECIAL] = how many
  const uint32_t tid = threadIdx.x;
  for (uint32_t x = tid; x < GS_NSTAT * 32u; x += GS_BLOCK) s_stat[x] = 0u;
  for (uint32_t x = tid; x < 32u * 32u; x += GS_BLOCK) s_heard[x] = 0u;
  if (tid == 64u) s_q[0] = 0u;
  if (tid == 65u) s_q[1] = GS_NEVER;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (tid == 66u) s_spec[GS_MAX_SPECIAL] = gs_special_members(*gp, s_spec);
  __syncthreads();
  const GsGlobals& g = *gp;
  const GsHot h = gs_hot(g);
  // mode bit 1: batches of four groups are dealt to the warps round-robin (neighbouring warps stream
  // neighbouring lines) instead of one contiguous run per warp
  const bool cyclic = (mode & 2u) != 0u;
  const uint32_t world = g.world, rank = g.rank, n_spec = s_spec[GS_MAX_SPECIAL];
  uint32_t* const qs = d.qstate[rank];
  const uint32_t t0 = *d.tick_base + k_off;
  // Where the chain of windows stands and how far it may go.  Both words are stable for the whole
  // launch: siblings only raise WIN_END to this window's own end, and lower HORIZON to ticks
  // >= t0 + ProbeInterval >= t0 + n_ticks.
  const uint32_t reached = __ldcg(qs + GS_Q_WIN_END), horizon = __ldcg(qs + GS_Q_HORIZON);
  if (reached < t0) return;  // an earlier window of this chain stopped at the horizon
  uint32_t w1 = t0 + n_ticks;
  if (horizon < w1) w1 = horizon;  // (GS_NEVER = no probe in flight anywhere)
  if (w1 <= t0) return;            // the horizon is here: the host goes back to single ticks
  if (world > 1u) gs_ranks_wait(d, g, t0);
  const uint32_t P = h.P, T = h.T, lane = tid & 31u, wib = tid >> 5;
  // this rank's groups of 32 members (4 per tile), dealt to the warps in contiguous runs: inside a
  // window rows are independent, so the unit of work need not be the 128-member phase tile
  uint32_t tile_lo = 0, tile_hi = (h.n + GS_TILE - 1u) / GS_TILE;
  if (world > 1u) {
    const uint32_t per = g.rows_per_rank / GS_TILE;
    tile_lo = rank * per < tile_hi ? rank * per : tile_hi;
    tile_hi = tile_lo + per < tile_hi ? tile_lo + per : tile_hi;
  }
  const uint32_t n_warps = gridDim.x * GS_WARPS, grp_lo = tile_lo * 4u, grp_hi = tile_hi * 4u;
  const uint32_t run = (grp_hi - grp_lo + n_warps - 1u) / n_warps;
  const uint32_t wid = blockIdx.x * GS_WARPS + wib;
  const uint32_t g_begin = grp_lo + wid * run < grp_hi ? grp_lo + wid * run : grp_hi;
  const uint32_t g_end = g_begin + run < grp_hi ? g_begin + run : grp_hi;
  const uint32_t shift = g.phase_shift + 2u, t0_mod = t0 % P, rot_p = g.rot_p;
  const uint32_t win_q = (w1 - t0) / P, win_r = (w1 - t0) - win_q * P;
  // the batch is taken through the probe fast path together if the pool allows the fast path at all
  const bool fast_ok = h.loss_thr == 0u && h.graph_n == 0u && d.coord == nullptr && h.pp_interval == 0u;
  DevSinkT<COORDS> sink{s_stat, s_heard, s_q};
  bool did_work = false;
  uint32_t n_probe = 0, n_ack = 0;
  // phase of the first group, then incrementally (one division per warp, not per tile)
  uint32_t pg = g_begin >> shift;              // phase group of the current group
  uint32_t pp = (pg % P + rot_p) % P;          // its probe phase
  const uint32_t g_first = cyclic ? (grp_lo + wid * 4u < grp_hi ? grp_lo + wid * 4u : grp_hi) : g_begin;
  const uint32_t g_step = cyclic ? n_warps * 4u : 4u, g_lim = cyclic ? grp_hi : g_end;
  for (uint32_t gb = g_first; gb < g_lim; gb += g_step) {
    if (cyclic) {  // (a division per batch instead of one per warp)
      pg = gb >> shift;
      pp = (pg % P + rot_p) % P;
    }
    uint32_t tf0[4], tx0[4];
    // ---- 0. the first ticks >= t0 at which each group of the batch can be due ----
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t grp = gb + u;
      if (grp < g_lim) {
        const uint32_t q = grp >> shift;
        if (q != pg) {                                   // groups are consecutive: the next phase group, phase + 1 (mod P)
          pp = pp + 1u == P ? 0u : pp + 1u;
          pg = q;
        }
        uint32_t a = pp + P - t0_mod;                    // first tick >= t0 congruent to the phase ...
        a = a >= P ? a - P : a;
        uint32_t b = a + T;                              // ... and to phase + ProbeTimeout
        b = b >= P ? b - P : b;
        tf0[u] = t0 + a;
        tx0[u] = t0 + b;
      } else {
        tf0[u] = tx0[u] = GS_NEVER;
      }
    }
    // ---- 1. fast-forward.  A member that is up, listed alive, idle and due at its ticker phase keeps its
    // probe state in registers and runs ALL its probes of the launch in a row: ring entry -> target ->
    // the target's status byte -> ack -> awareness - 1, due + ProbeInterval, cursor + 1.  A launch covers
    // one ProbeInterval in general and many when the host knows that no probe can go unanswered; either
    // way the loop stops at the first thing that is not this common case (ring wrap, a target that is
    // not up-alive-established, a slow link), writes the member's state back as it stood BEFORE that
    // probe, and the generic code below carries on from there.  Four groups in lock step: four
    // independent permutations and four gathers in flight per lane.
    // After an obstacle the generic path (2.) takes the ONE ProbeInterval that contains it and the
    // fast-forward resumes behind it: `lo` = the tick up to which this batch has been through 2.
    uint32_t lo = t0;
#pragma unroll 1
    for (;;) {
      uint32_t stuck = GS_NEVER;  // earliest ticker firing still inside the launch after the fast-forward
      if constexpr (PRISTINE) {
        // Closed form (gs_pristine_probes_k): every own column of the batch in ONE round of loads, then per
        // member one inverse ring permutation, no ring entries, no gathers; written back at once.
        uint32_t cnt = 0;
        uint32_t du[4], kk[4], mm[4], cu[4], pa[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t i = (gb + u) * 32u + lane;
          du[u] = GS_NEVER;
          kk[u] = mm[u] = cu[u] = pa[u] = 0u;
          if (gb + u < g_lim) {
            du[u] = __ldcg(d.due + i);
            if (fast_ok) {
              kk[u] = d.key[tf0[u] & 1u][i];  // (parity of the group's first firing; the rare other case reloads)
              mm[u] = d.meta[i];
              cu[u] = d.cursor[i];
              pa[u] = d.pass[i];
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (gb + u >= g_lim) continue;
          const uint32_t i = (gb + u) * 32u + lane;
          uint32_t due = du[u];
          if (fast_ok && due >= lo && due < w1) {
            // on the ticker schedule of its group: the first firing of the launch, or (after an obstacle) a later one
            uint32_t later = 0u;
            bool on_phase = due == tf0[u];
            if (!on_phase && due > tf0[u]) {
              later = (due - tf0[u]) / P;
              on_phase = later * P == due - tf0[u];
            }
            if (on_phase) {
              const uint32_t k0 = ((due ^ tf0[u]) & 1u) ? d.key[due & 1u][i] : kk[u];
              const uint32_t m = mm[u];
              if (gs_key_truth(k0) == GS_TRUTH_UP && gs_key_rank(k0) == GS_RANK_ALIVE && gs_meta_stage(m) == GS_STAGE_IDLE &&
                  !(m & (GS_META_DIRTY | GS_META_ISOLATED))) {
                const GsU4 rk = gs_perm_keys(h.seed_lo, h.seed_hi, i, pa[u]);
                // firings inside the launch: ceil((w1 - tf0) / P) without a division (w1 - t0 = win_q P + win_r)
                const uint32_t kt = win_q + (win_r > tf0[u] - t0 ? 1u : 0u) - later;
                const uint32_t k = gs_pristine_probes_k(h.n, h.perm_bits, rk, i, cu[u], kt, s_spec, n_spec);
                if (k) {
                  const uint32_t aw = gs_meta_aw(m);
                  if (aw) d.meta[i] = gs_meta_set_aw(m, aw > k ? aw - k : 0u);
                  d.cursor[i] = cu[u] + k;
                  due += k * P;
                  d.due[i] = due;
                  cnt += k;
                }
              }
            }
          }
          if (due >= lo && due < w1 && due < stuck) stuck = due;  // still something due inside the launch
        }
        n_probe += cnt;  // per lane; summed over the warp once, at the end
        n_ack += cnt;
      } else
      {
        uint32_t mm[4], cu[4], du[4], m_in[4], cu_in[4], du_in[4], kt[4];
        GsU4 rk[4];
        bool live[4], in_rng[4];
        uint32_t cnt = 0;
        {
          // every own column of the batch in ONE round of loads (a member that turns out not to be due costs
          // 16 bytes it did not need; waiting for `due` first would cost every member a second round trip).
          // The key is read at the parity of the group's first firing and again in the rare other case.
          uint32_t kk[4], pa[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t i = (gb + u) * 32u + lane;
            in_rng[u] = gb + u < g_lim;
            du[u] = GS_NEVER;
            kk[u] = mm[u] = cu[u] = pa[u] = 0u;
            if (in_rng[u]) {
              du[u] = __ldcg(d.due + i);
              if (fast_ok) {
                kk[u] = d.key[tf0[u] & 1u][i];
                mm[u] = d.meta[i];
                cu[u] = d.cursor[i];
                pa[u] = d.pass[i];
              }
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t i = (gb + u) * 32u + lane;
            live[u] = false;
            kt[u] = 0u;
            m_in[u] = mm[u];
            cu_in[u] = cu[u];
            du_in[u] = du[u];
            if (!in_rng[u] || !fast_ok || du[u] < lo || du[u] >= w1) continue;
            // on the ticker schedule of its group: the first firing of the launch, or (after an obstacle) a later one
            uint32_t later = 0u;
            if (du[u] != tf0[u]) {
              if (du[u] < tf0[u]) continue;
              later = (du[u] - tf0[u]) / P;
              if (later * P != du[u] - tf0[u]) continue;
            }
            const uint32_t k = ((du[u] ^ tf0[u]) & 1u) ? d.key[du[u] & 1u][i] : kk[u];
            live[u] = gs_key_truth(k) == GS_TRUTH_UP && gs_key_rank(k) == GS_RANK_ALIVE &&
                      gs_meta_stage(mm[u]) == GS_STAGE_IDLE && !(mm[u] & (GS_META_DIRTY | GS_META_ISOLATED));
            rk[u] = gs_perm_keys(h.seed_lo, h.seed_hi, i, pa[u]);
            // firings inside the launch: ceil((w1 - tf0) / P) without a division (w1 - t0 = win_q P + win_r)
            kt[u] = win_q + (win_r > tf0[u] - t0 ? 1u : 0u) - later;
          }
        }
        for (;;) {
          bool go[4];
          bool any = false;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            go[u] = live[u] && du[u] < w1;
            any |= go[u];
          }
          if (!__any_sync(0xFFFFFFFFu, any)) break;
          uint32_t c[4], kc[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            c[u] = 0u;
            if (go[u]) {
              if (cu[u] >= h.n) {  // ring wrap: re-keyed by the generic step
                live[u] = go[u] = false;
              } else {
                c[u] = gs_perm(cu[u], h.n, h.perm_bits, rk[u]);
                if (c[u] == (gb + u) * 32u + lane) live[u] = go[u] = false;  // own entry: skipped by the generic step
              }
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) kc[u] = go[u] ? gs_peer_key(d, du[u] & 1u, c[u], false) : 0u;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (!go[u]) continue;
            const uint32_t i = (gb + u) * 32u + lane;
            if (gs_key_truth(kc[u]) != GS_TRUTH_UP || gs_key_rank(kc[u]) != GS_RANK_ALIVE || gs_key_pending(kc[u]) ||
                gs_extra(h, i, c[u]) + gs_extra(h, c[u], i) > T) {
              live[u] = false;  // anything but a prompt ack: the generic step decides
              continue;
            }
            const uint32_t aw = gs_meta_aw(mm[u]);
            mm[u] = gs_meta_set_aw(mm[u], aw ? aw - 1u : 0u);
            du[u] += P;
            cu[u] += 1u;
            ++cnt;
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (!in_rng[u]) continue;
          const uint32_t i = (gb + u) * 32u + lane;
          if (cu[u] != cu_in[u]) d.cursor[i] = cu[u];
          if (du[u] != du_in[u]) d.due[i] = du[u];
          if (mm[u] != m_in[u]) d.meta[i] = mm[u];
          if (du[u] >= lo && du[u] < w1 && du[u] < stuck) stuck = du[u];  // still something due inside the launch
        }
        n_probe += cnt;  // per lane; summed over the warp once, at the end
        n_ack += cnt;
      }
      stuck = __reduce_min_sync(0xFFFFFFFFu, stuck);
      if (stuck == GS_NEVER) break;
      // ---- 2. the ProbeInterval of the earliest obstacle takes the generic path (out of line: it is rare,
      // and its staging arrays would cost the loop above its registers)
      {
        const uint32_t off = (stuck - t0) / P * P, s_lo = t0 + off, s_hi = s_lo + P < w1 ? s_lo + P : w1;
        uint32_t add[2] = {0u, 0u};
        gs_window_generic<COORDS>(&d, gp, gb, g_lim, tf0[0] + off, tf0[1] + off, tf0[2] + off, tf0[3] + off, tx0[0] + off,
                                  tx0[1] + off, tx0[2] + off, tx0[3] + off, s_lo, s_hi, s_stat, s_heard, s_q, add);
        n_probe += add[0];
        n_ack += add[1];
        did_work = true;
        lo = s_lo + P;
        if (lo >= w1) break;
      }
    }
  }
  did_work |= n_probe != 0u;
  if (n_probe) {  // one shared-memory counter per lane (DevSinkT::stat)
    atomicAdd(&s_stat[GS_ST_PROBES * 32 + lane], n_probe);
    atomicAdd(&s_stat[GS_ST_ACTIVE_ROWS * 32 + lane], n_probe);
    if (n_ack) atomicAdd(&s_stat[GS_ST_ACKS * 32 + lane], n_ack);
  }
  if (world > 1u && did_work) __threadfence_system();  // horizon words on the peers, before the release
  __syncthreads();
  if (tid < GS_NSTAT) {
    uint32_t v = 0;
    for (uint32_t x = 0; x < 32u; ++x) v += s_stat[tid * 32u + ((x + tid) & 31u)];
    if (v) atomicAdd(&d.stats[tid], (unsigned long long)v);
  }
  if (tid == 0u) {
    // a quiet window never meets mail and never posts: if it did, the scheduling invariant is broken
    // ... and a launch that covers several ProbeIntervals was promised that no probe goes unanswered
    if (s_q[0] != 0u || (n_ticks > P && s_q[1] != GS_NEVER)) atomicExch(qs + GS_Q_VIOLATION, t0 + 1u);
    s_q[0] = 0u;
    gs_q_publish(d, g, s_q, t0);
    atomicMax(qs + GS_Q_WIN_END, w1);
  }
  if (world > 1u) gs_ranks_release(d, g, w1);
}

// Horizon of the pool as it stands (run before the first window after single ticks): the minimum,
// over running members with a probe in flight, of the tick at which it can end in an accusation.
__global__ void __launch_bounds__(GS_BLOCK)
    gs_quiet_scan_kernel(GsDev d, const GsGlobals* __restrict__ gp, uint32_t now, uint32_t first, uint32_t count) {
  __shared__ uint32_t s_min;
  if (threadIdx.x == 0u) s_min = GS_NEVER;
  __syncthreads();
  const GsGlobals& g = *gp;
  uint32_t h = GS_NEVER;
  for (uint32_t x = blockIdx.x * GS_BLOCK + threadIdx.x; x < count; x += gridDim.x * GS_BLOCK) {
    const uint32_t i = first + x;
    if (gs_key_truth(d.key[now & 1u][i]) != GS_TRUTH_UP) continue;
    const uint32_t stage = gs_meta_stage(d.meta[i]);
    if (stage == GS_STAGE_IDLE) continue;
    const uint32_t due = d.due[i];
    const uint32_t e = stage == GS_STAGE_WAIT_T ? due - g.T + g.P : due;  // probe start + P, or the deadline itself
    if (e < h) h = e;
  }
  h = __reduce_min_sync(0xFFFFFFFFu, h);
  if ((threadIdx.x & 31u) == 0u && h != GS_NEVER) atomicMin(&s_min, h);
  __syncthreads();
  if (threadIdx.x == 0u && s_min != GS_NEVER) {
    if (g.world <= 1u) atomicMin(d.qstate[0] + GS_Q_HORIZON, s_min);
    else for (uint32_t r = 0; r < g.world; ++r) atomicMin_system(d.qstate[r] + GS_Q_HORIZON, s_min);
  }
}

// End of a chain of windows: the device clock moves to wherever the chain got.
__global__ void gs_window_advance_kernel(uint32_t* tick_base, const uint32_t* qs) { *tick_base = qs[GS_Q_WIN_END]; }

__global__ void gs_advance_kernel(uint32_t* tick_base, uint32_t k, uint32_t* done_ctr) {
  *tick_base += k;
  if (done_ctr) *done_ctr = 0u;
}

// Cross-GPU barrier (sharded pools).  One warp: lane r publishes this rank's new epoch into
// slot `rank` of rank r's flag array (release, system scope, over NVLink) and then spins on
// slot r of its own array until rank r has published the same epoch.  Everything the preceding
// tick kernel wrote — including remote atomics into peers' mailboxes — happens-before the
// release, so a rank that leaves the barrier sees every delivery addressed to it.
__global__ void gs_xbar_kernel(GsXbar xb) {
  const uint32_t lane = threadIdx.x;
  const uint32_t e = *xb.epoch + 1u;
  __threadfence_system();
  if (lane < xb.world) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(xb.flags[lane] + xb.rank), "r"(e) : "memory");
    uint32_t v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(xb.flags[xb.rank] + lane) : "memory");
    } while ((int32_t)(v - e) < 0);
  }
  __syncwarp();
  __threadfence_system();
  if (lane == 0) *xb.epoch = e;
}

__global__ void __launch_bounds__(GS_BLOCK)
    gs_init_kernel(GsDev d, const GsGlobals* __restrict__ gp, uint32_t first, uint32_t count,
                   uint32_t now) {
  uint32_t x = blockIdx.x * GS_BLOCK + threadIdx.x;
  if (x < count) gs_init_row(d, *gp, first + x, now);
}

__global__ void __launch_bounds__(GS_BLOCK)
    gs_crash_kernel(GsDev d, const GsGlobals* __restrict__ gp, uint32_t thr, uint32_t salt,
                    uint32_t* n_crashed) {
  uint32_t i = blockIdx.x * GS_BLOCK + threadIdx.x;
  bool c = false;
  if (i < gp->n) c = gs_crash_row(d, *gp, i, thr, salt);
  unsigned b = __ballot_sync(0xFFFFFFFFu, c);
  if ((threadIdx.x & 31u) == 0u && b) atomicAdd(n_crashed, (uint32_t)__popc(b));
}

__global__ void __launch_bounds__(GS_BLOCK)
    gs_reap_kernel(GsDev d, const GsGlobals* __restrict__ gp, uint32_t now, uint32_t reconnect_ticks,
                   uint32_t tombstone_ticks, uint32_t log_events, uint32_t* counts) {
  const uint32_t i = blockIdx.x * GS_BLOCK + threadIdx.x;
  uint32_t r = 0;
  if (i < gp->n) r = gs_reap_row(d, *gp, i, now, reconnect_ticks, tombstone_ticks);
  if (r && log_events) {
    DevSink sink{nullptr, nullptr, nullptr};
    sink.log_event(d, *gp, now, GS_EV_MEMBER_REAP, i, GS_EMPTY32, 0u);
  }
  const unsigned b0 = __ballot_sync(0xFFFFFFFFu, (r & 1u) != 0u), b1 = __ballot_sync(0xFFFFFFFFu, (r & 2u) != 0u);
  if ((threadIdx.x & 31u) == 0u) {
    if (b0) atomicAdd(&counts[0], (uint32_t)__popc(b0));
    if (b1) atomicAdd(&counts[1], (uint32_t)__popc(b1));
  }
}

__global__ void __launch_bounds__(GS_BLOCK)
    gs_recount_kernel(GsDev d, const GsGlobals* __restrict__ gp, uint32_t now, uint32_t first, uint32_t count, GsRecount* out) {
  __shared__ GsRecount s;
  uint32_t* sw = reinterpret_cast<uint32_t*>(&s);
  for (uint32_t x = threadIdx.x; x < sizeof(GsRecount) / 4; x += GS_BLOCK) sw[x] = 0u;
  __syncthreads();
  const GsGlobals& g = *gp;
  const uint32_t x = blockIdx.x * GS_BLOCK + threadIdx.x, i = first + x;
  if (x < count && i < g.n) {
    uint32_t k = d.key[now & 1u][i];
    uint32_t truth = gs_key_truth(k), rank = gs_key_rank(k);
    atomicAdd(&s.truth_cnt[truth], 1u);
    if (truth != GS_TRUTH_NONE) atomicAdd(&s.rank_cnt[rank], 1u);
    if (truth == GS_TRUTH_CRASHED && rank < GS_RANK_DEAD) atomicAdd(&s.crashed_alive, 1u);
    if ((truth == GS_TRUTH_CRASHED || truth == GS_TRUTH_GONE) && rank < GS_RANK_DEAD) atomicAdd(&s.unreachable_live, 1u);
    if (truth == GS_TRUTH_UP && (d.meta[i] & GS_META_ISOLATED)) atomicAdd(&s.isolated_up, 1u);
    if (truth != GS_TRUTH_NONE && gs_key_pending(k)) atomicAdd(&s.pending, 1u);
    if (truth == GS_TRUTH_UP && g.active_mask) {
      uint32_t h = d.heard[i] & g.active_mask, q = d.queued[i] & g.active_mask;
      while (h) {
        uint32_t r = __ffs(h) - 1;
        h &= h - 1;
        atomicAdd(&s.heard_cnt[r], 1u);
      }
      while (q) {
        uint32_t r = __ffs(q) - 1;
        q &= q - 1;
        atomicAdd(&s.queued_cnt[r], 1u);
      }
    }
  }
  __syncthreads();
  uint32_t* ow = reinterpret_cast<uint32_t*>(out);
  for (uint32_t x = threadIdx.x; x < sizeof(GsRecount) / 4; x += GS_BLOCK)
    if (sw[x]) atomicAdd(&ow[x], sw[x]);
}

__global__ void __launch_bounds__(GS_BLOCK)
    gs_hash_kernel(GsDev d, const GsGlobals* __restrict__ gp, uint32_t now,
                   unsigned long long* out) {
  __shared__ unsigned long long s[4];
  if (threadIdx.x < 4) s[threadIdx.x] = 0ull;
  __syncthreads();
  uint32_t i = blockIdx.x * GS_BLOCK + threadIdx.x;
  if (i < gp->n) {
    uint64_t h = gs_hash_row(d, *gp, i, now);
    if (h) {
      uint64_t lanes[4];
      gs_hash_lanes(h, lanes);
      for (int q = 0; q < 4; ++q) atomicAdd(&s[q], (unsigned long long)lanes[q]);
    }
  }
  __syncthreads();
  if (threadIdx.x < 4 && s[threadIdx.x]) atomicAdd(&out[threadIdx.x], s[threadIdx.x]);
}

// Tick launches use programmatic stream serialization (PDL) so consecutive ticks overlap
// launch latency and prologue with the previous tick's tail.
static cudaError_t gs_launch_tick(uint32_t blocks, cudaStream_t stream, const GsDev& d,
                                  const GsGlobals* g_dev, uint32_t k, bool pdl) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(blocks);
  cfg.blockDim = dim3(GS_BLOCK);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return d.coord ? cudaLaunchKernelEx(&cfg, gs_tick_kernel<true>, d, g_dev, k)
                 : cudaLaunchKernelEx(&cfg, gs_tick_kernel<false>, d, g_dev, k);
}

static cudaError_t gs_launch_window(uint32_t blocks, cudaStream_t stream, const GsDev& d, const GsGlobals* g_dev,
                                    uint32_t k_off, uint32_t n_ticks, bool pdl, uint32_t mode) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(blocks);
  cfg.blockDim = dim3(GS_BLOCK);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  if (mode & 1u)  // pristine pool: the closed-form instantiation
    return d.coord ? cudaLaunchKernelEx(&cfg, gs_window_kernel<true, true>, d, g_dev, k_off, n_ticks, mode)
                   : cudaLaunchKernelEx(&cfg, gs_window_kernel<false, true>, d, g_dev, k_off, n_ticks, mode);
  return d.coord ? cudaLaunchKernelEx(&cfg, gs_window_kernel<true, false>, d, g_dev, k_off, n_ticks, mode)
                 : cudaLaunchKernelEx(&cfg, gs_window_kernel<false, false>, d, g_dev, k_off, n_ticks, mode);
}

__global__ void gs_row_read_kernel(GsDev d, uint32_t i, uint32_t* out) {
  const uint32_t* col[8] = {d.key[0], d.key[1], d.meta, d.heard, d.queued, d.ltime_member, d.ltime_event, d.event_min};
  if (threadIdx.x < 8u) out[threadIdx.x] = col[threadIdx.x][i];
}

__global__ void __launch_bounds__(GS_BLOCK) gs_fill32_kernel(uint32_t* dst, uint32_t value, size_t count) {
  for (size_t x = (size_t)blockIdx.x * GS_BLOCK + threadIdx.x; x < count; x += (size_t)gridDim.x * GS_BLOCK)
    dst[x] = value;
}

__global__ void __launch_bounds__(GS_BLOCK) gs_and_kernel(GsDev d, uint32_t first, uint32_t count, uint32_t keep) {
  const uint32_t x = blockIdx.x * GS_BLOCK + threadIdx.x, i = first + x;
  if (x >= count) return;
  uint32_t v;
  v = d.heard[i];
  if (v & ~keep) d.heard[i] = v & keep;
  v = d.queued[i];
  if (v & ~keep) d.queued[i] = v & keep;
  for (uint32_t s = 0; s < GS_RING_MAX && d.inbox[s] != nullptr; ++s) {
    v = d.inbox[s][i];
    if (v & ~keep) d.inbox[s][i] = v & keep;
  }
}

class CudaBackend : public GsBackend {
 public:
  explicit CudaBackend(int dev) : dev_(dev) {
    err_[0] = 0;
    cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking);
    cudaEventCreate(&ev0_);
    cudaEventCreate(&ev1_);
    int sms = 148, occ = 4;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gs_tick_kernel<false>, GS_BLOCK, 0) != cudaSuccess || occ < 1)
      occ = 4;
    full_grid_ = (uint32_t)(sms * occ);
    int wocc = GS_WIN_BLOCKS;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&wocc, gs_window_kernel<false, false>, GS_BLOCK, 0) != cudaSuccess || wocc < 1)
      wocc = GS_WIN_BLOCKS;
    win_grid_ = (uint32_t)(sms * wocc);
    scratch_ = nullptr;
    cudaMalloc(&scratch_, 4096);
  }
  ~CudaBackend() override {
    cudaSetDevice(dev_);
    for (auto& kv : graphs_) cudaGraphExecDestroy(kv.second);
    for (auto& kv : wgraphs_) cudaGraphExecDestroy(kv.second);
    if (sharded_) vmm_.destroy();
    if (scratch_) cudaFree(scratch_);
    cudaEventDestroy(ev0_);
    cudaEventDestroy(ev1_);
    cudaStreamDestroy(stream_);
  }
  const char* name() const override { return "cuda-sm_100a"; }
  void* alloc(size_t bytes) override {
    cudaSetDevice(dev_);
    void* p = nullptr;
    if (!ok(cudaMalloc(&p, bytes ? bytes : 4), "cudaMalloc")) return nullptr;
    return p;
  }
  void release(void* p) override {
    cudaSetDevice(dev_);
    if (p && !sharded_) cudaFree(p);
  }
  bool h2d(void* dst, const void* src, size_t bytes) override {
    cudaSetDevice(dev_);
    return ok(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream_), "h2d") &&
           ok(cudaStreamSynchronize(stream_), "h2d sync");
  }
  bool d2h(void* dst, const void* src, size_t bytes) override {
    cudaSetDevice(dev_);
    return ok(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream_), "d2h") &&
           ok(cudaStreamSynchronize(stream_), "d2h sync");
  }
  void* host_alloc(size_t bytes) override {
    void* q = nullptr;
    cudaSetDevice(dev_);
    return cudaHostAlloc(&q, bytes, cudaHostAllocDefault) == cudaSuccess ? q : nullptr;
  }
  void host_free(void* q) override { cudaFreeHost(q); }
  bool h2d_word(void* dst, const void* src, size_t bytes) override {
    if (bytes > 64) return h2d(dst, src, bytes);
    cudaSetDevice(dev_);
    return ok(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream_), "h2d");
  }
  bool h2d_async(void* dst, const void* src, size_t bytes) override {
    cudaSetDevice(dev_);
    return ok(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream_), "h2d");
  }
  bool row_read(const GsDev& d, uint32_t i, uint32_t out[8]) override {
    cudaSetDevice(dev_);
    uint32_t* w = reinterpret_cast<uint32_t*>(scratch_) + 256;  // (the first KB of scratch belongs to the counters)
    gs_row_read_kernel<<<1, 32, 0, stream_>>>(d, i, w);
    ++launches_;
    return ok(cudaGetLastError(), "row read launch") && d2h(out, w, 32);
  }
  bool fill32(uint32_t* dst, uint32_t value, size_t count) override {
    cudaSetDevice(dev_);
    if ((value & 0xFFu) == ((value >> 8) & 0xFFu) && (value & 0xFFFFu) == (value >> 16))
      return ok(cudaMemsetAsync(dst, (int)(value & 0xFFu), count * 4, stream_), "memset");
    return ok(cudaMemsetD32Async_(dst, value, count), "memset32");
  }
  bool fill8(uint8_t* dst, uint8_t value, size_t count) override {
    cudaSetDevice(dev_);
    return ok(cudaMemsetAsync(dst, value, count, stream_), "memset8");
  }
  bool init_rows(const GsDev& d, const GsGlobals* g_dev, const GsGlobals&, uint32_t first,
                 uint32_t count, uint32_t now) override {
    if (!count) return true;
    cudaSetDevice(dev_);
    gs_init_kernel<<<(count + GS_BLOCK - 1) / GS_BLOCK, GS_BLOCK, 0, stream_>>>(d, g_dev, first,
                                                                                count, now);
    ++launches_;
    return ok(cudaGetLastError(), "init launch") && ok(cudaStreamSynchronize(stream_), "init");
  }
  bool run_ticks(const GsDev& d, const GsGlobals* g_dev, const GsGlobals& g, uint32_t t0,
                 uint32_t nticks, bool use_graph, double* kernel_ms, uint64_t* launches,
                 const GsXbar* xbar) override {
    (void)t0;
    if (!nticks || !g.n) {
      if (nticks) {  // no members: just advance time
        gs_advance_kernel<<<1, 1, 0, stream_>>>(d.tick_base, nticks, nullptr);
        ++launches_;
        return ok(cudaGetLastError(), "advance") && ok(cudaStreamSynchronize(stream_), "advance");
      }
      return true;
    }
    cudaSetDevice(dev_);
    // performance variant: keep the status replica (1 byte per member, gathered at random by every
    // prober) resident in L2 — persisting hits for the window, streaming for everything else.
    // Set on the stream before any capture, so graph kernel nodes inherit it.
    if (d.kst != nullptr && !l2_window_set_ && getenv("GSIM_NO_L2_WINDOW") == nullptr) {
      l2_window_set_ = true;
      cudaDeviceProp prop;
      if (cudaGetDeviceProperties(&prop, dev_) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
        size_t bytes = g.cap;
        if (bytes > (size_t)prop.accessPolicyMaxWindowSize) bytes = (size_t)prop.accessPolicyMaxWindowSize;
        size_t carve = bytes < (size_t)prop.persistingL2CacheMaxSize ? bytes : (size_t)prop.persistingL2CacheMaxSize;
        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
        cudaStreamAttrValue v;
        memset(&v, 0, sizeof(v));
        v.accessPolicyWindow.base_ptr = d.kst;
        v.accessPolicyWindow.num_bytes = bytes;
        v.accessPolicyWindow.hitRatio = bytes <= carve ? 1.0f : (float)carve / (float)bytes;
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        cudaStreamSetAttribute(stream_, cudaStreamAttributeAccessPolicyWindow, &v);
        cudaGetLastError();  // best effort: an unsupported attribute must not fail the step
      }
    }
    // persistent launch: one warp per 128-member tile up to a full machine (SMs x resident CTAs)
    uint32_t tiles = (g.n + GS_TILE - 1) / GS_TILE;
    if (g.world > 1 && tiles > g.rows_per_rank / GS_TILE) tiles = g.rows_per_rank / GS_TILE;
    const uint32_t warps_per_block = GS_BLOCK / 32;
    uint32_t blocks = (tiles + warps_per_block - 1) / warps_per_block;
    if (blocks > full_grid_) blocks = full_grid_;
    if (!ok(cudaEventRecord(ev0_, stream_), "event")) return false;
    uint32_t left = nticks;
    if (use_graph && (!xbar || !no_shard_graph_) && left >= GS_GRAPH_TICKS) {
      cudaGraphExec_t ge = graph_for(d, g_dev, blocks, xbar);
      if (!ge) return false;
      while (left >= GS_GRAPH_TICKS) {
        if (!ok(cudaGraphLaunch(ge, stream_), "graph launch")) return false;
        left -= GS_GRAPH_TICKS;
        launches_ += GS_GRAPH_TICKS + 1;
      }
    }
    if (left) {
      for (uint32_t k = 0; k < left; ++k) {
        if (!ok(gs_launch_tick(blocks, stream_, d, g_dev, k, pdl_ && !xbar), "tick launch")) return false;
      }
      gs_advance_kernel<<<1, 1, 0, stream_>>>(d.tick_base, left, nullptr);
      launches_ += left + 1;
      if (!ok(cudaGetLastError(), "tick launch")) return false;
    }
    if (!ok(cudaEventRecord(ev1_, stream_), "event")) return false;
    // the word a kernel raises when one of its internal invariants breaks (a bulk copy that never
    // completed): read back with the synchronisation that happens anyway, so that it fails loudly
    uint32_t violation = 0;
    if (!ok(cudaMemcpyAsync(&violation, d.qstate[g.rank] + GS_Q_VIOLATION, 4, cudaMemcpyDeviceToHost, stream_), "tick d2h"))
      return false;
    if (!ok(cudaStreamSynchronize(stream_), "tick sync")) return false;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ev0_, ev1_);
    if (kernel_ms) *kernel_ms += ms;
    if (launches) *launches += nticks;
    if (violation != 0u) {
      snprintf(err_, sizeof(err_), "tick %u: a bulk copy of the mailbox scan did not complete (kernel invariant broken)", violation - 1u);
      return false;
    }
    return true;
  }
  // Quiet windows (gs_window_kernel): `nticks` ticks as a chain of launches of up to ProbeInterval
  // ticks each.  The chain stops by itself at the horizon; *ticks_done says how far it got.
  bool run_windows(const GsDev& d, const GsGlobals* g_dev, const GsGlobals& g, uint32_t t0, uint32_t nticks,
                   uint32_t per_launch, bool use_graph, double* kernel_ms, uint64_t* launches, uint32_t* ticks_done,
                   const GsXbar* xbar, bool pristine) override {
    cudaSetDevice(dev_);
    *ticks_done = 0;
    if (!nticks || !g.n) return true;
    uint32_t* qs = d.qstate[g.rank];
    uint32_t init[2] = {t0, 0u};  // WIN_END = t0, VIOLATION = 0
    if (!ok(cudaMemcpyAsync(qs + GS_Q_WIN_END, init, 8, cudaMemcpyHostToDevice, stream_), "window init")) return false;
    uint32_t tiles = (g.n + GS_TILE - 1) / GS_TILE;
    if (g.world > 1 && tiles > g.rows_per_rank / GS_TILE) tiles = g.rows_per_rank / GS_TILE;
    uint32_t blocks = (tiles * 4u + GS_WARPS - 1) / GS_WARPS;  // a warp per group of 32 members, up to a full machine
    if (blocks > win_grid_) blocks = win_grid_;
    const uint32_t K = per_launch < g.P ? g.P : per_launch;
    const bool sharded = xbar != nullptr;
    const bool pdl = pdl_ && !sharded;
    if (!ok(cudaEventRecord(ev0_, stream_), "event")) return false;
    uint32_t left = nticks, n_launch = 0;
    if (use_graph && K == g.P && (!sharded || !no_shard_graph_)) {
      while (left >= GS_WIN_GRAPH * K) {
        cudaGraphExec_t ge = window_graph_for(d, g_dev, blocks, K, pdl, g.rank);
        if (!ge) return false;
        if (!ok(cudaGraphLaunch(ge, stream_), "window graph launch")) return false;
        left -= GS_WIN_GRAPH * K;
        n_launch += GS_WIN_GRAPH;
        launches_ += GS_WIN_GRAPH + 1;
      }
    }
    if (left) {
      uint32_t k = 0;
      while (left) {
        const uint32_t c = left < K ? left : K;
        if (!ok(gs_launch_window(blocks, stream_, d, g_dev, k, c, pdl, (pristine ? 1u : 0u) | win_mode_), "window launch"))
          return false;
        k += c;
        left -= c;
        ++n_launch;
        ++launches_;
      }
      gs_window_advance_kernel<<<1, 1, 0, stream_>>>(d.tick_base, qs);
      ++launches_;
      if (!ok(cudaGetLastError(), "window launch")) return false;
    }
    if (!ok(cudaEventRecord(ev1_, stream_), "event")) return false;
    uint32_t back[2] = {0, 0};
    if (!ok(cudaMemcpyAsync(back, qs + GS_Q_WIN_END, 8, cudaMemcpyDeviceToHost, stream_), "window d2h")) return false;
    if (!ok(cudaStreamSynchronize(stream_), "window sync")) return false;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ev0_, ev1_);
    if (kernel_ms) *kernel_ms += ms;
    if (launches) *launches += n_launch;
    if (back[1] != 0u) {
      snprintf(err_, sizeof(err_), "quiet window starting at tick %u met mail or posted some (scheduling invariant broken)", back[1] - 1u);
      return false;
    }
    if (back[0] < t0 || back[0] > t0 + nticks) {
      snprintf(err_, sizeof(err_), "window chain ended at tick %u outside [%u, %u]", back[0], t0, t0 + nticks);
      return false;
    }
    *ticks_done = back[0] - t0;
    return true;
  }
  bool quiet_scan(const GsDev& d, const GsGlobals* g_dev, const GsGlobals& g, uint32_t now, uint32_t first,
                  uint32_t count) override {
    cudaSetDevice(dev_);
    if (!count) return true;
    uint32_t blocks = (count + GS_BLOCK - 1) / GS_BLOCK;
    if (blocks > 148u * 8u) blocks = 148u * 8u;
    gs_quiet_scan_kernel<<<blocks, GS_BLOCK, 0, stream_>>>(d, g_dev, now, first, count);
    ++launches_;
    (void)g;
    return ok(cudaGetLastError(), "quiet scan launch") && ok(cudaStreamSynchronize(stream_), "quiet scan");
  }
  bool crash_fraction(const GsDev& d, const GsGlobals* g_dev, const GsGlobals& g, uint32_t thr,
                      uint32_t salt, uint32_t, uint32_t* n_crashed) override {
    cudaSetDevice(dev_);
    uint32_t* cnt = reinterpret_cast<uint32_t*>(scratch_);
    if (!ok(cudaMemsetAsync(cnt, 0, 4, stream_), "memset")) return false;
    if (g.n) {
      gs_crash_kernel<<<(g.n + GS_BLOCK - 1) / GS_BLOCK, GS_BLOCK, 0, stream_>>>(d, g_dev, thr,
                                                                                 salt, cnt);
      ++launches_;
    }
    return ok(cudaGetLastError(), "crash launch") && d2h(n_crashed, cnt, 4);
  }
  bool reap_rows(const GsDev& d, const GsGlobals* g_dev, const GsGlobals& g, uint32_t now,
                 uint32_t reconnect_ticks, uint32_t tombstone_ticks, bool log_events,
                 uint32_t counts[2]) override {
    cudaSetDevice(dev_);
    uint32_t* cnt = reinterpret_cast<uint32_t*>(scratch_);
    if (!ok(cudaMemsetAsync(cnt, 0, 8, stream_), "memset")) return false;
    if (g.n) {
      gs_reap_kernel<<<(g.n + GS_BLOCK - 1) / GS_BLOCK, GS_BLOCK, 0, stream_>>>(
          d, g_dev, now, reconnect_ticks, tombstone_ticks, log_events ? 1u : 0u, cnt);
      ++launches_;
    }
    return ok(cudaGetLastError(), "reap launch") && d2h(counts, cnt, 8);
  }
  bool recount(const GsDev& d, const GsGlobals* g_dev, const GsGlobals& g, uint32_t now, uint32_t first, uint32_t count,
               GsRecount* out) override {
    cudaSetDevice(dev_);
    GsRecount* dr = reinterpret_cast<GsRecount*>(scratch_);
    if (!ok(cudaMemsetAsync(dr, 0, sizeof(GsRecount), stream_), "memset")) return false;
    if (first < g.n && count) {
      if (count > g.n - first) count = g.n - first;
      gs_recount_kernel<<<(count + GS_BLOCK - 1) / GS_BLOCK, GS_BLOCK, 0, stream_>>>(d, g_dev, now, first, count, dr);
      ++launches_;
    }
    return ok(cudaGetLastError(), "recount launch") && d2h(out, dr, sizeof(GsRecount));
  }
  bool state_hash(const GsDev& d, const GsGlobals* g_dev, const GsGlobals& g, uint32_t now,
                  uint64_t out[4]) override {
    cudaSetDevice(dev_);
    unsigned long long* dh = reinterpret_cast<unsigned long long*>(scratch_);
    if (!ok(cudaMemsetAsync(dh, 0, 32, stream_), "memset")) return false;
    if (g.n) {
      gs_hash_kernel<<<(g.n + GS_BLOCK - 1) / GS_BLOCK, GS_BLOCK, 0, stream_>>>(d, g_dev, now, dh);
      ++launches_;
    }
    return ok(cudaGetLastError(), "hash launch") && d2h(out, dh, 32);
  }
  // ---- sharded pools -----------------------------------------------------------------------
  bool shard_begin(uint32_t world, uint32_t rank) override {
    cudaSetDevice(dev_);
    cudaFree(0);  // make sure the primary context exists before driver-API calls
    sharded_ = vmm_.init(dev_, world, rank, err_, sizeof(err_));
    return sharded_;
  }
  size_t shard_granularity() override { return vmm_.granularity(); }
  void* shard_alloc(size_t slice_bytes, size_t planes) override {
    void* q = vmm_.reserve(slice_bytes, planes);
    if (!q) snprintf(err_, sizeof(err_), "%s", vmm_.last_error());
    return q;
  }
  bool shard_commit(const int** fds, size_t* n) override {
    if (!vmm_.commit()) {
      snprintf(err_, sizeof(err_), "%s", vmm_.last_error());
      return false;
    }
    *fds = vmm_.export_fds().data();
    *n = vmm_.export_fds().size();
    return true;
  }
  bool shard_attach(uint32_t peer, const int* fds, size_t n) override {
    cudaSetDevice(dev_);
    if (!vmm_.attach(peer, fds, n)) {
      snprintf(err_, sizeof(err_), "%s", vmm_.last_error());
      return false;
    }
    return true;
  }
  bool xbar_host(const GsXbar& xb) override {
    cudaSetDevice(dev_);
    gs_xbar_kernel<<<1, 32, 0, stream_>>>(xb);
    ++launches_;
    return ok(cudaGetLastError(), "xbar launch") && ok(cudaStreamSynchronize(stream_), "xbar");
  }
  bool and_columns(const GsDev& d, const GsGlobals& g, uint32_t keep, uint32_t first, uint32_t count) override {
    cudaSetDevice(dev_);
    if (first >= g.n || !count) return true;
    if (count > g.n - first) count = g.n - first;
    gs_and_kernel<<<(count + GS_BLOCK - 1) / GS_BLOCK, GS_BLOCK, 0, stream_>>>(d, first, count, keep);
    ++launches_;
    return ok(cudaGetLastError(), "and launch") && ok(cudaStreamSynchronize(stream_), "and");
  }
  bool sync() override {
    cudaSetDevice(dev_);
    return ok(cudaStreamSynchronize(stream_), "sync");
  }
  const char* last_error() const override { return err_; }
  uint64_t total_launches() const override { return launches_; }

 private:
  cudaError_t cudaMemsetD32Async_(uint32_t* dst, uint32_t value, size_t count) {
    // the runtime API has no 32-bit memset: a grid-stride fill kernel on the pool's stream
    if (!count) return cudaSuccess;
    size_t blocks = (count + GS_BLOCK - 1) / GS_BLOCK;
    if (blocks > 148u * 16u) blocks = 148u * 16u;
    gs_fill32_kernel<<<(unsigned)blocks, GS_BLOCK, 0, stream_>>>(dst, value, count);
    ++launches_;
    return cudaGetLastError();
  }
  cudaGraphExec_t graph_for(const GsDev& d, const GsGlobals* g_dev, uint32_t blocks, const GsXbar* xbar) {
    // the column pointers are baked into the captured launches: if they changed (a peer graph was
    // attached or removed), every cached graph is stale
    if (have_graph_dev_ && memcmp(&graph_dev_, &d, sizeof(GsDev)) != 0) {
      for (auto& kv : graphs_) cudaGraphExecDestroy(kv.second);
      graphs_.clear();
      for (auto& kv : wgraphs_) cudaGraphExecDestroy(kv.second);
      wgraphs_.clear();
    }
    graph_dev_ = d;
    have_graph_dev_ = true;
    auto it = graphs_.find(blocks);
    if (it != graphs_.end()) return it->second;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t ge = nullptr;
    if (!ok(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal), "capture"))
      return nullptr;
    for (uint32_t k = 0; k < GS_GRAPH_TICKS; ++k)
      if (!ok(gs_launch_tick(blocks, stream_, d, g_dev, k, pdl_ && !xbar), "tick capture")) {
        cudaGraph_t dead = nullptr;
        cudaStreamEndCapture(stream_, &dead);
        if (dead) cudaGraphDestroy(dead);
        return nullptr;
      }

    gs_advance_kernel<<<1, 1, 0, stream_>>>(d.tick_base, GS_GRAPH_TICKS, nullptr);
    if (!ok(cudaStreamEndCapture(stream_, &graph), "end capture")) return nullptr;
    if (!ok(cudaGraphInstantiate(&ge, graph, 0), "instantiate")) {
      cudaGraphDestroy(graph);
      return nullptr;
    }
    cudaGraphDestroy(graph);
    graphs_[blocks] = ge;
    return ge;
  }
  cudaGraphExec_t window_graph_for(const GsDev& d, const GsGlobals* g_dev, uint32_t blocks, uint32_t K, bool pdl, uint32_t rank) {
    if (have_graph_dev_ && memcmp(&graph_dev_, &d, sizeof(GsDev)) != 0) {
      for (auto& kv : graphs_) cudaGraphExecDestroy(kv.second);
      graphs_.clear();
      for (auto& kv : wgraphs_) cudaGraphExecDestroy(kv.second);
      wgraphs_.clear();
    }
    graph_dev_ = d;
    have_graph_dev_ = true;
    const uint64_t key = ((uint64_t)blocks << 32) | K;
    auto it = wgraphs_.find(key);
    if (it != wgraphs_.end()) return it->second;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t ge = nullptr;
    if (!ok(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal), "capture")) return nullptr;
    bool good = true;
    for (uint32_t j = 0; j < GS_WIN_GRAPH && good; ++j)
      good = ok(gs_launch_window(blocks, stream_, d, g_dev, j * K, K, pdl, win_mode_), "window capture");
    if (good) gs_window_advance_kernel<<<1, 1, 0, stream_>>>(d.tick_base, d.qstate[rank]);
    if (!ok(cudaStreamEndCapture(stream_, &graph), "end capture") || !good) {
      if (graph) cudaGraphDestroy(graph);
      return nullptr;
    }
    if (!ok(cudaGraphInstantiate(&ge, graph, 0), "instantiate")) {
      cudaGraphDestroy(graph);
      return nullptr;
    }
    cudaGraphDestroy(graph);
    wgraphs_[key] = ge;
    return ge;
  }
  bool ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    snprintf(err_, sizeof(err_), "%s: %s", what, cudaGetErrorString(e));
    return false;
  }
  int dev_;
  cudaStream_t stream_;
  cudaEvent_t ev0_, ev1_;
  void* scratch_;
  uint32_t full_grid_ = 592;
  uint32_t win_grid_ = 592;
  GsVmm vmm_;
  bool sharded_ = false;
  bool pdl_ = getenv("GSIM_NO_PDL") == nullptr;
  // sharded pools: stream launches measured faster than graph replay (21 vs 28 us/tick at 2 Mi
  // members per GPU on 2 GPUs); GSIM_SHARD_GRAPH=1 turns the graph path on
  bool no_shard_graph_ = getenv("GSIM_SHARD_GRAPH") == nullptr;
  // window kernel: how groups are dealt to the warps (bit 1 of the kernel's mode word); GSIM_WIN_CYCLIC=0/1
  uint32_t win_mode_ = getenv("GSIM_WIN_CYCLIC") && atoi(getenv("GSIM_WIN_CYCLIC")) ? 2u : 0u;
  std::map<uint32_t, cudaGraphExec_t> graphs_;
  std::map<uint64_t, cudaGraphExec_t> wgraphs_;
  GsDev graph_dev_;
  bool have_graph_dev_ = false;
  bool l2_window_set_ = false;
  uint64_t launches_ = 0;
  char err_[256];
};

}  // namespace

GsBackend* gs_make_cuda_backend(int device, char* err, size_t err_cap) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    snprintf(err, err_cap, "no CUDA device: %s (libgsim has no CPU fallback)",
             e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return nullptr;
  }
  if (device < 0) {
    if (cudaGetDevice(&device) != cudaSuccess) device = 0;
  }
  if (device >= count) {
    snprintf(err, err_cap, "CUDA device %d out of range (%d devices)", device, count);
    return nullptr;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
    snprintf(err, err_cap, "device %d is not sm_100-class (libgsim ships sm_100a SASS only)",
             device);
    return nullptr;
  }
  if (cudaSetDevice(device) != cudaSuccess) {
    snprintf(err, err_cap, "cudaSetDevice(%d) failed", device);
    return nullptr;
  }
  return new CudaBackend(device);
}
