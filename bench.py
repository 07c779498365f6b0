#!/usr/bin/env python
"""bench.py — BASELINE metric: million node-ticks/sec (+ ticks-to-full-convergence).

Workload at N=1 GPU = BASELINE.json configs[1]: 1,000,000 converged virtual members, default
LAN config (probe 1 s / 500 ms, gossip 200 ms x 3, tau = 100 ms), single join cascade.
One STEP = one joiner is created and joins through seed 0 (serf.Create + Join), then the pool
advances TICKS_PER_STEP lock-step ticks (the cascade converges in ~30 ticks, the rest is
steady-state probing, SURVEY §8d C2 "time a >= 2000-tick window").

  value      node-ticks/s with the cluster state already resident in HBM (wall clock around
             exactly K steps, barrier + cuda synchronize on both sides, max over ranks)
  e2e        the same through the reference-facing C ABI with HOST buffers: every step restores
             the cluster from a pinned host snapshot (H2D), joins, ticks, and reads Members()
             and the stats back (D2H)
  roofline   gs_tick_kernel: algorithmic bytes / CUDA-event time of the tick launches
  cpu_baseline / --impl reference   the oracle (CPU restatement) on the host cores

Multi-GPU (`torchrun ... --gpus N`): see DESIGN.md §7.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark runs from the tree build() left, which may be read-only: no bytecode caches in it
sys.dont_write_bytecode = True

N_MEMBERS = 1_000_000
TICKS_PER_STEP = 2048
SEED = 0x5EED0001
N_HBM = 67_108_864          # secondary roofline point: 268 MB mailbox column + cold columns exceed the 126 MB L2
HBM_TICKS = 256
MEMBERS_PER_GPU_SHARDED = 1024 * 1024   # ~ the single-GPU workload per GPU: an honest weak-scaling curve

# Algorithmic bytes (DESIGN.md §4): useful bytes the algorithm has to move, not sectors.
# gs_tick_kernel (one tick per launch): every member reads its 4-byte mailbox word; tiles whose
# ticker phase can be due at this tick (2 of every P ticks) also read `due`; members that act pay
# for the cold columns they touch.
B_SCAN = 4.0        # inbox[t&1][i]
B_DUE = 4.0         # due[i], on 2/P of the ticks
B_ACTIVE = 24.0     # key, meta, due, queued reads; inbox clear; wake / write-back word
B_PROBE = 12.0      # extra for a probe start: cursor r/w, pass, target key gather, due write
B_ACCEPT = 21.0     # heard r/w, queued write, tx init, Lamport clock witness
B_PACKET = 12.0     # peer key gather + mailbox atomic RMW
B_RUMOR_TX = 2.0    # tx counter r/w per broadcast carried
# gs_window_kernel (a whole window of ticks per launch, quiet pool): no mailbox word is read at all.  A
# member's probe state is read once per launch (due, key, meta, cursor, pass), kept in registers while it
# runs all its probes of the launch, and written back once (cursor, due); each probe gathers the target's
# status byte.
B_WIN_ROW = 4.0 * 5 + 4.0 * 2
B_WIN_PROBE = 1.0


def split_bytes(d: dict, sc: dict, n_members: float, P: int) -> dict:
    """Algorithmic bytes of the timed region by kernel.  `d` = counter deltas, `sc` = scheduling
    deltas (window launches / ticks, single ticks).  Inside quiet windows every member starts exactly
    one probe per P ticks and nothing else happens, so the window kernel's share of the shared
    counters is window_ticks * n / P probes."""
    win_probes = min(float(d["probes"]), sc["window_ticks"] * n_members / P)
    # (launches in closed form — pristine pool — gather no status bytes: their probes cost no bytes at all)
    gathered = min(win_probes, (sc["window_ticks"] - sc.get("closed_form_ticks", 0)) * n_members / P)
    win = sc["window_launches"] * n_members * B_WIN_ROW + gathered * B_WIN_PROBE
    tick_nt = sc["tick_launches"] * n_members
    tick = (tick_nt * (B_SCAN + B_DUE * 2.0 / P) + max(0.0, d["active_rows"] - win_probes) * B_ACTIVE +
            max(0.0, d["probes"] - win_probes) * B_PROBE + d["rumors_accepted"] * B_ACCEPT +
            d["gossip_packets"] * B_PACKET + d["rumors_sent"] * B_RUMOR_TX)
    return {"window": win, "tick": tick}


def roofline_of(kernel: str, bytes_: float, ms: float, launches: int, ticks: int, n_members: float, peak: float,
                peak_src: str, traffic) -> dict:
    if launches == 0 or ms <= 0:
        return None
    achieved = bytes_ / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "per_gpu": True, "traffic": traffic, "peak_source": peak_src,
            "bytes_per_launch": bytes_ / launches, "launch_us": ms * 1e3 / launches, "launches": launches,
            "ticks_per_launch": ticks / launches, "bytes_per_node_tick": bytes_ / max(1.0, ticks * n_members),
            "share_of_kernel_time": None}


def stat_delta(a: dict, b: dict) -> dict:
    return {k: b[k] - a[k] for k in ("node_ticks", "probes", "rumors_accepted", "gossip_packets",
                                     "rumors_sent", "active_rows")}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self) -> dict:
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples if len(s) >= 7 for i in range(4)
                          if s[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------
# CPU side: the oracle (oracle/oracle.cpp, kind "port" — the Go modules that hold the reference
# arithmetic are not in /root/reference and there is no Go toolchain, SURVEY §8c).  Nothing below
# imports the product package's loader or maps consul_b200/libgsim.so.
CASCADE_TICKS = 128          # the join cascade and its retransmissions end well before this


def _oracle():
    """oracle_binding without building or loading anything of the product."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIBORACLE):     # build() made it; the tree is not written otherwise
        ge.build_oracle()
    import oracle_binding
    return oracle_binding


def host_cores() -> dict:
    """Logical CPUs this process may run on, and how many distinct physical cores they are."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        allowed = list(range(os.cpu_count() or 1))
    cores = set()
    for c in allowed:
        try:
            base = f"/sys/devices/system/cpu/cpu{c}/topology/"
            with open(base + "physical_package_id") as f1, open(base + "core_id") as f2:
                cores.add((f1.read().strip(), f2.read().strip()))
        except OSError:
            cores.add(("?", str(c)))
    return {"logical": len(allowed), "physical": len(cores)}


def pick_threads(o, probe_ticks: int = 4) -> tuple:
    """Give the CPU arm its best thread count: time a few ticks at each candidate (all logical
    CPUs, the physical cores, half of them) and keep the fastest.  OpenMP with static chunks and a
    barrier per tick collapses when threads outnumber the cores it really gets (round 1: 128 threads
    on the bench box ran 32x slower than 64), so the count is measured, not assumed."""
    hc = host_cores()
    cands = sorted({hc["logical"], hc["physical"], max(1, hc["physical"] // 2)}, reverse=True)
    best, tried = None, {}
    for th in cands:
        o.set_threads(th)
        o.step(1)
        t0 = time.perf_counter()
        o.step(probe_ticks)
        dt = time.perf_counter() - t0
        tried[th] = dt / probe_ticks
        if best is None or dt < best[1]:
            best = (th, dt)
    o.set_threads(best[0])
    return best[0], {"host": hc, "s_per_tick_by_threads": {str(k): round(v, 5) for k, v in tried.items()}}


def oracle_step_sampled(o, ticks: int, budget_s: float) -> tuple:
    """One step (after the join) on the oracle: the cascade part is always timed in full; the steady
    remainder is timed until `ticks` are done or the budget is spent, and then scaled to `ticks`.
    Returns (seconds for the whole step — measured or scaled —, ticks actually executed)."""
    t0 = time.perf_counter()
    head = min(ticks, CASCADE_TICKS)
    o.step(head)
    t_head = time.perf_counter() - t0
    done, t_tail = head, 0.0
    while done < ticks and (done == head or (t_head + t_tail) < budget_s):   # at least one steady chunk
        c = min(64, ticks - done)
        t1 = time.perf_counter()
        o.step(c)
        t_tail += time.perf_counter() - t1
        done += c
    if done == ticks:
        return t_head + t_tail, done
    per_tick = t_tail / (done - head) if done > head else t_head / head
    return t_head + t_tail + per_tick * (ticks - done), done


def workload_config(n: int, ticks: int, world: int, sharded: bool) -> dict:
    """The `config` object of the bench line — built by ONE function for both arms so that the
    reference line carries exactly the repo arm's config."""
    return {"workload": f"C2: {n:,} converged members + 1 joiner per step, LAN defaults "
                        f"(probe 1s/500ms, gossip 200ms x3), tau=100 ms, {ticks} ticks/step",
            "members": n, "members_per_gpu": n // world if sharded else n, "ticks_per_step": ticks, "seed": hex(SEED),
            "parallelism": (f"one pool range-sharded over {world} GPUs, P2P mailboxes over NVLink inside the tick "
                            "kernel, device barrier per tick") if sharded else "single GPU",
            "l2": "not flushed: a step is 2048 dependent ticks over the same state, whose hot "
                  "columns are L2-resident by construction; see roofline_hbm for the >L2 size"}


def workload_shape(args, world: int) -> tuple:
    """(members, capacity, sharded) of the pool both arms simulate at this --gpus."""
    total_steps = args.steps + args.warmup
    if world > 1:
        per_gpu = args.members_per_gpu
        return per_gpu * world - 256, per_gpu * world, True
    return args.members, args.members + 2 * total_steps + 8, False


DUMP_BYTES = 64 << 20       # --dump-outputs writes at most this much


def dump_outputs(out_dir: str, pool, with_members: bool) -> None:
    """What the last timed step leaves a caller with, as float64 .npy files (every value is an
    integer below 2**53, so float64 holds it exactly):
      stats.npy       Stats() in the order of consul_b200.pool.Pool.stats(), without active_rows
                      (how many rows left the kernels' idle fast path: a scheduling count, not a result)
      state_hash.npy  the 256-bit state digest as eight 32-bit words, high word of each 64-bit lane first
      members.npy     Members() as member 0 reports it, one row (id, status, incarnation, rank) per
                      member; beyond the byte budget, a fixed seeded sample of rows in id order
    Members() of a sharded pool would pull every row through rank 0, so it is left out there.  Every
    rank of a sharded pool must issue the same reads; the ranks other than 0 pass out_dir=None.
    (The reference arm's state is that of the ticks it executed: reproducible when its line's
    cpu_baseline.sample says every tick was.)"""
    import numpy as np
    st = pool.stats()
    st.pop("active_rows")
    stats = [float(x) for v in st.values() for x in (v if isinstance(v, list) else [v])]
    digest = [float(w) for h in pool.state_hash() for w in (h >> 32, h & 0xFFFFFFFF)]
    members = np.array(pool.members(0), dtype=np.float64) if with_members else None
    if out_dir is None:
        return
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "stats.npy"), np.array(stats, dtype=np.float64))
    np.save(os.path.join(out_dir, "state_hash.npy"), np.array(digest, dtype=np.float64))
    if members is not None:
        max_rows = (DUMP_BYTES - (1 << 20)) // members.itemsize // 4
        if len(members) > max_rows:
            rows = np.sort(np.random.default_rng(SEED).choice(len(members), max_rows, replace=False))
            members = members[rows]
        np.save(os.path.join(out_dir, "members.npy"), members)


def mapped_native_libs() -> list:
    out = set()
    try:
        with open("/proc/self/maps") as f:
            for ln in f:
                path = ln.split()[-1]
                if path.startswith(ROOT) and path.endswith(".so"):
                    out.add(os.path.relpath(path, ROOT))
    except OSError:
        pass
    return sorted(out)


def run_reference(args, rank: int, world: int):
    """Reference arm: the CPU implementation of the path on the host cores, the SAME cluster
    (members, seed, config) and the same step (join + `--ticks` ticks) as the repo arm at this
    --gpus.  Under torchrun only rank 0 works."""
    if rank != 0:
        return
    # torchrun pins OMP_NUM_THREADS=1 in its workers: this arm is a CPU program and takes the cores
    os.environ.pop("OMP_NUM_THREADS", None)
    ob = _oracle()
    n, cap, sharded = workload_shape(args, max(world, args.gpus))
    w = max(world, args.gpus)
    ticks = args.ticks
    cfg = ob.oracle_config("lan", capacity=cap, n_initial=n, seed=SEED)
    o = ob.OraclePool(cfg, threads=0)
    threads, tune = pick_threads(o)
    total = args.steps + args.warmup
    budget = float(os.environ.get("GSIM_REF_BUDGET_S", "300")) / max(1, total)

    def one_step():
        t0 = time.perf_counter()
        x = o.member_add()
        assert o.join(x, [0]) == 1
        t_host = time.perf_counter() - t0
        secs, done = oracle_step_sampled(o, ticks, budget)
        return t_host + secs, done

    for _ in range(args.warmup):
        one_step()
    secs, executed = 0.0, 0
    for _ in range(args.steps):
        s_, d_ = one_step()
        secs += s_
        executed += d_
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, o, with_members=True)
    n_now = o.stats()["n_members"]
    val = float(n_now) * ticks * args.steps / secs / 1e6
    exact = executed == ticks * args.steps
    sample = (f"{args.steps} steps x (join + {ticks} ticks) x {n_now:,} members, every tick executed" if exact else
              f"{args.steps} steps x {n_now:,} members: join + ticks 0..{CASCADE_TICKS} timed in full, then "
              f"{executed // args.steps - CASCADE_TICKS} steady ticks per step timed and scaled to {ticks} "
              f"(budget {budget:.0f} s per step)")
    line = {
        "impl": "reference", "metric": "million node-ticks/sec", "value": val, "unit": "M node-ticks/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(n, ticks, w, sharded),
        "cpu_baseline": {"value": val, "unit": "M node-ticks/s", "cores": threads, "kind": "port",
                         "sample": sample, "thread_tuning": tune},
        "e2e": {"value": val, "unit": "M node-ticks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "digest": "%016x" % o.state_hash()[0],
        "native_so_loaded": mapped_native_libs(),
    }
    assert not any("libgsim" in x for x in line["native_so_loaded"]), line["native_so_loaded"]
    print(json.dumps(line), flush=True)


def cpu_baseline_sample(n: int, cap: int, ticks: int, budget_s: float = 15.0) -> dict:
    """cpu_baseline of the repo arm's line: one step of the same workload on the oracle."""
    os.environ.pop("OMP_NUM_THREADS", None)
    ob = _oracle()
    o = ob.OraclePool(ob.oracle_config("lan", capacity=cap, n_initial=n, seed=SEED), threads=0)
    threads, tune = pick_threads(o)
    x = o.member_add()
    o.join(x, [0])
    secs, done = oracle_step_sampled(o, ticks, budget_s)
    return {"value": float(n + 1) * ticks / secs / 1e6, "unit": "M node-ticks/s", "cores": threads, "kind": "port",
            "sample": (f"one step of the same workload ({n + 1:,} members, join + {ticks} ticks): "
                       + ("every tick executed" if done == ticks else
                          f"ticks 0..{CASCADE_TICKS} in full + {done - CASCADE_TICKS} steady ticks scaled to {ticks}")
                       + f", {secs:.1f} s"), "thread_tuning": tune}


PARITY_TICKS = 96


def parity_script(p) -> dict:
    """The parity replay both sides run on a fresh pool: one joiner through seed 0, PARITY_TICKS
    ticks (cascade converged and retransmissions finished), digest + the counters that must match."""
    x = p.member_add()
    joined = p.join(x, [0])
    p.step(PARITY_TICKS)
    st = p.stats()
    return {"digest": "%016x" % p.state_hash()[0], "joined": joined, "now": p.now,
            "counters": {k: st[k] for k in ("probes", "acks", "gossip_packets", "rumors_sent", "rumors_accepted")}}


# --------------------------------------------------------------------------------------------
def kernel_source_sha() -> str:
    """Identity of the tick-kernel sources: profiles/traffic.json is trusted only for this build."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "consul_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".h", ".cu", ".cpp")):
            with open(os.path.join(csrc, f), "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()[:16]


def measured_traffic(key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel from the
    `ncu --set full` capture of THIS build (tools/ncu_traffic.py writes profiles/traffic.json with
    the source hash it profiled); null when the kernel sources have changed since."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        if t.get("kernel_source_sha") != kernel_source_sha():
            return None
        return t.get(key)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gsim", choices=["gsim", "reference"])
    ap.add_argument("--members", type=int, default=N_MEMBERS, help="members of the single-GPU pool")
    ap.add_argument("--members-per-gpu", type=int, default=MEMBERS_PER_GPU_SHARDED,
                    help="members per GPU of the sharded pool (--gpus > 1)")
    ap.add_argument("--ticks", type=int, default=TICKS_PER_STEP)
    ap.add_argument("--skip-hbm-point", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — libgsim has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from consul_b200.pool import Pool, lan_config, PRED_RUMOR_CONVERGED

    ticks = args.ticks
    n, cap, sharded = workload_shape(args, world)
    if sharded:
        # one pool sharded over all ranks (DESIGN.md §7); the last 256 ids are left for joiners
        from consul_b200.sharded import ShardedPool
        cfg = lan_config(capacity=cap, n_initial=n, seed=SEED, device=local_rank)
        pool = ShardedPool(cfg)
    else:
        cfg = lan_config(capacity=cap, n_initial=n, seed=SEED, device=local_rank)
        pool = Pool(cfg)
    gi = pool.stats()["probe_interval_ticks"]  # P: the due column is read on 2/P of the ticks

    # ---- parity of THIS run's pool: the first step is replayed on the CPU oracle (and, for a
    # sharded pool, on one GPU) and the 256-bit state digests must be equal ---------------------
    parity = None
    if not args.skip_parity:
        got = parity_script(pool)
        parity = {"what": f"fresh pool of {n:,} members: member_add + join(seed 0) + {PARITY_TICKS} ticks; "
                          "first 64 bits of the 256-bit order-independent state digest + counters",
                  "digest": got["digest"]}
        if rank == 0:
            omp_saved = os.environ.pop("OMP_NUM_THREADS", None)
            ob = _oracle()
            # (no thread tuning on THIS pool: tuning steps the clock; half the physical cores is what the
            # tuning picks on the bench boxes)
            o = ob.OraclePool(ob.oracle_config("lan", capacity=cap, n_initial=n, seed=SEED),
                              threads=max(1, host_cores()["physical"] // 2))
            want = parity_script(o)
            o.close()
            if omp_saved is not None:
                os.environ["OMP_NUM_THREADS"] = omp_saved
            parity["digest_oracle"] = want["digest"]
            ok = got == want
            if sharded:
                ref = Pool(lan_config(capacity=cap, n_initial=n, seed=SEED, device=local_rank))
                one = parity_script(ref)
                ref.close()
                parity["digest_single_gpu"] = one["digest"]
                ok = ok and got == one
            parity["parity_ok"] = bool(ok)
            if not ok:
                sys.stderr.write(f"bench.py: PARITY MISMATCH got={got} oracle={want}\n")

    def step_resident():
        x = pool.member_add()
        assert pool.join(x, [0]) == 1
        t_start = pool.now
        pool.step(ticks)
        return x, t_start

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local_rank)
    sampler.start()
    s0 = pool.stats()
    l0 = pool.launch_count()
    c0 = pool.sched_counts()
    kernel_ms, tick_launches = 0.0, 0
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        x, t_start = step_resident()
        ms, nl = pool.last_step_timing()
        kernel_ms += ms
        tick_launches += nl
    barrier()
    dt = time.perf_counter() - t0
    s1 = pool.stats()
    l1 = pool.launch_count()
    c1 = pool.sched_counts()
    d = stat_delta(s0, s1)
    sc = {k: c1[k] - c0[k] for k in c1}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if rank == 0 else None, pool, with_members=not sharded)

    # ticks-to-full-convergence of one cascade (untimed, exact tick recorded on the device)
    x = pool.member_add()
    pool.join(x, [0])
    t_join = pool.now
    slot_alive = None
    for r in range(30):
        try:
            info = pool.rumor_info(r)
        except Exception:
            continue
        if info["kind"] == 1 and info["subject"] == x:
            slot_alive = r
    t_conv = pool.run_until(PRED_RUMOR_CONVERGED, slot_alive, 400, 1)
    ticks_to_conv = int(t_conv - t_join + 1) if t_conv != 0xFFFFFFFF else None
    pool.step(64)

    # ---- e2e: HOST buffers through the C ABI, H2D + D2H inside the timed region -----------
    import ctypes as C
    restore_ok = False
    if sharded:
        # sharded pool: the cluster stays resident on the GPUs; the per-step host traffic is the
        # join operation (pokes) and the result read-back (stats, NumNodes of the joiner)
        def step_e2e():
            xx, _ = step_resident()
            # the result a caller reads back: cluster-wide counts (recount kernels on every GPU, a few hundred
            # bytes to the host) — not Members(), which on a sharded pool would pull every key through rank 0
            return pool.stats()["n_view_alive"]
        for _ in range(min(args.warmup, 3)):
            step_e2e()
        barrier()
        te0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        barrier()
        dte = time.perf_counter() - te0
        sampler.stop_flag.set()
        sampler.join(timeout=2)
        n_now = pool.stats()["n_members"]
        e2e_nodeticks = float(n_now) * ticks * args.steps
        h2d, d2h = 4096, 4096
        blob = None
    else:
        blob = pool.snapshot()
        pinned = torch.empty(len(blob), dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = memoryview(blob)
        blob_ptr = C.c_void_p(pinned.data_ptr())
        from consul_b200._lib import GsimMember
        mem_cap = cap
        mem_buf = (GsimMember * mem_cap)()
        mem_n = C.c_size_t()
        lib = pool.lib

        # self-check of the checkpoint path before it is timed: a few ticks forward, restore, and the
        # digest must be the one taken with the snapshot.  If it is not, the e2e number keeps the
        # cluster resident (and says so) instead of taking the bench line down with it.
        h_snap = pool.state_hash()
        try:
            pool.step(3)
            restore_ok = lib.gsim_restore(pool.h, blob_ptr, len(blob)) == 0 and pool.state_hash() == h_snap
        except Exception:
            restore_ok = False
        if not restore_ok:
            sys.stderr.write("bench.py: snapshot/restore self-check FAILED; e2e runs with the cluster resident\n")

        def step_e2e():
            if restore_ok:
                rc = lib.gsim_restore(pool.h, blob_ptr, len(blob))
                assert rc == 0, rc
            xx = pool.member_add()
            assert pool.join(xx, [0]) == 1
            pool.step(ticks)
            rc = lib.gsim_members(pool.h, 0, mem_buf, mem_cap, C.byref(mem_n))
            assert rc == 0 and mem_n.value == xx + 1
            return pool.stats()["n_view_alive"]

        for _ in range(min(args.warmup, 3)):
            step_e2e()
        barrier()
        te0 = time.perf_counter()
        for _ in range(args.steps):
            alive = step_e2e()
        barrier()
        dte = time.perf_counter() - te0
        sampler.stop_flag.set()
        sampler.join(timeout=2)
        n_now = pool.stats()["n_members"]
        e2e_nodeticks = float(n_now) * ticks * args.steps
        h2d = len(blob) if restore_ok else 4096
        d2h = mem_n.value * C.sizeof(GsimMember) + n_now * 4 + 512

    # ---- max over ranks, aggregate ------------------------------------------------------------
    tt = torch.tensor([dt, dte, kernel_ms], dtype=torch.float64, device="cuda")
    nt = torch.tensor([float(d["node_ticks"]), e2e_nodeticks], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        # a sharded pool's counters are already global (every rank reports the same totals)
    dt_max, dte_max, kms_max = [float(v) for v in tt.tolist()]
    node_ticks_all, e2e_all = [float(v) for v in nt.tolist()]

    # ---- roofline per kernel, PER GPU (a sharded pool's counters are whole-job totals: each GPU moves
    # 1/world of the bytes against one GPU's peak).  `roofline` = the kernel that took more of the time.
    peak, peak_src = measured_peak_gbs()
    by = split_bytes(d, sc, float(n), gi)
    one_m = (not sharded and n == N_MEMBERS)
    r_tick = roofline_of("gs_tick_kernel", by["tick"] / world, sc["tick_ms"], sc["tick_launches"], sc["tick_launches"],
                         float(n) / world, peak, peak_src, measured_traffic("traffic_tick_cascade_1m_bytes") if one_m else None)
    r_win = roofline_of("gs_window_kernel", by["window"] / world, sc["window_ms"], sc["window_launches"], sc["window_ticks"],
                        float(n) / world, peak, peak_src, measured_traffic("traffic_window_1m_bytes") if one_m else None)
    total_ms = sc["tick_ms"] + sc["window_ms"]
    for r, ms_ in ((r_tick, sc["tick_ms"]), (r_win, sc["window_ms"])):
        if r:
            r["share_of_kernel_time"] = ms_ / total_ms if total_ms > 0 else None
    roofline = r_tick if (r_tick and (not r_win or sc["tick_ms"] >= sc["window_ms"])) else r_win
    roofline = dict(roofline)
    roofline["note"] = ("the kernel with the larger share of the step's kernel time; both kernels are in roofline_kernels. "
                        "1M members: the hot columns are L2-resident by construction (2048 dependent ticks over the same "
                        "state); roofline_hbm below is the HBM-bound size")
    # SURVEY §8(d)'s per-unit figure (every member's 32-byte row read and written every tick + rumor columns +
    # 0.2 messages: 82 B per node-tick in LAN steady state) x the node-ticks of the timed region: the yardstick
    # of a kernel that streams the whole state every tick.  This path does not touch idle rows, so it runs
    # above 1.0 of it; the byte models above are the honest ones.
    roofline["survey_model"] = {"bytes_per_node_tick": 82.0,
                                "achieved": 82.0 * d["node_ticks"] / world / (total_ms * 1e-3) / 1e9 if total_ms > 0 else None,
                                "unit": "GB/s", "frac": (82.0 * d["node_ticks"] / world / (total_ms * 1e-3) / 1e9 / peak) if total_ms > 0 else None}
    roofline["whole_step"] = {"achieved": (by["tick"] + by["window"]) / world / (total_ms * 1e-3) / 1e9 if total_ms > 0 else None,
                              "unit": "GB/s", "bytes_per_node_tick": (by["tick"] + by["window"]) / max(1.0, d["node_ticks"])}

    roofline_hbm = None
    if sharded:
        pool.close()
    if not args.skip_hbm_point and rank == 0 and not sharded:
        pool.close()
        big = Pool(lan_config(capacity=N_HBM, n_initial=N_HBM, seed=SEED, device=local_rank))
        big.step(64)
        b0, q0 = big.stats(), big.sched_counts()
        big.step(HBM_TICKS)
        b1, q1 = big.stats(), big.sched_counts()
        db = stat_delta(b0, b1)
        qd = {k: q1[k] - q0[k] for k in q1}
        byb = split_bytes(db, qd, float(N_HBM), gi)
        dominant_win = qd["window_ms"] >= qd["tick_ms"]
        roofline_hbm = roofline_of("gs_window_kernel" if dominant_win else "gs_tick_kernel",
                                   byb["window"] if dominant_win else byb["tick"],
                                   qd["window_ms"] if dominant_win else qd["tick_ms"],
                                   qd["window_launches"] if dominant_win else qd["tick_launches"],
                                   qd["window_ticks"] if dominant_win else qd["tick_launches"], float(N_HBM), peak, peak_src,
                                   measured_traffic("traffic_window_64m_bytes") if dominant_win else None)
        roofline_hbm.update({"members": N_HBM, "ticks": HBM_TICKS, "sched": qd,
                             "node_ticks_per_s": db["node_ticks"] / ((qd["window_ms"] + qd["tick_ms"]) * 1e-3),
                             "workload": f"{N_HBM:,} members, LAN steady state (4x BASELINE config 4 on one GPU; hot columns exceed L2)"})
        big.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    if not args.skip_cpu_baseline:
        cpu = cpu_baseline_sample(n, cap, ticks)

    # BASELINE's second metric for the other configs: recorded by tools/configs_report.py on a B200 and
    # committed (profiles/r2_configs.jsonl); carried in the line as a recorded artefact, not re-measured here
    conv = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_configs.jsonl")) as f:
            conv = [json.loads(ln) for ln in f if ln.strip().startswith("{")]
    except Exception:
        pass

    value = node_ticks_all / dt_max / 1e6
    line = {
        "metric": "million node-ticks/sec", "value": value, "unit": "M node-ticks/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(n, ticks, world, sharded),
        "ticks_to_convergence": ticks_to_conv,
        "ticks_to_convergence_other_configs": conv,
        "parity": parity, "digest": parity["digest"] if parity else None,
        "digest_oracle": parity.get("digest_oracle") if parity else None,
        "parity_ok": parity.get("parity_ok") if parity else None,
        "kernel_ms_per_step": kms_max / args.steps,
        "e2e": {"value": e2e_all / dte_max / 1e6, "unit": "M node-ticks/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": dte_max / args.steps * 1e3,
                "path": ("member_add -> join -> step -> stats (cluster resident, sharded)" if sharded else
                         "gsim_restore(pinned host snapshot) -> member_add -> join -> step -> members + stats" if restore_ok else
                         "member_add -> join -> step -> members + stats (cluster resident: restore self-check failed)")},
        "gpu_launches": int(l1 - l0),
        "sched": sc,
        "roofline": roofline, "roofline_kernels": {"gs_tick_kernel": r_tick, "gs_window_kernel": r_win},
        "roofline_hbm": roofline_hbm,
        "cpu_baseline": cpu,
        "clocks": sampler.summary(),
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
