"""Per-tick profile of one join cascade (dev tool): for each libgsim build given on the command line, a
1 M-member pool takes one joiner and is stepped one tick at a time; prints the CUDA-event time of every
tick (sched_counts tick_ms / window_ms deltas), the cascade's ramp / plateau / tail split and the final
state hash.  Builds that compute the same thing print the same hash."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from consul_b200 import _lib
from consul_b200.pool import Pool, lan_config

N, TICKS = 1_000_000, 64
for path in sys.argv[1:]:
    lib = _lib.load(path)
    p = Pool(lan_config(lib, capacity=N + 16, n_initial=N, seed=0x5EED0001), lib)
    p.step(64)
    x = p.member_add(); p.join(x, [0])
    us = []
    for _ in range(TICKS):
        c0 = p.sched_counts()
        p.step(1)
        c1 = p.sched_counts()
        us.append((c1["tick_ms"] - c0["tick_ms"] + c1["window_ms"] - c0["window_ms"]) * 1e3)
    busy = [k for k, u in enumerate(us) if u >= 0.5 * max(us)]
    lo, hi = (busy[0], busy[-1] + 1) if busy else (0, 0)
    parts = {"ramp": us[:lo], "plateau": us[lo:hi], "tail": us[hi:]}
    print(f"{path}: hash {p.state_hash()[0]:016x}, {sum(us) / 1e3:.3f} ms over {TICKS} ticks; " +
          ", ".join(f"{k} {len(v)} ticks {sum(v) / 1e3:.3f} ms" for k, v in parts.items()), flush=True)
    print("  us/tick: " + " ".join(f"{u:.0f}" for u in us), flush=True)
    p.close()
