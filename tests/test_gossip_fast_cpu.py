"""The fast gossip tier (gs_fast_gossip, DESIGN.md §4.1) on the host emulation: members with mail that
only repeats what they heard, or brings fresh alive / intent rumors, with their gossip turn and probe
ticker, skip the generic row step.  It is a schedule change, not a model change: with the tier, without
it (GSIM_FLAG_NO_FAST_GOSSIP) and on the oracle, every column, counter and the digest are equal at every
checkpoint — in cascades the tier takes, and in scenarios where it declines some or all rows."""
import ctypes as C

import pytest

from consul_b200.pool import (FLAG_NO_FAST_GOSSIP, FLAG_NO_WINDOWS, PRED_ALL_RUMORS_CONVERGED,
                              PRED_CRASHED_ALL_DEAD, NEVER, Pool, lan_config)
from oracle_binding import OraclePool
from parity import compare_pools


def row_counts(lib):
    """(rows the fast gossip tier took, rows that took the generic step) in single-tick launches so far"""
    out = (C.c_uint64 * 2)()
    lib.gsim_hostemu_row_counts(out)
    return out[0], out[1]


def trio(lib, flags=0, **kw):
    """the same pool with the tier, without it, and on the oracle"""
    return [Pool(lan_config(lib, flags=flags, **kw), lib),
            Pool(lan_config(lib, flags=flags | FLAG_NO_FAST_GOSSIP, **kw), lib),
            OraclePool(lan_config(lib, flags=flags, **kw))]


def all3(pools, fn):
    out = [fn(p) for p in pools]
    assert out[0] == out[1] == out[2], out
    return out[0]


def check(pools, where):
    compare_pools(pools[0], pools[2], where + " (tier vs oracle)")
    compare_pools(pools[0], pools[1], where + " (tier vs generic)")


def run(pools, ticks, every, where):
    done = 0
    while done < ticks:
        k = min(every, ticks - done)
        for p in pools:
            p.step(k)
        done += k
        check(pools, f"{where} +{done}")


def counted(lib, pool, ticks):
    """step one pool, return the rows each tier took meanwhile"""
    a = row_counts(lib)
    pool.step(ticks)
    b = row_counts(lib)
    return b[0] - a[0], b[1] - a[1]


@pytest.mark.parametrize("n", [1000, 20000])
@pytest.mark.parametrize("seed", [0x5EED0001, 7, 1234567])
def test_c2_cascade(hostemu_lib, n, seed):
    """BASELINE config 2: one joiner into a converged pool, checked every 8 ticks through the cascade"""
    pools = trio(hostemu_lib, capacity=n + 1, n_initial=n, seed=seed, flags=FLAG_NO_WINDOWS)
    for p in pools:
        p.step(16)
    x = all3(pools, lambda p: p.member_add())
    assert all3(pools, lambda p: p.join(x, [0])) == 1
    fast, generic_on = 0, 0
    generic_off = 0
    for k in range(12):
        f, g = counted(hostemu_lib, pools[0], 8)
        fast, generic_on = fast + f, generic_on + g
        generic_off += counted(hostemu_lib, pools[1], 8)[1]
        pools[2].step(8)
        check(pools, f"cascade +{8 * (k + 1)}")
    assert all(p.stats()["rumors_accepted"] == 2 * n - 1 for p in pools)
    if n == 20000:
        # the tier really is used: it takes at least 90 % of the rows the generic step took without it
        assert fast >= 0.9 * generic_off, (fast, generic_on, generic_off)


def test_joiners_in_flight(hostemu_lib):
    """two joiners (4 tracked broadcasts, taken), then nine more at once (22: more than the tier holds)"""
    n = 3000
    pools = trio(hostemu_lib, capacity=n + 16, n_initial=n, seed=41)
    for p in pools:
        p.step(12)
    for s in (5, 900):
        x = all3(pools, lambda p: p.member_add())
        all3(pools, lambda p: p.join(x, [s]))
    run(pools, 24, 4, "two joiners")
    for k in range(9):
        x = all3(pools, lambda p: p.member_add())
        all3(pools, lambda p: p.join(x, [17 * k + 3]))
    run(pools, 80, 8, "nine joiners")
    all3(pools, lambda p: p.run_until(PRED_ALL_RUMORS_CONVERGED, 0, 600, 8))
    check(pools, "converged")


def test_watched_member(hostemu_lib):
    """a watched member logs the join it hears: the generic step takes its fresh mail"""
    n = 2000
    pools = trio(hostemu_lib, capacity=n + 2, n_initial=n, seed=43, flags=1)
    for p in pools:
        p.member_watch(17)
        p.member_watch(1500)
    x = all3(pools, lambda p: p.member_add(watched=True))
    all3(pools, lambda p: p.join(x, [17]))
    run(pools, 60, 5, "watched")
    all3(pools, lambda p: [(e.tick, e.type, e.subject, e.observer) for e in p.poll_events()])


def test_user_event_during_cascade(hostemu_lib):
    n = 2000
    pools = trio(hostemu_lib, capacity=n + 2, n_initial=n, seed=47)
    x = all3(pools, lambda p: p.member_add())
    all3(pools, lambda p: p.join(x, [3]))
    run(pools, 6, 2, "cascade")
    all3(pools, lambda p: p.user_event(9, b"deploy", b"x" * 16, False))
    run(pools, 60, 4, "event in cascade")


@pytest.mark.parametrize("kind", ["loss", "latency", "push_pull", "graph", "budget"])
def test_declining_pools(hostemu_lib, kind):
    """pools the tier declines as a whole: identical with and without it"""
    n = 1200
    kw = dict(capacity=n + 4, n_initial=n, seed=53)
    if kind == "loss":
        kw["packet_loss_ppm"] = 50000
    elif kind == "budget":
        kw["udp_buffer_size"] = 120
    elif kind == "push_pull":
        kw["flags"] = 32
        kw["push_pull_interval_ns"] = 2_000_000_000
    elif kind == "latency":
        kw["mailbox_depth"] = 4
    pools = trio(hostemu_lib, **kw)
    if kind == "latency":
        lat = [[1 + ((a + b) % 3) for b in range(4)] for a in range(4)]
        for p in pools:
            p.latency_set(lat)
    if kind == "graph":
        import numpy as np
        rows = [sorted({(i + d) % n for d in (1, 2, 3, 5, 8, 13, 21, 34)}) for i in range(n)]
        row_ptr = np.cumsum([0] + [len(r) for r in rows]).astype(np.uint32)
        col_idx = np.concatenate([np.array(r, dtype=np.uint32) for r in rows])
        for p in pools:
            p.graph_set(row_ptr, col_idx)
    if kind == "graph":  # the member list of a graph pool is static: a user event and crashes instead
        all3(pools, lambda p: p.user_event(9, b"deploy", b"x" * 16, False))
        for p in pools:
            p.crash_many([10, 11, 12])
    for k in range(0 if kind == "graph" else 2 if kind == "budget" else 1):
        x = all3(pools, lambda p: p.member_add(alive_msg_size=60 if kind == "budget" else 0))
        all3(pools, lambda p: p.join(x, [k + 1]))
    before = row_counts(hostemu_lib)[0]
    run(pools, 60, 6, kind)
    if kind != "latency":
        assert row_counts(hostemu_lib)[0] == before  # declined: not one row taken


def test_crash_wave(hostemu_lib):
    """a crash wave during a cascade: SUSPECT and DEAD gossip candidates, suspicion, refutation-free deaths"""
    n = 2000
    pools = trio(hostemu_lib, capacity=n + 2, n_initial=n, seed=59)
    all3(pools, lambda p: p.crash_fraction(60000, 5))
    x = all3(pools, lambda p: p.member_add())
    all3(pools, lambda p: p.join(x, [0]))
    run(pools, 120, 10, "crash wave")
    t = all3(pools, lambda p: p.run_until(PRED_CRASHED_ALL_DEAD, 0, 6000, 50))
    assert t != NEVER
    check(pools, "all dead")
    run(pools, 200, 50, "gossip to the dead")
