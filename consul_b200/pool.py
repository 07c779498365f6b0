"""Pool — one simulated gossip pool (LAN or WAN) of virtual members on one B200.

Thin object wrapper over the C ABI; all simulation state lives in HBM behind libgsim.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import (COLUMNS, GSIM_MAX_RUMORS, GSIM_MAX_SUSPICION_SLOTS, STAT_NAMES, GsimConfig,
                   GsimEvent, GsimMember, GsimMemberDesc, GsimRumorInfo, GsimStats)

PRED_RUMOR_CONVERGED = 1
PRED_ALL_RUMORS_CONVERGED = 2
PRED_CRASHED_ALL_DEAD = 3
NEVER = 0xFFFFFFFF

FLAG_LOG_GLOBAL_EVENTS = 1
FLAG_NO_GRAPH = 2
FLAG_NO_WINDOWS = 16
FLAG_PUSH_PULL = 32
FLAG_COORDINATES = 64
FLAG_NO_FAST_GOSSIP = 256
MEMBER_WATCHED = 1


class GsimError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"gsim error {code}: {msg}")
        self.code = code


def lan_config(lib=None, **kw) -> GsimConfig:
    lib = lib or _lib.lib()
    c = GsimConfig()
    lib.gsim_config_default_lan(C.byref(c))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def wan_config(lib=None, **kw) -> GsimConfig:
    lib = lib or _lib.lib()
    c = GsimConfig()
    lib.gsim_config_default_wan(C.byref(c))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def consul_test_config(lib=None, **kw) -> GsimConfig:
    lib = lib or _lib.lib()
    c = GsimConfig()
    lib.gsim_config_consul_test(C.byref(c))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


@dataclass
class Event:
    tick: int
    type: int
    subject: int
    observer: int
    ltime: int


class Pool:
    def __init__(self, cfg: GsimConfig, lib=None):
        self.lib = lib or _lib.lib()
        self.cfg = cfg
        h = C.c_void_p()
        rc = self.lib.gsim_pool_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise GsimError(rc, self.lib.gsim_strerror(rc).decode())
        self.h = h
        self.capacity = cfg.capacity

    # -- lifecycle -----------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self.lib.gsim_pool_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc: int):
        if rc != 0:
            msg = self.lib.gsim_last_error(self.h).decode() or self.lib.gsim_strerror(rc).decode()
            raise GsimError(rc, msg)

    # -- membership operations --------------------------------------------------
    def member_add(self, alive_msg_size: int = 0, watched: bool = False, name_len: int = 0, meta_len: int = 0) -> int:
        d = GsimMemberDesc(alive_msg_size, MEMBER_WATCHED if watched else 0, name_len, meta_len)
        out = C.c_uint32()
        self._ck(self.lib.gsim_member_add(self.h, C.byref(d), C.byref(out)))
        return out.value

    def join(self, member: int, seeds, ignore_old: bool = True) -> int:
        arr = (C.c_uint32 * len(seeds))(*seeds)
        n_ok = C.c_int()
        self._ck(self.lib.gsim_join(self.h, member, arr, len(seeds), int(ignore_old), C.byref(n_ok)))
        return n_ok.value

    def leave(self, member: int):
        self._ck(self.lib.gsim_leave(self.h, member))

    def crash(self, member: int):
        self._ck(self.lib.gsim_crash(self.h, member))

    def crash_many(self, ids):
        arr = (C.c_uint32 * len(ids))(*ids)
        self._ck(self.lib.gsim_crash_many(self.h, arr, len(ids)))

    def crash_fraction(self, ppm: int, salt: int = 0) -> int:
        out = C.c_uint32()
        self._ck(self.lib.gsim_crash_fraction(self.h, ppm, salt, C.byref(out)))
        return out.value

    def force_leave(self, via: int, target: int, prune: bool = False):
        self._ck(self.lib.gsim_force_leave(self.h, via, target, int(prune)))

    def user_event(self, member: int, name: bytes, payload: bytes, coalesce: bool = False) -> int:
        out = C.c_uint32()
        self._ck(self.lib.gsim_user_event(self.h, member, name, len(name), payload, len(payload),
                                          int(coalesce), C.byref(out)))
        return out.value

    def rumor_inject(self, slot: int, member: int) -> bool:
        """Out-of-band delivery of tracked broadcast `slot` to `member` (WAN bridges)."""
        out = C.c_int()
        self._ck(self.lib.gsim_rumor_inject(self.h, slot, member, C.byref(out)))
        return bool(out.value)

    def member_watch(self, member: int, on: bool = True):
        self._ck(self.lib.gsim_member_watch(self.h, member, int(on)))

    def member_update(self, member: int, alive_msg_size: int = 0) -> int:
        """(*Serf).SetTags: re-announce under the next incarnation; returns the rumor slot."""
        out = C.c_uint32()
        self._ck(self.lib.gsim_member_update(self.h, member, alive_msg_size, C.byref(out)))
        return out.value

    def graph_set(self, row_ptr, col_idx):
        """CSR peer graph: member i's memberlist = col_idx[row_ptr[i]:row_ptr[i+1]]; None removes it."""
        if row_ptr is None:
            self._ck(self.lib.gsim_graph_set(self.h, 0, None, None))
            return
        rp = np.ascontiguousarray(row_ptr, dtype=np.uint32)
        ci = np.ascontiguousarray(col_idx, dtype=np.uint32)
        self._ck(self.lib.gsim_graph_set(self.h, len(rp) - 1, rp.ctypes.data_as(C.POINTER(C.c_uint32)),
                                         ci.ctypes.data_as(C.POINTER(C.c_uint32))))

    def member_reconnect_timeout_set(self, member: int, timeout_ns: int):
        """serf.Config.ReconnectTimeoutOverride result for one member (0 = the pool's value)."""
        self._ck(self.lib.gsim_member_reconnect_timeout_set(self.h, member, timeout_ns))

    def coordinate(self, member: int):
        """(*Serf).GetCoordinate: (vec[8], error, adjustment, height) in seconds."""
        out = (C.c_double * 11)()
        self._ck(self.lib.gsim_coordinate_get(self.h, member, out))
        v = [float(x) for x in out]
        return v[:8], v[8], v[9], v[10]

    def latency_set(self, lat):
        """lat: square matrix (n_dcs x n_dcs) of one-way latencies in ticks (>= 1), or None."""
        if lat is None:
            self._ck(self.lib.gsim_latency_set(self.h, 0, None))
            return
        m = np.ascontiguousarray(lat, dtype=np.uint8)
        assert m.ndim == 2 and m.shape[0] == m.shape[1]
        self._ck(self.lib.gsim_latency_set(self.h, m.shape[0], m.ctypes.data_as(C.POINTER(C.c_uint8))))

    # -- time ---------------------------------------------------------------------
    def step(self, ticks: int = 1):
        self._ck(self.lib.gsim_step(self.h, ticks))

    def run_until(self, predicate: int, arg: int = 0, max_ticks: int = 10000,
                  check_every: int = 16) -> int:
        out = C.c_uint32()
        self._ck(self.lib.gsim_run_until(self.h, predicate, arg, max_ticks, check_every,
                                         C.byref(out)))
        return out.value

    @property
    def now(self) -> int:
        return self.lib.gsim_now(self.h)

    # -- observation ------------------------------------------------------------------
    def members(self, observer: int):
        n = C.c_size_t()
        self._ck(self.lib.gsim_members(self.h, observer, None, 0, C.byref(n)))
        buf = (GsimMember * max(1, n.value))()
        self._ck(self.lib.gsim_members(self.h, observer, buf, n.value, C.byref(n)))
        return [(m.id, m.status, m.incarnation, m.rank) for m in buf[: n.value]]

    def num_nodes(self, observer: int) -> int:
        out = C.c_uint32()
        self._ck(self.lib.gsim_num_nodes(self.h, observer, C.byref(out)))
        return out.value

    def poll_events(self, cap: int = 65536):
        buf = (GsimEvent * cap)()
        n = C.c_size_t()
        self._ck(self.lib.gsim_poll_events(self.h, buf, cap, C.byref(n)))
        return [Event(e.tick, e.type, e.subject, e.observer, e.ltime) for e in buf[: n.value]]

    def rumor_info(self, slot: int) -> dict:
        out = GsimRumorInfo()
        self._ck(self.lib.gsim_rumor_info_get(self.h, slot, C.byref(out)))
        return {n: getattr(out, n) for n, _ in GsimRumorInfo._fields_}

    def rumor_retire(self, slot: int):
        self._ck(self.lib.gsim_rumor_retire(self.h, slot))

    def user_event_get(self, slot: int):
        nl, pl = C.c_size_t(), C.c_size_t()
        nb, pb = C.create_string_buffer(1024), C.create_string_buffer(1024)
        self._ck(self.lib.gsim_user_event_get(self.h, slot, nb, 1024, C.byref(nl), pb, 1024,
                                              C.byref(pl)))
        return nb.raw[: nl.value], pb.raw[: pl.value]

    def stats(self) -> dict:
        s = GsimStats()
        self._ck(self.lib.gsim_stats_get(self.h, C.byref(s)))
        out = {n: int(s.counters[i]) for i, n in enumerate(STAT_NAMES)}
        for n, _ in GsimStats._fields_:
            if n == "counters":
                continue
            v = getattr(s, n)
            out[n] = list(v) if n == "suspicion_ticks" else int(v)
        return out

    def state_hash(self):
        out = (C.c_uint64 * 4)()
        self._ck(self.lib.gsim_state_hash(self.h, out))
        return tuple(int(x) for x in out)

    def column(self, name: str) -> np.ndarray:
        cap = self.capacity
        if name == "tx":
            arr = np.zeros((GSIM_MAX_RUMORS, cap), dtype=np.uint8)
        elif name == "sus_from":
            arr = np.zeros((GSIM_MAX_SUSPICION_SLOTS, cap), dtype=np.uint32)
        else:
            arr = np.zeros(cap, dtype=np.uint32)
        n = C.c_size_t()
        self._ck(self.lib.gsim_column_read(self.h, COLUMNS[name], arr.ctypes.data_as(C.c_void_p),
                                           arr.nbytes, C.byref(n)))
        return arr

    # -- checkpoint -----------------------------------------------------------------------
    def snapshot(self) -> bytes:
        n = C.c_size_t()
        self._ck(self.lib.gsim_snapshot_size(self.h, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        self._ck(self.lib.gsim_snapshot(self.h, buf, n.value, C.byref(n)))
        return buf.raw[: n.value]

    def restore(self, blob: bytes):
        self._ck(self.lib.gsim_restore(self.h, blob, len(blob)))

    # -- measurement ----------------------------------------------------------------------
    def last_step_timing(self):
        ms = C.c_double()
        n = C.c_uint64()
        self._ck(self.lib.gsim_last_step_timing(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def sched_counts(self) -> dict:
        out = (C.c_uint64 * 8)()
        self._ck(self.lib.gsim_sched_counts(self.h, out))
        return {"window_launches": int(out[0]), "window_ticks": int(out[1]), "tick_launches": int(out[2]),
                "horizon_scans": int(out[3]), "window_ms": out[4] / 1e6, "tick_ms": out[5] / 1e6,
                "closed_form_launches": int(out[6]), "closed_form_ticks": int(out[7])}

    def launch_count(self) -> int:
        return int(self.lib.gsim_launch_count(self.h))
