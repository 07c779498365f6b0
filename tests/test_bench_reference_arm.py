"""bench.py's CPU arm (`--impl reference`): same config object as the repo arm, oracle only —
the product library must not be mapped into that process (VERDICT r1, weak #12)."""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_oracle_presets_equal_libgsim_presets(hostemu_lib):
    """The oracle restates the LAN / WAN / test-harness defaults on its own; they must be the
    product's, field by field (both cite agent/config/runtime.go:1271-1413, server_test.go:221-237)."""
    from consul_b200 import _lib
    from oracle_binding import oracle_config
    for preset, fn in (("lan", "gsim_config_default_lan"), ("wan", "gsim_config_default_wan"),
                       ("consul_test", "gsim_config_consul_test")):
        a = oracle_config(preset)
        b = _lib.GsimConfig()
        getattr(hostemu_lib, fn)(C.byref(b))
        for name, _ in _lib.GsimConfig._fields_:
            assert getattr(a, name) == getattr(b, name), (preset, name)


def test_reference_arm_runs_without_the_product_library(tmp_path):
    env = dict(os.environ, OMP_NUM_THREADS="1", GSIM_REF_BUDGET_S="20")     # as under torchrun
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1", "--members", "30000", "--ticks", "160", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["native_so_loaded"] == ["oracle/liboracle.so"]
    assert line["config"]["ticks_per_step"] == 160 and line["config"]["members"] == 30000
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["value"] == line["value"] > 0
    # --dump-outputs: the state the last timed step left, the one the line's digest was taken from
    import numpy as np
    words = np.load(tmp_path / "state_hash.npy")
    assert words.dtype == np.float64 and words.shape == (8,)
    assert "%016x" % (int(words[0]) << 32 | int(words[1])) == line["digest"]
    members = np.load(tmp_path / "members.npy")
    assert members.shape == (30000 + 1 + 2, 4) and (members[:, 0] == np.arange(len(members))).all()
    assert np.load(tmp_path / "stats.npy").dtype == np.float64
    # the config object is produced by the one function the repo arm uses
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.workload_config(30000, 160, 1, False)


def test_sampled_step_scales_to_the_full_step():
    """A budget too small for the whole step still reports the time of the WHOLE step (cascade in
    full + steady ticks scaled), never a shorter step."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle_binding import OraclePool, oracle_config
    o = OraclePool(oracle_config("lan", capacity=20002, n_initial=20000, seed=7), threads=1)
    x = o.member_add()
    o.join(x, [0])
    secs, done = bench.oracle_step_sampled(o, 2048, budget_s=0.0)
    assert done == bench.CASCADE_TICKS + 64 and secs > 0
    o2 = OraclePool(oracle_config("lan", capacity=20002, n_initial=20000, seed=7), threads=1)
    x = o2.member_add()
    o2.join(x, [0])
    secs2, done2 = bench.oracle_step_sampled(o2, 2048, budget_s=1e9)
    assert done2 == 2048
    assert 0.3 < secs / secs2 < 3.0          # the scaled figure is the same order as the measured one
