"""The fast gossip tier on the B200 (DESIGN.md §4.1): a 1 M-member join cascade and the benchmark's own
step sequence give the same digest and counters with the tier and without it (GSIM_FLAG_NO_FAST_GOSSIP),
and the same as the oracle."""
import pytest

from consul_b200.pool import FLAG_NO_FAST_GOSSIP, Pool, lan_config
from oracle_binding import OraclePool
from parity import compare_pools

pytestmark = pytest.mark.gpu


def test_cascade_1m_tier_on_off(cuda_lib):
    n = 1_000_000
    cfg = dict(capacity=n + 1, n_initial=n, seed=0x5EED0001)
    on, off = Pool(lan_config(cuda_lib, **cfg), cuda_lib), Pool(lan_config(cuda_lib, flags=FLAG_NO_FAST_GOSSIP, **cfg), cuda_lib)
    ora = OraclePool(lan_config(cuda_lib, **cfg))
    for p in (on, off, ora):
        x = p.member_add()
        assert p.join(x, [0]) == 1
    for k in range(12):
        for p in (on, off):
            p.step(8)
        compare_pools(on, off, f"cascade +{8 * (k + 1)}", columns=False)
    ora.step(96)
    compare_pools(on, ora, "cascade end (tier vs oracle)")
    assert on.stats()["rumors_accepted"] == 2 * n - 1


def test_bench_sequence_tier_on_off(cuda_lib):
    """bench.py's step: member_add + join + 2048 ticks, three times"""
    n = 1_000_000
    cfg = dict(capacity=n + 16, n_initial=n, seed=0x5EED0001)
    on, off = Pool(lan_config(cuda_lib, **cfg), cuda_lib), Pool(lan_config(cuda_lib, flags=FLAG_NO_FAST_GOSSIP, **cfg), cuda_lib)
    for s in range(3):
        for p in (on, off):
            x = p.member_add()
            p.join(x, [s])
            p.step(2048)
        compare_pools(on, off, f"bench step {s}", columns=False)
