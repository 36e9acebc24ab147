"""
gbm_series_sum's chunking (engine.gbm_sum_chunk_steps): a multiple of 32 steps, at most 2048 rows, and S rows
plus statistics workspace within chunk_bytes whatever N and H are.  CPU only (the sizes are host arithmetic).
"""
import pytest

from rlmd_b200 import _lib, engine


@pytest.mark.parametrize("n,g,h", [(300, 3, 70_000), (2000, 4, 10_000), (1, 1, 5), (4099, 11, 97),
                                   (1_000_000, 10, 500), (1_000_000, 64, 2000)])
def test_chunk_steps_are_capped(n, g, h):
    tc = engine.gbm_sum_chunk_steps(n, g, h)
    assert tc % 32 == 0 and 32 <= tc <= 2048
    assert tc <= -(-(h - 1) // 32) * 32 or tc == 32
    per_row = 8 * n + _lib.lib.b200_gbm_sum_stats_workspace_bytes(1, n, g)
    assert tc == 32 or tc * per_row <= 256 << 20
    assert _lib.lib.b200_gbm_sum_stats_workspace_bytes(tc, n, g) == tc * (per_row - 8 * n)
    # an explicit chunk is rounded down to 32 and capped the same way
    assert engine.gbm_sum_chunk_steps(n, g, h, chunk_steps=10 ** 6) == min(2048, -(-(h - 1) // 32) * 32)
    assert engine.gbm_sum_chunk_steps(n, g, h, chunk_steps=100) == min(96, max(32, -(-(h - 1) // 32) * 32))


def test_small_investor_count_long_horizon_stays_small():
    """N = 300, H = 7e4: 2048 rows (within the kernel's 65535 per call), workspace under 300 MB."""
    tc = engine.gbm_sum_chunk_steps(300, 3, 70_000)
    assert tc <= 2048
    assert _lib.lib.b200_gbm_sum_stats_workspace_bytes(tc, 300, 3) <= 300 << 20
