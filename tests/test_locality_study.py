"""tools/locality_study.py (the per-SM L1 model of the lidar kernel's schedules) at a tiny size, on the CPU."""
import os
import sys

import pytest


def test_locality_study_tiny():
    """Every schedule replays the same warp-lookups, the rates are rates, and home segments bring fewer lines into the
    SMs than the global queue."""
    pytest.importorskip('numba')
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tools'))
    import locality_study
    r = locality_study.main(['--envs', '32', '--sms', '4', '--warps', '8', '--homes', '4'])
    g, h = r['schedules']['global'], r['schedules']['homes_4']
    assert r['units'] == 32 * 34
    assert g['warp_lookups'] == h['warp_lookups'] == r['warp_lookups']
    for v in (g, h):
        assert 0.0 <= v['warp_lookups_all_hit_share'] <= 1.0 and 0.0 <= v['sector_hit_rate'] <= 1.0
    assert h['line_fills'] < g['line_fills']
