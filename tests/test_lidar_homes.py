"""Home segments of the lidar kernel's scheduler (launches above 48 units per resident warp, or forced): every SM serves a
contiguous stretch of the units first and steals from the nearest other stretches once its own is drained.  Only the order in which units run may depend on the segments
(F110_LIDAR_HOMES=n forces n of them, include/f110_b200.h); scans, observations, flags and counts may not."""
import os

import numpy as np
import pytest

from tests import helpers as H

# default (one queue at these sizes), one queue forced, far more segments than SMs (most have no resident warp)
HOMES = (None, '1', '1000')


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _sim(homes, *args, **kw):
    from f110_gymnasium_ros2_jazzy_b200 import BatchSim
    old = os.environ.pop('F110_LIDAR_HOMES', None)
    if homes is not None:
        os.environ['F110_LIDAR_HOMES'] = homes
    try:
        return BatchSim(*args, **kw)
    finally:
        os.environ.pop('F110_LIDAR_HOMES', None)
        if old is not None:
            os.environ['F110_LIDAR_HOMES'] = old


@pytest.mark.gpu
@pytest.mark.parametrize('homes', HOMES)
@pytest.mark.parametrize('envs', [None, 8])
def test_scans_equal_the_reference(homes, envs):
    """Noise-free scans against the reference's own, bit for bit; envs = 8 is a grid of fewer CTAs than SMs
    (one queue by default, forced segments with no resident warp otherwise)."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS
    g = H.load('scans')
    poses, ref = g['Shanghai_map__poses'][:envs], g['Shanghai_map__scans'][:envs]
    sim = _sim(homes, len(poses), 1, outputs=ALL_OUTPUTS, noise_std=0.0)
    s, c = H.tables()[:2]
    sim.set_tables(s, c)
    sim.set_map_arrays(*H.golden_map('Shanghai_map'))
    for _ in range(3):      # the later launches run in the order the first one recorded
        sim.sim_reset(poses[:, None, :])
        out = sim.step(None, np.zeros((len(poses), 1, 1080)))
        torch.cuda.synchronize()
        assert np.array_equal(out['scans_f64'].cpu().numpy()[:, 0], ref)
    sim.close()


@pytest.mark.gpu
def test_rollout_does_not_depend_on_the_segments():
    """A 512-env rollout with device noise and auto-reset (K1 appends the units of reset cars to their segment's list):
    observations, flags and state equal across the segment counts at every step, and the lookup-counting variant counts
    every ray once per step."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, workloads
    dt, res, origin = H.golden_map('Shanghai_map')
    start = workloads.start_poses(512)
    rng = np.random.default_rng(11)
    acts = rng.uniform([-0.4189, 0.0], [0.4189, 12.0], size=(120, 512, 1, 2)).astype(np.float32)
    s, c = H.tables()[:2]
    runs = {}
    for homes in HOMES:
        for count in (False, True):
            sim = _sim(homes, 512, 1, outputs=ALL_OUTPUTS, noise_std=0.01, seed=5, count_lookups=count)
            sim.set_tables(s, c)
            sim.set_map_arrays(dt, res, origin)
            out = sim.reset(start)
            rays0 = sim.lookup_count()[1] if count else 0     # the reset's own launch
            mask, trace = None, []
            for t in range(120):
                out = sim.step(acts[t], reset_mask=mask, reset_poses=start) if mask is not None else sim.step(acts[t])
                torch.cuda.synchronize()
                mask = out['terminated'].clone()
                trace.append([out[k].cpu().numpy().copy() for k in ('obs', 'terminated', 'state', 'collisions')])
                if count:
                    assert sim.lookup_count()[1] - rays0 == (t + 1) * 512 * 1080
            sim.close()
            runs[(homes, count)] = trace
    base = runs[(None, False)]
    assert sum(int(tr[1].sum()) for tr in base) > 0             # episodes ended and restarted on the way
    for key, trace in runs.items():
        for a, b in zip(base, trace):
            for x, y in zip(a, b):
                assert np.array_equal(x, y), key


@pytest.mark.gpu
@pytest.mark.parametrize('homes', HOMES)
def test_every_timeline_entry_is_from_the_current_launch(homes):
    """The lookup-counting variant writes every unit's (start, end) each launch, whichever SM ran it."""
    torch = _torch()
    import ctypes as C
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, _lib, workloads
    n = 1024
    sim = _sim(homes, n, 1, outputs=ALL_OUTPUTS, noise_std=0.01, count_lookups=True)
    s, c = H.tables()[:2]
    sim.set_tables(s, c)
    sim.set_map_arrays(*H.golden_map('Shanghai_map'))
    sim.reset(workloads.start_poses(n))
    units = int(sim.lib.f110_debug_unit_timeline(sim.h, None, 0))
    assert units == n * 34
    prev_end = None
    for _ in range(4):
        sim.step(np.zeros((n, 1, 2), np.float32))
        torch.cuda.synchronize()
        buf = np.zeros((units, 4), np.uint32)
        _lib.check(min(0, int(sim.lib.f110_debug_unit_timeline(sim.h, buf.ctypes.data_as(C.c_void_p), units))))
        # %globaltimer_lo wraps every 4.3 s: times are compared as signed 32-bit differences
        if prev_end is not None:
            assert ((buf[:, 0] - prev_end).astype(np.int32) > 0).all()
        t0 = buf[0, 0]
        prev_end = np.uint32(t0 + np.uint32((buf[:, 1] - t0).astype(np.int32).max()))
    sim.close()


@pytest.mark.gpu
def test_default_segments_of_a_large_launch():
    """Above 48 units per resident warp every SM gets a home segment by default: observations, flags and state equal those
    of one shared queue, and every ray is counted once per step."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, workloads
    n = 12288
    start = workloads.start_poses(n)
    acts = np.random.default_rng(2).uniform([-0.4189, 0.0], [0.4189, 12.0], size=(6, n, 1, 2)).astype(np.float32)
    s, c = H.tables()[:2]
    runs = []
    for homes in (None, '1'):
        sim = _sim(homes, n, 1, outputs=ALL_OUTPUTS, noise_std=0.01, seed=9, count_lookups=True)
        sim.set_tables(s, c)
        sim.set_map_arrays(*H.golden_map('Shanghai_map'))
        sim.reset(start)
        rays0 = sim.lookup_count()[1]
        trace = []
        for t in range(6):
            out = sim.step(acts[t])
            torch.cuda.synchronize()
            trace.append([out[k].cpu().numpy().copy() for k in ('obs', 'terminated', 'state')])
            assert sim.lookup_count()[1] - rays0 == (t + 1) * n * 1080
        sim.close()
        runs.append(trace)
    for a, b in zip(*runs):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
