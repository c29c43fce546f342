"""Per-unit timeline of one lidar launch (development aid; needs a GPU).

  python tools/unit_timeline.py [--envs 4096] [--steps 30] [--flush]

Steps the C3 workload with the lookup-counting variant of the lidar kernel, then reads back, for every 32-beam work unit
of the last launch, when it started and ended (%globaltimer), its longest ray and the SM / queue position it ran at, and
prints: kernel span, when the longest units ran, per-warp-slot busy time, and the makespan a perfect packing would reach."""
import argparse
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from f110_gymnasium_ros2_jazzy_b200 import F110VecEnv, _lib  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--flush', action='store_true')
    a = ap.parse_args()
    args = argparse.Namespace(map='Shanghai_map', map_upsample=1, agents=1, beams=1080, envs=a.envs)
    map_arrays, poses = bench.load_workload(args, a.envs, 0, a.envs)
    env = F110VecEnv(a.envs, num_agents=1, num_beams=1080, seed=42, device=0, auto_reset=True,
                     outputs=('obs', 'reward', 'terminated'), noise_std=0.01, count_lookups=True, map_arrays=map_arrays)
    env.reset(poses)
    acts = bench.action_stream(torch, a.steps, a.envs, 1, torch.device('cuda', 0))
    flush = torch.empty(2 * bench.L2_BYTES, dtype=torch.uint8, device='cuda') if a.flush else None
    for k in range(a.steps):
        if flush is not None:
            flush.fill_(k & 0xFF)
        env.step(acts[k])
    torch.cuda.synchronize()
    L = env.backend.lib
    n = int(L.f110_debug_unit_timeline(env.backend.h, None, 0))
    buf = np.zeros((n, 4), np.uint32)
    _lib.check(min(0, int(L.f110_debug_unit_timeline(env.backend.h, buf.ctypes.data_as(C.c_void_p), n))))
    t0 = buf[:, 0].astype(np.int64); t1 = buf[:, 1].astype(np.int64)
    base = t0.min()
    s, e = (t0 - base) / 1e3, (t1 - base) / 1e3        # us
    look, redo, sm, pos = buf[:, 2] & 0xFFFFFF, buf[:, 2] >> 24, buf[:, 3] >> 24, buf[:, 3] & 0xFFFFFF
    dur = e - s
    os.makedirs('gpurun_out', exist_ok=True)
    np.savez_compressed('gpurun_out/unit_timeline_%d.npz' % a.envs, start_us=s, end_us=e, lookups=look, sm=sm, pos=pos, redo=redo)
    print("units %d, kernel span (first unit start -> last unit end) %.1f us" % (n, e.max()))
    print("sum of unit durations %.0f us = %.1f us per warp slot over %d slots" % (dur.sum(), dur.sum() / (148 * 48), 148 * 48))
    order = np.argsort(-look.astype(np.int64))[:8]
    for u in order:
        print("  unit %7d pos %6d sm %3d lookups %4d  start %7.1f end %7.1f (%.1f us, %.0f ns/lookup)"
              % (u, pos[u], sm[u], look[u], s[u], e[u], dur[u], 1e3 * dur[u] / max(look[u], 1)))
    last = np.argsort(-e)[:8]
    print("last units to finish:")
    for u in last:
        print("  unit %7d pos %6d sm %3d lookups %4d  start %7.1f end %7.1f" % (u, pos[u], sm[u], look[u], s[u], e[u]))
    for q in (1, 10, 50):
        print("  units started by %.1f us: %d%%" % (np.percentile(s, q), q))
    for q in (50, 90, 99, 100):
        print("  units ended by %.1f us: %d%%" % (np.percentile(e, q), q))
    # light units: duration vs lookups
    for lo, hi in ((0, 4), (4, 8), (8, 16), (16, 24), (24, 48), (48, 96), (96, 1000)):
        sel = (look >= lo) & (look < hi)
        if sel.any():
            print("  lookups [%3d,%4d): %6d units, mean %.2f us (%.0f ns/lookup), start median %.1f us"
                  % (lo, hi, sel.sum(), dur[sel].mean(), 1e3 * dur[sel].sum() / max(look[sel].sum(), 1), np.median(s[sel])))
    r = redo > 0
    if r.any():
        print("units with rays redone in exact arithmetic: %d, mean %.2f us (%.0f ns/lookup) against %.2f us (%.0f ns/lookup) for the others below 24 lookups"
              % (r.sum(), dur[r].mean(), 1e3 * dur[r].sum() / look[r].sum(), dur[~r & (look < 24)].mean(),
                 1e3 * dur[~r & (look < 24)].sum() / look[~r & (look < 24)].sum()))
        print("  of the 50 units that finish last, %d had a redone ray" % int(r[np.argsort(-e)[:50]].sum()))
    per_sm = np.bincount(sm, weights=dur, minlength=148)
    print("per-SM busy warp-us: min %.0f mean %.0f max %.0f" % (per_sm.min(), per_sm.mean(), per_sm.max()))


if __name__ == '__main__':
    main()
