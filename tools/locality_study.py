"""L1 locality of the lidar kernel's schedule, replayed on the CPU (analysis, not product): how many of a launch's map
lookups an SM's L1 could serve when the SMs take units from one device-wide queue, against when every SM has a home
stretch of contiguous scans.

The march is the reference's (tools/tile_study.py, laser_models.py:106-146) on the C3 start poses; each lookup is placed in
the device's padded map (cell (r, c) at [r + 1][c + 1] of prows x pitch fp64 cells, MapView), so a 128-byte line is 16
cells of one row and a 32-byte sector 4.  A unit is 32 consecutive beams of one scan, a warp-lookup the lookups its live
lanes issue together at one step of the march.  Per SM the model runs `--warps` resident warps round robin, one
warp-lookup each per turn, every warp taking the SM's next unit when its own is done, against a fully associative LRU L1
of `--l1-kb` with sectored fills (a miss fills the missing sectors only; a line is allocated on its first sector).
Compulsory and capacity misses only: no other work shares the L1, and the stealing at the end of a homed launch is not
modelled.

Schedules:
  * global: the queue order of today's kernel (the heavy units first, longest class first, then the light ones in natural
    order) cut into chunks of `--chunk` units, each chunk going to the SM of a random warp (fetch order is a race);
  * homes Q: the scans cut into Q contiguous segments, SM k serving segment k * Q // SMs (the SMs that share a segment take
    its chunks in random turns); inside a segment heavy units first, then light, as in the global queue.

Reported per schedule: line fills and sector hit rate (sum and per-SM mean / max), and the share of warp-lookups whose
lanes all hit L1 -- the ones that do not wait for an L2 round trip.

  python tools/locality_study.py [--envs 4096] [--homes 37,74,148,296] [--out profiles/r03_locality_study.json]
"""
import argparse
import json
import os
import sys

import numpy as np
from numba import njit

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from f110_gymnasium_ros2_jazzy_b200 import workloads   # noqa: E402

HEAVY_T = (96, 48, 24)   # the lidar kernel's class thresholds (HEAVY_T0..2)


@njit(cache=False)
def march(poses, dt, res, ox, oy, sines, cosines, B, inc, fov, cap, ray_len, cell):
    """The reference march; -> lookups recorded.  ray_len[ray] = lookups of ray p * B + i, cell[k] = (row, col) of lookup
    k, rays in order."""
    H_, W_ = dt.shape
    k = 0
    for p in range(poses.shape[0]):
        ti = 2000 * (poses[p, 2] - fov / 2.) / (2. * np.pi)
        ti = np.fmod(ti, 2000.)
        while ti < 0:
            ti += 2000
        for i in range(B):
            s = sines[int(ti)]
            c = cosines[int(ti)]
            x = poses[p, 0]
            y = poses[p, 1]
            total = 0.0
            n = 0
            while True:
                xr = x - ox
                yr = y - oy
                if xr < 0 or xr >= W_ * res or yr < 0 or yr >= H_ * res:
                    r_, c_ = H_ - 1, W_ - 1
                else:
                    r_, c_ = int(yr / res), int(xr / res)
                d = dt[r_, c_]
                if k < cap:
                    cell[k, 0] = r_
                    cell[k, 1] = c_
                k += 1
                n += 1
                total += d
                if not (d > 1e-4 and total <= 30.0):
                    break
                x += d * c
                y += d * s
            ray_len[p * B + i] = n
            ti += inc
            while ti >= 2000:
                ti -= 2000
    return k


def padded_geometry(H, W):
    """(prows, pitch) of the device's padded map (f110_capi.cu set_map): fx_bits = 32 - bit_length(max(W, H) + 1)."""
    fx_bits = 32 - (max(W, H) + 1).bit_length()
    prows = 1 << (32 - fx_bits)
    return prows, prows + 16


@njit(cache=False)
def simulate_sm(units, unit_off, wl_off, wl_sec, warps, cap_lines, prev, nxt, present, stat):
    """One SM: `units` in the order the SM takes them, `warps` resident warps round robin.  Unit u's warp-lookups are
    unit_off[u] .. unit_off[u + 1]; warp-lookup w's sectors (line << 2 | sector, deduplicated) are wl_sec[wl_off[w] ..
    wl_off[w + 1]].  prev / nxt / present: LRU list over line ids (all -1 / 0 on entry, restored on exit).
    stat += (warp-lookups, of them all-hit, sector requests, sector hits, line fills)."""
    head = -1
    tail = -1
    size = 0
    slot_unit = np.full(warps, -1, np.int64)
    slot_wl = np.zeros(warps, np.int64)
    nxt_unit = 0
    active = 0
    for w in range(warps):
        if nxt_unit < units.size:
            slot_unit[w] = units[nxt_unit]
            slot_wl[w] = unit_off[units[nxt_unit]]
            nxt_unit += 1
            active += 1
    touched = []
    while active > 0:
        for w in range(warps):
            u = slot_unit[w]
            if u < 0:
                continue
            if slot_wl[w] >= unit_off[u + 1]:
                if nxt_unit < units.size:
                    u = units[nxt_unit]
                    nxt_unit += 1
                    slot_unit[w] = u
                    slot_wl[w] = unit_off[u]
                else:
                    slot_unit[w] = -1
                    active -= 1
                    continue
                if slot_wl[w] >= unit_off[u + 1]:
                    continue
            wl = slot_wl[w]
            slot_wl[w] += 1
            all_hit = True
            for q in range(wl_off[wl], wl_off[wl + 1]):
                code = wl_sec[q]
                line = code >> 2
                bit = np.uint8(1 << (code & 3))
                stat[2] += 1
                if present[line] != 0:
                    if present[line] & bit:
                        stat[3] += 1
                    else:
                        all_hit = False
                        present[line] |= bit
                    # move to front
                    if head != line:
                        p = prev[line]
                        n = nxt[line]
                        if p >= 0:
                            nxt[p] = n
                        if n >= 0:
                            prev[n] = p
                        if tail == line:
                            tail = p
                        prev[line] = -1
                        nxt[line] = head
                        if head >= 0:
                            prev[head] = line
                        head = line
                else:
                    all_hit = False
                    stat[4] += 1
                    if size == cap_lines:
                        ev = tail
                        tail = prev[ev]
                        if tail >= 0:
                            nxt[tail] = -1
                        else:
                            head = -1
                        present[ev] = 0
                        prev[ev] = -1
                        nxt[ev] = -1
                        size -= 1
                    present[line] = bit
                    touched.append(line)
                    prev[line] = -1
                    nxt[line] = head
                    if head >= 0:
                        prev[head] = line
                    head = line
                    if tail < 0:
                        tail = line
                    size += 1
            stat[0] += 1
            if all_hit:
                stat[1] += 1
    for line in touched:
        present[line] = 0
        prev[line] = -1
        nxt[line] = -1


def build_trace(envs, B=1080):
    dt, res, origin = workloads.shanghai_map(1)
    poses = workloads.start_poses(envs)[:, 0]
    th = np.linspace(0, 2 * np.pi, 2000, endpoint=False)    # laser_models.py:379-381 uses theta_dis = 2000
    fov = 4.7
    inc = 2000 * (fov / (B - 1)) / (2 * np.pi)
    cap = int(envs * B * 12)
    ray_len = np.zeros(envs * B, np.int64)
    cell = np.zeros((cap, 2), np.int32)
    n = march(poses, dt, res, origin[0], origin[1], np.sin(th), np.cos(th), B, inc, fov, cap, ray_len, cell)
    assert n <= cap, (n, cap)
    cell = cell[:n]
    prows, pitch = padded_geometry(*dt.shape)
    # lookup -> (unit, step of its ray, lane)
    ray = np.repeat(np.arange(envs * B, dtype=np.int64), ray_len)
    starts = np.concatenate(([0], np.cumsum(ray_len)[:-1]))
    step = np.arange(n, dtype=np.int64) - np.repeat(starts, ray_len)
    ups = -(-B // 32)
    env, beam = ray // B, ray % B
    unit = env * ups + beam // 32
    lines = (cell[:, 0].astype(np.int64) + 1) * (pitch // 16) + (cell[:, 1].astype(np.int64) + 1) // 16
    sector = ((cell[:, 1].astype(np.int64) + 1) // 4) & 3
    # warp-lookups: (unit, step); the sectors one warp-lookup requests, deduplicated
    wl_key = unit * 4096 + step
    code = lines * 4 + sector
    order = np.lexsort((code, wl_key))
    wl_key, code = wl_key[order], code[order]
    keep = np.ones(n, bool)
    keep[1:] = (wl_key[1:] != wl_key[:-1]) | (code[1:] != code[:-1])
    wl_key, code = wl_key[keep], code[keep]
    new_wl = np.ones(wl_key.size, bool)
    new_wl[1:] = wl_key[1:] != wl_key[:-1]
    wl_off = np.concatenate((np.flatnonzero(new_wl), [wl_key.size])).astype(np.int64)
    wl_unit = wl_key[new_wl] // 4096
    num_units = envs * ups
    unit_off = np.searchsorted(wl_unit, np.arange(num_units + 1)).astype(np.int64)
    # unit classes as the kernel records them: the longest ray of the unit, spread to its two neighbours in the scan
    lane_len = np.zeros(num_units * 32, np.int64)
    rays = np.arange(envs * B)
    lane_len[(rays // B * ups + rays % B // 32) * 32 + rays % B % 32] = ray_len
    wmax = lane_len.reshape(num_units, 32).max(1)
    own = np.where(wmax >= HEAVY_T[0], 0, np.where(wmax >= HEAVY_T[1], 1, np.where(wmax >= HEAVY_T[2], 2, 3)))
    cls = own.copy()
    k = np.arange(num_units) % ups
    left = np.where(k > 0, np.roll(own, 1), 3)
    right = np.where(k + 1 < ups, np.roll(own, -1), 3)
    cls = np.minimum(cls, np.minimum(left, right))
    meta = {'envs': envs, 'beams': B, 'lookups': int(n), 'lookups_per_ray': n / (envs * B), 'units': int(num_units),
            'warp_lookups': int(wl_off.size - 1), 'sector_requests': int(code.size),
            'heavy_units': int((cls < 3).sum()), 'padded_map': [prows, pitch]}
    return dict(meta=meta, cls=cls, unit_off=unit_off, wl_off=wl_off, wl_sec=code, lines_total=prows * pitch // 16)


def longest_first(units, cls):
    """Heavy units first (class 0, 1, 2), then the light ones, each in natural order."""
    return units[np.argsort(cls[units], kind='stable')]


def schedule_global(num_units, cls, sms, chunk, rng):
    q = longest_first(np.arange(num_units), cls)
    chunks = np.array_split(q, -(-q.size // chunk))
    owner = rng.integers(0, sms, len(chunks))
    return [np.concatenate([c for c, o in zip(chunks, owner) if o == k] or [np.zeros(0, np.int64)]) for k in range(sms)]


def schedule_homes(num_units, ups, cls, sms, homes, chunk, rng):
    scans = num_units // ups
    seg_of_scan = (np.arange(scans) * homes) // scans          # contiguous, sizes differ by at most one scan
    seg_of_unit = np.repeat(seg_of_scan, ups)
    home_of_sm = (np.arange(sms) * homes) // sms if homes <= sms else None
    out = [[] for _ in range(sms)]
    for g in range(homes):
        q = longest_first(np.flatnonzero(seg_of_unit == g), cls)
        if homes <= sms:
            owners = np.flatnonzero(home_of_sm == g)
            chunks = np.array_split(q, max(1, -(-q.size // chunk)))
            pick = owners[rng.integers(0, owners.size, len(chunks))]
            for c, o in zip(chunks, pick):
                out[o].append(c)
        else:   # several homes per SM, served one after the other
            out[g * sms // homes].append(q)
    return [np.concatenate(o) if o else np.zeros(0, np.int64) for o in out]


def evaluate(trace, per_sm, warps, l1_kb):
    cap_lines = l1_kb * 1024 // 128
    L = trace['lines_total']
    prev = np.full(L, -1, np.int64)
    nxt = np.full(L, -1, np.int64)
    present = np.zeros(L, np.uint8)
    rows = []
    for units in per_sm:
        stat = np.zeros(5, np.int64)
        simulate_sm(units.astype(np.int64), trace['unit_off'], trace['wl_off'], trace['wl_sec'], warps, cap_lines,
                    prev, nxt, present, stat)
        rows.append(stat)
    s = np.array(rows)
    tot = s.sum(0)
    sec_hit = s[:, 3] / np.maximum(s[:, 2], 1)
    return {'warp_lookups': int(tot[0]), 'warp_lookups_all_hit_share': float(tot[1] / tot[0]),
            'sector_hit_rate': float(tot[3] / tot[2]), 'line_fills': int(tot[4]),
            'line_fills_per_sm_mean': float(s[:, 4].mean()), 'line_fills_per_sm_max': int(s[:, 4].max()),
            'sector_hit_rate_per_sm_min': float(sec_hit.min()), 'sector_hit_rate_per_sm_max': float(sec_hit.max()),
            'units_per_sm_min': int(min(u.size for u in per_sm)), 'units_per_sm_max': int(max(u.size for u in per_sm))}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--envs', type=int, default=4096)
    ap.add_argument('--beams', type=int, default=1080)
    ap.add_argument('--sms', type=int, default=148)
    ap.add_argument('--warps', type=int, default=48, help='resident warps per SM (12 CTAs of 4 warps)')
    ap.add_argument('--chunk', type=int, default=4, help='units per fetch (LIDAR_CHUNK)')
    ap.add_argument('--l1-kb', type=int, default=224)
    ap.add_argument('--homes', default='37,74,148,296')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--out', default=None)
    a = ap.parse_args(argv)
    trace = build_trace(a.envs, a.beams)
    ups = -(-a.beams // 32)
    num_units = trace['meta']['units']
    res = {'what': 'tools/locality_study.py: per-SM LRU model of L1 over the exact lidar march on the C3 start poses '
                   '(Shanghai, %d beams)' % a.beams,
           'model': {'sms': a.sms, 'warps_per_sm': a.warps, 'chunk': a.chunk, 'l1_kb': a.l1_kb, 'seed': a.seed},
           **trace['meta'], 'schedules': {}}
    rng = np.random.default_rng(a.seed)
    res['schedules']['global'] = evaluate(trace, schedule_global(num_units, trace['cls'], a.sms, a.chunk, rng),
                                          a.warps, a.l1_kb)
    for q in [int(v) for v in a.homes.split(',') if v]:
        res['schedules']['homes_%d' % q] = evaluate(
            trace, schedule_homes(num_units, ups, trace['cls'], a.sms, q, a.chunk, rng), a.warps, a.l1_kb)
    print(json.dumps(res, indent=1), flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)
    return res


if __name__ == '__main__':
    main()
