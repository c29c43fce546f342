"""The post kernel (K3: post_kernel, post_single_kernel in f110_kernels.cu) held to the oracle beam for beam.

Rollouts compared with the oracle's rollouts drift apart by about 1e-15 per step, which forces a loose lidar tolerance
(0.1 % of beams may be off); that allowance is about the size of the errors K3 can make (an off-by-one at the edge of a
ray-cast window is two beams in two thousand).  So these tests do not compare trajectories.  At every step of a GPU rollout
they recompute what K3 must have produced from that step's own GPU outputs, with the oracle's primitives:

* the wall scan is oracle.scan(agent pose) + the injected noise -- on an axis-aligned map origin the lidar kernel's march
  is the oracle's bit for bit -- and the expected scan is that, lowered by ray_cast for each opponent from the ray-cast
  origin (x, y, state yaw): the yaw the iTTC zeroed for a stopped car (base_classes.py:225), the opponents' vertices from
  their poses before the zeroing and the observing car's own length and width (:223);
* GJK with the construction-time length and width (:562), the iTTC against the wall scan (a stopped car's speed before the
  zeroing comes from a twin handle whose iTTC threshold is 0), _check_done (f110_env.py:320-348) in numpy, the pose slots of
  the observation and the episode counters.

Beams no opponent lowers must be bit-identical, flags exact.  A lowered beam ends on a ray / edge intersection formed
from vertices and beam directions that come from CUDA's sincos on the GPU and from libm in the oracle, an ulp apart; it
must lie within 4 units of (an ulp of the range + an ulp of the coordinates the vertices are formed in) / the sine of the
angle at which the beam meets the edge.  Four ulp of the range alone, the budget of test_lidar_variants.py, holds only near
the world origin: 60 m from it an ulp of a vertex is 7e-15 m, 60 ulp of a 0.5 m range.  Two things are exempt, counted and printed, and their counts bounded: a GJK pair
whose separation is below 1e-9 m, and a window edge whose vertex angle is within 1e-12 rad of the midpoint between two beams
(the kernel's atan2 shortcut, stage B).  Then constructed geometries at reset steps, where poses are exact and every path
of the ray-cast can be reached on purpose, and the lap bookkeeping and episode counters at the finish-zone edges.
"""
import math

import numpy as np
import pytest

from tests import helpers as H
from tests.test_post_cone_model import (collinear_geometries, kernel_vertex_angles, near_tie, reference_vertex_angles,
                                        vertices, window, wrap_yaw)

pytestmark = pytest.mark.gpu

EPISODES, EPISODE_STEPS, EGO_COLLISIONS, LAPS_DONE, EPISODE_TIME = range(5)   # F110_STAT_* (include/f110_b200.h)
DT = 0.01
LM = np.float32(30.0)


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _post_envs_per_cta(A):
    """post_envs_per_cta (f110_kernels.cu) with 128 threads and the cap of 16."""
    by_items, by_segs = 256 // (11 * A * (A - 1)) if A > 1 else 16, 16 // A
    return max(1, min(by_items, by_segs, 16))


def obs_lidar(x):
    """_pack_flat_obs's lidar channel (f110_env.py:552-584): float32 clip to [0, lidar_max], divided by lidar_max."""
    r = np.asarray(x).astype(np.float32)
    r = np.where(np.isnan(r), LM, r)
    return (np.clip(r, np.float32(0), LM) / LM).astype(np.float32)


def separation(v1, v2):
    """Signed separation of two rectangles along their best edge normal (> 0 apart, < 0 overlapping)."""
    best = -np.inf
    for poly in (v1, v2):
        for k in range(2):
            e = poly[k + 1] - poly[k]
            n = np.array([-e[1], e[0]]) / np.hypot(*e)
            p1, p2 = v1 @ n, v2 @ n
            best = max(best, p2.min() - p1.max(), p1.min() - p2.max())
    return best


def _oracle(B, fov, m, A=1, N=1):
    from oracle.f110_oracle import Oracle
    o = Oracle(N, A, num_beams=B, fov=fov)
    o.set_map_arrays(*m)
    return o


def _sim(N, A, B, fov, m, outputs=None, **kw):
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    sim = BatchSim(N, A, outputs=outputs or ALL_OUTPUTS, noise_std=0.0, num_beams=B, fov=fov, **kw)
    if isinstance(m, list):
        sim.set_maps(m)
    else:
        sim.set_map_arrays(*m)
    return sim


def _np(sim):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in sim.out.items()}


class Replay(object):
    """What K3 must have written, recomputed per step from the GPU's own agent poses and state."""

    def __init__(self, N, A, B, fov, oracles, lengths, widths, ego=0, sim_lw=(0.58, 0.31)):
        self.N, self.A, self.B, self.fov, self.ego = N, A, B, fov, ego
        self.oracles, self.L, self.W, self.sim_lw = oracles, lengths, widths, sim_lw
        self.angles = list(oracles[0].get_beam_tables()[0])
        self.start = np.zeros((N, A, 3))
        self.near = np.ones((N, A), bool)
        self.tog = np.zeros((N, A), np.int64)
        self.lap_times = np.zeros((N, A))
        self.time = np.zeros(N)
        self.steps = np.zeros(N, np.int64)
        self.stats = np.zeros(5)
        self.c = dict(beams=0, lowered=0, max_err=0.0, gjk=0, ittc=0, laps=0, gjk_exempt=0, tie_exempt=0, tie_pairs=0)

    def reset(self, e, poses):
        self.start[e] = poses
        self.near[e] = True
        self.tog[e] = 0
        self.time[e] = 0.0
        self.steps[e] = -1

    def check(self, e, g, slot=0, noise=None, twin_v=None, f64=True, where=''):
        """g: the step's outputs (numpy); noise [A, B] or None; twin_v [A]: speeds of the zero-threshold twin."""
        A, B, o = self.A, self.B, self.oracles[slot]
        poses, st = g['agent_poses'][e], g['state'][e]
        tag = (where, e)
        assert np.array_equal(poses[:, :2], st[:, :2]), tag
        hit = np.all(st[:, 3:] == 0, axis=1)
        origin = np.stack([st[:, 0], st[:, 1], st[:, 4]], 1)
        assert np.array_equal(origin[~hit, 2], poses[~hit, 2]), tag
        wall = np.stack([o.scan(poses[a])[0] for a in range(A)])
        if noise is not None:
            wall = wall + noise
        # iTTC (base_classes.py:243-252) on the wall scan
        for a in range(A):
            if hit[a]:
                assert twin_v is not None and o.check_ttc(wall[a], twin_v[a]), (tag, a, 'zeroed without an iTTC hit')
            else:
                assert not o.check_ttc(wall[a], st[a, 3]), (tag, a, 'iTTC hit not applied')
                assert twin_v is None or twin_v[a] == st[a, 3], (tag, a)
        self.c['ittc'] += int(hit.sum())
        # opponent ray-cast
        exp = wall.copy()
        edges = [set() for _ in range(A)]
        for a in range(A):
            for b in range(A):
                if b == a:
                    continue
                vb = o.get_vertices(poses[b], self.L[a], self.W[a])
                exp[a] = o.ray_cast(origin[a], exp[a], vb)
                verts = vertices(poses[b], self.L[a], self.W[a])
                ra, ka = reference_vertex_angles(origin[a], verts), kernel_vertex_angles(origin[a], verts)
                if any(near_tie(self.angles, x) for x in ra + ka):
                    self.c['tie_pairs'] += 1
                    edges[a] |= set(window(self.angles, ra)) | set(window(self.angles, ka))
        lowered = exp.view(np.int64) != wall.view(np.int64)
        tol = [self._tolerance(o, origin[a], poses, a, exp[a], lowered[a]) for a in range(A)]
        for a in range(A):
            got32 = g['scans_f32'][e, a]
            if f64:
                got = g['scans_f64'][e, a]
                bad_u = ~lowered[a] & (got.view(np.int64) != wall[a].view(np.int64))
                err = np.abs(got - exp[a])
                bad_l = lowered[a] & ~(err <= 4 * tol[a])
                if lowered[a].any():
                    self.c['max_err'] = max(self.c['max_err'], float((err / tol[a])[lowered[a]].max()))
            else:
                bad_u = bad_l = np.zeros(B, bool)
            want32 = exp[a].astype(np.float32)
            bad_u |= ~lowered[a] & (got32.view(np.int32) != wall[a].astype(np.float32).view(np.int32))
            bad_l |= lowered[a] & ~(np.abs(got32 - want32) <= np.spacing(want32))
            if a == 0 and 'obs' in g:
                ob, wo = g['obs'][e, :B], obs_lidar(exp[a])
                bad_u |= ~lowered[a] & (ob.view(np.int32) != obs_lidar(wall[a]).view(np.int32))
                bad_l |= lowered[a] & ~(np.abs(ob - wo) <= np.spacing(wo))
            bad = np.flatnonzero(bad_u | bad_l)
            ex = [i for i in bad if i in edges[a]]
            self.c['tie_exempt'] += len(ex)
            assert len(ex) == len(bad), (tag, a, 'beams differ', [i for i in bad if i not in edges[a]][:8],
                                         'lowered' if bad_l.any() else 'not lowered')
            self.c['lowered'] += int(lowered[a].sum())
        self.c['beams'] += A * B
        # GJK (Simulator.check_collision, base_classes.py:549-563) with the construction-time length / width
        coll = g['collisions'][e].astype(bool)
        if A > 1:
            sv = np.stack([o.get_vertices(poses[a], *self.sim_lw) for a in range(A)])
            gjk = o.collision_multiple(sv)[0] != 0
            self.c['gjk'] += int(gjk.sum())
            for a in np.flatnonzero((gjk | hit) != coll):
                assert any(abs(separation(sv[a], sv[b])) < 1e-9 for b in range(A) if b != a), (tag, a, 'collision flag')
                self.c['gjk_exempt'] += 1
        else:
            assert np.array_equal(coll, hit), tag
        # _check_done (f110_env.py:320-348) on the GPU's positions
        self.time[e] = self.time[e] + DT
        self.steps[e] += 1
        th = -self.start[e, self.ego, 2]
        rc, rs = math.cos(th), math.sin(th)
        for a in range(A):
            dx, dy = st[a, 0] - self.start[e, a, 0], st[a, 1] - self.start[e, a, 1]
            lx, ty = rc * dx + (-rs) * dy, rs * dx + rc * dy
            ty = ty - 2 if ty > 2 else (-2 - ty if ty < -2 else 0.0)
            closes = lx * lx + ty * ty <= 0.1
            if closes != self.near[e, a]:
                self.near[e, a] = closes
                self.tog[e, a] += 1
            if self.tog[e, a] < 4:
                self.lap_times[e, a] = self.time[e]
        assert np.array_equal(g['toggles'][e], self.tog[e]), (tag, g['toggles'][e], self.tog[e])
        assert np.array_equal(g['lap_counts'][e], (self.tog[e] // 2).astype(np.float64)), tag
        assert np.array_equal(g['lap_times'][e], self.lap_times[e]), tag
        assert g['time'][e] == self.time[e], tag
        all_laps = bool((self.tog[e] >= 4).all())
        done = bool(coll[self.ego]) or all_laps
        assert bool(g['terminated'][e]) == done, tag
        if done:
            self.stats += [1, self.steps[e] + 1, bool(coll[self.ego]), all_laps, self.time[e]]
        self.c['laps'] += int((g['toggles'][e] >= 2).sum())
        # pose slots of the observation (f110_env.py:563-579)
        if 'obs' in g:
            q = np.zeros(8, np.float32)
            for k in range(min(A, 2)):
                q[4 * k:4 * k + 4] = (st[k, 0], st[k, 1], wrap_yaw(st[k, 4]), 1.0 if coll[k] else 0.0)
            assert np.array_equal(g['obs'][e, B:].view(np.int32), q.view(np.int32)), (tag, g['obs'][e, B:], q)

    def _tolerance(self, o, org, poses, a, exp, lowered):
        """One unit of the lowered beams' error budget: an ulp of the range plus an ulp of the coordinates the vertices
        and the origin are formed in (the vertices come from CUDA's sincos, the reference's from libm), divided by the
        sine of the angle at which the beam meets the edge it ends on (a grazing beam magnifies both)."""
        tol = np.spacing(exp)
        idx = np.flatnonzero(lowered)
        if not len(idx):
            return tol
        th = org[2] + np.asarray(self.angles)[idx]
        ux, uy = np.cos(th), np.sin(th)
        px, py = org[0] + exp[idx] * ux, org[1] + exp[idx] * uy
        best_d, sin_t = np.full(len(idx), np.inf), np.ones(len(idx))
        scale = abs(org[:2]).max()
        for b in range(self.A):
            if b == a:
                continue
            v = o.get_vertices(poses[b], self.L[a], self.W[a])
            scale = max(scale, abs(v).max())
            for k in range(4):
                p0, p1 = v[k], v[(k + 1) % 4]
                ex, ey = p1 - p0
                t = np.clip(((px - p0[0]) * ex + (py - p0[1]) * ey) / (ex * ex + ey * ey), 0, 1)
                d = np.hypot(px - p0[0] - t * ex, py - p0[1] - t * ey)
                s = abs(ex * uy - ey * ux) / math.hypot(ex, ey)
                sin_t = np.where(d < best_d, s, sin_t)
                best_d = np.minimum(best_d, d)
        tol[idx] = (tol[idx] + np.spacing(scale)) / np.maximum(sin_t, 1e-6)
        return tol

    def check_stats(self, sim):
        got = sim.stats(reset=True).cpu().numpy()
        assert np.array_equal(got[:4], self.stats[:4]), (got[:5], self.stats)
        assert abs(got[EPISODE_TIME] - self.stats[EPISODE_TIME]) <= 1e-12 * max(1.0, self.stats[EPISODE_TIME])
        assert not got[5:].any()

    def report(self, label):
        c = self.c
        print('%s: lowered beams checked %d of %d (max %.2f of the budget unit), GJK collisions %d, iTTC stops %d, cars past a lap %d, '
              'exempt: GJK %d, window near-ties %d beams in %d pairs' % (label, c['lowered'], c['beams'], c['max_err'],
                                                                         c['gjk'], c['ittc'], c['laps'], c['gjk_exempt'],
                                                                         c['tie_exempt'], c['tie_pairs']))
        assert c['gjk_exempt'] + c['tie_exempt'] <= 1e-6 * c['beams'] + 2, c


# ----------------------------------------------------------------------------- 1. replay of GPU rollouts

SHANGHAI = 'Shanghai_map'


def _arc_poses(rng, A, cl, arclen, m):
    """A cars one behind the other along the (doubled) centerline, 0.3-1.5 m apart, car 0 the last, with lateral offsets of
    up to 0.25 m; about every third car is turned to face the nearer side of the track from 0.3 m (the iTTC stops it)."""
    j0 = rng.integers(0, len(cl) // 2)
    s = np.concatenate([[0.0], np.cumsum(rng.uniform(0.3, 1.5, A - 1))])
    p = cl[np.searchsorted(arclen, arclen[j0] + s)].copy()
    dt, res, org = m
    half = dt[((p[:, 1] - org[1]) / res).astype(int), ((p[:, 0] - org[0]) / res).astype(int)]
    turn = rng.choice([-1.0, 1.0], A) * (rng.uniform(size=A) < 1 / 3)
    lat = np.where(turn != 0, turn * (half - 0.3), rng.uniform(-0.25, 0.25, A))
    p[:, 0] -= lat * np.sin(p[:, 2])
    p[:, 1] += lat * np.cos(p[:, 2])
    p[:, 2] += rng.uniform(-0.1, 0.1, A) + turn * np.pi / 2
    return p


def _square_poses(rng, A):
    c = rng.uniform(-4, 4, 2)
    th = rng.uniform(-np.pi, np.pi)
    s = np.concatenate([[0.0], np.cumsum(rng.uniform(0.3, 1.5, A - 1))])
    lat = rng.uniform(-0.25, 0.25, A)
    return np.stack([c[0] + s * np.cos(th) - lat * np.sin(th), c[1] + s * np.sin(th) + lat * np.cos(th),
                     np.full(A, th) + rng.uniform(-0.1, 0.1, A)], 1)


def _drive(rng, g, e, A, cl, slot):
    """Pure pursuit towards the centerline 0.8 m ahead (Shanghai) or a circle (open square); the car behind is faster, and
    every fourth car steers hard into the wall."""
    st = g['state'][e]
    act = np.zeros((A, 2))
    for a in range(A):
        if (e + a) % 4 == 0:
            steer = 0.4 if e % 2 else -0.4
        elif slot == 0:
            j = int(np.argmin((cl[:, 0] - st[a, 0]) ** 2 + (cl[:, 1] - st[a, 1]) ** 2))
            tx, ty = cl[(j + 10) % len(cl), :2]
            steer = wrap_yaw(math.atan2(ty - st[a, 1], tx - st[a, 0]) - st[a, 4])
        else:
            steer = 0.25
        act[a] = (np.clip(steer + rng.normal(0, 0.05), -0.4, 0.4), 7.0 - 4.0 * a / max(A - 1, 1) + rng.uniform(-0.5, 0.5))
    return act


def _replay_run(A, N, B, fov, steps=50, maps=(SHANGHAI,), ego=0, per_agent=False, holes=False, lean=False, seed=0):
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS
    from oracle.f110_oracle import DEFAULT_PARAMS
    rng = np.random.default_rng(seed)
    mdata = [H.golden_map(m) for m in maps]
    outputs = tuple(k for k in ALL_OUTPUTS if k != 'scans_f64') if lean else ALL_OUTPUTS
    m = mdata if len(maps) > 1 else mdata[0]
    sim = _sim(N, A, B, fov, m, outputs=outputs, ego_idx=ego)
    twin = _sim(N, A, B, fov, m, outputs=('state',), ego_idx=ego, ttc_thresh=0.0)
    L, W = [DEFAULT_PARAMS['length']] * A, [DEFAULT_PARAMS['width']] * A
    if per_agent:
        for a, (la, wa) in enumerate([(0.75, 0.42), (0.45, 0.22), (0.9, 0.31)][:A]):
            p = dict(DEFAULT_PARAMS, length=la, width=wa)
            sim.update_params(p, a)
            twin.update_params(p, a)
            L[a], W[a] = la, wa
    oracles = [_oracle(B, fov, md) for md in mdata]
    from f110_gymnasium_ros2_jazzy_b200.params import beam_tables
    assert np.array_equal(oracles[0].get_beam_tables()[0], beam_tables(DEFAULT_PARAMS, B, fov)[0])
    slots = (np.arange(N) * len(maps)) // N
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    arclen = np.concatenate([[0.0], np.cumsum(np.hypot(*np.diff(cl[:, :2], axis=0).T))])
    cl2 = np.concatenate([cl, cl])
    arclen2 = np.concatenate([arclen, arclen + arclen[-1] + 0.08])
    rep = Replay(N, A, B, fov, oracles, L, W, ego=ego)
    sim.stats(reset=True)
    g = None
    for t in range(steps):
        poses = np.stack([_arc_poses(rng, A, cl2, arclen2, mdata[0]) if slots[e] == 0 else _square_poses(rng, A) for e in range(N)])
        if t == 0:
            rm = np.ones(N, np.uint8)
        else:
            rm = (g['terminated'] | ((np.arange(N) + t) % 40 == 0)).astype(np.uint8)
        act = np.zeros((N, A, 2)) if g is None else np.stack([_drive(rng, g, e, A, cl, slots[e]) for e in range(N)])
        noise = None if lean else rng.normal(0, 0.01, (N, A, B))
        am = None
        if holes and t > 0:
            am = np.ones(N, np.uint8)
            am[[1, 2, 5, N - 2]] = rng.integers(0, 2, 4)
        twin.load_state_dict(sim.state_dict())
        twin.step(act, noise, reset_mask=rm, reset_poses=poses, active_mask=am)
        sim.step(act, noise, reset_mask=rm, reset_poses=poses, active_mask=am)
        if lean:
            assert sim.lidar_variant()['mode'] == 3
        g = _np(sim)
        tv = _np(twin)['state'][:, :, 3]
        for e in range(N):
            if am is not None and not am[e]:
                continue
            if rm[e]:
                rep.reset(e, poses[e])
            rep.check(e, g, slots[e], None if noise is None else noise[e], tv[e], f64=not lean,
                      where=('step', t))
    rep.check_stats(sim)
    rep.report('A %d B %d fov %.1f envs/CTA %d N %d%s' % (A, B, fov, _post_envs_per_cta(A) if A > 1 else 128, N,
                                                         ' lean' if lean else ''))
    return rep.c


REPLAY_RUNS = {
    'A1': dict(A=1, N=37, B=1080, fov=4.7),
    'A2_holes': dict(A=2, N=29, B=1080, fov=4.7, holes=True),
    'A3_params_ego1': dict(A=3, N=20, B=541, fov=4.7, per_agent=True, ego=1),
    'A4_unstaged': dict(A=4, N=9, B=2049, fov=4.7),
    'A6_wide': dict(A=6, N=5, B=2048, fov=6.2),
    'A8_narrow': dict(A=8, N=4, B=32, fov=1.0),
    'A16': dict(A=16, N=3, B=4320, fov=4.7, steps=25),
    'A2_maps': dict(A=2, N=21, B=1080, fov=4.7, maps=(SHANGHAI, 'open_square')),
    'A2_lean': dict(A=2, N=19, B=1080, fov=4.7, lean=True),
    'A3_lean_unstaged': dict(A=3, N=11, B=2049, fov=6.2, lean=True),
}


@pytest.mark.parametrize('name', sorted(REPLAY_RUNS))
def test_post_kernel_replays_exactly(name):
    kw = REPLAY_RUNS[name]
    c = _replay_run(seed=sorted(REPLAY_RUNS).index(name), **kw)
    assert c['ittc'] > 0, c
    if kw['A'] > 1:
        assert c['lowered'] > 0 and c['gjk'] > 0, c


# ----------------------------------------------------------------------------- 2. constructed geometries at reset steps

def _constructed(A, B, fov, angles, L=0.58, W=0.31):
    """Reset poses [n, A, 3] on the open square: car 0 at the origin, the others placed on purpose."""
    out = []
    R = 0.5 * math.hypot(L, W)

    def two(ego_yaw, bear, d, yaw):
        th = ego_yaw + bear
        return [(0.0, 0.0, ego_yaw), (d * math.cos(th), d * math.sin(th), yaw)]
    for y in (0.0, 0.4, -2.0, math.pi / 2):
        out.append(two(y, math.pi, 1.2, y))                          # straight behind: vertex beams clamp to 0 and B - 1
        out.append(two(y, math.pi - 0.2, 0.8, 0.3))
        for s in (-1, 1):
            out.append(two(y, s * fov / 2, 1.0, 0.0))                 # straddling +-fov/2
            out.append(two(y, s * 1.6, 0.45, 1.0))                   # forward and backward cones overlap and merge
        out.append(two(y, 0.3, 0.2, 0.5))                            # overlapping cars, dist <= R
        out.append(two(y, 0.0, 0.0, y))                              # identical poses
        out.append(two(y, 0.1, 3.0, 2.0))
        out.append(two(y, 0.0, 25.0, 1.0))                           # far: a tiny cone
        out.append(two(y, -0.05, 45.0, 0.0))                         # beyond max_range
        out.append(two(y, 0.7, R * (1 + 5e-7), 0.0))                 # on the bounding circle's pruning edge
    out.append([(0.0, 0.0, 0.7), (L / 2, -W / 2, 0.0)])              # a vertex exactly at the observer (NaN -> beam 0)
    for i in range(B // 2 - 5, B // 2 + 5):                          # the collinear fallback, both ways, on and 1e-9 off
        out += [[ego, opp] for ego, opp, _, _ in collinear_geometries(angles, i, L, W)]
    if A == 2:
        return np.array(out)
    if A >= 16:                                                      # a ring of 15 cars at mixed distances
        rng = np.random.default_rng(A)
        rings = []
        for k in range(6):
            ego = (0.0, 0.0, rng.uniform(-np.pi, np.pi))
            d = rng.choice([0.35, 0.6, 1.0, 2.0, 4.0], A - 1)
            th = np.linspace(-np.pi, np.pi, A - 1, endpoint=False) + rng.uniform(-0.1, 0.1, A - 1)
            rings.append([ego] + [(d[j] * math.cos(th[j]), d[j] * math.sin(th[j]), rng.uniform(-3, 3)) for j in range(A - 1)])
        return np.array(rings)
    # A = 3: each two-car geometry with a third car out of the way, and swapped observers
    return np.array([g + [(3.0, -3.0, 0.0)] for g in out] + [[g[1], g[0], (-3.0, 3.0, 1.0)] for g in out])


CONSTRUCTED = [(2, 1080, 4.7), (2, 32, 4.7), (2, 541, 1.0), (2, 2049, 6.2), (2, 4320, 4.7), (3, 1080, 4.7), (16, 1080, 4.7),
               (16, 2049, 6.2)]


@pytest.mark.parametrize('A,B,fov', CONSTRUCTED)
def test_constructed_geometries_at_reset(A, B, fov):
    _torch()
    m = H.golden_map('open_square')
    o1 = _oracle(B, fov, m)
    angles = list(o1.get_beam_tables()[0])
    poses = _constructed(A, B, fov, angles)
    N = len(poses)
    sim = _sim(N, A, B, fov, m)
    orc = _oracle(B, fov, m, A, N)
    rep = Replay(N, A, B, fov, [o1], [0.58] * A, [0.31] * A)
    ones = np.ones(N, np.uint8)
    noise = np.zeros((N, A, B))
    for t in range(2):
        p = poses if t == 0 else poses[::-1].copy()
        sim.step(None, noise, reset_mask=ones, reset_poses=p)
        g = _np(sim)
        want = orc.step(None, noise, reset_mask=ones, reset_poses=p)
        for e in range(N):
            rep.reset(e, p[e])
            rep.check(e, g, noise=noise[e], where=('reset', t))
        low = want['scans'] != np.stack([[o1.scan(q)[0] for q in env] for env in p])
        d = np.abs(g['scans_f64'] - want['scans'])
        assert np.array_equal(g['scans_f64'][~low], want['scans'][~low])
        tol = np.stack([[rep._tolerance(o1, p[e, a, [0, 1, 2]], p[e], a, want['scans'][e, a], low[e, a]) for a in range(A)]
                        for e in range(N)])
        assert (d[low] <= 4 * tol[low]).all()
        for k in ('collisions', 'terminated', 'toggles'):
            assert np.array_equal(g[k], want[k]), k
    rep.report('constructed A %d B %d fov %.1f, %d geometries' % (A, B, fov, N))
    assert rep.c['lowered'] > 0 and rep.c['gjk'] > 0


@pytest.mark.parametrize('i', [540, 545, 549])
def test_collinear_fallback_on_the_gpu(i):
    """The only geometry that needs the backward cone: the beam that points straight away from the opponent's rear edge
    is lowered to 1 - W/2, by the GPU as by the oracle, and no other beam is."""
    _torch()
    m = H.golden_map('open_square')
    o1 = _oracle(1080, 4.7, m)
    geos = collinear_geometries(list(o1.get_beam_tables()[0]), i)
    poses = np.array([[ego, opp] for ego, opp, _, _ in geos])
    sim = _sim(len(poses), 2, 1080, 4.7, m)
    sim.step(None, np.zeros((len(poses), 2, 1080)), reset_mask=np.ones(len(poses), np.uint8), reset_poses=poses)
    g = _np(sim)
    for e, (ego, opp, _, W) in enumerate(geos):
        wall = o1.scan(np.array(ego))[0]
        lowered = np.flatnonzero(g['scans_f64'][e, 0] != wall)
        assert i in lowered and abs(g['scans_f64'][e, 0, i] - (1 - W / 2)) < 1e-8, (e, lowered)
        if opp[1] > 0:
            assert list(lowered) == [i], (e, lowered)


# ----------------------------------------------------------------------------- 3. laps, done and the episode counters

def _edge_values():
    p = math.sqrt(0.1)
    while p * p > 0.1:
        p = math.nextafter(p, 0.0)
    while math.nextafter(p, 1.0) ** 2 <= 0.1:
        p = math.nextafter(p, 1.0)
    p_out = math.nextafter(p, 1.0)                         # p * p <= 0.1 < p_out * p_out
    q_in, q_out = None, None
    for k in range(-200, 200):                            # 2 + q with (2 + q - 2)^2 at the edge
        y = 2.0 + p + k * 2.0 ** -51
        if (y - 2) ** 2 <= 0.1:
            q_in = y
        elif q_in is not None and q_out is None:
            q_out = y
    return p, p_out, q_in, q_out


def _lap_walk(A, n_env, rng):
    """Per env and step, a position offset from the start for every car: in and out of the finish zone across its edges."""
    p, p_out, q_in, q_out = _edge_values()
    two_up = math.nextafter(2.0, 3.0)
    inside = [(p, 0.0), (-p, 0.0), (0.0, 2.0), (0.0, -2.0), (0.0, two_up), (0.0, -two_up), (0.0, q_in), (0.0, -q_in),
              (p, 2.0), (-p, -2.0), (0.0, 0.0)]
    outside = [(p_out, 0.0), (-p_out, 0.0), (0.0, q_out), (0.0, -q_out), (p_out, 2.0), (0.5, 0.0), (0.0, 3.0)]
    walks = []
    for e in range(n_env):
        cars = []
        for a in range(A):
            seq = []
            for k in range(12):
                pool = outside if k % 2 == 0 else inside
                seq.append(pool[rng.integers(0, len(pool))])
                if rng.uniform() < 0.3:                     # stay a step: no toggle
                    seq.append(seq[-1])
            cars.append(seq)
        T = min(len(c) for c in cars)
        walks.append([[c[t] for c in cars] for t in range(T)])
    T = min(len(w) for w in walks)
    return np.array([w[:T] for w in walks])                  # [N, T, A, 2]


@pytest.mark.parametrize('A', [1, 2, 3])
def test_laps_done_and_episode_counters(A):
    """Cars moved by sim_reset (Simulator.reset: poses only; start poses, toggles and time untouched, on both sides) and a
    zero-action step that leaves them where they were put.  With start yaw 0 the start rotation is exactly (1, 0), so the
    finish-zone edges -- dist2 = 0.1 and one ulp above, |ty| = 2 and one ulp beyond -- are exact on both sides."""
    _torch()
    m = H.golden_map('open_square')
    rng = np.random.default_rng(A)
    N = 10
    starts = np.zeros((N, A, 3))
    starts[:, :, 0] = np.arange(A)[None, :] * 2.5           # the ego starts at the origin: its offsets are exact
    starts[:, 1:, 1] = -2.0 + np.arange(N)[:, None] * 0.25
    walk = _lap_walk(A, N, rng)
    sim = _sim(N, A, 1080, 4.7, m)
    orc = _oracle(1080, 4.7, m, A, N)
    sim.stats(reset=True)
    ones, zeros = np.ones(N, np.uint8), np.zeros((N, A, 1080))
    stats = np.zeros(5)
    steps = np.zeros(N, np.int64)

    def step(*args, **kw):
        sim.step(*args, **kw)
        g, want = _np(sim), orc.step(*args, **kw)
        act = kw.get('active_mask')
        act = np.ones(N, bool) if act is None else act.astype(bool)
        for k in ('toggles', 'lap_counts', 'lap_times', 'time', 'terminated', 'collisions'):
            assert np.array_equal(g[k][act], want[k][act]), (k, g[k][act], want[k][act])
        for e in np.flatnonzero(act):
            # the env's step count: 0 on a reset step and after sim_reset, + 1 on every other step it runs
            steps[e] = 0 if kw.get('reset_mask') is not None else steps[e] + 1
            if want['terminated'][e]:
                laps = bool((want['toggles'][e] >= 4).all())
                stats[:] += [1, steps[e] + 1, bool(want['collisions'][e, 0]), laps, want['time'][e]]
        return g

    for rnd in range(2):
        step(None, zeros, reset_mask=ones, reset_poses=starts)
        for t in range(walk.shape[1]):
            pos = starts.copy()
            pos[:, :, :2] += walk[:, t]
            if A > 1 and t == walk.shape[1] - 2:
                pos[0, 1] = pos[0, 0]                           # env 0: the ego rammed, done by collision
            am = None
            if rnd == 1:
                am = ones.copy()
                am[[3, 7]] = t % 2                              # done envs hidden every other step
            # the oracle's sim_reset moves every env; a hidden env does not step, and is moved again before it next does
            sim.sim_reset(pos, env_mask=am)
            orc.sim_reset(pos)
            steps[:] = np.where(am == 0, steps, 0) if am is not None else 0
            step(None, zeros, active_mask=am)
        got = sim.stats(reset=True).cpu().numpy()
        print('A %d round %d: episodes %d, steps %d, ego collisions %d, laps done %d, time %.2f' % ((A, rnd) + tuple(got[:5])))
        assert np.array_equal(got[:4], stats[:4]), (got[:5], stats)
        assert abs(got[EPISODE_TIME] - stats[EPISODE_TIME]) <= 1e-12 * max(1.0, stats[EPISODE_TIME])
        assert stats[LAPS_DONE] > 0 and (A == 1 or stats[EGO_COLLISIONS] > 0)
        stats[:] = 0
