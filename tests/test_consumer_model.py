"""The oracle's consumers (oracle/f110_oracle.c: f110o_gap_follow and the shaped reward) pinned to the numpy and scipy
calls the reference makes, at every parameter, shape and branch.  CPU only.

Gap follow: a numpy restatement of rl_training/utils/gap_follow.py:3-58 with every parameter (np.clip, np.mean of float32
slices, np.argmin, the bubble, the first longest run, (s + e) // 2, the np.radians speed bands), pinned to the recorded
reference on tests/golden/gap_follow.npz; the oracle must then equal it bit for bit over a grid of window sizes, bubble
radii, thresholds, distances, beam counts and non-finite beams.  numpy sums a float32 slice of 8 or more elements as an
eight-way tree, and np.argmin returns the first NaN: windows of 8 to 15 beams and NaN beams are where a sequential sum or a
NaN-blind argmin part from the reference.

Reward: the float32 wall quantile against np.quantile, the lateral segment lookup against np.searchsorted, the 5 nearest
midpoints against scipy's cKDTree.  reward_cases() builds seeded centerlines and episodes, each aimed at a branch of the
reward; test_reward_cases_reach_their_branches checks on the oracle's per-env breakdown that each one gets there.  The GPU
tests (test_consumer_kernels.py) hold both reward kernels to the oracle on the same cases.
"""
import numpy as np
import pytest

from oracle.f110_oracle import REWARD_TERM as T, RewardOracle, gap_follow_action, quantile_f32
from tests import helpers as H

# ----------------------------------------------------------------------------------------------------- gap follow


def np_gap_follow(scan, angle_min=-np.pi / 2, angle_increment=np.pi / 1080, max_distance=3.0, window_size=5,
                  bubble_radius=30, threshold=0.5):
    """gap_follow.py:3-58 in numpy: float32 scan -> (steer, speed) float64 and the window means (before the bubble)."""
    ranges = np.asarray(scan, np.float32)
    n = len(ranges)
    clipped = np.clip(ranges, 0, np.float32(max_distance))                    # preprocess_lidar :3-12
    half = window_size // 2
    proc = np.array([np.mean(clipped[max(0, i - half):min(n - 1, i + half) + 1]) for i in range(n)], np.float32)
    free = proc.copy()
    closest = int(np.argmin(free))                                             # create_bubble :14-19
    free[max(0, closest - bubble_radius):min(n - 1, closest + bubble_radius) + 1] = 0
    masked = free > np.float32(threshold)                                      # find_max_gap :21-38
    gaps, start = [], None
    for i, val in enumerate(masked):
        if val and start is None:
            start = i
        elif not val and start is not None:
            gaps.append((start, i - 1))
            start = None
    if start is not None:
        gaps.append((start, n - 1))
    s, e = max(gaps, key=lambda g: g[1] - g[0]) if gaps else (0, n - 1)
    best = (s + e) // 2                                                        # find_best_point :40-41
    steering = angle_min + best * angle_increment                             # :49
    speed = 2.5 if abs(steering) < np.radians(10) else (2.0 if abs(steering) < np.radians(20) else 1.5)
    return np.array([steering, speed]), proc


def _poison(rng, scans, max_distance):
    """Non-finite, negative and clipped beams in a few rows of a batch of scans (in place)."""
    n = scans.shape[1]
    k = len(scans)
    scans[0, rng.integers(0, n)] = np.nan
    if k > 1:
        scans[1, rng.integers(0, n, size=3)] = np.nan
        scans[1, 0] = np.nan if n > 1 else scans[1, 0]
    if k > 2:
        scans[2, rng.integers(0, n, size=max(1, n // 9))] = np.inf
    if k > 3:
        scans[3, ::3] = -np.inf
    if k > 4:
        scans[4, rng.integers(0, n, size=max(1, n // 5))] *= -1
    if k > 5:
        scans[5] = np.nan
    if k > 6:
        scans[6, : n // 2] = 2 * max_distance + 1
    return scans


def _scans(rng, num, n, max_distance=3.0):
    """Blocky scans (runs of every length, level ties) plus uniform ones, then a few poisoned rows."""
    out = np.empty((num, n), np.float32)
    for row in out[: num // 2]:
        i = 0
        while i < n:
            ln = int(rng.choice([1, 2, 3, 7, 8, 9, 15, 16, 33, 70]))
            row[i:i + ln] = rng.choice([0.0, 0.3, 0.5, 0.6, 1.0, 2.5, 3.0, 9.0])
            i += ln
    out[num // 2:] = rng.uniform(0.0, 1.5 * max_distance, size=(num - num // 2, n)).astype(np.float32)
    return _poison(rng, out, max_distance)


def gap_follow_grid():
    """[(label, scans [k, n] float32, kwargs)]: every window size 1..15, bubble radii 0, 1, 30 and >= n, several
    thresholds and distances, the beam counts around the warp and shared-memory sizes, the speed bands hit exactly."""
    rng = np.random.default_rng(2024)
    cases = []
    for w in range(1, 16):
        cases.append(('window%d' % w, _scans(rng, 12, 1080), dict(window_size=w)))
    for br in (0, 1, 30, 1080, 5000):
        cases.append(('bubble%d' % br, _scans(rng, 8, 1080), dict(bubble_radius=br, window_size=9)))
    for thr, md in ((0.0, 3.0), (0.5, 1.0), (2.9, 3.0), (3.0, 3.0), (0.25, 10.0), (-1.0, 3.0), (1.0, 0.0)):
        cases.append(('thr%g_md%g' % (thr, md), _scans(rng, 8, 1080, md), dict(threshold=thr, max_distance=md, window_size=11)))
    for n in (1, 2, 31, 32, 33, 1080, 6049, 6050, 8192):
        for w in (5, 9):
            cases.append(('n%d_w%d' % (n, w), _scans(rng, 8 if n < 6000 else 3, n), dict(window_size=w, angle_increment=np.pi / n)))
    # the speed bands' boundaries hit exactly: angle_increment 0 makes the steering angle_min itself
    edge = _scans(rng, 4, 64)
    for a in (np.radians(10), -np.radians(10), np.radians(20), -np.radians(20), np.nextafter(np.radians(10), 0),
              np.nextafter(np.radians(20), 0), np.nextafter(np.radians(20), 1), 0.0):
        cases.append(('band%.17g' % a, edge, dict(angle_min=float(a), angle_increment=0.0, window_size=8)))
    return cases


def test_numpy_gap_follow_matches_recorded_reference():
    """The restatement reproduces the reference's actions on the 214 recorded scans and its window means on 8 of them."""
    g = H.load('gap_follow')
    for s, a in zip(g['scans'], g['actions']):
        assert np.array_equal(np_gap_follow(s)[0], a)
    for k in range(len(g['proc'])):
        assert np.array_equal(np_gap_follow(g['scans'][k])[1], g['proc'][k])


@pytest.mark.parametrize('label,scans,kw', [pytest.param(*c, id=c[0]) for c in gap_follow_grid()])
def test_oracle_gap_follow_equals_numpy(label, scans, kw):
    """f110o_gap_follow == the numpy restatement, actions and window means bit for bit (NaN where numpy has NaN)."""
    for s in scans:
        want, wproc = np_gap_follow(s, **kw)
        got, gproc = gap_follow_action(s, want_proc=True, **kw)
        assert np.array_equal(got, want), (label, got, want)
        assert np.array_equal(gproc.view(np.uint32), wproc.view(np.uint32)) or np.array_equal(gproc, wproc, equal_nan=True), label


def test_gap_follow_grid_reaches_the_numpy_divergences():
    """The grid holds windows whose numpy mean differs from a sequential float32 sum, scans where np.argmin lands on a NaN
    that is not beam 0, and both speed band boundaries: the cases the oracle once got wrong are in it."""
    seq_differs = nan_first = 0
    for label, scans, kw in gap_follow_grid():
        w = kw.get('window_size', 5)
        for s in scans:
            _, proc = np_gap_follow(s, **kw)
            if np.isnan(proc).any() and not np.isnan(proc[0]) and np.argmin(proc) > 0:
                nan_first += 1
            if w >= 8 and label.startswith('window'):
                c = np.clip(s, 0, np.float32(kw.get('max_distance', 3.0)))
                h = w // 2
                for i in range(h, len(c) - h, 7):
                    acc = np.float32(0)
                    for v in c[i - h:i + h + 1]:
                        acc = np.float32(acc + v)
                    seq_differs += np.float32(acc / np.float32(2 * h + 1)) != proc[i]
    assert seq_differs > 100 and nan_first > 10, (seq_differs, nan_first)
    speeds = {lab: gap_follow_action(sc[0], **kw)[1] for lab, sc, kw in gap_follow_grid() if lab.startswith('band')}
    assert sorted(set(speeds.values())) == [1.5, 2.0, 2.5]


# ----------------------------------------------------------------------------------------------------- reward internals

QUANTILE_BEAMS = (1, 2, 3, 31, 33, 1080, 4097, 8192)
QUANTILES = (0.0, 0.05, 0.1, 0.5, 1.0)


@pytest.mark.parametrize('B', QUANTILE_BEAMS)
def test_wall_quantile_equals_numpy(B):
    rng = np.random.default_rng(B)
    arrays = [rng.uniform(0, 1, B).astype(np.float32),
              rng.choice(np.float32([0.1, 0.25, 0.5, 1.0]), B),                       # heavy ties
              np.full(B, 0.3, np.float32),                                            # all equal
              np.round(rng.uniform(0, 1, B) * 8).astype(np.float32) / np.float32(8.0)]
    for a in arrays:
        for q in QUANTILES:
            want = np.quantile(a, q)
            assert want.dtype == np.float32
            assert quantile_f32(a, q).tobytes() == want.tobytes(), (B, q)


def _track_knots(xy):
    seg = np.diff(xy, axis=0)
    return np.concatenate([[0.0], np.cumsum(np.sqrt(seg[:, 0] * seg[:, 0] + seg[:, 1] * seg[:, 1]))])


def test_lateral_segment_index_equals_searchsorted():
    """np.searchsorted(s, e_s, 'right') - 1 clamped to [0, n - 2], on knots exactly, between them, beyond both ends and
    on repeated knots (zero-length segments)."""
    rng = np.random.default_rng(5)
    xy = np.cumsum(rng.uniform(-1, 1, size=(200, 2)), axis=0)
    xy[50] = xy[49]; xy[51] = xy[49]; xy[120] = xy[119]                               # repeated points
    for pts in (xy, xy[:2], xy[:3], np.concatenate([xy[:1], xy[:1], xy[:5]])):
        o = RewardOracle(1, pts, num_beams=8)
        s = _track_knots(pts)
        n = len(pts)
        qs = np.concatenate([s, np.nextafter(s, -np.inf), np.nextafter(s, np.inf), rng.uniform(-1, s[-1] + 1, 200),
                             [-1e300, 1e300, 0.0, -0.0]])
        for q in qs:
            want = int(np.clip(np.searchsorted(s, q, 'right') - 1, 0, n - 2))
            assert o.seg_index(q) == want, (n, q)


def _lattice(n_side=12):
    """A serpentine polyline through an integer lattice: midpoints on half-integers, so lattice cars see exact ties."""
    pts = []
    for r in range(n_side):
        cols = range(n_side) if r % 2 == 0 else range(n_side - 1, -1, -1)
        pts += [(float(c), float(r)) for c in cols]
    return np.array(pts)


def test_five_nearest_midpoints_equal_ckdtree():
    """The oracle's 5 nearest midpoints against scipy.spatial.cKDTree(mid).query(p, k=5): the same index sets except
    among exact ties, ordered by (distance, index); sqrt of the oracle's squared distance within one ulp of cKDTree's."""
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(11)
    shanghai = H.reward_recording()['centerline'][:, :2]
    tracks = [('shanghai', shanghai, shanghai[rng.integers(0, len(shanghai), 300)] + rng.normal(0, 1.0, (300, 2))),
              ('lattice', _lattice(), np.concatenate([rng.integers(0, 12, (200, 2)).astype(float),
                                                      rng.integers(0, 24, (100, 2)) / 2.0])),
              ('hairpin', hairpin_xy(), hairpin_xy()[rng.integers(0, 400, 200)] + rng.normal(0, 0.3, (200, 2)))]
    bit_equal = total = 0
    for name, xy, cars in tracks:
        o = RewardOracle(1, xy, num_beams=8)
        mid = (xy[:-1] + xy[1:]) * 0.5
        tree = cKDTree(mid)
        dist, idx = tree.query(cars, k=6)
        for p, dd, ii in zip(cars, dist, idx):
            got, _ = o.knn(p[0], p[1])
            dx, dy = mid[got, 0] - p[0], mid[got, 1] - p[1]
            d2 = dx * dx + dy * dy
            order = np.lexsort((got, d2))
            assert np.array_equal(order, np.arange(5)), (name, p)               # (distance, index) order
            dg = np.sqrt(d2)
            assert (np.abs(dg - dd[:5]) <= np.spacing(dd[:5])).all(), (name, p, dg, dd)
            bit_equal += int((dg == dd[:5]).sum()); total += 5
            if dd[4] < dd[5] and len(set(np.round(dd[:5], 12))) == 5:
                assert set(got) == set(ii[:5]), (name, p)
            # the full answer in the contract's order: every midpoint sorted by (distance, index), first five
            all_d2 = (mid[:, 0] - p[0]) * (mid[:, 0] - p[0]) + (mid[:, 1] - p[1]) * (mid[:, 1] - p[1])
            assert np.array_equal(got, np.lexsort((np.arange(len(mid)), all_d2))[:5]), (name, p)
    print('knn distances bit-equal to cKDTree: %d of %d' % (bit_equal, total))


# ----------------------------------------------------------------------------------------------------- reward cases

def hairpin_xy(n=401, gap=0.5):
    """Two 20 m legs 0.5 m apart joined by a half circle: a car's 5 neighbours come from both legs, far apart in index."""
    leg = np.linspace(0, 20, (n - 41) // 2)
    th = np.linspace(-np.pi / 2, np.pi / 2, 41)[1:-1]
    a = np.stack([leg, np.zeros_like(leg)], 1)
    b = np.stack([20 + gap / 2 * np.cos(th), gap / 2 + gap / 2 * np.sin(th)], 1)
    c = np.stack([leg[::-1], np.full_like(leg, gap)], 1)
    return np.concatenate([a, b, c])


def circle_xy(n=200, r=6.0):
    """A closed loop whose last point repeats the first: cars circling it cross the seam at s = 0 = L."""
    th = np.linspace(0, 2 * np.pi, n)
    xy = np.stack([r * np.cos(th), r * np.sin(th)], 1)
    xy[-1] = xy[0]
    return xy


def s_curve_xy(n=300):
    t = np.linspace(0, 1, n)
    return np.stack([30 * t, 4 * np.sin(2 * np.pi * t)], 1)


def pose_along(xy, s_knots, s, t, closed):
    """The point at arclength s (wrapped when closed), moved t along the left normal, and its heading."""
    L = s_knots[-1]
    s = np.mod(s, L) if closed else np.clip(s, 0, L)
    i = np.clip(np.searchsorted(s_knots, s, 'right') - 1, 0, len(xy) - 2)
    seg = xy[i + 1] - xy[i]
    ln = np.maximum(np.hypot(seg[:, 0], seg[:, 1]), 1e-12)
    u = seg / ln[:, None]
    f = np.clip((s - s_knots[i]) / ln, 0, 1)
    p = xy[i] + f[:, None] * seg + t[:, None] * np.stack([-u[:, 1], u[:, 0]], 1)
    return p, np.arctan2(u[:, 1], u[:, 0])


def lidar(rng, N, B, lidar_max):
    """Uniform lidar with heavy ties and, in some rows, zeros, NaN, inf, negatives and values above lidar_max."""
    x = rng.uniform(0.0, 1.3 * lidar_max, (N, B)).astype(np.float32)
    x[::2] = np.round(x[::2] * 16) / 16
    for e in range(0, N, 3):
        k = rng.integers(0, B, size=max(1, B // 10))
        x[e, k] = rng.choice(np.float32([0.0, np.nan, np.inf, -np.inf, -0.5, 2 * lidar_max, -0.0]), len(k))
    x[x.shape[0] // 2, :] = 0.0 if N > 1 else x[0]
    x[-1, : B // 3] = np.float32(lidar_max) * np.float32(0.001)             # near a wall
    return x


class Case(object):
    """One reward scenario: centerline, parameters and T steps of N envs' observations (and reset masks)."""

    def __init__(self, name, centerline, obs, masks, closed=True, num_beams=32, check=None, **kw):
        self.name, self.centerline, self.obs, self.masks, self.closed = name, centerline, obs, masks, closed
        self.num_beams, self.check, self.kw = num_beams, check, kw

    def oracle_run(self):
        """-> totals [T, N], terms [T, N, 32] from the oracle."""
        o = RewardOracle(self.obs.shape[1], self.centerline, num_beams=self.num_beams, closed=self.closed, **self.kw)
        out = [o.compute_terms(self.obs[t], None if self.masks is None else self.masks[t]) for t in range(len(self.obs))]
        return np.stack([a for a, _ in out]), np.stack([b for _, b in out])


def episodes(rng, xy, closed, N, T, B, lidar_max=1.0, speed=None, lateral=None, opp_gap=None, theta_noise=0.3, phase=True,
             crash=None, hold=None, opp_speed=None):
    """Observations [T, N, B+8] of N envs driving along the centerline: env e at speed[e] m/step (negative: backward)
    from step hold[e] on (standing still before), lateral offset lateral[e], the opponent opp_gap[e] m ahead (or driving
    on its own at opp_speed m/step); reset masks with a period and phase per env."""
    s_knots = _track_knots(xy)
    L = s_knots[-1]
    speed = rng.uniform(0.02, 0.3, N) if speed is None else np.asarray(speed, float)
    lateral = rng.uniform(-1.2, 1.2, N) if lateral is None else np.asarray(lateral, float)
    opp_gap = rng.uniform(-1.5, 1.5, N) if opp_gap is None else np.asarray(opp_gap, float)
    hold = np.zeros(N) if hold is None else np.asarray(hold, float)
    s0 = rng.uniform(0, L, N)
    obs = np.zeros((T, N, B + 8), np.float32)
    for t in range(T):
        s = s0 + speed * np.maximum(t - hold, 0)
        pe, th = pose_along(xy, s_knots, s, lateral * np.cos(0.1 * np.maximum(t - hold, 0)), closed)
        so = s + opp_gap if opp_speed is None else s0 + opp_gap + np.asarray(opp_speed, float) * t
        po, tho = pose_along(xy, s_knots, so, -0.5 * lateral, closed)
        obs[t, :, :B] = lidar(rng, N, B, lidar_max)
        obs[t, :, B + 0:B + 2] = pe
        obs[t, :, B + 2] = th
        obs[t, :, B + 4:B + 6] = po
        obs[t, :, B + 6] = tho + rng.uniform(-theta_noise, theta_noise, N) + 2 * np.pi * rng.integers(-2, 3, N)
        if crash is not None:
            obs[t, :, B + 3] = crash[t, :, 0]
            obs[t, :, B + 7] = crash[t, :, 1]
    period = rng.integers(7, 31, N) if phase else np.full(N, 10 ** 9)
    ph = rng.integers(0, 31, N)
    masks = np.array([[(t + ph[e]) % period[e] == 0 or t == 0 for e in range(N)] for t in range(T)], np.uint8)
    return obs, masks


def _widths(rng, n):
    return np.stack([rng.uniform(0.1, 2.0, n), rng.uniform(0.1, 2.0, n)], 1)


def _has(terms, key, pred):
    v = terms[..., T[key]]
    return bool(pred(v[~np.isnan(v)]).any())


def reward_cases():
    """The seeded reward scenarios; every one carries a check of the branches it was built to reach."""
    rng = np.random.default_rng(77)
    shanghai = H.reward_recording()['centerline'][:, :2]
    cases = []

    def add(name, xy, N, T, B=32, closed=True, widths=True, check=None, ep=None, **kw):
        cl = np.concatenate([xy, _widths(rng, len(xy))], 1) if widths else xy
        obs, masks = episodes(rng, xy, closed, N, T, B, lidar_max=kw.get('lidar_max', 1.0), **(ep or {}))
        cases.append(Case(name, cl, obs, masks, closed=closed, num_beams=B, check=check, **kw))

    def lat_both_sides(tm):
        assert _has(tm, 'e_t', lambda v: v > 0) and _has(tm, 'e_t', lambda v: v < 0)

    add('shanghai_widths', shanghai, 5, 40, B=1080, check=lat_both_sides,
        near_wall_dist=0.2, grace_steps_wall=1, grace_steps_opp=0, w_rel_lead=0.5, lead_clip=0.05, opp_safe_dist=2.0)
    cases[-1].check = lambda tm: (lat_both_sides(tm), _lead_clipped(tm, 0.5), _has(tm, 'r_wall', lambda v: v < 0),
                                  _has(tm, 'r_opp', lambda v: v < 0), _has(tm, 'r_flank', lambda v: v > 0),
                                  _has(tm, 'w_eff', lambda v: v == 0.2), _has(tm, 'w_eff', lambda v: v > 0.2))
    add('shanghai_2col', shanghai, 3, 30, B=1080, widths=False, default_half_width=0.7, lat_cap=0.5,
        check=lambda tm: _has(tm, 'w_eff', lambda v: v == 0.7) and _lat_capped(tm, 0.5))
    # backward driving flips at step 20; a stationary car (buf_sum == 0) does not; forward_sign -1
    add('open_s_curve', s_curve_xy(), 4, 45, closed=False, forward_sign=-1.0,
        ep=dict(speed=[-0.05, 0.0, 0.08, -0.2], lateral=[0.3, 0.0, 0.3, -0.3], phase=False),
        check=lambda tm: (_flipped(tm, [0, 3], [1, 2])))
    add('closed_seam', circle_xy(), 4, 60,
        ep=dict(speed=[0.9, -0.9, 0.75, 0.3], phase=False),
        check=lambda tm: _crosses_seam(tm, _track_knots(circle_xy())[-1]))
    # the direction flip is decided on the first 20 steps: env 0 stands still through step 20 and then drives forward
    # (buf_sum == 0: no flip), env 1 likewise and then backward (no flip either), env 2 moves backward at step 20 (flip);
    # the opponent drives on and w_rel_lead != 0, so a wrong flip shows in r_prog and r_lead
    add('hold20', circle_xy(), 3, 40, w_rel_lead=0.3, lead_clip=5.0,
        ep=dict(speed=[0.2, -0.2, -0.2], lateral=[0.0, 0.0, 0.0], hold=[20, 20, 18], opp_speed=[0.1, 0.15, 0.05], phase=False),
        check=lambda tm: (_flipped(tm, [2], [0, 1]), _has(tm, 'r_lead', lambda v: v != 0),
                          bool((tm[21:, 0, T['r_prog']] > 0).all()), bool((tm[21:, 1, T['r_prog']] < 0).all())))
    # one car, next to a one-midpoint last block (n - 1 = 193): its nearest midpoint is that one, the 4 others lie in a
    # block whose lower bound exceeds that midpoint's distance, and its projection belongs on segment 191, not 192.  Only
    # blocks of >= 5 midpoints may bound the 5th-nearest distance.
    k = np.arange(192)
    prune = np.concatenate([np.stack([-0.5 + 0.4 * np.cos(0.3 * k), 0.5 + 0.4 * np.sin(0.3 * k)], 1)[:-1],
                            [[0.0, 0.0], [10.0, 0.0], [10.0, 1.0]]])
    add('prune_last_block', prune, 1, 4, closed=False, ep=dict(phase=False),
        check=lambda tm: bool((tm[..., T['knn_ego0']] == 192).all() and (tm[..., T['knn_ego1']] == 191).all()
                              and (tm[..., T['seg']] == 191).all()))
    ob = cases[-1].obs
    B = cases[-1].num_beams
    ob[:, 0, B:B + 2] = (9.0, 0.6); ob[:, 0, B + 4:B + 6] = (9.5, 0.7)
    add('hairpin', hairpin_xy(), 6, 30, ep=dict(lateral=np.linspace(-0.4, 0.4, 6)),
        check=lambda tm: _knn_spread(tm))
    for n in (2, 3, 6, 7):
        xy = np.cumsum(np.random.default_rng(n).uniform(0.2, 1.0, (n, 2)), 0)
        add('short%d' % n, xy, 3, 24, closed=False, check=lambda tm, n=n: _knn_count(tm, min(5, n - 1)))
    for r in (0, 1, 4, 5):
        n = 64 * 3 + r + 1
        xy = np.stack([np.linspace(0, 100, n), 3 * np.sin(np.linspace(0, 6, n))], 1)
        # cars next to the last block: its midpoints are the ones with index >= 192
        add('tail%d' % r, xy, 4, 20, closed=False, ep=dict(speed=[0.0] * 4, lateral=[0.3, -0.3, 1.0, 0.0], phase=False),
            check=None)
        obs = cases[-1].obs
        B = cases[-1].num_beams
        obs[:, :, B + 0] = np.float32(99.9); obs[:, :, B + 4] = np.float32(100.5)
        cases[-1].check = lambda tm: _has(tm, 'knn_ego0', lambda v: v >= 190)
    # cars on lattice points and cell centres: at (c + 0.5, r + 0.5) the midpoints of rows r and r + 1 (driven in opposite
    # directions) tie at 0.5 and so do both projections, so the (distance, index) order alone decides e_s
    add('lattice', _lattice(), 8, 20, closed=False, ep=dict(phase=False), w_rel_lead=0.3,
        check=None)
    ob = cases[-1].obs
    B = cases[-1].num_beams
    lat = np.random.default_rng(3).integers(0, 12, (20, 8, 4)).astype(np.float32)
    lat[:, :4] += np.float32(0.5)                  # envs 0-3: both cars at cell centres
    lat[:, 4:, 2:] /= 2
    ob[:, :, B + 0], ob[:, :, B + 1], ob[:, :, B + 4], ob[:, :, B + 5] = lat[..., 0], lat[..., 1], lat[..., 2], lat[..., 3]
    cases[-1].check = lambda tm, ob=ob, B=B: _lattice_ties(tm, ob, B)
    # the same tie with both midpoints in one warp lane: on a 20-wide serpentine the segments of rows r and r + 1 at
    # column 3 are 2 * 20 - 2 - 2 * 3 = 32 apart (r even), so only a lane's own (distance, index) order separates them
    add('lattice_lane', _lattice(20), 4, 12, closed=False, ep=dict(phase=False), w_rel_lead=0.3, check=None)
    ob = cases[-1].obs
    B = cases[-1].num_beams
    r = 2 * np.random.default_rng(4).integers(0, 10, (12, 4, 2)).astype(np.float32)     # even rows run left to right
    ob[:, :, B + 0] = 3.5; ob[:, :, B + 1] = r[..., 0] + np.float32(0.5)
    ob[:, :, B + 4] = 12.5; ob[:, :, B + 5] = r[..., 1] + np.float32(0.5)
    cases[-1].check = lambda tm: bool((np.abs(tm[..., T['knn_ego1']] - tm[..., T['knn_ego0']]) == 32).all())
    # zero-length segments: a cluster of repeated points at the start, cars on it fall back to the nearest node
    dup = np.concatenate([np.zeros((6, 2)), np.stack([np.linspace(1, 30, 60), np.zeros(60)], 1)])
    dup = np.concatenate([dup[:30], dup[29:30], dup[30:]])                                   # and one in the middle
    add('duplicates', dup, 4, 20, closed=False, ep=dict(speed=[0.0, 0.1, 0.0, 0.2], lateral=[0.0, 0.3, 0.0, -0.3]), check=None)
    ob = cases[-1].obs
    B = cases[-1].num_beams
    ob[:, 0, B:B + 2] = 0.01; ob[:, 2, B + 4:B + 6] = -0.02
    cases[-1].check = lambda tm: _has(tm, 'fallback_ego', lambda v: v == 1) and _has(tm, 'fallback_opp', lambda v: v == 1)
    add('degenerate2', np.array([[1.0, 1.0], [1.0, 1.0]]), 2, 5, closed=False,
        check=lambda tm: _has(tm, 'fallback_ego', lambda v: v == 1))
    # crashes, bonus 0 and > 0, grace steps at 0, 1 and 25 with crash steps just before the boundaries
    for bonus, gw, go in ((0.0, 0, 1), (7.5, 1, 25), (50.0, 25, 0)):
        T_, N_ = 30, 4
        crash = np.zeros((T_, N_, 2), np.float32)
        crash[[3, 23, 24], 0, 0] = 1.0
        crash[[0, 24, 25], 1, 1] = 1.0
        crash[[23, 24], 2, :] = 1.0
        add('crash_b%g_g%d_%d' % (bonus, gw, go), shanghai, N_, T_, opp_crash_bonus=bonus, grace_steps_wall=gw,
            grace_steps_opp=go, near_wall_dist=0.5, opp_safe_dist=3.0, ep=dict(phase=False, crash=crash),
            check=lambda tm, bonus=bonus: (_has(tm, 'early', lambda v: v == 1),
                                           _has(tm, 'early', lambda v: v == 2) == (bonus > 0)))
    # flank boxes hit on their edges: oth = 0 (sincos exact), the ego at x_rel, y_rel on the box's edges
    edges = [(0.2, 0.25), (1.8, 0.8), (1.8, -0.25), (0.2, -0.8), (1.0, 0.525), (0.19999, 0.3), (1.0, 0.80001), (1.0, 0.0)]
    N_ = len(edges)
    obs = np.zeros((3, N_, 40), np.float32)
    obs[:, :, :32] = 0.5
    for e, (xr, yr) in enumerate(edges):
        obs[:, e, 32 + 4] = np.float32(5.0); obs[:, e, 32 + 5] = np.float32(1.0)
        obs[:, e, 32 + 0] = np.float32(5.0 + xr); obs[:, e, 32 + 1] = np.float32(1.0 + yr)
    cases.append(Case('flank_edges', np.concatenate([shanghai, _widths(rng, len(shanghai))], 1), obs, None, num_beams=32,
                      opp_safe_dist=1e-9, near_wall_dist=1e-9, check=lambda tm: _has(tm, 'r_flank', lambda v: v > 0)))
    # far off the track and NaN poses, lidar_max != 1
    add('off_track_nan', shanghai, 6, 12, B=33, lidar_max=4.5, near_wall_dist=1.0, check=None)
    ob = cases[-1].obs
    B = cases[-1].num_beams
    ob[:, 0, B:B + 2] = 1e4; ob[:, 1, B + 4] = np.nan; ob[5:, 2, B + 6] = np.nan; ob[:, 3, B + 1] = -np.inf
    cases[-1].check = lambda tm: _has(tm, 'fallback_opp', lambda v: v == 1)
    for B in (1, 2, 3, 31, 4097, 8192):
        add('beams%d' % B, shanghai, 3, 6, B=B, lidar_max=2.0, grace_steps_wall=0, near_wall_dist=1.5,
            wall_quantile=float(np.random.default_rng(B).choice([0.0, 0.05, 0.5, 1.0])),
            check=lambda tm: _has(tm, 'dmin', lambda v: v >= 0))
    add('batch4099', shanghai, 4099, 8, B=64, grace_steps_wall=2, grace_steps_opp=3, w_rel_lead=0.2, lead_clip=0.1,
        check=lambda tm: _lead_clipped(tm, 0.2))
    xy = np.stack([np.linspace(0, 2000, 16385), 5 * np.sin(np.linspace(0, 40, 16385))], 1)
    add('n16385', xy, 3, 6, closed=False, check=lambda tm: _has(tm, 'knn_ego0', lambda v: v >= 16380))
    B = cases[-1].num_beams
    cases[-1].obs[:, 0, B:B + 2] = xy[-2] + (0.05, 0.3)                 # next to the 256th block's midpoints
    return cases


def _lead_clipped(tm, w):
    r = tm[..., T['r_lead']]
    assert (r == w).any() and (r == -w).any(), 'lead clip not bound on both sides'


def _lat_capped(tm, cap):
    return bool((tm[..., T['r_lat']] == -0.35 * cap).any())


def _flipped(tm, flip_envs, keep_envs):
    f = tm[..., T['flip']]
    assert (f[25:, flip_envs] == -1).all() and (f[:19, flip_envs] == 1).all(), f[:, flip_envs]
    assert (f[:, keep_envs] == 1).all()


def _crosses_seam(tm, L):
    """Some car's consecutive arclengths jump by more than half a lap: it crossed s = 0 = L."""
    e_s = tm[..., T['e_s']]
    assert (np.abs(np.diff(e_s, axis=0)) > 0.5 * L).any()
    return True


def _knn_spread(tm):
    k = tm[..., T['knn_ego0']:T['knn_ego0'] + 5]
    spread = np.nanmax(k, -1) - np.nanmin(k, -1)
    return bool((spread > 100).any())


def _knn_count(tm, K):
    k = tm[..., T['knn_ego0']:T['knn_ego0'] + 5]
    k = k[~np.isnan(k[..., 0])]
    assert ((k >= 0).sum(-1) == K).all()
    return True


def _lattice_ties(tm, obs, B):
    """Lattice cars sit at exactly equal distances from several midpoints: the 5th neighbour ties with a 6th for some."""
    xy = _lattice()
    mid = (xy[:-1] + xy[1:]) * 0.5
    ties = 0
    for t in range(len(obs)):
        for e in range(obs.shape[1]):
            p = obs[t, e, B:B + 2].astype(np.float64)
            d2 = np.sort((mid[:, 0] - p[0]) ** 2 + (mid[:, 1] - p[1]) ** 2)
            ties += d2[4] == d2[5]
    assert ties > 10, ties
    centre = (obs[:, :, B:B + 2] % 1 == 0.5).all(-1) & (obs[:, :, B:B + 2] < 11).all(-1)
    k = tm[..., T['knn_ego0']:T['knn_ego0'] + 2][centre]
    assert (np.abs(k[:, 1] - k[:, 0]) > 1).sum() > 10, k                 # the two nearest: midpoints of two rows
    return True


def check_branches(c, tm):
    """Assert that case c's oracle breakdown tm [T, N, terms] reaches the branches the case was built for."""
    if c.check is None:
        return
    res = c.check(tm)
    assert all(x is not False for x in (res if isinstance(res, tuple) else (res,))), (c.name, res)


def test_reward_cases_reach_their_branches():
    """Each constructed case drives the oracle down the branch it was built for (e.g. the flip at step 20, the fallback
    projection, the lead clip on both sides, the early returns), so no case quietly misses its purpose."""
    seen = {}
    for c in reward_cases():
        tot, tm = c.oracle_run()
        check_branches(c, tm)
        for k in ('r_wall', 'r_opp', 'r_flank', 'r_lead'):
            seen[k] = seen.get(k, False) or _has(tm, k, lambda v: v != 0)
        seen['early1'] = seen.get('early1', False) or _has(tm, 'early', lambda v: v == 1)
        seen['early2'] = seen.get('early2', False) or _has(tm, 'early', lambda v: v == 2)
        seen['nan_total'] = seen.get('nan_total', False) or bool(np.isnan(tot).any())
    assert all(v for k, v in seen.items() if k != 'nan_total'), seen
