"""A numpy model of the post kernel's ray-cast work list, checked against the CPU oracle's ray_cast (no GPU).

The opponent ray-cast of post_kernel (f110_kernels.cu, stages B-D) does not walk the reference's window of beams
(get_blocked_view_indices, laser_models.py:282-315) but only the beams of that window that lie within
alpha = asin(R / dist) + 1e-6 of the bearing of the opponent's bounding circle, or of the opposite bearing (the collinear
fallback of get_range can lower a beam that points straight away from an edge), each interval widened by one beam.  The
model below forms the same list in the same way -- the four vertex beams with nearest_beam's semantics, the window, the
forward and backward cones, their clip to the window and their merge -- and the test asserts that every beam the oracle's
ray_cast lowers (from an all-inf scan) is on it.  The window itself is the kernel's shortcut
yaw - atan2(vy, vx) for the reference's atan2(sin yaw, cos yaw) - atan2(uy, ux); the two agree except where a vertex angle
lies within an ulp or so of the midpoint between two beams, and those near-ties are counted.  A GPU mismatch of the
ray-cast on these inputs (tests/test_post_kernel.py) is then a kernel fault, not a hole in the pruning argument.
"""
import bisect
import math

import numpy as np
import pytest

from tests import helpers as H

# the window edge's angle is this close to the midpoint of two beams: the kernel's atan2 shortcut may pick the other beam
TIE_RAD = 1e-12


def nearest_beam(angles, a):
    """np.argmin(np.abs(angles - a)) over a strictly increasing table (first minimum); NaN -> 0."""
    if a != a:
        return 0
    k = bisect.bisect_left(angles, a)
    if k <= 0:
        return 0
    if k >= len(angles):
        return len(angles) - 1
    return k - 1 if abs(angles[k - 1] - a) <= abs(angles[k] - a) else k


def near_tie(angles, a):
    """a within TIE_RAD of the midpoint between two neighbouring beams."""
    if a != a:
        return False
    k = bisect.bisect_left(angles, a)
    for j in (k - 1, k):
        if 0 < j < len(angles) and abs(a - 0.5 * (angles[j - 1] + angles[j])) <= TIE_RAD:
            return True
    return False


def vertices(pose, length, width):
    """get_vertices (collision_models.py:218-260) in libm's trig: order rl, rr, fr, fl."""
    c, s = math.cos(pose[2]), math.sin(pose[2])
    out = []
    for hx, hy in ((-length / 2, width / 2), (-length / 2, -width / 2), (length / 2, -width / 2), (length / 2, width / 2)):
        out.append((c * hx + -s * hy + pose[0], s * hx + c * hy + pose[1]))
    return out


def _wrap(ang):
    if ang > math.pi:
        return ang - 2 * math.pi
    if ang < -math.pi:
        return ang + 2 * math.pi
    return ang


def reference_vertex_angles(pose, verts):
    """-angle of get_blocked_view_indices for each vertex (NaN where the vertex is the observer's position)."""
    ex, ey = math.cos(pose[2]), math.sin(pose[2])
    out = []
    for vx, vy in verts:
        dx, dy = vx - pose[0], vy - pose[1]
        norm = math.sqrt(dx * dx + dy * dy)
        if norm == 0.0:
            out.append(math.nan)
            continue
        out.append(-_wrap(math.atan2(ey, ex) - math.atan2(dy / norm, dx / norm)))
    return out


def kernel_vertex_angles(pose, verts):
    """stage B's vertex angle: yaw - atan2(vy, vx), NaN for a vertex at the observer."""
    out = []
    for vx, vy in verts:
        dx, dy = vx - pose[0], vy - pose[1]
        out.append(math.nan if dx == 0.0 and dy == 0.0 else -_wrap(pose[2] - math.atan2(dy, dx)))
    return out


def window(angles, vertex_angles):
    ind = [nearest_beam(angles, a) for a in vertex_angles]
    return min(ind), max(ind)


def work_list(angles, fov, pose, opp_pose, length, width):
    """The beams stage D visits for one observer (pose = ray-cast origin) and one opponent (its pose before iTTC zeroing),
    with the observer's length / width: -> (window (lo, hi), list of (first, last) beam intervals)."""
    B = len(angles)
    verts = vertices(opp_pose, length, width)
    lo, hi = window(angles, kernel_vertex_angles(pose, verts))
    R = 0.5 * math.sqrt(length * length + width * width) * (1.0 + 1e-9) + 1e-9
    dx, dy = opp_pose[0] - pose[0], opp_pose[1] - pose[1]
    dist = math.sqrt(dx * dx + dy * dy)
    f0, f1, b0, b1 = 0, B - 1, B, -1
    alpha = math.asin(R / dist) + 1e-6 if dist >= R else math.nan
    cone_max = min(0.75, math.pi - 0.5 * fov - 0.01)
    if dist > R * (1.0 + 1e-6) and alpha < cone_max:
        phi = _wrap(math.atan2(dy, dx) - pose[2])
        back = phi - math.pi if phi > 0. else phi + math.pi
        amin, amax = angles[0], angles[-1]
        if phi + alpha < amin or phi - alpha > amax:
            f0, f1 = B, -1
        else:
            f0, f1 = nearest_beam(angles, phi - alpha) - 1, nearest_beam(angles, phi + alpha) + 1
        if not (back + alpha < amin or back - alpha > amax):
            b0, b1 = nearest_beam(angles, back - alpha) - 1, nearest_beam(angles, back + alpha) + 1
    f0, f1, b0, b1 = max(lo, f0), min(hi, f1), max(lo, b0), min(hi, b1)
    if b0 <= f1 and f0 <= b1:
        f0, f1, b0, b1 = min(f0, b0), max(f1, b1), B, -1
    return (lo, hi), [(i0, i1) for i0, i1 in ((f0, f1), (b0, b1)) if i1 >= i0]


def in_items(items, i):
    return any(i0 <= i <= i1 for i0, i1 in items)


def oracle_for(B, fov):
    from oracle.f110_oracle import Oracle
    return Oracle(1, 2, num_beams=B, fov=fov)


def geometries(rng, B, fov, angles, n):
    """(observer pose, opponent pose, length, width): random pairs at every distance and bearing, and constructed ones --
    straight behind, on the fov edges, overlapping and identical cars, a vertex at the observer, the collinear fallback
    both ways, far and beyond max_range."""
    out = []
    for _ in range(n):
        L, W = rng.uniform(0.2, 1.2), rng.uniform(0.1, 0.8)
        ego = (rng.uniform(-5, 5), rng.uniform(-5, 5), rng.uniform(-math.pi, math.pi))
        kind = rng.integers(0, 6)
        if kind == 0:       # anywhere, log-uniform distance
            d, bear = math.exp(rng.uniform(math.log(0.05), math.log(40.0))), rng.uniform(-math.pi, math.pi)
        elif kind == 1:     # behind, within a cone's width of straight behind
            d, bear = rng.uniform(0.3, 6.0), math.pi + rng.uniform(-0.5, 0.5)
        elif kind == 2:     # straddling +-fov/2
            d, bear = rng.uniform(0.3, 6.0), rng.choice([-1, 1]) * fov / 2 + rng.uniform(-0.3, 0.3)
        elif kind == 3:     # overlapping
            d, bear = rng.uniform(0.0, 0.6), rng.uniform(-math.pi, math.pi)
        elif kind == 4:     # near the bounding circle
            R = 0.5 * math.hypot(L, W)
            d, bear = R * (1 + rng.choice([-1e-6, 0.0, 1e-7, 2e-6, 1e-3])), rng.uniform(-math.pi, math.pi)
        else:               # cones that overlap: wide fov, close and to the side
            d, bear = rng.uniform(0.35, 1.0), rng.choice([-1, 1]) * rng.uniform(1.2, 1.9)
        th = ego[2] + bear
        opp = (ego[0] + d * math.cos(th), ego[1] + d * math.sin(th), rng.choice([0.0, rng.uniform(-math.pi, math.pi)]))
        out.append((ego, opp, L, W))
    L, W = 0.58, 0.31
    out.append(((1.0, 2.0, 0.3), (1.0, 2.0, 0.3), L, W))                # identical poses
    out.append(((0.0, 0.0, 0.7), (L / 2, -W / 2, 0.0), L, W))            # vertex rl exactly at the observer
    out.append(((0.0, 0.0, 0.0), (45.0, 0.0, 0.0), L, W))                # beyond max_range
    out.append(((0.0, 0.0, 0.0), (25.0, 0.3, 1.0), L, W))               # far, tiny cone
    out += [g for i in range(B // 2 - 8, B // 2 + 8) for g in collinear_geometries(angles, i, L, W)]
    return out


def collinear_geometries(angles, i, L=0.58, W=0.31):
    """Observer at the origin with yaw y, y + angles[i] == -pi/2 exactly, so beam i points along -y with
    (cos, sin)(theta + pi/2) == (1, 0); an opponent with yaw 0 whose rear edge lies exactly on the line x = 0, above the
    observer (beam i points away from it: only the backward cone holds beam i) and below it (along the beam), each also
    moved 1e-9 m off the line, inside get_range's 1e-8 collinearity tolerance.  [] when no such yaw exists for beam i."""
    y = -math.pi / 2 - angles[i]
    for _ in range(8):
        if wrap_yaw(y) == y and y + angles[i] == -math.pi / 2:
            break
        y = math.nextafter(y, -math.inf if y + angles[i] > -math.pi / 2 else math.inf)
    else:
        return []
    out = []
    for sy in (1.0, -1.0):
        px = L / 2
        while -L / 2 + px != 0.0:
            px = math.nextafter(px, math.inf if -L / 2 + px < 0 else -math.inf)
        for shift in (0.0, 1e-9):
            out.append(((0.0, 0.0, y), (px + shift, sy, 0.0), L, W))
    return out


def wrap_yaw(a):
    """The dynamics' post clamp of the yaw (base_classes.py:408): Python's float modulo, as numpy scalars do it."""
    m = math.fmod(a + math.pi, 2 * math.pi)
    if m != 0.0:
        if m < 0.0:
            m += 2 * math.pi
    else:
        m = 0.0
    return m - math.pi


CASES = [(32, 4.7), (541, 4.7), (1080, 4.7), (1080, 6.2), (1080, 1.0), (2049, 4.7), (4320, 6.2), (541, 1.0)]


@pytest.mark.parametrize('B,fov', CASES)
def test_work_list_covers_every_lowered_beam(B, fov):
    o = oracle_for(B, fov)
    angles = list(o.get_beam_tables()[0])
    rng = np.random.default_rng(B * 10 + int(fov * 10))
    geos = geometries(rng, B, fov, angles, 12000)
    inf = np.full(B, np.inf)
    lowered = ties = window_ties = pruned = 0
    for ego, opp, L, W in geos:
        from_ref = o.ray_cast(np.array(ego), inf, o.get_vertices(np.array(opp), L, W))
        hit = np.flatnonzero(from_ref < np.inf)
        (lo, hi), items = work_list(angles, fov, ego, opp, L, W)
        verts = vertices(opp, L, W)
        ref_lo, ref_hi = window(angles, reference_vertex_angles(ego, verts))
        tie = any(near_tie(angles, a) for a in reference_vertex_angles(ego, verts) + kernel_vertex_angles(ego, verts))
        ties += tie
        if (lo, hi) != (ref_lo, ref_hi):
            assert tie, ('window differs from the reference without a near-tie', ego, opp, L, W, (lo, hi), (ref_lo, ref_hi))
            window_ties += 1
        missed = [i for i in hit if not in_items(items, i)]
        if missed:
            assert tie and all(i in (lo, hi, ref_lo, ref_hi) for i in missed), \
                ('lowered beam outside the work list', ego, opp, L, W, missed[:5], items, (lo, hi))
        lowered += len(hit)
        pruned += (hi - lo + 1) - sum(i1 - i0 + 1 for i0, i1 in items)
    print('B %d fov %.1f: %d geometries, %d beams lowered, %d beams of the windows pruned, near-ties %d (windows moved %d)'
          % (B, fov, len(geos), lowered, pruned, ties, window_ties))
    assert window_ties <= 1e-3 * len(geos)
    assert lowered > 0 and (pruned > 0 or fov > 6.0)


@pytest.mark.parametrize('i', range(540, 550))
def test_collinear_fallback_lowers_the_beam_pointing_away(i):
    """The recipe of the backward cone: the reference lowers beam i, which points straight away from the opponent, to
    1 - W/2 and nothing else; the work list holds beam i only through its backward cone."""
    o = oracle_for(1080, 4.7)
    angles = list(o.get_beam_tables()[0])
    geos = collinear_geometries(angles, i)
    assert geos, i
    for ego, opp, L, W in geos:
        ray = o.ray_cast(np.array(ego), np.full(1080, np.inf), o.get_vertices(np.array(opp), L, W))
        hit = np.flatnonzero(ray < np.inf)
        (lo, hi), items = work_list(angles, 4.7, ego, opp, L, W)
        if opp[1] > 0:
            assert list(hit) == [i] and abs(ray[i] - (1 - W / 2)) < 1e-8, (hit, ray[hit])
            assert (lo, hi) == (0, 1079)
            assert len(items) == 1 and items[0][0] <= i <= items[0][1] and items[0][1] - items[0][0] < 200, items
        else:
            assert i in hit and abs(ray[i] - (1 - W / 2)) < 1e-8
        assert all(in_items(items, k) for k in hit)
