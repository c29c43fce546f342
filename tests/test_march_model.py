"""A numpy model of the lidar kernel's guarded fixed-point march, checked against the CPU oracle (no GPU).

The kernel's correctness argument (f110_kernels.cu, the comment on the march above lidar_kernel, and the loop in
f110_lidar_body.cuh) is that every lookup whose fixed-point fraction clears the guard band addresses exactly the cell the
reference's world-frame arithmetic addresses, so a ray that is decided on the fast path has the reference's distance bit
for bit; everything else (guard band, sentinel, non-finite coordinates) is redone in the reference's own arithmetic.  The
model below performs the same operations in the same order as the kernel -- the scan head of dynamics_kernel, the direction
table of f110_capi.cu direction_table, __double2uint_rz, the guard mask, the padded index and its -1 sentinels -- and the
test asserts that every ray it decides on the fast path equals the oracle's scan.  The library is built with -fmad=false,
so numpy's separately rounded products and sums are the kernel's.  A GPU mismatch on these inputs is then a kernel,
dispatch or compile fault, not a hole in the argument.

The argument has a limit this model shows: the reference marches in world coordinates, and each of its steps rounds the
car's world position by up to half an ulp of it.  That rounding must stay far below one fixed-point unit (res / 2^fb).
Near the world origin it is negligible; with a map placed 1e9 m from the world origin, half an ulp is 6e-8 m, which on a
200-cell map at 0.05 m (24 fraction bits) is 20 units per step, ten times the guard band, and the model then finds fast
rays one cell (0.05 m) off the reference.  The origins checked here go up to 3e7 m.
"""
import numpy as np
import pytest

from tests import helpers as H

B = 1080


def march_model(dt, res, origin, poses, fb, eps=1e-4, max_range=30.0, guard=2):
    """-> [len(poses), B] scans of the rays the fast march decides (NaN for the ones it hands to the exact path)."""
    Hm, Wm = dt.shape
    gm = ((1 << fb) - 1) & ~(2 * guard - 1)
    fx_off = float(1 << fb) - guard
    inv_fx = (1.0 / res) * float(1 << fb)
    oc, os_ = np.cos(origin[2]), np.sin(origin[2])
    sines, cosines = H.tables()[:2]
    theta_inc = H.THETA_DIS * (H.FOV / (B - 1)) / (2 * np.pi)
    out = np.full((len(poses), B), np.nan)
    for p, (x, y, th) in enumerate(poses):
        # the reference's running theta index (laser_models.py:174-184)
        t = np.fmod(H.THETA_DIS * (th - H.FOV / 2.) / (2. * np.pi), H.THETA_DIS)
        while t < 0:
            t += H.THETA_DIS
        ti = np.empty(B, np.int64)
        for i in range(B):
            ti[i] = int(t)
            t += theta_inc
            while t >= H.THETA_DIS:
                t -= H.THETA_DIS
        cs, sn = cosines[ti], sines[ti]
        DX = (cs * oc + sn * os_) * inv_fx
        DY = (-cs * os_ + sn * oc) * inv_fx
        xt, yt = x - origin[0], y - origin[1]
        X = np.full(B, (xt * oc + yt * os_) * inv_fx + fx_off)
        Y = np.full(B, (-xt * os_ + yt * oc) * inv_fx + fx_off)
        total = np.zeros(B)
        alive = np.ones(B, bool)
        fast = np.ones(B, bool)
        while alive.any():
            # __double2uint_rz: NaN and negative -> 0, beyond 2^32 - 1 -> 2^32 - 1
            ux = np.clip(np.nan_to_num(X, nan=0.0), 0, 4294967295.0).astype(np.uint64)
            uy = np.clip(np.nan_to_num(Y, nan=0.0), 0, 4294967295.0).astype(np.uint64)
            decided = ((~ux & gm) != 0) & ((~uy & gm) != 0)
            r, c = (uy >> fb).astype(np.int64) - 1, (ux >> fb).astype(np.int64) - 1     # the map sits one cell in
            inside = (r >= 0) & (r < Hm) & (c >= 0) & (c < Wm)
            d = np.where(inside, dt[np.clip(r, 0, Hm - 1), np.clip(c, 0, Wm - 1)], -1.0)   # sentinel outside
            handed_over = alive & (~decided | (d < 0))
            fast &= ~handed_over
            alive &= ~handed_over
            total = np.where(alive, total + d, total)
            alive &= (d > eps) & (total <= max_range)
            X = np.where(alive, X + d * DX, X)
            Y = np.where(alive, Y + d * DY, Y)
        out[p] = np.where(fast, np.minimum(total, max_range), np.nan)
    return out


def _oracle_scans(dt, res, origin, poses):
    from oracle.f110_oracle import Oracle
    o = Oracle(1, 1)
    o.set_map_arrays(dt, res, origin)
    return np.stack([o.scan(p)[0] for p in poses])


def _check(dt, res, origin, poses, fb):
    want = _oracle_scans(dt, res, origin, poses)
    got = march_model(dt, res, origin, poses, fb)
    fast = ~np.isnan(got)
    bad = fast & (got.view(np.int64) != want.view(np.int64))
    assert not bad.any(), ("fast-path rays differ from the oracle", int(bad.sum()), np.argwhere(bad)[:5])
    return fast.mean()


def test_synthetic_yaws_are_libm_exact():
    import math
    for y in H.SYNTH_YAWS:
        assert np.cos(y) == math.cos(y) and np.sin(y) == math.sin(y), y


@pytest.mark.parametrize('name', sorted(H.SYNTH_MAPS))
def test_fast_march_equals_oracle_at_every_width(name):
    _, dt, res, origin = H.synthetic_map(name)
    frac = _check(dt, res, origin, H.synthetic_poses(name), H.fraction_bits(max(dt.shape)))
    assert frac > 0.2, frac       # not vacuous: poses outside the map and in walls hand every ray over


@pytest.mark.parametrize('shift', [0.0, 1e4, 1e5, 1e6, 5e6, 3e7])
@pytest.mark.parametrize('yaw', [0.0, 0.3, 2.5])
def test_fast_march_far_from_the_world_origin(shift, yaw):
    """A map moved and rotated far from the world origin, marched at the narrowest width (17 fraction bits) and at its own."""
    _, dt, res, origin = H.synthetic_map('w24_200')
    org = (origin[0] + shift, origin[1] - shift, yaw)
    # the same map-frame points, cell corners among them, placed through the moved origin
    m = np.array([(40 * res, 20 * res), (40.5 * res, 20 * res), (150.3 * res, 24.6 * res), (3 * res, 3 * res),
                  (60.7 * res, 10.2 * res)])
    co, so = np.cos(yaw), np.sin(yaw)
    poses = np.stack([org[0] + co * m[:, 0] - so * m[:, 1], org[1] + so * m[:, 0] + co * m[:, 1],
                      yaw + np.array([0.0, 1.0, -2.0, 0.7, 2.2])], 1)
    for fb in (17, H.fraction_bits(max(dt.shape))):
        assert _check(dt, res, org, poses, fb) > 0.2
