"""Shared test helpers: golden fixture access (nothing here touches /root/reference)."""
import functools
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@functools.lru_cache(maxsize=None)
def load(name):
    return dict(np.load(os.path.join(GOLDEN, name + '.npz')))


@functools.lru_cache(maxsize=None)
def golden_map(name):
    """-> (dt fp64 [H,W], resolution, origin[3]) rebuilt from the packed occupancy exactly as
    laser_models.py:398-425 does (255/0 image -> scipy EDT -> * resolution)."""
    from scipy.ndimage import distance_transform_edt
    m = load('maps')
    shape = tuple(int(v) for v in m[name + '__shape'])
    free = np.unpackbits(m[name + '__bits'])[:shape[0] * shape[1]].reshape(shape).astype(bool)
    img = np.where(free, 255., 0.)
    res = float(m[name + '__resolution'])
    return res * distance_transform_edt(img), res, [float(v) for v in m[name + '__origin']]


LARGE_MAPS = ('levine', 'Shanghai_x2', 'Shanghai_x4', 'Shanghai_x2_rot')


@functools.lru_cache(maxsize=2)
def large_map(name):
    """BASELINE config C4 'large maps' -> (dt fp64 [H,W], resolution, origin[3], poses, reference scans).
    levine (2048 x 2048) comes packed in maps_large.npz; Shanghai_x2 / _x4 / _x2_rot are rebuilt from the Shanghai bits by
    pixel replication (np.kron), exactly what make_golden.py wrote to disk for the reference (resolution / k)."""
    from scipy.ndimage import distance_transform_edt
    g = load('scans_large')
    if name == 'levine':
        m = load('maps_large')
        shape = tuple(int(v) for v in m['levine__shape'])
        free = np.unpackbits(m['levine__bits'])[:shape[0] * shape[1]].reshape(shape).astype(bool)
        res, origin = float(m['levine__resolution']), [float(v) for v in m['levine__origin']]
    else:
        m = load('maps')
        shape = tuple(int(v) for v in m['Shanghai_map__shape'])
        free = np.unpackbits(m['Shanghai_map__bits'])[:shape[0] * shape[1]].reshape(shape).astype(bool)
        k = int(name.split('_x')[1][0])
        free = np.kron(free, np.ones((k, k), bool))
        res, origin = float(g[name + '__resolution']), [float(v) for v in g[name + '__origin']]
    dt = res * distance_transform_edt(np.where(free, 255., 0.))
    probe = g[name + '__dt_probe']
    assert dt[-1, -1] == probe[0] and dt[0, 0] == probe[1] and dt.max() == probe[2], "EDT differs from the reference's"
    return dt, res, origin, g[name + '__poses'], g[name + '__scans']


def write_map_files(name, directory):
    """Materialise a golden map as <directory>/<name>.yaml + .png (the reference's on-disk format)."""
    from PIL import Image
    m = load('maps')
    shape = tuple(int(v) for v in m[name + '__shape'])
    free = np.unpackbits(m[name + '__bits'])[:shape[0] * shape[1]].reshape(shape).astype(bool)
    img = np.where(free, 254, 0).astype(np.uint8)[::-1]       # undo FLIP_TOP_BOTTOM
    Image.fromarray(img, mode='L').save(os.path.join(directory, name + '.png'))
    o = m[name + '__origin']
    with open(os.path.join(directory, name + '.yaml'), 'w') as f:
        f.write("image: %s.png\nresolution: %r\norigin: [%r, %r, %r]\nnegate: 0\noccupied_thresh: 0.45\nfree_thresh: 0.196\n"
                % (name, float(m[name + '__resolution']), float(o[0]), float(o[1]), float(o[2])))
    return directory + '/', name


def tables():
    m = load('maps')
    return m['sines'], m['cosines'], m['scan_angles'], m['beam_cosines'], m['side_distances']


FOV, THETA_DIS = 4.7, 2000
# Yaws whose np.cos / np.sin equal libm's: the handle gets the origin's cos / sin from numpy, the oracle from libm
SYNTH_YAWS = (0.0, 0.3, np.pi / 2, -1.5708, np.pi, 2.5)
# Thin synthetic maps at both ends of every fixed-point width of the lidar kernel's march, 32 - bit_length(side + 1)
# capped at 24 (f110_capi.cu fixed_point_format): name -> (long side, short side, resolution, long side vertical, origin)
SYNTH_MAPS = {
    'w24_200': (200, 48, 0.05, False, (-3.0, 2.0, 0.0)),
    'w23_254': (254, 64, 0.1, True, (4.5e5, 5.4e6, 0.3)),
    'w22_511': (511, 48, 0.025, False, (-12.0, -1.0, np.pi / 2)),
    'w22_1022': (1022, 80, 0.04, True, (100.0, -250.0, -1.5708)),
    'w21_1500': (1500, 96, 0.05, False, (4.5e5, 5.4e6, np.pi)),
    'w20_4094': (4094, 56, 0.05, False, (-40.0, 7.5, 2.5)),
    'w19_4095': (4095, 48, 0.1, True, (0.0, 0.0, 0.0)),
    'w19_8190': (8190, 64, 0.025, False, (4.5e5, 5.4e6, 0.3)),
    'w18_8191': (8191, 48, 0.05, True, (-7.0, 3.0, np.pi / 2)),
    'w17_16383': (16383, 48, 0.1, False, (4.5e5, 5.4e6, 2.5)),
    'w17_20000': (20000, 48, 0.03, True, (-1.0e3, 2.0e3, np.pi)),
}


def fraction_bits(side):
    """The lidar march's fixed-point fraction bits for a map (or map set) whose larger side is `side` cells."""
    return min(24, 32 - int(side + 1).bit_length())


@functools.lru_cache(maxsize=None)
def synthetic_map(name):
    """-> (free mask bool [H, W], dt fp64 [H, W] = resolution * scipy EDT, resolution, origin).  Border walls with a gap in
    the far end wall (rays leave the map through it), boxes and single-cell obstacles in the first 40 % of the long axis,
    and a free run after them (rays reach max_range where the map is long enough)."""
    from scipy.ndimage import distance_transform_edt
    side, thick, res, vertical, origin = SYNTH_MAPS[name]
    rng = np.random.default_rng(side)
    free = np.ones((thick, side), bool)
    free[0, :] = free[-1, :] = free[:, 0] = free[:, -1] = False
    free[thick // 3:2 * thick // 3, -1] = True
    region = max(8, int(0.4 * side))
    for _ in range(max(2, side // 150)):
        h, w = rng.integers(2, thick // 4), rng.integers(2, 12)
        r, c = rng.integers(2, thick - 2 - h), rng.integers(2, region - w)
        free[r:r + h, c:c + w] = False
    for _ in range(max(4, side // 60)):
        free[rng.integers(2, thick - 2), rng.integers(2, region)] = False
    if vertical:
        free = np.ascontiguousarray(free.T)
    dt = res * distance_transform_edt(np.where(free, 255., 0.))
    return free, dt, res, tuple(origin)


def synthetic_poses(name, n_free=6, seed=0):
    """World-frame poses [n, 3] on synthetic map `name`: exact cell corners and edge midpoints in the map frame, free cells,
    an obstacle cell, the map border, outside the map on every side and beyond the far corner, and headings on exact
    theta-table indices; yaws from SYNTH_YAWS otherwise."""
    free, _, res, origin = synthetic_map(name)
    H, W = free.shape
    rng = np.random.default_rng(seed)
    ok = free.copy()
    ok[:-1] &= free[1:]; ok[:, :-1] &= free[:, 1:]; ok[1:] &= free[:-1]; ok[:, 1:] &= free[:, :-1]
    cells = np.argwhere(ok)
    pick = cells[rng.integers(0, len(cells), n_free)]
    m = []                                             # map-frame (x, y)
    for k, (r, c) in enumerate(pick):
        m.append((c * res, r * res) if k % 3 == 0 else (c * res + 0.5 * res, r * res) if k % 3 == 1 else
                 (c * res + rng.uniform(0, res), r * res + rng.uniform(0, res)))
    occ = np.argwhere(~free[1:-1, 1:-1]) + 1
    r, c = occ[len(occ) // 2]
    m.append(((c + 0.5) * res, (r + 0.5) * res))       # inside an obstacle
    m += [(0.0, H * res / 2), (W * res / 2, 0.0), (0.5 * res, 0.5 * res)]          # on the border
    m += [(-0.5, H * res / 2), (W * res + 0.5, H * res / 2), (W * res / 2, -0.5), (W * res / 2, H * res + 0.5),
          (W * res + 1.0, H * res + 1.0)]              # outside, every side, and beyond the far corner
    yaws = [SYNTH_YAWS[k % len(SYNTH_YAWS)] for k in range(len(m))]
    # the free run, looking along the long axis towards the gap in the end wall: from its start and from near its end
    for f in (0.42, 0.97):
        m.append((f * W * res, (H / 2 + 0.25) * res) if W > H else ((W / 2 + 0.25) * res, f * H * res))
        yaws.append(0.0 if W > H else np.pi / 2)
    m, yaws = np.array(m, np.float64), np.array(yaws)
    co, so = np.cos(origin[2]), np.sin(origin[2])
    out = np.stack([origin[0] + co * m[:, 0] - so * m[:, 1], origin[1] + so * m[:, 0] + co * m[:, 1], yaws + origin[2]], 1)
    # headings on exact theta-table indices: theta_dis * (yaw - fov / 2) / (2 pi) an integer
    out[1::4, 2] = FOV / 2 + 2 * np.pi * rng.integers(0, THETA_DIS, len(out[1::4])) / THETA_DIS
    return out


def noise_stream(seed, steps, beams=1080, expect_sha=None):
    """The reference's lidar noise: one Generator.normal(0, 0.01, beams) per agent per step, every agent
    seeded identically (base_classes.py:204, laser_models.py:450-452) -> [steps, beams]."""
    rng = np.random.default_rng(seed)
    out = np.stack([rng.normal(0., 0.01, size=beams) for _ in range(steps)])
    if expect_sha is not None:
        got = hashlib.sha256(out.tobytes()).hexdigest()
        assert got == str(expect_sha), "numpy PCG64 normal stream differs from the one the golden rollout was recorded with"
    return out


@functools.lru_cache(maxsize=None)
def reward_recording():
    """reward.npz with its flat observations 'obs' [T, 1088] f32.  The file keeps what the recorded reference rollout was
    driven with (start poses per episode, the actions applied, the lidar noise seed) and the SHA-256 of every observation
    the reference returned; the oracle, whose env reproduces the reference's bit for bit (test_env_rollouts), replays the
    rollout here and every observation must hash to the recorded one."""
    from oracle.f110_oracle import Oracle
    g = dict(load('reward'))
    o = Oracle(1, 2)
    s, c, a, bc, sd = tables()
    o.set_tables(s, c)
    o.set_beam_tables(a, bc, sd)
    o.set_map_arrays(*golden_map('Shanghai_map'))
    obs, episode = [], -1
    for k in range(len(g['actions'])):
        if g['episode_start'][k]:
            # F110Env.reset restarts the noise stream of every agent and draws one scan (the reset observation)
            episode += 1
            rng = np.random.default_rng(int(g['seed']))
            nz = rng.normal(0., 0.01, size=1080)
            o.reset(g['poses'][episode][None], noise=np.stack([nz, nz])[None])
        nz = rng.normal(0., 0.01, size=1080)
        ob = np.array(o.step(g['actions'][k][None], noise=np.stack([nz, nz])[None])['obs'][0], np.float32)   # a copy
        assert hashlib.sha256(ob.tobytes()).digest() == g['obs_sha256'][k].tobytes(), \
            ("replayed observation differs from the reference's", k)
        obs.append(ob)
    g['obs'] = np.stack(obs)
    return g


ROLLOUT_MAP = {
    'rollout_c2_shanghai': 'Shanghai_map', 'rollout_const_shanghai': 'Shanghai_map',
    'rollout_circles_open': 'open_square', 'rollout_headon_open': 'open_square',
    'rollout_three_euler_open': 'open_square', 'rollout_corridor': 'straight_corridor',
}
ROLLOUT_KW = {'rollout_three_euler_open': dict(integrator=2, lidar_dist=0.275, ego_idx=1)}


def compare_rollout(name, make_backend, state_tol, scan_tol, scan_frac=0.999, obs_tol=None):
    """Replay a golden F110Env rollout through `make_backend(num_agents, map_name, **kw)` which must return
    an object with .reset(poses[1,A,3], noise[1,A,B]) and .step(actions[1,A,2], noise) -> dict of numpy
    arrays (state, collisions, terminated, toggles, lap_times, lap_counts, time, scans, obs).
    Flags must match bit-exactly; returns a summary dict."""
    g = load(name)
    T, A = g['actions'].shape[0], g['actions'].shape[1]
    nz = noise_stream(int(g['seed']), T + 1, expect_sha=g['noise_sha256'])
    be = make_backend(A, ROLLOUT_MAP[name], **ROLLOUT_KW.get(name, {}))
    every = int(g['every'])
    worst_state, worst_scan, outliers, beams, worst_obs = 0.0, 0.0, 0, 0, 0.0
    for k in range(T + 1):
        noise = np.broadcast_to(nz[k], (1, A, nz.shape[1]))
        out = be.reset(g['poses'][None], noise) if k == 0 else be.step(g['actions'][k - 1][None], noise)
        assert np.array_equal(out['collisions'][0], g['collisions'][k]), (name, 'collisions', k)
        assert bool(out['terminated'][0]) == bool(g['terminated'][k]), (name, 'terminated', k)
        assert np.array_equal(out['toggles'][0], g['toggles'][k]), (name, 'toggles', k)
        assert np.array_equal(out['lap_counts'][0], g['lap_counts'][k]), (name, 'lap_counts', k)
        assert np.allclose(out['lap_times'][0], g['lap_times'][k], rtol=0, atol=1e-12), (name, 'lap_times', k)
        assert abs(out['time'][0] - g['time'][k]) < 1e-12
        d = np.abs(out['state'][0] - g['state'][k]).max()
        worst_state = max(worst_state, d)
        assert d <= state_tol, (name, 'state', k, d)
        if k % every == 0:
            ds = np.abs(out['scans'][0] - g['scans'][k // every])
            outliers += int((ds > scan_tol).sum()); beams += ds.size
            worst_scan = max(worst_scan, float(ds.max()))
            do = np.abs(out['obs'][0] - g['obs'][k // every])
            worst_obs = max(worst_obs, float(do.max()))
    assert outliers <= (1 - scan_frac) * beams, (name, 'scan outliers', outliers, beams)
    if obs_tol is not None:
        assert worst_obs <= obs_tol, (name, 'obs', worst_obs)
    return dict(state=worst_state, scan=worst_scan, outliers=outliers, beams=beams, obs=worst_obs)
