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
