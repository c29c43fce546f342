"""The scenarios of test_reference_differential.py, without the reference: the oracle driven exactly as those tests drive it,
against tests/golden/differential.npz.

That recording was made with the oracle (tests/golden/make_differential.py) whose source has not changed since it passed
those tests against the live reference -- state, flat observation, flags, time and reward bit-exact, scans within 1e-12 --
so it stands for what the reference computed on these scenarios.  Per step it keeps the flags, time and reward, and a
SHA-256 of the state + flat observation and one of the scans (the scans of a 4-car, 200-step run alone are 7 MB)."""
import hashlib

import numpy as np
import pytest

from oracle.f110_oracle import DEFAULT_PARAMS, Oracle, gap_follow_action
from tests import helpers as H

ROLLOUTS = ('random_11', 'random_12', 'kwargs_0', 'kwargs_1', 'update_map', 'per_agent_params')


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def _oracle(num_agents, map_name='Shanghai_map', **kw):
    o = Oracle(1, num_agents, **kw)
    s, c, a, bc, sd = H.tables()
    o.set_tables(s, c)
    o.set_beam_tables(a, bc, sd)
    o.set_map_arrays(*H.golden_map(map_name))
    return o


def _centerline_pose(cl, k):
    return [cl[k, 0], cl[k, 1], np.arctan2(cl[k + 1, 1] - cl[k, 1], cl[k + 1, 0] - cl[k, 0])]


def run_rollout(name):
    """-> per-step records (the reset observation first) of the oracle on one scenario of test_reference_differential.py:
    same poses, actions, lidar noise, map swaps and parameters, same stopping rule."""
    cl = H.load('reward')['centerline']                    # rl_training/maps/cenerlines/Shanghai_map.csv
    if name.startswith('random_'):
        steps, A, stop_on_term = 250, 2, False
        rng = np.random.default_rng(int(name.split('_')[1]))
        i = int(rng.integers(0, len(cl) - 60))
        poses = np.array([_centerline_pose(cl, i), _centerline_pose(cl, i + int(rng.integers(8, 50)))])
        o, noise = _oracle(2), np.random.default_rng(42)
        act = lambda: rng.uniform([-0.4189, 0], [0.4189, 9], size=(2, 2)).astype(np.float32)
    elif name.startswith('kwargs_'):
        kw = (dict(num_agents=3, timestep=0.02, integrator=2, lidar_dist=0.2, ego_idx=1, seed=7),
              dict(num_agents=4, timestep=0.005, integrator=1, lidar_dist=-0.15, ego_idx=3, seed=123))[int(name[-1])]
        steps, A, stop_on_term = 200, kw['num_agents'], True
        o = _oracle(A, timestep=kw['timestep'], integrator=kw['integrator'], lidar_dist=kw['lidar_dist'], ego_idx=kw['ego_idx'])
        poses = np.array([_centerline_pose(cl, 1000 + 30 * a) for a in range(A)])
        noise, rng = np.random.default_rng(kw['seed']), np.random.default_rng(1)
        act = lambda: rng.uniform([-0.4189, 0], [0.4189, 8], size=(A, 2)).astype(np.float32)
    elif name == 'update_map':
        steps, A, stop_on_term = 120, 2, True
        poses = np.array([[0., 0., 1.5], [0.3, 4.0, 1.5]])
        o, noise, rng = _oracle(2), np.random.default_rng(42), np.random.default_rng(8)
        act = lambda: rng.uniform([-0.2, 0], [0.2, 4], size=(2, 2)).astype(np.float32)
    else:
        steps, A, stop_on_term = 150, 2, True
        poses = np.array([[0., 0., 0.], [1.2, 0.25, 0.1]])
        p1 = dict(DEFAULT_PARAMS)
        p1.update(m=5.1, I=0.09, lf=0.17, lr=0.19, length=0.9, width=0.5, mu=0.8, a_max=6.0, v_max=12.0, sv_max=2.0)
        o = _oracle(2)
        o.update_params(p1, 1)
        noise, rng = np.random.default_rng(42), np.random.default_rng(5)
        act = lambda: rng.uniform([-0.4189, 0], [0.4189, 6], size=(2, 2)).astype(np.float32)
    nz = noise.normal(0., 0.01, size=1080)
    records = [o.reset(poses[None], noise=np.stack([nz] * A)[None])]
    for t in range(steps):
        if name == 'update_map' and t in (40, 80):
            o.set_map_arrays(*H.golden_map('straight_corridor' if t == 40 else 'Shanghai_map'))
        a = act()
        nz = noise.normal(0., 0.01, size=1080)
        records.append(o.step(a[None], noise=np.stack([nz] * A)[None]))
        if stop_on_term and records[-1]['terminated'][0]:
            break
    return [{k: np.array(v[0]) for k, v in r.items()} for r in records]


def record(name):
    """The arrays differential.npz keeps for one scenario."""
    rs = run_rollout(name)
    return {'digest_state_obs': np.stack([_digest(r['state'], r['obs']) for r in rs]),
            'digest_scans': np.stack([_digest(r['scans']) for r in rs]),
            'collisions': np.stack([r['collisions'] for r in rs]), 'terminated': np.stack([r['terminated'] for r in rs]),
            'toggles': np.stack([r['toggles'] for r in rs]), 'time': np.stack([r['time'] for r in rs]),
            'reward': np.stack([r['reward'] for r in rs])}


def gap_follow_scans():
    """The 60 scans of test_gap_follow_and_reward_vs_live_reference."""
    rng = np.random.default_rng(3)
    out = []
    for _ in range(60):
        s = rng.uniform(0, 6, 1080).astype(np.float32)
        s[rng.integers(0, 1000):][:rng.integers(1, 80)] = rng.uniform(0, 0.4)
        out.append(s)
    return out


@pytest.mark.parametrize('name', ROLLOUTS)
def test_oracle_rollout_matches_recording(name):
    g = H.load('differential')
    want = {k.split('__', 1)[1]: v for k, v in g.items() if k.startswith(name + '__')}
    got = record(name)
    assert len(got['time']) == len(want['time']), (name, 'steps', len(got['time']), len(want['time']))
    for k in ('collisions', 'terminated', 'toggles', 'time', 'reward'):
        assert np.array_equal(got[k], want[k]), (name, k)
    for k in ('digest_state_obs', 'digest_scans'):
        bad = np.flatnonzero((got[k] != want[k]).any(axis=1))
        assert bad.size == 0, (name, k, 'first step that differs', int(bad[0]) if bad.size else None)
    # what each live scenario asserts about how it ends
    t = len(got['time']) - 2                              # index of the last step (the reset comes first)
    if name.startswith('kwargs_'):
        assert t > 50
    elif name == 'update_map':
        assert t >= 45                                    # past the first map swap
    elif name == 'per_agent_params':
        assert got['collisions'].any()                    # the cars start 1.2 m apart: a GJK collision ends the run


def test_gap_follow_matches_recording():
    want = H.load('differential')['gap_follow__actions']
    assert np.array_equal(np.stack([gap_follow_action(s) for s in gap_follow_scans()]), want)
