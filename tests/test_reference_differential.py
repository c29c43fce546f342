"""Differential tests of the oracle against the LIVE reference (only where F110_REFERENCE_ROOT names a checkout of it;
skipped otherwise).  The committed golden fixtures pin fixed scenarios; these draw fresh ones."""
import os
import sys
import warnings

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
from ref_loader import REF_MAPS, fresh_statics, load_reference, reference_available  # noqa: E402

pytestmark = pytest.mark.skipif(not reference_available(), reason="F110_REFERENCE_ROOT does not name a checkout of the reference")


@pytest.fixture(scope="module")
def ref():
    warnings.filterwarnings('ignore')
    return load_reference()


@pytest.mark.parametrize("seed", [11, 12])
def test_random_rollout_oracle_vs_live_reference(ref, seed):
    """Fresh start poses on the centerline, fresh random f32 actions, 250 steps: state and flat obs bit-exact, flags exact,
    scans within 1e-12 (BLAS dots in the reference's opponent ray-cast)."""
    from oracle.f110_oracle import Oracle
    rng = np.random.default_rng(seed)
    cl = np.loadtxt(os.path.join(os.path.dirname(REF_MAPS.rstrip('/')), 'maps/cenerlines/Shanghai_map.csv'), delimiter=',', comments='#')
    i = int(rng.integers(0, len(cl) - 60))
    def pose(k):
        return [cl[k, 0], cl[k, 1], np.arctan2(cl[k + 1, 1] - cl[k, 1], cl[k + 1, 0] - cl[k, 0])]
    poses = np.array([pose(i), pose(i + int(rng.integers(8, 50)))])
    fresh_statics(ref)
    env = ref.F110Env(map_dir=REF_MAPS, map='Shanghai_map', map_ext='.png', num_agents=2)
    o = Oracle(1, 2)
    o.set_map(REF_MAPS + 'Shanghai_map.yaml', '.png')
    noise = np.random.default_rng(42)
    obs, info = env.reset(options=poses)
    nz = noise.normal(0., 0.01, size=1080)
    out = o.reset(poses[None], noise=np.stack([nz, nz])[None])
    assert np.array_equal(obs, out['obs'][0])
    for t in range(250):
        act = rng.uniform([-0.4189, 0], [0.4189, 9], size=(2, 2)).astype(np.float32)
        obs, r, term, trunc, info = env.step(act)
        nz = noise.normal(0., 0.01, size=1080)
        out = o.step(act[None], noise=np.stack([nz, nz])[None])
        st = np.stack([a.state for a in env.sim.agents])
        assert np.array_equal(st, out['state'][0]), t
        assert np.array_equal(obs, out['obs'][0]), t
        assert bool(out['terminated'][0]) == term and np.array_equal(info['collisions'], out['collisions'][0])
        assert np.array_equal(env.toggle_list, out['toggles'][0])
        assert np.abs(np.stack(ref.F110Env.current_obs['scans']) - out['scans'][0]).max() < 1e-12


@pytest.mark.parametrize("case", [0, 1])
def test_env_kwargs_oracle_vs_live_reference(ref, case):
    """F110Env constructor kwargs away from their defaults (f110_env.py:104-185): 3-4 agents, time step, Euler, lidar
    offset, ego index, seed.  State / flat obs bit-exact, flags and time exact, scans within 1e-12."""
    from oracle.f110_oracle import Oracle
    kw = (dict(num_agents=3, timestep=0.02, integrator=ref.Integrator.Euler, lidar_dist=0.2, ego_idx=1, seed=7),
          dict(num_agents=4, timestep=0.005, lidar_dist=-0.15, ego_idx=3, seed=123))[case]
    A = kw['num_agents']
    cl = np.loadtxt(os.path.join(os.path.dirname(REF_MAPS.rstrip('/')), 'maps/cenerlines/Shanghai_map.csv'), delimiter=',', comments='#')
    def pose(k):
        return [cl[k, 0], cl[k, 1], np.arctan2(cl[k + 1, 1] - cl[k, 1], cl[k + 1, 0] - cl[k, 0])]
    fresh_statics(ref)
    env = ref.F110Env(map_dir=REF_MAPS, map='Shanghai_map', map_ext='.png', **kw)
    o = Oracle(1, A, timestep=kw['timestep'], integrator=getattr(kw.get('integrator', 1), 'value', 1),
               lidar_dist=kw['lidar_dist'], ego_idx=kw['ego_idx'])
    o.set_map(REF_MAPS + 'Shanghai_map.yaml', '.png')
    poses = np.array([pose(1000 + 30 * a) for a in range(A)])
    noise, rng = np.random.default_rng(kw['seed']), np.random.default_rng(1)
    obs, info = env.reset(options=poses)
    nz = noise.normal(0., 0.01, size=1080)
    out = o.reset(poses[None], noise=np.stack([nz] * A)[None])
    assert np.array_equal(obs, out['obs'][0])
    for t in range(200):
        act = rng.uniform([-0.4189, 0], [0.4189, 8], size=(A, 2)).astype(np.float32)
        obs, r, term, trunc, info = env.step(act)
        nz = noise.normal(0., 0.01, size=1080)
        out = o.step(act[None], noise=np.stack([nz] * A)[None])
        st = np.stack([a.state for a in env.sim.agents])
        assert np.array_equal(st, out['state'][0]) and np.array_equal(obs, out['obs'][0]), t
        assert bool(out['terminated'][0]) == term and np.array_equal(info['collisions'], out['collisions'][0]), t
        assert info['time'] == float(out['time'][0]) and np.float32(r) == out['reward'][0], t
        assert np.abs(np.stack(ref.F110Env.current_obs['scans']) - out['scans'][0]).max() < 1e-12
        if term:
            break
    assert t > 50


def test_update_map_mid_episode_oracle_vs_live_reference(ref):
    """F110Env.update_map (f110_env.py:474-485) between steps: the cars keep their state, the scans come from the new map
    (here one whose yaml origin is rotated by -pi/2)."""
    from oracle.f110_oracle import Oracle
    poses = np.array([[0., 0., 1.5], [0.3, 4.0, 1.5]])
    fresh_statics(ref)
    env = ref.F110Env(map_dir=REF_MAPS, map='Shanghai_map', map_ext='.png', num_agents=2)
    o = Oracle(1, 2)
    o.set_map(REF_MAPS + 'Shanghai_map.yaml', '.png')
    noise, rng = np.random.default_rng(42), np.random.default_rng(8)
    obs, info = env.reset(options=poses)
    nz = noise.normal(0., 0.01, size=1080)
    out = o.reset(poses[None], noise=np.stack([nz, nz])[None])
    assert np.array_equal(obs, out['obs'][0])
    for t in range(120):
        if t == 40:
            env.update_map(REF_MAPS + 'straight_corridor.yaml', '.png')
            o.set_map(REF_MAPS + 'straight_corridor.yaml', '.png')
        if t == 80:
            env.update_map(REF_MAPS + 'Shanghai_map.yaml', '.png')
            o.set_map(REF_MAPS + 'Shanghai_map.yaml', '.png')
        act = rng.uniform([-0.2, 0], [0.2, 4], size=(2, 2)).astype(np.float32)
        obs, r, term, trunc, info = env.step(act)
        nz = noise.normal(0., 0.01, size=1080)
        out = o.step(act[None], noise=np.stack([nz, nz])[None])
        st = np.stack([a.state for a in env.sim.agents])
        assert np.array_equal(st, out['state'][0]) and np.array_equal(obs, out['obs'][0]), t
        assert bool(out['terminated'][0]) == term and np.array_equal(info['collisions'], out['collisions'][0]), t
        assert np.abs(np.stack(ref.F110Env.current_obs['scans']) - out['scans'][0]).max() < 1e-12
        if term:
            break
    assert t >= 45          # the run got past the first map swap


def test_per_agent_params_oracle_vs_live_reference(ref):
    """Simulator.update_params(params, agent_idx) (base_classes.py:529-547): a heavier, longer, wider second car.  Dynamics
    use the agent's own parameters, its ray-cast the agent's own length/width (:223), GJK the Simulator's (:556-560)."""
    from oracle.f110_oracle import DEFAULT_PARAMS, Oracle
    poses = np.array([[0., 0., 0.], [1.2, 0.25, 0.1]])
    p1 = dict(DEFAULT_PARAMS)
    p1.update(m=5.1, I=0.09, lf=0.17, lr=0.19, length=0.9, width=0.5, mu=0.8, a_max=6.0, v_max=12.0, sv_max=2.0)
    fresh_statics(ref)
    env = ref.F110Env(map_dir=REF_MAPS, map='Shanghai_map', map_ext='.png', num_agents=2)
    env.update_params(p1, index=1)
    o = Oracle(1, 2)
    o.set_map(REF_MAPS + 'Shanghai_map.yaml', '.png')
    o.update_params(p1, 1)
    noise, rng = np.random.default_rng(42), np.random.default_rng(5)
    obs, info = env.reset(options=poses)
    nz = noise.normal(0., 0.01, size=1080)
    out = o.reset(poses[None], noise=np.stack([nz, nz])[None])
    assert np.array_equal(obs, out['obs'][0])
    collided = False
    for t in range(150):
        act = rng.uniform([-0.4189, 0], [0.4189, 6], size=(2, 2)).astype(np.float32)
        obs, r, term, trunc, info = env.step(act)
        nz = noise.normal(0., 0.01, size=1080)
        out = o.step(act[None], noise=np.stack([nz, nz])[None])
        st = np.stack([a.state for a in env.sim.agents])
        assert np.array_equal(st, out['state'][0]) and np.array_equal(obs, out['obs'][0]), t
        assert bool(out['terminated'][0]) == term and np.array_equal(info['collisions'], out['collisions'][0]), t
        assert np.abs(np.stack(ref.F110Env.current_obs['scans']) - out['scans'][0]).max() < 1e-12
        collided = collided or bool(info['collisions'].any())
        if term:
            break
    assert collided          # the two cars start 1.2 m apart: the run ends in a GJK collision


def test_gap_follow_and_reward_vs_live_reference(ref):
    from oracle.f110_oracle import RewardOracle, gap_follow_action
    sys.path.insert(0, os.path.join(os.path.dirname(REF_MAPS.rstrip('/'))))
    from utils.gap_follow import gap_follow_action as ref_gf
    rng = np.random.default_rng(3)
    for _ in range(60):
        s = rng.uniform(0, 6, 1080).astype(np.float32)
        s[rng.integers(0, 1000):][:rng.integers(1, 80)] = rng.uniform(0, 0.4)
        assert np.array_equal(gap_follow_action(s), ref_gf(s.copy()))


def test_replay_buffer_vs_live_reference():
    """DeviceReplayBuffer against rl_training/DDPG/replay_buffer.py on the same insert / update sequence: ring position,
    priorities, sampling probabilities, and -- for the indices the reference drew -- the importance weights."""
    import importlib.util
    import torch
    from f110_gymnasium_ros2_jazzy_b200.rollout import DeviceReplayBuffer
    path = os.path.join(os.path.dirname(REF_MAPS.rstrip('/')), 'DDPG', 'replay_buffer.py')
    spec = importlib.util.spec_from_file_location('ref_replay_buffer', path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    ref = mod.PrioritizedExperienceReplayBuffer(buffer_size=50, batch_size=8, alpha=0.6, seed=3)
    mine = DeviceReplayBuffer(capacity=50, batch_size=8, obs_dim=4, act_dim=2, alpha=0.6, device='cpu')
    rng = np.random.default_rng(0)
    for rnd in range(9):
        n = 7
        o = rng.normal(size=(n, 4)).astype(np.float32)
        for i in range(n):
            ref.add(('exp', rnd, i))
        mine.add(torch.from_numpy(o), torch.zeros(n, 2), torch.zeros(n), torch.from_numpy(o), torch.zeros(n, dtype=torch.uint8))
        assert len(ref) == len(mine) and ref._next_idx == mine.next_idx
        idxs, _, w_ref = ref.sample(beta=0.4)
        pr = np.abs(rng.normal(size=8)).astype(np.float32) * 3
        pr[0] = np.inf if rnd == 4 else (np.nan if rnd == 6 else pr[0])      # clamped to f32 max / replaced by 1e-6
        ref.update_priorities(idxs, pr)
        mine.update_priorities(idxs, pr)
        assert np.array_equal(ref._buffer['priority'][:len(ref)], mine.priority[:len(mine)].numpy())
        probs = mine.probabilities().numpy()
        idxs2, _, w_ref2 = ref.sample(beta=0.7)
        w = np.power(len(mine) * probs[idxs2], -0.7)
        assert np.allclose((w / w.max()).astype(np.float32), w_ref2, rtol=1e-6, atol=0)
