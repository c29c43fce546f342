"""GPU parity suite (-m gpu): the CUDA path, called through the C ABI, against
  * the golden vectors recorded from the unmodified reference (tests/golden), and
  * the CPU oracle on the same seeded inputs, at sizes the oracle finishes in seconds, and
  * size-independent properties at the BASELINE.json batch sizes.

Tolerances are BASELINE.json's north_star: collision / done / lap flags bit-exact over the rollout, fp64
vehicle state within 1e-9 absolute, lidar within 1e-6 m on >= 99.9 % of beams (outliers counted).
"""
import os

import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu

STATE_TOL = 1e-9
SCAN_TOL = 1e-6
SCAN_FRAC = 0.999


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


class GpuBackend(object):
    """Adapter: BatchSim (device tensors) -> the numpy dict compare_rollout expects."""

    def __init__(self, num_envs, num_agents, map_name, **kw):
        _torch()
        from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
        self.sim = BatchSim(num_envs, num_agents, outputs=ALL_OUTPUTS, noise_std=kw.pop('noise_std', 0.0), **kw)
        s, c, a, bc, sd = H.tables()
        self.sim.set_tables(s, c)
        if self.sim.B == len(a) and kw.get('fov', 4.7) == 4.7:     # the fixture tables are the reference's 1080 x 4.7 rad ones
            self.sim.set_beam_tables(a, bc, sd)
        self.sim.set_map_arrays(*H.golden_map(map_name))

    def _np(self, o):
        import torch
        torch.cuda.synchronize()
        d = {k: v.cpu().numpy() for k, v in o.items()}
        d['scans'] = d['scans_f64']
        return d

    def reset(self, poses, noise=None):
        return self._np(self.sim.reset(poses, noise))

    def step(self, actions, noise=None, **kw):
        return self._np(self.sim.step(actions, noise, **kw))


def make_gpu(num_agents, map_name, **kw):
    return GpuBackend(1, num_agents, map_name, **kw)


def make_oracle(num_envs, num_agents, map_name, **kw):
    from oracle.f110_oracle import Oracle
    o = Oracle(num_envs, num_agents, **kw)
    s, c, a, bc, sd = H.tables()
    o.set_tables(s, c)
    if o.B == len(a) and kw.get('fov', 4.7) == 4.7:
        o.set_beam_tables(a, bc, sd)
    o.set_map_arrays(*H.golden_map(map_name))
    return o


# ----------------------------------------------------------------------------- golden rollouts

@pytest.mark.parametrize("name", sorted(H.ROLLOUT_MAP))
def test_golden_rollouts(name):
    r = H.compare_rollout(name, make_gpu, state_tol=STATE_TOL, scan_tol=SCAN_TOL, scan_frac=SCAN_FRAC, obs_tol=1e-6)
    print(name, r)


@pytest.mark.parametrize("map_name", ["Shanghai_map", "straight_corridor"])
def test_golden_scans_noise_free(map_name):
    """ScanSimulator2D.scan(pose, None): the ray-march alone; expected bit-exact (same tables, no FMA)."""
    g = H.load('scans')
    poses, ref = g[map_name + '__poses'], g[map_name + '__scans']
    be = GpuBackend(len(poses), 1, map_name)
    be.sim.sim_reset(poses[:, None, :])
    # a zero-velocity car does not move in one zero-action step: the scan is taken at the reset pose
    out = be.step(None, np.zeros((len(poses), 1, 1080)))
    d = np.abs(out['scans'][:, 0] - ref)
    # wrap() of the yaw happens before the scan; poses outside [-pi, pi) only change theta by an exact 2*pi multiple
    frac_exact = float((d == 0).mean())
    print(map_name, 'max', d.max(), 'exact fraction', frac_exact)
    assert (d <= SCAN_TOL).mean() >= SCAN_FRAC


def _rotated_map_and_poses(theta, n=96):
    """The Shanghai map under an origin with yaw theta (ScanSimulator2D.set_map keeps orig_c/orig_s, laser_models.py:421),
    and centerline poses carried into that world frame."""
    dt, res, o = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    cl = cl[np.linspace(0, len(cl) - 1, n).round().astype(int)]
    o2 = [3.5, -7.25, theta]
    mx, my = cl[:, 0] - o[0], cl[:, 1] - o[1]                    # map-frame coordinates
    c, s = np.cos(theta), np.sin(theta)
    poses = np.stack([o2[0] + c * mx - s * my, o2[1] + s * mx + c * my, cl[:, 2] + theta], axis=1)
    return (dt, res, o2), poses


@pytest.mark.parametrize('theta', [0.0, 0.3])
def test_exact_finishing_path_scans(theta):
    """F110_FLAG_NARROW_FRACTION leaves the fixed-point cell index 6 fraction bits, so about 6 % of lookups fall in the
    guard band and their rays are finished by the lidar kernel's exact-arithmetic loop (normally 1e-6 of lookups).
    The scans must not change by a bit, and must equal the oracle's -- on an axis-aligned and on a rotated map origin."""
    from oracle.f110_oracle import Oracle
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    m, poses = _rotated_map_and_poses(theta)
    n = len(poses)
    orc = Oracle(1, 1); orc.set_map_arrays(*m)
    s, c, _, _, _ = H.tables()
    orc.set_tables(s, c)
    want = np.stack([orc.scan(p)[0] for p in poses])
    outs = []
    for narrow in (False, True):
        sim = BatchSim(n, 1, outputs=ALL_OUTPUTS, noise_std=0.0, narrow_fraction=narrow)
        sim.set_tables(s, c)
        sim.set_map_arrays(*m)
        sim.sim_reset(poses[:, None, :])
        o = sim.step(None, np.zeros((n, 1, 1080)))
        import torch
        torch.cuda.synchronize()
        outs.append(o['scans_f64'].cpu().numpy()[:, 0])
        sim.close()
    assert np.array_equal(outs[0], outs[1])
    d = np.abs(outs[1] - want)
    print('theta', theta, 'max', d.max(), 'exact fraction', float((d == 0).mean()))
    assert (d <= SCAN_TOL).mean() >= SCAN_FRAC
    if theta == 0.0:
        assert d.max() == 0.0


def test_rotated_origin_scans_golden():
    """Map origin with a yaw (non-identity rotation in every lookup): against the reference's own scans."""
    _torch()
    import torch
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    g = H.load('scans_rotated')
    dt, res, _ = H.golden_map('Shanghai_map')
    poses = g['poses']
    n = len(poses)
    sim = BatchSim(n, 1, outputs=ALL_OUTPUTS, noise_std=0.0)
    s, c, _, _, _ = H.tables()
    sim.set_tables(s, c)
    sim.set_map_arrays(dt, res, [float(v) for v in g['origin']])
    sim.sim_reset(poses[:, None, :])
    o = sim.step(None, np.zeros((n, 1, 1080)))
    torch.cuda.synchronize()
    d = np.abs(o['scans_f64'].cpu().numpy()[:, 0] - g['scans'])
    print('rotated origin: max', d.max(), 'exact fraction', float((d == 0).mean()))
    assert (d <= SCAN_TOL).mean() >= SCAN_FRAC
    sim.close()


@pytest.mark.parametrize("name", H.LARGE_MAPS)
def test_large_map_scans_golden_and_oracle(name):
    """BASELINE config C4 'large maps': levine 2048^2, Shanghai x2 (4000^2, 128 MB), x4 (8000^2, 512 MB: not L2-resident)
    and x2 under a rotated origin.  The guarded fixed-point cell index keeps 20 / 20 / 19 fraction bits on these maps
    instead of the 21 of the 2000^2 map.  Noise-free scans against the reference's own (tests/golden/scans_large.npz)
    and against the oracle: bit-exact on the axis-aligned origins, <= 1e-6 m on >= 99.9 % of beams on the rotated one;
    poses on the track, next to the map border, on it and outside."""
    from oracle.f110_oracle import Oracle
    _torch()
    import torch
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    dt, res, origin, poses, ref = H.large_map(name)
    n = len(poses)
    s, c, _, _, _ = H.tables()
    orc = Oracle(1, 1); orc.set_tables(s, c); orc.set_map_arrays(dt, res, origin)
    want = np.stack([orc.scan(p)[0] for p in poses])
    sim = BatchSim(n, 1, outputs=ALL_OUTPUTS, noise_std=0.0)
    sim.set_tables(s, c)
    sim.set_map_arrays(dt, res, origin)
    sim.sim_reset(poses[:, None, :])
    o = sim.step(None, np.zeros((n, 1, 1080)))
    torch.cuda.synchronize()
    got = o['scans_f64'].cpu().numpy()[:, 0]
    sim.close()
    d_ref, d_orc = np.abs(got - ref), np.abs(got - want)
    print(name, dt.shape, 'vs reference max', d_ref.max(), 'exact', float((d_ref == 0).mean()), '| vs oracle max', d_orc.max())
    assert (d_ref <= SCAN_TOL).mean() >= SCAN_FRAC
    assert d_orc.max() == 0.0 or name.endswith('_rot')
    assert (d_orc <= SCAN_TOL).mean() >= SCAN_FRAC
    if not name.endswith('_rot'):
        assert d_ref.max() == 0.0


def test_lean_lidar_variants_equal_the_general_one():
    """The lidar kernel has variants without the tests and address arithmetic for outputs that were not asked for (single
    agent: float32 observation only; opponents: no fp64 scan; both: device noise, no env mask).  Same seed, same actions:
    the observation, reward and terminated flags equal those of the general variant (ALL_OUTPUTS) bit for bit."""
    _torch()
    import torch
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim, workloads
    dt, res, origin = H.golden_map('Shanghai_map')
    rng = np.random.default_rng(13)
    for agents, lean in ((1, ('obs', 'reward', 'terminated')), (2, ('obs', 'scans_f32', 'reward', 'terminated'))):
        N = 300
        start = workloads.start_poses(N, agents)
        acts = rng.uniform([-0.4189, 0.0], [0.4189, 10.0], size=(120, N, agents, 2)).astype(np.float32)
        traces = []
        for outputs in (ALL_OUTPUTS, lean):
            sim = BatchSim(N, agents, outputs=outputs, noise_std=0.01, seed=17)
            sim.set_map_arrays(dt, res, origin)
            out = sim.reset(start)
            mask, tr = None, []
            for t in range(120):
                out = sim.step(acts[t], reset_mask=mask, reset_poses=start) if mask is not None else sim.step(acts[t])
                torch.cuda.synchronize()
                mask = out['terminated'].clone()
                tr.append((out['obs'].cpu().numpy().copy(), out['terminated'].cpu().numpy().copy()))
            sim.close()
            traces.append(tr)
        for (o0, t0), (o1, t1) in zip(*traces):
            assert np.array_equal(t0, t1) and np.array_equal(o0, o1), agents
        assert sum(int(t.sum()) for _, t in traces[1]) > 0


@pytest.mark.parametrize('agents', [2, 4])
def test_opponent_raycast_in_float_outputs_equals_the_fp64_path(agents):
    """K3 lowers the beams that hit an opponent in the caller's own buffers (ray_cast_agents, base_classes.py:206-227).  With an
    fp64 scan among the outputs that is the reference's min(scan, range) in fp64; without one the float outputs are lowered
    each in its own domain.  Float conversion and the observation's clip / scale are monotone, so both give the same floats:
    checked bit for bit over a rollout in which cars see, occlude and hit each other."""
    _torch()
    import torch
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim, workloads
    N = 256
    dt, res, origin = H.golden_map('Shanghai_map')
    start = workloads.start_poses(N, agents)            # opponents 25 centerline rows (about 1.6 m) ahead of each other
    rng = np.random.default_rng(11)
    acts = rng.uniform([-0.3, 0.0], [0.3, 6.0], size=(150, N, agents, 2)).astype(np.float32)
    traces = []
    for outputs in (ALL_OUTPUTS, ('obs', 'scans_f32', 'reward', 'terminated')):
        sim = BatchSim(N, agents, outputs=outputs, noise_std=0.01, seed=5)
        sim.set_map_arrays(dt, res, origin)
        out = sim.reset(start)
        mask, tr = None, []
        for t in range(150):
            out = sim.step(acts[t], reset_mask=mask, reset_poses=start) if mask is not None else sim.step(acts[t])
            torch.cuda.synchronize()
            mask = out['terminated'].clone()
            tr.append((out['obs'].cpu().numpy().copy(), out['scans_f32'].cpu().numpy().copy(), out['terminated'].cpu().numpy().copy()))
        sim.close()
        traces.append(tr)
    for (o0, s0, t0), (o1, s1, t1) in zip(*traces):
        assert np.array_equal(t0, t1) and np.array_equal(s0, s1) and np.array_equal(o0, o1)
    # the opponent ahead is in view: the beams straight ahead of car 0 end on it, not on a wall tens of metres away
    assert np.median(traces[1][0][1][:, 0, 520:560].min(axis=1)) < 2.5


def test_c1_single_agent_sim_rollout():
    g = H.load('rollout_c1_single')
    be = make_gpu(1, 'Shanghai_map')
    rng = None
    worst = 0.0
    for t in range(g['state'].shape[0]):
        if g['resets'][t] or t == 0:
            rng = np.random.default_rng(int(g['seed']))
            be.sim.sim_reset(g['pose'][None, None])
        out = be.step(g['action'][None], rng.normal(0., 0.01, size=1080)[None, None])
        worst = max(worst, np.abs(out['state'][0, 0] - g['state'][t]).max())
        assert out['collisions'][0, 0] == g['collisions'][t], t
        if t % int(g['every']) == 0:
            assert (np.abs(out['scans'][0, 0] - g['scans'][t // int(g['every'])]) <= SCAN_TOL).mean() >= SCAN_FRAC
    assert worst <= STATE_TOL
    print('c1 worst state diff', worst)


def test_integration_stub_simulator(tmp_path):
    """integration/native_simulator.py -- the ctypes-only `Simulator` INTEGRATION.md hands to a maintainer of the
    reference -- replays the reference's recorded single-agent Simulator rollout (golden C1) and raises the reference's
    exceptions.  It imports nothing from this package: the C ABI is the whole interface."""
    import importlib.util
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    from f110_gymnasium_ros2_jazzy_b200.params import default_params
    _torch()
    os.environ.setdefault('F110_B200_LIB', _lib.LIB_PATH)
    spec = importlib.util.spec_from_file_location(
        'native_simulator', os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'integration', 'native_simulator.py'))
    ns = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ns)
    map_dir, name = H.write_map_files('Shanghai_map', str(tmp_path))
    g = H.load('rollout_c1_single')
    sim = ns.Simulator(default_params(), 1, int(g['seed']))
    with pytest.raises(ValueError, match='Map is not set'):
        sim.reset(g['pose'][None]); sim.step(g['action'])
    sim.set_map(map_dir + name + '.yaml', '.png')
    with pytest.raises(ValueError, match='Number of poses'):
        sim.reset(np.zeros((2, 3)))
    with pytest.raises(IndexError):
        sim.update_params(default_params(), agent_idx=3)
    worst = 0.0
    for t in range(600):
        if g['resets'][t] or t == 0:
            sim.reset(g['pose'][None])
        obs = sim.step(g['action'])
        st = np.array([obs['poses_x'][0], obs['poses_y'][0], obs['poses_theta'][0], obs['linear_vels_x'][0], obs['ang_vels_z'][0]])
        worst = max(worst, np.abs(st - g['state'][t][[0, 1, 4, 3, 5]]).max())
        assert obs['collisions'][0] == g['collisions'][t], t
        if t % int(g['every']) == 0:
            assert (np.abs(obs['scans'][0] - g['scans'][t // int(g['every'])]) <= SCAN_TOL).mean() >= SCAN_FRAC
    assert worst <= STATE_TOL
    print('integration stub: worst state diff', worst)


# ----------------------------------------------------------------------------- oracle on seeded batches

@pytest.mark.parametrize("num_envs,num_agents", [(64, 1), (48, 2), (16, 3)])
def test_batched_vs_oracle(num_envs, num_agents):
    """Random start poses on the Shanghai centerline, random f32 actions, injected noise, masks and resets."""
    rng = np.random.default_rng(100 + num_envs)
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    idx = rng.integers(0, len(cl), size=num_envs)
    poses = np.zeros((num_envs, num_agents, 3))
    for a in range(num_agents):
        j = (idx + 18 * a) % len(cl)
        poses[:, a] = cl[j]
        poses[:, a, 1] += 0.25 * a
    be = GpuBackend(num_envs, num_agents, 'Shanghai_map')
    orc = make_oracle(num_envs, num_agents, 'Shanghai_map')
    T = 120
    stats = dict(state=0.0, outl=0, beams=0)
    prev_term = np.zeros(num_envs, np.uint8)
    for t in range(T):
        noise = rng.normal(0, 0.01, size=(num_envs, num_agents, 1080))
        if t == 0:
            g = be.reset(poses, noise)
            c = orc.reset(poses, noise)
        else:
            act = rng.uniform([-0.4189, 0], [0.4189, 12], size=(num_envs, num_agents, 2)).astype(np.float32)
            kw = {}
            if t % 7 == 0:       # auto-reset of the envs that terminated + a partial active mask
                kw = dict(reset_mask=prev_term.copy(), reset_poses=poses)
            if t % 11 == 0:
                kw['active_mask'] = (rng.uniform(size=num_envs) < 0.7).astype(np.uint8)
            g = be.step(act, noise, **kw)
            c = orc.step(act, noise, **kw)
        for k in ('collisions', 'terminated', 'toggles', 'lap_counts'):
            assert np.array_equal(g[k], c[k]), (k, t)
        assert np.allclose(g['lap_times'], c['lap_times'], rtol=0, atol=1e-12)
        assert np.allclose(g['time'], c['time'], rtol=0, atol=1e-12)
        d = np.abs(g['state'] - c['state']).max()
        stats['state'] = max(stats['state'], d)
        assert d <= STATE_TOL, (t, d)
        ds = np.abs(g['scans'] - c['scans'])
        stats['outl'] += int((ds > SCAN_TOL).sum()); stats['beams'] += ds.size
        assert np.abs(g['obs'] - c['obs']).max() <= 1e-6 or (ds > SCAN_TOL).any()
        prev_term = c['terminated'].copy()
    print('batched vs oracle', num_envs, num_agents, stats)
    assert stats['outl'] <= (1 - SCAN_FRAC) * stats['beams']


@pytest.mark.parametrize("kw", [
    dict(theta_dis=360, eps=1e-3, max_range=12.0, lidar_dist=0.3, timestep=0.02, ttc_thresh=0.01),
    dict(theta_dis=4001, integrator=2, ego_idx=1, max_range=45.0, lidar_dist=-0.1),       # Euler (Integrator.Euler == 2); ego = the second car
])
def test_constructor_parameters_vs_oracle(kw):
    """Every Simulator / ScanSimulator2D constructor parameter away from its default (base_classes.py:478-510,
    laser_models.py:356-381): table size, march threshold and range, lidar offset, time step, integrator, ego index."""
    _torch()
    import torch
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    from oracle.f110_oracle import Oracle
    N, A = 24, 2
    m = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    rng = np.random.default_rng(31)
    idx = rng.integers(0, len(cl), size=N)
    poses = np.stack([cl[idx], cl[(idx + 25) % len(cl)]], axis=1)
    sim = BatchSim(N, A, outputs=ALL_OUTPUTS, noise_std=0.0, **kw)
    orc = Oracle(N, A, **kw)
    sim.set_map_arrays(*m); orc.set_map_arrays(*m)
    worst, outl, beams = 0.0, 0, 0
    for t in range(80):
        noise = rng.normal(0, 0.01, size=(N, A, 1080))
        if t == 0:
            g = sim.reset(poses, noise); c = orc.reset(poses, noise)
        else:
            act = rng.uniform([-0.4189, 0], [0.4189, 10], size=(N, A, 2)).astype(np.float32)
            g = sim.step(act, noise); c = orc.step(act, noise)
        torch.cuda.synchronize()
        g = {k: v.cpu().numpy() for k, v in g.items()}
        for k in ('collisions', 'terminated', 'toggles'):
            assert np.array_equal(g[k], c[k]), (k, t)
        worst = max(worst, np.abs(g['state'] - c['state']).max())
        ds = np.abs(g['scans_f64'] - c['scans'])
        outl += int((ds > SCAN_TOL).sum()); beams += ds.size
        assert np.abs(g['time'] - c['time']).max() <= 1e-12
    print('constructor parameters', kw, 'state', worst, 'lidar outliers', outl, '/', beams)
    assert worst <= STATE_TOL and outl <= (1 - SCAN_FRAC) * beams
    sim.close()


def test_per_agent_params_vs_oracle():
    """update_params on one agent (heavier, longer, wider car; the oracle is pinned to the reference for this in
    test_reference_differential, and to its recording in test_differential_golden): dynamics and ray-cast use the
    agent's parameters, GJK the Simulator's."""
    from oracle.f110_oracle import DEFAULT_PARAMS
    N, A = 16, 3
    p1 = dict(DEFAULT_PARAMS)
    p1.update(m=5.1, I=0.09, lf=0.17, lr=0.19, length=0.9, width=0.5, mu=0.8, a_max=6.0, v_max=12.0, sv_max=2.0)
    p2 = dict(DEFAULT_PARAMS)
    p2.update(length=0.4, width=0.2, C_Sf=5.0, C_Sr=5.5, h=0.05, s_max=0.3, s_min=-0.3)
    be = GpuBackend(N, A, 'Shanghai_map')
    orc = make_oracle(N, A, 'Shanghai_map')
    be.sim.update_params(p1, 1); orc.update_params(p1, 1)
    be.sim.update_params(p2, 2); orc.update_params(p2, 2)
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    rng = np.random.default_rng(77)
    idx = rng.integers(0, len(cl), size=N)
    poses = np.stack([cl[idx], cl[(idx + 14) % len(cl)], cl[(idx + 30) % len(cl)]], axis=1)
    poses[:, 1, 1] += 0.2
    worst, outl, beams, coll = 0.0, 0, 0, 0
    for t in range(150):
        noise = rng.normal(0, 0.01, size=(N, A, 1080))
        if t == 0:
            g = be.reset(poses, noise); c = orc.reset(poses, noise)
        else:
            act = rng.uniform([-0.4189, 0], [0.4189, 7], size=(N, A, 2)).astype(np.float32)
            act[:, 0, 1] += 3.0                      # the ego is faster: it runs into the car ahead
            g = be.step(act, noise); c = orc.step(act, noise)
        for k in ('collisions', 'terminated', 'toggles'):
            assert np.array_equal(g[k], c[k]), (k, t)
        worst = max(worst, np.abs(g['state'] - c['state']).max())
        ds = np.abs(g['scans'] - c['scans'])
        outl += int((ds > SCAN_TOL).sum()); beams += ds.size
        coll += int(c['collisions'].sum())
    print('per-agent params: state', worst, 'lidar outliers', outl, '/', beams, 'collision flags', coll)
    assert worst <= STATE_TOL and outl <= (1 - SCAN_FRAC) * beams and coll > 0


def test_map_swap_between_steps_vs_oracle():
    """f110_set_map between steps (F110Env.update_map, f110_env.py:474-485; the oracle is pinned to the reference for this):
    state carries over, scans come from the new map -- a different size, resolution and a rotated origin -- and back."""
    N, A = 8, 2
    be = GpuBackend(N, A, 'Shanghai_map')
    orc = make_oracle(N, A, 'Shanghai_map')
    rng = np.random.default_rng(21)
    poses = np.tile(np.array([[0., 0., 1.5], [0.3, 4.0, 1.5]]), (N, 1, 1))
    poses[:, :, 0] += rng.uniform(-0.2, 0.2, size=(N, 1))
    outl = beams = 0
    for t in range(90):
        noise = rng.normal(0, 0.01, size=(N, A, 1080))
        if t == 30 or t == 60:
            name = 'straight_corridor' if t == 30 else 'Shanghai_map'
            be.sim.set_map_arrays(*H.golden_map(name)); orc.set_map_arrays(*H.golden_map(name))
        if t == 0:
            g = be.reset(poses, noise); c = orc.reset(poses, noise)
        else:
            act = rng.uniform([-0.2, 0], [0.2, 4], size=(N, A, 2)).astype(np.float32)
            g = be.step(act, noise); c = orc.step(act, noise)
        for k in ('collisions', 'terminated', 'toggles'):
            assert np.array_equal(g[k], c[k]), (k, t)
        assert np.abs(g['state'] - c['state']).max() <= STATE_TOL, t
        ds = np.abs(g['scans'] - c['scans'])
        outl += int((ds > SCAN_TOL).sum()); beams += ds.size
    assert outl <= (1 - SCAN_FRAC) * beams


def test_non_finite_actions():
    """NaN / inf commands.  A NaN steer is swallowed by pid (its comparison is false) and an infinite speed by the
    acceleration clip: both match the oracle (and the reference, probed in the build container) to the usual
    tolerances.  A NaN speed or an infinite steer (pid forms inf/inf) poisons the state; the reference -- and the
    oracle, which restates it -- then index the map with int(NaN) and segfault, so there is nothing to be equal to:
    here those envs must stay memory-safe and must not disturb their neighbours."""
    poses = np.array([[0., 0., 0.], [3.0, 0.5, 0.]])
    bad = [[np.nan, 3.0], [0.1, np.inf], [0.05, 3.0], [np.nan, np.nan], [-np.inf, 2.0]]
    N, M = len(bad), 3                                      # the first M envs have a counterpart in the oracle
    be = GpuBackend(N, 2, 'Shanghai_map')
    orc = make_oracle(M, 2, 'Shanghai_map')
    rng = np.random.default_rng(9)
    P = np.broadcast_to(poses, (N, 2, 3)).copy()
    for t in range(45):
        noise = rng.normal(0, 0.01, size=(N, 2, 1080))
        if t == 0:
            g = be.reset(P, noise); c = orc.reset(P[:M], noise[:M])
        else:
            act = np.tile(np.array([[0.05, 3.0], [0.0, 2.0]]), (N, 1, 1))
            if t == 20:
                act[:, 0] = bad
            g = be.step(act, noise); c = orc.step(act[:M], noise[:M])
        for k in ('collisions', 'terminated', 'toggles'):
            assert np.array_equal(g[k][:M], c[k]), (k, t)
        assert np.abs(g['state'][:M] - c['state']).max() <= STATE_TOL, t
        assert (np.abs(g['scans'][:M] - c['scans']) <= SCAN_TOL).mean() >= SCAN_FRAC
        assert np.isfinite(g['state'][:M]).all()
    for e in range(M, N):                                   # the poisoned cars stay poisoned; nothing else happened
        assert not np.isfinite(g['state'][e, 0]).all(), e


def test_known_answer_dynamics_on_device():
    """The reference's stiff high-speed test state (dynamic_models.py:262-266, CommonRoad vehicle-2 params
    :232-253) through ONE Euler step of the device kernel: x1 == x0 + dt * f(x0, u) with f from the oracle,
    whose RHS is pinned to f_st_gt (:258) by tests/test_oracle_golden.py."""
    torch = _torch()
    from oracle.f110_oracle import Oracle
    from tests.test_oracle_golden import TEST_PARAMS
    x_st = np.array([2.0233348142065677, 0.0041907137716636, 0.0197545248559617, 15.7216236334290116,
                     0.0025857914776859, 0.0529001056654038, 0.0033012170610298])
    p = dict(TEST_PARAMS)
    p['lidar_max'] = 30.0
    dt = 1e-3
    be = GpuBackend(1, 1, 'open_square', params=p, integrator=2, timestep=dt)
    # inject the state through the checkpoint blob: after the 64-byte header, x[k] are the first seven 256-byte-aligned
    # arrays of the arena (NA = 1)
    blob = be.sim.state_dict()['blob'].clone()
    blob.view(torch.float64)[8:8 + 7 * 32:32] = torch.tensor(x_st, dtype=torch.float64, device=blob.device)
    be.sim.load_state_dict({'blob': blob, 'N': 1, 'A': 1, 'B': 1080})
    out = be.step(np.array([[[0.5, 30.0]]], np.float64), np.zeros((1, 1, 1080)))
    # pid(): the steering FIFO is still empty -> steer = 0 -> sv = -sv_max; speed error -> accl clipped to +a_max
    f = Oracle(1, 1).vehicle_dynamics_st(x_st, np.array([-p['sv_max'], p['a_max']]), p)
    x1 = x_st + dt * f
    assert np.abs(out['state'][0, 0] - x1).max() < 1e-13


def test_gjk_known_answer_on_device():
    """collision_models.py:313-324 geometry as cars: overlapping / separated poses -> collision flags."""
    be = GpuBackend(1, 4, 'open_square')
    poses = np.array([[[0.0, 0.0, 0.0], [0.3, 0.1, 0.4], [3.0, 3.0, 1.0], [-4.0, 2.0, 0.0]]])
    out = be.reset(poses, np.zeros((1, 4, 1080)))
    assert out['collisions'][0].tolist() == [1, 1, 0, 0]
    assert bool(out['terminated'][0])
    from oracle.f110_oracle import Oracle
    orc = make_oracle(1, 4, 'open_square')
    c = orc.reset(poses, np.zeros((1, 4, 1080)))
    assert np.array_equal(c['collisions'], out['collisions'])
    assert (np.abs(c['scans'] - out['scans']) <= SCAN_TOL).all()


# ----------------------------------------------------------------------------- properties at full size

def test_full_size_properties():
    """BASELINE config 3 shape (4096 envs x 1 agent x 1080 beams): replicated envs must produce replicated
    results (no cross-env leakage), scans bounded by max_range + noise, state finite, and a checkpoint
    round-trip must reproduce the same next step bit for bit."""
    torch = _torch()
    N = 4096
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    idx = np.linspace(0, len(cl) - 1, N // 4).round().astype(int)
    poses = np.repeat(cl[idx][:, None, :], 4, axis=0)              # every start pose 4x
    be = GpuBackend(N, 1, 'Shanghai_map')
    rng = np.random.default_rng(5)
    be.sim.reset(poses, None)
    for t in range(30):
        act = np.repeat(rng.uniform([-0.4189, 0], [0.4189, 10], size=(N // 4, 1, 2)).astype(np.float32), 4, axis=0)
        out = be.sim.step(act, None)
    torch.cuda.synchronize()
    st = out['state'].cpu().numpy().reshape(N // 4, 4, 7)
    sc = out['scans_f64'].cpu().numpy().reshape(N // 4, 4, 1080)
    assert np.isfinite(st).all()
    assert (st == st[:, :1]).all() and (sc == sc[:, :1]).all()
    assert sc.max() <= 30.0 and sc.min() >= 0.0
    obs = out['obs'].cpu().numpy()
    assert obs[:, :1080].min() >= 0.0 and obs[:, :1080].max() <= 1.0
    # checkpoint round trip
    sd = be.sim.state_dict()
    act = rng.uniform([-0.4189, 0], [0.4189, 10], size=(N, 1, 2)).astype(np.float32)
    a1 = {k: v.clone() for k, v in be.sim.step(act, None).items()}
    be.sim.load_state_dict(sd)
    a2 = be.sim.step(act, None)
    torch.cuda.synchronize()
    for k in a1:
        assert torch.equal(a1[k], a2[k]), k


def test_device_noise_statistics():
    """Throughput mode: on-device Philox + Box-Muller noise ~ N(0, 0.01^2), independent across envs."""
    torch = _torch()
    N = 512
    be = GpuBackend(N, 1, 'open_square', noise_std=0.01, seed=7)
    poses = np.zeros((N, 1, 3))
    a = {k: v.clone() for k, v in be.sim.reset(poses, None).items()}
    clean = GpuBackend(1, 1, 'open_square')
    c = clean.reset(poses[:1], np.zeros((1, 1, 1080)))
    torch.cuda.synchronize()
    nz = a['scans_f64'].cpu().numpy()[:, 0] - c['scans'][0, 0][None]
    assert abs(nz.mean()) < 2e-4 and abs(nz.std() - 0.01) < 2e-4
    assert abs(np.corrcoef(nz[0], nz[1])[0, 1]) < 0.15
    k = ((nz / 0.01) ** 4).mean()
    assert 2.8 < k < 3.2


def test_device_noise_law_and_stream_semantics():
    """The on-device noise stream beyond its first two moments: Kolmogorov-Smirnov against N(0, 0.01^2) over 1.1e6 rays,
    the Box-Muller tail (u1 has 24 bits: |z| <= sqrt(50 ln 2) = 5.89), no correlation between neighbouring beams, between
    consecutive steps of the same ray or between envs, and the reference's episode semantics -- RaceCar.reset re-seeds the
    generator (base_classes.py:204), so every reset replays the same noise."""
    from scipy import stats
    N = 512
    be = GpuBackend(N, 1, 'open_square', noise_std=0.01, seed=11)
    ref = GpuBackend(1, 1, 'open_square')                     # the same env without noise: every env of `be` is this one
    poses = np.zeros((N, 1, 3))
    zero, none = np.zeros((N, 1, 2), np.float32), np.zeros((1, 1, 1080))
    clean = [ref.reset(poses[:1], none)['scans'][0, 0]] + [ref.step(zero[:1], none)['scans'][0, 0].copy() for _ in range(2)]
    noisy = [be.reset(poses, None)['scans'][:, 0]] + [be.step(zero, None)['scans'][:, 0].copy() for _ in range(2)]
    first, second, third = (n - c[None] for n, c in zip(noisy, clean))
    z = np.concatenate([first.ravel(), second.ravel()]) / 0.01
    d, _ = stats.kstest(z, 'norm')
    assert d < 0.004, d                                        # 1.1e6 samples: the 0.1 % critical value is 0.0019
    assert 4.0 < np.abs(z).max() < 5.95
    rho = lambda a, b: abs(np.corrcoef(a.ravel(), b.ravel())[0, 1])
    assert rho(first[:, :-1], first[:, 1:]) < 0.008            # neighbouring beams (5.5e5 pairs: sigma = 0.0013)
    assert rho(first, second) < 0.008 and rho(second, third) < 0.008       # the same ray, consecutive steps
    assert rho(first[:-1], first[1:]) < 0.008                  # the same ray of neighbouring envs
    again = be.reset(poses, None)['scans'][:, 0]
    assert np.array_equal(again, noisy[0])                     # a reset restarts the stream
    assert np.array_equal(be.step(zero, None)['scans'][:, 0], noisy[1])


def test_env_api_matches_reference_surface(tmp_path):
    """F110Env drop-in: kwargs, return types, info keys/dtypes (f110_env.py:586-602) and the golden rollout."""
    _torch()
    import f110_gymnasium_ros2_jazzy_b200 as f
    map_dir, name = H.write_map_files('Shanghai_map', str(tmp_path))
    env = f.make('f110_gym:f110-v0', map_dir=map_dir, map=name, map_ext='.png', num_agents=2)
    s, c, a, bc, sd = H.tables()
    env.sim.backend.set_tables(s, c)
    g = H.load('rollout_const_shanghai')
    obs, info = env.reset(options=g['poses'])
    assert obs.dtype == np.float32 and obs.shape == (1088,)
    assert info['time'] == pytest.approx(0.01)
    assert np.abs(obs - g['obs'][0]).max() <= 1e-6
    for k, dt_ in [('poses_x', np.float32), ('poses_y', np.float32), ('poses_theta', np.float32),
                   ('linear_vels_x', np.float32), ('linear_vels_y', np.float32), ('ang_vels_z', np.float32),
                   ('collisions', np.int8), ('lap_times', np.float32), ('lap_counts', np.float32)]:
        assert info[k].dtype == dt_ and info[k].shape == (2,), k
    assert len(info['scans']) == 2 and info['scans'][1].dtype == np.float32 and info['scans'][1].shape == (1080,)
    first_term = None
    for t in range(g['actions'].shape[0]):
        obs, r, term, trunc, info = env.step(g['actions'][t])
        assert r == 0.01 and trunc is False and isinstance(term, bool)
        assert term == bool(g['terminated'][t + 1]), t
        assert np.array_equal(info['collisions'], g['collisions'][t + 1].astype(np.int8))
        if term and first_term is None:
            first_term = t
    assert first_term == 220     # SURVEY 8c: ego terminates (TTC) at the 221st step
    with pytest.raises(ValueError):
        env.reset(options=np.zeros((3, 3)))
    with pytest.raises(IndexError):
        env.update_params(env.params, index=5)
    env.close()


def test_map_not_set_raises():
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import BatchSim
    sim = BatchSim(2, 1)
    with pytest.raises(ValueError, match="Map is not set"):
        sim.step(None)


def test_step_host_matches_device_path():
    torch = _torch()
    N = 32
    be = GpuBackend(N, 2, 'open_square')
    b2 = GpuBackend(N, 2, 'open_square')
    rng = np.random.default_rng(3)
    poses = np.zeros((N, 2, 3)); poses[:, 1, 0] = 2.0; poses[:, :, 1] = rng.uniform(-3, 3, size=(N, 1))
    noise = rng.normal(0, 0.01, size=(N, 2, 1080))
    d = be.reset(poses, noise)
    h = b2.sim.step_host(None, noise, np.ones(N, np.uint8), poses)
    for t in range(5):
        act = rng.uniform([-0.4, 0], [0.4, 8], size=(N, 2, 2)).astype(np.float32)
        d = be.step(act, noise)
        h = b2.sim.step_host(act, noise)
    for k in ('obs', 'state', 'scans_f64', 'terminated', 'collisions'):
        assert np.array_equal(d[k], h[k].numpy()), k


@pytest.mark.parametrize("A,chunks,extra", [(1, 3, ()), (2, (1, 3), ('scans_f32', 'state', 'toggles')), (2, 1, ('scans_f64',))])
def test_host_vec_env_matches_device_vec_env(A, chunks, extra):
    """F110HostVecEnv (chunked f110_step_host_async pipeline, block-laid-out pinned buffers, merged copies) == one F110VecEnv
    batch, noise off, auto-reset on -- one and two cars, even and uneven chunks, with and without extra outputs."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import FAST_OUTPUTS, F110HostVecEnv, F110VecEnv
    N = 96
    m = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    idx = np.linspace(0, len(cl) - 1, N).round().astype(int)
    poses = np.stack([cl[(idx + 25 * a) % len(cl)] for a in range(A)], axis=1)
    outs = FAST_OUTPUTS + tuple(extra)
    dev = F110VecEnv(N, num_agents=A, map_arrays=m, noise_std=0.0, outputs=outs)
    host = F110HostVecEnv(N, chunks=chunks, map_arrays=m, num_agents=A, noise_std=0.0, outputs=outs)
    rng = np.random.default_rng(11)
    od, _ = dev.reset(poses)
    oh, _ = host.reset(poses)
    torch.cuda.synchronize()
    assert np.array_equal(od.cpu().numpy(), oh)
    terms = 0
    for t in range(150):
        act = rng.uniform([-0.4189, 0], [0.4189, 20], size=(N, A, 2)).astype(np.float32)
        od, rd, td, _, infod = dev.step(torch.from_numpy(act).cuda())
        oh, rh, th, _, infoh = host.step(act)
        torch.cuda.synchronize()
        assert np.array_equal(td.cpu().numpy(), th), t
        assert np.array_equal(od.cpu().numpy(), oh), t
        assert np.array_equal(rd.cpu().numpy(), rh), t
        for k in extra:
            assert np.array_equal(infod[k].cpu().numpy(), infoh[k].numpy()), (k, t)
        terms += int(th.sum())
    assert terms > 0      # the auto-reset path was exercised
    host.close(); dev.close()


def test_host_vec_env_send_recv_pipeline():
    """send/recv per chunk, with the chunks out of phase across step boundaries, gives every chunk exactly the
    trajectory the synchronous step() gives it."""
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import F110HostVecEnv
    N, K, T = 90, 3, 60
    m = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    poses = cl[np.linspace(0, len(cl) - 1, N).round().astype(int)][:, None, :]
    sync = F110HostVecEnv(N, chunks=K, map_arrays=m, num_agents=1, noise_std=0.01)
    pipe = F110HostVecEnv(N, chunks=K, map_arrays=m, num_agents=1, noise_std=0.01)
    sync.reset(poses); pipe.reset(poses)
    acts = np.random.default_rng(5).uniform([-0.4189, 0], [0.4189, 20], size=(T, N, 1, 2)).astype(np.float32)
    want = []
    for t in range(T):
        o, r, d, _, _ = sync.step(acts[t])
        want.append((o.copy(), r.copy(), d.copy()))
    # chunk k runs k steps ahead of chunk K-1: start them staggered, then recv/send round-robin
    step_of = [0] * K
    for k in range(K):
        pipe.send(k, acts[0][pipe.chunk_slice(k)])
    done = 0
    while done < K:
        done = 0
        for k in range(K):
            if step_of[k] >= T:
                done += 1
                continue
            o, r, d = pipe.recv(k)
            t = step_of[k]
            sl = pipe.chunk_slice(k)
            assert np.array_equal(o, want[t][0][sl]), (k, t)
            assert np.array_equal(r, want[t][1][sl]) and np.array_equal(d, want[t][2][sl]), (k, t)
            step_of[k] += 1
            if step_of[k] < T:
                pipe.send(k, acts[step_of[k]][sl])
                if k == 0 and step_of[k] + 1 < T and step_of[k] % 7 == 0:      # let chunk 0 run ahead now and then
                    o, r, d = pipe.recv(0)
                    assert np.array_equal(o, want[step_of[0]][0][sl])
                    step_of[0] += 1
                    pipe.send(0, acts[step_of[0]][sl])
    sync.close(); pipe.close()


def test_step_is_cuda_graph_capturable():
    """f110_step neither allocates nor synchronises: a step can be captured and replayed by torch.cuda.graph."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    N = 64
    m = H.golden_map('open_square')
    a = BatchSim(N, 2, outputs=ALL_OUTPUTS, noise_std=0.0); a.set_map_arrays(*m)
    b = BatchSim(N, 2, outputs=ALL_OUTPUTS, noise_std=0.0); b.set_map_arrays(*m)
    rng = np.random.default_rng(2)
    poses = np.zeros((N, 2, 3)); poses[:, 1, 0] = 2.5; poses[:, :, 1] = rng.uniform(-4, 4, size=(N, 1))
    a.reset(poses); b.reset(poses)
    act = torch.zeros((N, 2, 2), dtype=torch.float32, device='cuda')
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        b.step(act)                       # warm-up on the side stream
    torch.cuda.current_stream().wait_stream(s)
    sd = b.state_dict()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.step(act)
    b.load_state_dict(sd)                 # undo the capture-time bookkeeping and the warm-up step
    a.step(act)
    for t in range(20):
        act.copy_(torch.from_numpy(rng.uniform([-0.4, 0], [0.4, 8], size=(N, 2, 2)).astype(np.float32)))
        a.step(act)
        g.replay()
    torch.cuda.synchronize()
    for k in a.out:
        assert torch.equal(a.out[k], b.out[k]), k


def test_gap_follow_kernel_bit_exact():
    """f110_gap_follow against the reference's gap_follow_action (golden) and the oracle, through strided views."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import gap_follow_actions
    from oracle.f110_oracle import gap_follow_action
    g = H.load('gap_follow')
    scans = g['scans']
    N = len(scans)
    rng = np.random.default_rng(9)
    more = rng.uniform(0, 5, size=(300, 1080)).astype(np.float32)
    more[:, 200:260] *= rng.uniform(0, 0.2, size=(300, 1)).astype(np.float32)
    allscans = np.concatenate([scans, more])
    M = len(allscans)
    t = torch.zeros((M, 2, 1080), dtype=torch.float32, device='cuda')
    t[:, 1] = torch.from_numpy(allscans).cuda()
    t[:, 0] = 7.0
    act = torch.full((M, 2, 2), -9.0, dtype=torch.float32, device='cuda')
    gap_follow_actions(t, act, agent_idx=1)
    torch.cuda.synchronize()
    a = act.cpu().numpy()
    assert (a[:, 0] == -9.0).all()                                   # the ego slot is untouched
    assert np.array_equal(a[:N, 1], g['actions'].astype(np.float32))
    ref = np.stack([gap_follow_action(s) for s in more]).astype(np.float32)
    assert np.array_equal(a[N:, 1], ref)
    # 8000 beams: 64 KB of dynamic shared memory, above the 48 KB a kernel gets without opting in
    wide = np.random.default_rng(9).uniform(0.3, 8.0, size=(3, 8000)).astype(np.float32)
    tw = torch.from_numpy(np.stack([wide, wide], axis=1).copy()).cuda()
    actw = torch.zeros((3, 2, 2), dtype=torch.float32, device='cuda')
    gap_follow_actions(tw, actw, agent_idx=1, angle_increment=np.pi / 8000)
    torch.cuda.synchronize()
    refw = np.stack([gap_follow_action(s, angle_increment=np.pi / 8000) for s in wide]).astype(np.float32)
    assert np.array_equal(actw.cpu().numpy()[:, 1], refw)
    # run structure: the kernel joins per-lane run summaries associatively -- blocky scans with runs of every length and
    # position (ends on lane boundaries, equal-length runs where the first must win, all / none above the threshold), and
    # beam counts around the warp size
    rs = np.random.default_rng(21)
    for nb in (31, 32, 33, 64, 100, 340, 1080, 1088):
        blocky = np.zeros((200, nb), np.float32)
        for row in blocky:
            i = 0
            while i < nb:
                ln = int(rs.choice([1, 2, 3, 5, 8, 13, 33, 34, 35, 68, 100]))
                row[i:i + ln] = rs.choice([0.0, 0.2, 0.6, 1.0, 3.0, 9.0])
                i += ln
        blocky[0] = 3.0; blocky[1] = 0.0; blocky[2] = 0.55
        if nb >= 100:
            blocky[3] = 0.0; blocky[3, 10:30] = 2.0; blocky[3, 60:80] = 2.0      # two equal runs far from the bubble's centre
        tb = torch.from_numpy(np.stack([blocky, blocky], axis=1).copy()).cuda()
        ab = torch.zeros((len(blocky), 2, 2), dtype=torch.float32, device='cuda')
        gap_follow_actions(tb, ab, agent_idx=1, angle_increment=np.pi / nb)
        torch.cuda.synchronize()
        refb = np.stack([gap_follow_action(sc, angle_increment=np.pi / nb) for sc in blocky]).astype(np.float32)
        assert np.array_equal(ab.cpu().numpy()[:, 1], refb), nb


def test_consumers_survive_non_finite_inputs():
    """The observation of a poisoned car (NaN pose, NaN/inf beams) goes through the gap-follow and reward kernels without
    a fault, the rows next to it come out exactly as they do without it, and the poisoned rows equal the oracle's."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward, gap_follow_actions
    from tests.test_oracle_golden import REWARD_KW
    g, r = H.load('gap_follow'), H.reward_recording()
    scans = g['scans'][:64].copy()
    bad = scans.copy()
    bad[5] = np.nan
    bad[9, 100:300] = np.inf
    bad[11, ::7] = -np.inf
    out = []
    for arr in (scans, bad):
        t = torch.zeros((64, 2, 1080), dtype=torch.float32, device='cuda')
        t[:, 1] = torch.from_numpy(arr).cuda()
        act = torch.zeros((64, 2, 2), dtype=torch.float32, device='cuda')
        gap_follow_actions(t, act, agent_idx=1)
        torch.cuda.synchronize()
        out.append(act.cpu().numpy())
    keep = np.ones(64, bool); keep[[5, 9, 11]] = False
    assert np.array_equal(out[0][keep], out[1][keep])
    from oracle.f110_oracle import RewardOracle, gap_follow_action
    for k in (5, 9, 11):
        assert np.array_equal(out[1][k, 1], gap_follow_action(bad[k]).astype(np.float32)), k

    obs = r['obs'][:8].copy()
    badobs = obs.copy()
    badobs[2, 1080:1083] = np.nan          # pose
    badobs[3, :1080] = np.nan              # lidar
    badobs[4, 1080] = np.inf
    from tests.test_consumer_kernels import DeviceMath, expected_reward
    dm = DeviceMath()
    res = []
    for arr in (obs, badobs):
        rw = ShapedReward(8, r['centerline'], **REWARD_KW)
        orc = RewardOracle(8, r['centerline'], **REWARD_KW)
        mask = torch.ones(8, dtype=torch.uint8, device='cuda')
        for _ in range(3):
            got = rw(torch.from_numpy(arr).cuda(), mask)
            tot, terms = orc.compute_terms(arr, mask.cpu().numpy())
            mask = torch.zeros(8, dtype=torch.uint8, device='cuda')
            torch.cuda.synchronize()
            want, _ = expected_reward(dm, arr, tot, terms, 1080, REWARD_KW)
            assert np.array_equal(got.cpu().numpy(), want, equal_nan=True)
        res.append(got.cpu().numpy())
        rw.close()
    keep = np.ones(8, bool); keep[[2, 3, 4]] = False
    assert np.array_equal(res[0][keep], res[1][keep])


def test_device_rollout_runs_without_host_sync():
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import Actor, DeviceRollout, F110VecEnv
    N = 64
    m = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    idx = np.linspace(0, len(cl) - 1, N).round().astype(int)
    poses = np.stack([cl[idx], cl[(idx + 40) % len(cl)]], axis=1)
    env = F110VecEnv(N, num_agents=2, map_arrays=m, outputs=('obs', 'reward', 'terminated', 'scans_f32', 'state'))
    torch.manual_seed(42)
    actor = Actor(1088, 2, [-0.4189, 0.0], [0.4189, 20.0]).cuda()
    ro = DeviceRollout(env, actor)
    ro.reset(poses)
    for _ in range(50):
        obs, r, term, trunc, info = ro.step()
    torch.cuda.synchronize()
    st = info['state'].cpu().numpy()
    assert np.isfinite(st).all() and obs.shape == (N, 1088)
    # the gap-follow opponent drives (its speed can exceed the 2.5 m/s command: with the env's default v_min = 1e-8 a
    # braking request accelerates, the pid quirk of dynamic_models.py:204-219 that is reproduced on purpose)
    assert (st[:, 1, 3] > 0.5).mean() > 0.5
    env.close()


def test_device_rollout_fills_device_replay_buffer():
    """DeviceRollout(replay=DeviceReplayBuffer): every transition lands in the device buffer in env order --
    (obs before the step, the ego action that was applied, reward, obs after, done) -- and a prioritised batch can be
    drawn, all without a host copy (train_ddpg.py:160-188's remember / replay shape).  The step that auto-resets an env
    which terminated on the previous step is the reference's env.reset() between episodes (:152), not a transition: it
    must not reach the buffer (the reference breaks on done, :197), its reward is 0, and the shaped reward restarts so
    that its first value of the new episode is computed on the first real next_obs."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import Actor, DeviceReplayBuffer, DeviceRollout, F110VecEnv, ShapedReward
    N, T = 32, 60
    m = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    idx = np.linspace(0, len(cl) - 1, N).round().astype(int)
    poses = np.stack([cl[idx], cl[(idx + 40) % len(cl)]], axis=1)
    env = F110VecEnv(N, num_agents=2, map_arrays=m, outputs=('obs', 'reward', 'terminated', 'scans_f32'))

    class FullLock(torch.nn.Module):                  # steers into the wall at speed: episodes end within the rollout
        def forward(self, obs):
            return torch.tensor([0.4189, 9.0], device=obs.device).expand(obs.shape[0], 2)
    g = H.load('reward')
    rfn = ShapedReward(N, g['centerline'])
    solo = ShapedReward(N, g['centerline'])           # the same reward objects driven by hand, reset exactly at episode starts
    buf = DeviceReplayBuffer(capacity=N * T, batch_size=64, device='cuda')
    ro = DeviceRollout(env, FullLock(), reward_fn=rfn, replay=buf)
    obs0 = ro.reset(poses).clone()
    want, resetting_prev, first = [], torch.zeros(N, dtype=torch.bool, device='cuda'), torch.ones(N, dtype=torch.bool, device='cuda')
    n_reset_steps = 0
    for t in range(T):
        before = ro.obs.clone()
        resetting = env.backend.out['terminated'].clone().bool()          # envs this step auto-resets
        obs, r, term, trunc, info = ro.step()
        # hand-driven reference: no call at all on a reset step; restart flag on the first real step of an episode
        expect = solo(obs.clone(), (first | resetting).to(torch.uint8)).clone()   # (value on reset steps is discarded, as in the rollout)
        real = ~resetting
        assert torch.all(r[resetting] == 0)
        assert torch.equal(r[real], expect[real])
        n_reset_steps += int(resetting.sum())
        for e in torch.nonzero(real).flatten().tolist():
            want.append((before[e].clone(), ro.actions[e, 0].clone(), r[e].clone(), obs[e].clone(), term[e].clone()))
        first = resetting
    torch.cuda.synchronize()
    assert n_reset_steps > 0, "the scenario must contain terminations"
    assert len(buf) == N * T - n_reset_steps == len(want) and buf.obs.is_cuda
    for k, (o, a, r, no, d) in enumerate(want):
        assert torch.equal(buf.obs[k], o) and torch.equal(buf.next_obs[k], no) and torch.equal(buf.action[k], a)
        assert float(buf.reward[k]) == float(r.float()) and int(buf.done[k]) == int(d)
    assert torch.equal(buf.obs[:N], obs0)
    idxs, (o, a, r, no, d), w = buf.sample(beta=0.4)
    assert o.shape == (64, 1088) and w.is_cuda and float(w.max()) == 1.0 and len(set(idxs.tolist())) == 64
    buf.update_priorities(idxs, torch.rand(64, device='cuda') + 0.1)
    # a second reset() of the rollout restarts every reward object on the next step
    ro.reset(poses)
    ro.step()
    assert bool(torch.all(ro._fresh == 1))
    env.close()


def test_checkpoint_is_versioned_and_env_level_resume_is_exact():
    """f110_get_state / f110_set_state carry a header (magic, layout version, N, A, B): a blob of another shape or a corrupted
    one is refused.  F110VecEnv.state_dict adds what lives above the C ABI (terminated flags = next reset mask, start
    poses): a fresh env loaded from it continues bit for bit, including the auto-reset of envs that had just terminated."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import F110VecEnv
    N = 64
    m = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    poses = cl[np.linspace(0, len(cl) - 1, N).round().astype(int)][:, None, :]
    kw = dict(num_agents=1, map_arrays=m, outputs=('obs', 'reward', 'terminated', 'state'), noise_std=0.01, seed=7)
    env = F110VecEnv(N, **kw)
    env.reset(poses)
    g = torch.Generator(device='cuda'); g.manual_seed(3)
    acts = torch.rand((80, N, 1, 2), generator=g, device='cuda') * torch.tensor([0.8378, 12.0], device='cuda') + torch.tensor([-0.4189, 2.0], device='cuda')
    for k in range(40):
        env.step(acts[k])
    assert int(env.backend.out['terminated'].sum()) >= 0
    sd = env.state_dict()
    ref = []
    for k in range(40, 80):
        o, r, t, _, info = env.step(acts[k])
        ref.append((o.clone(), t.clone(), info['state'].clone()))
    # a second env, as another process would build it
    env2 = F110VecEnv(N, **kw)
    env2.reset(poses[::-1].copy())            # different history before the load
    env2.load_state_dict(sd)
    for k in range(40, 80):
        o, r, t, _, info = env2.step(acts[k])
        assert torch.equal(o, ref[k - 40][0]) and torch.equal(t, ref[k - 40][1]) and torch.equal(info['state'], ref[k - 40][2]), k
    # the blob is refused by a handle of another shape, and when its header is damaged
    env3 = F110VecEnv(N // 2, **kw)
    with pytest.raises(Exception):
        env3.backend.load_state_dict(dict(sd['backend'], N=N // 2))
    bad = dict(sd['backend'], blob=sd['backend']['blob'].clone())
    bad['blob'][0] ^= 0xFF
    with pytest.raises(Exception):
        env2.backend.load_state_dict(bad)
    for e in (env, env2, env3):
        e.close()


def test_cuda_graph_is_dropped_when_the_map_changes():
    """The step kernels take the map descriptor by value: a graph captured before set_map would replay with the freed map.
    F110VecEnv re-captures (also when the map is changed on the backend directly)."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import F110VecEnv
    N = 32
    m1 = H.golden_map('Shanghai_map')
    dt2, res2, o2 = H.golden_map('open_square')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    poses = np.zeros((N, 1, 3)); poses[:, 0, 0] = np.linspace(-3, 3, N)
    kw = dict(num_agents=1, outputs=('obs', 'reward', 'terminated', 'scans_f64'), noise_std=0.0)
    envs = [F110VecEnv(N, map_arrays=m1, cuda_graph=cg, **kw) for cg in (True, False)]
    act = torch.zeros((N, 1, 2), device='cuda'); act[..., 1] = 1.0
    for e in envs:
        e.reset(cl[np.linspace(0, len(cl) - 1, N).round().astype(int)][:, None, :])
        for _ in range(4):
            e.step(act)
    assert envs[0]._graph is not None
    envs[0].backend.set_map_arrays(dt2, res2, o2)        # behind the env's back
    envs[1].set_map_arrays(dt2, res2, o2)
    for e in envs:
        e.reset(poses)
        for _ in range(4):
            e.step(act)
    torch.cuda.synchronize()
    assert envs[0]._graph is not None
    assert torch.equal(envs[0].backend.out['scans_f64'], envs[1].backend.out['scans_f64'])
    for e in envs:
        e.close()


def test_c4_full_size_sharded_properties():
    """BASELINE config 4 size: 262 144 envs on one handle (the 1-GPU end of the sweep).  Replicated start poses must
    give replicated results across the whole batch (index arithmetic survives 2.8e8 rays), outputs stay in range,
    and the launch-order history must not change any result (same step from the same checkpoint, twice)."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import BatchSim
    N = 262144
    free, total = torch.cuda.mem_get_info()
    if free < 12 * 2**30:
        pytest.skip("needs ~8 GB of device memory")
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    R = 512
    base = cl[np.linspace(0, len(cl) - 1, R).round().astype(int)]
    poses = np.tile(base[None], (N // R, 1, 1)).reshape(N, 1, 3)      # env e has pose base[e % R]
    sim = BatchSim(N, 1, outputs=('obs', 'terminated', 'state'), noise_std=0.0)
    sim.set_map_arrays(*H.golden_map('Shanghai_map'))
    sim.reset(torch.from_numpy(poses).cuda())
    rng = np.random.default_rng(17)
    for t in range(6):
        a = rng.uniform([-0.4189, 0], [0.4189, 12], size=(R, 1, 2)).astype(np.float32)
        act = torch.from_numpy(np.tile(a[None], (N // R, 1, 1, 1)).reshape(N, 1, 2)).cuda()
        out = sim.step(act)
    torch.cuda.synchronize()
    obs = out['obs'].view(N // R, R, -1)
    assert torch.equal(obs, obs[:1].expand_as(obs))
    st = out['state'].view(N // R, R, 7)
    assert torch.equal(st, st[:1].expand_as(st)) and torch.isfinite(st).all()
    assert float(out['obs'][:, :1080].min()) >= 0.0 and float(out['obs'][:, :1080].max()) <= 1.0
    sd = sim.state_dict()
    o1 = {k: v.clone() for k, v in sim.step(act).items()}
    sim.load_state_dict(sd)
    o2 = sim.step(act)          # same state, different launch-order history
    torch.cuda.synchronize()
    for k in o1:
        assert torch.equal(o1[k], o2[k]), k
    sim.close()


@pytest.mark.parametrize('form', ['warp', 'cta'])
def test_shaped_reward_kernel_matches_reference_and_oracle(form, monkeypatch):
    """f110_reward_compute: (a) the recorded reference episodes, each replayed in its own env slot of one batch, within
    1e-9 of the reference (numpy, BLAS and glibc there), (b) the oracle on the same batch of independent envs, exactly,
    once its opponent and flank terms are recomputed with the device's hypot and sincos.  Both forms of the kernel: a warp
    per env (the default) and a CTA per env (scans too long for a warp's shared memory; forced)."""
    monkeypatch.setenv('F110_REWARD_CTA', '1' if form == 'cta' else '0')
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward
    from oracle.f110_oracle import RewardOracle
    from tests.test_consumer_kernels import DeviceMath, expected_reward
    from tests.test_oracle_golden import REWARD_ALT_KW, REWARD_KW
    dm = DeviceMath()
    g = H.reward_recording()
    obs, starts = g['obs'], g['episode_start']
    T = len(obs)
    for kw, key in ((REWARD_KW, 'reward'), (REWARD_ALT_KW, 'reward_alt')):
        # env slot 0 replays the recording; slots 1..3 replay it shifted in time (independent state per env)
        N = 4
        rw = ShapedReward(N, g['centerline'], **kw)
        orc = RewardOracle(N, g['centerline'], **kw)
        for t in range(T):
            batch = np.stack([obs[(t + 37 * k) % T] for k in range(N)])
            mask = np.array([starts[(t + 37 * k) % T] or t == 0 for k in range(N)], np.uint8)
            got = rw(torch.from_numpy(batch).cuda(), torch.from_numpy(mask).cuda()).cpu().numpy()
            tot, terms = orc.compute_terms(batch, mask)
            want, _ = expected_reward(dm, batch, tot, terms, 1080, kw)
            assert np.array_equal(got, want), (key, t, got, want)
            assert abs(got[0] - g[key][t]) < 1e-9, (key, t, got[0], g[key][t])
        rw.close()


def test_device_edt_bit_identical_to_scipy():
    """f110_set_map_image: the exact integer EDT on the device reproduces resolution * scipy.ndimage.distance_transform_edt
    (laser_models.py:40-53) bit for bit -- on the three fixture maps and on random occupancy with thin / isolated obstacles."""
    _torch()
    from scipy.ndimage import distance_transform_edt
    from f110_gymnasium_ros2_jazzy_b200 import BatchSim
    sim = BatchSim(1, 1)
    m = H.load('maps')
    for name in ('Shanghai_map', 'straight_corridor', 'open_square'):
        shape = tuple(int(v) for v in m[name + '__shape'])
        free = np.unpackbits(m[name + '__bits'])[:shape[0] * shape[1]].reshape(shape)
        ref, res, origin = H.golden_map(name)
        sim.set_map_image(free, res, origin)
        got = sim.get_map()
        assert got.shape == ref.shape and np.array_equal(got, ref), name
    rng = np.random.default_rng(4)
    for shape, p in (((257, 131), 0.01), ((64, 700), 0.2), ((300, 300), 0.0005), ((5, 1000), 0.05), ((1, 77), 0.1), ((200, 1), 0.05),
                     ((130, 1030), 0.00002)):
        free = (rng.uniform(size=shape) > p).astype(np.uint8)
        free[rng.integers(0, shape[0]), rng.integers(0, shape[1])] = 0      # at least one obstacle
        ref = 0.0731 * distance_transform_edt(np.where(free, 255., 0.))
        # both forms: the banded 16-bit kernels every real map takes, and the general one (H + W > 32766), forced
        for wide in ('0', '1'):
            os.environ['F110_EDT_WIDE'] = wide
            try:
                sim.set_map_image(free, 0.0731, [0.0, 0.0, 0.0])
            finally:
                os.environ.pop('F110_EDT_WIDE')
            assert np.array_equal(sim.get_map(), ref), (shape, wide)
        assert sim.edt_kernel_ms() > 0.0
    # and the scans taken on a device-built map equal the ones on the host-built map
    g = H.load('scans')
    poses = g['Shanghai_map__poses']
    be = GpuBackend(len(poses), 1, 'Shanghai_map')
    shape = tuple(int(v) for v in m['Shanghai_map__shape'])
    free = np.unpackbits(m['Shanghai_map__bits'])[:shape[0] * shape[1]].reshape(shape)
    _, res, origin = H.golden_map('Shanghai_map')
    be.sim.set_map_image(free, res, origin)
    be.sim.sim_reset(poses[:, None, :])
    out = be.step(None, np.zeros((len(poses), 1, 1080)))
    assert np.array_equal(out['scans'][:, 0], g['Shanghai_map__scans'])
    sim.close()


def test_ros_bridge_call_sequence_as_written(tmp_path):
    """The literal call sequence of jazzy_bridge/.../gym_bridge.py, nothing added: gym.make('f110_gym:f110-v0', map=<path
    without extension>, map_ext=..., num_agents=...) (:77-80), reset(options=np.array([[sx, sy, stheta], [sx1, sy1, stheta1]]))
    followed by list(obs[0]) / list(obs[1]) (:112-114), step(np.array([[steer, speed], [steer, speed]])) in float64 (:224-229),
    _update_sim_state's reads of obs[i] and info['poses_x' | 'poses_y' | 'poses_theta' | 'linear_vels_x' | 'linear_vels_y' |
    'ang_vels_z'][i] (:264-280), and the pose-reset callbacks (:197-210).  'f110_gym' resolves through the alias package at
    the repository root exactly as gymnasium resolves a 'module:id' string; the scans layout is selected by the bridge's own
    calling convention (map= without map_dir=)."""
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import gym_compat as gym        # gymnasium itself when it is installed
    map_dir, name = H.write_map_files('open_square', str(tmp_path))
    map_path = map_dir + name
    sx, sy, stheta, sx1, sy1, stheta1 = 0.0, 0.0, 0.0, 2.0, 0.5, 0.0
    # ---- two agents (:77-80, :100-114)
    env = gym.make('f110_gym:f110-v0', map=map_path, map_ext='.png', num_agents=2)
    obs, info = env.reset(options=np.array([[sx, sy, stheta], [sx1, sy1, stheta1]]))
    ego_scan = list(obs[0]); opp_scan = list(obs[1])
    assert len(ego_scan) == 1080 and len(opp_scan) == 1080 and isinstance(ego_scan[0], np.floating)
    ego_pose, ego_speed, opp_pose, opp_speed = [sx, sy, stheta], [0.0, 0.0, 0.0], [sx1, sy1, stheta1], [0.0, 0.0, 0.0]
    ego_steer, ego_requested_speed, opp_steer, opp_requested_speed = 0.3, 1.0, 0.0, 1.5
    for _ in range(20):
        obs, reward, terminated, truncated, info = env.step(np.array([[ego_steer, ego_requested_speed], [opp_steer, opp_requested_speed]]))
        ego_scan = list(obs[0])
        opp_scan = list(obs[1])
        opp_pose[0] = info['poses_x'][1]; opp_pose[1] = info['poses_y'][1]; opp_pose[2] = info['poses_theta'][1]
        opp_speed[0] = info['linear_vels_x'][1]; opp_speed[1] = info['linear_vels_y'][1]; opp_speed[2] = info['ang_vels_z'][1]
        ego_pose[0] = info['poses_x'][0]; ego_pose[1] = info['poses_y'][0]; ego_pose[2] = info['poses_theta'][0]
        ego_speed[0] = info['linear_vels_x'][0]; ego_speed[1] = info['linear_vels_y'][0]; ego_speed[2] = info['ang_vels_z'][0]
    assert reward == env.unwrapped.timestep and truncated is False and terminated in (True, False)
    assert opp_pose[0] > sx1 and ego_pose[2] > 0.0 and ego_speed[1] == 0.0 and np.isfinite(ego_speed + opp_speed).all()
    assert len(ego_scan) == 1080 and max(ego_scan) <= 30.05
    # pose reset from rviz (:197, :210)
    rx, ry, rtheta = -1.0, 1.0, 0.5
    obs, info = env.reset(options=np.array([[rx, ry, rtheta], opp_pose]))
    assert abs(info['poses_x'][0] - rx) < 1e-6 and len(list(obs[1])) == 1080
    obs, info = env.reset(options=np.array([list(ego_pose), [rx, ry, rtheta]]))
    assert abs(info['poses_y'][1] - ry) < 1e-6
    env.close()
    # ---- one agent (:124-125, :226)
    env = gym.make('f110_gym:f110-v0', map=map_path, map_ext='.png', num_agents=1)
    obs, info = env.reset(options=np.array([[sx, sy, stheta]]))
    ego_scan = list(obs[0])
    obs, reward, terminated, truncated, info = env.step(np.array([[ego_steer, ego_requested_speed]]))
    assert len(list(obs[0])) == 1080 and info['poses_x'].shape == (1,)
    env.close()


def test_train_ddpg_loop_shape(tmp_path):
    """rl_training/train_ddpg.py:58-65 and :150-202 with the env swapped in and nothing else changed in the calls: gym.make(
    'f110_gym:f110-v0', render_mode=..., map_dir=..., map=..., map_ext=..., num_agents=2), reset(options=float32 start poses),
    then per step the opponent's action from info["scans"][1], np.stack([ego, opp]).astype(float32), env.step(actions) ->
    (next_obs, _, terminated, truncated, info), the shaped reward on next_obs, done = terminated or truncated.  The opponent
    is the reference's gap-follow controller (oracle restatement, pinned on tests/golden/gap_follow.npz); the whole rollout is
    compared with the oracle stepping the same actions."""
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import gym_compat as gym
    from oracle.f110_oracle import Oracle, gap_follow_action as gap_follow
    map_dir, name = H.write_map_files('Shanghai_map', str(tmp_path))
    env = gym.make('f110_gym:f110-v0', render_mode='human_fast', map_dir=map_dir, map=name, map_ext='.png', num_agents=2)
    assert env.unwrapped.timestep == 0.01
    start_poses = [[0.0, 0.0, 0.0], [3.0, 0.5, 0.0]]                         # ddpg_config.yaml:11-12
    orc = Oracle(1, 2); orc.set_map_arrays(*H.golden_map('Shanghai_map'))
    s, c, a, bc, sd = H.tables(); orc.set_tables(s, c); orc.set_beam_tables(a, bc, sd)
    rng = np.random.default_rng(0)
    nz = np.random.default_rng(42)                                          # the env's lidar noise stream (seed 42, re-seeded on reset)
    obs, info = env.reset(options=np.array(start_poses, dtype=np.float32))
    noise = nz.normal(0., 0.01, size=1080)
    ref = orc.reset(np.array(start_poses, dtype=np.float32).astype(np.float64)[None], np.broadcast_to(noise, (1, 2, 1080)))
    assert obs.shape == (1088,) and obs.dtype == np.float32
    assert np.abs(obs - ref['obs'][0]).max() <= 1e-6
    steps, done = 0, False
    action_low, action_high = np.array([-0.4189, 0.0], np.float32), np.array([0.4189, 6.0], np.float32)
    for step in range(120):
        ego_action = rng.uniform(low=action_low, high=action_high).astype(np.float32)
        opp_action = gap_follow(info["scans"][1]).astype(np.float32)
        actions = np.stack([ego_action, opp_action], axis=0).astype(np.float32)
        next_obs, _, terminated, truncated, info = env.step(actions)
        noise = nz.normal(0., 0.01, size=1080)
        ref = orc.step(actions[None], np.broadcast_to(noise, (1, 2, 1080)))
        assert bool(terminated) == bool(ref['terminated'][0]) and truncated is False
        assert np.array_equal(info['collisions'], ref['collisions'][0].astype(np.int8))
        assert np.abs(next_obs - ref['obs'][0]).max() <= 1e-6
        assert (np.abs(info['scans'][1] - ref['scans'][0, 1].astype(np.float32)) <= 1e-5).mean() >= SCAN_FRAC
        done = bool(terminated or truncated)
        obs = next_obs
        steps += 1
        if done:
            break
    assert steps >= 20
    env.close()


@pytest.mark.parametrize("num_envs,num_agents,num_beams,fov", [(5, 16, 1080, 4.7), (33, 6, 64, 3.0), (7, 4, 4320, 4.7), (1, 2, 32, 1.0),
                                                              (6, 3, 720, 6.2),    # 355-degree lidar: no cone pruning in K3, beams wrap the table
                                                              (3, 1, 270, 4.7), (2, 2, 541, 4.7),    # C4's shortest scan; an odd beam count
                                                              (2, 1, 2160, 4.7)])
def test_shape_extremes_vs_oracle(num_envs, num_agents, num_beams, fov):
    """Edges of the supported shapes: the maximum agent count (one env per post-kernel CTA), the minimum beam count, a
    non-default field of view, 4320 beams, ragged env counts, the beam counts of BASELINE config 4's sweep that are not
    multiples of a warp, an odd beam count -- each against the oracle with injected noise."""
    from f110_gymnasium_ros2_jazzy_b200.params import beam_tables, default_params, theta_tables
    rng = np.random.default_rng(1000 + num_agents)
    be = GpuBackend(num_envs, num_agents, 'open_square', num_beams=num_beams, fov=fov)
    orc = make_oracle(num_envs, num_agents, 'open_square', num_beams=num_beams, fov=fov)
    # the fixture tables are for 1080 beams / 4.7 rad: rebuild them for this shape, identically on both sides
    s, c = theta_tables(2000)
    a, bc, sd = beam_tables(default_params(), num_beams, fov)
    for x in (be.sim, orc):
        x.set_tables(s, c)
        x.set_beam_tables(a, bc, sd)
    poses = np.zeros((num_envs, num_agents, 3))
    poses[..., 0] = rng.uniform(-7, 7, size=(num_envs, num_agents))
    poses[..., 1] = rng.uniform(-7, 7, size=(num_envs, num_agents))
    poses[..., 2] = rng.uniform(-np.pi, np.pi, size=(num_envs, num_agents))
    if num_agents >= 2:
        poses[:, 1, :2] = poses[:, 0, :2] + rng.uniform(-0.3, 0.3, size=(num_envs, 2))     # a guaranteed overlap per env
    outl = beams = 0
    for t in range(40):
        noise = rng.normal(0, 0.01, size=(num_envs, num_agents, num_beams))
        if t == 0:
            g, o = be.reset(poses, noise), orc.reset(poses, noise)
            assert num_agents < 2 or g['collisions'][:, :2].all()          # the overlapping pair is flagged by GJK
        else:
            act = rng.uniform([-0.4189, 0], [0.4189, 6], size=(num_envs, num_agents, 2)).astype(np.float32)
            g, o = be.step(act, noise), orc.step(act, noise)
        for k in ('collisions', 'terminated', 'toggles'):
            assert np.array_equal(g[k], o[k]), (k, t)
        assert np.abs(g['state'] - o['state']).max() <= STATE_TOL
        d = np.abs(g['scans'] - o['scans'])
        outl += int((d > SCAN_TOL).sum()); beams += d.size
    assert outl <= (1 - SCAN_FRAC) * beams


def test_vec_env_cuda_graph_mode_matches_eager():
    """F110VecEnv(cuda_graph=True): capture once, replay per step -- same results as the eager env (noise off)."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import F110VecEnv
    N = 128
    m = H.golden_map('Shanghai_map')
    cl = H.load('maps')['Shanghai_map__centerline_poses']
    poses = cl[np.linspace(0, len(cl) - 1, N).round().astype(int)][:, None, :]
    a = F110VecEnv(N, num_agents=1, map_arrays=m, noise_std=0.0)
    b = F110VecEnv(N, num_agents=1, map_arrays=m, noise_std=0.0, cuda_graph=True)
    a.reset(poses); b.reset(poses)
    rng = np.random.default_rng(8)
    for t in range(120):
        act = torch.from_numpy(rng.uniform([-0.4189, 0], [0.4189, 18], size=(N, 1, 2)).astype(np.float32)).cuda()
        oa = a.step(act); ob = b.step(act)
        torch.cuda.synchronize()
        assert torch.equal(oa[0], ob[0]) and torch.equal(oa[2], ob[2]), t
    assert b._graph is not None
    a.close(); b.close()
