"""CPU suite: pins the oracle (oracle/f110_oracle.c) against
  (a) the reference's own embedded known-answer tests, and
  (b) golden vectors recorded from the unmodified reference (tests/golden/make_golden.py).
"""
import numpy as np
import pytest

from oracle.f110_oracle import DEFAULT_PARAMS, Oracle
from tests import helpers as H

# CommonRoad vehicle-2 parameters of the reference's DynamicsTest (dynamic_models.py:232-253)
TEST_PARAMS = dict(mu=1.0489, C_Sf=21.92 / 1.0489, C_Sr=21.92 / 1.0489, lf=0.3048 * 3.793293, lr=0.3048 * 4.667707,
                   h=0.3048 * 2.01355, m=4.4482216152605 / 0.3048 * 74.91452, I=4.4482216152605 * 0.3048 * 1321.416,
                   s_min=-1.066, s_max=1.066, sv_min=-0.4, sv_max=0.4, v_switch=7.319, a_max=11.5, v_min=-13.6,
                   v_max=50.8, width=0.31, length=0.58)


def make_oracle(num_agents, map_name, **kw):
    o = Oracle(1, num_agents, **kw)
    s, c, a, bc, sd = H.tables()
    o.set_tables(s, c)
    o.set_beam_tables(a, bc, sd)
    o.set_map_arrays(*H.golden_map(map_name))
    return o


def test_derivatives_known_answer():
    """dynamic_models.py:255-270 test_derivatives (assertAlmostEqual, 7 places -> we require 1e-12)."""
    f_ks_gt = [16.3475935934250209, 0.4819314886013121, 0.1500000000000000, 5.1464424102339752, 0.2401426578627629]
    f_st_gt = [15.7213512030862397, 0.0925527979719355, 0.1500000000000000, 5.3536773276413925, 0.0529001056654038,
               0.6435589397748606, 0.0313297971641291]
    g = 9.81
    x_ks = np.array([3.9579422297936526, 0.0391650102771405, 0.0378491427211811, 16.3546957860883566, 0.0294717351052816])
    x_st = np.array([2.0233348142065677, 0.0041907137716636, 0.0197545248559617, 15.7216236334290116, 0.0025857914776859,
                     0.0529001056654038, 0.0033012170610298])
    u = np.array([0.15, 0.63 * g])
    o = Oracle(1, 1)
    assert np.abs(o.vehicle_dynamics_ks(x_ks, u, TEST_PARAMS) - f_ks_gt).max() < 1e-12
    assert np.abs(o.vehicle_dynamics_st(x_st, u, TEST_PARAMS) - f_st_gt).max() < 1e-12


def _odeint_like(o, x0, u, t_final=1.0, dt=1e-4):
    """The reference integrates with scipy odeint (dynamic_models.py:281-423); a fine RK4 reproduces the
    end states well inside the 1e-2 the reference asserts."""
    x = np.array(x0, float)
    f = lambda s: o.vehicle_dynamics_st(s, u, TEST_PARAMS)
    for _ in range(int(round(t_final / dt))):
        k1 = f(x); k2 = f(x + dt * k1 / 2); k3 = f(x + dt * k2 / 2); k4 = f(x + dt * k3)
        x = x + dt / 6 * (k1 + 2 * k2 + 2 * k3 + k4)
    return x


@pytest.mark.parametrize("u,gt", [
    # test_zeroinit_roll :281-305
    ([0.0, 0.0], [0.0] * 7),
    # test_zeroinit_dec :307-345
    ([0.0, -0.7 * 9.81], [-3.4335000000000013, 0.0, 0.0, -6.8670000000000018, 0.0, 0.0, 0.0]),
    # test_zeroinit_acc :347-383
    ([0.0, 0.63 * 9.81], [3.0901500000000009, 0.0, 0.0, 6.1803000000000017, 0.0, 0.0, 0.0]),
    # test_zeroinit_rollleft :385-423
    ([0.15, 0.0], [0.0, 0.0, 0.15, 0.0, 0.0, 0.0, 0.0]),
])
def test_zeroinit_rollouts(u, gt):
    o = Oracle(1, 1)
    x = _odeint_like(o, np.zeros(7), np.array(u), dt=1e-3)
    assert np.abs(x - np.array(gt)).max() < 1e-2


def test_pid_brake_quirk():
    """SURVEY a6: with v_min=1e-8 a braking request yields a huge positive acceleration."""
    o = Oracle(1, 1)
    a, sv = o.pid(2.0, 0.0, 3.0, 0.0, 3.2, 9.51, 20.0, 1e-8)
    assert a == (10.0 * 9.51 / (-1e-8)) * (2.0 - 3.0) and a > 9e9 and sv == 0.0


def test_gjk_known_answer():
    """collision_models.py:273-324 CollisionTests: random-perturbation overlap + the exact multi-body result."""
    np.random.seed(1234)
    vertices1 = np.asarray([[4, 11.], [5, 5], [9, 9], [10, 10]])
    length, width = 0.32, 0.22
    o = Oracle(1, 1)
    for _ in range(1000):
        a = vertices1 + np.random.normal(size=(vertices1.shape)) / 100.
        b = vertices1 + np.random.normal(size=(vertices1.shape)) / 100.
        assert o.collision(a, b)
    vertices2 = np.asarray([[0, 0.], [1, 1], [3, 0], [2, 1]])   # unused by the reference's multi test as well
    all_vertices = np.stack([o.get_vertices(np.array(p, float), length, width) for p in
                             [[0, 0, 0], [0.2, 0.1, 0.1], [10, 10, 0], [10.1, 10.05, 1.0], [20, 0, 0], [20.05, 0.02, 0.5],
                              [50, 50, 0]]])
    col, idx = o.collision_multiple(all_vertices)
    assert col.tolist() == [1, 1, 1, 1, 1, 1, 0]
    assert idx.tolist() == [1, 0, 3, 2, 5, 4, -1]


def test_gjk_reference_fixture():
    """collision_models.py:313-324 verbatim geometry: 5 copies of one quad, one shifted, one far away."""
    vertices1 = np.asarray([[4, 11.], [5, 5], [9, 9], [10, 10]])
    all_vertices = np.stack([vertices1] * 5 + [vertices1 + 0.5, vertices1 + 100.0])
    # (the reference perturbs with seeded noise of 1e-2 scale; the boolean outcome is perturbation-independent)
    o = Oracle(1, 1)
    col, idx = o.collision_multiple(all_vertices)
    assert col.tolist() == [1, 1, 1, 1, 1, 1, 0]
    assert idx.tolist() == [5, 5, 5, 5, 5, 4, -1]


@pytest.mark.parametrize("map_name", ["Shanghai_map", "straight_corridor"])
def test_scans_bit_exact(map_name):
    g = H.load('scans')
    o = make_oracle(1, map_name)
    for pose, ref in zip(g[map_name + '__poses'], g[map_name + '__scans']):
        mine, _ = o.scan(pose)
        assert np.array_equal(mine, ref)


def test_scans_rotated_origin():
    """yaml origin with a yaw: the rotated branch of xy_2_rc (laser_models.py:70-77), golden from the reference."""
    from oracle.f110_oracle import Oracle
    g = H.load('scans_rotated')
    dt, res, _ = H.golden_map('Shanghai_map')
    o = Oracle(1, 1)
    o.set_map_arrays(dt, res, [float(v) for v in g['origin']])
    s, c, _, _, _ = H.tables()
    o.set_tables(s, c)
    d = np.abs(np.stack([o.scan(p)[0] for p in g['poses']]) - g['scans'])
    # the oracle takes cos/sin(origin yaw) from libm, the reference from numpy: equal here, else allow the 1e-6 bar
    print('rotated origin: max', d.max(), 'exact fraction', float((d == 0).mean()))
    assert (d <= 1e-6).mean() >= 0.999
    assert d.max() == 0.0 or not (np.cos(g['origin'][2]) == g['orig_c'] and np.sin(g['origin'][2]) == g['orig_s'])


def test_dt_probe():
    dt, res, _ = H.golden_map('Shanghai_map')
    p = H.load('scans')['Shanghai_map__dt_probe']
    assert dt[-1, -1] == p[0] and dt[0, 0] == p[1] and dt.max() == p[2] and dt.sum() == p[3]


@pytest.mark.parametrize("name", sorted(H.ROLLOUT_MAP))
def test_env_rollouts(name):
    """Flags bit-exact; fp64 state bit-exact except where BLAS-evaluated vertices enter (never the state);
    scans within 1e-9 everywhere (opponent ray-cast goes through BLAS dots in the reference)."""
    r = H.compare_rollout(name, make_oracle, state_tol=0.0, scan_tol=1e-9, scan_frac=1.0, obs_tol=0.0)
    assert r['outliers'] == 0


def test_single_agent_sim_rollout():
    """Config C1 at Simulator level (the env cannot pack a 1-agent observation, f110_env.py:554)."""
    g = H.load('rollout_c1_single')
    o = make_oracle(1, 'Shanghai_map')
    T = g['state'].shape[0]
    rng = np.random.default_rng(int(g['seed']))
    for t in range(T):
        if g['resets'][t] or t == 0:
            # Simulator.reset only: re-seed the noise stream, no zero-action step
            rng = np.random.default_rng(int(g['seed']))
            o.sim_reset(g['pose'][None, None])
        out = o.step(g['action'][None], noise=rng.normal(0., 0.01, size=1080)[None, None])
        assert np.array_equal(out['state'][0, 0], g['state'][t]), t
        assert out['collisions'][0, 0] == g['collisions'][t], t
        if t % int(g['every']) == 0:
            assert np.array_equal(out['scans'][0, 0], g['scans'][t // int(g['every'])])


def test_map_not_set_and_bad_index():
    o = Oracle(1, 2)
    with pytest.raises(ValueError):
        o.step()
    with pytest.raises(IndexError):
        o.update_params(DEFAULT_PARAMS, 5)


def test_gap_follow_oracle_matches_reference():
    """rl_training/utils/gap_follow.py:43-58 on 214 recorded / synthetic float32 scans: actions bit-exact."""
    from oracle.f110_oracle import gap_follow_action
    g = H.load('gap_follow')
    for s, a in zip(g['scans'], g['actions']):
        assert np.array_equal(gap_follow_action(s), a)
    for k in range(len(g['proc'])):
        _, p = gap_follow_action(g['scans'][k], want_proc=True)
        assert np.array_equal(p, g['proc'][k])


REWARD_KW = dict(w_prog=5.0, alive_bonus=0.5, grace_steps_wall=25, grace_steps_opp=175, w_lat=0.25, lat_cap=3.0,
                 near_wall_dist=0.30 / 30, w_wall=0.30, wall_quantile=0.10, opp_safe_dist=0.60, w_opp=0.30,
                 w_rel_lead=0.0)       # train_ddpg.py:127-145
REWARD_ALT_KW = dict(w_rel_lead=0.3, grace_steps_wall=5, grace_steps_opp=5, wall_quantile=0.05)


def test_shaped_reward_oracle_matches_reference():
    """rewards.py:185-355 + track_progress.py over 754 recorded steps (4 episodes incl. a crash), two parameter sets:
    within 1e-12 of the reference's float (BLAS dots / libm ulps), and the float32 quantile path bit-exact."""
    from oracle.f110_oracle import RewardOracle
    g = H.reward_recording()
    for kw, key in ((REWARD_KW, 'reward'), (REWARD_ALT_KW, 'reward_alt')):
        o = RewardOracle(1, g['centerline'], **kw)
        got = np.array([o(g['obs'][k], np.array([g['episode_start'][k]], np.uint8))[0] for k in range(len(g[key]))])
        assert np.abs(got - g[key]).max() < 1e-12
        assert (got == -50.0).any() and (np.abs(got) < 5).any()


@pytest.mark.parametrize("name", H.LARGE_MAPS)
def test_large_map_scans_golden(name):
    """BASELINE config C4 'large maps' (levine 2048^2, Shanghai x2 = 4000^2, x4 = 8000^2, x2 under a rotated origin):
    the oracle's noise-free scans against the reference's own (laser_models.py:55-186), poses on the track, at the map
    border and outside it.  Axis-aligned origins are bit-exact; the rotated one within 1e-6 m on >= 99.9 % of beams."""
    dt, res, origin, poses, ref = H.large_map(name)
    o = Oracle(1, 1)
    s, c, _, _, _ = H.tables()
    o.set_tables(s, c)
    o.set_map_arrays(dt, res, origin)
    got = np.stack([o.scan(p)[0] for p in poses])
    d = np.abs(got - ref)
    print(name, dt.shape, 'max', d.max(), 'exact fraction', float((d == 0).mean()))
    assert (d <= 1e-6).mean() >= 0.999
    if not name.endswith('_rot'):
        assert d.max() == 0.0
