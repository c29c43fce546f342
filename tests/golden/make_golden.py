"""Generate the committed golden fixtures from the UNMODIFIED reference.

Needs a checkout of the reference:  F110_REFERENCE_ROOT=<dir> python tests/golden/make_golden.py
Writes tests/golden/*.npz.  The tests read these fixtures; only the optional differential
tests read the reference itself.

What is recorded
  maps.npz         binarised occupancy (bit-packed, after the reference's flip+threshold,
                   laser_models.py:398-404) + yaml metadata for every map the tests/bench use,
                   the Shanghai centerline start poses (SURVEY 8d C3), and the numpy-computed
                   lookup tables (laser_models.py:379-381, base_classes.py:122-158).
  scans.npz        noise-free ScanSimulator2D.scan(pose, None) at fixed poses.
  scans_rotated.npz  the same on a map whose yaml origin has a yaw (the rotated branch of xy_2_rc).
  rollout_*.npz    F110Env / Simulator rollouts: per-step fp64 states, flags, lap bookkeeping,
                   and sub-sampled scans / flat observations.
"""
import hashlib
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
warnings.filterwarnings('ignore')
from ref_loader import REF_MAPS, REF_ROOT, fresh_statics, load_reference  # noqa: E402

ns = load_reference()
TMP = '/tmp/f110_golden_maps/'
os.makedirs(TMP, exist_ok=True)


def write_open_map():
    """20 m x 20 m free square with a 3-pixel wall, used for the lap / GJK scenarios."""
    from PIL import Image
    img = np.full((400, 400), 254, np.uint8)
    img[:3, :] = 0; img[-3:, :] = 0; img[:, :3] = 0; img[:, -3:] = 0
    img[150:160, 300:360] = 0   # an interior block so the scan is not symmetric
    Image.fromarray(img, mode='L').save(TMP + 'open_square.png')
    with open(TMP + 'open_square.yaml', 'w') as f:
        f.write("image: open_square.png\nresolution: 0.05\norigin: [-10.0, -10.0, 0.0]\nnegate: 0\n"
                "occupied_thresh: 0.65\nfree_thresh: 0.196\n")


def pack_map(map_dir, name, ext='.png'):
    import yaml
    from PIL import Image
    img = np.array(Image.open(map_dir + name + ext).transpose(Image.FLIP_TOP_BOTTOM)).astype(np.float64)
    free = img > 128.
    meta = yaml.safe_load(open(map_dir + name + '.yaml'))
    return {name + '__bits': np.packbits(free, axis=None), name + '__shape': np.array(free.shape),
            name + '__resolution': np.float64(meta['resolution']),
            name + '__origin': np.array(meta['origin'], np.float64)}


def make_env(map_dir, name, num_agents=2, **kw):
    fresh_statics(ns)
    return ns.F110Env(map_dir=map_dir, map=name, map_ext='.png', num_agents=num_agents, **kw)


def noise_digest(seed, steps, beams=1080):
    rng = np.random.default_rng(seed)
    h = hashlib.sha256()
    for _ in range(steps):
        h.update(rng.normal(0., 0.01, size=beams).tobytes())
    return h.hexdigest()


def record_env_rollout(env, poses, actions, every=50, seed=42):
    """F110Env rollout; scans are the obs-dict fp64 scans (after noise and opponent ray-cast)."""
    T, A = actions.shape[0], env.num_agents
    rec = dict(poses=np.asarray(poses, np.float64), actions=actions, every=np.int64(every), seed=np.int64(seed))
    st = np.zeros((T + 1, A, 7)); col = np.zeros((T + 1, A), np.uint8); term = np.zeros(T + 1, np.uint8)
    tog = np.zeros((T + 1, A), np.int32); lt = np.zeros((T + 1, A)); lc = np.zeros((T + 1, A)); tm = np.zeros(T + 1)
    ks = list(range(0, T + 1, every))
    scans = np.zeros((len(ks), A, 1080)); obs = np.zeros((len(ks), 1088), np.float32)

    def grab(k, o, done, info):
        st[k] = np.stack([a.state for a in env.sim.agents])
        col[k] = info['collisions']; term[k] = done; tog[k] = env.toggle_list
        lt[k] = env.lap_times; lc[k] = env.lap_counts; tm[k] = info['time']
        if k % every == 0:
            scans[k // every] = np.stack(ns.F110Env.current_obs['scans']); obs[k // every] = o
    o, info = env.reset(options=np.array(poses, np.float64))
    grab(0, o, False, info)   # index 0 = state after reset (which already contains one zero-action step)
    for t in range(T):
        o, r, done, trunc, info = env.step(actions[t])
        assert r == env.timestep and trunc is False
        grab(t + 1, o, done, info)
    rec.update(state=st, collisions=col, terminated=term, toggles=tog, lap_times=lt, lap_counts=lc, time=tm,
               scans=scans, obs=obs, noise_sha256=np.array(noise_digest(seed, T + 1)))
    return rec


def record_sim_rollout(map_dir, name, pose, action, T, every=100, seed=42):
    """C1: Simulator-level single agent (F110Env cannot pack a 1-agent observation, f110_env.py:554)."""
    fresh_statics(ns)
    params = make_env(map_dir, name).params
    fresh_statics(ns)
    sim = ns.Simulator(params, 1, seed, time_step=0.01, integrator=ns.Integrator.RK4)
    sim.set_map(map_dir + name + '.yaml', '.png')
    st = np.zeros((T, 7)); col = np.zeros(T, np.uint8); resets = np.zeros(T, np.uint8)
    ks = list(range(0, T, every)); scans = np.zeros((len(ks), 1080))
    pose = np.asarray(pose, np.float64)
    sim.reset(pose[None])
    act = np.asarray(action, np.float32)[None]
    for t in range(T):
        if t > 0 and col[t - 1]:
            sim.reset(pose[None]); resets[t] = 1
        obs = sim.step(act)
        st[t] = sim.agents[0].state; col[t] = obs['collisions'][0]
        if t % every == 0:
            scans[t // every] = obs['scans'][0]
    return dict(pose=pose, action=act, state=st, collisions=col, resets=resets, scans=scans,
                every=np.int64(every), seed=np.int64(seed))


def main():
    write_open_map()
    out = {}
    out.update(pack_map(REF_MAPS, 'Shanghai_map'))
    out.update(pack_map(REF_MAPS, 'straight_corridor'))
    out.update(pack_map(TMP, 'open_square'))
    cl = np.loadtxt(os.path.join(REF_ROOT, 'rl_training/maps/cenerlines/Shanghai_map.csv'), delimiter=',', comments='#')
    nxt = np.roll(cl[:, :2], -1, axis=0)
    yaw = np.arctan2(nxt[:, 1] - cl[:, 1], nxt[:, 0] - cl[:, 0])
    out['Shanghai_map__centerline_poses'] = np.column_stack([cl[:, 0], cl[:, 1], yaw])
    env = make_env(REF_MAPS, 'Shanghai_map')
    R = ns.RaceCar
    out.update(sines=R.scan_simulator.sines, cosines=R.scan_simulator.cosines, scan_angles=R.scan_angles,
               beam_cosines=R.cosines, side_distances=R.side_distances)
    np.savez_compressed(os.path.join(HERE, 'maps.npz'), **out)

    # ---- noise-free scans
    sc = {}
    rng = np.random.default_rng(7)
    poses = np.array([[0, 0, 0]] + [[rng.uniform(-70, 50), rng.uniform(-30, 60), rng.uniform(-4, 4)] for _ in range(23)])
    poses[1] = [-200.0, 0.0, 1.0]     # outside the map
    cp = out['Shanghai_map__centerline_poses']
    poses[2:12] = cp[np.linspace(0, len(cp) - 1, 10).round().astype(int)]
    sc['Shanghai_map__poses'] = poses
    sc['Shanghai_map__scans'] = np.stack([R.scan_simulator.scan(p, None) for p in poses])
    sc['Shanghai_map__dt_probe'] = np.array([R.scan_simulator.dt[-1, -1], R.scan_simulator.dt[0, 0], R.scan_simulator.dt.max(),
                                             R.scan_simulator.dt.sum()])
    env = make_env(REF_MAPS, 'straight_corridor')
    poses = np.array([[0, 0, 0], [0.2, 5.0, 1.5], [-0.3, 40.0, -1.0], [0.0, 99.0, 1.57], [5.0, 5.0, 0.0], [0.1, -0.5, 3.0]])
    sc['straight_corridor__poses'] = poses
    sc['straight_corridor__scans'] = np.stack([R.scan_simulator.scan(p, None) for p in poses])
    np.savez_compressed(os.path.join(HERE, 'scans.npz'), **sc)

    # ---- S1: config C2, random actions on Shanghai
    env = make_env(REF_MAPS, 'Shanghai_map')
    acts = np.random.default_rng(0).uniform([-0.4189, 0], [0.4189, 20], size=(1000, 2, 2)).astype(np.float32)
    np.savez_compressed(os.path.join(HERE, 'rollout_c2_shanghai.npz'),
                        **record_env_rollout(env, [[0, 0, 0], [3.0, 0.5, 0]], acts))
    # ---- S1b: constant action from the survey (ego TTC-terminates at step 221)
    acts = np.tile(np.array([[0.05, 3.0], [0.0, 2.0]], np.float32), (400, 1, 1))
    np.savez_compressed(os.path.join(HERE, 'rollout_const_shanghai.npz'),
                        **record_env_rollout(env, [[0, 0, 0], [3.0, 0.5, 0]], acts))
    # ---- S2: circles on the open map -> finish-zone toggles, lap counts, done by laps
    env = make_env(TMP, 'open_square')
    acts = np.tile(np.array([[0.4189, 1.5], [-0.4189, 2.0]], np.float32), (900, 1, 1))
    np.savez_compressed(os.path.join(HERE, 'rollout_circles_open.npz'),
                        **record_env_rollout(env, [[0, 0, 0.3], [2.0, -3.0, -1.0]], acts))
    # ---- S3: head-on on the open map -> GJK collision flags + opponent ray-cast in the scans
    acts = np.tile(np.array([[0.0, 3.0], [0.02, 2.5]], np.float32), (300, 1, 1))
    np.savez_compressed(os.path.join(HERE, 'rollout_headon_open.npz'),
                        **record_env_rollout(env, [[-4.0, 0, 0.0], [4.0, 0.15, np.pi - 0.01]], acts, every=10))
    # ---- S3b: three agents, Euler integrator, lidar offset, non-default ego
    env = make_env(TMP, 'open_square', num_agents=3, integrator=ns.Integrator.Euler, lidar_dist=0.275, ego_idx=1)
    acts = np.random.default_rng(3).uniform([-0.4189, 0], [0.4189, 8], size=(300, 3, 2)).astype(np.float32)
    np.savez_compressed(os.path.join(HERE, 'rollout_three_euler_open.npz'),
                        **record_env_rollout(env, [[-2.0, 0, 0.0], [0.0, 0.3, 0.1], [1.2, 0.2, 3.0]], acts, every=25))
    # ---- S4: rotated-origin corridor until the end wall (TTC)
    env = make_env(REF_MAPS, 'straight_corridor')
    acts = np.tile(np.array([[0.0, 8.0], [0.01, 6.0]], np.float32), (600, 1, 1))
    np.savez_compressed(os.path.join(HERE, 'rollout_corridor.npz'),
                        **record_env_rollout(env, [[0.0, 0.5, 1.5708], [0.3, 3.0, 1.5708]], acts))
    # ---- S5: config C1, Simulator-level single agent with resets on collision
    np.savez_compressed(os.path.join(HERE, 'rollout_c1_single.npz'),
                        **record_sim_rollout(REF_MAPS, 'Shanghai_map', [0, 0, 0], [0.0, 2.0], 10000))
    for f in sorted(os.listdir(HERE)):
        if f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, 'KiB')


def make_gap_follow_golden():
    """rl_training/utils/gap_follow.py:43-58 on recorded + synthetic scans -> tests/golden/gap_follow.npz"""
    sys.path.insert(0, os.path.join(REF_ROOT, 'rl_training'))
    from utils.gap_follow import gap_follow_action, preprocess_lidar
    rng = np.random.default_rng(5)
    scans = []
    for f in ('rollout_c2_shanghai', 'rollout_headon_open', 'rollout_corridor', 'rollout_circles_open'):
        g = np.load(os.path.join(HERE, f + '.npz'))
        scans.append(g['scans'].reshape(-1, 1080).astype(np.float32))
    scans = np.concatenate(scans)
    extra = [np.full(1080, 0.2, np.float32), np.full(1080, 5.0, np.float32), np.zeros(1080, np.float32),
             np.linspace(0, 6, 1080).astype(np.float32), np.linspace(6, 0, 1080).astype(np.float32)]
    for _ in range(40):
        s = rng.uniform(0.0, 4.0, 1080).astype(np.float32)
        s[rng.integers(0, 1080, 30)] = rng.uniform(0, 0.4, 30).astype(np.float32)   # narrow obstacles
        k = rng.integers(0, 900); s[k:k + rng.integers(5, 180)] = 0.3                 # a wall segment
        extra.append(s)
    nanscan = rng.uniform(0.6, 3.0, 1080).astype(np.float32); nanscan[100] = 30.0
    extra.append(nanscan)
    scans = np.concatenate([scans, np.stack(extra)])
    acts = np.stack([gap_follow_action(s.copy()) for s in scans])
    proc = np.stack([preprocess_lidar(s) for s in scans[:8]])
    np.savez_compressed(os.path.join(HERE, 'gap_follow.npz'), scans=scans, actions=acts, proc=proc)
    print('gap_follow.npz', scans.shape, acts.dtype, proc.dtype)


REWARD_KW = dict(w_prog=5.0, alive_bonus=0.5, grace_steps_wall=25, grace_steps_opp=175, w_lat=0.25, lat_cap=3.0,
                 near_wall_dist=0.30 / 30, w_wall=0.30, wall_quantile=0.10, opp_safe_dist=0.60, w_opp=0.30,
                 w_rel_lead=0.0)     # train_ddpg.py:127-145


def make_reward_golden():
    """train_ddpg.py:150-202 loop shape with the reference's own env, gap-follow opponent and shaped reward
    (rewards.py:185-355 on CenterlineProgress, track_progress.py) -> tests/golden/reward.npz (obs + rewards)."""
    sys.path.insert(0, os.path.join(REF_ROOT, 'rl_training'))
    from utils.gap_follow import gap_follow_action
    from utils.rewards import CenterlineSafetyProgressReward
    from utils.track_progress import CenterlineProgress
    csv = os.path.join(REF_ROOT, 'rl_training/maps/cenerlines/Shanghai_map.csv')
    P = CenterlineProgress(csv, closed=True)
    env = make_env(REF_MAPS, 'Shanghai_map')
    rfn = CenterlineSafetyProgressReward(dt=env.timestep, progress=P, **REWARD_KW)
    rfn2 = CenterlineSafetyProgressReward(dt=env.timestep, progress=P, w_rel_lead=0.3, grace_steps_wall=5, grace_steps_opp=5,
                                          wall_quantile=0.05)   # defaults otherwise: exercises lead / bubble / flank terms
    cl = np.loadtxt(csv, delimiter=',', comments='#')
    rng = np.random.default_rng(21)
    obs_all, rew_all, rew2_all, first, acts_all, poses_all = [], [], [], [], [], []
    for ep, (i0, gap, kspeed) in enumerate([(0, 30, 1.6), (2500, 14, 1.2), (5200, 9, 2.2), (900, 12, 0.8)]):
        def pose(i):
            j = (i + 1) % len(cl)
            return [cl[i, 0], cl[i, 1], np.arctan2(cl[j, 1] - cl[i, 1], cl[j, 0] - cl[i, 0])]
        rfn.reset(); rfn2.reset()
        poses_all.append(np.array([pose(i0), pose((i0 + gap) % len(cl))], np.float32).astype(np.float64))
        obs, info = env.reset(options=poses_all[-1])
        for t in range(260):
            ego = gap_follow_action(info['scans'][0]).astype(np.float32)
            ego[1] *= kspeed
            ego[0] += np.float32(rng.normal(0, 0.03))
            if ep == 3 and t > 120:
                ego[0] = np.float32(0.35)        # drive it into the wall: crash penalty path
            opp = gap_follow_action(info['scans'][1]).astype(np.float32)
            acts_all.append(np.stack([ego, opp]).astype(np.float32))
            obs, _, term, trunc, info = env.step(acts_all[-1])
            obs_all.append(obs.copy()); rew_all.append(float(rfn(obs))); rew2_all.append(float(rfn2(obs)))
            first.append(1 if t == 0 else 0)
            if term and t > 150:
                break
    # the observations themselves (3 MB of noisy scans) are not stored: tests/helpers.py:reward_recording replays the
    # rollout from its poses, actions and noise seed (F110Env's default, 42) and checks each against its SHA-256
    sha = np.stack([np.frombuffer(hashlib.sha256(np.ascontiguousarray(o, np.float32).tobytes()).digest(), np.uint8)
                    for o in obs_all])
    np.savez_compressed(os.path.join(HERE, 'reward.npz'), actions=np.stack(acts_all), poses=np.stack(poses_all),
                        seed=np.int64(42), obs_sha256=sha, reward=np.array(rew_all), reward_alt=np.array(rew2_all),
                        episode_start=np.array(first, np.uint8), centerline=cl)
    print('reward.npz', len(rew_all), 'steps; reward range', min(rew_all), max(rew_all), 'alt', min(rew2_all), max(rew2_all))


def make_rotated_scan_golden(theta=0.3):
    """ScanSimulator2D on the Shanghai image under a yaml whose origin has a yaw (laser_models.py:410-422 keeps
    orig_c / orig_s; xy_2_rc rotates every lookup, :70-77) -> tests/golden/scans_rotated.npz"""
    import shutil
    from f110_gym.envs.laser_models import ScanSimulator2D
    shutil.copy(os.path.join(REF_MAPS, 'Shanghai_map.png'), os.path.join(TMP, 'Shanghai_rot.png'))
    origin = [3.5, -7.25, theta]
    with open(os.path.join(TMP, 'Shanghai_rot.yaml'), 'w') as f:
        f.write("image: Shanghai_rot.png\nresolution: 0.06505\norigin: [%r, %r, %r]\nnegate: 0\noccupied_thresh: 0.45\n"
                "free_thresh: 0.196\n" % tuple(origin))
    sim = ScanSimulator2D(1080, 4.7)
    sim.set_map(os.path.join(TMP, 'Shanghai_rot.yaml'), '.png')
    m = dict(np.load(os.path.join(HERE, 'maps.npz')))
    cl, o = m['Shanghai_map__centerline_poses'], m['Shanghai_map__origin']
    cl = cl[np.linspace(0, len(cl) - 1, 48).round().astype(int)]
    mx, my = cl[:, 0] - o[0], cl[:, 1] - o[1]                      # map-frame coordinates of the centerline
    c, s_ = np.cos(theta), np.sin(theta)
    poses = np.stack([origin[0] + c * mx - s_ * my, origin[1] + s_ * mx + c * my, cl[:, 2] + theta], axis=1)
    poses = np.concatenate([poses, [[0., 0., 0.], [500., 0., 1.]]])     # in free space or not, and outside the map
    scans = np.stack([sim.scan(p, None) for p in poses])
    np.savez_compressed(os.path.join(HERE, 'scans_rotated.npz'), origin=np.array(origin), poses=poses, scans=scans,
                        orig_c=np.float64(sim.orig_c), orig_s=np.float64(sim.orig_s))
    print('scans_rotated.npz', scans.shape, 'range', scans.min(), scans.max())


def make_c1_golden():
    """BASELINE config C1 at its full length: 10 000 Simulator.step calls, single agent, constant action, reset on
    every collision -> tests/golden/rollout_c1_single.npz"""
    np.savez_compressed(os.path.join(HERE, 'rollout_c1_single.npz'),
                        **record_sim_rollout(REF_MAPS, 'Shanghai_map', [0, 0, 0], [0.0, 2.0], 10000))
    print('rollout_c1_single.npz', os.path.getsize(os.path.join(HERE, 'rollout_c1_single.npz')) // 1024, 'KiB')


def large_map_poses(name, k=1, n=64):
    """Poses for the C4 large-map scans: n centerline poses of the Shanghai track (levine: free cells picked by a
    seeded generator), plus poses next to and beyond the map border and one far outside."""
    m = dict(np.load(os.path.join(HERE, 'maps.npz')))
    if name == 'levine':
        return None
    cl = m['Shanghai_map__centerline_poses']
    poses = cl[np.linspace(0, len(cl) - 1, n).round().astype(int)].copy()
    o, res, (h, w) = m['Shanghai_map__origin'], float(m['Shanghai_map__resolution']), m['Shanghai_map__shape']
    x1, y1 = o[0] + w * res, o[1] + h * res
    extra = [[o[0] + 0.013, o[1] + 0.021, 0.7], [x1 - 0.011, y1 - 0.017, -2.4], [o[0] + 0.5 * w * res, y1 - 1e-3, 1.6],
             [x1 + 3.0, o[1] + 0.5 * h * res, 3.0], [o[0] - 1e-9, o[1] + 10.0, 0.0], [-500.0, 0.0, 1.0]]
    return np.concatenate([poses, np.array(extra)])


def make_large_map_golden():
    """BASELINE config C4 'large maps': the reference's own ScanSimulator2D on (a) assets/maps/levine (2048 x 2048),
    (b) the Shanghai image upsampled x2 (4000 x 4000) and x4 (8000 x 8000) by pixel replication with the resolution
    divided accordingly, (c) the x2 map under an origin with a yaw.  Noise-free scans (laser_models.py:429-454 with
    rng None) -> tests/golden/scans_large.npz; the levine occupancy -> tests/golden/maps_large.npz.  The upsampled
    occupancies are rebuilt by the tests from the Shanghai bits (np.kron), exactly as written to disk here."""
    from PIL import Image
    from f110_gym.envs.laser_models import ScanSimulator2D
    out = {}
    # ---- (a) levine, as it lies in the reference tree
    lev_dir = os.path.join(REF_ROOT, 'assets', 'maps') + '/'
    packed = pack_map(lev_dir, 'levine')
    np.savez_compressed(os.path.join(HERE, 'maps_large.npz'), **packed)
    sim = ScanSimulator2D(1080, 4.7)
    sim.set_map(lev_dir + 'levine.yaml', '.png')
    free = np.argwhere(sim.dt > 0.3)
    rng = np.random.default_rng(11)
    pick = free[rng.choice(len(free), 72, replace=False)]
    o = packed['levine__origin']; res = float(packed['levine__resolution'])
    poses = np.column_stack([o[0] + (pick[:, 1] + rng.uniform(0, 1, 72)) * res, o[1] + (pick[:, 0] + rng.uniform(0, 1, 72)) * res,
                             rng.uniform(-np.pi, np.pi, 72)])
    poses = np.concatenate([poses, [[o[0] + 1e-3, o[1] + 1e-3, 0.8], [o[0] + 2048 * res - 1e-3, o[1] + 2048 * res - 1e-3, -2.3],
                                    [o[0] - 5.0, o[1] + 20.0, 0.0], [300.0, 300.0, 1.0]]])
    out['levine__poses'] = poses
    out['levine__scans'] = np.stack([sim.scan(p, None) for p in poses])
    out['levine__dt_probe'] = np.array([sim.dt[-1, -1], sim.dt[0, 0], sim.dt.max(), sim.dt.sum()])
    print('levine', out['levine__scans'].shape, 'range', out['levine__scans'].min(), out['levine__scans'].max())
    # ---- (b), (c) upsampled Shanghai
    m = dict(np.load(os.path.join(HERE, 'maps.npz')))
    shape = tuple(int(v) for v in m['Shanghai_map__shape'])
    free = np.unpackbits(m['Shanghai_map__bits'])[:shape[0] * shape[1]].reshape(shape).astype(bool)
    o, res = m['Shanghai_map__origin'], float(m['Shanghai_map__resolution'])
    for k, theta in ((2, 0.0), (4, 0.0), (2, 0.3)):
        big = np.kron(free, np.ones((k, k), bool))
        name = 'Shanghai_x%d%s' % (k, '_rot' if theta else '')
        Image.fromarray(np.where(big, 254, 0).astype(np.uint8)[::-1], mode='L').save(TMP + name + '.png')
        origin = [float(o[0]), float(o[1]), 0.0] if not theta else [3.5, -7.25, theta]
        with open(TMP + name + '.yaml', 'w') as f:
            f.write("image: %s.png\nresolution: %r\norigin: [%r, %r, %r]\nnegate: 0\noccupied_thresh: 0.45\nfree_thresh: 0.196\n"
                    % (name, res / k, origin[0], origin[1], origin[2]))
        sim = ScanSimulator2D(1080, 4.7)
        sim.set_map(TMP + name + '.yaml', '.png')
        assert sim.dt.shape == (shape[0] * k, shape[1] * k)
        poses = large_map_poses('Shanghai', k)
        if theta:
            mx, my = poses[:, 0] - o[0], poses[:, 1] - o[1]
            c, s_ = np.cos(theta), np.sin(theta)
            poses = np.stack([origin[0] + c * mx - s_ * my, origin[1] + s_ * mx + c * my, poses[:, 2] + theta], axis=1)
        out[name + '__origin'] = np.array(origin)
        out[name + '__resolution'] = np.float64(res / k)
        out[name + '__poses'] = poses
        out[name + '__scans'] = np.stack([sim.scan(p, None) for p in poses])
        out[name + '__dt_probe'] = np.array([sim.dt[-1, -1], sim.dt[0, 0], sim.dt.max(), sim.dt.sum()])
        print(name, sim.dt.shape, out[name + '__scans'].shape, 'range', out[name + '__scans'].min(), out[name + '__scans'].max())
        del sim, big
    np.savez_compressed(os.path.join(HERE, 'scans_large.npz'), **out)
    for f in ('maps_large.npz', 'scans_large.npz'):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, 'KiB')


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == 'large':
        make_large_map_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == 'c1':
        make_c1_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == 'reward':
        make_reward_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == 'gap_follow':
        make_gap_follow_golden()     # only the consumer-side fixture
    elif len(sys.argv) > 1 and sys.argv[1] == 'rotated':
        make_rotated_scan_golden()
    else:
        main()
        make_gap_follow_golden()
        make_reward_golden()
        make_rotated_scan_golden()
        make_large_map_golden()
