"""ctypes binding of the CPU oracle (oracle/f110_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / ``--impl reference`` legs of bench.py.  The product package never imports it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

PARAM_KEYS = ['mu', 'C_Sf', 'C_Sr', 'lf', 'lr', 'h', 'm', 'I', 's_min', 's_max', 'sv_min', 'sv_max',
              'v_switch', 'a_max', 'v_min', 'v_max', 'width', 'length']

# f110_env.py:132-156
DEFAULT_PARAMS = {'mu': 1.0489, 'C_Sf': 4.718, 'C_Sr': 5.4562, 'lf': 0.15875, 'lr': 0.17145, 'h': 0.074,
                  'm': 3.74, 'I': 0.04712, 's_min': -0.4189, 's_max': 0.4189, 'sv_min': -3.2, 'sv_max': 3.2,
                  'v_switch': 7.319, 'a_max': 9.51, 'v_min': 0.00000001, 'v_max': 20.0, 'width': 0.31,
                  'length': 0.58, 'lidar_max': 30.0}


def build(force=False):
    so = os.path.join(_HERE, "libf110_oracle.so")
    src = os.path.join(_HERE, "f110_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libf110_oracle.so"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        dp, vp, u8p, fp, i32p = (C.POINTER(C.c_double), C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_float),
                                 C.POINTER(C.c_int32))
        L.f110o_create.restype = vp
        L.f110o_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double,
                                   C.c_double, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_uint64, vp]
        L.f110o_destroy.argtypes = [vp]
        L.f110o_set_threads.argtypes = [vp, C.c_int]
        L.f110o_set_map.argtypes = [vp, vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double]
        L.f110o_set_tables.argtypes = [vp, vp, vp]
        L.f110o_set_beam_tables.argtypes = [vp, vp, vp, vp]
        L.f110o_get_beam_tables.argtypes = [vp, vp, vp, vp]
        L.f110o_update_params.argtypes = [vp, vp, C.c_int]
        L.f110o_update_params.restype = C.c_int
        L.f110o_scan.argtypes = [vp, vp, vp, C.POINTER(C.c_long)]
        L.f110o_check_ttc.argtypes = [vp, vp, C.c_double]
        L.f110o_check_ttc.restype = C.c_int
        L.f110o_ray_cast.argtypes = [vp, vp, vp, vp]
        L.f110o_step.argtypes = [vp, vp, C.c_int] + [vp] * 14
        L.f110o_step.restype = C.c_int
        L.f110o_sim_reset.argtypes = [vp, vp, C.c_int]
        L.f110o_sim_reset.restype = C.c_int
        L.f110o_last_lookups.argtypes = [vp]
        L.f110o_last_lookups.restype = C.c_long
        L.f110o_vehicle_dynamics_st.argtypes = [vp] * 4
        L.f110o_vehicle_dynamics_ks.argtypes = [vp] * 4
        L.f110o_pid.argtypes = [C.c_double] * 8 + [dp, dp]
        L.f110o_update_pose.argtypes = [vp, C.c_double, C.c_int, C.c_int, vp, vp, vp, vp, vp]
        L.f110o_update_pose.restype = None
        L.f110o_get_vertices.argtypes = [vp, C.c_double, C.c_double, vp]
        L.f110o_collision.argtypes = [vp, vp]
        L.f110o_collision.restype = C.c_int
        L.f110o_collision_multiple.argtypes = [vp, C.c_int, vp, vp]
        L.f110o_reward_create.restype = vp
        L.f110o_reward_create.argtypes = [C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int]
        L.f110o_reward_destroy.argtypes = [vp]
        L.f110o_reward_compute.argtypes = [vp, vp, vp, vp]
        L.f110o_reward_compute_terms.argtypes = [vp, vp, vp, vp, vp]
        L.f110o_quantile_f32.argtypes = [vp, C.c_int, C.c_double]
        L.f110o_quantile_f32.restype = C.c_float
        L.f110o_reward_seg_index.argtypes = [vp, C.c_double]
        L.f110o_reward_seg_index.restype = C.c_int
        L.f110o_reward_knn.argtypes = [vp, C.c_double, C.c_double, vp, vp]
        L.f110o_gap_follow.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_float, C.c_int, C.c_int, C.c_float,
                                       dp, dp, C.POINTER(C.c_int), vp]
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def params_vector(params):
    return np.array([float(params[k]) for k in PARAM_KEYS], dtype=np.float64)


def load_map_dt(map_path, map_ext):
    """laser_models.py:383-427 restated: flip, threshold at 128, dt = resolution * EDT."""
    import yaml
    from PIL import Image
    from scipy.ndimage import distance_transform_edt
    img = np.array(Image.open(os.path.splitext(map_path)[0] + map_ext).transpose(Image.FLIP_TOP_BOTTOM))
    img = img.astype(np.float64)
    img[img <= 128.] = 0.
    img[img > 128.] = 255.
    with open(map_path, 'r') as f:
        meta = yaml.safe_load(f)
    res, origin = meta['resolution'], meta['origin']
    return res * distance_transform_edt(img), float(res), [float(v) for v in origin]


def numpy_tables(theta_dis=2000):
    """laser_models.py:379-381 (numpy's own sin/cos, which need not equal libm's bit for bit)."""
    th = np.linspace(0.0, 2 * np.pi, num=theta_dis)
    return np.sin(th), np.cos(th)


def numpy_beam_tables(params, num_beams=1080, fov=4.7):
    """base_classes.py:122-158, evaluated with numpy scalars exactly as the reference does."""
    incr = fov / (num_beams - 1)
    cosines = np.zeros((num_beams,)); angles = np.zeros((num_beams,)); side = np.zeros((num_beams,))
    dist_sides = params['width'] / 2.
    dist_fr = (params['lf'] + params['lr']) / 2.
    for i in range(num_beams):
        angle = -fov / 2. + i * incr
        angles[i] = angle
        cosines[i] = np.cos(angle)
        if angle > 0:
            if angle < np.pi / 2:
                to_side = dist_sides / np.sin(angle); to_fr = dist_fr / np.cos(angle)
            else:
                to_side = dist_sides / np.cos(angle - np.pi / 2.); to_fr = dist_fr / np.sin(angle - np.pi / 2.)
        else:
            if angle > -np.pi / 2:
                to_side = dist_sides / np.sin(-angle); to_fr = dist_fr / np.cos(-angle)
            else:
                to_side = dist_sides / np.cos(-angle - np.pi / 2); to_fr = dist_fr / np.sin(-angle - np.pi / 2)
        side[i] = min(to_side, to_fr)
    return angles, cosines, side


class Oracle(object):
    """N independent envs x A agents, stepped on the CPU exactly as F110Env.step does."""

    def __init__(self, num_envs=1, num_agents=2, num_beams=1080, fov=4.7, theta_dis=2000, eps=1e-4,
                 max_range=30.0, timestep=0.01, integrator=1, ego_idx=0, lidar_dist=0.0, ttc_thresh=0.005,
                 params=None, noise_std=0.0, seed=42, threads=1, numpy_trig=True):
        self.L = lib()
        self.params = dict(DEFAULT_PARAMS if params is None else params)
        self.N, self.A, self.B = num_envs, num_agents, num_beams
        pv = params_vector(self.params)
        self.h = self.L.f110o_create(num_envs, num_agents, num_beams, fov, theta_dis, eps, max_range, timestep,
                                     integrator, ego_idx, lidar_dist, ttc_thresh,
                                     float(self.params.get('lidar_max', 30.0)), noise_std, seed, _p(pv))
        self.L.f110o_set_threads(self.h, threads)
        if numpy_trig:
            s, c = numpy_tables(theta_dis)
            self.set_tables(s, c)
            self.set_beam_tables(*numpy_beam_tables(self.params, num_beams, fov))

    def __del__(self):
        if getattr(self, 'h', None):
            self.L.f110o_destroy(self.h)
            self.h = None

    def set_threads(self, n):
        self.L.f110o_set_threads(self.h, n)

    def set_tables(self, sines, cosines):
        s = np.ascontiguousarray(sines, np.float64); c = np.ascontiguousarray(cosines, np.float64)
        self.L.f110o_set_tables(self.h, _p(s), _p(c))

    def set_beam_tables(self, scan_angles, cosines, side_distances):
        a, c, s = (np.ascontiguousarray(v, np.float64) for v in (scan_angles, cosines, side_distances))
        self.L.f110o_set_beam_tables(self.h, _p(a), _p(c), _p(s))

    def get_beam_tables(self):
        a, c, s = (np.empty(self.B) for _ in range(3))
        self.L.f110o_get_beam_tables(self.h, _p(a), _p(c), _p(s))
        return a, c, s

    def set_map_arrays(self, dt, resolution, origin):
        dt = np.ascontiguousarray(dt, np.float64)
        self.L.f110o_set_map(self.h, _p(dt), dt.shape[0], dt.shape[1], resolution, origin[0], origin[1], origin[2])

    def set_map(self, map_path, map_ext):
        self.set_map_arrays(*load_map_dt(map_path, map_ext))

    def update_params(self, params, agent_idx=-1):
        if self.L.f110o_update_params(self.h, _p(params_vector(params)), agent_idx) != 0:
            raise IndexError('Index given is out of bounds for list of agents.')

    def scan(self, pose):
        out = np.empty(self.B)
        n = C.c_long(0)
        pose = np.ascontiguousarray(pose, np.float64)
        self.L.f110o_scan(self.h, _p(pose), _p(out), C.byref(n))
        return out, n.value

    def check_ttc(self, scan, vel):
        scan = np.ascontiguousarray(scan, np.float64)
        return bool(self.L.f110o_check_ttc(self.h, _p(scan), float(vel)))

    def ray_cast(self, pose, scan, vertices):
        scan = np.array(scan, np.float64)
        pose = np.ascontiguousarray(pose, np.float64); vertices = np.ascontiguousarray(vertices, np.float64)
        self.L.f110o_ray_cast(self.h, _p(pose), _p(scan), _p(vertices))
        return scan

    def step(self, actions=None, noise=None, reset_mask=None, reset_poses=None, active_mask=None, want_scans=True):
        N, A, B = self.N, self.A, self.B
        if actions is None:
            actions = np.zeros((N, A, 2), np.float32)
        actions = np.ascontiguousarray(actions)
        if actions.dtype not in (np.float32, np.float64):
            actions = actions.astype(np.float64)
        assert actions.size == N * A * 2
        if noise is not None:
            noise = np.ascontiguousarray(noise, np.float64); assert noise.size == N * A * B
        if reset_mask is not None:
            reset_mask = np.ascontiguousarray(reset_mask, np.uint8)
            reset_poses = np.ascontiguousarray(reset_poses, np.float64); assert reset_poses.size == N * A * 3
        if active_mask is not None:
            active_mask = np.ascontiguousarray(active_mask, np.uint8)
        o = getattr(self, '_out', None)
        if o is None:
            o = dict(obs=np.zeros((N, B + 8), np.float32), reward=np.zeros(N, np.float32),
                     terminated=np.zeros(N, np.uint8), scans=np.zeros((N, A, B)), state=np.zeros((N, A, 7)),
                     collisions=np.zeros((N, A), np.uint8), toggles=np.zeros((N, A), np.int32),
                     lap_times=np.zeros((N, A)), lap_counts=np.zeros((N, A)), time=np.zeros(N))
            self._out = o
        rc = self.L.f110o_step(self.h, _p(actions), int(actions.dtype == np.float64), _p(noise), _p(reset_mask),
                               _p(reset_poses), _p(active_mask), _p(o['obs']), _p(o['reward']), _p(o['terminated']),
                               _p(o['scans']) if want_scans else None, _p(o['state']), _p(o['collisions']),
                               _p(o['toggles']), _p(o['lap_times']), _p(o['lap_counts']), _p(o['time']))
        if rc == -2:
            raise ValueError('Map is not set for scan simulator.')
        if rc != 0:
            raise RuntimeError('oracle step failed: %d' % rc)
        return o

    def reset(self, poses, noise=None):
        """F110Env.reset for every env: poses [N,A,3]; performs the zero-action step (f110_env.py:457-458)."""
        poses = np.ascontiguousarray(poses, np.float64).reshape(self.N, self.A, 3)
        return self.step(None, noise, np.ones(self.N, np.uint8), poses)

    def sim_reset(self, poses):
        """Simulator.reset (base_classes.py:627-643): set poses only, no step."""
        poses = np.ascontiguousarray(poses, np.float64)
        if poses.ndim == 2:
            poses = poses[None]
        if self.L.f110o_sim_reset(self.h, _p(poses), poses.shape[1]) != 0:
            raise ValueError('Number of poses for reset does not match number of agents.')

    @property
    def last_lookups(self):
        return self.L.f110o_last_lookups(self.h)

    # thin scalar entry points for the known-answer tests
    def vehicle_dynamics_st(self, x, u, params):
        f = np.empty(7); x = np.ascontiguousarray(x, np.float64); u = np.ascontiguousarray(u, np.float64)
        self.L.f110o_vehicle_dynamics_st(_p(x), _p(u), _p(params_vector(params)), _p(f))
        return f

    def vehicle_dynamics_ks(self, x, u, params):
        f = np.empty(5); x = np.ascontiguousarray(x, np.float64); u = np.ascontiguousarray(u, np.float64)
        self.L.f110o_vehicle_dynamics_ks(_p(x), _p(u), _p(params_vector(params)), _p(f))
        return f

    def pid(self, speed, steer, current_speed, current_steer, max_sv, max_a, max_v, min_v):
        a, s = C.c_double(), C.c_double()
        self.L.f110o_pid(speed, steer, current_speed, current_steer, max_sv, max_a, max_v, min_v, C.byref(a), C.byref(s))
        return a.value, s.value

    @staticmethod
    def update_pose(state, steer_buf, steer_cnt, raw_steer, speed, params, timestep=0.01, integrator=1):
        """RaceCar.update_pose (base_classes.py:256-417) of n cars with one parameter set, one step each: state [n, 7],
        steer_buf [n, 2] (newest first), steer_cnt [n], raw_steer / speed [n] (float32 actions are widened as the env
        does) -> new (state, steer_buf, steer_cnt)."""
        x = np.array(state, np.float64).reshape(-1, 7)
        n = x.shape[0]
        b = np.array(steer_buf, np.float64).reshape(n, 2)
        c = np.array(steer_cnt, np.int32).reshape(n)
        rs = np.ascontiguousarray(np.asarray(raw_steer).astype(np.float64).reshape(n))
        sp = np.ascontiguousarray(np.asarray(speed).astype(np.float64).reshape(n))
        lib().f110o_update_pose(_p(params_vector(params)), float(timestep), int(integrator), n, _p(x), _p(b), _p(c),
                                _p(rs), _p(sp))
        return x, b, c

    def get_vertices(self, pose, length, width):
        v = np.empty((4, 2)); pose = np.ascontiguousarray(pose, np.float64)
        self.L.f110o_get_vertices(_p(pose), length, width, _p(v))
        return v

    def collision(self, v1, v2):
        v1 = np.ascontiguousarray(v1, np.float64); v2 = np.ascontiguousarray(v2, np.float64)
        return bool(self.L.f110o_collision(_p(v1), _p(v2)))

    def collision_multiple(self, vertices):
        vertices = np.ascontiguousarray(vertices, np.float64)
        n = vertices.shape[0]
        c, i = np.empty(n), np.empty(n)
        self.L.f110o_collision_multiple(_p(vertices), n, _p(c), _p(i))
        return c, i


def gap_follow_action(scan, angle_min=-np.pi / 2, angle_increment=np.pi / 1080, max_distance=3.0, window_size=5,
                      bubble_radius=30, threshold=0.5, want_proc=False):
    """rl_training/utils/gap_follow.py:43-58 restated (oracle): float32 scan -> (steer, speed) as float64.  The keyword
    arguments are the reference's parameters with its defaults; want_proc also returns the window means."""
    L = lib()
    scan = np.ascontiguousarray(scan, np.float32)
    st, sp, best = C.c_double(), C.c_double(), C.c_int()
    proc = np.empty(scan.shape[0], np.float32) if want_proc else None
    L.f110o_gap_follow(_p(scan), scan.shape[0], float(angle_min), float(angle_increment), float(max_distance), int(window_size),
                       int(bubble_radius), float(threshold), C.byref(st), C.byref(sp), C.byref(best), _p(proc))
    out = np.array([st.value, sp.value])
    return (out, proc) if want_proc else out


REWARD_PARAM_KEYS = ['dt', 'w_prog', 'forward_sign', 'alive_bonus', 'w_rel_lead', 'lead_clip', 'w_lat', 'lat_cap',
                     'default_half_width', 'lidar_max', 'near_wall_dist', 'w_wall', 'wall_quantile', 'opp_safe_dist', 'w_opp',
                     'ego_crash_penalty', 'opp_crash_bonus']
# CenterlineSafetyProgressReward.__init__ defaults (rewards.py:196-222)
REWARD_DEFAULTS = dict(dt=0.01, w_prog=1.2, forward_sign=+1.0, alive_bonus=0.02, w_rel_lead=0.0, lead_clip=5.0, w_lat=0.35,
                       lat_cap=4.0, default_half_width=1.5, lidar_max=1.0, near_wall_dist=0.35 / 30.0, w_wall=1.0,
                       wall_quantile=0.05, opp_safe_dist=0.7, w_opp=0.8, ego_crash_penalty=50.0, opp_crash_bonus=50.0,
                       grace_steps_wall=25, grace_steps_opp=25)


# the columns of RewardOracle.terms (f110o_reward_compute_terms in f110_oracle.c)
REWARD_TERM_NAMES = (['knn_ego%d' % k for k in range(5)] + ['knn_opp%d' % k for k in range(5)] +
                     ['fallback_ego', 'fallback_opp', 'e_s', 'e_t', 'o_s', 'o_t', 'seg', 'de', 'dop', 'flip', 'dmin',
                      'r_prog', 'r_alive', 'r_lead', 'r_lat', 'r_wall', 'r_opp', 'r_flank', 'early', 'steps', 'oth', 'w_eff'])
REWARD_TERM = {k: i for i, k in enumerate(REWARD_TERM_NAMES)}


def quantile_f32(values, q):
    """The oracle's np.quantile(float32 array, q) (method 'linear')."""
    v = np.ascontiguousarray(values, np.float32)
    return np.float32(lib().f110o_quantile_f32(_p(v), len(v), float(q)))


class RewardOracle(object):
    """CenterlineSafetyProgressReward (rewards.py:185-355) over a CenterlineProgress (track_progress.py), one
    independent instance per env.  centerline: [n, 4] rows x_m, y_m, w_tr_right_m, w_tr_left_m, or [n, 2] without the
    widths (the reward then uses default_half_width on both sides)."""

    def __init__(self, num_envs, centerline, num_beams=1080, closed=True, **kw):
        self.L = lib()
        p = dict(REWARD_DEFAULTS); p.update(kw)
        cl = np.ascontiguousarray(centerline, np.float64)
        xy = np.ascontiguousarray(cl[:, :2])
        wR = np.ascontiguousarray(cl[:, 2]) if cl.shape[1] >= 4 else None
        wL = np.ascontiguousarray(cl[:, 3]) if cl.shape[1] >= 4 else None
        pv = np.array([float(p[k]) for k in REWARD_PARAM_KEYS])
        self.N, self.B = num_envs, num_beams
        self.h = self.L.f110o_reward_create(num_envs, num_beams, _p(xy), _p(wR), _p(wL), len(xy), int(closed), _p(pv),
                                            int(p['grace_steps_wall']), int(p['grace_steps_opp']))

    def __del__(self):
        if getattr(self, 'h', None):
            self.L.f110o_reward_destroy(self.h); self.h = None

    def __call__(self, obs, reset_mask=None):
        return self.compute_terms(obs, reset_mask)[0]

    def compute_terms(self, obs, reset_mask=None):
        """One reward call -> (total [N], terms [N, len(REWARD_TERM_NAMES)]): the per-env breakdown of what the call
        did (neighbours, projections, branch taken, each summand); NaN where the call did not get that far."""
        obs = np.ascontiguousarray(obs, np.float32).reshape(self.N, self.B + 8)
        out = np.empty(self.N)
        terms = np.empty((self.N, len(REWARD_TERM_NAMES)))
        rm = None if reset_mask is None else np.ascontiguousarray(reset_mask, np.uint8)
        self.L.f110o_reward_compute_terms(self.h, _p(obs), _p(rm), _p(out), _p(terms))
        return out, terms

    def seg_index(self, s):
        """The lateral term's segment lookup: np.searchsorted(s_knots, s, 'right') - 1 clamped to [0, n - 2]."""
        return self.L.f110o_reward_seg_index(self.h, float(s))

    def knn(self, x, y):
        """The 5 nearest segment midpoints of (x, y) in the oracle's order (distance, then index), and (s, t)."""
        k, st = np.empty(5), np.empty(2)
        self.L.f110o_reward_knn(self.h, float(x), float(y), _p(k), _p(st))
        return k.astype(np.int64), st
