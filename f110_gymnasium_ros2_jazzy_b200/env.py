"""F110Env ('f110-v0') and its batched form F110VecEnv on the B200 backend.

F110Env keeps the reference's Gymnasium surface (f110_env.py:55-602): the same kwargs with the same
defaults, ``reset(seed=None, options=poses) -> (obs f32[1088], info)``, ``step(action (A, 2)) -> (obs,
reward, terminated, truncated, info)``, the same ``info`` keys and dtypes, ``update_map``,
``update_params``, ``add_render_callback``, ``render``, and the attributes consumers touch (``timestep``,
``sim``, ``lap_times``, ``lap_counts``, ``action_space``, ``observation_space``, ``unwrapped``).

Documented extensions (SURVEY 7.7, 7.8):
  * ``num_agents=1`` works: the flat observation keeps its 1088 layout with the opponent slots = 0
    (the reference raises IndexError in _pack_flat_obs, f110_env.py:554,566).
  * ``obs_mode='scans'`` returns the (A, B) f32 scans instead of the flat vector, the shape
    jazzy_bridge/gym_bridge.py:113-114,265-267 indexes.
  * ``map`` may be given without ``map_dir`` as a path without extension (gym_bridge.py:77-80); that call selects
    ``obs_mode='scans'`` by default, which is what the bridge's ``list(obs[0])`` / ``list(obs[1])`` need.
  * ``noise`` selects the lidar-noise source, see simulator.Simulator.
  * ``edt='device'`` builds the distance transform with the exact EDT kernel instead of scipy (same bits; update_map
    in milliseconds).
"""
import os

import numpy as np
import torch

from .backend import BatchSim, FAST_OUTPUTS
from .gym_compat import gym, spaces
from .maps import map_bounds
from .params import default_params
from .simulator import Integrator, Simulator

# rendering constants kept for API parity (f110_env.py:48-52)
VIDEO_W, VIDEO_H, WINDOW_W, WINDOW_H = 600, 400, 1000, 800


class F110Env(gym.Env):
    metadata = {'render_modes': ['human', 'human_fast'], 'render_fps': 30}

    renderer = None
    current_obs = None
    render_callbacks = []

    def __init__(self, **kwargs):
        # kwargs extraction, defaults as f110_env.py:104-185
        self.conf = kwargs.get('conf', None)
        self.seed = kwargs.get('seed', 42)
        if 'map_dir' in kwargs and 'map' in kwargs:
            self.map_dir = kwargs['map_dir']
            self.map_name = kwargs['map']
            self.map_path = self.map_dir + self.map_name + '.yaml'
        elif 'map' in kwargs:
            # The ROS bridge's calling convention (gym_bridge.py:77-80): `map` alone, a path without extension.  The bridge
            # then indexes the observation per agent -- list(obs[0]), list(obs[1]) are the scans it publishes
            # (:112-114, :264-267) -- so in this mode the observation is the (A, B) f32 scan array unless obs_mode says
            # otherwise.  (With the reference's flat observation obs[0] is a scalar and the bridge cannot run.)
            kwargs.setdefault('obs_mode', 'scans')
            base = os.path.splitext(kwargs['map'])[0]
            self.map_dir = os.path.dirname(base) + '/'
            self.map_name = os.path.basename(base)
            self.map_path = base + '.yaml'
        else:
            # the reference falls back to envs/maps/vegas.yaml, a file that does not exist in its tree
            raise FileNotFoundError("F110Env needs map_dir= and map= (the reference's default maps/vegas.yaml is absent)")
        self.map_ext = kwargs.get('map_ext', '.png')
        self.params = kwargs.get('params', None) or default_params()
        self.num_agents = kwargs.get('num_agents', 2)
        self.timestep = kwargs.get('timestep', 0.01)
        self.ego_idx = kwargs.get('ego_idx', 0)
        self.integrator = kwargs.get('integrator', Integrator.RK4)
        self.lidar_dist = kwargs.get('lidar_dist', 0.0)
        self.obs_mode = kwargs.get('obs_mode', 'flat')
        self.render_mode = kwargs.get('render_mode', None)
        noise = kwargs.get('noise', 'numpy')

        self.start_thresh = 0.1
        self.poses_x, self.poses_y, self.poses_theta = [], [], []
        self.collisions = np.zeros((self.num_agents,))
        self.lidar_max = self.params.get("lidar_max", 30.0)
        self.near_start = True
        self.num_toggles = 0
        self.lap_times = np.zeros((self.num_agents,))
        self.lap_counts = np.zeros((self.num_agents,))
        self.current_time = 0.0
        self.near_starts = np.array([True] * self.num_agents)
        self.toggle_list = np.zeros((self.num_agents,))
        self.start_xs = np.zeros((self.num_agents,))
        self.start_ys = np.zeros((self.num_agents,))
        self.start_thetas = np.zeros((self.num_agents,))
        self.start_rot = np.eye(2)

        self.sim = Simulator(self.params, self.num_agents, self.seed, time_step=self.timestep, ego_idx=self.ego_idx,
                             integrator=self.integrator, lidar_dist=self.lidar_dist, noise=noise,
                             device=kwargs.get('device', None), edt=kwargs.get('edt', 'host'))
        self.sim.set_map(self.map_path, self.map_ext)

        self.x_min, self.x_max, self.y_min, self.y_max = map_bounds(self.map_path, self.map_dir)
        self.render_obs = None

        low = np.array([self.params['s_min'], self.params['v_min']], dtype=np.float32)
        high = np.array([self.params['s_max'], self.params['v_max']], dtype=np.float32)
        self.action_space = spaces.Box(low=np.tile(low, (self.num_agents, 1)), high=np.tile(high, (self.num_agents, 1)),
                                       dtype=np.float32)
        nb = self.sim.num_beams
        low = np.array([0.0] * nb + [self.x_min, self.y_min, -np.pi, 0.0, self.x_min, self.y_min, -np.pi, 0.0], dtype=np.float32)
        high = np.array([1.0] * nb + [self.x_max, self.y_max, np.pi, 1.0, self.x_max, self.y_max, np.pi, 1.0], dtype=np.float32)
        self.observation_space = spaces.Box(low=low, high=high, dtype=np.float32)

    # ------------------------------------------------------------------ gym API
    def _finish(self, o):
        """Everything F110Env.step does after Simulator.step (f110_env.py:389-421), read back from the device."""
        A = self.num_agents
        st = o['state'][0]
        obs_dict = self.sim._observations(o)
        # the obs dict carries the lap arrays as they were BEFORE this step's _check_done (f110_env.py:389-390)
        obs_dict['lap_times'] = self.lap_times.astype(np.float32)
        obs_dict['lap_counts'] = self.lap_counts.astype(np.float32)
        F110Env.current_obs = obs_dict
        self.render_obs = {k: obs_dict[k] for k in ('ego_idx', 'poses_x', 'poses_y', 'poses_theta', 'lap_times',
                                                    'lap_counts', 'scans')}
        reward = self.timestep
        self.current_time = float(o['time'][0])
        self.poses_x, self.poses_y, self.poses_theta = obs_dict['poses_x'], obs_dict['poses_y'], obs_dict['poses_theta']
        self.collisions = obs_dict['collisions']
        self.toggle_list = o['toggles'][0].astype(np.float64)
        self.lap_times = o['lap_times'][0].copy()
        self.lap_counts = o['lap_counts'][0].copy()
        terminated = bool(o['terminated'][0])
        toggle_done = self.toggle_list >= 4
        if self.obs_mode == 'scans':
            obs = o['scans_f32'][0].copy()
        else:
            obs = o['obs'][0].copy()
        info = {
            "ego_idx": int(self.ego_idx),
            "poses_x": st[:, 0].astype(np.float32),
            "poses_y": st[:, 1].astype(np.float32),
            "poses_theta": st[:, 4].astype(np.float32),
            "linear_vels_x": st[:, 3].astype(np.float32),
            "linear_vels_y": np.zeros(A, np.float32),
            "ang_vels_z": st[:, 5].astype(np.float32),
            "collisions": o['collisions'][0].astype(np.int8),
            "lap_times": self.lap_times.astype(np.float32),
            "lap_counts": self.lap_counts.astype(np.float32),
            "scans": [o['scans_f32'][0, i].copy() for i in range(A)],
            "checkpoint_done": toggle_done,
            "time": float(self.current_time),
        }
        return obs, reward, terminated, False, info

    def step(self, action):
        action = np.asarray(action)
        if action.dtype != np.float32:
            action = action.astype(np.float64)
        o = self.sim._step_raw(action.reshape(1, self.num_agents, 2))
        return self._finish(o)

    def reset(self, seed=None, options=None):
        poses = options
        if poses is None:
            # the reference dereferences None here (f110_env.py:438,448)
            raise TypeError("'NoneType' object is not subscriptable: F110Env.reset needs options=poses (num_agents, 3)")
        poses = np.asarray(poses, dtype=np.float64)
        if poses.shape[0] != self.num_agents:
            raise ValueError('Number of poses for reset does not match number of agents.')
        self.num_toggles = 0
        self.near_start = True
        self.near_starts = np.array([True] * self.num_agents)
        self.start_xs, self.start_ys, self.start_thetas = poses[:, 0], poses[:, 1], poses[:, 2]
        th = -self.start_thetas[self.ego_idx]
        self.start_rot = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        # RaceCar.reset re-seeds every car's generator (base_classes.py:204)
        self.sim._rngs = [np.random.default_rng(seed=self.sim.seed) for _ in range(self.num_agents)]
        o = self.sim._step_raw(None, reset_mask=np.ones(1, np.uint8), reset_poses=poses[None])
        obs, reward, terminated, truncated, info = self._finish(o)
        return obs, info

    def update_map(self, map_path, map_ext):
        self.sim.set_map(map_path, map_ext)

    def update_params(self, params, index=-1):
        self.sim.update_params(params, agent_idx=index)

    def add_render_callback(self, callback_func):
        F110Env.render_callbacks.append(callback_func)

    def render(self, mode='human'):
        """The pyglet viewer (rendering.py) is visualisation only and out of scope; callbacks still run."""
        assert mode in ['human', 'human_fast']
        for render_callback in F110Env.render_callbacks:
            render_callback(F110Env.renderer)

    def state_dict(self):
        """Checkpoint of the env: the library's versioned state blob, the host generators of the reference's lidar-noise
        stream (noise='numpy') and the lap bookkeeping this class mirrors on the host."""
        rng = None if self.sim._rngs is None else [r.bit_generator.state for r in self.sim._rngs]
        return {'backend': self.sim.backend.state_dict(), 'noise_rng': rng, 'current_time': self.current_time,
                'lap_times': self.lap_times.copy(), 'lap_counts': self.lap_counts.copy(), 'toggle_list': self.toggle_list.copy(),
                'start': (np.array(self.start_xs), np.array(self.start_ys), np.array(self.start_thetas), self.start_rot.copy())}

    def load_state_dict(self, sd):
        self.sim.backend.load_state_dict(sd['backend'])
        torch.cuda.current_stream(self.sim.backend.device).synchronize()
        if sd['noise_rng'] is not None:
            self.sim._rngs = [np.random.default_rng() for _ in sd['noise_rng']]
            for r, st in zip(self.sim._rngs, sd['noise_rng']):
                r.bit_generator.state = st
        self.current_time = sd['current_time']
        self.lap_times, self.lap_counts, self.toggle_list = sd['lap_times'].copy(), sd['lap_counts'].copy(), sd['toggle_list'].copy()
        self.start_xs, self.start_ys, self.start_thetas, self.start_rot = sd['start']

    def close(self):
        if getattr(self, 'sim', None) is not None:
            self.sim.backend.close()


def _map_specs(map_dir=None, map=None, map_arrays=None, maps=None):
    """The vector envs' map arguments as one BatchSim.set_maps spec list: one map is the set of one."""
    if maps is not None:
        if map is not None or map_arrays is not None:
            raise ValueError("give either maps= (a map set) or map= / map_arrays= (one map), not both")
        return maps
    if map_arrays is not None:
        dt, resolution, origin = map_arrays
        return [(np.asarray(dt, np.float64), resolution, origin)]
    return [map_dir + map + '.yaml']


class F110VecEnv(object):
    """N F110Envs stepped as one batch on one GPU; torch CUDA tensors in and out (zero-copy).

    ``step(actions [N, A, 2])`` -> ``(obs [N, B+8] f32, reward [N] f32, terminated [N] u8, truncated [N] u8, info)``.
    The returned tensors are persistent buffers rewritten by the next step.  With ``auto_reset=True`` an env
    that terminated is reset to its start poses by the NEXT step call, which is then that env's zero-action
    reset step (gymnasium's next-step autoreset; F110Env.reset semantics f110_env.py:425-472).

    ``maps=[spec, ...]`` instead of ``map=`` / ``map_arrays=`` installs a map set (BatchSim.set_maps): every env drives on
    the map of its slot, env e on slot floor(e * K / N) unless ``env_maps`` (int [N]) says otherwise; ``reassign`` moves envs
    to other maps at their next reset.  ShapedReward(centerlines=[...]) with one centerline per map, in slot order, scores
    each env on its own map's centerline (DeviceRollout passes it the slots).
    """

    def __init__(self, num_envs, map_dir=None, map=None, map_ext='.png', num_agents=2, params=None, seed=42,
                 timestep=0.01, ego_idx=0, integrator=Integrator.RK4, lidar_dist=0.0, device=None, auto_reset=True,
                 outputs=FAST_OUTPUTS, noise_std=0.01, num_beams=1080, fov=4.7, count_lookups=False, map_arrays=None,
                 cuda_graph=False, maps=None, env_maps=None):
        specs = _map_specs(map_dir, map, map_arrays, maps)
        self.num_envs, self.num_agents = num_envs, num_agents
        self.timestep = timestep
        self.auto_reset = auto_reset
        outs = tuple(dict.fromkeys(tuple(outputs) + ('obs', 'reward', 'terminated')))
        self.backend = BatchSim(num_envs, num_agents, params=params, seed=seed, timestep=timestep, integrator=integrator,
                                ego_idx=ego_idx, lidar_dist=lidar_dist, noise_std=noise_std, device=device, outputs=outs,
                                num_beams=num_beams, fov=fov, count_lookups=count_lookups)
        self.backend.set_maps(specs, map_ext=map_ext)
        if maps is not None and env_maps is not None:
            self.backend.set_env_maps(env_maps)
        self.device = self.backend.device
        self.start_poses = None
        self.truncated = torch.zeros(num_envs, dtype=torch.uint8, device=self.device)
        self.single_observation_shape = (num_beams + 8,)
        self.single_action_shape = (num_agents, 2)
        # cuda_graph=True: the step (3-4 kernel launches) is captured once and replayed, one launch per step on the host side
        self.cuda_graph = cuda_graph
        self._graph = None
        self._act = torch.zeros((num_envs, num_agents, 2), dtype=torch.float32, device=self.device)
        self._steps_eager = 0
        self._map_generation = self.backend.map_generation

    def reset(self, poses, noise=None):
        """poses [N, A, 3] (or [A, 3], broadcast to every env)."""
        p = torch.as_tensor(np.asarray(poses, np.float64) if not torch.is_tensor(poses) else poses, dtype=torch.float64)
        if p.ndim == 2:
            p = p[None].expand(self.num_envs, -1, -1)
        self.start_poses = p.to(self.device).contiguous()
        self._graph = None          # the captured step holds the old start-pose tensor
        self._steps_eager = 0
        o = self.backend.reset(self.start_poses, noise)
        return o['obs'], o

    def step(self, actions, noise=None):
        o = self.backend.out
        if self._graph is not None and self._map_generation != self.backend.map_generation:
            self._drop_graph()      # the map was changed behind the env's back (backend.set_map*): see set_maps
        if self.cuda_graph and noise is None and self.auto_reset and self.start_poses is not None:
            self._act.copy_(torch.as_tensor(actions, device=self.device).reshape(self._act.shape))
            if self._graph is None and self._steps_eager >= 1:
                # capture on a side stream (the first step ran eagerly and warmed everything up); capture does not execute
                side = torch.cuda.Stream(self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                g = torch.cuda.CUDAGraph()
                with torch.cuda.stream(side):
                    with torch.cuda.graph(g, stream=side):
                        self.backend.step(self._act, None, reset_mask=o['terminated'], reset_poses=self.start_poses)
                torch.cuda.current_stream(self.device).wait_stream(side)
                self._graph = g
            if self._graph is not None:
                self._graph.replay()
                return o['obs'], o['reward'], o['terminated'], self.truncated, o
            self._steps_eager += 1
            o = self.backend.step(self._act, None, reset_mask=o['terminated'], reset_poses=self.start_poses)
            return o['obs'], o['reward'], o['terminated'], self.truncated, o
        if self.auto_reset:
            # `terminated` of the previous step doubles as this step's reset mask (read by K1 before K3 rewrites it)
            o = self.backend.step(actions, noise, reset_mask=o['terminated'], reset_poses=self.start_poses)
        else:
            o = self.backend.step(actions, noise)
        return o['obs'], o['reward'], o['terminated'], self.truncated, o

    def set_map(self, map_path, map_ext, edt='host'):
        """update_map for the whole batch: the set of one map (set_maps)."""
        self.set_maps([map_path], edt=edt, map_ext=map_ext)

    def set_map_arrays(self, dt, resolution, origin):
        self.set_maps(_map_specs(map_arrays=(dt, resolution, origin)))

    def set_maps(self, specs, edt='host', map_ext='.png'):
        """Installs a map set for the whole batch (BatchSim.set_maps; env e on slot floor(e * K / N)).  A captured CUDA graph
        holds the previous (freed) map by value: it is dropped here and re-captured by the next steps."""
        self.backend.set_maps(specs, edt=edt, map_ext=map_ext)
        self._drop_graph()

    def reassign(self, env_mask, slots, start_poses):
        """Moves the masked envs to map `slots` with new start poses, effective at their reset on the next step: sets their
        slots (BatchSim.set_env_maps) and start poses and ORs the mask into `terminated`, the next step's reset mask.  All
        three are in-place, stream-ordered device writes, so a captured CUDA graph replays them without re-capture.
        env_mask [N] (non-zero = move), slots int [N] (or one int), start_poses [N, A, 3] (or [A, 3]); entries of unmasked
        envs are ignored.  Needs auto_reset=True (without it nothing would reset the envs)."""
        if not self.auto_reset:
            raise ValueError("reassign needs auto_reset=True: the moved envs are reset by the next step")
        if self.start_poses is None:
            raise ValueError("reset() the batch before reassign()")
        N = self.num_envs
        m = torch.as_tensor(np.asarray(env_mask) if not torch.is_tensor(env_mask) else env_mask).to(self.device)
        m = (m.reshape(N) != 0)
        sl = torch.as_tensor(np.asarray(slots) if not torch.is_tensor(slots) else slots).to(self.device, torch.int32)
        sl = sl.expand(N).contiguous() if sl.ndim == 0 else sl.reshape(N).contiguous()
        p = torch.as_tensor(np.asarray(start_poses, np.float64) if not torch.is_tensor(start_poses) else start_poses,
                            dtype=torch.float64).to(self.device)
        if p.ndim == 2:
            p = p[None].expand(N, -1, -1)
        self.backend.set_env_maps(sl, m.to(torch.uint8))
        self.start_poses.copy_(torch.where(m[:, None, None], p, self.start_poses))
        term = self.backend.out['terminated']
        term.bitwise_or_(m.to(torch.uint8))

    def _drop_graph(self):
        self._graph = None
        self._steps_eager = 0
        self._map_generation = self.backend.map_generation

    def state_dict(self):
        """Everything needed to continue the batch bit for bit in another process: the library's state blob (versioned,
        BatchSim.state_dict), plus what lives on this side of the C ABI -- the terminated flags (the next step's reset mask
        under auto-reset) and the start poses."""
        return {'backend': self.backend.state_dict(), 'terminated': self.backend.out['terminated'].clone(),
                'start_poses': None if self.start_poses is None else self.start_poses.clone(), 'auto_reset': self.auto_reset,
                'env_maps': self.backend.env_maps().clone()}

    def load_state_dict(self, sd):
        self.backend.load_state_dict(sd['backend'])
        if sd.get('env_maps') is not None:
            self.backend.set_env_maps(sd['env_maps'].cpu().numpy())      # host form: a slot this env's maps lack raises
        self.backend.out['terminated'].copy_(sd['terminated'].to(self.device))
        self.start_poses = None if sd['start_poses'] is None else sd['start_poses'].to(self.device).contiguous()
        self._drop_graph()          # a captured step holds the old start-pose tensor

    def close(self):
        self.backend.close()


class F110HostVecEnv(object):
    """N F110Envs for a HOST-side consumer: numpy actions in, pinned-host observations out, every step.

    This is the end-to-end shape of the reference's own use (train_ddpg.py:160-202 reads the observation on the
    host every step).  The envs are split over ``chunks`` independent library handles, each with its own stream;
    a step enqueues, per chunk, the upload, the three kernels and the downloads (f110_step_host_async), then waits
    for all of them (f110_host_sync) -- so one chunk's PCIe traffic overlaps the other chunks' kernels.  Per chunk the
    inputs (actions, start poses, reset mask) sit back to back in one pinned block and so do reward and terminated,
    which the library then moves with one copy each (include/f110_b200.h, f110_step_host_async); the observation
    goes straight into its slice of one contiguous [N, B+8] pinned array.  Auto-reset as in F110VecEnv.

    ``chunks``: an int (equal chunks) or relative sizes, e.g. (1, 3): a small first chunk starts the downloads sooner.
    """

    def __init__(self, num_envs, chunks=2, map_arrays=None, map_dir=None, map=None, map_ext='.png', num_agents=1,
                 seed=42, device=None, outputs=FAST_OUTPUTS, num_beams=1080, maps=None, env_maps=None, **kw):
        specs = _map_specs(map_dir, map, map_arrays, maps)
        self.num_envs, self.num_agents, self.num_beams = num_envs, num_agents, num_beams
        if maps is not None:
            # the whole batch's assignment (F110VecEnv's default: env e on slot floor(e K / N)); each chunk gets its slice
            slots = (np.arange(num_envs) * len(maps)) // num_envs if env_maps is None else np.asarray(env_maps, np.int32)
        if isinstance(chunks, int):
            chunks = max(1, min(chunks, num_envs))
            self.bounds = [(num_envs * k) // chunks for k in range(chunks + 1)]
        else:
            w = np.cumsum([0.0] + [float(v) for v in chunks])
            self.bounds = sorted(set(int(round(num_envs * v / w[-1])) for v in w))
            chunks = len(self.bounds) - 1
        self.parts = []
        for k in range(chunks):
            n = self.bounds[k + 1] - self.bounds[k]
            b = BatchSim(n, num_agents, seed=seed + 7919 * k, device=device, outputs=('obs',), num_beams=num_beams,
                         host_stream_rank=k + 1, **kw)
            b.set_maps(specs, map_ext=map_ext)
            if maps is not None:
                b.set_env_maps(slots[self.bounds[k]:self.bounds[k + 1]])
            self.parts.append(b)
        outs = tuple(dict.fromkeys(tuple(outputs) + ('obs', 'reward', 'terminated')))
        from .backend import _OUT_SPECS
        # Every output buffer is a slice of ONE pinned allocation (that is what F110_HOST_MERGE_ADJACENT vouches for).
        # reward / terminated live in per-chunk [reward f32 | terminated u8] blocks, which the library downloads with one
        # copy, and are gathered into plain whole-batch arrays after a step; everything else is a whole-batch array
        # the copy engine writes directly.
        specs = [(key,) + _OUT_SPECS[key] for key in outs if key not in ('reward', 'terminated')]
        sizes = [int(np.prod(shape(num_envs, num_agents, num_beams))) * torch.zeros(0, dtype=dt).element_size()
                 for _, shape, dt in specs]
        offs = np.cumsum([0] + [(b + 255) // 256 * 256 for b in sizes])
        small0 = int(offs[-1])
        self._arena = torch.zeros(small0 + sum((5 * (self.bounds[k + 1] - self.bounds[k]) + 255) // 256 * 256
                                               for k in range(chunks)), dtype=torch.uint8, pin_memory=True)
        self.out, self._np = {}, {}
        for (key, shape, dt), off, nb in zip(specs, offs, sizes):
            self.out[key] = self._arena[int(off):int(off) + nb].view(dt).view(shape(num_envs, num_agents, num_beams))
            self._np[key] = self.out[key].numpy()
        self._np['reward'] = np.zeros(num_envs, np.float32)
        self._np['terminated'] = np.ones(num_envs, np.uint8)
        self.out['reward'] = torch.from_numpy(self._np['reward'])
        self.out['terminated'] = torch.from_numpy(self._np['terminated'])
        self._rew_k, self._term_k = [], []
        off = small0
        for k in range(chunks):
            n = self.bounds[k + 1] - self.bounds[k]
            self._rew_k.append(self._arena[off:off + 4 * n].view(torch.float32).numpy())
            self._term_k.append(self._arena[off + 4 * n:off + 5 * n].numpy())
            off += (5 * n + 255) // 256 * 256
        self._in = {}            # action dtype -> per-chunk input blocks (built at the first step with that dtype)
        self.start_poses = None

    def _input_blocks(self, dtype):
        """Per chunk one pinned block [actions | start poses f64 | reset mask u8] for actions of this dtype, and the
        F110StepIO of every chunk pointing into it: all buffers are persistent, a step only fills them."""
        import ctypes as C
        from . import _lib
        if dtype in self._in:
            return self._in[dtype]
        K, A = len(self.parts), self.num_agents
        ios = (_lib.F110StepIO * K)()
        acts, masks, keep = [], [], []
        for k in range(K):
            lo, hi = self.bounds[k], self.bounds[k + 1]
            n = hi - lo
            ab = n * A * 2 * dtype.itemsize
            blk = torch.zeros(ab + n * A * 24 + n, dtype=torch.uint8, pin_memory=True)
            a = blk[:ab].numpy().view(dtype).reshape(n, A, 2)
            p = blk[ab:ab + n * A * 24].numpy().view(np.float64).reshape(n, A, 3)
            p[...] = self.start_poses[lo:hi]
            m = blk[ab + n * A * 24:].numpy()
            io = ios[k]
            io.actions, io.actions_f64 = a.ctypes.data, int(dtype == np.float64)
            io.host_flags = _lib.F110_HOST_MERGE_ADJACENT      # adjacent buffers below are slices of one pinned block
            io.reset_poses, io.reset_mask = p.ctypes.data, m.ctypes.data
            io.reward, io.terminated = self._rew_k[k].ctypes.data, self._term_k[k].ctypes.data
            for key, t in self.out.items():
                if key not in ('reward', 'terminated'):
                    setattr(io, key, t[lo:hi].data_ptr())
            acts.append(a); masks.append(m); keep.append(blk)
        handles = (C.c_void_p * K)(*[b.h for b in self.parts])
        self._in[dtype] = (ios, handles, acts, masks, keep)
        self._lib = _lib
        return self._in[dtype]

    def _fill(self, k, blocks, actions):
        """chunk k's inputs for the next step: its actions (None = zero action: a reset step) and, as reset mask, the
        `terminated` its previous step produced."""
        ios, _, acts, masks, _ = blocks
        np.copyto(masks[k], self._term_k[k])
        if actions is None:
            ios[k].actions = None
        else:
            ios[k].actions = acts[k].ctypes.data
            np.copyto(acts[k], actions.reshape(acts[k].shape))

    def _gather(self, k):
        sl = slice(self.bounds[k], self.bounds[k + 1])
        self._np['reward'][sl] = self._rew_k[k]
        self._np['terminated'][sl] = self._term_k[k]

    @staticmethod
    def _as_actions(actions):
        a = np.asarray(actions)
        return a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)

    def _run(self, actions):
        K = len(self.parts)
        a = None if actions is None else self._as_actions(actions)
        blocks = self._input_blocks(np.dtype(np.float32) if a is None else a.dtype)
        if a is not None:
            assert a.size == self.num_envs * self.num_agents * 2
            a = a.reshape(self.num_envs, self.num_agents, 2)
        for k in range(K):
            self._fill(k, blocks, None if a is None else a[self.bounds[k]:self.bounds[k + 1]])
        self._lib.check(self._lib.load().f110_step_host_multi(blocks[1], blocks[0], K))
        for k in range(K):
            self._gather(k)
        return self.out

    def reset(self, poses):
        p = np.asarray(poses, np.float64)
        if p.ndim == 2:
            p = np.broadcast_to(p[None], (self.num_envs,) + p.shape)
        self.start_poses = np.ascontiguousarray(p)
        self._in = {}
        for t in self._term_k:
            t[:] = 1
        o = self._run(None)
        return self._np['obs'], o

    def step(self, actions):
        """actions: numpy [N, A, 2] f32/f64.  The previous step's `terminated` is this step's reset mask."""
        o = self._run(actions)
        return self._np['obs'], self._np['reward'], self._np['terminated'], None, o

    # ---- pipelined use (EnvPool-style): the chunks step independently, so the host can prepare chunk k's next
    # actions while the other chunks' kernels and downloads are in flight ACROSS step boundaries.  Per chunk the
    # order is recv(k) -> read chunk_out(k) -> send(k, actions); a chunk's buffers must not be touched between
    # send and recv.
    def chunk_slice(self, k):
        return slice(self.bounds[k], self.bounds[k + 1])

    def send(self, k, actions):
        """Enqueue one step of chunk k (upload, kernels, downloads) and return at once.  actions: [n_k, A, 2]."""
        a = self._as_actions(actions)
        blocks = self._input_blocks(a.dtype)
        assert a.size == (self.bounds[k + 1] - self.bounds[k]) * self.num_agents * 2
        self._fill(k, blocks, a)
        self._lib.check(self._lib.load().f110_step_host_async(self.parts[k].h, blocks[0][k]))

    def recv(self, k):
        """Wait for chunk k's step; returns (obs, reward, terminated) views of the pinned buffers for that chunk."""
        self._lib.check(self._lib.load().f110_host_sync(self.parts[k].h))
        return self._np['obs'][self.chunk_slice(k)], self._rew_k[k], self._term_k[k]

    def close(self):
        for b in self.parts:
            b.close()
