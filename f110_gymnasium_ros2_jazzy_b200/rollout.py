"""Device-resident rollout loop (SURVEY 8f row 1 / BASELINE config 5).

The reference's training loop (rl_training/train_ddpg.py:160-202) does, per step and on the host:
ego action from the actor, opponent action ``gap_follow_action(info["scans"][1])``, ``np.stack``, ``env.step``.
Here the same loop shape runs with every tensor on the GPU: the actor is a torch module evaluated on the observation
tensor the step kernels wrote (zero-copy), the opponent is the ``f110_gap_follow`` kernel reading the opponent's scan
in place and writing its action slot in place, and the step consumes the action tensor in place.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib


def gap_follow_actions(scans_f32, actions, agent_idx=1, angle_min=-np.pi / 2, angle_increment=np.pi / 1080,
                       max_distance=3.0, window_size=5, bubble_radius=30, threshold=0.5):
    """Batched gap_follow_action (gap_follow.py:43-58): for every env, agent ``agent_idx``'s scan -> its action slot.

    scans_f32: CUDA float32 [N, A, B] (F110VecEnv output 'scans_f32'); actions: CUDA float32 [N, A, 2], written in place.
    """
    if not (scans_f32.is_cuda and actions.is_cuda and scans_f32.dtype == torch.float32 and actions.dtype == torch.float32):
        raise ValueError("gap_follow_actions needs CUDA float32 tensors")
    if not (scans_f32.is_contiguous() and actions.is_contiguous()):
        raise ValueError("gap_follow_actions needs contiguous tensors")
    N, A, B = scans_f32.shape
    lib = _lib.load()
    stream = C.c_void_p(torch.cuda.current_stream(scans_f32.device).cuda_stream)
    _lib.check(lib.f110_gap_follow(C.c_void_p(scans_f32.data_ptr() + 4 * agent_idx * B), N, A * B, B,
                                   C.c_void_p(actions.data_ptr() + 4 * 2 * agent_idx), 2 * A, angle_min, angle_increment,
                                   max_distance, window_size, bubble_radius, threshold, stream))
    return actions


class Actor(torch.nn.Module):
    """The reference's DDPG actor architecture (rl_training/DDPG/agent.py:25-62): obs -> 128 -> 128 -> act, ReLU,
    tanh scaled to the action bounds.  The learner itself is out of scope; this is what a rollout evaluates."""

    def __init__(self, obs_dim, act_dim, action_low, action_high):
        super().__init__()
        self.fc1 = torch.nn.Linear(obs_dim, 128)
        self.fc2 = torch.nn.Linear(128, 128)
        self.fc3 = torch.nn.Linear(128, act_dim)
        self.register_buffer("action_low", torch.tensor(action_low, dtype=torch.float32))
        self.register_buffer("action_high", torch.tensor(action_high, dtype=torch.float32))
        # the two constants of the output scaling, formed once instead of with four small kernels per forward
        self.register_buffer("_scale", 0.5 * (self.action_high - self.action_low), persistent=False)
        self.register_buffer("_offset", 0.5 * (self.action_high + self.action_low), persistent=False)
        torch.nn.init.kaiming_uniform_(self.fc1.weight, nonlinearity="relu")
        torch.nn.init.kaiming_uniform_(self.fc2.weight, nonlinearity="relu")
        torch.nn.init.uniform_(self.fc3.weight, -3e-3, 3e-3)
        for b in (self.fc1.bias, self.fc2.bias, self.fc3.bias):
            torch.nn.init.zeros_(b)

    def forward(self, obs):
        x = torch.relu(self.fc1(obs))
        x = torch.relu(self.fc2(x))
        t = torch.tanh(self.fc3(x))
        return self._scale * t + self._offset


class DeviceRollout(object):
    """ego = policy(obs), opponent = gap-follow on its own scan, env.step -- no host round trip per step.

    ``reward_fn`` (optional, e.g. ShapedReward) replaces the env's constant reward, as train_ddpg.py:179 does.  A reward
    with K > 1 centerlines needs a map set of K maps (F110VecEnv(maps=...)): every step it is passed the envs' slots, so
    each env is scored on its own map's centerline, whatever moved it there (set_env_maps, reassign, load_state_dict).
    ``replay`` (optional, e.g. DeviceReplayBuffer) receives every transition (obs, ego action, reward, next obs, done)
    except the auto-reset steps (see step).
    ``env`` is an F110VecEnv with num_agents == 2 and 'scans_f32' among its outputs; ``policy`` maps the observation
    tensor [N, B+8] to ego actions [N, 2] (e.g. Actor).  ``opponent`` may be 'gap_follow' or a constant (steer, speed).
    """

    def __init__(self, env, policy, opponent='gap_follow', reward_fn=None, replay=None):
        if env.num_agents != 2:
            raise ValueError("DeviceRollout mirrors the reference's two-car loop (ego + opponent)")
        if opponent == 'gap_follow' and 'scans_f32' not in env.backend.out:
            raise ValueError("the gap-follow opponent needs the env's 'scans_f32' output")
        self.env, self.policy, self.opponent = env, policy, opponent
        self.actions = torch.zeros((env.num_envs, 2, 2), dtype=torch.float32, device=env.device)
        if opponent != 'gap_follow':
            self.actions[:, 1, 0] = float(opponent[0])
            self.actions[:, 1, 1] = float(opponent[1])
        self.obs = None
        self.reward_fn = reward_fn          # e.g. ShapedReward: train_ddpg.py:179 discards the env's reward for it
        self._slots = None
        k = getattr(reward_fn, 'num_centerlines', 1)
        if k > 1:
            if env.backend.num_maps != k:
                raise ValueError("a reward with %d centerlines needs a map set of %d maps (the env has %d)"
                                 % (k, k, env.backend.num_maps))
            self._slots = torch.zeros(env.num_envs, dtype=torch.int32, device=env.device)   # refreshed every step
        self.reward = None
        self.replay = replay                # e.g. DeviceReplayBuffer: agent.remember(obs, ego_action, r, next_obs, done), :185
        self._prev_obs = None if replay is None else torch.zeros((env.num_envs,) + tuple(env.single_observation_shape),
                                                                 dtype=torch.float32, device=env.device)

    def reset(self, poses):
        self.obs, o = self.env.reset(poses)
        n, dev = self.env.num_envs, self.env.device
        # envs whose NEXT step is the first real step of an episode: every env, right after a reset
        self._first = torch.ones(n, dtype=torch.uint8, device=dev)
        self._resetting = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._fresh = torch.zeros(n, dtype=torch.uint8, device=dev)
        return self.obs

    @torch.no_grad()
    def step(self):
        """One step of the loop train_ddpg.py:160-202 runs per env.  An env that terminated on the previous step is auto-reset
        by this one: that step is the reference's ``env.reset()`` between episodes (:152), not a transition -- its action is
        ignored by the env, its observation is the reset observation.  Such envs are kept out of the replay memory (the
        reference ``break``s on done and never stores a terminal -> reset pair), get reward 0, and their reward object starts
        over (``reward_fn.reset()``, :151) so that its first call is on the first real next_obs, as in the reference."""
        self.actions[:, 0, :] = self.policy(self.obs)
        if self.opponent == 'gap_follow':
            gap_follow_actions(self.env.backend.out['scans_f32'], self.actions, agent_idx=1)
        self._resetting.copy_(self.env.backend.out['terminated'])      # this step resets these envs (auto-reset)
        if self.env.backend.out['terminated'].data_ptr() == self._resetting.data_ptr():
            raise RuntimeError("internal: the terminated flags must be copied before the step rewrites them")
        if self.replay is not None:
            self._prev_obs.copy_(self.obs)          # the env rewrites its observation tensor in place
        self.obs, reward, terminated, truncated, info = self.env.step(self.actions)
        if self.reward_fn is not None:
            # reward object restarted on the reset step itself (its value there is discarded) and again on the first real step
            torch.maximum(self._resetting, self._first, out=self._fresh)
            if self._slots is None:
                reward = self.reward_fn(self.obs, self._fresh)
            else:
                reward = self.reward_fn(self.obs, self._fresh, slots=self.env.backend.env_maps(out=self._slots))
            reward.masked_fill_(self._resetting.bool(), 0.0)
        self.reward = reward
        if self.replay is not None:
            self.replay.add(self._prev_obs, self.actions[:, 0, :], reward, self.obs, terminated, keep=self._resetting == 0)
        self._first.copy_(self._resetting)          # the step after a reset step is an episode's first real step
        return self.obs, reward, terminated, truncated, info


class DeviceReplayBuffer(object):
    """The replay memory of the reference's DDPG agent (rl_training/DDPG/replay_buffer.py:6-135,
    PrioritizedExperienceReplayBuffer) as device-resident tensors, filled a whole batch of envs at a time, so that
    transitions go from the env's output tensors into the buffer without touching the host (SURVEY 8f row 1).

    Same semantics: ring-buffer insertion (:46-71) with a new transition's priority = the current maximum (1.0 when
    empty); sampling probabilities (prio + eps)^alpha / sum (:86-95), without replacement when the buffer holds at
    least a batch (:97-101); importance weights (len * p)^-beta normalised by their maximum (:103-113);
    update_priorities clamps to [1e-8, f32 max] and maps non-finite values to 1e-6 (:120-135).
    Layout: SoA tensors [capacity, ...] (obs and next_obs f32 [capacity, obs_dim]: 8.7 KB per transition at 1088).
    """

    def __init__(self, capacity, batch_size, obs_dim=1088, act_dim=2, alpha=0.6, priority_epsilon=1e-6, device=None, seed=42):
        assert capacity > 0 and batch_size > 0
        self.capacity, self.batch_size, self.alpha, self.eps = int(capacity), int(batch_size), float(alpha), float(priority_epsilon)
        dev = torch.device(device) if device is not None else torch.device('cuda' if torch.cuda.is_available() else 'cpu')
        self.device = dev
        # one row more than the capacity: transitions masked out of an add() are written there, so that a masked add needs
        # neither a compaction nor a host round trip
        self._obs = torch.zeros((capacity + 1, obs_dim), dtype=torch.float32, device=dev)
        self._next_obs = torch.zeros((capacity + 1, obs_dim), dtype=torch.float32, device=dev)
        self._action = torch.zeros((capacity + 1, act_dim), dtype=torch.float32, device=dev)
        self._reward = torch.zeros(capacity + 1, dtype=torch.float32, device=dev)
        self._done = torch.zeros(capacity + 1, dtype=torch.uint8, device=dev)
        self._priority = torch.zeros(capacity + 1, dtype=torch.float32, device=dev)
        self.obs, self.next_obs, self.action = self._obs[:capacity], self._next_obs[:capacity], self._action[:capacity]
        self.reward, self.done, self.priority = self._reward[:capacity], self._done[:capacity], self._priority[:capacity]
        self._len = torch.zeros((), dtype=torch.int64, device=dev)      # ring-buffer counters live on the device
        self._next = torch.zeros((), dtype=torch.int64, device=dev)
        self._max_prio = torch.ones((), dtype=torch.float32, device=dev)     # running maximum, kept on the device
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(seed)

    @property
    def length(self):
        return int(self._len)        # (synchronises)

    @property
    def next_idx(self):
        return int(self._next)

    def __len__(self):
        return self.length

    @torch.no_grad()
    def add(self, obs, action, reward, next_obs, done, priority=None, keep=None):
        """One transition per env: obs/next_obs [n, obs_dim], action [n, act_dim], reward [n], done [n].
        ``keep`` [n] (optional): only the rows where it is non-zero are stored, in order, without a host round trip."""
        n = obs.shape[0]
        if n > self.capacity:
            raise ValueError("more transitions in one add() than the buffer holds")
        empty = self._len == 0
        if priority is None:
            p0 = torch.where(empty, torch.ones_like(self._max_prio), self._max_prio).expand(n)
        else:
            p0 = torch.as_tensor(priority, dtype=torch.float32, device=self.device).expand(n)
        p0 = torch.clamp(p0, 1e-8, torch.finfo(torch.float32).max)
        if keep is None:
            count = torch.full((), n, dtype=torch.int64, device=self.device)
            idx = (self._next + torch.arange(n, device=self.device)) % self.capacity
        else:
            k = keep.to(device=self.device).reshape(n) != 0
            rank = torch.cumsum(k, 0)
            count = rank[-1]
            idx = torch.where(k, (self._next + rank - 1) % self.capacity, torch.full_like(rank, self.capacity))
        self._obs.index_copy_(0, idx, obs.to(torch.float32))
        self._next_obs.index_copy_(0, idx, next_obs.to(torch.float32))
        self._action.index_copy_(0, idx, action.to(torch.float32))
        self._reward.index_copy_(0, idx, reward.to(torch.float32).reshape(n))
        self._done.index_copy_(0, idx, done.to(torch.uint8).reshape(n))
        self._priority.index_copy_(0, idx, p0)
        new_max = torch.where(empty, p0.max(), torch.maximum(self._max_prio, p0.max()))
        self._max_prio = torch.where(count > 0, new_max, self._max_prio)
        self._len = torch.clamp(self._len + count, max=self.capacity)
        self._next = (self._next + count) % self.capacity

    def probabilities(self):
        ps = (self.priority[:self.length] + self.eps).double() ** self.alpha     # the sum is formed in float32, as numpy does (:88)
        den = ps.sum()
        if not bool(torch.isfinite(den)) or float(den) <= 0.0:
            return torch.full((self.length,), 1.0 / self.length, dtype=torch.float64, device=self.device)
        return ps / den

    @torch.no_grad()
    def sample(self, beta=0.4):
        """-> idxs [B] int64, (obs, action, reward, next_obs, done) gathered on the device, weights [B] f32."""
        if self.length == 0:
            raise ValueError("Cannot sample from an empty buffer.")
        probs = self.probabilities()
        idxs = torch.multinomial(probs, self.batch_size, replacement=self.length < self.batch_size, generator=self.gen)
        w = (self.length * probs[idxs]) ** (-float(beta))
        m = w.max()
        w = torch.ones_like(w) if (not bool(torch.isfinite(m)) or float(m) <= 0.0) else w / m
        batch = (self.obs[idxs], self.action[idxs], self.reward[idxs], self.next_obs[idxs], self.done[idxs])
        return idxs, batch, w.to(torch.float32)

    @torch.no_grad()
    def update_priorities(self, idxs, priorities):
        pr = torch.as_tensor(priorities, dtype=torch.float32, device=self.device).reshape(-1)
        pr = torch.clamp(pr, 1e-8, torch.finfo(torch.float32).max)
        pr = torch.where(torch.isfinite(pr), pr, torch.full_like(pr, 1e-6))
        self.priority.index_copy_(0, torch.as_tensor(idxs, device=self.device).reshape(-1).long(), pr)
        self._max_prio = self.priority[:self.length].max()


# CenterlineSafetyProgressReward.__init__ defaults (rl_training/utils/rewards.py:196-222)
REWARD_DEFAULTS = dict(dt=0.01, w_prog=1.2, forward_sign=+1.0, alive_bonus=0.02, w_rel_lead=0.0, lead_clip=5.0, w_lat=0.35,
                       lat_cap=4.0, default_half_width=1.5, lidar_max=1.0, near_wall_dist=0.35 / 30.0, w_wall=1.0,
                       wall_quantile=0.05, opp_safe_dist=0.7, w_opp=0.8, ego_crash_penalty=50.0, opp_crash_bonus=50.0,
                       grace_steps_wall=25, grace_steps_opp=25)


class ShapedReward(object):
    """Batched CenterlineSafetyProgressReward (rewards.py:185-355) on a CenterlineProgress (track_progress.py): one
    independent reward object per env, evaluated by ``f110_reward_compute`` straight from the observation tensor.

    ``centerline``: [n, 2] (x_m, y_m) or [n, 4] (+ w_tr_right_m, w_tr_left_m), the CSV train_ddpg.py loads.  Keyword
    arguments are the reference constructor's.  ``__call__(obs, reset_mask=None)`` returns a float64 CUDA tensor [N];
    ``reset_mask`` plays the role of ``reward_fn.reset()`` per env.

    ``centerlines=[cl_0, ..., cl_{K-1}]`` instead of ``centerline`` (1 <= K <= 256, each [n, 2] or [n, 4] with
    2 <= n <= 16385) holds one centerline per map of a map set, in slot order; ``closed`` is then one flag for all or a
    list of K.  ``__call__`` then needs ``slots`` (CUDA int32 [N], e.g. BatchSim.env_maps()): env e is scored exactly as a
    reward on ``centerlines[slots[e]]`` alone would score it.  A changed slot restarts that env's record, as its reset mask
    does; a slot outside [0, K) gives NaN and leaves the env's record alone.  Parameters are shared by the whole set.
    """

    def __init__(self, num_envs, centerline=None, num_beams=1080, closed=True, device=None, centerlines=None, **kw):
        unknown = set(kw) - set(REWARD_DEFAULTS)
        if unknown:
            raise TypeError("unknown reward arguments: %s" % sorted(unknown))
        if (centerline is None) == (centerlines is None):
            raise ValueError("give either centerline= or centerlines=, not both and not neither")
        lines = _check_centerlines(centerlines, closed) if centerlines is not None else None
        p = dict(REWARD_DEFAULTS)
        p.update(kw)
        self.lib = _lib.load()
        self.device = torch.device('cuda', torch.cuda.current_device() if device is None else device)
        cfg = _lib.F110RewardConfig(num_envs=num_envs, num_beams=num_beams, device=self.device.index,
                                    grace_steps_wall=int(p['grace_steps_wall']), grace_steps_opp=int(p['grace_steps_opp']),
                                    **{k: float(v) for k, v in p.items() if not k.startswith('grace_')})
        h = C.c_void_p()
        if lines is None:
            cl = np.ascontiguousarray(centerline, np.float64)
            xy = np.ascontiguousarray(cl[:, :2])
            wR = np.ascontiguousarray(cl[:, 2]) if cl.shape[1] >= 4 else None
            wL = np.ascontiguousarray(cl[:, 3]) if cl.shape[1] >= 4 else None
            cfg.num_points, cfg.closed = len(xy), int(closed)
            _lib.check(self.lib.f110_reward_create(C.byref(cfg), xy.ctypes.data_as(C.c_void_p),
                                                   None if wR is None else wR.ctypes.data_as(C.c_void_p),
                                                   None if wL is None else wL.ctypes.data_as(C.c_void_p), C.byref(h)))
            self.num_centerlines = 1
        else:
            descs = (_lib.F110Centerline * len(lines))()
            for d, (xy, wR, wL, c) in zip(descs, lines):
                d.xy = xy.ctypes.data
                d.wR = None if wR is None else wR.ctypes.data
                d.wL = None if wL is None else wL.ctypes.data
                d.num_points, d.closed = len(xy), int(c)
            _lib.check(self.lib.f110_reward_create_set(C.byref(cfg), descs, len(lines), C.byref(h)))
            self.num_centerlines = len(lines)
        self.h = h
        self.N, self.B = num_envs, num_beams
        self.out = torch.zeros(num_envs, dtype=torch.float64, device=self.device)

    def __call__(self, obs, reset_mask=None, slots=None):
        if not (obs.is_cuda and obs.dtype == torch.float32 and obs.is_contiguous() and obs.numel() == self.N * (self.B + 8)):
            raise ValueError("obs must be a contiguous CUDA float32 tensor [N, B+8]")
        if slots is None and self.num_centerlines > 1:
            raise ValueError("a reward with %d centerlines needs each env's slot (slots=)" % self.num_centerlines)
        rm = sl = None
        if reset_mask is not None:
            rm = reset_mask.to(device=self.device, dtype=torch.uint8).contiguous()
            self._keep = rm
        if slots is not None:
            if not (torch.is_tensor(slots) and slots.is_cuda and slots.dtype == torch.int32 and slots.is_contiguous()
                    and slots.numel() == self.N):
                raise ValueError("slots must be a contiguous CUDA int32 tensor [N]")
            sl = slots
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        _lib.check(self.lib.f110_reward_compute_slots(self.h, ptr(obs), ptr(rm), ptr(sl), ptr(self.out), None, stream))
        return self.out

    def close(self):
        if getattr(self, 'h', None):
            self.lib.f110_reward_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _check_centerlines(centerlines, closed):
    """-> [(xy [n, 2], wR [n] or None, wL [n] or None, closed)] per line, or ValueError naming the first bad line; no
    library call, so the checks hold without a device."""
    lines = list(centerlines)
    if not 1 <= len(lines) <= _lib.F110_MAX_MAPS:
        raise ValueError("centerlines: %d given; 1 to %d allowed" % (len(lines), _lib.F110_MAX_MAPS))
    if isinstance(closed, (list, tuple, np.ndarray)):
        flags = [bool(c) for c in closed]
        if len(flags) != len(lines):
            raise ValueError("closed: %d flags for %d centerlines" % (len(flags), len(lines)))
    else:
        flags = [bool(closed)] * len(lines)
    out = []
    for k, (cl, c) in enumerate(zip(lines, flags)):
        cl = np.asarray(cl, np.float64)
        if cl.ndim != 2 or cl.shape[1] not in (2, 4):
            raise ValueError("centerline %d: shape %s; [n, 2] (x, y) or [n, 4] (+ w_right, w_left) expected" % (k, cl.shape))
        if not 2 <= len(cl) <= 16385:
            raise ValueError("centerline %d has %d points; 2 to 16385 allowed" % (k, len(cl)))
        wide = cl.shape[1] == 4
        out.append((np.ascontiguousarray(cl[:, :2]), np.ascontiguousarray(cl[:, 2]) if wide else None,
                    np.ascontiguousarray(cl[:, 3]) if wide else None, c))
    return out
