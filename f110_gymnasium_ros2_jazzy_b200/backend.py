"""BatchSim: N independent F1TENTH envs x A agents stepped on one B200 through libf110_b200.so.

The simulation state lives in a device arena owned by the library; every input and output of a
step is a torch CUDA tensor owned by the caller's process and handed over as a raw pointer
(zero-copy with the RL loop).  torch is plumbing only: device memory, streams, (optionally) CUDA
graphs.  A step never allocates or synchronises, so it can be captured by ``torch.cuda.graph``.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .maps import load_map
from .params import beam_tables, default_params, params_vector, theta_tables

RK4, EULER = 1, 2   # Integrator enum values (base_classes.py:40-42)

_OUT_SPECS = {
    # name: (shape fn, dtype)
    'obs': (lambda N, A, B: (N, B + 8), torch.float32),
    'reward': (lambda N, A, B: (N,), torch.float32),
    'terminated': (lambda N, A, B: (N,), torch.uint8),
    'scans_f64': (lambda N, A, B: (N, A, B), torch.float64),
    'scans_f32': (lambda N, A, B: (N, A, B), torch.float32),
    'state': (lambda N, A, B: (N, A, 7), torch.float64),
    'collisions': (lambda N, A, B: (N, A), torch.uint8),
    'toggles': (lambda N, A, B: (N, A), torch.int32),
    'lap_times': (lambda N, A, B: (N, A), torch.float64),
    'lap_counts': (lambda N, A, B: (N, A), torch.float64),
    'time': (lambda N, A, B: (N,), torch.float64),
    'agent_poses': (lambda N, A, B: (N, A, 3), torch.float64),
}
ALL_OUTPUTS = tuple(_OUT_SPECS)
FAST_OUTPUTS = ('obs', 'reward', 'terminated')


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class HostBlocks(object):
    """The pinned buffers of BatchSim.host_blocks (plain attribute bag)."""


class BatchSim(object):
    """Device-resident batch of F110 simulations (the native backend of Simulator + F110Env.step)."""

    def __init__(self, num_envs, num_agents=2, params=None, seed=42, timestep=0.01, integrator=RK4, ego_idx=0,
                 lidar_dist=0.0, num_beams=1080, fov=4.7, theta_dis=2000, eps=1e-4, max_range=30.0,
                 ttc_thresh=0.005, noise_std=0.01, device=None, outputs=ALL_OUTPUTS, count_lookups=False,
                 host_stream_rank=0, narrow_fraction=False):
        if not torch.cuda.is_available():
            raise RuntimeError("f110_gymnasium_ros2_jazzy_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device('cuda', torch.cuda.current_device() if device is None else
                                   (device if isinstance(device, int) else torch.device(device).index or 0))
        self.N, self.A, self.B = int(num_envs), int(num_agents), int(num_beams)
        self.params = dict(default_params() if params is None else params)
        self.timestep = float(timestep)
        self.theta_dis = int(theta_dis)
        integ = getattr(integrator, 'value', integrator)
        cfg = _lib.F110Config(abi_version=_lib.F110_ABI_VERSION, device=self.device.index, num_envs=self.N,
                              num_agents=self.A, num_beams=self.B, theta_dis=theta_dis, integrator=int(integ),
                              ego_idx=int(ego_idx), flags=(_lib.F110_FLAG_COUNT_LOOKUPS if count_lookups else 0) |
                              (_lib.F110_FLAG_NARROW_FRACTION if narrow_fraction else 0),   # narrow_fraction: test hook
                              host_stream_rank=int(host_stream_rank),
                              fov=fov, eps=eps, max_range=max_range, timestep=timestep, lidar_dist=lidar_dist,
                              ttc_thresh=ttc_thresh, lidar_max=float(self.params.get('lidar_max', 30.0)),
                              noise_std=noise_std, seed=int(seed) & 0xFFFFFFFFFFFFFFFF)
        pv = params_vector(self.params)
        h = C.c_void_p()
        _lib.check(self.lib.f110_create(C.byref(cfg), pv.ctypes.data_as(C.c_void_p), C.byref(h)))
        self.h = h
        # host-side tables, numpy-evaluated like the reference
        s, c = theta_tables(theta_dis)
        self.set_tables(s, c)
        self.set_beam_tables(*beam_tables(self.params, self.B, fov))
        with torch.cuda.device(self.device):
            self.out = {k: torch.zeros(_OUT_SPECS[k][0](self.N, self.A, self.B), dtype=_OUT_SPECS[k][1], device=self.device)
                        for k in outputs}
        self._keep = []   # tensors referenced by the last enqueued step

    # ------------------------------------------------------------------ setup (host pointers)
    def close(self):
        if getattr(self, 'h', None):
            self.lib.f110_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_tables(self, sines, cosines):
        s = np.ascontiguousarray(sines, np.float64)
        c = np.ascontiguousarray(cosines, np.float64)
        if not (s.size == c.size == self.theta_dis):
            raise ValueError("sin/cos tables must have theta_dis = %d entries" % self.theta_dis)
        _lib.check(self.lib.f110_set_tables(self.h, s.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p)))

    def set_beam_tables(self, scan_angles, cosines, side_distances):
        a, c, s = (np.ascontiguousarray(v, np.float64) for v in (scan_angles, cosines, side_distances))
        if not (a.size == c.size == s.size == self.B):
            raise ValueError("beam tables must have num_beams = %d entries" % self.B)
        _lib.check(self.lib.f110_set_beam_tables(self.h, a.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p),
                                                 s.ctypes.data_as(C.c_void_p)))

    def set_map_arrays(self, dt, resolution, origin):
        """One map from its distance transform (any dtype, converted to float64): the set of one."""
        self.set_maps([(np.asarray(dt, np.float64), resolution, origin)])

    def set_map_image(self, free_mask, resolution, origin):
        """Map from the binarised image (non-zero = free, row 0 = bottom row): the EDT runs on the device
        (f110_set_map_image) and reproduces resolution * scipy.ndimage.distance_transform_edt(img) bit for bit."""
        self.set_maps([(np.asarray(free_mask) != 0, resolution, origin)])

    def edt_kernel_ms(self):
        """Device time of the EDT kernels of the last set_map_image call (CUDA events)."""
        return float(self.lib.f110_edt_kernel_ms(self.h))

    def get_map(self, slot=0):
        """The fp64 map of `slot` (0 for a single map) as the device holds it."""
        dt = np.empty(self.map_shapes[slot], np.float64)
        _lib.check(self.lib.f110_get_map_slot(self.h, int(slot), dt.ctypes.data_as(C.c_void_p), dt.size))
        return dt

    @property
    def num_maps(self):
        """Maps installed: 1 for a single map, K after set_maps with K maps, 0 before any."""
        return int(self.lib.f110_map_count(self.h))

    def set_maps(self, specs, edt='host', map_ext='.png'):
        """Installs a map set (f110_set_maps): env e then drives on map floor(e * K / N) until set_env_maps says otherwise.
        Each spec is a yaml path (loaded like set_map: scipy's EDT on the host, or the device EDT with edt='device'), a
        (dt float64 [H, W], resolution, origin) tuple, or a (free_mask bool / uint8 [H, W], resolution, origin) tuple (device
        EDT).  ShapedReward(centerlines=[...]) with one centerline per map scores each env on the line of its slot.
        Every other map setter installs the set of one map through here."""
        from .maps import load_map_image
        descs, keep, shapes = (_lib.F110MapDesc * len(specs))(), [], []
        for k, spec in enumerate(specs):
            if isinstance(spec, (str, bytes)) or hasattr(spec, '__fspath__'):
                spec = load_map_image(spec, map_ext) if edt == 'device' else load_map(spec, map_ext)
                if edt == 'device':
                    spec = (spec[0].astype(bool),) + tuple(spec[1:])
            arr, res, origin = spec
            arr = np.asarray(arr)
            d = descs[k]
            if arr.dtype == np.float64:
                a = np.ascontiguousarray(arr)
                d.dt = a.ctypes.data
            elif arr.dtype in (np.bool_, np.uint8):
                # numpy stores a bool as one byte 0 / 1: a bool mask goes to the library as it is, without another pass
                a = np.ascontiguousarray(arr if arr.dtype == np.bool_ else arr != 0).view(np.uint8)
                d.free_mask = a.ctypes.data
            else:
                raise ValueError("map %d: a distance transform must be float64, a free mask bool or uint8 (got %s)" % (k, arr.dtype))
            keep.append(a)
            d.height, d.width = a.shape
            # orig_s / orig_c are numpy-evaluated on the host like laser_models.py:421-422
            d.resolution, d.orig_x, d.orig_y = float(res), float(origin[0]), float(origin[1])
            d.orig_cos, d.orig_sin = float(np.cos(origin[2])), float(np.sin(origin[2]))
            shapes.append(a.shape)
        _lib.check(self.lib.f110_set_maps(self.h, descs, len(specs)))
        self.map_shapes = shapes

    def set_env_maps(self, slots, env_mask=None):
        """Each (masked) env's map slot.  numpy / list input: validated on the host first -- a slot outside
        [0, num_maps) raises IndexError and changes nothing.  CUDA tensors: stream-ordered on the current stream (capturable;
        entries out of range leave that env's slot unchanged).  A slot change is not a reset: see F110VecEnv.reassign."""
        if torch.is_tensor(slots) and slots.is_cuda:
            sl = slots.to(device=self.device, dtype=torch.int32).contiguous()
            m = None if env_mask is None else env_mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if sl.numel() != self.N or (m is not None and m.numel() != self.N):
                raise ValueError("slots and env_mask need %d entries" % self.N)
            self._keep_slots = (sl, m)
            _lib.check(self.lib.f110_set_env_maps(self.h, _ptr(sl), _ptr(m), self._stream()))
            return
        sl = np.ascontiguousarray(np.asarray(slots.cpu() if torch.is_tensor(slots) else slots), np.int32).reshape(-1)
        m = None
        if env_mask is not None:
            m = np.ascontiguousarray(np.asarray(env_mask.cpu() if torch.is_tensor(env_mask) else env_mask) != 0, np.uint8).reshape(-1)
        if sl.size != self.N or (m is not None and m.size != self.N):
            raise ValueError("slots and env_mask need %d entries" % self.N)
        _lib.check(self.lib.f110_set_env_maps_host(self.h, sl.ctypes.data_as(C.c_void_p),
                                                   None if m is None else m.ctypes.data_as(C.c_void_p)))

    def env_maps(self, out=None):
        """Device int32 [N]: each env's map slot (all 0 for a single map), valid in stream order.  ``out``: a contiguous
        device int32 [N] tensor to write instead of a new one (one stream-ordered copy, capturable into a CUDA graph)."""
        if out is None:
            out = torch.empty(self.N, dtype=torch.int32, device=self.device)
        elif not (out.is_cuda and out.dtype == torch.int32 and out.is_contiguous() and out.numel() == self.N):
            raise ValueError("env_maps(out=...) needs a contiguous CUDA int32 tensor of %d entries" % self.N)
        _lib.check(self.lib.f110_get_env_maps(self.h, _ptr(out), self._stream()))
        return out

    def set_map(self, map_path, map_ext, edt='host'):
        """edt='host': scipy on the host, as the reference; edt='device': the device EDT, as set_map_image."""
        self.set_maps([map_path], edt=edt, map_ext=map_ext)

    def update_params(self, params, agent_idx=-1):
        pv = params_vector(params)
        _lib.check(self.lib.f110_set_params(self.h, pv.ctypes.data_as(C.c_void_p), int(agent_idx)))

    # ------------------------------------------------------------------ step path (device pointers)
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, x, dtype, shape):
        if x is None:
            return None
        if not torch.is_tensor(x):
            x = torch.as_tensor(np.ascontiguousarray(x), dtype=dtype)
        x = x.to(device=self.device, dtype=dtype, non_blocking=True).contiguous()
        if x.numel() != int(np.prod(shape)):
            raise ValueError("expected %s elements, got %s" % (shape, tuple(x.shape)))
        return x

    def sim_reset(self, poses, env_mask=None):
        """Simulator.reset (base_classes.py:627-643): set poses, do not step.  poses [N, A, 3] (or [A, 3] if N == 1)."""
        p = poses if torch.is_tensor(poses) else np.asarray(poses, np.float64)
        if p.ndim == 2:
            p = p[None]
        num_poses = p.shape[1]
        if num_poses != self.A:
            _lib.check(self.lib.f110_sim_reset(self.h, C.c_void_p(8), num_poses, None, self._stream()))
        p = self._dev(p, torch.float64, (self.N, self.A, 3))
        m = self._dev(env_mask, torch.uint8, (self.N,))
        self._keep = [p, m]
        _lib.check(self.lib.f110_sim_reset(self.h, _ptr(p), num_poses, _ptr(m), self._stream()))

    def step(self, actions=None, noise=None, reset_mask=None, reset_poses=None, active_mask=None):
        """One batched F110Env.step.  Returns self.out (dict of persistent CUDA tensors, valid in stream order)."""
        N, A, B = self.N, self.A, self.B
        act = None
        f64 = 0
        if actions is not None:
            if torch.is_tensor(actions):
                f64 = int(actions.dtype == torch.float64)
                act = self._dev(actions, torch.float64 if f64 else torch.float32, (N, A, 2))
            else:
                a = np.asarray(actions)
                f64 = int(a.dtype == np.float64)
                act = self._dev(a, torch.float64 if f64 else torch.float32, (N, A, 2))
        nz = self._dev(noise, torch.float64, (N, A, B))
        rm = self._dev(reset_mask, torch.uint8, (N,))
        rp = self._dev(reset_poses, torch.float64, (N, A, 3))
        am = self._dev(active_mask, torch.uint8, (N,))
        o = self.out
        io = _lib.F110StepIO(actions=_ptr(act), actions_f64=f64, noise=_ptr(nz), reset_mask=_ptr(rm), reset_poses=_ptr(rp),
                             active_mask=_ptr(am), **{k: _ptr(o[k]) for k in o})
        self._keep = [act, nz, rm, rp, am]
        _lib.check(self.lib.f110_step(self.h, C.byref(io), self._stream()))
        return o

    def reset(self, poses, noise=None, env_mask=None):
        """F110Env.reset for the masked envs (all when env_mask is None): reset + the zero-action step."""
        p = poses if torch.is_tensor(poses) else np.asarray(poses, np.float64)
        if p.ndim == 2:
            p = p[None]
        if p.shape[1] != self.A:
            raise ValueError('Number of poses for reset does not match number of agents.')
        if env_mask is None:
            mask = torch.ones(self.N, dtype=torch.uint8, device=self.device)
            return self.step(None, noise, mask, p, None)
        return self.step(None, noise, env_mask, p, env_mask)

    def step_host(self, actions=None, noise=None, reset_mask=None, reset_poses=None, out=None, sync=True):
        """Host-buffer entry (f110_step_host): numpy in, numpy out, copies inside the call.  With sync=False the
        call only enqueues (f110_step_host_async); the buffers are valid after host_sync()."""
        N, A, B = self.N, self.A, self.B
        if out is None:
            out = self.host_out()
        f64 = 0
        act = None
        if actions is not None:
            act = np.ascontiguousarray(actions)
            if act.dtype not in (np.float32, np.float64):
                act = act.astype(np.float64)
            f64 = int(act.dtype == np.float64)
            assert act.size == N * A * 2
        nz = None if noise is None else np.ascontiguousarray(noise, np.float64)
        rm = None if reset_mask is None else np.ascontiguousarray(reset_mask, np.uint8)
        rp = None if reset_poses is None else np.ascontiguousarray(reset_poses, np.float64)

        def hp(a):
            if a is None:
                return None
            return C.c_void_p(a.data_ptr()) if torch.is_tensor(a) else a.ctypes.data_as(C.c_void_p)
        io = _lib.F110StepIO(actions=hp(act), actions_f64=f64, noise=hp(nz), reset_mask=hp(rm), reset_poses=hp(rp),
                             active_mask=None, **{k: hp(out[k]) for k in out})
        self._keep_host = (act, nz, rm, rp, out)   # the async copies read / write these after we return
        if sync:
            _lib.check(self.lib.f110_step_host(self.h, C.byref(io)))
        else:
            _lib.check(self.lib.f110_step_host_async(self.h, C.byref(io)))
        return out

    # merge order of f110_step_host_async (include/f110_b200.h)
    _IN_ORDER = ('actions', 'reset_poses', 'noise', 'reset_mask')
    _OUT_ORDER = ('scans_f64', 'state', 'agent_poses', 'lap_times', 'lap_counts', 'time', 'obs', 'scans_f32', 'reward', 'toggles',
                  'terminated', 'collisions')

    def host_blocks(self, outputs=ALL_OUTPUTS, actions_dtype=np.float32, noise=True):
        """Pinned host buffers for step_host_blocks: one allocation per direction, the fields back to back in the
        library's merge order, so that a step moves them with ONE copy each way (F110_HOST_MERGE_ADJACENT).
        -> HostBlocks with numpy views .actions [N,A,2], .reset_poses [N,A,3], .noise [N,A,B] (or None),
        .reset_mask [N] and the dict .out of output views."""
        N, A, B = self.N, self.A, self.B
        adt = np.dtype(actions_dtype)
        hb = HostBlocks()
        in_specs = {'actions': ((N, A, 2), adt), 'reset_poses': ((N, A, 3), np.dtype(np.float64)),
                    'noise': ((N, A, B), np.dtype(np.float64)), 'reset_mask': ((N,), np.dtype(np.uint8))}
        keys = [k for k in self._IN_ORDER if noise or k != 'noise']
        nbytes = [int(np.prod(in_specs[k][0])) * in_specs[k][1].itemsize for k in keys]
        hb._in = torch.zeros(sum(nbytes), dtype=torch.uint8, pin_memory=True)
        raw, off = hb._in.numpy(), 0
        hb.noise = None
        for k, nb in zip(keys, nbytes):
            setattr(hb, k, raw[off:off + nb].view(in_specs[k][1]).reshape(in_specs[k][0]))
            off += nb
        okeys = [k for k in self._OUT_ORDER if k in outputs]
        onb = [int(np.prod(_OUT_SPECS[k][0](N, A, B))) * torch.zeros(0, dtype=_OUT_SPECS[k][1]).element_size() for k in okeys]
        hb._out = torch.zeros(sum(onb), dtype=torch.uint8, pin_memory=True)
        hb.out, off = {}, 0
        for k, nb in zip(okeys, onb):
            hb.out[k] = hb._out[off:off + nb].view(_OUT_SPECS[k][1]).view(_OUT_SPECS[k][0](N, A, B))
            off += nb
        hb.np = {k: v.numpy() for k, v in hb.out.items()}
        hb.io = _lib.F110StepIO(actions=C.c_void_p(hb.actions.ctypes.data), actions_f64=int(adt == np.float64),
                                host_flags=_lib.F110_HOST_MERGE_ADJACENT,
                                noise=None if hb.noise is None else C.c_void_p(hb.noise.ctypes.data),
                                reset_mask=C.c_void_p(hb.reset_mask.ctypes.data),
                                reset_poses=C.c_void_p(hb.reset_poses.ctypes.data), active_mask=None,
                                **{k: C.c_void_p(v.data_ptr()) for k, v in hb.out.items()})
        return hb

    def step_host_blocks(self, hb, sync=True):
        """One step on the buffers of host_blocks(): the caller has filled hb.actions / hb.noise / hb.reset_mask
        (non-zero: that env is reset to hb.reset_poses and its action ignored)."""
        if sync:
            _lib.check(self.lib.f110_step_host(self.h, C.byref(hb.io)))
        else:
            _lib.check(self.lib.f110_step_host_async(self.h, C.byref(hb.io)))
        return hb.np

    def host_sync(self):
        _lib.check(self.lib.f110_host_sync(self.h))

    def host_out(self, outputs=None, pinned=True):
        """Pinned host tensors shaped like the outputs, for step_host."""
        keys = outputs if outputs is not None else tuple(self.out)
        return {k: torch.zeros(_OUT_SPECS[k][0](self.N, self.A, self.B), dtype=_OUT_SPECS[k][1],
                               pin_memory=pinned) for k in keys}

    # ------------------------------------------------------------------ checkpoint / stats
    @property
    def map_generation(self):
        """Incremented by every map change; F110VecEnv compares it to know that a captured CUDA graph is stale."""
        return int(self.lib.f110_map_generation(self.h))

    def state_dict(self):
        """The library's checkpoint blob: a versioned header (layout, N, A, B) + the whole persistent state arena."""
        n = int(self.lib.f110_state_nbytes(self.h))
        blob = torch.empty(n, dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.f110_get_state(self.h, _ptr(blob), self._stream()))
        return {'blob': blob, 'N': self.N, 'A': self.A, 'B': self.B}

    def load_state_dict(self, sd):
        if (sd['N'], sd['A'], sd['B']) != (self.N, self.A, self.B):
            raise ValueError("checkpoint shape mismatch")
        blob = sd['blob'].to(self.device).contiguous()
        if blob.numel() != int(self.lib.f110_state_nbytes(self.h)):
            raise ValueError("checkpoint size mismatch")
        self._keep = [blob]
        _lib.check(self.lib.f110_set_state(self.h, _ptr(blob), self._stream()))

    def stats(self, reset=False):
        """Device tensor of F110_NUM_STATS episode counters (sum-reducible across ranks)."""
        t = torch.zeros(_lib.F110_NUM_STATS, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.f110_get_stats(self.h, _ptr(t), int(reset), self._stream()))
        return t

    def lookup_count(self):
        a, b = C.c_uint64(0), C.c_uint64(0)
        _lib.check(self.lib.f110_get_lookup_count(self.h, C.byref(a), C.byref(b)))
        self.max_lookups = int(self.lib.f110_max_lookups(self.h))
        self.redone_rays = int(self.lib.f110_redone_rays(self.h))
        return a.value, b.value

    def lidar_variant(self):
        """The lidar kernel variant the last step ran (f110_get_lidar_variant): dict with fraction_bits, template_fb (0 =
        generic), mode (0..3) and maps (a map set's kernel)."""
        v = np.zeros(4, np.int32)
        _lib.check(self.lib.f110_get_lidar_variant(self.h, v.ctypes.data_as(C.c_void_p)))
        return dict(zip(('fraction_bits', 'template_fb', 'mode', 'maps'), (int(x) for x in v)))

    @property
    def kernel_launches(self):
        return int(self.lib.f110_kernel_launches(self.h))
