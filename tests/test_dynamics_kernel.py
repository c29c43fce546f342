"""The dynamics kernel (K1: dynamics_kernel, dynamics_maps_kernel and sim_reset_kernel in f110_kernels.cu) held to the model
of test_dynamics_model.py bit for bit.

The model is pinned to the oracle bit for bit when it takes glibc's trig.  Here it takes the device's: f110_trig_probe runs
K1's own sincos / tan / cos calls, compiled in the same nvcc command as K1.  Everything else in K1 is IEEE arithmetic in the
reference's order without contraction, so state and steering FIFO must then equal K1's exactly, and the only difference
between K1 and the oracle is the device's trig.  The tests print how often the device's trig differs from glibc's and by how
many ulp, and check that the glibc-trig model does miss K1 somewhere in the rollouts: that difference must be exercised.

Every handle runs with an iTTC threshold of 0, so the post kernel never zeroes a state: a step's `state` output is K1's
result.  State and FIFO are read back from (and written into) the checkpoint blob, whose layout is parsed below.
"""
import ctypes as C

import numpy as np
import pytest

from tests import helpers as H
from tests.test_dynamics_model import (AGENT1_PARAMS, DEFAULT_PARAMS, EULER, LIBM, PARAM_SETS, REVERSE_PARAMS, RK4,
                                       TIMESTEPS, VSWITCH_PARAMS, check_expectations, dynamics_step, edge_cases,
                                       params_matrix, random_cars, same, sim_reset, stack_edges)

pytestmark = pytest.mark.gpu

CKPT_MAGIC, CKPT_LAYOUT = 0x30313146, 2


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


class DeviceTrig(object):
    """K1's trig from f110_trig_probe.  Counts the values that differ from glibc's and the largest difference in ulp."""

    def __init__(self):
        from f110_gymnasium_ros2_jazzy_b200 import _lib
        self.torch, self._lib = _torch(), _lib
        self.lib = _lib.load()
        self.evals = self.differ = 0
        self.max_ulp = 0.0

    def _probe(self, x):
        torch = self.torch
        x = np.ascontiguousarray(x, np.float64).reshape(-1)
        if x.size == 0:
            return np.empty((4, 0))
        xd = torch.from_numpy(x).cuda()
        out = torch.empty(4 * x.size, dtype=torch.float64, device=xd.device)
        self._lib.check(self.lib.f110_trig_probe(C.c_void_p(xd.data_ptr()), x.size, C.c_void_p(out.data_ptr()),
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return out.cpu().numpy().reshape(4, x.size)

    def _count(self, dev, ref):
        d = ~same(dev, ref)
        self.evals += dev.size
        self.differ += int(d.sum())
        fin = d & np.isfinite(dev) & np.isfinite(ref)
        if fin.any():
            self.max_ulp = max(self.max_ulp, float((np.abs(dev[fin] - ref[fin]) / np.spacing(np.abs(ref[fin]))).max()))

    def sincos(self, x):
        o = self._probe(x)
        s, c = LIBM.sincos(x)
        self._count(o[0], s)
        self._count(o[1], c)
        return o[0], o[1]

    def tan(self, x):
        o = self._probe(x)
        self._count(o[2], LIBM.tan(x))
        return o[2]

    def cos(self, x):
        o = self._probe(x)
        self._count(o[3], LIBM.cos(x))
        return o[3]

    def summary(self):
        return 'device trig: %d of %d values differ from glibc, by at most %.3g ulp' % (self.differ, self.evals, self.max_ulp)


# ---------------------------------------------------------------------------------------------------------- checkpoint

def blob_layout(N, A):
    """name -> (byte offset in the blob, dtype, count): a 64-byte header, then layout_state's arena (f110_capi.cu), every
    array at a 256-byte-aligned offset of the arena."""
    NA, off, out = N * A, 0, {}
    arrays = [('x%d' % k, np.float64, NA) for k in range(7)] + [
        (k, np.float64, NA) for k in ('steer_buf0', 'steer_buf1', 'start_x', 'start_y', 'start_th', 'lap_times', 'lap_counts')] + [
        (k, np.float64, N) for k in ('time', 'rot_c', 'rot_s')] + [
        ('steer_cnt', np.int32, NA), ('toggles', np.int32, NA), ('step_count', np.uint32, N),
        ('near_start', np.uint8, NA), ('collisions', np.uint8, NA)]
    for name, dt, n in arrays:
        off = (off + 255) & ~255
        out[name] = (64 + off, np.dtype(dt), n)
        off += n * np.dtype(dt).itemsize
    return out


class Blob(object):
    """The checkpoint blob of a handle on the host: state x [NA, 7], FIFO b0, b1, cnt [NA]."""

    def __init__(self, sim):
        self.sim = sim
        sd = sim.state_dict()
        self.raw = sd['blob'].cpu().numpy().copy()
        hdr = self.raw[:64].view(np.uint32)
        assert hdr[0] == CKPT_MAGIC and hdr[1] == CKPT_LAYOUT, 'checkpoint layout %d: the parser reads layout %d' % (
            hdr[1], CKPT_LAYOUT)
        assert tuple(self.raw[8:20].view(np.int32)) == (sim.N, sim.A, sim.B)
        self.layout = blob_layout(sim.N, sim.A)
        last = max(o + d.itemsize * n for o, d, n in self.layout.values())
        assert last <= self.raw.size == 64 + int(self.raw[24:32].view(np.uint64)[0])

    def get(self, name):
        o, d, n = self.layout[name]
        return self.raw[o:o + n * d.itemsize].view(d)

    def set(self, name, v):
        self.get(name)[:] = np.asarray(v).astype(self.layout[name][1])

    @property
    def x(self):
        return np.stack([self.get('x%d' % k) for k in range(7)], 1)

    @x.setter
    def x(self, v):
        for k in range(7):
            self.set('x%d' % k, v[:, k])

    def fifo(self):
        return self.get('steer_buf0').copy(), self.get('steer_buf1').copy(), self.get('steer_cnt').copy()

    def load(self):
        torch = _torch()
        sim = self.sim
        sim.load_state_dict({'blob': torch.from_numpy(self.raw.copy()).to(sim.device), 'N': sim.N, 'A': sim.A, 'B': sim.B})


def _sim(N, A, params=None, maps=('open_square',), **kw):
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    sim = BatchSim(N, A, outputs=ALL_OUTPUTS, noise_std=0.0, ttc_thresh=0.0, **kw)
    if len(maps) == 1:
        sim.set_map_arrays(*H.golden_map(maps[0]))
    else:
        sim.set_maps([H.golden_map(m) for m in maps])
    for a, p in enumerate(params or []):
        if p is not DEFAULT_PARAMS:
            sim.update_params(p, a)
    return sim


def _state(sim):
    torch = _torch()
    torch.cuda.synchronize()
    return sim.out['state'].cpu().numpy().reshape(-1, 7).copy()


def _start_poses(rng, N, A):
    return np.concatenate([rng.uniform(-5, 5, (N, A, 2)), rng.uniform(-np.pi, np.pi, (N, A, 1))], 2)


def _assert_cars(got, want, what):
    ok = same(got, want)
    ok = ok.all(1) if ok.ndim == 2 else ok
    bad = np.flatnonzero(~ok)
    assert bad.size == 0, (what, 'cars differ:', bad.size, bad[:6], got[bad[:2]], want[bad[:2]])


# ---------------------------------------------------------------------------------------------------------- a. edges

EDGE_AGENTS = ('default', 'reverse', 'vswitch', 'agent1')
EDGE_ENVS = 97          # 4 x 97 = 388 cars: four CTAs of 128 threads, the last one partly filled


@pytest.mark.parametrize('f64', [True, False], ids=['f64', 'f32'])
@pytest.mark.parametrize('integrator', [RK4, EULER], ids=['rk4', 'euler'])
@pytest.mark.parametrize('dt', TIMESTEPS)
def test_constructed_states_one_step(dt, integrator, f64):
    """The edge list of test_dynamics_model.py, one car per entry, injected through the checkpoint blob next to random
    cars, then one step: state and FIFO bit for bit."""
    N, A = EDGE_ENVS, len(EDGE_AGENTS)
    NA = N * A
    rng = np.random.default_rng(int(dt * 1e4) + 10 * integrator + int(f64))
    sets = [PARAM_SETS[k] for k in EDGE_AGENTS]
    sim = _sim(N, A, params=sets, timestep=dt, integrator=integrator)
    pv = params_matrix(sets * N, NA)
    # random cars everywhere, then the edge entries, each in the next free env of its parameter set's agent column
    x, b0, b1, cnt, rs, sp = (np.empty((NA, 7)), np.empty(NA), np.empty(NA), np.empty(NA, np.int32), np.empty(NA),
                              np.empty(NA))
    for a, p in enumerate(sets):
        x[a::A], b0[a::A], b1[a::A], cnt[a::A], rs[a::A], sp[a::A] = random_cars(rng, N, p)
    cases = edge_cases(dt)
    ex, eb0, eb1, ecnt, ers, esp, _ = stack_edges(cases)
    slots, used = [], [0] * A
    for c in cases:
        a = EDGE_AGENTS.index(c['params'])
        slots.append(used[a] * A + a)
        used[a] += 1
    assert max(used) <= N
    slots = np.array(slots)
    x[slots], b0[slots], b1[slots], cnt[slots], rs[slots], sp[slots] = ex, eb0, eb1, ecnt, ers, esp
    act = np.stack([rs, sp], 1).reshape(N, A, 2).astype(np.float64 if f64 else np.float32)
    # a reset step, then the parser checks itself against the state output before anything is injected
    sim.reset(_start_poses(rng, N, A))
    st = _state(sim)
    blob = Blob(sim)
    assert np.array_equal(blob.x.view(np.int64), st.view(np.int64))
    assert (blob.get('steer_cnt') == 1).all() and not blob.get('steer_buf0').any() and not blob.get('steer_buf1').any()
    blob.x = x
    blob.set('steer_buf0', b0); blob.set('steer_buf1', b1); blob.set('steer_cnt', cnt)
    blob.load()
    sim.step(act)
    got = _state(sim)
    after = Blob(sim)
    trig = DeviceTrig()
    wx, wb0, wb1, wcnt, tr = dynamics_step(x, b0, b1, cnt, act[..., 0].reshape(-1), act[..., 1].reshape(-1), pv, dt,
                                           integrator, trig)
    _assert_cars(got, wx, 'state')
    _assert_cars(after.x, wx, 'blob state')
    gb0, gb1, gcnt = after.fifo()
    _assert_cars(gb0, wb0, 'steer_buf0')
    _assert_cars(gb1, wb1, 'steer_buf1')
    assert np.array_equal(gcnt, wcnt)
    if f64:
        check_expectations(cases, {k: (v[:, slots] if k == 'kin' else v[slots]) for k, v in tr.items()}, integrator)
    print(len(cases), 'edge cases,', NA, 'cars;', trig.summary())


# ---------------------------------------------------------------------------------------------------------- b, c. replay

def replay(sim, steps, params, integrator, rng, f64=False, reset_rate=0.0, hole_rate=0.0, sim_reset_at=None, map_set=False):
    """Step a handle with random actions and check every car at every step against the model run on the previous step's
    GPU state and the model's own FIFO (the FIFO is checked against the blob too).  -> (DeviceTrig, steps on which the
    glibc-trig model missed K1)."""
    N, A = sim.N, sim.A
    NA = N * A
    pv = params_matrix(list(params) * N, NA)
    trig = DeviceTrig()
    poses = _start_poses(rng, N, A)
    sim.reset(poses)
    x = _state(sim)
    b0, b1, cnt = np.zeros(NA), np.zeros(NA), np.ones(NA, np.int32)
    libm_missed = 0
    for t in range(steps):
        if t == sim_reset_at:
            mask = (rng.random(N) < 0.5).astype(np.uint8)
            mask[0] = 1
            p2 = _start_poses(rng, N, A)
            sim.sim_reset(p2, env_mask=mask)
            x, b0, b1, cnt = sim_reset(x, b0, b1, cnt, p2.reshape(-1, 3), np.repeat(mask, A))
            bl = Blob(sim)
            _assert_cars(bl.x, x, ('sim_reset', t))
            _assert_cars(np.stack(bl.fifo()[:2], 1), np.stack([b0, b1], 1), ('sim_reset fifo', t))
            assert np.array_equal(bl.get('steer_cnt'), cnt)
        steer = rng.uniform(-0.5, 0.5, (N, A))
        speed = np.where(rng.random((N, A)) < 0.3, rng.uniform(-1.0, 1.0, (N, A)), rng.uniform(-3.0, 9.0, (N, A)))
        act = np.stack([steer, speed], 2).astype(np.float64 if f64 else np.float32)
        rm = (rng.random(N) < reset_rate).astype(np.uint8) if reset_rate else None
        am = (rng.random(N) >= hole_rate).astype(np.uint8) if hole_rate and t > 2 else None
        rp = _start_poses(rng, N, A) if rm is not None else None
        sim.step(act, reset_mask=rm, reset_poses=rp, active_mask=am)
        got = _state(sim)
        bl = Blob(sim)
        kw = dict(reset=None if rm is None else np.repeat(rm, A), poses=None if rp is None else rp.reshape(-1, 3),
                  active=None if am is None else np.repeat(am, A))
        args = (x, b0, b1, cnt, act[..., 0].reshape(-1), act[..., 1].reshape(-1), pv, sim.timestep, integrator)
        wx, b0, b1, cnt, _ = dynamics_step(*args, trig=trig, **kw)
        lx = dynamics_step(*args, trig=LIBM, **kw)[0]
        libm_missed += int(not same(lx, bl.x).all())
        _assert_cars(bl.x, wx, ('blob state', t))
        on = np.ones(NA, bool) if am is None else np.repeat(am, A) != 0
        _assert_cars(got[on], wx[on], ('state', t))
        gb0, gb1, gcnt = bl.fifo()
        _assert_cars(np.stack([gb0, gb1], 1), np.stack([b0, b1], 1), ('fifo', t))
        assert np.array_equal(gcnt, cnt), t
        x = bl.x
    if map_set:
        assert sim.lidar_variant()['maps'] == 1     # dynamics_maps_kernel ran
    return trig, libm_missed


REPLAYS = {
    # A: (handle keywords, per-agent parameters, f64 actions, sim_reset step, map set)
    1: (dict(timestep=0.01, integrator=RK4), [DEFAULT_PARAMS], False, None, False),
    2: (dict(timestep=0.005, integrator=EULER, ego_idx=1), [DEFAULT_PARAMS, AGENT1_PARAMS], True, 150, True),
    3: (dict(timestep=0.02, integrator=RK4, ego_idx=1), [REVERSE_PARAMS, AGENT1_PARAMS, PARAM_SETS['agent2']], False, 120,
        False),
    4: (dict(timestep=0.01, integrator=RK4), [DEFAULT_PARAMS, REVERSE_PARAMS, PARAM_SETS['test'], VSWITCH_PARAMS], True,
        90, True),
}


@pytest.mark.parametrize('A', sorted(REPLAYS))
def test_rollout_replay(A):
    """250 steps with random actions, reset steps, inactive envs, a masked Simulator.reset, per-agent parameters, Euler,
    ego_idx 1 and a map set (dynamics_maps_kernel): every car bit for bit at every step.  (The rollouts step at 5 ms and
    more: at 1 ms a one-ulp trig difference times dt falls below an ulp of the state, and the glibc-trig control matched K1
    on all 250 steps; that timestep is held by the constructed states.)"""
    kw, params, f64, sr, maps = REPLAYS[A]
    N = 61 if A < 3 else 37
    sim = _sim(N, A, params=params, maps=('open_square', 'straight_corridor') if maps else ('open_square',), **kw)
    rng = np.random.default_rng(100 + A)
    trig, missed = replay(sim, 250, params, kw['integrator'], rng, f64=f64, reset_rate=0.03, hole_rate=0.1, sim_reset_at=sr, map_set=maps)
    print('A = %d: %s; the glibc-trig model missed K1 on %d of 250 steps' % (A, trig.summary(), missed))
    assert trig.differ > 0 and missed > 0


@pytest.mark.parametrize('N,A', [(4096, 1), (8192, 2)])
def test_launch_sizes(N, A):
    """20 steps at the C3 shape (4096 x 1) and at 8192 x 2, every car bit for bit."""
    sim = _sim(N, A, timestep=0.01, integrator=RK4)
    trig, missed = replay(sim, 20, [DEFAULT_PARAMS] * A, RK4, np.random.default_rng(N + A))
    print('%d x %d: %s; the glibc-trig model missed K1 on %d of 20 steps' % (N, A, trig.summary(), missed))


# ---------------------------------------------------------------------------------------------------------- d. lidar offset

@pytest.mark.parametrize('lidar_dist', [0.275, -0.1])
def test_lidar_offset_scan_origin(lidar_dist):
    """K1 puts the scan origin at x + lidar_dist * (cos, sin)(yaw) with the device's sincos.  On the axis-aligned
    open_square map the lidar kernel's march is the oracle's, so scans_f64 must equal Oracle.scan of that origin bit for bit
    (the oracle's own rollout adds the offset with glibc's trig and so cannot be used)."""
    from oracle.f110_oracle import Oracle
    N, steps = 6, 40
    sim = _sim(N, 1, timestep=0.01, integrator=RK4, lidar_dist=lidar_dist)
    o = Oracle(1, 1, ttc_thresh=0.0)
    o.set_map_arrays(*H.golden_map('open_square'))
    trig = DeviceTrig()
    rng = np.random.default_rng(int(abs(lidar_dist) * 1000))
    sim.reset(np.concatenate([rng.uniform(-4, 4, (N, 1, 2)), rng.uniform(-np.pi, np.pi, (N, 1, 1))], 2))
    libm_origin_differs = 0
    for t in range(steps):
        if t:
            act = np.stack([rng.uniform(-0.4, 0.4, (N, 1)), rng.uniform(0.0, 4.0, (N, 1))], 2).astype(np.float32)
            sim.step(act)
        st = _state(sim)
        scans = sim.out['scans_f64'].cpu().numpy().reshape(N, -1)
        s, c = trig.sincos(st[:, 4])
        ox, oy = st[:, 0] + lidar_dist * c, st[:, 1] + lidar_dist * s
        ls, lc = LIBM.sincos(st[:, 4])
        libm_origin_differs += int(((st[:, 0] + lidar_dist * lc) != ox).sum() + ((st[:, 1] + lidar_dist * ls) != oy).sum())
        for e in range(N):
            want = o.scan(np.array([ox[e], oy[e], st[e, 4]]))[0]
            bad = np.flatnonzero(~same(scans[e], want))
            assert bad.size == 0, (t, e, bad[:8], scans[e][bad[:4]], want[bad[:4]])
    print('lidar_dist %g: %s; glibc trig would move %d origin coordinates' % (lidar_dist, trig.summary(),
                                                                           libm_origin_differs))
