"""A numpy restatement of the dynamics kernel (K1: dynamics_body in f110_kernels.cu), pinned to the oracle bit for bit.

K1 is IEEE add / multiply / divide in the reference's operator order, built without contraction, plus three trig calls:
sincos for the heading terms and tan / cos of the steering angle in the kinematic branch.  The model below repeats that
arithmetic on a batch of cars and takes its trig from a callable.  With glibc's trig (through `math`, the libm the oracle
links; numpy's own sin / cos / tan are not glibc's and must not be used) it must equal Oracle.update_pose bit for bit,
which this file checks on random steps of both branches and on a constructed list of branch edges.  With the device's trig
(f110_trig_probe, compiled with the library's flags) it must then equal K1 bit for bit: test_dynamics_kernel.py.

Each entry of the edge list names the branch it is built to reach, and the model's trace of the branches it took is
checked against that, so that an entry cannot quietly miss its purpose.
"""
import math
import types

import numpy as np
import pytest

from oracle.f110_oracle import DEFAULT_PARAMS, PARAM_KEYS, Oracle
from tests.test_oracle_golden import TEST_PARAMS

PI = 3.141592653589793
RK4, EULER = 1, 2
TIMESTEPS = (0.01, 0.02, 0.005, 1e-3)
YAW_RATE_CAP = 10.0
SLIP_CAP = 60 * (PI / 180.0)

# the two per-agent sets of test_gpu_parity.test_per_agent_params_vs_oracle
AGENT1_PARAMS = dict(DEFAULT_PARAMS, m=5.1, I=0.09, lf=0.17, lr=0.19, length=0.9, width=0.5, mu=0.8, a_max=6.0, v_max=12.0,
                     sv_max=2.0)
AGENT2_PARAMS = dict(DEFAULT_PARAMS, length=0.4, width=0.2, C_Sf=5.0, C_Sr=5.5, h=0.05, s_max=0.3, s_min=-0.3)
# a_max * v_switch / v_switch rounds below a_max here (with the defaults it is == a_max), so vel == v_switch taken as above
# the switch caps a clipped acceleration one ulp lower (with a pair that rounds above, such as 7.5 and 5.1, the cap never
# binds).  v_switch < 0.5 puts the tie on the kinematic branch, where x5 = dt * u1 / lwb * tan(x2) carries the ulp into the
# state; at higher speeds x3 + dt * u1 absorbs it.
VSWITCH_PARAMS = dict(DEFAULT_PARAMS, a_max=5.5, v_switch=0.12)
VSWITCH_STEER = (0.1, 0.2, -0.15, 0.3, 0.05, -0.35)     # between them, a steering angle where the tie shows at every dt
# v_min < 0: the car can reverse, and pid can brake (with the default v_min = 1e-8, -v_min < 0 makes every gain push the
# speed up)
REVERSE_PARAMS = dict(DEFAULT_PARAMS, v_min=-5.0)
PARAM_SETS = {'default': DEFAULT_PARAMS, 'test': dict(TEST_PARAMS, lidar_max=30.0), 'agent1': AGENT1_PARAMS,
              'agent2': AGENT2_PARAMS, 'vswitch': VSWITCH_PARAMS, 'reverse': REVERSE_PARAMS}


def params_matrix(params, n):
    """[n, 18] parameter rows from one dict or a list of n dicts."""
    if isinstance(params, dict):
        params = [params] * n
    return np.array([[float(p[k]) for k in PARAM_KEYS] for p in params], np.float64)


# ---------------------------------------------------------------------------------------------------------- trig sources

class LibmTrig(object):
    """glibc's sin / cos / tan through `math` (the libm the oracle links).  A non-finite argument gives NaN, as in C."""

    @staticmethod
    def _map(f, x):
        return np.array([f(v) if math.isfinite(v) else math.nan for v in np.asarray(x, np.float64).tolist()], np.float64)

    def sincos(self, x):
        return self._map(math.sin, x), self._map(math.cos, x)

    def tan(self, x):
        return self._map(math.tan, x)

    def cos(self, x):
        return self._map(math.cos, x)


LIBM = LibmTrig()


# ---------------------------------------------------------------------------------------------------------- the model

def _clip(x, lo, hi):
    """np.clip on scalars: x < lo -> lo, then x > hi -> hi; NaN passes."""
    x = np.where(x < lo, lo, x)
    return np.where(x > hi, hi, x)


def _params(pv):
    return types.SimpleNamespace(**{k: pv[:, i] for i, k in enumerate(PARAM_KEYS)})


def accl_constraints(vel, accl, p, rec=None):
    pos_limit = np.where(vel > p.v_switch, p.a_max * p.v_switch / vel, p.a_max)
    hold = ((vel <= p.v_min) & (accl <= 0)) | ((vel >= p.v_max) & (accl >= 0))
    lo = ~hold & (accl <= -p.a_max)
    hi = ~hold & ~lo & (accl >= pos_limit)
    if rec is not None:
        rec.update(above_switch=vel > p.v_switch, accl_hold=hold, accl_lo=lo, accl_hi=hi)
    return np.where(hold, 0., np.where(lo, -p.a_max, np.where(hi, pos_limit, accl)))


def steering_constraint(sa, sv, p, rec=None):
    hold = ((sa <= p.s_min) & (sv <= 0)) | ((sa >= p.s_max) & (sv >= 0))
    lo = ~hold & (sv <= p.sv_min)
    hi = ~hold & ~lo & (sv >= p.sv_max)
    if rec is not None:
        rec.update(steer_hold=hold, sv_lo=lo, sv_hi=hi)
    return np.where(hold, 0., np.where(lo, p.sv_min, np.where(hi, p.sv_max, sv)))


def vehicle_dynamics_st(x, u_sv, u_accl, p, trig, rec=None):
    """f(x, u) of both branches, chosen per car by |x3| < 0.5 -> (f [n, 7], kinematic mask)."""
    g = 9.81
    x2, x3, x4, x5, x6 = x[:, 2], x[:, 3], x[:, 4], x[:, 5], x[:, 6]
    u0 = steering_constraint(x2, u_sv, p, rec)
    u1 = accl_constraints(x3, u_accl, p, rec)
    kin = np.abs(x3) < 0.5
    s, c = trig.sincos(np.where(kin, x4, x6 + x4))
    t2, c2 = np.zeros_like(x2), np.ones_like(x2)
    if kin.any():
        t2[kin], c2[kin] = trig.tan(x2[kin]), trig.cos(x2[kin])
    # kinematic branch: vehicle_dynamics_ks re-applies the constraints to the constrained input
    lwb = p.lf + p.lr
    k0, k1 = steering_constraint(x2, u0, p), accl_constraints(x3, u1, p)
    fk = [x3 * c, x3 * s, k0, k1, x3 / lwb * t2, u1 / lwb * t2 + x3 / (lwb * (c2 * c2)) * u0, np.zeros_like(x2)]
    mu, C_Sf, C_Sr, lf, lr, h, m, I = p.mu, p.C_Sf, p.C_Sr, p.lf, p.lr, p.h, p.m, p.I
    fs = [x3 * c, x3 * s, u0, u1, x5,
          -mu * m / (x3 * I * (lr + lf)) * (lf * lf * C_Sf * (g * lr - u1 * h) + lr * lr * C_Sr * (g * lf + u1 * h)) * x5
          + mu * m / (I * (lr + lf)) * (lr * C_Sr * (g * lf + u1 * h) - lf * C_Sf * (g * lr - u1 * h)) * x6
          + mu * m / (I * (lr + lf)) * lf * C_Sf * (g * lr - u1 * h) * x2,
          (mu / (x3 * x3 * (lr + lf)) * (C_Sr * (g * lf + u1 * h) * lr - C_Sf * (g * lr - u1 * h) * lf) - 1) * x5
          - mu / (x3 * (lr + lf)) * (C_Sr * (g * lf + u1 * h) + C_Sf * (g * lr - u1 * h)) * x6
          + mu / (x3 * (lr + lf)) * (C_Sf * (g * lr - u1 * h)) * x2]
    return np.stack([np.where(kin, a, b) for a, b in zip(fk, fs)], 1), kin


def pid(speed, steer, cur_speed, cur_steer, p):
    steer_diff = steer - cur_steer
    sv_on = np.abs(steer_diff) > 1e-4
    sv = np.where(sv_on, (steer_diff / np.abs(steer_diff)) * p.sv_max, 0.0)
    vel_diff = speed - cur_speed
    fast, up = cur_speed > 0., vel_diff > 0
    kp = np.where(fast, np.where(up, 10.0 * p.a_max / p.v_max, 10.0 * p.a_max / (-p.v_min)),
                  np.where(up, 2.0 * p.a_max / p.v_max, 2.0 * p.a_max / (-p.v_min)))
    return kp * vel_diff, sv, dict(sv_on=sv_on, pid_fast=fast, vd_up=up)


def wrap_yaw(a):
    """Python's (a + pi) % (2 pi) - pi with a floored fmod."""
    m = np.fmod(a + PI, 2 * PI)
    m = np.where(m != 0.0, np.where(m < 0.0, m + 2 * PI, m), 0.0)
    return m - PI


def dynamics_step(x, b0, b1, cnt, raw_steer, speed, pv, dt, integrator, trig=LIBM, reset=None, poses=None, active=None):
    """One step of K1 for n cars.  x [n, 7]; FIFO b0 (newest), b1 [n], cnt [n]; the action [n] (a float32 action is
    widened); pv [n, 18] parameter rows (or one dict); reset [n] with reset poses [n, 3]: the car is put at its pose, its
    FIFO cleared and the step uses a zero action; active [n]: an inactive car keeps state and FIFO.
    -> (x, b0, b1, cnt, trace): trace maps a branch name to a bool [n] (kin: [stages, n])."""
    with np.errstate(all='ignore'):
        x0 = np.array(x, np.float64).reshape(-1, 7)
        n = x0.shape[0]
        pv = params_matrix(pv, n) if isinstance(pv, (dict, list)) else np.asarray(pv, np.float64)
        p = _params(pv)
        x = x0.copy()
        b0, b1 = np.array(b0, np.float64).reshape(n), np.array(b1, np.float64).reshape(n)
        cnt = np.array(cnt, np.int64).reshape(n)
        fifo_in = b0, b1, cnt
        rs = np.asarray(raw_steer).astype(np.float64).reshape(n)
        sp = np.asarray(speed).astype(np.float64).reshape(n)
        rst = np.zeros(n, bool) if reset is None else np.asarray(reset).reshape(n) != 0
        if rst.any():
            poses = np.asarray(poses, np.float64).reshape(n, 3)
            x[rst] = 0.0
            x[rst, 0], x[rst, 1], x[rst, 4] = poses[rst, 0], poses[rst, 1], poses[rst, 2]
            b0, b1 = np.where(rst, 0.0, b0), np.where(rst, 0.0, b1)
            cnt = np.where(rst, 0, cnt)
            rs, sp = np.where(rst, 0.0, rs), np.where(rst, 0.0, sp)
        # steering delay FIFO
        fill = cnt < 2
        steer = np.where(fill, 0.0, b1)
        n_cnt = np.where(fill, cnt + 1, cnt)
        n_b1, n_b0 = b0, rs
        accl, sv, tr = pid(sp, steer, x[:, 3], x[:, 2], p)
        sv = _clip(sv, p.sv_min, p.sv_max)
        accl = _clip(accl, -p.a_max, p.a_max)
        tr.update(fifo_fill=fill, reset=rst)
        if integrator == RK4:
            k1, kin1 = vehicle_dynamics_st(x, sv, accl, p, trig, tr)
            k2, kin2 = vehicle_dynamics_st(x + dt * (k1 / 2), sv, accl, p, trig)
            k3, kin3 = vehicle_dynamics_st(x + dt * (k2 / 2), sv, accl, p, trig)
            k4, kin4 = vehicle_dynamics_st(x + dt * k3, sv, accl, p, trig)
            x = x + dt * (1.0 / 6.0) * (k1 + 2 * k2 + 2 * k3 + k4)     # (dt * (1/6)) * sum, the reference's grouping
            tr['kin'] = np.stack([kin1, kin2, kin3, kin4])
        else:
            f, kin = vehicle_dynamics_st(x, sv, accl, p, trig, tr)
            x = x + dt * f
            tr['kin'] = kin[None]
        tr.update(clamp_s=(x[:, 2] < p.s_min) | (x[:, 2] > p.s_max), clamp_v=(x[:, 3] < p.v_min) | (x[:, 3] > p.v_max))
        x[:, 2] = _clip(x[:, 2], p.s_min, p.s_max)
        x[:, 3] = _clip(x[:, 3], p.v_min, p.v_max)
        yaw = wrap_yaw(x[:, 4])
        tr['wrap'] = yaw.view(np.int64) != x[:, 4].view(np.int64)
        x[:, 4] = yaw
        r = x[:, 5]
        tr.update(yaw_nan=np.isnan(r), yaw_inf=np.isinf(r))
        r = np.where(np.isnan(r), 0.0, np.where(np.isinf(r), np.where(r > 0, YAW_RATE_CAP, -YAW_RATE_CAP), r))
        tr['yaw_cap'] = np.abs(r) > YAW_RATE_CAP
        x[:, 5] = _clip(r, -YAW_RATE_CAP, YAW_RATE_CAP)
        sl = x[:, 6]
        tr['slip_nan'] = np.isnan(sl)
        sl = np.where(np.isnan(sl), 0.0, sl)
        tr['slip_cap'] = np.abs(sl) > SLIP_CAP
        x[:, 6] = _clip(sl, -SLIP_CAP, SLIP_CAP)
        if active is not None:
            off = np.asarray(active).reshape(n) == 0
            x[off] = x0[off]
            n_b0, n_b1, n_cnt = (np.where(off, a, b) for a, b in zip(fifo_in, (n_b0, n_b1, n_cnt)))
        return x, n_b0, n_b1, n_cnt.astype(np.int32), tr


def sim_reset(x, b0, b1, cnt, poses, mask=None):
    """Simulator.reset (sim_reset_kernel): the masked cars to their poses at rest, FIFO cleared, no step."""
    x, b0, b1, cnt = np.array(x, np.float64), np.array(b0, np.float64), np.array(b1, np.float64), np.array(cnt, np.int32)
    poses = np.asarray(poses, np.float64).reshape(-1, 3)
    m = np.ones(len(x), bool) if mask is None else np.asarray(mask).reshape(-1) != 0
    x[m] = 0.0
    x[m, 0], x[m, 1], x[m, 4] = poses[m, 0], poses[m, 1], poses[m, 2]
    b0[m] = b1[m] = 0.0
    cnt[m] = 0
    return x, b0, b1, cnt


def same(a, b):
    """Elementwise bit equality, NaN equal to any NaN."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return (a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))


# ---------------------------------------------------------------------------------------------------------- inputs

def random_cars(rng, n, params):
    """(x [n, 7], b0, b1, cnt, raw_steer, speed): a third of the speeds around the branch switch, headings past +-pi."""
    p = params
    x = np.empty((n, 7))
    x[:, 0:2] = rng.uniform(-60, 60, (n, 2))
    x[:, 2] = rng.uniform(1.2 * p['s_min'], 1.2 * p['s_max'], n)
    x[:, 3] = np.where(rng.random(n) < 0.35, rng.uniform(-0.6, 0.6, n), rng.uniform(min(p['v_min'], 0) - 1, p['v_max'] + 1, n))
    x[:, 4] = np.where(rng.random(n) < 0.8, rng.uniform(-3.3, 3.3, n), rng.uniform(-40, 40, n))
    x[:, 5] = rng.uniform(-12, 12, n)
    x[:, 6] = rng.uniform(-1.2, 1.2, n)
    b = rng.uniform(1.2 * p['s_min'], 1.2 * p['s_max'], (3, n))
    cnt = rng.integers(0, 3, n)
    speed = rng.uniform(min(p['v_min'], 0) - 2, p['v_max'] + 2, n)
    return x, b[0], b[1], cnt, b[2], speed


def edge_cases(dt):
    """The constructed edge list: dicts of name, params (a PARAM_SETS key), x [7], b0, b1, cnt, action (raw_steer, speed)
    and expect: the branches the entry is built to reach (trace name -> bool; kin: per RK4 stage, the first for Euler)."""
    D, R = PARAM_SETS['default'], PARAM_SETS['reverse']
    up = lambda v: np.nextafter(v, np.inf)
    dn = lambda v: np.nextafter(v, -np.inf)
    out = []

    def add(name, x3=2.0, x2=0.0, x4=0.3, x5=0.0, x6=0.0, b0=0.0, b1=0.0, cnt=2, steer=0.0, speed=None, params='default',
            **expect):
        x = [1.25, -2.5, x2, x3, x4, x5, x6]
        out.append(dict(name=name, params=params, x=np.array(x, np.float64), b0=b0, b1=b1, cnt=cnt,
                        action=(steer, x3 if speed is None else speed), expect=expect))

    # the switch between the kinematic and the single-track model, |x3| < 0.5 (with a steering angle, yaw rate and slip
    # on which the two models disagree: at x2 = x5 = x6 = 0 and a zero command they give the same derivative)
    sw = dict(x2=0.1, x5=0.3, x6=0.05)
    add('v=0.5', x3=0.5, kin=[False] * 4, **sw)
    add('v=0.5-ulp', x3=dn(0.5), kin=[True] * 4, **sw)
    add('v=0.5+ulp', x3=up(0.5), kin=[False] * 4, **sw)
    add('v=-0.5', x3=-0.5, params='reverse', kin=[False] * 4, **sw)
    add('v=-0.5+ulp', x3=up(-0.5), params='reverse', kin=[True] * 4, **sw)
    add('v=-0.5-ulp', x3=dn(-0.5), params='reverse', kin=[False] * 4, **sw)
    a = R['a_max']
    add('braking across the switch', x3=0.5 + 0.3 * a * dt, speed=0.0, params='reverse', accl_lo=True,
        kin=[False, True, True, True], **sw)
    add('accelerating across the switch', x3=0.5 - 0.3 * a * dt, speed=5.0, params='reverse', accl_hi=True,
        kin=[True, False, False, False], **sw)
    # pid's steering dead band, |steer - x2| > 1e-4
    add('steer diff 1e-4', b1=1e-4, sv_on=False)
    add('steer diff -1e-4', b1=-1e-4, sv_on=False)
    add('steer diff 1e-4+ulp', b1=up(1e-4), sv_on=True)
    add('steer diff -1e-4-ulp', b1=dn(-1e-4), sv_on=True)
    # pid's gains, cur_speed > 0
    add('v=0 up', x3=0.0, speed=1.0, pid_fast=False, vd_up=True, kin=[True] * 4)
    add('v=-0 up', x3=-0.0, speed=1.0, pid_fast=False, vd_up=True)
    add('v=0 down', x3=0.0, speed=-1.0, params='reverse', pid_fast=False, vd_up=False)
    add('v=subnormal up', x3=5e-324, speed=1.0, pid_fast=True, vd_up=True)
    add('v=subnormal down', x3=5e-324, speed=0.0, pid_fast=True, vd_up=False)
    add('v=-subnormal down', x3=-5e-324, speed=-1.0, params='reverse', pid_fast=False, vd_up=False)
    # accl_constraints at v_min / v_max: acceleration outward, zero, inward
    add('v=v_max out', x3=D['v_max'], speed=25.0, accl_hold=True)
    add('v=v_max zero', x3=D['v_max'], speed=D['v_max'], accl_hold=True)
    add('v=v_min zero', x3=D['v_min'], speed=D['v_min'], accl_hold=True)
    add('v=v_min in', x3=D['v_min'], speed=0.0, accl_hold=False)
    add('reverse v=v_min out', x3=R['v_min'], speed=-6.0, params='reverse', accl_hold=True)
    add('reverse v=v_min zero', x3=R['v_min'], speed=R['v_min'], params='reverse', accl_hold=True)
    add('reverse v=v_min in', x3=R['v_min'], speed=-4.0, params='reverse', accl_hold=False)
    add('reverse v=v_max out', x3=R['v_max'], speed=25.0, params='reverse', accl_hold=True)
    add('reverse v=v_max in', x3=R['v_max'], speed=15.0, params='reverse', accl_hold=False, accl_lo=True)
    # the positive-acceleration limit at vel == v_switch
    V = PARAM_SETS['vswitch']
    for s in VSWITCH_STEER:
        add('v=v_switch, x2=%g' % s, x3=V['v_switch'], x2=s, b1=s, speed=8.0, params='vswitch', above_switch=False,
            accl_hi=True, kin=[True] * 4)
    add('v=v_switch+ulp', x3=up(V['v_switch']), speed=8.0, params='vswitch', above_switch=True, accl_hi=True)
    add('v=v_switch-ulp', x3=dn(V['v_switch']), speed=8.0, params='vswitch', above_switch=False, accl_hi=True)
    # steering_constraint at s_min / s_max: steering velocity < 0, = 0, > 0
    for lim, sgn in (('s_max', 1.0), ('s_min', -1.0)):
        s = D[lim]
        add('x2=%s out' % lim, x2=s, b1=s + 0.1 * sgn, sv_on=True, steer_hold=True)
        add('x2=%s zero' % lim, x2=s, b1=s, sv_on=False, steer_hold=True)
        add('x2=%s in' % lim, x2=s, b1=0.0, sv_on=True, steer_hold=False, sv_lo=sgn > 0, sv_hi=sgn < 0)
        add('x2 short of %s' % lim, x2=s - sgn * 0.25 * D['sv_max'] * dt, b1=s + 0.1 * sgn, steer_hold=False, clamp_s=True)
    # the yaw wrap
    add('yaw=pi', x4=PI, wrap=True)
    add('yaw=-pi', x4=-PI, wrap=False)
    add('yaw=pi+ulp', x4=up(PI), wrap=True)
    add('yaw=-pi-ulp', x4=dn(-PI), wrap=True)
    add('yaw=31.4', x4=31.4, wrap=True)
    add('yaw=-47.1', x4=-47.1, wrap=True)
    add('yaw=2pi', x4=2 * PI, wrap=True)
    # yaw rate and slip beyond their caps, infinite, NaN
    add('yaw rate 15', x3=0.2, x5=15.0, kin=[True] * 4, yaw_cap=True)
    add('yaw rate -15', x3=0.2, x5=-15.0, kin=[True] * 4, yaw_cap=True)
    add('yaw rate inf', x3=0.2, x5=np.inf, kin=[True] * 4, yaw_inf=True)
    add('yaw rate -inf', x3=0.2, x5=-np.inf, kin=[True] * 4, yaw_inf=True)
    add('yaw rate nan', x3=0.2, x5=np.nan, kin=[True] * 4, yaw_nan=True)
    add('yaw rate 40 st', x3=8.0, x5=40.0, kin=[False] * 4, yaw_cap=True)
    add('yaw rate inf st', x3=2.0, x5=np.inf, kin=[False] * 4, yaw_inf=False, yaw_nan=True)
    add('slip 1.5', x3=0.2, x6=1.5, kin=[True] * 4, slip_cap=True)
    add('slip -1.5', x3=0.2, x6=-1.5, kin=[True] * 4, slip_cap=True)
    add('slip inf', x3=0.2, x6=np.inf, kin=[True] * 4, slip_cap=True, slip_nan=False)
    add('slip -inf', x3=0.2, x6=-np.inf, kin=[True] * 4, slip_cap=True, slip_nan=False)
    add('slip nan', x3=0.2, x6=np.nan, kin=[True] * 4, slip_nan=True)
    add('slip nan st', x3=2.0, x6=np.nan, kin=[False] * 4, slip_nan=True)
    # reverse driving
    add('reverse st', x3=-3.0, speed=-4.0, params='reverse', kin=[False] * 4, pid_fast=False, vd_up=False)
    add('reverse kin', x3=-0.3, speed=-1.0, b1=0.2, params='reverse', kin=[True] * 4, pid_fast=False, sv_on=True)
    # the FIFO and non-finite actions
    for c in (0, 1, 2):
        add('fifo cnt %d' % c, b0=0.3, b1=-0.2, cnt=c, steer=0.1, fifo_fill=c < 2, sv_on=c == 2)
    for v in (np.nan, np.inf, -np.inf):
        add('steer %r' % v, steer=v, fifo_fill=False)
        add('steer %r, fifo filling' % v, steer=v, cnt=1, fifo_fill=True)
        add('fifo delivers %r' % v, b1=v, fifo_fill=False)
        add('speed %r' % v, speed=v)
    return out


def stack_edges(cases, key_params=None):
    """Arrays of an edge list: x [n, 7], b0, b1, cnt, raw_steer, speed, pv [n, 18]."""
    x = np.stack([c['x'] for c in cases])
    b0, b1 = (np.array([c[k] for c in cases], np.float64) for k in ('b0', 'b1'))
    cnt = np.array([c['cnt'] for c in cases], np.int32)
    act = np.array([c['action'] for c in cases], np.float64)
    pv = params_matrix([PARAM_SETS[c['params']] for c in cases], len(cases))
    return x, b0, b1, cnt, act[:, 0], act[:, 1], pv


def check_expectations(cases, tr, integrator):
    """Every entry reached the branches it was built for."""
    for i, c in enumerate(cases):
        for k, want in c['expect'].items():
            if k == 'kin':
                got = [bool(v) for v in tr['kin'][:, i]]
                want = want if integrator == RK4 else want[:1]
            else:
                got = bool(tr[k][i])
            assert got == want, (c['name'], k, got, want)


def oracle_update(x, b0, b1, cnt, raw_steer, speed, pv, dt, integrator):
    """Oracle.update_pose over cars whose parameter rows may differ (grouped by row)."""
    n = len(x)
    xo, bo, co = np.empty((n, 7)), np.empty((n, 2)), np.empty(n, np.int32)
    rows, inv = np.unique(pv, axis=0, return_inverse=True)
    for r in range(len(rows)):
        sel = np.flatnonzero(inv.reshape(-1) == r)
        p = dict(zip(PARAM_KEYS, rows[r]))
        xo[sel], bo[sel], co[sel] = Oracle.update_pose(x[sel], np.stack([b0[sel], b1[sel]], 1), cnt[sel], raw_steer[sel],
                                                       speed[sel], p, dt, integrator)
    return xo, bo[:, 0], bo[:, 1], co


def assert_same_as_oracle(x, b0, b1, cnt, raw_steer, speed, pv, dt, integrator, names=None):
    got = dynamics_step(x, b0, b1, cnt, raw_steer, speed, pv, dt, integrator)
    want = oracle_update(x, b0, b1, cnt, raw_steer, speed, pv, dt, integrator)
    for k, (g, w) in enumerate(zip(got[:4], want)):
        ok = same(g, w)
        if ok.ndim == 2:
            ok = ok.all(1)
        bad = np.flatnonzero(~ok)
        assert bad.size == 0, ('state b0 b1 cnt'.split()[k], len(bad), [names[i] if names else i for i in bad[:5]],
                               g[bad[:2]], w[bad[:2]])
    return got[4]


# ---------------------------------------------------------------------------------------------------------- tests

@pytest.mark.parametrize('integrator', [RK4, EULER])
@pytest.mark.parametrize('dt', TIMESTEPS)
def test_random_steps_match_oracle(dt, integrator):
    """3000 random (state, FIFO, action) triples per parameter set: 6 sets x 8 (timestep, integrator) pairs = 144 000 steps
    in all, about a third of them on the kinematic branch."""
    rng = np.random.default_rng(int(dt * 1e5) + 7 * integrator)
    n, kin = 3000, 0
    for name, p in PARAM_SETS.items():
        x, b0, b1, cnt, rs, sp = random_cars(rng, n, p)
        if name == 'agent1':
            rs, sp = rs.astype(np.float32), sp.astype(np.float32)      # f32 actions, widened
        tr = assert_same_as_oracle(x, b0, b1, cnt, rs, sp, params_matrix(p, n), dt, integrator)
        kin += int(tr['kin'][0].sum())
        assert 0 < tr['kin'][0].sum() < n and 0 < tr['fifo_fill'].sum() < n, name
    assert kin > 0.25 * n * len(PARAM_SETS)


@pytest.mark.parametrize('integrator', [RK4, EULER])
@pytest.mark.parametrize('dt', TIMESTEPS)
def test_edge_list_matches_oracle(dt, integrator):
    cases = edge_cases(dt)
    x, b0, b1, cnt, rs, sp, pv = stack_edges(cases)
    tr = assert_same_as_oracle(x, b0, b1, cnt, rs, sp, pv, dt, integrator, names=[c['name'] for c in cases])
    check_expectations(cases, tr, integrator)


def test_edge_list_reaches_its_ties():
    """The ties the edge list is built on are real: for the v_switch pair a_max * v_switch / v_switch rounds below a_max
    (the defaults give a_max), the yaw at +pi wraps to -pi, and the names of the edge list are unique."""
    V, D = PARAM_SETS['vswitch'], PARAM_SETS['default']
    assert V['a_max'] * V['v_switch'] / V['v_switch'] < V['a_max']
    assert D['a_max'] * D['v_switch'] / D['v_switch'] == D['a_max']
    x, *_ = dynamics_step(np.array([[0.0, 0.0, 0.0, 2.0, PI, 0.0, 0.0]]), [0.], [0.], [2], [0.], [2.0], D, 0.01, RK4)
    assert x[0, 4] == -PI
    names = [c['name'] for c in edge_cases(0.01)]
    assert len(names) == len(set(names))


@pytest.mark.parametrize('integrator', [RK4, EULER])
@pytest.mark.parametrize('dt', TIMESTEPS)
def test_edge_list_shows_the_v_switch_tie(dt, integrator, monkeypatch):
    """vel >= v_switch in place of vel > v_switch changes the state of at least one v_switch entry."""
    import sys
    cases = [c for c in edge_cases(dt) if c['name'].startswith('v=v_switch, ')]
    args = stack_edges(cases)[:6] + (params_matrix(VSWITCH_PARAMS, len(cases)), dt, integrator)
    right = dynamics_step(*args)[0]

    def above_or_at(vel, accl, p, rec=None):
        pos_limit = np.where(vel >= p.v_switch, p.a_max * p.v_switch / vel, p.a_max)
        return np.where(accl >= pos_limit, pos_limit, accl)      # the entries reach neither the hold nor the lower clip
    monkeypatch.setattr(sys.modules[__name__], 'accl_constraints', above_or_at)
    assert not same(dynamics_step(*args)[0], right).all()


def test_env_rules_match_oracle():
    """The env-level rules of the model -- reset steps with a zero action, inactive envs untouched, Simulator.reset with an
    env mask, per-agent parameters, f32 actions -- against the oracle's env on CPU (iTTC threshold 0, so its state is the
    dynamics' own), under RK4 and Euler."""
    from tests import helpers as H
    N, A = 5, 3
    for integrator, dt in ((RK4, 0.01), (EULER, 0.005)):
        o = Oracle(N, A, timestep=dt, integrator=integrator, ego_idx=1, ttc_thresh=0.0)
        o.set_map_arrays(*H.golden_map('open_square'))
        o.update_params(AGENT1_PARAMS, 1)
        o.update_params(REVERSE_PARAMS, 2)
        pv = params_matrix([DEFAULT_PARAMS, AGENT1_PARAMS, REVERSE_PARAMS] * N, N * A)
        rng = np.random.default_rng(integrator)
        poses = np.concatenate([rng.uniform(-3, 3, (N, A, 2)), rng.uniform(-PI, PI, (N, A, 1))], 2)
        x = np.zeros((N * A, 7)); b0 = np.zeros(N * A); b1 = np.zeros(N * A); cnt = np.zeros(N * A, np.int32)
        for t in range(40):
            act = np.stack([rng.uniform(-0.5, 0.5, (N, A)), rng.uniform(-3, 8, (N, A))], 2).astype(np.float32)
            rm = np.ones(N, np.uint8) if t == 0 else (rng.random(N) < 0.1).astype(np.uint8)
            am = None if t < 5 or t == 20 else (rng.random(N) < 0.8).astype(np.uint8)
            if t == 20:     # the oracle's Simulator.reset has no env mask, and its state output skips inactive envs
                o.sim_reset(poses[::-1])
                x, b0, b1, cnt = sim_reset(x, b0, b1, cnt, poses[::-1].reshape(-1, 3))
            out = o.step(act, reset_mask=rm, reset_poses=poses, active_mask=am)
            rep = lambda m: None if m is None else np.repeat(m, A)
            x, b0, b1, cnt, _ = dynamics_step(x, b0, b1, cnt, act[..., 0], act[..., 1], pv, dt, integrator,
                                              reset=rep(rm), poses=poses.reshape(-1, 3), active=rep(am))
            assert same(x, out['state'].reshape(-1, 7)).all(), (integrator, t)
