"""The consumer kernels (csrc/f110_consumers.cu) held to the oracle bit for bit.

gap_follow_kernel: over the parameter grid of test_consumer_model.py (every window size, bubble radius, threshold, beam
count up to 8192 with the shared-memory opt-in, the speed band boundaries, non-finite beams), through strided [N, 3, n]
views, agent 0 and agent 2, with the other slots asserted untouched.

shaped_reward_warp_kernel: the reward is built with -fmad=false, and every operation in it is
IEEE-exact except hypot (the opponent bubble) and sincos (the flank).  The expected value is the oracle's breakdown with
those two terms recomputed in numpy from the device's own hypot and sincos (f110_hypot_probe, f110_trig_probe), summed
in the kernel's order: it must equal out_f64 exactly, and out_f32 must equal its float32 rounding, on every case of
reward_cases().
"""
import ctypes as C

import numpy as np
import pytest

from oracle.f110_oracle import REWARD_DEFAULTS, REWARD_TERM as T, gap_follow_action
from tests.test_consumer_model import check_branches, gap_follow_grid, reward_cases

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


# ----------------------------------------------------------------------------------------------------- gap follow

def _gap_follow_device(scans, agent_idx, A=3, **kw):
    """Scans [N, n] placed in slot agent_idx of [N, A, n]; -> the actions [N, A, 2] after the kernel (other slots -7)."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import gap_follow_actions
    N, n = scans.shape
    t = torch.full((N, A, n), 5.0, dtype=torch.float32, device='cuda')
    if N:
        t[:, agent_idx] = torch.from_numpy(np.ascontiguousarray(scans)).cuda()
    act = torch.full((N, A, 2), -7.0, dtype=torch.float32, device='cuda')
    gap_follow_actions(t, act, agent_idx=agent_idx, **kw)
    torch.cuda.synchronize()
    return act.cpu().numpy()


def _check_gap_follow(scans, agent_idx, **kw):
    a = _gap_follow_device(scans, agent_idx, **kw)
    want = np.stack([gap_follow_action(s, **kw) for s in scans]).astype(np.float32) if len(scans) else np.zeros((0, 2), np.float32)
    others = [k for k in range(a.shape[1]) if k != agent_idx]
    assert (a[:, others] == -7.0).all()
    bad = np.nonzero((a[:, agent_idx] != want).any(1))[0]
    assert len(bad) == 0, (kw, bad[:10], a[bad[:3], agent_idx], want[bad[:3]])


@pytest.mark.parametrize('label,scans,kw', [pytest.param(*c, id=c[0]) for c in gap_follow_grid()])
def test_gap_follow_kernel_equals_oracle(label, scans, kw):
    for agent_idx in (0, 2):
        _check_gap_follow(scans, agent_idx, **kw)


@pytest.mark.parametrize('N', [0, 1, 7, 8193])
@pytest.mark.parametrize('w', [5, 9])
def test_gap_follow_kernel_batch_sizes(N, w):
    rng = np.random.default_rng(N + w)
    scans = rng.uniform(0, 4, (N, 1080)).astype(np.float32)
    if N > 1:
        scans[::5, rng.integers(0, 1080)] = np.nan
        scans[1::7, 200:400] = rng.uniform(0, 0.4, (len(scans[1::7]), 200)).astype(np.float32)
    _check_gap_follow(scans, 2, window_size=w)


def test_gap_follow_rejects_bad_arguments():
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import gap_follow_actions
    t = torch.zeros((2, 2, 64), dtype=torch.float32, device='cuda')
    act = torch.zeros((2, 2, 2), dtype=torch.float32, device='cuda')
    for kw in (dict(bubble_radius=-1), dict(window_size=0), dict(window_size=16)):
        with pytest.raises(ValueError):
            gap_follow_actions(t, act, **kw)


# ----------------------------------------------------------------------------------------------------- shaped reward

class DeviceMath(object):
    """The reward kernels' hypot and sincos, evaluated by the library's probes."""

    def __init__(self):
        from f110_gymnasium_ros2_jazzy_b200 import _lib
        self.torch, self._lib, self.L = _torch(), _lib, _lib.load()

    def _run(self, fn, *arrays, rows=1):
        torch = self.torch
        n = len(arrays[0])
        ins = [torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda() for a in arrays]
        out = torch.zeros(rows * max(n, 1), dtype=torch.float64, device='cuda')
        self._lib.check(fn(*[C.c_void_p(x.data_ptr()) for x in ins], n, C.c_void_p(out.data_ptr()), None))
        torch.cuda.synchronize()
        return out.cpu().numpy()[:rows * n].reshape(rows, n)

    def hypot(self, a, b):
        return self._run(self.L.f110_hypot_probe, a, b)[0]

    def sincos(self, x):
        o = self._run(self.L.f110_trig_probe, x, rows=4)
        return o[0], o[1]


def expected_reward(dm, obs, tot, terms, B, kw):
    """The oracle's totals [N] with r_opp and r_flank recomputed from the device's hypot and sincos, summed in the kernel's
    order (the oracle's total itself where the call returned early)."""
    p = dict(REWARD_DEFAULTS); p.update(kw)
    o = obs.astype(np.float64)
    ex, ey, ox, oy = o[:, B], o[:, B + 1], o[:, B + 4], o[:, B + 5]
    dx, dy = ex - ox, ey - oy
    rho = dm.hypot(dx, dy)
    safe = p['opp_safe_dist']
    y = (safe - rho) / (safe if safe > 1e-6 else 1e-6)
    r_opp = np.where((terms[:, T['steps']] >= p['grace_steps_opp']) & (rho < safe), -p['w_opp'] * (y * y), 0.0)
    sn, cs = dm.sincos(-terms[:, T['oth']])
    with np.errstate(invalid='ignore'):                   # poisoned poses: NaN and inf products, outside the box
        x_rel, y_rel = cs * dx - sn * dy, sn * dx + cs * dy
        ay = np.abs(y_rel)
        inside = (0.2 <= x_rel) & (x_rel <= 1.8) & (0.25 <= ay) & (ay <= 0.8)
        yb = np.maximum(0.8 - np.abs(ay - 0.525), 0.0)
        r_flank = np.where(inside, 0.1 * (x_rel / 1.8) * (yb / 0.8), 0.0)
    t = terms
    total = (((((t[:, T['r_prog']] + t[:, T['r_alive']]) + t[:, T['r_lead']]) + t[:, T['r_lat']]) + t[:, T['r_wall']]) + r_opp) + r_flank
    early = t[:, T['early']] > 0
    return np.where(early, tot, total), int((r_opp != t[:, T['r_opp']]).sum() + (r_flank != t[:, T['r_flank']]).sum())


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize('c', reward_cases(), ids=lambda c: c.name)
def test_shaped_reward_kernels_equal_oracle(c):
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward, _lib
    from oracle.f110_oracle import RewardOracle
    dm = DeviceMath()
    L = _lib.load()
    Tn, N, _ = c.obs.shape
    rw = ShapedReward(N, c.centerline, num_beams=c.num_beams, closed=c.closed, **c.kw)
    orc = RewardOracle(N, c.centerline, num_beams=c.num_beams, closed=c.closed, **c.kw)
    o64 = torch.full((N,), -123.0, dtype=torch.float64, device='cuda')
    o32 = torch.full((N,), -123.0, dtype=torch.float32, device='cuda')
    breakdown = []
    libm_differs = 0
    for t in range(Tn):
        ob = torch.from_numpy(c.obs[t]).cuda()
        mask = None if c.masks is None else torch.from_numpy(c.masks[t]).cuda()
        mode = t % 3                                  # f64 and f32, f64 only, f32 only
        p64 = C.c_void_p(o64.data_ptr()) if mode in (0, 1) else None
        p32 = C.c_void_p(o32.data_ptr()) if mode in (0, 2) else None
        o64.fill_(-123.0); o32.fill_(-123.0)
        _lib.check(L.f110_reward_compute(rw.h, C.c_void_p(ob.data_ptr()), None if mask is None else C.c_void_p(mask.data_ptr()),
                                         p64, p32, None))
        torch.cuda.synchronize()
        tot, terms = orc.compute_terms(c.obs[t], None if c.masks is None else c.masks[t])
        breakdown.append(terms)
        want, nd = expected_reward(dm, c.obs[t], tot, terms, c.num_beams, c.kw)
        libm_differs += nd
        g64, g32 = o64.cpu().numpy(), o32.cpu().numpy()
        if mode in (0, 1):
            bad = np.nonzero(~((g64 == want) | (np.isnan(g64) & np.isnan(want))))[0]
            assert len(bad) == 0, (c.name, t, bad[:5], g64[bad[:5]], want[bad[:5]])
        else:
            assert (g64 == -123.0).all()
        if mode in (0, 2):
            assert _same(g32, want.astype(np.float32)), (c.name, t)
        else:
            assert (g32 == -123.0).all()
    rw.close()
    check_branches(c, np.stack(breakdown))          # the case reached what it was built for
    print(c.name, 'reward terms where the device hypot / sincos differ from glibc:', libm_differs)


def test_reward_centerline_point_limit():
    """ceil((n - 1) / 64) <= 256 midpoint blocks: 16 385 points are accepted, 16 386 refused with that number."""
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward
    xy = np.stack([np.linspace(0, 100, 16386), np.zeros(16386)], 1)
    ShapedReward(1, xy[:16385], num_beams=8).close()
    with pytest.raises(ValueError, match='16385'):
        ShapedReward(1, xy, num_beams=8)
