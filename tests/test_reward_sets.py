"""The shaped reward on a set of centerlines (f110_reward_create_set, f110_reward_compute_slots, ShapedReward(centerlines=),
DeviceRollout on a map set; DESIGN.md section 10).

The expected value throughout: K single-centerline references, each run over all N envs, env e read from reference
slots[e], each reference given reset_mask | slot changed.  The references are the oracle (with the device's hypot and
sincos, as test_consumer_kernels.py holds the single-line kernels to it) or single-line ShapedReward objects, which that
file holds to the oracle bit for bit.  The GPU tests run at a short scan, where four envs share a CTA, and at the
longest, 8192 beams, where a warp's scratch leaves room for only one env per CTA.

CPU: the argument checks of ShapedReward(centerlines=...) and of f110_reward_create_set (both refuse before any device
call), and a static guard on the reward kernels' stack frames in the built library.
"""
import ctypes as C
import re

import numpy as np
import pytest

from tests import helpers as H
from tests.test_consumer_model import circle_xy, episodes, hairpin_xy, s_curve_xy

INT32_MAX = 2 ** 31 - 1


# ----------------------------------------------------------------------------------------------------- CPU

def test_shaped_reward_argument_checks():
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward
    line = np.stack([np.linspace(0, 10, 50), np.zeros(50)], 1)
    bad = [
        (dict(centerline=line, centerlines=[line]), 'either'),
        (dict(), 'either'),
        (dict(centerlines=[]), '0 given'),
        (dict(centerlines=[line] * 257), '257 given'),
        (dict(centerlines=[line, line[:1]]), 'centerline 1 has 1 points'),
        (dict(centerlines=[line, line, np.zeros((16386, 2))]), 'centerline 2 has 16386 points; 2 to 16385'),
        (dict(centerlines=[line, np.zeros((10, 3))]), r'centerline 1: shape \(10, 3\)'),
        (dict(centerlines=[line, np.zeros(10)]), 'centerline 1: shape'),
        (dict(centerlines=[line, line], closed=[True]), '1 flags for 2 centerlines'),
        (dict(centerlines=[line, line], closed=[True, False, True]), '3 flags for 2 centerlines'),
    ]
    for kw, msg in bad:
        with pytest.raises(ValueError, match=msg):
            ShapedReward(4, num_beams=8, **kw)


def _lines_c(lines, closed=1):
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    arr = (_lib.F110Centerline * max(len(lines), 1))()
    keep = []
    for d, xy in zip(arr, lines):
        xy = np.ascontiguousarray(xy, np.float64)
        keep.append(xy)
        d.xy, d.num_points, d.closed = xy.ctypes.data, len(xy), closed
    return arr, keep


def test_create_set_validates_every_line_before_allocating():
    """The C entry point refuses bad sets before any device call, so it answers without a GPU too, naming the line."""
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    L = _lib.load()
    cfg = _lib.F110RewardConfig(num_envs=4, num_beams=8)
    line = np.stack([np.linspace(0, 10, 50), np.zeros(50)], 1)
    cases = [([line] * 257, 257, '257 centerlines; 1 to 256'),
             ([line], 0, '0 centerlines'),
             ([line, line, line, np.zeros((16386, 2))], 4, 'centerline 3 has 16386 points; 2 to 16385'),
             ([line, line[:1]], 2, 'centerline 1 has 1 points')]
    for lines, count, msg in cases:
        arr, keep = _lines_c(lines)
        h = C.c_void_p()
        assert L.f110_reward_create_set(C.byref(cfg), arr, count, C.byref(h)) == _lib.F110_ERR_INVALID
        assert msg in L.f110_last_error().decode(), (msg, L.f110_last_error())
        assert not h.value
    arr, keep = _lines_c([line, line])
    arr[1].xy = None
    h = C.c_void_p()
    assert L.f110_reward_create_set(C.byref(cfg), arr, 2, C.byref(h)) == _lib.F110_ERR_INVALID
    assert 'centerline 1 has no points' in L.f110_last_error().decode()


def test_reward_kernels_stack_frames():
    """Exactly the two reward kernels exist, and the set kernel's local memory is at most 16 bytes above the single-line
    kernel's 80-byte stack frame: the line's view (pointers, L, closed) does not go to local memory."""
    from tests.test_kernel_shape import CUOBJDUMP, _functions
    if not CUOBJDUMP:
        pytest.skip("cuobjdump neither on PATH nor under CUDA_HOME")
    res = _functions(["-res-usage"])
    local = {}
    for name, lines in res.items():
        m = re.search(r"(shaped_reward_(?:set_)?(?:warp_)?kernel)", name)
        if m:
            local[m.group(1)] = int(re.search(r"LOCAL:(\d+)", " ".join(lines)).group(1))
    assert set(local) == {'shaped_reward_warp_kernel', 'shaped_reward_set_warp_kernel'}, local
    assert local['shaped_reward_warp_kernel'] <= 80, local
    assert local['shaped_reward_set_warp_kernel'] <= 80 + 16, local


# ----------------------------------------------------------------------------------------------------- GPU

def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


KW = dict(near_wall_dist=0.2, grace_steps_wall=1, grace_steps_opp=0, w_rel_lead=0.5, lead_clip=0.05, opp_safe_dist=2.0)


def _prune_xy():
    k = np.arange(192)
    return np.concatenate([np.stack([-0.5 + 0.4 * np.cos(0.3 * k), 0.5 + 0.4 * np.sin(0.3 * k)], 1)[:-1],
                           [[0.0, 0.0], [10.0, 0.0], [10.0, 1.0]]])


def _lines():
    """(centerline [n, 2 | 4], closed): Shanghai with its widths and with 2 columns, the open s-curve, the closed circle
    with its seam, the hairpin, and the open line whose last block holds one midpoint."""
    sh = H.load('reward')['centerline']
    return [(sh, True), (sh[:, :2], True), (s_curve_xy(), False), (circle_xy(), True), (hairpin_xy(), True),
            (_prune_xy(), False)]


def _assemble(rng, lines, slots_t, T, B, **ep):
    """Observations [T, N, B+8]: env e at step t takes the step-t row of an episode driven on line slots_t[t][e] (its own
    episode per line), plus the per-line reset masks read the same way.  Slots outside [0, K) read line 0."""
    N = slots_t.shape[1]
    per = [episodes(rng, np.asarray(cl)[:, :2], closed, N, T, B, **ep) for cl, closed in lines]
    idx = np.clip(slots_t, 0, len(lines) - 1)
    obs = np.stack([np.stack([per[idx[t, e]][0][t, e] for e in range(N)]) for t in range(T)])
    masks = np.stack([np.array([per[idx[t, e]][1][t, e] for e in range(N)], np.uint8) for t in range(T)])
    return obs, masks


class SetRun(object):
    """A set reward object driven through f110_reward_compute_slots with both outputs."""

    def __init__(self, N, lines, B, **kw):
        torch = _torch()
        from f110_gymnasium_ros2_jazzy_b200 import ShapedReward, _lib
        self.torch, self.lib, self._lib = torch, _lib.load(), _lib
        self.rw = ShapedReward(N, centerlines=[cl for cl, _ in lines], closed=[c for _, c in lines], num_beams=B, **kw)
        self.o64 = torch.zeros(N, dtype=torch.float64, device='cuda')
        self.o32 = torch.zeros(N, dtype=torch.float32, device='cuda')

    def __call__(self, obs, mask, slots):
        torch = self.torch
        ob = torch.from_numpy(np.ascontiguousarray(obs)).cuda()
        m = None if mask is None else torch.from_numpy(np.ascontiguousarray(mask, np.uint8)).cuda()
        sl = torch.from_numpy(np.ascontiguousarray(slots, np.int32)).cuda()
        self.o64.fill_(-123.0); self.o32.fill_(-123.0)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        self._lib.check(self.lib.f110_reward_compute_slots(self.rw.h, p(ob), p(m), p(sl), p(self.o64), p(self.o32), None))
        torch.cuda.synchronize()
        return self.o64.cpu().numpy().copy(), self.o32.cpu().numpy().copy()


def _changed(slots_t):
    """[T, N]: the env's slot differs from the one of its previous call (-1 before the first)."""
    T, N = slots_t.shape
    prev = np.full(N, -1)
    out = np.zeros((T, N), bool)
    for t in range(T):
        out[t] = slots_t[t] != prev
        prev = slots_t[t]
    return out


def _single_refs(lines, N, B, obs, masks, slots_t, **kw):
    """What K single-line ShapedReward objects give, env e read from reference slots[t][e] -> f64 [T, N]."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward
    refs = [ShapedReward(N, cl, num_beams=B, closed=c, **kw) for cl, c in lines]
    chg = _changed(slots_t)
    want = np.zeros(slots_t.shape)
    for t in range(len(obs)):
        ob = torch.from_numpy(np.ascontiguousarray(obs[t])).cuda()
        m = (chg[t] | (masks[t] != 0 if masks is not None else False)).astype(np.uint8)
        got = [r(ob, torch.from_numpy(m).cuda()).cpu().numpy() for r in refs]
        want[t] = np.choose(slots_t[t], got)
    for r in refs:
        r.close()
    return want


def _check_step(g64, g32, want, where):
    bad = np.nonzero(g64.view(np.int64) != want.view(np.int64))[0]
    assert len(bad) == 0 or np.array_equal(g64[bad], want[bad], equal_nan=True), (where, bad[:5], g64[bad[:5]], want[bad[:5]])
    assert np.array_equal(g32, want.astype(np.float32), equal_nan=True), where


@pytest.mark.gpu
@pytest.mark.parametrize('B', [1080, 8192])
def test_set_equals_oracle(B):
    """Envs in blocks and interleaved, reset masks from the episodes: out_f64 equals the oracle of each env's line bit
    for bit, out_f32 is its rounding.  1080 beams on six lines; the longest scan, 8192 beams (one warp per CTA), on two."""
    _torch()
    from oracle.f110_oracle import RewardOracle
    from tests.test_consumer_kernels import DeviceMath, expected_reward
    dm = DeviceMath()
    rng = np.random.default_rng(31)
    lines = _lines()
    per_line, T, sub = (5, 30, lines) if B == 1080 else (2, 6, [lines[0], lines[3]])
    K = len(sub)
    for slots in (np.repeat(np.arange(K), per_line), np.arange(K * per_line) % K):       # blocks, interleaved
        N = len(slots)
        slots_t = np.broadcast_to(slots, (T, N)).copy()
        obs, masks = _assemble(rng, sub, slots_t, T, B)
        run = SetRun(N, sub, B, **KW)
        orcs = [RewardOracle(N, cl, num_beams=B, closed=c, **KW) for cl, c in sub]
        chg = _changed(slots_t)
        for t in range(T):
            g64, g32 = run(obs[t], masks[t], slots_t[t])
            m = (masks[t] != 0) | chg[t]
            want = np.zeros(N)
            for k, o in enumerate(orcs):
                tot, terms = o.compute_terms(obs[t], m.astype(np.uint8))
                wk, _ = expected_reward(dm, obs[t], tot, terms, B, KW)
                want[slots == k] = wk[slots == k]
            _check_step(g64, g32, want, (B, t))
        run.rw.close()


def _three_lines():
    sh = H.load('reward')['centerline']
    return [(sh, True), (circle_xy(), True), (s_curve_xy(), False)]


@pytest.mark.gpu
@pytest.mark.parametrize('B', [64, 8192])
def test_slot_change_restarts_only_the_moved_envs(B):
    """At step 15 a third of the envs move to another line with no reset mask: they restart (their value is a fresh
    reward object's first), the others go on; every step equals the single-line references."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward
    lines = _three_lines()
    K, N, T, tc = len(lines), 12, 30, 15
    rng = np.random.default_rng(5)
    slots = np.arange(N) % K
    moved = np.arange(N) % 3 == 1
    slots_t = np.broadcast_to(slots, (T, N)).copy()
    slots_t[tc:, moved] = (slots[moved] + 1) % K
    obs, _ = _assemble(rng, lines, slots_t, T, B, phase=False)
    run = SetRun(N, lines, B, **KW)
    want = _single_refs(lines, N, B, obs, None, slots_t, **KW)
    for t in range(T):
        g64, g32 = run(obs[t], None, slots_t[t])
        _check_step(g64, g32, want[t], t)
        if t == tc:
            fresh = [ShapedReward(N, cl, num_beams=B, closed=c, **KW) for cl, c in lines]
            first = np.choose(slots_t[t], [f(torch.from_numpy(obs[t]).cuda()).cpu().numpy() for f in fresh])
            assert np.array_equal(g64[moved], first[moved])
            assert (g64[~moved] != first[~moved]).any()
            for f in fresh:
                f.close()
    run.rw.close()


@pytest.mark.gpu
@pytest.mark.parametrize('B', [64, 8192])
def test_out_of_range_slot_leaves_the_record(B):
    """At step 8 every env has a slot outside [0, K) (-1, K, INT32_MAX): NaN in both outputs.  Back on a valid slot, each
    env goes on exactly as a set that never saw that call -- which counts a return to another line as a slot change."""
    _torch()
    lines = _three_lines()
    K, N, T, tb = len(lines), 12, 20, 8
    rng = np.random.default_rng(8)
    slots = np.arange(N) % K
    slots_t = np.broadcast_to(slots, (T, N)).copy()
    slots_t[tb] = np.array([-1, K, INT32_MAX])[np.arange(N) % 3]
    slots_t[tb + 1:, np.arange(N) % 2 == 1] = (slots[np.arange(N) % 2 == 1] + 1) % K     # half come back elsewhere
    obs, masks = _assemble(rng, lines, slots_t, T, B)
    a, b = SetRun(N, lines, B, **KW), SetRun(N, lines, B, **KW)
    keep = np.arange(T) != tb
    want = _single_refs(lines, N, B, obs[keep], masks[keep], slots_t[keep], **KW)
    j = 0
    for t in range(T):
        ga64, ga32 = a(obs[t], masks[t], slots_t[t])
        if t == tb:
            assert np.isnan(ga64).all() and np.isnan(ga32).all()
            continue
        gb64, gb32 = b(obs[t], masks[t], slots_t[t])
        assert np.array_equal(ga64.view(np.int64), gb64.view(np.int64)) and np.array_equal(ga32.view(np.int32), gb32.view(np.int32)), t
        _check_step(gb64, gb32, want[j], t)
        j += 1
    a.rw.close(); b.rw.close()


@pytest.mark.gpu
@pytest.mark.parametrize('B', [1080, 8192])
def test_set_of_one_is_the_single_reward(B):
    """f110_reward_create_set with one line equals f110_reward_create bit for bit, through f110_reward_compute_slots with
    no slots and with slots that would be out of range (a set of one does not read them).  On a set of two,
    f110_reward_compute and f110_reward_compute_slots without slots refuse."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward, _lib
    L = _lib.load()
    sh = H.load('reward')['centerline']
    N, T = 8, 12
    obs, masks = episodes(np.random.default_rng(2), sh[:, :2], True, N, T, B)
    one = ShapedReward(N, sh, num_beams=B, **KW)
    sets = [ShapedReward(N, centerlines=[sh], num_beams=B, **KW) for _ in range(2)]
    assert one.num_centerlines == 1 and sets[0].num_centerlines == 1 and L.f110_reward_count(sets[0].h) == 1
    far = torch.full((N,), 5, dtype=torch.int32, device='cuda')
    for t in range(T):
        ob = torch.from_numpy(obs[t]).cuda()
        m = torch.from_numpy(masks[t]).cuda()
        want = one(ob, m).clone()
        assert torch.equal(sets[0](ob, m).view(torch.int64), want.view(torch.int64)), t
        assert torch.equal(sets[1](ob, m, slots=far).view(torch.int64), want.view(torch.int64)), t
    two = ShapedReward(N, centerlines=[sh, circle_xy()], num_beams=B)
    assert two.num_centerlines == 2 and L.f110_reward_count(two.h) == 2
    ob = torch.from_numpy(obs[0]).cuda()
    out = torch.zeros(N, dtype=torch.float64, device='cuda')
    assert L.f110_reward_compute(two.h, C.c_void_p(ob.data_ptr()), None, C.c_void_p(out.data_ptr()), None, None) == _lib.F110_ERR_INVALID
    assert 'f110_reward_compute_slots' in L.f110_last_error().decode()
    assert L.f110_reward_compute_slots(two.h, C.c_void_p(ob.data_ptr()), None, None, C.c_void_p(out.data_ptr()), None,
                                       None) == _lib.F110_ERR_INVALID
    with pytest.raises(ValueError, match='slots'):
        two(ob)
    for r in [one, two] + sets:
        r.close()


@pytest.mark.gpu
def test_set_limits():
    """256 lines are accepted, 257 refused; 16 386 points and 1 point refused with the line's index."""
    _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward, _lib
    tiny = np.stack([np.linspace(0, 1, 3), np.zeros(3)], 1)
    rw = ShapedReward(4, centerlines=[tiny + k for k in range(256)], num_beams=8)
    assert _lib.load().f110_reward_count(rw.h) == 256
    rw.close()
    L = _lib.load()
    cfg = _lib.F110RewardConfig(num_envs=4, num_beams=8)
    for lines, count, msg in (([tiny] * 257, 257, '257 centerlines'), ([tiny, np.zeros((16386, 2))], 2, 'centerline 1 has 16386'),
                              ([tiny, tiny, tiny[:1]], 3, 'centerline 2 has 1 points')):
        arr, keep = _lines_c(lines)
        h = C.c_void_p()
        assert L.f110_reward_create_set(C.byref(cfg), arr, count, C.byref(h)) == _lib.F110_ERR_INVALID
        assert msg in L.f110_last_error().decode()
    with pytest.raises(ValueError, match='closed'):
        ShapedReward(4, centerlines=[tiny, tiny], closed=[True], num_beams=8)


def _carry(xy_or_poses, origin_from, origin_to):
    """Points (or poses, yaw in column 2) of one map frame carried to the same map installed at another origin."""
    a = xy_or_poses.copy()
    d = origin_to[2] - origin_from[2]
    c, s = np.cos(d), np.sin(d)
    x, y = a[..., 0] - origin_from[0], a[..., 1] - origin_from[1]
    a[..., 0] = origin_to[0] + c * x - s * y
    a[..., 1] = origin_to[1] + s * x + c * y
    if a.shape[-1] == 3:
        a[..., 2] += d
    return a


@pytest.mark.gpu
@pytest.mark.parametrize('cuda_graph', [False, True])
def test_device_rollout_on_a_map_set(cuda_graph):
    """Two-car envs on Shanghai and on the same map installed again at another origin (the scans_rotated one), each slot
    with its centerline carried into that frame.  At step 25 a third of the envs move to the other map (reassign).  The
    rollout's reward equals single-line rewards driven by hand with the same observations, restarted at episode starts
    and slot changes; reset steps give 0."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import Actor, DeviceRollout, F110VecEnv, ShapedReward, workloads
    N, T = 48, 50
    dt, res, org = H.golden_map('Shanghai_map')
    org2 = [float(v) for v in H.load('scans_rotated')['origin']]
    cl = H.load('reward')['centerline']
    cl2 = cl.copy()
    cl2[:, :2] = _carry(cl[:, :2], org, org2)
    slots = (np.arange(N) * 2) // N
    base = workloads.start_poses(N, 2)
    poses = np.where(slots[:, None, None] == 1, _carry(base, org, org2), base)
    env = F110VecEnv(N, num_agents=2, maps=[(dt, res, org), (dt, res, org2)], outputs=('obs', 'reward', 'terminated', 'scans_f32'),
                     cuda_graph=cuda_graph)
    torch.manual_seed(0)
    actor = Actor(1088, 2, [-0.4189, 0.0], [0.4189, 9.0]).cuda()
    rfn = ShapedReward(N, centerlines=[cl, cl2])
    solo = [ShapedReward(N, cl), ShapedReward(N, cl2)]
    with pytest.raises(ValueError, match='3 centerlines'):
        DeviceRollout(env, actor, reward_fn=ShapedReward(N, centerlines=[cl, cl2, cl]))
    ro = DeviceRollout(env, actor, reward_fn=rfn)
    ro.reset(poses)
    moved = np.arange(N) % 3 == 0
    new_slots = np.where(moved, 1 - slots, slots).astype(np.int32)
    new_poses = np.where(new_slots[:, None, None] == 1, _carry(base, org, org2), base)
    prev = torch.full((N,), -1, dtype=torch.int32, device='cuda')
    first = torch.ones(N, dtype=torch.bool, device='cuda')
    resets = 0
    for t in range(T):
        if t == 25:
            env.reassign(moved.astype(np.uint8), new_slots, new_poses)
        resetting = env.backend.out['terminated'].clone().bool()
        obs, r, term, trunc, info = ro.step()
        cur = env.backend.env_maps()
        restart = (first | resetting | (cur != prev)).to(torch.uint8)
        got = [s(obs.clone(), restart).clone() for s in solo]
        expect = torch.where(cur == 0, got[0], got[1])
        real = ~resetting
        assert torch.all(r[resetting] == 0), t
        assert torch.equal(r[real].view(torch.int64), expect[real].view(torch.int64)), t
        resets += int(resetting.sum())
        prev, first = cur, resetting
    assert np.array_equal(env.backend.env_maps().cpu().numpy(), new_slots)
    assert resets > 0
    for s in [rfn] + solo:
        s.close()
    env.close()
