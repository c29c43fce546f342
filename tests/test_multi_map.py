"""Map sets: several maps in one handle, each env on the map of its slot (f110_set_maps, DESIGN.md section 10).

GPU tests hold every env of a set handle to what a single-map handle holding that env's map produces, bit for bit, and
to the reference's scans at the bar of the single-map scan tests.  CPU tests: static guards on the compiled
lidar_maps_kernel (the same bars test_kernel_shape.py keeps on lidar_kernel) and argument checks that need no device."""
import re

import numpy as np
import pytest

from tests import helpers as H

SCAN_TOL = 1e-6
SCAN_FRAC = 0.999


# ----------------------------------------------------------------------------- CPU: static guards on lidar_maps_kernel

def _maps_variants():
    from tests.test_kernel_shape import CUOBJDUMP, _functions
    if not CUOBJDUMP:
        pytest.skip("cuobjdump neither on PATH nor under CUDA_HOME")
    fns = _functions(["-sass"])
    res = _functions(["-res-usage"])
    pick = lambda d: {k: v for k, v in d.items() if "lidar_maps_kernel" in k}
    return pick(fns), pick(res)


def test_lidar_maps_kernel_register_budget():
    _, res = _maps_variants()
    assert len(res) == 40                                       # fraction bits {generic, 19..22} x COUNT x MODE, like lidar_kernel
    for name, lines in res.items():
        text = " ".join(lines)
        assert int(re.search(r"REG:(\d+)", text).group(1)) <= 40, name
        assert int(re.search(r"LOCAL:(\d+)", text).group(1)) <= 128, name


def test_lidar_maps_kernel_hot_loop():
    fns, _ = _maps_variants()
    assert len(fns) == 40
    for name, lines in fns.items():
        ins = []
        for line in lines:
            m = re.search(r"/\*([0-9a-f]{4,5})\*/\s+(.*?);", line)
            if m:
                ins.append((int(m.group(1), 16), m.group(2)))
        loops = []
        for addr, text in ins:
            m = re.search(r"BRA\s+(?:P\d,\s*)?(?:`\(\.L_x_\d+\)|0x([0-9a-f]+))", text)
            if m and m.group(1) and int(m.group(1), 16) < addr:
                body = [t for a, t in ins if int(m.group(1), 16) <= a <= addr]
                if any("F2I.U32.F64" in t for t in body) and any("LDG" in t for t in body):
                    loops.append(body)
        assert loops, name
        hot = min(loops, key=len)
        assert not any("CALL" in t for t in hot), name
        assert not any(("LDL" in t) or ("STL" in t) for t in hot), name
        lookups = sum("LDG" in t for t in hot)
        assert lookups in (1, 2), (name, lookups)
        tuned = "lidar_maps_kernelILi0E" not in name
        assert len(hot) / lookups <= (21 if tuned else 34), (name, len(hot), lookups)
        if tuned:
            assert sum(("LDC" in t) or ("LDCU" in t) for t in hot) <= 1, name


def test_vec_env_refuses_a_map_and_a_map_set():
    from f110_gymnasium_ros2_jazzy_b200 import F110VecEnv
    with pytest.raises(ValueError):
        F110VecEnv(4, map_arrays=H.golden_map('open_square'), maps=[H.golden_map('open_square')])


# ----------------------------------------------------------------------------- GPU

def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _golden_free(name):
    m = H.load('maps')
    shape = tuple(int(v) for v in m[name + '__shape'])
    free = np.unpackbits(m[name + '__bits'])[:shape[0] * shape[1]].reshape(shape).astype(bool)
    return free, float(m[name + '__resolution']), [float(v) for v in m[name + '__origin']]


def _sim(n, a=1, outputs=None, **kw):
    """BatchSim with the reference's own sin / cos and beam tables (the fixtures' tables)."""
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, BatchSim
    sim = BatchSim(n, a, outputs=outputs or ALL_OUTPUTS, **kw)
    s, c, ang, bc, sd = H.tables()
    sim.set_tables(s, c)
    sim.set_beam_tables(ang, bc, sd)
    return sim


def _scan_once(sim, poses):
    import torch
    sim.sim_reset(poses[:, None, :])
    o = sim.step(None, np.zeros((len(poses), 1, 1080)))
    torch.cuda.synchronize()
    return o['scans_f64'].cpu().numpy()[:, 0].copy()


@pytest.mark.gpu
def test_reference_scans_through_one_handle():
    """Seven maps in one set -- Shanghai_x4 makes it 19 fraction bits for all -- one env per recorded reference pose, each on
    its own map; one noise-free step.  Every map is held to the bar of its single-map scan test, and every env equals a
    single-map handle of its map bit for bit.  Then again with the envs interleaved, and after a reassignment that permutes
    the slots."""
    torch = _torch()
    g, gl, gr = H.load('scans'), H.load('scans_large'), H.load('scans_rotated')
    sh = H.golden_map('Shanghai_map')
    members = [  # (map, poses, reference scans, bit-exact against the reference)
        (sh, g['Shanghai_map__poses'], g['Shanghai_map__scans'], False),
        (H.golden_map('straight_corridor'), g['straight_corridor__poses'], g['straight_corridor__scans'], False),
        (H.golden_map('open_square'), np.zeros((0, 3)), np.zeros((0, 1080)), False),
    ]
    for name in ('levine', 'Shanghai_x2_rot', 'Shanghai_x4'):
        dt, res, origin, poses, ref = H.large_map(name)
        members.append(((dt, res, origin), poses, ref, not name.endswith('_rot')))
    members.append(((sh[0], sh[1], [float(v) for v in gr['origin']]), gr['poses'], gr['scans'], False))
    K = len(members)
    slots = np.concatenate([np.full(len(p), k) for k, (_, p, _, _) in enumerate(members)]).astype(np.int32)
    poses = np.concatenate([p for _, p, _, _ in members])
    refs = np.concatenate([r for _, _, r, _ in members])
    n = len(poses)
    # what a single-map handle of each map gives
    want = np.zeros((n, 1080))
    for k, (m, p, _, _) in enumerate(members):
        if len(p):
            one = _sim(len(p), noise_std=0.0)
            one.set_map_arrays(*m)
            want[slots == k] = _scan_once(one, p)
            one.close()
    sim = _sim(n, noise_std=0.0)
    sim.set_maps([m for m, _, _, _ in members])
    assert sim.num_maps == K

    def check(order):
        # env j drives pose order[j] on its map
        sim.set_env_maps(slots[order])
        assert np.array_equal(sim.env_maps().cpu().numpy(), slots[order])
        got = _scan_once(sim, poses[order])
        assert np.array_equal(got, want[order])
        for k, (_, _, _, exact) in enumerate(members):
            sel = slots[order] == k
            if not sel.any():
                continue
            d = np.abs(got[sel] - refs[order][sel])
            assert (d <= SCAN_TOL).mean() >= SCAN_FRAC, (k, d.max())
            if exact:
                assert d.max() == 0.0, k

    check(np.arange(n))                                            # blocks
    check(np.argsort(np.arange(n) % 7, kind='stable'))             # interleaved
    check(np.random.default_rng(3).permutation(n))                 # a reassignment that permutes the envs' slots
    sim.close()


def _start_poses(name, n, a, rng):
    """Valid start poses on a map: Shanghai's centerline rows, or a golden rollout's start poses with seeded jitter."""
    from f110_gymnasium_ros2_jazzy_b200 import workloads
    if name == 'Shanghai_map':
        return workloads.start_poses(n, a)
    base = H.load({'open_square': 'rollout_circles_open', 'straight_corridor': 'rollout_corridor'}[name])['poses'][:a]
    p = np.broadcast_to(base, (n, a, 3)).copy()
    p[..., :2] += rng.normal(0, 0.05, size=(n, a, 2))
    p[..., 2] += rng.normal(0, 0.05, size=(n, a))
    return p


ROLLOUT_MAPS = ('Shanghai_map', 'open_square', 'straight_corridor')


def _rollout_inputs(N, A, slots, seed=0):
    rng = np.random.default_rng(seed)
    poses = np.zeros((N, A, 3))
    for k, name in enumerate(ROLLOUT_MAPS):
        sel = slots == k
        poses[sel] = _start_poses(name, int(sel.sum()), A, rng)
    return poses


def _eq(a, b):
    import torch
    if a.dtype.is_floating_point:
        a, b = a.contiguous().view(torch.int32 if a.element_size() == 4 else torch.int64), \
            b.contiguous().view(torch.int32 if b.element_size() == 4 else torch.int64)
    return bool(torch.equal(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("N,A,fast", [(512, 2, False), (512, 1, False), (512, 1, True), (32768, 1, True)])
def test_rollout_bit_identical_to_single_map_handles(N, A, fast):
    """300 steps, random actions, device noise, auto-reset: env e of the set handle equals, every step and in every output,
    a single-map handle of its map that steps the same N envs with active_mask = (slot == k).  Lookups and rays of the set
    handle are the sums over the single-map handles."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, FAST_OUTPUTS
    outs = FAST_OUTPUTS if fast else ALL_OUTPUTS
    K = len(ROLLOUT_MAPS)
    slots = (np.arange(N) * K) // N
    poses = torch.as_tensor(_rollout_inputs(N, A, slots), device='cuda')
    maps = [H.golden_map(n) for n in ROLLOUT_MAPS]
    count = N <= 4096
    st = _sim(N, A, outputs=outs, count_lookups=count)
    st.set_maps(maps)
    singles, masks = [], []
    for k in range(K):
        one = _sim(N, A, outputs=outs, count_lookups=count)
        one.set_map_arrays(*maps[k])
        singles.append(one)
        masks.append(torch.as_tensor((slots == k).astype(np.uint8), device='cuda'))
    sel = [torch.as_tensor(slots == k, device='cuda') for k in range(K)]
    gen = torch.Generator(device='cuda').manual_seed(1)
    lo = torch.tensor([-0.4, 0.0], device='cuda', dtype=torch.float32)
    span = torch.tensor([0.8, 6.0], device='cuda', dtype=torch.float32)
    st.reset(poses)
    for k in range(K):
        singles[k].reset(poses, env_mask=masks[k])
    for t in range(301):
        if t:
            act = torch.rand((N, A, 2), generator=gen, device='cuda') * span + lo
            st.step(act, None, reset_mask=st.out['terminated'], reset_poses=poses)
            for k in range(K):
                singles[k].step(act, None, reset_mask=singles[k].out['terminated'], reset_poses=poses, active_mask=masks[k])
        for key in outs:
            for k in range(K):
                assert _eq(st.out[key][sel[k]], singles[k].out[key][sel[k]]), (t, key, k)
    torch.cuda.synchronize()
    if count:
        look, rays = st.lookup_count()
        parts = [s.lookup_count() for s in singles]
        assert look == sum(p[0] for p in parts) and rays == sum(p[1] for p in parts)
    for s in [st] + singles:
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cuda_graph", [False, True])
def test_reassign_at_reset(cuda_graph):
    """Mid-rollout a third of the envs move to another map with new start poses (F110VecEnv.reassign), eagerly and under a
    captured CUDA graph (no re-capture): equal to single-map handles that reset those envs at the same step.  reassign
    leaves map_generation alone; set_maps bumps it."""
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, F110VecEnv
    N, A, K = 384, 2, len(ROLLOUT_MAPS)
    maps = [H.golden_map(n) for n in ROLLOUT_MAPS]
    slots = (np.arange(N) * K) // N
    poses = _rollout_inputs(N, A, slots)
    from f110_gymnasium_ros2_jazzy_b200 import BatchSim
    env = F110VecEnv(N, num_agents=A, maps=maps, outputs=ALL_OUTPUTS, cuda_graph=cuda_graph)
    singles = []
    for k in range(K):
        one = BatchSim(N, A, seed=42, noise_std=0.01, outputs=ALL_OUTPUTS)     # the vec env's settings and tables
        one.set_map_arrays(*maps[k])
        singles.append(one)
    gen0 = env.backend.map_generation
    env.reset(poses)
    dposes = torch.as_tensor(poses, device='cuda')
    cur = slots.copy()
    for k in range(K):
        singles[k].reset(dposes, env_mask=torch.as_tensor((cur == k).astype(np.uint8), device='cuda'))
    gen = torch.Generator(device='cuda').manual_seed(2)
    lo = torch.tensor([-0.4, 0.0], device='cuda')
    span = torch.tensor([0.8, 6.0], device='cuda')
    moved = np.arange(N) % 3 == 0
    new_slots = np.where(moved, (slots + 1) % K, slots)
    new_poses = _rollout_inputs(N, A, new_slots, seed=5)
    starts = dposes.clone()
    for t in range(1, 121):
        extra = None
        if t == 60:
            env.reassign(moved.astype(np.uint8), new_slots.astype(np.int32), new_poses)
            cur = new_slots
            starts = torch.where(torch.as_tensor(moved, device='cuda')[:, None, None], torch.as_tensor(new_poses, device='cuda'), starts)
            extra = torch.as_tensor(moved.astype(np.uint8), device='cuda')
        act = torch.rand((N, A, 2), generator=gen, device='cuda') * span + lo
        env.step(act)
        for k in range(K):
            m = torch.as_tensor((cur == k).astype(np.uint8), device='cuda')
            rm = singles[k].out['terminated'] if extra is None else singles[k].out['terminated'] | extra
            singles[k].step(act, None, reset_mask=rm, reset_poses=starts, active_mask=m)
        o = env.backend.out
        for key in ALL_OUTPUTS:
            for k in range(K):
                s = torch.as_tensor(cur == k, device='cuda')
                assert _eq(o[key][s], singles[k].out[key][s]), (t, key, k)
    assert np.array_equal(env.backend.env_maps().cpu().numpy(), new_slots)
    assert env.backend.map_generation == gen0
    if cuda_graph:
        assert env._graph is not None
    env.set_maps(maps)
    assert env.backend.map_generation == gen0 + 1
    env.close()
    for s in singles:
        s.close()


@pytest.mark.gpu
def test_set_construction_limits_and_slots():
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    from scipy.ndimage import distance_transform_edt
    # mixed dt and free-mask specs: each slot's map is scipy's EDT bit for bit
    free_o, res_o, org_o = _golden_free('open_square')
    free_c, res_c, org_c = _golden_free('straight_corridor')
    sim = _sim(64, noise_std=0.0)
    sim.set_maps([(free_o, res_o, org_o), H.golden_map('straight_corridor'), (free_c.astype(np.uint8), res_c, org_c)])
    assert sim.num_maps == 3
    assert np.array_equal(sim.get_map(0), res_o * distance_transform_edt(np.where(free_o, 255., 0.)))
    assert np.array_equal(sim.get_map(1), H.golden_map('straight_corridor')[0])
    assert np.array_equal(sim.get_map(2), res_c * distance_transform_edt(np.where(free_c, 255., 0.)))
    assert np.array_equal(sim.env_maps().cpu().numpy(), (np.arange(64) * 3) // 64)
    with pytest.raises(IndexError):
        sim.get_map(3)
    # out-of-range slots: the host form raises and changes nothing, the device form leaves those envs alone
    before = sim.env_maps().cpu().numpy()
    bad = np.zeros(64, np.int32); bad[5] = 3
    with pytest.raises(IndexError):
        sim.set_env_maps(bad)
    assert np.array_equal(sim.env_maps().cpu().numpy(), before)
    dev = torch.full((64,), 2, dtype=torch.int32, device='cuda'); dev[7] = -1; dev[9] = 3
    mask = torch.ones(64, dtype=torch.uint8, device='cuda'); mask[11] = 0
    sim.set_env_maps(dev, mask)
    want = np.full(64, 2); want[[7, 9, 11]] = before[[7, 9, 11]]
    assert np.array_equal(sim.env_maps().cpu().numpy(), want)
    sim.close()
    # limits: the handle keeps its previous map and steps as before
    sh = H.golden_map('Shanghai_map')
    poses = H.load('scans')['Shanghai_map__poses']
    sim = _sim(len(poses), noise_std=0.0)
    sim.set_map_arrays(*sh)
    first = _scan_once(sim, poses)
    gen = sim.map_generation
    tiny = (np.full((4, 4), 0.5), 0.05, [0.0, 0.0, 0.0])
    wide = (np.full((1, 4096), 0.5), 0.05, [0.0, 0.0, 0.0])   # pads every member to 8192 x 8208 cells: 32 exceed 2^31
    huge = (np.full((1, 40000), 0.5), 0.05, [0.0, 0.0, 0.0])  # pads to 65536 x 65552 cells: alone beyond 2^31
    for install in (lambda: sim.set_maps([]), lambda: sim.set_maps([tiny] * (_lib.F110_MAX_MAPS + 1)),
                    lambda: sim.set_maps([wide] * 32), lambda: sim.set_maps([huge]), lambda: sim.set_map_arrays(*huge)):
        with pytest.raises(ValueError):
            install()
        assert sim.num_maps == 1 and sim.map_generation == gen
        assert np.array_equal(_scan_once(sim, poses), first)
    # back to one map: f110_set_map after a set gives what a fresh single-map handle gives
    sim.set_maps([H.golden_map('open_square'), sh])
    assert sim.num_maps == 2 and sim.map_generation == gen + 1
    sim.set_map_arrays(*sh)
    assert sim.num_maps == 1 and np.array_equal(sim.env_maps().cpu().numpy(), np.zeros(len(poses)))
    assert np.array_equal(_scan_once(sim, poses), first)
    sim.close()


@pytest.mark.gpu
def test_a_set_of_one_is_the_single_map():
    """The rotated-origin Shanghai map installed four ways -- set_maps of its dt, set_map_arrays, set_map_image and set_maps
    of its free mask -- gives one map_generation bump, one map, all slots 0, the same map and the single-map kernel each, and
    bit-identical outputs over a 40-step rollout.  set_tables after a set of one rebuilds its direction table: the scans then
    equal those of a fresh handle given the same tables before its map."""
    torch = _torch()
    free, res, _ = _golden_free('Shanghai_map')
    dt = H.golden_map('Shanghai_map')[0]
    gr = H.load('scans_rotated')
    origin = [float(v) for v in gr['origin']]
    N = len(gr['poses'])
    poses = torch.as_tensor(gr['poses'][:, None, :], device='cuda')
    installs = {'set_maps(dt)': lambda s: s.set_maps([(dt, res, origin)]),
                'set_map_arrays': lambda s: s.set_map_arrays(dt, res, origin),
                'set_map_image': lambda s: s.set_map_image(free, res, origin),
                'set_maps(mask)': lambda s: s.set_maps([(free, res, origin)])}
    gen = torch.Generator(device='cuda').manual_seed(6)
    acts = [torch.rand((N, 1, 2), generator=gen, device='cuda') * torch.tensor([0.8, 6.0], device='cuda')
            + torch.tensor([-0.4, 0.0], device='cuda') for _ in range(40)]
    want = None
    for name, install in installs.items():
        sim = _sim(N)
        gen0 = sim.map_generation
        install(sim)
        assert sim.map_generation == gen0 + 1 and sim.num_maps == 1, name
        assert np.array_equal(sim.get_map(0), dt), name
        assert not sim.env_maps().cpu().numpy().any(), name
        outs = [{k: v.clone() for k, v in sim.reset(poses).items()}]
        for a in acts:
            sim.step(a, None, reset_mask=sim.out['terminated'], reset_poses=poses)
            outs.append({k: v.clone() for k, v in sim.out.items()})
        assert sim.lidar_variant()['maps'] == 0, name
        want = outs if want is None else want
        for t, (o, w) in enumerate(zip(outs, want)):
            for k in o:
                assert _eq(o[k], w[k]), (name, t, k)
        sim.close()
    s, c = H.tables()[:2]
    s2, c2 = np.roll(s, 100), np.roll(c, 100)      # every table direction turned by 100 entries
    sim = _sim(N)
    sim.set_maps([(dt, res, origin)])
    before = _scan_once(sim, gr['poses'])
    sim.set_tables(s2, c2)
    fresh = _sim(N)
    fresh.set_tables(s2, c2)
    fresh.set_maps([(dt, res, origin)])
    after = _scan_once(sim, gr['poses'])
    assert np.array_equal(after, _scan_once(fresh, gr['poses']))
    assert not np.array_equal(after, before)
    sim.close(); fresh.close()


@pytest.mark.gpu
def test_checkpoint_resumes_bit_identical():
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import ALL_OUTPUTS, F110VecEnv
    N, A, K = 256, 2, len(ROLLOUT_MAPS)
    maps = [H.golden_map(n) for n in ROLLOUT_MAPS]
    slots = (np.arange(N) * K) // N
    env = F110VecEnv(N, num_agents=A, maps=maps, outputs=ALL_OUTPUTS)
    env.reset(_rollout_inputs(N, A, slots))
    gen = torch.Generator(device='cuda').manual_seed(4)
    acts = [torch.rand((N, A, 2), generator=gen, device='cuda') * torch.tensor([0.8, 6.0], device='cuda')
            + torch.tensor([-0.4, 0.0], device='cuda') for _ in range(80)]
    moved = np.arange(N) % 4 == 1
    for t in range(40):
        if t == 20:
            env.reassign(moved.astype(np.uint8), ((slots + 2) % K).astype(np.int32), _rollout_inputs(N, A, (slots + 2) % K, 7))
        env.step(acts[t])
    sd = env.state_dict()
    a_out = []
    for t in range(40, 80):
        env.step(acts[t])
        a_out.append({k: v.clone() for k, v in env.backend.out.items()})
    env2 = F110VecEnv(N, num_agents=A, maps=maps, outputs=ALL_OUTPUTS)
    env2.load_state_dict(sd)
    assert torch.equal(env2.backend.env_maps(), env.backend.env_maps())
    for t in range(40, 80):
        env2.step(acts[t])
        for k, v in env2.backend.out.items():
            assert _eq(v, a_out[t - 40][k]), (t, k)
    env.close(); env2.close()


@pytest.mark.gpu
def test_host_vec_env_with_a_map_set():
    torch = _torch()
    from f110_gymnasium_ros2_jazzy_b200 import F110VecEnv
    from f110_gymnasium_ros2_jazzy_b200.env import F110HostVecEnv
    N, K = 300, len(ROLLOUT_MAPS)
    maps = [H.golden_map(n) for n in ROLLOUT_MAPS]
    slots = ((np.arange(N) * 7) % K).astype(np.int32)
    poses = _rollout_inputs(N, 1, slots)
    host = F110HostVecEnv(N, chunks=(1, 3), num_agents=1, maps=maps, env_maps=slots, noise_std=0.0)
    dev = F110VecEnv(N, num_agents=1, maps=maps, env_maps=slots, noise_std=0.0)
    ho, _ = host.reset(poses)
    do, _ = dev.reset(poses)
    assert np.array_equal(ho, do.cpu().numpy())
    rng = np.random.default_rng(9)
    for t in range(60):
        a = rng.uniform([-0.4, 0.0], [0.4, 6.0], size=(N, 1, 2)).astype(np.float32)
        hobs, hrew, hterm, _, _ = host.step(a)
        dobs, drew, dterm, _, _ = dev.step(torch.as_tensor(a, device='cuda'))
        assert np.array_equal(hobs, dobs.cpu().numpy()), t
        assert np.array_equal(hrew, drew.cpu().numpy()) and np.array_equal(hterm, dterm.cpu().numpy()), t
    host.close(); dev.close()
