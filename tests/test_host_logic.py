"""CPU suite for the host side: map/param tables, the gym shim, env-index sharding and the gloo all-reduce of the
episode statistics (world_size 2), and that the C-ABI library loads and exports every declared symbol.
No compute call is made without a GPU."""
import os
import re
import socket
import sys

import numpy as np
import pytest

from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    L = _lib.load()
    hdr = open(os.path.join(ROOT, 'include', 'f110_b200.h')).read()
    declared = set(re.findall(r'\b(f110_[a-z0-9_]+)\s*\(', hdr))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(L, name), name
    assert L.f110_abi_version() == _lib.F110_ABI_VERSION


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from f110_gymnasium_ros2_jazzy_b200 import BatchSim
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        BatchSim(1)
    # and the C entry point itself refuses
    import ctypes as C
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    from f110_gymnasium_ros2_jazzy_b200.params import default_params, params_vector
    L = _lib.load()
    cfg = _lib.F110Config(abi_version=_lib.F110_ABI_VERSION, device=0, num_envs=1, num_agents=1, num_beams=1080,
                          theta_dis=2000, integrator=1, ego_idx=0, fov=4.7, eps=1e-4, max_range=30.0, timestep=0.01,
                          ttc_thresh=0.005, lidar_max=30.0, noise_std=0.01, seed=1)
    h = C.c_void_p()
    pv = params_vector(default_params())
    rc = L.f110_create(C.byref(cfg), pv.ctypes.data_as(C.c_void_p), C.byref(h))
    assert rc == _lib.F110_ERR_NO_DEVICE and not h.value
    assert b"no CPU fallback" in L.f110_last_error()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'f110_gymnasium_ros2_jazzy_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'oracle' not in src.lower().replace('the oracle', ''), os.path.join(dirpath, f)


def test_tables_match_reference_tables():
    from f110_gymnasium_ros2_jazzy_b200.params import beam_tables, default_params, theta_tables
    s, c, a, bc, sd = H.tables()
    ms, mc = theta_tables(2000)
    ma, mbc, msd = beam_tables(default_params(), 1080, 4.7)
    # numpy's sin/cos may differ from the recording machine's by an ulp on another CPU: allow 2 ulp
    for mine, ref in ((ms, s), (mc, c), (ma, a), (mbc, bc), (msd, sd)):
        assert np.allclose(mine, ref, rtol=0, atol=5e-16 * max(1.0, np.abs(ref).max()))
    assert np.array_equal(ma, a)


def test_map_loader_reproduces_reference_dt(tmp_path):
    from f110_gymnasium_ros2_jazzy_b200.maps import load_map, map_bounds
    for name in ('straight_corridor', 'open_square'):
        d, n = H.write_map_files(name, str(tmp_path))
        dt, res, origin = load_map(d + n + '.yaml', '.png')
        gdt, gres, gorigin = H.golden_map(name)
        assert np.array_equal(dt, gdt) and res == gres and origin == gorigin
        x0, x1, y0, y1 = map_bounds(d + n + '.yaml', d)
        assert x1 > x0 and y1 > y0


def test_gym_shim_surface():
    from f110_gymnasium_ros2_jazzy_b200 import gym_compat as g
    box = g.spaces.Box(low=np.zeros((2, 2), np.float32), high=np.ones((2, 2), np.float32), dtype=np.float32)
    x = box.sample()
    assert x.shape == (2, 2) and x.dtype == np.float32 and box.contains(x)
    with pytest.raises(ValueError):
        g.make('nope-v0')


def test_shard_range_partitions():
    from f110_gymnasium_ros2_jazzy_b200 import shard_range
    for n in (1, 7, 4096, 262144):
        for w in (1, 2, 3, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _stats_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from f110_gymnasium_ros2_jazzy_b200.dist import EpisodeStats, shard_range
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    lo, hi = shard_range(10, rank, world)
    local = torch.zeros(8, dtype=torch.float64)
    local[0] = hi - lo            # episodes
    local[1] = 100.0 * (hi - lo)  # steps
    local[2] = rank
    out = EpisodeStats().reduce(local)
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_episode_stats_allreduce_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_stats_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = dict(q.get(timeout=120) for _ in ps)
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r in (0, 1):
        assert res[r]['episodes'] == 10.0 and res[r]['episode_steps'] == 1000.0 and res[r]['ego_collisions'] == 1.0
        assert res[r]['mean_episode_steps'] == 100.0


def test_bench_reference_arm_runs_on_cpu():
    """bench.py --impl reference must work without a GPU and print one JSON line with the contract's keys."""
    import json
    import subprocess
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '2',
                                   '--warmup', '1', '--cpu-envs', '16'], cwd=ROOT, timeout=300)
    line = json.loads(out.decode().strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['unit'] == 'env-steps/s' and line['value'] > 0
    assert line['cpu_baseline']['kind'] == 'port' and line['e2e']['h2d_bytes_per_step'] == 0


def test_bench_dump_outputs_writes_every_returned_array(tmp_path, monkeypatch):
    """bench.py --dump-outputs: each array of a step's return value as <name>.npy, float64 kept, the rest as float32, and
    above the size cap the same seeded sample of envs from every array, named by env_index.npy."""
    import torch
    import bench
    n = 50
    obs, rew = torch.rand((n, 12)), torch.rand(n)
    term, trunc = (torch.arange(n) % 3 == 0).to(torch.uint8), torch.zeros(n, dtype=torch.uint8)
    info = {'obs': obs, 'reward': rew, 'terminated': term, 'state': torch.rand((n, 2, 7), dtype=torch.float64),
            'toggles': torch.arange(2 * n, dtype=torch.int32).reshape(n, 2)}
    bench.dump_outputs(str(tmp_path / 'all'), (obs, rew, term, trunc, info), torch)
    got = {f[:-4]: np.load(str(tmp_path / 'all' / f)) for f in os.listdir(str(tmp_path / 'all'))}
    assert sorted(got) == ['env_index', 'obs', 'reward', 'state', 'terminated', 'toggles', 'truncated']
    assert got['state'].dtype == np.float64 and np.array_equal(got['state'], info['state'].numpy())
    assert got['toggles'].dtype == np.float32 and np.array_equal(got['toggles'], info['toggles'].numpy())
    assert np.array_equal(got['terminated'], term.numpy()) and np.array_equal(got['env_index'], np.arange(n))
    row = 8 + 4 * 12 + 4 + 4 + 4 + 8 * 14 + 4 * 2
    cap = 20 * row + 7 * bench.NPY_HEADER_BYTES           # 7 files
    monkeypatch.setattr(bench, 'DUMP_BYTES', cap)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), (obs, rew, term, trunc, info), torch)
    keep = np.load(str(tmp_path / 'a' / 'env_index.npy')).astype(int)
    assert len(keep) == 20 and np.array_equal(keep, np.load(str(tmp_path / 'b' / 'env_index.npy')))
    assert sum(os.path.getsize(str(tmp_path / 'a' / f)) for f in os.listdir(str(tmp_path / 'a'))) <= cap
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'obs.npy')), obs.numpy()[keep])
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'state.npy')), info['state'].numpy()[keep])


def test_bind_host_to_gpu_uses_the_gpus_numa_node(tmp_path):
    """bind_host_to_gpu reads <sysfs>/bus/pci/devices/<id>/numa_node and node<N>/cpulist; here against a fake sysfs."""
    import os
    from f110_gymnasium_ros2_jazzy_b200.dist import _parse_cpulist, bind_host_to_gpu
    assert _parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    before = os.sched_getaffinity(0)
    if len(before) < 2:
        pytest.skip("needs two CPUs")
    keep = sorted(before)[: len(before) // 2]
    dev = tmp_path / "bus/pci/devices/0000:1b:00.0"
    dev.mkdir(parents=True)
    (dev / "numa_node").write_text("1\n")
    node = tmp_path / "devices/system/node/node1"
    node.mkdir(parents=True)
    (node / "cpulist").write_text(",".join(str(c) for c in keep) + "\n")
    try:
        prev = bind_host_to_gpu(0, pci_bus_id="0000:1B:00.0", sysfs=str(tmp_path))
        assert prev == before and os.sched_getaffinity(0) == set(keep)
        # no NUMA information (-1) or an unknown device: nothing changes
        (dev / "numa_node").write_text("-1\n")
        assert bind_host_to_gpu(0, pci_bus_id="0000:1b:00.0", sysfs=str(tmp_path)) is None
        assert bind_host_to_gpu(0, pci_bus_id="0000:ff:00.0", sysfs=str(tmp_path)) is None
    finally:
        os.sched_setaffinity(0, before)


def test_device_replay_buffer_ring_and_per_formulas():
    """DeviceReplayBuffer (torch tensors, here on the CPU) against the reference's PrioritizedExperienceReplayBuffer
    formulas (rl_training/DDPG/replay_buffer.py:46-135): ring insertion, new-transition priority = current max,
    sampling probabilities, importance weights, priority clamping."""
    import torch
    from f110_gymnasium_ros2_jazzy_b200.rollout import DeviceReplayBuffer
    buf = DeviceReplayBuffer(capacity=10, batch_size=4, obs_dim=3, act_dim=2, alpha=0.6, device='cpu', seed=1)
    def batch(n, base):
        o = torch.arange(n * 3, dtype=torch.float32).reshape(n, 3) + base
        return o, torch.ones(n, 2) * base, torch.full((n,), float(base)), o + 0.5, torch.zeros(n, dtype=torch.uint8)
    buf.add(*batch(4, 100))
    assert len(buf) == 4 and buf.next_idx == 4 and torch.all(buf.priority[:4] == 1.0)
    buf.update_priorities([1, 2], [5.0, float('nan')])
    assert buf.priority[1] == 5.0 and abs(float(buf.priority[2]) - 1e-6) < 1e-12
    buf.add(*batch(8, 200))                                  # wraps: slots 4..9 then 0..1
    assert len(buf) == 10 and buf.next_idx == 2
    assert torch.all(buf.priority[4:10] == 5.0) and torch.all(buf.priority[0:2] == 5.0)    # new ones get the running max
    assert float(buf.reward[0]) == 200.0 and float(buf.reward[3]) == 100.0
    # probabilities and weights, restated in numpy exactly as the reference computes them
    ps = buf.priority[:10].numpy().astype(np.float32)
    pa = np.power(ps + 1e-6, 0.6, dtype=np.float64)
    want = pa / pa.sum()
    assert np.allclose(buf.probabilities().numpy(), want, rtol=1e-12, atol=0)
    idxs, (o, a, r, no, d), w = buf.sample(beta=0.4)
    assert len(set(idxs.tolist())) == 4                       # without replacement once a batch fits
    wr = np.power(10 * want[idxs.numpy()], -0.4)
    assert np.allclose(w.numpy(), (wr / wr.max()).astype(np.float32), rtol=1e-6)
    assert torch.equal(o, buf.obs[idxs]) and torch.equal(no, buf.next_obs[idxs]) and w.dtype == torch.float32
    small = DeviceReplayBuffer(capacity=8, batch_size=4, obs_dim=3, device='cpu')
    with pytest.raises(ValueError):
        small.sample()
    small.add(*batch(2, 1))
    assert small.sample()[0].shape == (4,)                    # fewer than a batch stored: with replacement
    # clamping (replay_buffer.py:120-135): +inf -> float32 max, tiny -> 1e-8; the probabilities stay finite
    small.update_priorities([0, 1], [float('inf'), 1e-12])
    assert float(small.priority[0]) == np.finfo(np.float32).max and float(small.priority[1]) == float(np.float32(1e-8))
    p = small.probabilities().numpy()
    assert np.isfinite(p).all() and abs(p.sum() - 1.0) < 1e-12 and p[0] > 0.999


def test_f110_gym_alias_resolves_like_gymnasium():
    """gym.make('f110_gym:f110-v0', ...) -- the id string of train_ddpg.py:58 and gym_bridge.py:77 -- imports a module called
    f110_gym and looks the id up afterwards (f110_gymnasium/gym/f110_gym/__init__.py:1-5).  The alias package at the repository
    root must register the id with an entry point that is the B200 F110Env, and f110_gym.envs must export the classes the
    reference's does."""
    import importlib
    for name in [k for k in sys.modules if k == "f110_gym" or k.startswith("f110_gym.")]:
        del sys.modules[name]                      # (the differential tests load the REFERENCE's package under this name)
    import f110_gym
    import f110_gym.envs as envs
    assert f110_gym.__file__.startswith(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from f110_gymnasium_ros2_jazzy_b200 import F110Env, Integrator, Simulator, gym_compat
    assert envs.F110Env is F110Env and envs.Simulator is Simulator and envs.Integrator is Integrator
    assert hasattr(envs, 'RaceCar')
    if gym_compat.HAVE_GYMNASIUM:
        import gymnasium
        spec = gymnasium.spec('f110-v0')
        entry = spec.entry_point
    else:
        entry, _ = gym_compat._REGISTRY['f110-v0']
    mod, _, attr = entry.partition(':')
    assert getattr(importlib.import_module(mod), attr) is F110Env
    with pytest.raises(Exception):
        gym_compat.make('f110_gym:no-such-env-v0')
    for name in [k for k in sys.modules if k == "f110_gym" or k.startswith("f110_gym.")]:
        del sys.modules[name]


def test_package_workload_data_equals_the_golden_fixture():
    """The Shanghai map and centerline the package ships for bench.py / smoke() are the arrays recorded from the reference."""
    from f110_gymnasium_ros2_jazzy_b200 import workloads
    g = H.load('maps')
    free, res, origin = workloads.shanghai_free_mask()
    shape = tuple(int(v) for v in g['Shanghai_map__shape'])
    assert np.array_equal(np.packbits(free, axis=None), g['Shanghai_map__bits']) and free.shape == shape
    assert res == float(g['Shanghai_map__resolution']) and origin == [float(v) for v in g['Shanghai_map__origin']]
    assert np.array_equal(workloads.centerline_poses(), g['Shanghai_map__centerline_poses'])
    dt, _, _ = workloads.shanghai_map()
    assert np.array_equal(dt, H.golden_map('Shanghai_map')[0])
    p = workloads.start_poses(16, 2, env_offset=4, total_envs=64)
    assert p.shape == (16, 2, 3) and np.array_equal(p[0, 0], g['Shanghai_map__centerline_poses'][np.linspace(0, 6686, 64).round().astype(int)[4]])
