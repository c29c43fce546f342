#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched F110Env step path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--agents A] [--beams B]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      # the CPU arm: oracle port on all host cores
  python bench.py --config c4|c5 ...        # BASELINE configs 4 / 5 (the default is C3)
  python bench.py --dump-outputs DIR ...    # also write what the last timed step returned, DIR/<name>.npy

Workload (config C3 of BASELINE.json / SURVEY 8d): E = 4096 single-agent envs per GPU on the Shanghai map
(2000x2000 cells, 0.06505 m), 1080-beam 270-degree lidar, RK4 single-track dynamics, start poses spread over
the centerline, iid uniform actions in the action-space bounds (pre-generated on the device, torch Philox seed
1234), lidar noise from the on-device Philox stream, auto-reset to the start pose on the step after done.
One "step" = one batched F110Env.step over all E envs of the rank.  Weak scaling: every rank owns E envs.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how every field is obtained.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

S_MIN, S_MAX, V_MIN, V_MAX = -0.4189, 0.4189, 0.0, 20.0   # ddpg_config.yaml:19-20 / f110_env.py action space
L2_BYTES = 126 * 1024 * 1024


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=["c3", "c4", "c5"],
                    help="c3 (default, the metric's configuration): 4096 single-agent envs per GPU.  c4: 262 144 envs in total, sharded "
                         "over the GPUs (combine with --beams 270..4320 and --map-upsample 2|4 for the sweep).  c5: 65 536 two-agent envs "
                         "in total driven by DeviceRollout (actor 1088-128-128-2 + gap-follow opponent, observations consumed on the device)")
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: 4096 for c3, 262144 / N for c4, 65536 / N for c5)")
    ap.add_argument("--agents", type=int, default=1)
    ap.add_argument("--beams", type=int, default=1080)
    ap.add_argument("--map", default="Shanghai_map")
    ap.add_argument("--map-upsample", type=int, default=1, help="nearest-neighbour upsample factor (C4 large maps)")
    ap.add_argument("--cpu-envs", type=int, default=0, help="envs in the CPU sample (0 = auto)")
    ap.add_argument("--cpu-steps", type=int, default=0, help="steps in the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--host-chunks", default="1,3", help="env chunks pipelined by the e2e host path: a count, or relative sizes "
                    "(a small first chunk starts the downloads sooner)")
    ap.add_argument("--pipe-chunks", type=int, default=4, help="env chunks of the e2e send/recv (cross-step pipelined) figure")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the last timed step returned as DIR/<name>.npy "
                    "(rank 0's envs; a seeded sample of them above 64 MiB, see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.config == "c5":
        a.agents = 2
    if a.envs <= 0:
        a.envs = {"c3": 4096, "c4": 262144 // world, "c5": 65536 // world}[a.config]
    return a


def load_workload(args, num_envs, env_offset=0, total_envs=None):
    """Map + start poses from the arrays the package ships (nothing reads /root/reference or tests/ at run time)."""
    from f110_gymnasium_ros2_jazzy_b200 import workloads
    if args.map != "Shanghai_map":
        raise SystemExit("bench.py ships the Shanghai map only (--map-upsample 2|4 gives BASELINE C4's large maps)")
    map_arrays = workloads.shanghai_map(args.map_upsample)
    poses = workloads.start_poses(num_envs, args.agents, env_offset, total_envs or num_envs)
    return map_arrays, poses


def action_stream(torch, steps, n, a, device, seed=1234):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    u = torch.rand((steps, n, a, 2), generator=g, device=device, dtype=torch.float32)
    lo = torch.tensor([S_MIN, V_MIN], device=device)
    hi = torch.tensor([S_MAX, V_MAX], device=device)
    return (lo + u * (hi - lo)).contiguous()


class ClockSampler(object):
    """SM clock and throttle reasons sampled through NVML every ~5 ms in a background thread while the timed
    region runs (nvidia-smi -lms 200 would see one or two samples of a 40 ms region)."""

    def __init__(self, gpu_index):
        import threading
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES: map the CUDA ordinal to the NVML device through its PCI bus id
            import torch
            bus = torch.cuda.get_device_properties(gpu_index).pci_bus_id if hasattr(torch.cuda.get_device_properties(gpu_index), 'pci_bus_id') else None
            h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hi).bus == bus:
                        h = hi
            self.h = h or pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        except Exception:
            self._t = None

    def _loop(self):
        nv = self.nv
        masks = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                 "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, m in masks.items():
                    if r & m:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if self._t is None:
            return out
        self._stop.set()
        self._t.join(timeout=2)
        if self.samples:
            out.update(sm_mhz=float(np.median(self.samples)), reasons=sorted(self.reasons), samples=len(self.samples))
        return out


def cpu_arm(args, steps, warmup, envs=None, threads=None):
    """The reference's CPU implementation of the path: the oracle port (the reference itself is Python/numba and
    cannot travel to the GPU box), all host threads, a bounded sample of the same workload."""
    from oracle.f110_oracle import Oracle
    threads = threads or (os.cpu_count() or 1)
    try:
        threads = min(threads, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    n = envs or args.cpu_envs or max(256, 64 * threads)   # >= 64 envs per thread: amortises the per-step fork/join
    n = min(n, args.envs)
    map_arrays, poses = load_workload(args, n, 0, args.envs)
    o = Oracle(n, args.agents, num_beams=args.beams, noise_std=0.01, seed=42, threads=threads)
    o.set_map_arrays(*map_arrays)
    rng = np.random.default_rng(1234)
    acts = rng.uniform([S_MIN, V_MIN], [S_MAX, V_MAX], size=(steps + warmup, n, args.agents, 2)).astype(np.float32)
    out = o.reset(poses)
    term = out['terminated'].copy()
    for k in range(warmup):
        term = o.step(acts[k], reset_mask=term, reset_poses=poses, want_scans=False)['terminated'].copy()
    look = 0
    t0 = time.perf_counter()
    for k in range(warmup, warmup + steps):
        term = o.step(acts[k], reset_mask=term, reset_poses=poses, want_scans=False)['terminated'].copy()
        look += o.last_lookups
    el = time.perf_counter() - t0
    return dict(value=n * steps / el, seconds=el, envs=n, steps=steps, threads=threads,
                lookups_per_ray=look / float(n * steps * args.agents * args.beams))


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # size the sample so that W+K steps finish in a couple of minutes on any box
    probe = cpu_arm(args, 2, 1)
    per_step = probe['seconds'] / 2
    budget = 60.0
    envs = probe['envs']
    if per_step * (args.steps + args.warmup) > budget:
        envs = max(8, int(envs * budget / (per_step * (args.steps + args.warmup))))
    r = cpu_arm(args, args.steps, args.warmup, envs=envs)
    rays = r['value'] * args.agents * args.beams
    line = {
        "impl": "reference", "metric": "env-steps/s (1080-beam lidar)", "value": r['value'], "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r['seconds'] / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "rays_per_s": rays,
        "config": workload_config(args, r['envs'], note="CPU arm: bounded sample of the same workload"),
        "cpu_baseline": {"value": r['value'], "unit": "env-steps/s", "cores": r['threads'], "kind": "port",
                         "sample": "%d envs x %d steps of the C3 workload (oracle/f110_oracle.c, pthreads)" % (r['envs'], r['steps'])},
        "e2e": {"value": r['value'], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def workload_config(args, envs_per_gpu, note=None):
    names = {"c3": "C3", "c4": "C4", "c5": "C5"}
    what = ("%d single-agent f110-v0 envs per GPU" % envs_per_gpu) if args.agents == 1 else \
           ("%d %d-agent f110-v0 envs per GPU" % (envs_per_gpu, args.agents))
    extra = ", DeviceRollout: actor 1088-128-128-2 + gap-follow opponent on the device" if args.config == "c5" else ""
    c = {"workload": "%s: %s, %s%s, RK4 ST dynamics, %d-beam 4.7 rad lidar, uniform random actions, auto-reset on done%s"
                     % (names[args.config], what, args.map, "" if args.map_upsample == 1 else " x%d" % args.map_upsample, args.beams, extra),
         "envs_per_gpu": envs_per_gpu, "agents": args.agents, "beams": args.beams, "map": args.map,
         "map_upsample": args.map_upsample, "parallelism": "env-index sharding, no step-path collective"}
    if note:
        c["note"] = note
    return c


def emit(line):
    """The one JSON line, on the process's ORIGINAL stdout (see main)."""
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


_JSON_OUT = sys.stdout


def numba_reference():
    """The baseline north_star names -- the unmodified numba reference under a one-process-per-core lock-step vector runner --
    as measured in the BUILD CONTAINER by tools/numba_reference_baseline.py (numba and /root/reference do not exist on the
    GPU box).  Reported beside the in-run C-port figure, labelled as what it is."""
    p = os.path.join(ROOT, "profiles", "numba_reference.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    r = next((x for x in d["results"] if x["shape"] == "sim1" and x["workers"] > 1), None)
    if r is None:
        return None
    return {"value": r["env_steps_per_s"], "unit": "env-steps/s", "cores": r["workers"], "per_core": r["env_steps_per_s_per_core"],
            "where": d["where"], "runner": d["runner"], "shape": "Simulator.step, 1 agent (the C3 shape), scan + pose returned",
            "source": "profiles/numba_reference.json (tools/numba_reference_baseline.py)"}


def fabric_probe(torch, dist, dev, world, nbytes, iters=40):
    """Bare device->host copy of one step's download (same bytes, pinned destination), every rank at once, no kernels: the
    ceiling of the e2e figure on this box.  -> GB/s of this rank (max over nothing: the caller gathers)."""
    d = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
    h = torch.zeros(nbytes, dtype=torch.uint8, pin_memory=True)
    for _ in range(5):
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    return iters * nbytes / (time.perf_counter() - t0) / 1e9


def main():
    # Libraries write to fd 1 behind Python's back (NCCL prints its version banner there when NCCL_DEBUG is set in the
    # environment).  Keep the original stdout for the JSON line and point fd 1 at stderr for everything else.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        return reference_main(args)

    import torch
    import torch.distributed as dist
    import __graft_entry__
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device; there is no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()

    from f110_gymnasium_ros2_jazzy_b200 import EpisodeStats, F110VecEnv, shard_range
    E, A, B, K, W = args.envs, args.agents, args.beams, args.steps, args.warmup
    total_envs = E * world
    lo, hi = shard_range(total_envs, rank, world)
    map_arrays, poses = load_workload(args, hi - lo, lo, total_envs)
    rollout = args.config == "c5"
    outputs = ('obs', 'reward', 'terminated', 'scans_f32') if rollout else ('obs', 'reward', 'terminated')

    def make_env(count=False):
        env = F110VecEnv(E, num_agents=A, num_beams=B, seed=42 + rank, device=local, auto_reset=True,
                         outputs=outputs, noise_std=0.01, count_lookups=count, map_arrays=map_arrays)
        env.reset(poses)
        return env

    env = make_env()
    acts = None if rollout else action_stream(torch, W + K, E, A, dev, seed=1234 + rank)
    ro = None
    if rollout:
        from f110_gymnasium_ros2_jazzy_b200 import Actor, DeviceRollout
        torch.manual_seed(42)
        ro = DeviceRollout(env, Actor(B + 8, 2, [S_MIN, V_MIN], [S_MAX, V_MAX]).to(dev))
        ro.reset(poses)
    flush = None if args.no_flush else torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    def run(env, first, n, per_step_events=None, flush_buf=None):
        """-> what the last of the n steps returned."""
        result = None
        for k in range(first, first + n):
            if flush_buf is not None:
                flush_buf.fill_(k & 0xFF)          # evict L2 (252 MiB written) before every timed step
            if per_step_events is not None:
                per_step_events[k - first][0].record(stream)
            if ro is not None:
                result = ro.step()
            else:
                result = env.step(acts[k])
            if per_step_events is not None:
                per_step_events[k - first][1].record(stream)
        return result

    # ---- warm-up, then the timed region: K steps, device-timed per step so the flush is not counted
    run(env, 0, W, None, flush)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    launches0 = env.backend.kernel_launches
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    last = run(env, W, K, ev, flush)
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    launches = env.backend.kernel_launches - launches0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    dev_ms = float(sum(step_ms))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, torch)       # before kernel_breakdown steps this env again
    if world > 1:
        dist.barrier()
        t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    stats = EpisodeStats().reduce(env.backend.stats())   # the path's only collective, off the step path

    # ---- e2e on every rank: host buffers in and out through f110_step_host_async/f110_host_sync, and beside it the bare
    # device->host copy of the same bytes on every rank at once (what the box's host fabric gives, no kernels)
    e2e = None
    if not args.no_e2e and not rollout:
        el, el_pipe = e2e_run(args, map_arrays, poses, acts, W, K, E, A, B, local, torch)
        d2h_bytes = E * (B + 8) * 4 + E * 4 + E
        fab = torch.tensor([fabric_probe(torch, dist, dev, world, d2h_bytes)], dtype=torch.float64, device=dev)
        fab_all = [float(fab)]
        if world > 1:
            dist.barrier()
            t = torch.tensor([el, el_pipe], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            el, el_pipe = float(t[0].item()), float(t[1].item())
            g = [torch.zeros_like(fab) for _ in range(world)]
            dist.all_gather(g, fab)
            fab_all = [float(x) for x in g]
        floor_ms = 1e3 * d2h_bytes / (min(fab_all) * 1e9)
        e2e = {"value": total_envs * K / el, "unit": "env-steps/s", "h2d_bytes_per_step": E * A * 2 * 4 + E + E * A * 3 * 8,
               "d2h_bytes_per_step": d2h_bytes, "ms_per_step": 1e3 * el / K, "n_gpus": world,
               "api": "F110HostVecEnv.step -> f110_step_host_async + f110_host_sync (C ABI, pinned host buffers, env chunks %s)" % args.host_chunks,
               "bytes_are": "per GPU",
               "fabric": {"what": "bare cudaMemcpyAsync device->host of d2h_bytes_per_step into pinned memory, all %d ranks at once, no kernels" % world,
                          "d2h_gbs_per_rank": [round(x, 1) for x in fab_all], "d2h_gbs_aggregate": round(sum(fab_all), 1),
                          "download_floor_ms_per_step": floor_ms, "value_ceiling": total_envs / (floor_ms * 1e-3),
                          "frac_of_ceiling": (total_envs * K / el) / (total_envs / (floor_ms * 1e-3)),
                          "note": "the slowest rank's bare copy bounds a synchronous step from below; see profiles/r02_d2h_fabric.json "
                                  "for the 1 vs 8 rank figures (54.7 -> 12.0 GB/s per rank on this pool's boxes)"},
               "pipelined": {"value": total_envs * K / el_pipe, "ms_per_step": 1e3 * el_pipe / K,
                             "chunks": args.pipe_chunks,
                             "api": "F110HostVecEnv.send/recv per chunk (same copies per step; chunks out of phase across "
                                    "step boundaries, EnvPool-style) -- not the headline, which stays the synchronous step()"}}

    value = total_envs * K / (dev_ms * 1e-3)
    rays_per_s = value * A * B

    # ---- everything below runs on rank 0 ALONE: the other ranks leave now instead of spinning in a barrier (an NCCL barrier
    # is a busy wait that took host cores from the CPU arm and put a 100 % "busy" GPU beside an idle rank 0 in round 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        env.close()
        return 0

    # ---- roofline of the dominant kernel (lidar ray-march): kernel-only time via the library's event pairs
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    if ro is not None:
        acts = action_stream(torch, W + min(K, 50), E, A, dev, seed=1234 + rank)
    lidar_ms, kern_ms = kernel_breakdown(env, acts, W, min(K, 50), flush, torch)
    cenv = make_env(count=True)
    for k in range(W + min(K, 50)):
        cenv.step(acts[k])
    looks, rays = cenv.backend.lookup_count()
    max_lookups = cenv.backend.max_lookups
    redone_rays = cenv.backend.redone_rays
    cenv.close()
    lbar = looks / max(rays, 1)
    # SURVEY 8d: bytes_per_ray = L-bar * s_cell + s_out, with s_cell = 8 (the reference's fp64 cell) and s_out = what this
    # launch actually stores per ray: the f32 observation (4 B) here; + 4 / + 8 when the f32 / f64 scans are requested too.
    s_out = 4.0 + (4.0 if 'scans_f32' in outputs else 0.0)
    bytes_per_ray = 8.0 * lbar + s_out
    alg_bytes = bytes_per_ray * E * A * B                 # per launch
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (lidar_ms * 1e-3) / 1e9
    gather = gather_roofline(map_arrays[0], E * A * B, lbar, torch, dev)
    step_ms_unevented = dev_ms / K
    roofline = {"bound": "l2-gather",
                "bound_note": "the cells a launch touches stay in L2 (DRAM traffic is ~1 % of the algorithmic bytes, see traffic), so the HBM "
                              "figure below is the contract's denominator, not the limiter; gather_roofline is the same march's loads alone "
                              "against L2, and ncu (profiles/) shows instruction issue + L2-hit latency binding the kernel",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": load_traffic(), "traffic_note": "dram__bytes_read+write per lidar launch from the committed ncu capture "
                                                           "(profiles/traffic.json), not measured in this run",
                "kernel": "lidar_kernel", "kernel_ms": lidar_ms,
                "kernel_share_of_step": min(1.0, lidar_ms / max(step_ms_unevented, 1e-9)),
                "kernel_share_note": "kernel_ms (its own event pair: the events keep PDL from overlapping the neighbours) over the un-evented "
                                     "ms_per_step; all_kernels_ms are evented too and sum to more than ms_per_step",
                "lookups_per_ray": lbar, "longest_ray_lookups": max_lookups,
                "rays_redone_exactly": redone_rays, "rays_counted": rays,
                "bytes_per_ray": bytes_per_ray, "bytes_per_ray_is": "8 * lookups_per_ray + %g stored" % s_out,
                "sector_level": {"bytes_per_ray": 32.0 * lbar + s_out, "gbs": (32.0 * lbar + s_out) * E * A * B / (lidar_ms * 1e-3) / 1e9,
                                 "note": "32-byte sector per gather instead of the 8 useful bytes (SURVEY 8d)"},
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650",
                "all_kernels_ms": {"dynamics": kern_ms[0], "lidar": kern_ms[1], "post": kern_ms[2]},
                "gather_roofline": dict(gather, frac_of_whole_map=8.0 * lbar * E * A * B / (lidar_ms * 1e-3) / 1e9 / gather["whole_map_gbs"],
                                        frac_of_touched_window=8.0 * lbar * E * A * B / (lidar_ms * 1e-3) / 1e9 / gather["touched_window_gbs"])}
    # ---- CPU arm beside it (the other ranks have exited: every host core is free)
    cpu = None
    if not args.no_cpu_baseline:
        probe = cpu_arm(args, 5, 2)
        steps = args.cpu_steps or int(min(400, max(20, 2.0 / (probe['seconds'] / 5))))   # ~2 s wall on all threads
        c = cpu_arm(args, steps, 3)
        cpu = {"value": c['value'], "unit": "env-steps/s", "cores": c['threads'], "kind": "port",
               "sample": "%d envs x %d steps of the same workload, oracle/f110_oracle.c on %d threads (%.1f s)"
                         % (c['envs'], c['steps'], c['threads'], c['seconds']),
               "numba_reference": numba_reference()}
    line = {
        "metric": "env-steps/s (1080-beam lidar)", "value": value, "unit": "env-steps/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak" if args.config == "c3" else "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "rays_per_s": rays_per_s,
        "config": dict(workload_config(args, E), total_envs=total_envs,
                       l2="flushed between timed steps (252 MiB fill, outside the per-step events)" if flush is not None
                       else "not flushed; per-step working set %.0f MiB" % ((E * A * B * 12 + map_arrays[0].nbytes) / 2**20),
                       timing="sum of per-step CUDA-event intervals on the launch stream, max over ranks",
                       wall_ms_per_step_incl_flush=1e3 * t_wall / K),
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "episode_stats": {k: stats[k] for k in ('episodes', 'ego_collisions', 'mean_episode_steps')},
    }
    emit(line)
    return 0


DUMP_BYTES = 64 * 10 ** 6      # all files of a dump together, headers included
NPY_HEADER_BYTES = 4096        # bound on one .npy header (128 bytes for the short shapes written here)


def dump_outputs(directory, result, torch):
    """One step's return value -- (obs, reward, terminated, truncated, info) of F110VecEnv.step or DeviceRollout.step -- as
    <directory>/<name>.npy: obs, reward, terminated, truncated and every other tensor of info, float64 where the step
    computes float64, float32 otherwise.  Rows are envs.  When all of them would exceed DUMP_BYTES, a sample of envs drawn
    from a fixed seed is kept instead, so that two builds run with the same arguments write the same rows;
    env_index.npy names the rows written."""
    obs, reward, terminated, truncated, info = result
    arrays = dict(obs=obs, reward=reward, terminated=terminated, truncated=truncated)
    arrays.update((k, v) for k, v in info.items() if k not in arrays)
    n = obs.shape[0]
    row_bytes = 8 + sum((8 if v.dtype == torch.float64 else 4) * (v.numel() // n) for v in arrays.values())
    budget = DUMP_BYTES - NPY_HEADER_BYTES * (len(arrays) + 1)
    rows = np.arange(n)
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, budget // row_bytes, replace=False))
    idx = torch.from_numpy(rows).to(obs.device)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "env_index.npy"), rows.astype(np.float64))
    for k, v in arrays.items():
        v = v.index_select(0, idx)
        v = v if v.dtype == torch.float64 else v.to(torch.float32)
        np.save(os.path.join(directory, k + ".npy"), v.cpu().numpy())


def kernel_breakdown(env, acts, first, n, flush, torch):
    """Average per-launch duration of each of the three kernels, CUDA events on the launch stream."""
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    import ctypes as C
    L = env.backend.lib
    _lib.check(L.f110_set_kernel_timing(env.backend.h, 1))
    for k in range(first, first + n):
        if flush is not None:
            flush.fill_(k & 0xFF)
        env.step(acts[k])
    torch.cuda.synchronize()
    ms = (C.c_double * 3)()
    cnt = C.c_int64(0)
    _lib.check(L.f110_get_kernel_timing(env.backend.h, ms, C.byref(cnt)))
    _lib.check(L.f110_set_kernel_timing(env.backend.h, 0))
    per = [ms[i] / max(cnt.value, 1) for i in range(3)]
    return per[1], per


def e2e_run(args, map_arrays, poses, acts, W, K, E, A, B, local, torch):
    """Same workload through the host-buffer API: every step uploads the actions from pinned host memory and
    downloads observation / reward / terminated into pinned host memory, inside the timed region (wall clock
    around K synchronous steps).  Returns elapsed seconds."""
    from f110_gymnasium_ros2_jazzy_b200 import F110HostVecEnv
    from f110_gymnasium_ros2_jazzy_b200.dist import bind_host_to_gpu
    previous_affinity = bind_host_to_gpu(local) if int(os.environ.get("WORLD_SIZE", "1")) > 1 else None   # NUMA-local pinned buffers
    hc = [int(v) for v in str(args.host_chunks).split(",")]
    henv = F110HostVecEnv(E, chunks=hc[0] if len(hc) == 1 else tuple(hc), map_arrays=map_arrays, num_agents=A, num_beams=B,
                          device=local, noise_std=0.01)
    hacts = acts.cpu().pin_memory().numpy()
    henv.reset(poses)
    for k in range(min(W, 5)):
        henv.step(hacts[k])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(W, W + K):
        henv.step(hacts[k])
    el = time.perf_counter() - t0
    henv.close()
    henv = F110HostVecEnv(E, chunks=args.pipe_chunks, map_arrays=map_arrays, num_agents=A, num_beams=B, device=local,
                          noise_std=0.01)
    henv.reset(poses)
    for k in range(min(W, 5)):
        henv.step(hacts[k])
    # the same K steps with the chunks pipelined ACROSS step boundaries (send/recv per chunk): chunk g's next actions
    # go up as soon as its own observation has arrived, while the other chunk's download is still on the wire
    C = len(henv.parts)
    sl = [henv.chunk_slice(g) for g in range(C)]
    for g in range(C):
        henv.send(g, hacts[W - 1][sl[g]])
    for g in range(C):
        henv.recv(g)
    t0 = time.perf_counter()
    for g in range(C):
        henv.send(g, hacts[W][sl[g]])
    for k in range(W + 1, W + K):
        for g in range(C):
            henv.recv(g)
            henv.send(g, hacts[k][sl[g]])
    for g in range(C):
        henv.recv(g)
    el_pipe = time.perf_counter() - t0
    henv.close()
    if previous_affinity is not None:
        os.sched_setaffinity(0, previous_affinity)
    return el, el_pipe


def gather_roofline(dt, rays, lbar, torch, dev):
    """Empirical dependent-gather roofline (SURVEY 8d): f110_gather_probe with the lidar kernel's thread count and a
    chain of round(L-bar) dependent 8-byte loads, over the whole map (L2-resident random gather) and over a 4 MiB
    window (about what 4096 cars on the track actually touch).  GB/s of useful 8-byte cells."""
    import ctypes as C
    from f110_gymnasium_ros2_jazzy_b200 import _lib
    L = _lib.load()
    m = torch.from_numpy(np.ascontiguousarray(dt)).to(dev)
    sink = torch.zeros(1, dtype=torch.float64, device=dev)
    chain = max(1, int(round(lbar)))
    out = {"chain": chain, "threads": int(rays)}
    for key, window in (("whole_map_gbs", 0), ("touched_window_gbs", 512 * 1024)):
        ms = C.c_float(0)
        _lib.check(L.f110_gather_probe(C.c_void_p(m.data_ptr()), m.numel(), window, chain, int(rays), 5,
                                       C.c_void_p(sink.data_ptr()), C.byref(ms), None))
        out[key] = 8.0 * chain * rays / (ms.value * 1e-3) / 1e9
    # the HBM-resident regime (SURVEY 8d: an array far larger than L2), for the C4 large-map sweep
    del m
    big = torch.zeros(2 * 1024 ** 3 // 8, dtype=torch.float64, device=dev)
    ms = C.c_float(0)
    _lib.check(L.f110_gather_probe(C.c_void_p(big.data_ptr()), big.numel(), 0, chain, int(rays), 3,
                                   C.c_void_p(sink.data_ptr()), C.byref(ms), None))
    out["hbm_2gib_gbs"] = 8.0 * chain * rays / (ms.value * 1e-3) / 1e9
    del big
    return out


def load_traffic():
    """dram bytes per lidar launch from the committed ncu capture, if one exists (profiles/traffic.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("lidar_kernel_dram_bytes_per_launch")
        except Exception:
            return None
    return None


if __name__ == "__main__":
    sys.exit(main())
