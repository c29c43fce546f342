"""The shaped reward on a set of centerlines against one centerline (DESIGN.md section 10).

  python tools/reward_set_bench.py --out profiles/r06_reward_sets.json [--calls 300 --warmup 30 --steps 100]

Kernel: 8192 envs, 1080 beams, one observation per arm (cars along the Shanghai centerline, opponent 40 rows ahead,
seeded lidar).  Arms: `single`, today's single-line kernel on Shanghai; `set<K>_blocks` / `set<K>_interleaved`, the set
kernel with K = 2 and 8 copies of that centerline translated 500 m apart (env e on slot e * K // N, or e % K), each car
translated with its line, so every arm does the same geometric work.  CUDA events around each call, arms alternated call
by call, median per arm.  Each set arm's outputs are first held bit for bit to K single-line rewards on the translated
lines fed the same observations.  L2 is not flushed: an arm's observation (35.7 MB) and lines fit in the 126 MB L2.

Rollout (BASELINE C5 shape): DeviceRollout, 8192 two-car envs, actor 1088-128-128-2 + gap-follow opponent + shaped reward.
Arms: `one_map`, one map with the single-line reward; `set8`, a set of 8 translated Shanghai copies with the 8-line set
reward; `set8_workaround`, the same map set with 8 single-line rewards, each over all envs, selected by slot.  Windows of
--steps steps timed with CUDA events, arms alternated window by window, median env-steps/s per arm.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHIFT = 500.0       # m between the copies: far enough apart that no car of one copy is near another copy's line


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      timeout=30).decode().strip().splitlines()[0]
        name, power, clock = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:      # the numbers below still stand; say that the card could not be read
        return {"error": repr(e)}


def kernel_arms(torch, args, cl):
    from f110_gymnasium_ros2_jazzy_b200 import ShapedReward
    N, B = args.envs, 1080
    rng = np.random.default_rng(0)
    idx = np.linspace(0, len(cl) - 1, N).round().astype(int)
    base = np.zeros((N, B + 8), np.float32)
    base[:, :B] = rng.uniform(0.0, 1.0, (N, B)).astype(np.float32)
    base[:, B:B + 2] = cl[idx, :2] + rng.normal(0, 0.2, (N, 2))
    base[:, B + 2] = rng.uniform(-np.pi, np.pi, N)
    base[:, B + 4:B + 6] = cl[(idx + 40) % len(cl), :2]
    base[:, B + 6] = rng.uniform(-np.pi, np.pi, N)

    def line(k):
        c = cl.copy()
        c[:, 0] += k * SHIFT
        return c

    def obs_for(slots):
        o = base.copy()
        o[:, B] += (slots * SHIFT).astype(np.float32)
        o[:, B + 4] += (slots * SHIFT).astype(np.float32)
        return torch.from_numpy(o).cuda()

    arms, checks = {}, {}
    zero = np.zeros(N, np.int64)
    arms['single'] = (ShapedReward(N, cl), obs_for(zero), None)
    for K in args.ks:
        for layout, slots in (('blocks', (np.arange(N) * K) // N), ('interleaved', np.arange(N) % K)):
            name = 'set%d_%s' % (K, layout)
            ob = obs_for(slots)
            sl = torch.from_numpy(slots.astype(np.int32)).cuda()
            # the set's outputs, three calls, against K single-line rewards on the translated lines
            fresh = ShapedReward(N, centerlines=[line(k) for k in range(K)])
            refs = [ShapedReward(N, line(k)) for k in range(K)]
            ok = True
            for _ in range(3):
                got = fresh(ob, None, slots=sl).clone()
                want = torch.stack([r(ob).clone() for r in refs])
                want = want.gather(0, sl.long()[None]).squeeze(0)
                ok = ok and bool(torch.equal(got.view(torch.int64), want.view(torch.int64)))
            checks[name] = ok
            fresh.close()
            for r in refs:
                r.close()
            assert ok, name
            arms[name] = (ShapedReward(N, centerlines=[line(k) for k in range(K)]), ob, sl)
    names = list(arms)
    for _ in range(args.warmup):
        for n in names:
            rw, ob, sl = arms[n]
            rw(ob, None, slots=sl)
    torch.cuda.synchronize()
    ev = {n: [] for n in names}
    for _ in range(args.calls):
        for n in names:
            rw, ob, sl = arms[n]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rw(ob, None, slots=sl)
            e1.record()
            ev[n].append((e0, e1))
    torch.cuda.synchronize()
    out = {}
    for n in names:
        us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev[n]])
        out[n] = {"median_us": float(np.median(us)), "p10_us": float(np.percentile(us, 10)),
                  "p90_us": float(np.percentile(us, 90)), "calls": len(us)}
        if n in checks:
            out[n]["bit_identical_to_single_line_references"] = checks[n]
    for rw, _, _ in arms.values():
        rw.close()
    return out


class SelectBySlot(object):
    """Today's workaround: K single-line rewards, each over all envs, the env's value taken from its slot's."""

    def __init__(self, torch, env, rewards):
        self.torch, self.env, self.rewards = torch, env, rewards
        self.slots = torch.zeros(env.num_envs, dtype=torch.int64, device=env.device)
        self._s32 = torch.zeros(env.num_envs, dtype=torch.int32, device=env.device)

    def __call__(self, obs, reset_mask=None):
        torch = self.torch
        self.env.backend.env_maps(out=self._s32)
        self.slots.copy_(self._s32)
        vals = torch.stack([r(obs, reset_mask) for r in self.rewards])
        return vals.gather(0, self.slots[None]).squeeze(0)


def rollout_arms(torch, args, cl):
    from f110_gymnasium_ros2_jazzy_b200 import Actor, DeviceRollout, F110VecEnv, ShapedReward
    from tests import helpers as H
    N, K = args.envs, 8
    dt, res, org = H.golden_map('Shanghai_map')
    rows = H.load('maps')['Shanghai_map__centerline_poses']
    idx = np.linspace(0, len(rows) - 1, N).round().astype(int)
    poses = np.stack([rows[idx], rows[(idx + 40) % len(rows)]], axis=1)
    outs = ('obs', 'reward', 'terminated', 'scans_f32')
    kw = dict(w_prog=5.0, alive_bonus=0.5, grace_steps_wall=25, grace_steps_opp=175, w_lat=0.25, lat_cap=3.0,
              near_wall_dist=0.30 / 30, w_wall=0.30, wall_quantile=0.10, opp_safe_dist=0.60, w_opp=0.30)
    lines = []
    for k in range(K):
        c = cl.copy()
        c[:, 0] += k * SHIFT
        lines.append(c)
    slots = (np.arange(N) * K) // N
    set_poses = poses.copy()
    set_poses[..., 0] += (slots * SHIFT)[:, None]
    maps = [(dt, res, [org[0] + k * SHIFT, org[1], org[2]]) for k in range(K)]

    def actor():
        torch.manual_seed(42)
        return Actor(1088, 2, [-0.4189, 0.0], [0.4189, 20.0]).cuda()

    arms = {}
    env = F110VecEnv(N, num_agents=2, map_arrays=(dt, res, org), outputs=outs)
    arms['one_map'] = (DeviceRollout(env, actor(), reward_fn=ShapedReward(N, cl, **kw)), poses)
    env = F110VecEnv(N, num_agents=2, maps=maps, outputs=outs)
    arms['set8'] = (DeviceRollout(env, actor(), reward_fn=ShapedReward(N, centerlines=lines, **kw)), set_poses)
    env = F110VecEnv(N, num_agents=2, maps=maps, outputs=outs)
    arms['set8_workaround'] = (DeviceRollout(env, actor(), reward_fn=SelectBySlot(torch, env, [ShapedReward(N, c, **kw) for c in lines])),
                               set_poses)
    for ro, p in arms.values():
        ro.reset(p)
        for _ in range(args.warmup):
            ro.step()
    torch.cuda.synchronize()
    rates = {n: [] for n in arms}
    for _ in range(args.windows):
        for n, (ro, _) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                ro.step()
            e1.record()
            torch.cuda.synchronize()
            rates[n].append(N * args.steps / (e0.elapsed_time(e1) * 1e-3))
    # the set rollout's rewards against the workaround's: same maps, actor, poses and opponent, so the same observations
    same = bool(torch.equal(arms['set8'][0].reward.view(torch.int64), arms['set8_workaround'][0].reward.view(torch.int64)))
    out = {n: {"env_steps_per_s_median": float(np.median(r)), "env_steps_per_s_min": float(np.min(r)),
               "env_steps_per_s_max": float(np.max(r)), "windows": len(r)} for n, r in rates.items()}
    out["set8_reward_equals_workaround_after_last_window"] = same
    for ro, _ in arms.values():
        ro.env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--calls", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--ks", default="2,8")
    ap.add_argument("--steps", type=int, default=100, help="rollout steps per timed window")
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--skip-rollout", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    args.ks = [int(v) for v in args.ks.split(",") if v]
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("reward_set_bench.py needs a CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    from tests import helpers as H
    cl = H.load('reward')['centerline']
    res = {"gpu": gpu_info(), "envs": args.envs, "beams": 1080,
           "kernel": kernel_arms(torch, args, cl)}
    if not args.skip_rollout:
        res["rollout_c5"] = rollout_arms(torch, args, cl)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
