"""Map sets against the alternatives (DESIGN.md section 10): what one handle holding K maps costs per step, next to one map
and next to K handles of one map each.

  python tools/multimap_bench.py --out profiles/r04_multimap.json [--steps 200 --warmup 20 --ks 2,4,8]

The maps are K identical copies of the packaged Shanghai map, each in its own device memory, so the arms differ only in
where the cells live.  Arms (single agent, observation / reward / terminated only, device noise, auto-reset, as C3):
  a        C3: one map, 4096 envs
  b<K>     one handle with the K copies, 4096 envs in contiguous blocks on C3's start poses (C3's cars, split over K maps)
  c<K>     as b, but each block spread over its whole track (start_poses(N / K) per block): K x the touched L2 footprint
  d1_<K>   K handles x 4096 / K envs on one stream, one after the other
  dK_<K>   the same K handles, each on its own stream
  e1, e8   32 768 envs on one map, and over 8 copies (the home-segment path)
Per step: CUDA events around the step (all K steps for d), L2 flushed before every timed step as bench.py does (outside the
events).  The arms alternate step by step.  b's outputs are compared with a's bit for bit at every step: same cars, same
actions, same noise, the map copies are identical.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_BYTES = 126 * 1024 * 1024


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      timeout=30).decode().strip().splitlines()[0]
        name, power, clock = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:      # the numbers below still stand; say that the card could not be read
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--ks", default="2,4,8")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--big", type=int, default=32768)
    ap.add_argument("--arms", default="a,b,c,d,e", help="subset of a,b,c,d,e")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("multimap_bench.py needs a CUDA device")
    import __graft_entry__
    __graft_entry__.build()
    from f110_gymnasium_ros2_jazzy_b200 import F110VecEnv, workloads
    dev = torch.device("cuda", 0)
    N, W, T = args.envs, args.warmup, args.steps
    ks = [int(v) for v in args.ks.split(",") if v]
    arms_on = set(args.arms.split(","))
    sh = workloads.shanghai_map()
    copies = lambda k: [(sh[0].copy(), sh[1], list(sh[2])) for _ in range(k)]

    def vec(n, **kw):
        return F110VecEnv(n, num_agents=1, device=0, auto_reset=True, noise_std=0.01, seed=42, **kw)

    def spread(n, k):
        return np.concatenate([workloads.start_poses(n // k + (1 if b < n % k else 0)) for b in range(k)])

    g = torch.Generator(device=dev).manual_seed(1234)
    lo = torch.tensor([-0.4189, -5.0], device=dev)
    hi = torch.tensor([0.4189, 20.0], device=dev)

    def actions(n):
        return [(lo + torch.rand((n, 1, 2), generator=g, device=dev) * (hi - lo)).contiguous() for _ in range(W + T)]

    acts = actions(N)
    big_acts = actions(args.big) if "e" in arms_on else None
    arms = {}      # name -> (step fn(k), envs to close)
    c3 = workloads.start_poses(N)
    if "a" in arms_on or "b" in arms_on:
        a = vec(N, map_arrays=sh); a.reset(c3)
        arms["a"] = (lambda k, e=a: e.step(acts[k]), [a])
    for K in ks:
        if "b" in arms_on:
            b = vec(N, maps=copies(K)); b.reset(c3)
            arms["b%d" % K] = (lambda k, e=b: e.step(acts[k]), [b])
        if "c" in arms_on:
            c = vec(N, maps=copies(K)); c.reset(spread(N, K))
            arms["c%d" % K] = (lambda k, e=c: e.step(acts[k]), [c])
        if "d" in arms_on:
            bounds = [(N * j) // K for j in range(K + 1)]
            hs = []
            for j in range(K):
                h = vec(bounds[j + 1] - bounds[j], map_arrays=sh)
                h.reset(c3[bounds[j]:bounds[j + 1]])
                hs.append(h)
            sl = [slice(bounds[j], bounds[j + 1]) for j in range(K)]
            arms["d1_%d" % K] = (lambda k, hs=hs, sl=sl: [h.step(acts[k][s]) for h, s in zip(hs, sl)], hs)
            streams = [torch.cuda.Stream(dev) for _ in range(K)]

            def on_streams(k, hs=hs, sl=sl, streams=streams):
                main = torch.cuda.current_stream(dev)
                for h, s, st in zip(hs, sl, streams):
                    st.wait_stream(main)
                    with torch.cuda.stream(st):
                        h.step(acts[k][s])
                for st in streams:
                    main.wait_stream(st)
            arms["dK_%d" % K] = (on_streams, [])
    if "e" in arms_on:
        e1 = vec(args.big, map_arrays=sh); e1.reset(workloads.start_poses(args.big))
        e8 = vec(args.big, maps=copies(8)); e8.reset(workloads.start_poses(args.big))
        arms["e1"] = (lambda k, e=e1: e.step(big_acts[k]), [e1])
        arms["e8"] = (lambda k, e=e8: e.step(big_acts[k]), [e8])

    flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    ms = {n: [] for n in arms}
    mismatch = {n: 0 for n in arms if n.startswith("b")}
    for k in range(W + T):
        for name, (step, _) in arms.items():
            flush.fill_(k & 0xFF)
            e0, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            step(k)
            e1_.record(stream)
            if k >= W:
                ms[name].append((e0, e1_))
        if "a" in arms:
            ref = arms["a"][1][0].backend.out
            for name in mismatch:
                out = arms[name][1][0].backend.out
                for key in ("obs", "reward", "terminated"):
                    if not torch.equal(out[key], ref[key]):
                        mismatch[name] += 1
    torch.cuda.synchronize()
    res = {}
    for name, evs in ms.items():
        t = np.array([s.elapsed_time(e) for s, e in evs])
        res[name] = {"median_ms": float(np.median(t)), "mean_ms": float(t.mean()), "p10_ms": float(np.percentile(t, 10)),
                     "p90_ms": float(np.percentile(t, 90))}
    base = res.get("a", {}).get("median_ms")
    for name, r in res.items():
        if base and not name.startswith("e"):
            r["vs_a"] = r["median_ms"] / base
    if "e1" in res:
        res["e8"]["vs_e1"] = res["e8"]["median_ms"] / res["e1"]["median_ms"]
    for K in ks:
        d = [res[n]["median_ms"] for n in ("d1_%d" % K, "dK_%d" % K) if n in res]
        for arm in ("b%d" % K, "c%d" % K):
            if d and arm in res:
                res[arm]["speedup_vs_best_d"] = min(d) / res[arm]["median_ms"]
    out = {"gpu": gpu_info(), "measured": True, "steps": T, "warmup": W, "envs": N, "big_envs": args.big,
           "l2": "flushed before every timed step (252 MiB fill, outside the events)",
           "library": os.environ.get("F110_B200_LIB", "in-tree build"),
           "arms": res, "b_vs_a_output_mismatches (steps x outputs)": mismatch}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    for _, (_, envs) in arms.items():
        for e in envs:
            e.close()


if __name__ == "__main__":
    main()
