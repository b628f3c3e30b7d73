"""Device time of the prioritized replay (DevicePrioritizedReplay) against the uniform DeviceReplay at the bench shape
(65,536 envs x 16 assets, window 64, fp32 normalised windows, DSR n = 1), observation depth 16 and 64:
  add      step + add of each buffer, alternated, REPS x 50 steps -> the extra time of the prioritized add per step
  sample   sample(B) of each buffer, B = 4096 and 32768 (prioritized: descent + gather; beta 0.4)
  update   update_priorities(B) on the last prioritized sample's batch
CUDA events around each loop (one stream, device time including launch gaps); the median of REPS loops is printed.
  python profiles/per_cost.py [--out per_cost.json]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from madigan_b200.utils.replay import DevicePrioritizedReplay, DeviceReplay

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--reps", type=int, default=5)
args = ap.parse_args()

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                    "-i", "0"], capture_output=True, text=True).stdout.strip()
print(f"gpu: {q}")
dev = torch.device("cuda", 0)
env = bench.make_env(dev, 0)
acts = bench.synth_actions(4, bench.ENVS_PER_GPU, 1, device=dev)


def timed(f, n):
    """median over args.reps loops of n calls, microseconds per call"""
    out = []
    for _ in range(args.reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for i in range(n):
            f(i)
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / n * 1e3)
    return float(np.median(out))


res = {"gpu": q, "envs": bench.ENVS_PER_GPU, "reps": args.reps}
for depth in (16, 64):
    plain = DeviceReplay(env, depth=depth, norm_type="standard_normal", dtype=torch.float32)
    per = DevicePrioritizedReplay(env, alpha=.6, depth=depth, norm_type="standard_normal", dtype=torch.float32)
    for rp in (plain, per):
        rp.observe_start()

    def step_add(rp):
        def f(i):
            env.step(acts[i % 4], auto_reset=True)
            rp.add(acts[i % 4])
        return f

    for i in range(2 * depth):  # fill both rings past their capacity
        step_add(plain)(i)
        step_add(per)(i)
    r = {"capacity": per.capacity, "tree_size": per.tree_size}
    t_plain, t_per = [], []
    for _ in range(2):  # alternated
        t_plain.append(timed(step_add(plain), 50))
        t_per.append(timed(step_add(per), 50))
    r["step_add_uniform_us"], r["step_add_prioritized_us"] = min(t_plain), min(t_per)
    r["add_extra_us"] = r["step_add_prioritized_us"] - r["step_add_uniform_us"]
    print(f"depth {depth} (capacity {per.capacity:,}, {per.tree_size:,} leaves): step + add "
          f"{r['step_add_uniform_us']:.1f} us uniform, {r['step_add_prioritized_us']:.1f} us prioritized -> "
          f"prioritized add +{r['add_extra_us']:.1f} us per 65,536-env step")
    for B in (4096, 32768):
        plain.sample(B)
        per.sample(B, .4)
        r[f"sample_uniform_{B}_us"] = timed(lambda i: plain.sample(B), 50)
        r[f"sample_prioritized_{B}_us"] = timed(lambda i: per.sample(B, .4), 50)
        prio = torch.rand(B, dtype=torch.float64, device=dev) + .01
        per.update_priorities(prio)
        r[f"update_{B}_us"] = timed(lambda i: per.update_priorities(prio), 50)
        print(f"  B = {B}: sample uniform {r[f'sample_uniform_{B}_us']:.1f} us, prioritized "
              f"{r[f'sample_prioritized_{B}_us']:.1f} us; update_priorities {r[f'update_{B}_us']:.1f} us")
    res[f"depth_{depth}"] = r
    del plain, per
    torch.cuda.empty_cache()
print(json.dumps(res))
if args.out:
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
