"""Device time and memory of the replay row store (store="rows") against the window store at the bench shape
(65,536 envs x 16 assets, window 64, fp32 standard_normal windows, DSR n = 1):
  add      step + add of each store, alternated, REPS x 50 steps, at depth 16 and 64; the rows store also at depth
           1024 (the window store's byte count is given there: it cannot be allocated)
  sample   sample(B), B = 4096 and 32768, uniform and prioritized (beta 0.4), both stores, after steps that every
           buffer saw (the valid fraction printed is that of the prioritized sample)
  memory   device bytes of each buffer's tensors
CUDA events around each loop (one stream, device time including launch gaps); the median of REPS loops is printed.
  python profiles/replay_rows_cost.py [--out replay_rows_cost.json] [--depths 16,64,1024]"""
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
ap.add_argument("--depths", default="16,64,1024")
args = ap.parse_args()

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                    "-i", "0"], capture_output=True, text=True).stdout.strip()
print(f"gpu: {q}")
dev = torch.device("cuda", 0)
env = bench.make_env(dev, 0)
acts = bench.synth_actions(4, bench.ENVS_PER_GPU, 1, device=dev)
KW = dict(norm_type="standard_normal", dtype=torch.float32)


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


def nbytes(rp):
    ts = [rp.obs_port] + list(rp.t.values())
    ts += [rp.obs_price] if rp.obs_price is not None else [rp.rows, rp.row_end, rp.row_count, rp.last_ts]
    ts += list(getattr(rp, "per", {}).values())
    return sum(t.numel() * t.element_size() for t in ts)


def step_add(rp):
    def f(i):
        env.step(acts[i % 4], auto_reset=True)
        rp.add(acts[i % 4])
    return f


def window_store_bytes(depth):
    N, k, nA = env.N, env.k, env.nA
    return depth * N * (k * nA * 4 + (nA + 1) * 8) + N * (depth - 2) * (4 * 3 + 8 + 1 + 8 + nA * 8)


res = {"gpu": q, "envs": bench.ENVS_PER_GPU, "reps": args.reps}
for depth in (int(d) for d in args.depths.split(",")):
    r = {}
    stores = ["rows"] if depth > 64 else ["windows", "rows"]
    bufs = {}
    for st in stores:
        bufs[st] = (DeviceReplay(env, depth=depth, store=st, **KW),
                    DevicePrioritizedReplay(env, alpha=.6, depth=depth, store=st, **KW))
        for rp in bufs[st]:
            rp.observe_start()
            r[f"bytes_{st}_{type(rp).__name__}"] = nbytes(rp)
    if "windows" not in stores:
        r["bytes_windows_DeviceReplay_not_allocated"] = window_store_bytes(depth)
    def fill(n):  # every buffer sees every step (a buffer that misses steps appends whole windows)
        for i in range(n):
            env.step(acts[i % 4], auto_reset=True)
            for st in stores:
                for rp in bufs[st]:
                    rp.add(acts[i % 4])

    fill(min(2 * depth, 128))  # past capacity at depth 16 and 64; 128 steps of history at 1024
    t = {st: [] for st in stores}
    for _ in range(2):  # alternated
        for st in stores:
            t[st].append(timed(step_add(bufs[st][0]), 50))
    for st in stores:
        r[f"step_add_{st}_us"] = min(t[st])
    r["step_alone_us"] = timed(lambda i: env.step(acts[i % 4], auto_reset=True), 50)
    print(f"depth {depth}: " + ", ".join(f"step + add ({st}) {r[f'step_add_{st}_us']:.1f} us" for st in stores)
          + f"; step alone {r['step_alone_us']:.1f} us")
    fill(depth if depth <= 64 else 64)  # the timed loops fed one buffer each: a full depth of steps fed to all
    for st in stores:
        uni, per = bufs[st]
        for B in (4096, 32768):
            uni.sample(B)
            per.sample(B, .4)
            r[f"sample_{st}_uniform_{B}_us"] = timed(lambda i: uni.sample(B), 50)
            r[f"sample_{st}_prioritized_{B}_us"] = timed(lambda i: per.sample(B, .4), 50)
            print(f"  {st:7s} B = {B}: sample uniform {r[f'sample_{st}_uniform_{B}_us']:.1f} us, prioritized "
                  f"{r[f'sample_{st}_prioritized_{B}_us']:.1f} us; valid {float(per.last_valid.float().mean()):.4f}")
    print("  bytes: " + ", ".join(f"{k_[6:]} {v / 1e9:.2f} GB" for k_, v in r.items() if k_.startswith("bytes_")))
    res[f"depth_{depth}"] = r
    del bufs, uni, per
    torch.cuda.empty_cache()
print(json.dumps(res))
if args.out:
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
