"""What the auto-reset refill costs: (a) the refill alone, (b) its share of the bench's overlapped step.

(a) 8 slabs of 65,536 envs (the bench's shape: 16 assets = 8 OU pairs, window 64), each reset with a fixed seeded mask
    of ~0.4 %, 5 % and 100 % of its envs through Env.reset's path (mdg_reset_ws: header memset + list scan + refill),
    rotating over the slabs so that every call finds its slab evicted from L2 by the other seven.  CUDA events around
    R rounds x 8 calls on one stream; "floor" is the same call with an empty mask (memset + scan + a refill that finds
    no env).  Then, in a separate torch.profiler pass, the refill kernel's own mean duration per launch.
(b) bench.py's decomposition at its regime: 8 slabs on 8 streams, SETUP (default 16,384, bench.SETUP_STEPS) setup
    steps per slab, then K steps with auto-reset (step + refill, the bench's timed region) against K steps of the step
    kernel only (finished envs are left finished), alternated, REPS times.

  python profiles/refill_time.py [--part a|b|ab] [--generic]
--generic sets Env.flags |= FLAG_GENERIC_FILL: every refill takes the generic kernel (reset_fill_kernel).
MDG_FILL_GRID=<blocks> (read once per process) caps the refill's grid.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench

ap = argparse.ArgumentParser()
ap.add_argument("--part", default="ab", choices=["a", "b", "ab"])
ap.add_argument("--generic", action="store_true")
ap.add_argument("--steps", type=int, default=2000, help="K of part (b)")
ap.add_argument("--reps", type=int, default=3, help="repeats of part (b)")
args = ap.parse_args()

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                    "-i", "0"], capture_output=True, text=True).stdout.strip()
print(f"gpu: {q}")
dev = torch.device("cuda", 0)
n, slabs, W = 65536, 8, bench.WINDOW
envs = [bench.make_env(dev, s * n, n_envs=n) for s in range(slabs)]
if args.generic:
    from madigan_b200 import _abi as A
    for e in envs:
        e.flags |= A.FLAG_GENERIC_FILL
res = {"gpu": q, "generic": args.generic, "fill_grid": os.environ.get("MDG_FILL_GRID")}

if "a" in args.part:
    stream = torch.cuda.current_stream(dev)
    out = {}
    for rate, rounds in ((0.0, 50), (0.004, 50), (0.05, 20), (1.0, 3)):
        masks = [torch.from_numpy(np.random.default_rng(1000 + s).random(n) < rate).to(dev) for s in range(slabs)]
        listed = sum(int(m.sum()) for m in masks) / slabs
        for s in range(slabs):  # warm-up: every slab once
            envs[s]._reset_launch(masks[s], W, True, None, None)
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for r in range(rounds):
            for s in range(slabs):
                envs[s]._reset_launch(masks[s], W, True, None, None)
        t1.record(stream)
        torch.cuda.synchronize()
        us = t0.elapsed_time(t1) / (rounds * slabs) * 1e3
        # the refill kernel alone, in a run of its own under the profiler
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for r in range(min(rounds, 4)):
                for s in range(slabs):
                    envs[s]._reset_launch(masks[s], W, True, None, None)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if "reset_fill" in ev.key or "reset_scan" in ev.key:
                t = getattr(ev, "device_time_total", None)
                if t is None:
                    t = ev.cuda_time_total
                kern[ev.key.split("(")[0]] = round(t / max(ev.count, 1), 2)
        out[f"{rate:g}"] = {"listed_per_slab": listed, "us_per_reset_call": round(us, 2), "kernel_us": kern}
        print(f"(a) rate {rate:g}: {listed:.0f} envs listed per slab, {us:.2f} us per reset call "
              f"(events, {rounds} x {slabs} calls); per launch: {kern}", flush=True)
    res["a"] = out

if "b" in args.part:
    setup = int(os.environ.get("SETUP", bench.SETUP_STEPS))
    acts = bench.synth_actions(8, n, 1, device=dev)
    streams = [torch.cuda.Stream(dev) for _ in range(slabs)]
    for e, s in zip(envs, streams):
        e.bind_stream(s)
    for i in range(setup * slabs):
        envs[i % slabs].step(acts[i % 8], auto_reset=True)
    torch.cuda.synchronize()

    def run(auto, K):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cur = torch.cuda.current_stream()
        a.record(cur)
        for s in streams:
            s.wait_event(a)
        for i in range(K):
            envs[i % slabs].step(acts[i % 8], auto_reset=auto)
        for s in streams:
            ev = torch.cuda.Event(); ev.record(s); cur.wait_event(ev)
        b.record(cur)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / K * 1e3

    done = sum(float(e.t["done"].float().mean()) for e in envs) / slabs
    rows = []
    for rep in range(args.reps):
        t_auto = run(True, args.steps)
        t_step = run(False, args.steps)
        for i in range(8 * slabs):  # reset what the step-only run left finished
            envs[i % slabs].step(acts[i % 8], auto_reset=True)
        torch.cuda.synchronize()
        rows.append((t_auto, t_step))
        print(f"(b) {setup} setup steps/slab: step + refill {t_auto:.2f} us/step, step kernel only {t_step:.2f} "
              f"us/step, refill share {t_auto - t_step:.2f} us/step", flush=True)
    ta, ts = sorted(r[0] for r in rows)[len(rows) // 2], sorted(r[1] for r in rows)[len(rows) // 2]
    res["b"] = {"setup_steps": setup, "done_rate_before": done, "us_auto": [r[0] for r in rows],
                "us_step_only": [r[1] for r in rows], "median_auto": ta, "median_step_only": ts, "median_gap": ta - ts}
    for e in envs:
        e.bind_stream(None)
print(json.dumps(res))
