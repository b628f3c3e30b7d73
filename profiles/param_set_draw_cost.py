"""Cost of the per-episode set draw (Env(param_set_weights=...)) at the bench shape: device time per fused step +
auto-reset call, with and without the draw, for 65,536 envs x 8 OU pairs at S = 16 and S = 1024 (random initial
assignment, equal weights) and for the C4 composite at S = 16.  The slabs are param_sets_cost.py's (8 rotating slabs,
L2-cold, one stream, random set values); 256 fused calls back to back per shape, and the median of 256 single calls
timed with CUDA events.  Two passes in opposite order.
  python profiles/param_set_draw_cost.py [--out param_set_draw_cost.json]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

import param_sets_cost as pc

SHAPES = {  # name: (param_sets_cost shape, draw on)
    "pairs_S16": ("pairs_S16", False), "pairs_S16_draw": ("pairs_S16", True),
    "pairs_S1024": ("pairs_S1024", False), "pairs_S1024_draw": ("pairs_S1024", True),
    "c4_S16": ("c4_S16", False), "c4_S16_draw": ("c4_S16", True),
}


def measure(name):
    base, draw = SHAPES[name]
    cfg, reward, margins, costs, unit, S, assign, *broker = pc.SHAPES[base]
    envs = [pc.make(cfg, reward, margins, costs, S, assign, s, bool(broker)) for s in range(pc.SLABS)]
    if draw:
        for e in envs:
            e.set_param_set_weights([1.] * S)
    K, SL = pc.K, pc.SLABS
    g = torch.Generator().manual_seed(1)
    acts = [(torch.randint(-1, 2, (pc.N, 16), generator=g).double() * unit).to(pc.dev) for _ in range(4)]
    for i in range(40 * SL):  # leave the synchronised start
        envs[i % SL].step(acts[i % 4], auto_reset=True)
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    for i in range(K):
        ev[i][0].record()
        envs[i % SL].step(acts[i % 4], auto_reset=True)
        ev[i][1].record()
    torch.cuda.synchronize()
    single = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(K):
        envs[i % SL].step(acts[i % 4], auto_reset=True)
    b.record()
    torch.cuda.synchronize()
    fused = a.elapsed_time(b) * 1e3 / K
    done = float(torch.stack([e.t["done"].float().mean() for e in envs]).mean())
    del envs, acts
    torch.cuda.empty_cache()
    r = dict(step_autoreset_us=fused, step_autoreset_median_us=single[K // 2], step_autoreset_p10_us=single[K // 10],
             step_autoreset_p90_us=single[9 * K // 10], done_rate=done, n_sets=S, draw=draw)
    print(name, json.dumps(r), flush=True)
    return r


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = dict(card=torch.cuda.get_device_name(0), nvidia_smi=smi[0] if smi else None, n_envs=pc.N, slabs=pc.SLABS,
               launches=pc.K, results={})
    print(out["card"], out["nvidia_smi"], flush=True)
    for rep in range(2):  # two passes, in opposite order: the spread between them is the run-to-run noise
        for name in (SHAPES if rep == 0 else reversed(list(SHAPES))):
            out["results"].setdefault(name, []).append(measure(name))
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
