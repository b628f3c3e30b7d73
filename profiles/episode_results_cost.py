"""Cost of per-set episode results (EpisodeResults) at the bench shape: device time per fused step + auto-reset call,
65,536 envs x 8 OU pairs, DSR, about 2.5 % of envs resetting per step, for
  - no results;
  - results with n_offsets 6 and 0 (step, record + harvest, refill in one call);
  - the tearsheet= path with n_offsets 6 (step, tearsheet update, separate masked reset: scan + refill);
at S = 1 (a plain Env), 16, 1024 and N sets with the per-episode draw on (param_sets_cost.py's slabs: 8 rotating
slabs, L2-cold, one stream, random set values).  256 fused calls back to back per shape, and the median of 256 single
calls timed with CUDA events.  Two passes in opposite order.
  python profiles/episode_results_cost.py [--out episode_results_cost.json]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

import param_sets_cost as pc
from madigan_b200.utils.metrics import EpisodeResults, EpisodeTearsheet

BASES = {"S1": "pairs_nosets", "S16": "pairs_S16", "S1024": "pairs_S1024", "SN": "pairs_SN_identity"}
MODES = {"none": None, "results_J6": 6, "results_J0": 0, "tearsheet_J6": 6}


def measure(base, mode):
    cfg, reward, margins, costs, unit, S, assign, *broker = pc.SHAPES[BASES[base]]
    envs = [pc.make(cfg, reward, margins, costs, S, assign, s, bool(broker)) for s in range(pc.SLABS)]
    if S is not None:
        for e in envs:
            e.set_param_set_weights([1.] * S)
    kw = [{} for _ in envs]
    if mode.startswith("results"):
        kw = [dict(results=EpisodeResults(e, MODES[mode])) for e in envs]
    elif mode.startswith("tearsheet"):
        kw = [dict(tearsheet=EpisodeTearsheet(e, MODES[mode])) for e in envs]
    K, SL = pc.K, pc.SLABS
    g = torch.Generator().manual_seed(1)
    acts = [(torch.randint(-1, 2, (pc.N, 16), generator=g).double() * unit).to(pc.dev) for _ in range(4)]

    def call(i):
        envs[i % SL].step(acts[i % 4], auto_reset=True, **kw[i % SL])

    for i in range(40 * SL):  # leave the synchronised start
        call(i)
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    for i in range(K):
        ev[i][0].record()
        call(i)
        ev[i][1].record()
    torch.cuda.synchronize()
    single = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(K):
        call(i)
    b.record()
    torch.cuda.synchronize()
    fused = a.elapsed_time(b) * 1e3 / K
    done = float(torch.stack([e.t["done"].float().mean() for e in envs]).mean())
    episodes = None
    if mode.startswith("results"):
        episodes = int(sum(int(k["results"].table()["n_episodes"].sum()) for k in kw))
    del envs, acts, kw
    torch.cuda.empty_cache()
    r = dict(step_autoreset_us=fused, step_autoreset_median_us=single[K // 2], step_autoreset_p10_us=single[K // 10],
             step_autoreset_p90_us=single[9 * K // 10], done_rate=done, n_sets=S or 1, mode=mode,
             episodes_harvested=episodes)
    print(base, mode, json.dumps(r), flush=True)
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
    names = [(b, m) for b in BASES for m in MODES]
    for rep in range(2):  # two passes, in opposite order: the spread between them is the run-to-run noise
        for b, m in (names if rep == 0 else reversed(names)):
            out["results"].setdefault(f"{b}_{m}", []).append(measure(b, m))
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
