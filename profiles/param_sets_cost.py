"""Cost of generator parameter sets (Env(param_sets=...)) and of broker sets (Env(broker_sets=...)) at the bench
shape: device time of the step kernel alone and of step + auto-reset, for 65,536 envs x 8 OU pairs with no sets, S = 1,
16 and 1024 sets assigned at random, and S = N with the identity assignment; and for the C4 composite with no sets and
with S = 16.  The *_broker shapes add broker sets to the generator sets of the shape without the suffix.  L2-cold as
step_time.py: 8 rotating slabs, one stream, CUDA events around every launch (256 step launches per shape).
  python profiles/param_sets_cost.py [--out param_sets_cost.json]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from madigan_b200.environments import Env

dev = torch.device("cuda", 0)
N, SLABS, K = 65_536, 8, 32 * 8
C4_REWARD = dict(reward_shaper_config={"reward_shaper": "cosine_port_shaper", "desired_portfolio": [1.] + [0.] * 16,
                                       "cosine_temp": .025}, nstep_return=5, reduce_rewards=False)
SHAPES = {  # name: (data source config, reward, margins, costs, unit, S or None, assignment[, broker sets])
    "pairs_nosets": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, None, None),
    "pairs_S1": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, 1, "random"),
    "pairs_S16": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, 16, "random"),
    "pairs_S1024": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, 1024, "random"),
    "pairs_SN_identity": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, N, "identity"),
    "c4_nosets": (bench.COMPOSITE16, C4_REWARD, (.1, .25), (.001, 0.), 5000., None, None),
    "c4_S16": (bench.COMPOSITE16, C4_REWARD, (.1, .25), (.001, 0.), 5000., 16, "random"),
    "pairs_S16_broker": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, 16, "random", True),
    "pairs_S1024_broker": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, 1024, "random", True),
    "pairs_SN_identity_broker": (bench.PAIRS, bench.REWARD, (1., .25), (.02, .001), bench.UNIT, N, "identity", True),
    "c4_S16_broker": (bench.COMPOSITE16, C4_REWARD, (.1, .25), (.001, 0.), 5000., 16, "random", True),
}


def make(cfg, reward, margins, costs, S, assign, slab, broker=False):
    g = torch.Generator(device=dev).manual_seed(100 + slab)
    ids = None
    if S is not None:
        ids = (torch.arange(N, device=dev) if assign == "identity"
               else torch.randint(0, S, (N,), generator=g, device=dev)).to(torch.int32)
    e = Env("Composite", 1e6, {"data_source_config": cfg}, n_envs=N, window=bench.WINDOW, seed=bench.SEED, device=dev,
            env_offset=slab * N, reward=reward, param_sets=S, param_set=ids, broker_sets=S if broker else None)
    if S is not None:  # different markets: every slot of every set scaled by a factor in [0.9, 1.1]
        t = e.param_table
        t.mul_(0.9 + 0.2 * torch.rand(t.shape, generator=g, device=dev, dtype=torch.float64))
    e.setRequiredMargin(margins[0]); e.setMaintenanceMargin(margins[1])
    e.setTransactionCost(costs[0], 0.); e.setSlippage(costs[1], 0.)
    if broker:  # (the setters write every set) different frictions: every setting scaled by a factor in [0.9, 1.1]
        b = e.broker_table
        b.mul_(0.9 + 0.2 * torch.rand(b.shape, generator=g, device=dev, dtype=torch.float64))
    e.reset(fill_history=True)
    return e


def measure(name):
    cfg, reward, margins, costs, unit, S, assign, *broker = SHAPES[name]
    envs = [make(cfg, reward, margins, costs, S, assign, s, bool(broker)) for s in range(SLABS)]
    g = torch.Generator().manual_seed(1)
    acts = [(torch.randint(-1, 2, (N, 16), generator=g).double() * unit).to(dev) for _ in range(4)]
    for i in range(40 * SLABS):  # leave the synchronised start
        envs[i % SLABS].step(acts[i % 4], auto_reset=True)
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(K)]
    for i in range(K):
        ev[i][0].record()
        envs[i % SLABS].step(acts[i % 4])
        ev[i][1].record()
    torch.cuda.synchronize()
    st = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    for i in range(8 * SLABS):  # the steps above did not reset: back to the steady state
        envs[i % SLABS].step(acts[i % 4], auto_reset=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(K):
        envs[i % SLABS].step(acts[i % 4], auto_reset=True)
    b.record()
    torch.cuda.synchronize()
    fused = a.elapsed_time(b) * 1e3 / K
    done = float(torch.stack([e.t["done"].float().mean() for e in envs]).mean())
    del envs, acts
    torch.cuda.empty_cache()
    r = dict(step_kernel_median_us=st[K // 2], step_kernel_p10_us=st[K // 10], step_kernel_p90_us=st[9 * K // 10],
             step_autoreset_us=fused, done_rate=done, n_sets=S, assignment=assign, broker_sets=bool(broker))
    print(name, json.dumps(r), flush=True)
    return r


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out = dict(card=torch.cuda.get_device_name(0), nvidia_smi=smi[0] if smi else None, n_envs=N, slabs=SLABS,
               launches=K, results={})
    print(out["card"], out["nvidia_smi"], flush=True)
    for rep in range(2):  # two passes, in alternating order: the spread between them is the run-to-run noise
        for name in (SHAPES if rep == 0 else reversed(list(SHAPES))):
            out["results"].setdefault(name, []).append(measure(name))
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
