#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched Env.step hot path on B200 (BASELINE.json metric).

Workload (config.workload): C5 shape of SURVEY.md section 8(d) at the metric's 65,536 envs/GPU:
16-asset portfolios = 8 independent OU pairs (theta .015, phi .01, noise .03), transaction cost
.02 + slippage .001, required margin 1, DSR reward (adaptation .001, n-step 1, reduced), 64-step
observation ring, synthetic actions a*unit with a in {-1,0,+1}, envs auto-reset on done.

A "step" is one pass of the hot path (fused step kernel + masked auto-reset kernel) over one slab
of 65,536 envs.  The bench rotates over `--slabs` independent slabs so that a slab's state
(40 MB) has been evicted from the 126 MB L2 by the other slabs' traffic before it is stepped
again: every timed step streams its state from HBM ("inputs larger than L2").

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle) on host cores
  python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs as DIR/*.npy
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENVS_PER_GPU = 65_536
N_ASSETS = 16
WINDOW = 64
PAIRS = {f"pair{i}": {"data_source_type": "OUPair",
                      "data_source_config": {"theta": .015, "phi": .01, "noise": .03}} for i in range(8)}
REWARD = dict(reward_shaper_config={"reward_shaper": "DSR", "adaptation_rate": .001}, nstep_return=1,
              discount=0.99, reduce_rewards=True)
MARGINS = dict(required_margin=1., maintenance_margin=.25)
COSTS = dict(transaction_cost_rel=.02, transaction_cost_abs=0., slippage_rel=.001, slippage_abs=0.)
UNIT = 0.05 * 1_000_000. / 10.  # unit_size_proportion_avM .05 of init cash at the start price 10 (config.yaml:46)
SEED = 0x6d616469_67616e00 ^ 5
# Untimed steps per slab before the --warmup steps (see run_ours()).  The workload is not stationary at first: every
# env starts an episode at the same tick and the random policy ruins ~3 % of them per step, in waves; the finished
# share -- each a reset with a 64-tick history fill, ~half the cost of a step kernel at 3 % -- decays slowly as the
# population mixes: 3.0 % after 64 steps, 1.4 % after 256, 0.7 % after 1,024, 0.4 % after 4,096 (profiles/r2_notes.md).
# 16,384 steps per slab (~4 s; 20 steps cost 31.2 / 28.4 / 27.5 us per step after 2,048 / 8,192 / 16,384 of them)
# put the timed region into the long-run regime a training run spends its life in; the
# line reports the share it saw (done_rate_last_step).
SETUP_STEPS = 16384


def bytes_per_env_step(nA=N_ASSETS, G=8, R=2, ra=1, sh=1):
    """Algorithmic bytes per env-step, SURVEY.md 8(d) / BASELINE.md section 3."""
    return 8 * (14 * nA + 2 * G + 2 * R + 7 + ra + sh) + nA + 2


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([time.perf_counter()] + [x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self, t0=None, t1=None):
        """median SM clock / reasons over the samples taken between host times t0 and t1 (the timed region,
        which ends with a device synchronize); all samples when the window caught none"""
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        inside = [s[1:] for s in self.samples if t0 is None or (t0 <= s[0] <= t1)]
        if not inside:
            inside = [s[1:] for s in self.samples]
        for s in inside:
            try:
                sm.append(float(s[1])); mx.append(float(s[2]))
                for n, v in zip(names, s[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def make_env(device, env_offset, n_envs=ENVS_PER_GPU):
    from madigan_b200.environments import Env
    env = Env("Composite", 1_000_000., {"data_source_config": PAIRS}, n_envs=n_envs, window=WINDOW, seed=SEED,
              device=device, env_offset=env_offset, reward=REWARD)
    env.setRequiredMargin(MARGINS["required_margin"])
    env.setMaintenanceMargin(MARGINS["maintenance_margin"])
    env.setTransactionCost(COSTS["transaction_cost_rel"], COSTS["transaction_cost_abs"])
    env.setSlippage(COSTS["slippage_rel"], COSTS["slippage_abs"])
    env.reset(fill_history=True)
    return env


def synth_actions(n_batches, n_envs, generator_seed, device=None, pinned=False):
    import torch
    g = torch.Generator().manual_seed(generator_seed)
    out = []
    for _ in range(n_batches):
        a = torch.randint(-1, 2, (n_envs, N_ASSETS), generator=g).double() * UNIT
        if pinned:
            a = a.pin_memory()
        elif device is not None:
            a = a.to(device)
        out.append(a)
    return out


def reference_rate(seconds=6.0, threads=None):
    """The reference's own C++ env (oracle/_ref: Env.h/Broker/Account/Portfolio/DataSource compiled unmodified)
    stepping the same workload: one 16-asset env (8 reference OUPair sources) per host thread, each thread in
    its single-env `Env::step(units)` loop with reset on done -- the reference has no batching or threading of
    its own.  Returns (env-steps/s over all threads, threads, description)."""
    import threading as th
    import numpy as np
    from oracle import ref
    threads = threads or (os.cpu_count() or 1)
    rng = np.random.default_rng(0)
    acts = rng.integers(-1, 2, size=(64, N_ASSETS)).astype(np.float64) * UNIT
    envs = []
    for i in range(threads):
        e = ref.RefEnv(ref.MULTIPAIR, N_ASSETS, [.015, .01, .03], 1_000_000., seed=1000 + i)
        e.set(MARGINS["required_margin"], MARGINS["maintenance_margin"], COSTS["transaction_cost_rel"],
              COSTS["transaction_cost_abs"], COSTS["slippage_rel"], COSTS["slippage_abs"])
        e.reset()
        envs.append(e)
    # calibrate, then run every thread for about `seconds`
    t0 = time.perf_counter()
    envs[0].run(20_000, acts)
    per_step = (time.perf_counter() - t0) / 20_000
    steps = max(10_000, int(seconds / per_step))
    ts = [th.Thread(target=e.run, args=(steps, acts)) for e in envs]   # ctypes releases the GIL during the call
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    return steps * threads / dt, threads, (f"{threads} threads x {steps} Env::step(units) calls of one 16-asset env each "
                                           f"(reference C++ sources, g++ -O2 strict fp, reset on done; NO history fill, "
                                           f"no window, no agent reward: the C++ env alone), {dt:.2f} s")


def cpu_baseline(sample_envs=8192, sample_steps=24, threads=None):
    """CPU baseline on the host cores, a bounded sample of the same workload: the reference's own C++ env when
    oracle/_ref was built (kind "reference"), else the oracle port with OpenMP over envs (kind "port").
    A reported baseline, not the optimisation target."""
    try:
        from oracle import ref
        if ref.available():
            v, thr, desc = reference_rate(seconds=5.0, threads=threads)
            return {"value": v, "unit": "env-steps/s", "cores": thr, "kind": "reference", "sample": desc}
    except Exception:
        pass
    return port_rate(sample_envs, sample_steps, threads)


def port_rate(sample_envs=8192, sample_steps=24, threads=None):
    import numpy as np
    from madigan_b200.environments.data_source import make_params, make_reward
    from oracle.oracle import OracleBatch
    threads = threads or (os.cpu_count() or 1)
    P, _ = make_params("Composite", PAIRS, **MARGINS, **COSTS)
    R = make_reward(REWARD["reward_shaper_config"], 1, REWARD["discount"], True, n_assets=N_ASSETS)
    orc = OracleBatch(sample_envs, P, R, window=WINDOW, seed=SEED, threads=threads)
    orc.reset(fill_ticks=WINDOW)
    rng = np.random.default_rng(0)
    acts = [rng.integers(-1, 2, size=(sample_envs, N_ASSETS)).astype(np.float64) * UNIT for _ in range(4)]
    for i in range(2):
        orc.step(acts[i % 4])
    t0 = time.perf_counter()
    for i in range(sample_steps):
        orc.step(acts[i % 4])
        if orc.done.any():
            orc.reset(mask=orc.done.copy(), fill_ticks=WINDOW)
    dt = time.perf_counter() - t0
    return {"value": sample_envs * sample_steps / dt, "unit": "env-steps/s", "cores": threads, "kind": "port",
            "sample": f"{sample_envs} envs x {sample_steps} steps of the same workload (Philox noise, auto-reset with "
                      f"64-tick history fill, agent reward + DSR), oracle/mdg_oracle.c with OpenMP over envs, {dt:.2f} s"}


DUMP_LIMIT = 64 << 20  # bytes written by --dump-outputs


def write_outputs(out_dir, arrays, env_offset=0, limit=DUMP_LIMIT):
    """Write `arrays` (name -> numpy array with the env axis first) as <out_dir>/<name>.npy, floating arrays in their
    own precision and integer / bool ones as float64 / float32, plus env_index (the global index of each row's env).
    When they exceed `limit` bytes together, the rows of a fixed seeded sample of envs are written instead."""
    import numpy as np
    out = {k: (a if a.dtype.kind == "f" else a.astype(np.float64 if a.dtype.itemsize == 8 else np.float32))
           for k, a in arrays.items()}
    n = next(iter(out.values())).shape[0]
    per_env = sum(a.nbytes for a in out.values()) // n + 8
    keep = min(n, limit // per_env)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    out = {k: a[idx] for k, a in out.items()}
    out["env_index"] = (idx + env_offset).astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a))


def dump_outputs(out_dir, env, extra=None):
    """--dump-outputs: what the env's last Env.step call returned (State, reward, done and the BrokerResponse of
    EnvInfo, all views of live buffers that the next call overwrites), the agent and shaped rewards the same step
    computed, and `extra` tensors of the timed path; one row per env."""
    st, br, t = env._state(), env._info.brokerResponse, env.t
    arrays = {"state_price": st.price, "state_portfolio": st.portfolio, "state_timestamp": st.timestamp,
              "reward": t["reward"], "done": t["done"], "transaction_price": br.transactionPrice,
              "transaction_units": br.transactionUnits, "transaction_cost": br.transactionCost,
              "risk_info": br.riskInfo, "margin_call": br.marginCall, "agent_reward": env.agent_reward,
              "shaped_reward": t["shaped_reward"].permute(2, 0, 1)}
    arrays.update(extra or {})
    write_outputs(out_dir, {k: v.cpu().numpy() for k, v in arrays.items()}, env.env_offset)


def kernel_source_hash():
    import hashlib
    h = hashlib.sha256()
    for f in ("mdg_step_kernel.cuh", "mdg_common.cuh", "mdg_math.cuh"):
        h.update(open(os.path.join(ROOT, "madigan_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE step-kernel launch of this workload, from the committed
    `ncu --set full` capture (profiles/step_kernel_traffic.json names the report it was read from and the hash of the
    kernel sources it was taken with); bytes.  None when the kernel sources have changed since that capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")) as f:
            d = json.load(f)
        if d.get("kernel_source_hash") != kernel_source_hash():
            return None
        return d["dram_bytes_read"] + d["dram_bytes_write"]
    except Exception:
        return None


def ncu_pipes():
    """What the same committed capture says about the secondary ceilings (SURVEY 8d: say so when the kernel is bound
    by instruction issue / the fp64 pipe rather than by DRAM): per cent of peak; None when the sources have changed."""
    try:
        with open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")) as f:
            d = json.load(f)
        if d.get("kernel_source_hash") != kernel_source_hash():
            return None
        return {k: d[k] for k in ("issue_active_pct", "fp64_pipe_pct", "dram_throughput_pct", "duration_us") if k in d}
    except Exception:
        return None


def pin_to_gpu_numa_node(local):
    """Bind this process to the host cores nearest to GPU `local` (NVML's CPU affinity), before any pinned buffer is
    allocated: first-touch then places the staging buffers on the GPU's NUMA node, and 8 ranks stop sharing one
    root complex for their H2D streams.  Returns the number of cores, or None when NVML says nothing."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local])
                                              if os.environ.get("CUDA_VISIBLE_DEVICES", "").replace(",", "").isdigit()
                                              else local)
        n = (os.cpu_count() or 1)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = {64 * w + b for w, x in enumerate(words) for b in range(64) if (x >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus:
            pin_to_gpu_numa_node.before = allowed
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def config_dict(n_gpus, slabs, setup_steps=SETUP_STEPS):
    return {"workload": "C5 shape: 65,536 envs/GPU x 16-asset portfolios (8 OU pairs), cost .02 + slippage .001, "
                        "DSR reward n=1, 64-step observation ring, auto-reset on done",
            "envs_per_gpu": ENVS_PER_GPU, "n_assets": N_ASSETS, "window": WINDOW, "reward": "DSR(adaptation .001, n=1, reduced)",
            "slabs_per_gpu": slabs, "setup_steps_per_slab": setup_steps, "l2": f"rotating {slabs} slabs of 65,536 envs: resident state "
                                          f"{slabs} x 40 MB + rings exceeds the 126 MB L2, each step runs cold",
            "bytes_per_env_step": bytes_per_env_step(), "parallelism": f"env-slab sharding x{n_gpus}, no step-path collective"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from madigan_b200 import parallel

    rank, world, local = parallel.init_from_env("nccl")
    assert world == args.gpus or world == 1, f"WORLD_SIZE {world} != --gpus {args.gpus}"
    numa_cores = pin_to_gpu_numa_node(local)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    slabs, K, W = args.slabs, args.steps, args.warmup
    if slabs % max(1, min(args.streams, slabs)) != 0:
        raise SystemExit("--slabs must be a multiple of --streams (a slab always runs on the same stream)")
    per_rank = ENVS_PER_GPU * slabs
    envs = [make_env(dev, rank * per_rank + s * ENVS_PER_GPU) for s in range(slabs)]
    acts = synth_actions(8, ENVS_PER_GPU, 1234 + rank, device=dev)
    stream = torch.cuda.current_stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # Independent slabs are stepped round-robin on `--streams` CUDA streams, so that one slab's latency-bound
    # step kernel (65,536 envs = 14 warps per SM) overlaps the previous slab's reset kernels.
    n_str = max(1, min(args.streams, slabs))
    streams = [torch.cuda.Stream(dev) for _ in range(n_str)]

    def bind_all():  # slab i always runs on stream i % n_str: every launch and staging copy of the env follows it
        for i_, e_ in enumerate(envs):
            e_.bind_stream(streams[i_ % n_str])

    bind_all()

    def step_slab(i, acts_i):
        # the fused step kernel (dominant kernel) + masked auto-reset with history fill: one host call
        envs[i % slabs].step(acts_i, auto_reset=True)

    def fork(ev):
        for st in streams:
            st.wait_event(ev)

    def join():
        for st in streams:
            e_ = torch.cuda.Event()
            e_.record(st)
            stream.wait_event(e_)

    ev_w = torch.cuda.Event()
    ev_w.record(stream)
    fork(ev_w)
    # setup, untimed and independent of --warmup: every slab runs SETUP_STEPS steps, which allocates the per-stream
    # reset workspaces, loads the kernels and takes the slabs out of the synchronised start (all envs begin an episode
    # at the same tick, so the first ~40 steps see waves of simultaneous resets)
    for i in range(args.setup_steps * slabs):
        step_slab(i, acts[i % len(acts)])
    for i in range(W):
        step_slab(i, acts[i % len(acts)])
    join()
    barrier()

    # ---- timed regions.  The K steps of a region are issued R times (`--repeats`); the line reports the MEDIAN
    # repeat.  With `--graph` (default for K <= 512) the K-step sequence of a repeat -- kernels and, for the
    # end-to-end regions, the pinned-host copies, forked over the streams -- is captured into one CUDA graph
    # beforehand and the timed region is its launch: a 20-step region is ~1 ms of device work, less than the host
    # needs to enqueue it call by call.  The calls that are captured are the public ones (Env.step ...).
    R_ = max(1, args.repeats)
    use_graph = args.graph == "on" or (args.graph == "auto" and K <= 512)
    cap = torch.cuda.Stream(dev)  # capture origin stream
    counters = {"step_no": W, "t_issue": None}

    def timed_region(step_fn, restore_stream=False):
        """-> list of R_ region times (ms), each K calls of step_fn(i)"""
        graphs = []
        if use_graph:
            for r_ in range(R_):
                g_ = torch.cuda.CUDAGraph()
                torch.cuda.synchronize(dev)
                with torch.cuda.stream(cap):
                    g_.capture_begin(capture_error_mode="thread_local")
                    ev_f = torch.cuda.Event()
                    ev_f.record(cap)
                    for st in streams:
                        st.wait_event(ev_f)
                    for i in range(K):
                        step_fn(counters["step_no"] + i)
                    if restore_stream:
                        torch.cuda.set_stream(cap)
                    for st in streams:
                        e_ = torch.cuda.Event()
                        e_.record(st)
                        cap.wait_event(e_)
                    g_.capture_end()
                counters["step_no"] += K
                graphs.append(g_)
        out = []
        barrier()
        for r_ in range(R_):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            if use_graph:
                with torch.cuda.stream(cap):
                    ev0.record(cap)
                    graphs[r_].replay()
                    ev1.record(cap)
            else:
                ev0.record(stream)
                fork(ev0)
                t_i = time.perf_counter()
                for i in range(K):
                    step_fn(counters["step_no"] + i)
                t_i = (time.perf_counter() - t_i) / K * 1e3  # host time to enqueue one step
                counters["t_issue"] = t_i if counters["t_issue"] is None else min(counters["t_issue"], t_i)
                counters["step_no"] += K
                if restore_stream:
                    torch.cuda.set_stream(stream)
                join()
                ev1.record(stream)
            barrier()
            out.append(ev0.elapsed_time(ev1))
        return out

    # ---- timed region 1: device-resident inputs ("value")
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    launches0 = sum(e.launches for e in envs)
    t_region0 = time.perf_counter()
    ms_all = timed_region(lambda i: step_slab(i, acts[i % len(acts)]))
    # share of the envs that finished in each slab's last step of this region (the later regions use other action batches)
    done_rate_value = float(sum(float(e_.t["done"].float().mean()) for e_ in envs) / len(envs))
    launches = (sum(e.launches for e in envs) - launches0) // R_
    ms_total = sorted(ms_all)[len(ms_all) // 2]
    t_region1 = time.perf_counter()
    sampler.stop()
    clocks = sampler.summary(t_region0, t_region1)
    step_no = counters["step_no"]
    t_issue = counters["t_issue"]
    if args.dump_outputs and rank == 0:  # the slab of the last timed step, before the regions below step it again
        dump_outputs(args.dump_outputs, envs[(step_no - 1) % slabs])

    # ---- the dominant kernel alone (roofline): the step kernels of the `slabs` slabs back to back on ONE stream
    # between one pair of CUDA events (so that a launch's set-up overlaps its predecessor's execution, as it does in
    # the timed regions above; an event between two kernels exposes ~3 us of launch latency per kernel), the resets of
    # those slabs outside the pair.  `kernel_ms_single_launch` keeps the stricter one-event-pair-per-launch figure.
    for e_ in envs:
        e_.bind_stream(None)  # from here on the launches follow torch's current stream again
    rounds = max(4, min(K, 200) // slabs)
    g_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(rounds)]
    for r_ in range(rounds):
        g_ev[r_][0].record(stream)
        for s_ in range(slabs):
            envs[s_].step(acts[(r_ + s_) % len(acts)])
        g_ev[r_][1].record(stream)
        for s_ in range(slabs):
            envs[s_]._reset_launch(envs[s_].t["done"], WINDOW, True, None, None)
    barrier()
    kern_ms = sum(a.elapsed_time(b) for a, b in g_ev) / (rounds * slabs)
    KK = min(K, 200)
    k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KK)]
    for i in range(KK):
        env = envs[(step_no + i) % slabs]
        k_ev[i][0].record(stream)
        env.step(acts[i % len(acts)])
        k_ev[i][1].record(stream)
        env._reset_launch(env.t["done"], WINDOW, True, None, None)
    barrier()
    kern_ms_single = sum(a.elapsed_time(b) for a, b in k_ev) / KK

    # ---- timed region 2: end to end through the public API with HOST buffers ("e2e"): every step copies its
    # (N,16) fp64 units from pinned host memory, runs step + auto-reset, and reads reward/done back to the host;
    # the two streams let one slab's copies overlap the other's kernels
    host_acts = synth_actions(4, ENVS_PER_GPU, 999 + rank, pinned=True)
    host_reward = [torch.empty(ENVS_PER_GPU, dtype=torch.float64).pin_memory() for _ in range(n_str)]
    host_done = [torch.empty(ENVS_PER_GPU, dtype=torch.bool).pin_memory() for _ in range(n_str)]

    bind_all()
    set_stream = torch.cuda.set_stream  # (cheaper than a `with torch.cuda.stream(...)` context per call)

    def e2e_step(i):
        env = envs[i % slabs]
        j = i % n_str
        set_stream(streams[j])
        _s, r, d, _ = env.step(host_acts[i % 4], auto_reset=True)          # H2D of the units inside
        host_reward[j].copy_(env.shaped_reward[0, :, 0], non_blocking=True)  # D2H of the step's result
        host_done[j].copy_(d, non_blocking=True)

    ev_w.record(stream)
    fork(ev_w)
    for i in range(max(2 * slabs, W // 2)):  # every slab at least twice (first calls allocate staging buffers)
        e2e_step(i)
    set_stream(stream)
    join()
    barrier()
    e2e_all = timed_region(e2e_step, restore_stream=True)
    e2e_ms = sorted(e2e_all)[len(e2e_all) // 2]

    # ---- timed region 3 (extra key "e2e_actions"): the same end-to-end loop through Env.step_actions -- the agent's
    # DISCRETE actions (1 byte per asset) cross PCIe and DQN.action_to_transaction (dqn.py:160-179) runs fused in
    # front of the step, instead of a host-made fp64 units matrix (8 bytes per asset)
    g = torch.Generator().manual_seed(4242 + rank)
    host_a8 = [torch.randint(0, 3, (ENVS_PER_GPU, N_ASSETS), generator=g, dtype=torch.int8).pin_memory()
               for _ in range(4)]

    def e2e_actions_step(i):
        env = envs[i % slabs]
        j = i % n_str
        set_stream(streams[j])
        _s, r, d, _ = env.step_actions(host_a8[i % 4], action_atoms=3, unit_size=.05, auto_reset=True)
        host_reward[j].copy_(env.shaped_reward[0, :, 0], non_blocking=True)
        host_done[j].copy_(d, non_blocking=True)

    ev_w.record(stream)
    fork(ev_w)
    for i in range(max(2 * slabs, W // 2)):  # every slab at least twice (first calls allocate staging buffers)
        e2e_actions_step(i)
    set_stream(stream)
    join()
    barrier()
    e2e_act_all = timed_region(e2e_actions_step, restore_stream=True)
    e2e_act_ms = sorted(e2e_act_all)[len(e2e_act_all) // 2]
    for e_ in envs:
        e_.bind_stream(None)
    h2d = ENVS_PER_GPU * N_ASSETS * 8
    d2h = ENVS_PER_GPU * 8 + ENVS_PER_GPU

    # ---- episode statistics: the only cross-GPU data, gathered off the step path
    stats = envs[0].episode_stats()
    for e in envs[1:]:
        s2 = e.episode_stats()
        stats[:3] += s2[:3]; stats[5:] += s2[5:]
        stats[3] = torch.minimum(stats[3], s2[3]); stats[4] = torch.maximum(stats[4], s2[4])
    stats = parallel.reduce_episode_stats(stats, N_ASSETS)

    t = torch.tensor([ms_total, e2e_ms, kern_ms, e2e_act_ms, kern_ms_single], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, kern_ms, e2e_act_ms, kern_ms_single = (float(x) for x in t.cpu())
    if rank == 0:
        peak, which = peaks()
        B = bytes_per_env_step()
        value = world * ENVS_PER_GPU * K / (ms_total * 1e-3)
        achieved = B * ENVS_PER_GPU / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(world, slabs, args.setup_steps),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(), "ncu": ncu_pipes(), "peak_source": which,
                         "kernel": "mdg::step_kernel<PAIRS=true, 128 threads, 4 blocks/SM, TMA-staged operands>",
                         "kernel_ms": kern_ms, "kernel_ms_single_launch": kern_ms_single,
                         "kernel_timing": f"CUDA events around {slabs} consecutive launches (one per slab) on one stream, / {slabs}",
                         "algorithmic_bytes_per_launch": B * ENVS_PER_GPU},
            "e2e": {"value": world * ENVS_PER_GPU * K / (e2e_ms * 1e-3), "unit": "env-steps/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "e2e_actions": {"value": world * ENVS_PER_GPU * K / (e2e_act_ms * 1e-3), "unit": "env-steps/s",
                            "h2d_bytes_per_step": ENVS_PER_GPU * N_ASSETS, "d2h_bytes_per_step": d2h,
                            "api": "Env.step_actions(int8 actions, action_atoms=3, unit_size=.05): "
                                   "DQN.action_to_transaction fused in front of the step"},
            "gpu_launches": launches, "repeats": R_, "ms_per_repeat": ms_all, "e2e_ms_per_repeat": e2e_all,
            "timed_region": ("one CUDA graph launch per repeat (K steps x 2 kernels, forked over the streams)"
                             if use_graph else "K eager Env.step(auto_reset=True) calls"),
            "host_issue_ms_per_step": t_issue, "host_cores_bound": numa_cores, "clocks": clocks,
            "episode_stats": parallel.summarize_stats(stats, N_ASSETS),
        }
        es = line["episode_stats"]
        # share of the envs that finished (and were reset with a 64-tick history fill) in the last step: the random
        # policy ruins ~3 % of the envs per step early on and fewer once the survivors' equity has grown
        line["done_rate_last_step"] = es["n_done"] / max(es["n_envs"], 1)  # (not in config: both arms print the same config)
        line["done_rate_value_region"] = done_rate_value
        if world == 1 and not args.no_cpu_baseline:
            # in a subprocess: the reference's code is never loaded into the process that holds the product library
            try:
                before = getattr(pin_to_gpu_numa_node, "before", None)  # the baseline may use every host core again
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "5",
                                      "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT,
                                     preexec_fn=(lambda: os.sched_setaffinity(0, before)) if before else None)
                ref_line = json.loads(out.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref_line["cpu_baseline"]
            except Exception as ex:  # the oracle is test infrastructure; never let it break the GPU number
                line["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------
# The other BASELINE.json configurations (`--config c2|c3|c4|c5_1m`): parity-test cases first of all
# (tests/test_baseline_configs.py); here each gets a bench line with its own roofline (SURVEY.md section 8d's
# per-env-step bytes for ITS shape).  The driver's default run (`--config c5`, the metric's configuration) is unchanged.
# ---------------------------------------------------------------------------------------------------------------
COMPOSITE16 = {
    "sines": {"data_source_type": "Synth", "data_source_config": {
        "freq": [1., 0.3, 2., 0.5], "mu": [2., 2.1, 2.2, 2.3], "amp": [1., 1.2, 1.3, 1.],
        "phase": [0., 1., 2., 1.], "dX": 0.01, "noise": 0.01}},
    "ou": {"data_source_type": "OU", "data_source_config": {
        "mean": [10., 5., 1., 2.], "theta": [.08, .15, .15, .1], "phi": [.04, .04, .04, .04]}},
    "pair": {"data_source_type": "OUPair", "data_source_config": {"theta": .015, "phi": .01, "noise": .03}},
    "trend": {"data_source_type": "SimpleTrend", "data_source_config": {
        "trend_prob": [0.05, 0.02], "min_period": [5, 10], "max_period": [20, 30], "noise": [0.01, 0.005],
        "start": [10., 15.], "dYMin": [0.001, 0.01], "dYMax": [0.003, 0.03]}},
    "trendou": {"data_source_type": "TrendOU", "data_source_config": {
        "trend_prob": [0.05, 0.02], "min_period": [5, 10], "max_period": [20, 30], "dYMin": [0.001, 0.01],
        "dYMax": [0.003, 0.03], "start": [10., 15.], "theta": [.1, .05], "phi": [.02, .01],
        "noise_trend": [.01, .012], "ema_alpha": [0.1, 0.2]}},
    "trendyou": {"data_source_type": "TrendyOU", "data_source_config": {
        "trend_prob": [0.05, 0.02], "min_period": [5, 10], "max_period": [20, 30], "dYMin": [0.001, 0.01],
        "dYMax": [0.003, 0.03], "start": [10., 15.], "theta": [.1, .05], "phi": [.02, .01],
        "noise_trend": [.01, .012], "ema_alpha": [0.1, 0.2]}},
}
WORKLOADS = {
    # name: data source, envs (per GPU, or in total when "total"), nA, generator-state rows G, shaper moments R, ...
    "c2": dict(what="C2: 4,096 single-asset OU envs, log-return reward, window 64", ds=("OU", {"mean": [10.], "theta": [.08], "phi": [.04]}),
               envs=4096, nA=1, G=0, R=0, reward=dict(reward_shaper_config={"reward_shaper": None}, nstep_return=1, reduce_rewards=True),
               margins=(1., .25), costs=(0., 0.), unit=5000., kernel="mdg::step_kernel<generic>"),
    "c3": dict(what="C3: 65,536 OU-pair (2-asset stat-arb) envs/GPU, cost .02 + slippage .001, DSR n=1, window 64",
               ds=("OUPair", {"theta": .015, "phi": .01, "noise": .03}), envs=65536, nA=2, G=1, R=2,
               reward=dict(reward_shaper_config={"reward_shaper": "DSR", "adaptation_rate": .001}, nstep_return=1, reduce_rewards=True),
               margins=(1., .25), costs=(.02, .001), unit=5000., kernel="mdg::step_kernel<PAIRS>"),
    "c4": dict(what="C4: 65,536 composite-synth 16-asset portfolios/GPU (Synth4 + OU4 + OUPair + SimpleTrend2 + TrendOU2 + "
                    "TrendyOU2), required margin .1, cost .001, PPC reward n=5 per asset, standard_normal fp32 window every step",
               ds=("Composite", COMPOSITE16), envs=65536, nA=16, G=4 + 1 + 4 + 6 + 8, R=0,
               reward=dict(reward_shaper_config={"reward_shaper": "cosine_port_shaper", "desired_portfolio": [1.] + [0.] * 16,
                                                 "cosine_temp": .025}, nstep_return=5, reduce_rewards=False),
               margins=(.1, .25), costs=(.001, 0.), unit=5000., window_norm="standard_normal", kernel="mdg::step_kernel<generic>"),
    "c5_1m": dict(what="C5 sweep: 1,048,576 16-asset OU-pair portfolios IN TOTAL, sharded over the GPUs (one slab per GPU, one "
                       "launch per step), cost .02 + slippage .001, DSR n=1, window 64, episode statistics all-reduced (NCCL) every "
                       "1,000 steps inside the timed region",
                  ds=("Composite", PAIRS), envs=1_048_576, total=True, nA=16, G=8, R=2, reward=REWARD, margins=(1., .25),
                  costs=(.02, .001), unit=UNIT, stats_every=1000, setup=2048, kernel="mdg::step_kernel<PAIRS>"),
}


def run_workload(args):
    """One bench line for a non-default BASELINE configuration: K eager `Env.step(units, auto_reset=True)` calls on one
    slab per GPU (device-resident units; `e2e` repeats them with pinned-host units and a D2H read of reward/done)."""
    import torch
    import torch.distributed as dist
    from madigan_b200 import parallel
    from madigan_b200.environments import Env

    wl = WORKLOADS[args.config]
    rank, world, local = parallel.init_from_env("nccl")
    pin_to_gpu_numa_node(local)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    total = bool(wl.get("total"))
    if total:
        off, n = parallel.shard_envs(wl["envs"], world, rank)
    else:
        off, n = rank * wl["envs"], wl["envs"]
    nA, K, W = wl["nA"], args.steps, args.warmup
    env = Env(wl["ds"][0], 1_000_000., {"data_source_config": wl["ds"][1]}, n_envs=n, window=WINDOW, seed=SEED,
              device=dev, env_offset=off, reward=wl["reward"])
    env.setRequiredMargin(wl["margins"][0]); env.setMaintenanceMargin(wl["margins"][1])
    env.setTransactionCost(wl["costs"][0], 0.); env.setSlippage(wl["costs"][1], 0.)
    env.reset(fill_history=True)
    g = torch.Generator().manual_seed(77 + rank)
    acts = [(torch.randint(-1, 2, (n, nA), generator=g).double() * wl["unit"]).to(dev) for _ in range(4)]
    host_acts = [a.cpu().pin_memory() for a in acts[:2]]
    norm = wl.get("window_norm")
    wout = torch.empty((n, WINDOW, nA), dtype=torch.float32, device=dev) if norm else None
    stats_every = wl.get("stats_every")
    host_r = torch.empty(n, dtype=torch.float64).pin_memory()
    host_d = torch.empty(n, dtype=torch.bool).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one(i, a):
        env.step(a, auto_reset=True)
        if norm:
            env.window(norm, out=wout)
        if stats_every and (i + 1) % stats_every == 0:
            parallel.reduce_episode_stats(env.episode_stats(), nA)  # the only cross-GPU traffic, off the step path

    setup = wl.get("setup", args.setup_steps_small)
    for i in range(setup + W):
        one(i, acts[i % 4])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    ms_all = []
    l0 = env.launches
    t0 = time.perf_counter()
    for r_ in range(max(1, args.repeats)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(K):
            one(i, acts[i % 4])
        e1.record()
        barrier()
        ms_all.append(e0.elapsed_time(e1))
    t1 = time.perf_counter()
    launches = (env.launches - l0) // max(1, args.repeats)
    sampler.stop()
    clocks = sampler.summary(t0, t1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env, {"window": wout} if norm else None)
    ms_total = sorted(ms_all)[len(ms_all) // 2]
    # the dominant kernel alone: events around the step launch, the reset outside the pair
    KK = min(K, 100)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KK)]
    for i in range(KK):
        ev[i][0].record()
        env.step(acts[i % 4])
        ev[i][1].record()
        env._reset_launch(env.t["done"], WINDOW, True, None, None)
    barrier()
    kern_ms = sum(a.elapsed_time(b) for a, b in ev) / KK
    # end to end with host buffers
    for i in range(4):
        env.step(host_acts[i % 2], auto_reset=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        _s, r, d, _ = env.step(host_acts[i % 2], auto_reset=True)
        if norm:
            env.window(norm, out=wout)
        host_r.copy_(r, non_blocking=True)
        host_d.copy_(d, non_blocking=True)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    stats = parallel.reduce_episode_stats(env.episode_stats(), nA)
    t = torch.tensor([ms_total, e2e_ms, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, kern_ms = (float(x) for x in t.cpu())
    if rank == 0:
        peak, which = peaks()
        ra = 1 if wl["reward"]["reduce_rewards"] else nA
        B = bytes_per_env_step(nA, wl["G"], wl["R"], ra)
        n_all = wl["envs"] if total else wl["envs"] * world
        line = {
            "metric": "env-steps/sec", "value": n_all * K / (ms_total * 1e-3), "unit": "env-steps/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True,
            "scaling": "strong" if total else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["what"], "envs_total": n_all, "envs_this_gpu": n, "n_assets": nA, "window": WINDOW,
                       "bytes_per_env_step": B, "setup_steps": setup,
                       "l2": "one slab per GPU stepped repeatedly: its state is %s the 126 MB L2" %
                             ("larger than" if B * n > 126e6 else "SMALLER than (L2-warm, stated)"),
                       "parallelism": f"env-slab sharding x{world}, no step-path collective"},
            "roofline": {"bound": "hbm", "achieved": B * n / (kern_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": B * n / (kern_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": which,
                         "kernel": wl["kernel"], "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": B * n},
            "e2e": {"value": n_all * K / (e2e_ms * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": n * nA * 8,
                    "d2h_bytes_per_step": n * 9},
            "gpu_launches": launches, "repeats": max(1, args.repeats), "ms_per_repeat": ms_all, "clocks": clocks,
            "episode_stats": parallel.summarize_stats(stats, nA),
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()



def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path on the box's host cores, all threads.
    oracle/_ref (the reference's C++ sources compiled unmodified against an Eigen shim) when it was built, else
    the oracle port.  A "step" here is a bounded sample of the arm's workload: `sample` env-steps."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    cfg = config_dict(args.gpus, args.slabs, args.setup_steps)
    kind = "port"
    try:
        from oracle import ref
        if ref.available():
            kind = "reference"
    except Exception:
        pass
    if kind == "reference":
        # K timed steps, each = `threads` envs x `per` Env::step calls; W warm-up steps likewise
        for _ in range(max(1, min(args.warmup, 3))):
            reference_rate(seconds=0.2, threads=threads)
        t0 = time.perf_counter()
        n_rounds = max(1, min(args.steps, 20))
        rates = []
        for _ in range(n_rounds):
            v, thr, desc = reference_rate(seconds=1.0, threads=threads)
            rates.append(v)
        dt = time.perf_counter() - t0
        value = sum(rates) / len(rates)
        sample = desc
        ms_per_step = dt / n_rounds * 1e3
    else:
        r = port_rate(8192, max(4, min(args.steps, 40)), threads)
        value, sample, ms_per_step = r["value"], r["sample"], 8192 / r["value"] * 1e3
    line = {"impl": "reference", "reference_sample": sample, "metric": "env-steps/sec", "value": value, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps per repeat (default 4000 for c5 and the reference arm, 200 for the other --config)")
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--slabs", type=int, default=8)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="c5", choices=["c5"] + sorted(WORKLOADS),
                    help="c5 (default) = the metric's configuration; the others are BASELINE.json's remaining configurations")
    ap.add_argument("--setup-steps-small", type=int, default=256, help="untimed steps before the warm-up (--config != c5)")
    ap.add_argument("--setup-steps", type=int, default=SETUP_STEPS, help="untimed steps per slab before the warm-up")
    ap.add_argument("--repeats", type=int, default=5, help="the K timed steps are issued this many times; the median is reported")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="timed region as one CUDA graph launch (auto: when --steps <= 512)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0's envs; "
                         "a fixed seeded sample of them above 64 MB)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 200 if args.impl == "ours" and args.config != "c5" else 4000
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none")
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "c5":
        run_workload(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
