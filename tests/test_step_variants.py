"""Every instantiation of the fused step kernel, pinned to the oracle, and the episode statistics against fp64.

`launch_step` (csrc/mdg_step_kernel.cuh) compiles one template body into 40 kernels.  Which one runs depends on the
launch: all-OU-pairs sources or not (PAIRS), one wave or more (MINB 4 or 3; MINB 3 also switches on the predicated
TX2 gate and flat-position clean-up), N % 128 == 0 with the Env's slab layout (BULK, the TMA / row-copy ring), actions
or weights (ACTIONS), the MDG_BS64 knob (64-thread kernels), and parameter / broker sets.  Each row below drives one
of them and checks, with torch.profiler, that a step of each kind it takes launches exactly the kernel the row names
(profiled in a fresh child process, see `launched`), so that a row cannot silently drift to another instantiation
when the dispatcher changes.

`REGISTRY` maps every kernel name to the rows that cover it; a CPU test compares its keys with the step kernels `nm`
finds in the built library, so a new instantiation fails the suite until a row covers it.

The oracle rows use test_gpu_parity's machinery: injected noise, explicit masked resets with history fill, leverage,
costs and slippage; ledgers, units, risk codes and done flags bit-exact, prices bit-exact for arithmetic-only sources.
"""
import math
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from test_gpu_parity import (CASES, SHAPERS, close, compare_step, compare_windows, cpu, gen_units, make_pair, noise,
                             same_bits, sync_state_from_oracle)

ONE_WAVE = 148 * 512 * 2  # launch_step: up to two waves of four 128-thread blocks per SM take the MINB 4 kernels
BS64_MAX = 148 * 7 * 64   # MDG_BS64: one-wave launches of up to seven 64-thread blocks per SM
BULK1, RAGGED1 = 384, 385
BULK3, RAGGED3 = 1185 * 128, ONE_WAVE + 1  # 151,680 and 151,553
GATES = ("fast", "exact")
ACT_DRIVES = ("actions", "weights")
WINDOW = 8
MARGINS, COSTS, SCALE = (.1, .25), (.02, 1.5, .001, .002), 400_000.
ATOMS, UNIT = 7, .04
DSR = SHAPERS[0]                                                              # DSR n=1 reduced: the inline shaper
SORTINO = next(s for s in SHAPERS if s["reward_shaper_config"]["reward_shaper"] == "sortino_shaperA")  # n=6

# 7 OU pairs + one two-asset OU: 16 assets, exact prices, not all-pairs (the generic path)
OU_MIX = {**{f"pair{i}": {"data_source_type": "OUPair", "data_source_config": {"theta": .015, "phi": .01, "noise": .03}}
             for i in range(7)},
          "ou": {"data_source_type": "OU", "data_source_config": {"mean": [10., 5.], "theta": [.08, .15],
                                                                  "phi": [.04, .02]}}}
PAIRS_CASES = ("pairs8",)
ORACLE_THREADS = os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------- launch probe
_STEP_KERNEL = re.compile(r"mdg::(step_kernel64|step_kernel|step_sets_broker_kernel|step_sets_kernel)\s*<([^<>()]*)>")


def step_kernel_name(name):
    """`family<args>` without whitespace for a demangled (or mangled) mdg::step* kernel name, else None"""
    if name.startswith("_Z"):
        name = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip() or name
    m = _STEP_KERNEL.search(name)
    return None if m is None else f"{m.group(1)}<{re.sub(r'[ \t]+', '', m.group(2))}>"


def launched_step_kernels(fn):
    """Run fn under torch.profiler (CUDA activity) and return the set of step kernels it launched.  Fails when the
    profiler recorded no CUDA kernel at all: a probe that sees nothing must not pass."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [ev.name for ev in prof.events() if ev.device_type == DeviceType.CUDA]
    assert any(not n.startswith(("Memcpy", "Memset")) for n in names), \
        f"the profiler recorded no CUDA kernel (events: {[ev.name for ev in prof.events()]})"
    return {k for k in map(step_kernel_name, names) if k is not None}


def _on(knobs, name):
    v = knobs.get(name, "")
    try:
        return int(v) != 0  # launch_step reads the knobs with atoi
    except ValueError:
        return False


def expected_kernel(pairs, N, acts, family="step_kernel", knobs=None):
    """launch_step's choice for an Env of N envs (its state slab is aligned and equally spaced), restated"""
    knobs = os.environ if knobs is None else knobs
    b = lambda x: "true" if x else "false"
    bs = 64 if family == "step_kernel" and pairs and _on(knobs, "MDG_BS64") and N <= BS64_MAX else 128
    small = N <= ONE_WAVE
    # the row-copy ring (MDG_NO_TMA) is used in one-wave launches only
    bulk = pairs and not _on(knobs, "MDG_NO_BULK") and N % bs == 0 and (small or not _on(knobs, "MDG_NO_TMA"))
    if bs == 64:
        return f"step_kernel64<{b(acts)},{b(bulk)}>"
    return f"{family}<{b(pairs)},128,{4 if small else 3},{b(acts)},{b(bulk)}>"


def assert_launched(got, want, tag):
    assert got == {want}, f"{tag}: launched {sorted(got)}, the row names {want}"


# ---------------------------------------------------------------------------------------------------- rows
def _plain_rows():
    rows = [("pairs8", n, d, "fast") for n in (BULK1, RAGGED1) for d in ("units", "single_hold") + ACT_DRIVES]
    rows += [("pairs8", n, d, g) for n in (BULK3, RAGGED3) for d in ("units", "single_hold") + ACT_DRIVES for g in GATES]
    rows += [("trends6", RAGGED1, d, "fast") for d in ("units", "single_hold")]
    rows += [("composite16", RAGGED1, "units", "fast")] + [("ou3", RAGGED1, d, "fast") for d in ACT_DRIVES]
    rows += [("trends6", RAGGED3, d, g) for d in ("units", "single_hold") for g in GATES]
    rows += [("composite16", RAGGED3, "units", g) for g in GATES]
    rows += [("ou3", RAGGED3, d, g) for d in ACT_DRIVES for g in GATES]
    rows += [("trends6", RAGGED3, "sortino", "fast")]
    return rows


PLAIN_ROWS = _plain_rows()
KNIFE_ROWS = [(c, n, g) for c, n in (("pairs8", RAGGED3), ("pairs8", BULK3), ("ou_mix", RAGGED3)) for g in GATES]
FREE_ROWS = [("pairs8", BULK3), ("pairs8", RAGGED3), ("composite16", RAGGED3)]
SET_SHAPES = [("pairs8", n, act) for n in (BULK1, RAGGED1, BULK3, RAGGED3) for act in ("units", "acts")]
SET_SHAPES += [("composite", n, act) for n in (RAGGED1, RAGGED3) for act in ("units", "acts")]
# knob rows: plain oracle rows rerun in a child process with the knob set (knobs are read once per process)
KNOB_ROWS = {
    "MDG_BS64": [("pairs8", n, d, "fast") for n in (BULK1, RAGGED1) for d in ("units",) + ACT_DRIVES],
    "MDG_NO_TMA": [("pairs8", BULK1, d, "fast") for d in ACT_DRIVES],
    "MDG_NO_BULK": [("pairs8", BULK1, d, "fast") for d in ACT_DRIVES],
}


def row_id(r):
    return "-".join(str(x) for x in r)


def _registry():
    reg = {}

    def add(name, row):
        reg.setdefault(name, []).append(row)

    for r in PLAIN_ROWS:
        add(expected_kernel(r[0] in PAIRS_CASES, r[1], r[2] in ACT_DRIVES, knobs={}), f"test_plain_oracle[{row_id(r)}]")
    for knob, rows in KNOB_ROWS.items():
        for r in rows:
            add(expected_kernel(True, r[1], r[2] in ACT_DRIVES, knobs={knob: "1"}),
                f"test_knob_rows[{knob}] -> test_plain_oracle[{row_id(r)}]")
    for r in KNIFE_ROWS:
        add(expected_kernel(r[0] in PAIRS_CASES, r[1], False, knobs={}), f"test_knife_edge_multi_wave[{row_id(r)}]")
    for r in FREE_ROWS:
        add(expected_kernel(r[0] in PAIRS_CASES, r[1], False, knobs={}), f"test_free_running_multi_wave[{row_id(r)}]")
    add(expected_kernel(True, ONE_WAVE, False, knobs={}), "test_one_wave_boundary")
    for s in SET_SHAPES:
        for family in ("step_sets_kernel", "step_sets_broker_kernel", "step_kernel"):
            add(expected_kernel(s[0] in PAIRS_CASES, s[1], s[2] == "acts", family, knobs={}),
                f"test_sets_rows[{row_id(s)}]")
    return reg


REGISTRY = _registry()
ORACLE_TESTS = ("test_plain_oracle", "test_knob_rows", "test_knife_edge_multi_wave", "test_free_running_multi_wave")


# ---------------------------------------------------------------------------------------------------- probe pass
# torch.profiler stops recording device activity in a process that has done a lot of GPU and host work (seen on B200
# machines after a few of the multi-wave oracle rows: the runtime calls are still recorded, the kernels and copies are
# not).  So the launches are probed in a fresh child process that builds every row's Env exactly as the row does
# (same source, N, window, reward, flags and knobs; the Env allocates the same slab layout) and profiles one step of
# each kind the row takes.  Each row then asserts the kernel its configuration launched there.
def _plain_env(cfg, N, window, reward=None, margins=MARGINS, costs=COSTS, seed=7, env_offset=0, gate="fast",
               ds_type="Composite"):
    from madigan_b200.environments import Env
    env = Env(ds_type, 1e6, {"data_source_config": cfg}, n_envs=N, window=window, seed=seed, env_offset=env_offset,
              reward=reward)
    env.setRequiredMargin(margins[0]); env.setMaintenanceMargin(margins[1])
    env.setTransactionCost(costs[0], costs[1]); env.setSlippage(costs[2], costs[3])
    env.flags = A.FLAG_FORCE_EXACT_GATE if gate == "exact" else 0
    return env


def _probe_step(env, kind, nA, rng, injected=True):
    N = env.N
    kw = {}
    if injected:
        kw = dict(normals=rng.standard_normal((max(env.P.n_normals, 1), N)), uniforms=rng.random((max(env.P.n_uniforms,
                                                                                                        1), N)))
    if kind == "units":
        u = torch.from_numpy(rng.integers(-1, 2, size=(N, nA)) * 1000.)
        return launched_step_kernels(lambda: env.step(u, **kw))
    if kind == "single":
        u = torch.from_numpy(rng.integers(-1, 2, size=N) * 1000.)
        return launched_step_kernels(lambda: env.step(3 % nA, u, **kw))
    if kind == "hold":
        return launched_step_kernels(lambda: env.step(**kw))
    if kind == "actions":
        a = torch.from_numpy(rng.integers(0, ATOMS, size=(N, nA)).astype(np.int8))
        return launched_step_kernels(lambda: env.step_actions(a, action_atoms=ATOMS, unit_size=UNIT, **kw))
    w = torch.from_numpy(rng.random((N, nA + 1)).astype(np.float32))
    return launched_step_kernels(lambda: env.step_weights(w, **kw))


def probe_all(plain_rows):
    """{probe key: sorted kernel names}: one profiled step of every kind of every row (run in a fresh process)"""
    from test_broker_sets import BROKER, broker_env, plain_env
    from test_param_sets import COMPOSITE, COMPOSITE_SETS, PAIR_SETS, make_env
    rng = np.random.default_rng(0)
    out = {}
    for r in plain_rows:
        case, N, drive, gate = r
        env = _plain_env(CASES[case][1], N, WINDOW, SORTINO if drive == "sortino" else DSR, gate=gate,
                         ds_type=CASES[case][0])
        for kind in sorted({step_kind(drive, t) for t in range(3)}):
            out[f"plain:{row_id(r)}:{kind}"] = sorted(_probe_step(env, kind, env.nA, rng))
        del env
    if plain_rows is not PLAIN_ROWS:
        return out
    for r in KNIFE_ROWS:
        cfg = CASES["pairs8"][1] if r[0] == "pairs8" else OU_MIX
        env = _plain_env(cfg, r[1], 4, None, margins=(.2, .25), costs=(.002, .5, .001, .002), seed=5, gate=r[2])
        out[f"knife:{row_id(r)}"] = sorted(_probe_step(env, "units", 16, rng))
    for r in FREE_ROWS:
        env = _plain_env(CASES[r[0]][1], r[1], WINDOW, None, seed=1234, env_offset=1000, ds_type=CASES[r[0]][0])
        out[f"free:{row_id(r)}"] = sorted(_probe_step(env, "units", env.nA, rng, injected=False))
    env = _plain_env(CASES["pairs8"][1], ONE_WAVE, 4, None)
    out["boundary"] = sorted(_probe_step(env, "units", 16, rng))
    del env
    for sh in SET_SHAPES:
        cfg, N, drive = sh
        sets = PAIR_SETS[:2] if cfg == "pairs8" else COMPOSITE_SETS[:2]
        base = PAIR_SETS[0] if cfg == "pairs8" else COMPOSITE
        assign = torch.from_numpy(rng.integers(0, 2, N).astype(np.int32))
        envs = {"step_sets_kernel": make_env(base, N, sets, assign, reward=DSR, window=WINDOW),
                "step_sets_broker_kernel": broker_env(base, N, sets, BROKER[:2], assign, reward=DSR, window=WINDOW),
                "step_kernel": make_env(sets[0], N, reward=DSR, window=WINDOW)}
        for family, env in envs.items():
            kind = "units" if drive == "units" else "actions"
            out[f"sets:{row_id(sh)}:{family}"] = sorted(_probe_step(env, kind, env.nA, rng, injected=False))
        del envs
    return out


@pytest.fixture(scope="module")
def launched():
    """probe_all in a fresh child process (it inherits the knobs of this one)"""
    import json
    import tempfile
    here = os.path.dirname(os.path.abspath(__file__))
    rows = os.environ.get("MDG_PROBE_ROWS")  # a knob child probes only the rows it runs
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "launched.json")
        code = ("import json, sys; sys.path[:0] = [%r, %r]; import test_step_variants as T; rows = %s; "
                "json.dump(T.probe_all(T.PLAIN_ROWS if rows is None else [tuple(r) for r in rows]), open(%r, 'w'))"
                % (here, os.path.dirname(here), rows if rows else "None", path))
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        return {k: set(v) for k, v in json.load(open(path)).items()}


# ---------------------------------------------------------------------------------------------------- CPU
def _library():
    from madigan_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from madigan_b200.build import build
        build()
    return _lib.LIB_PATH


def test_registry_lists_every_step_instantiation():
    """REGISTRY's keys are exactly the step kernels of the built library; each has a row, and each plain (oracle-
    checkable) kernel an oracle row -- a sets row, which compares with plain Envs only, is not enough for it."""
    nm = shutil.which("nm")
    assert nm, "nm (binutils) is needed to list the library's kernels"
    out = subprocess.run([nm, "-C", "--defined-only", _library()], capture_output=True, text=True, check=True).stdout
    found = {k for k in map(step_kernel_name, out.splitlines()) if k is not None}
    assert found, "no mdg::step* kernel in the library"
    missing, stale = sorted(found - set(REGISTRY)), sorted(set(REGISTRY) - found)
    assert not missing and not stale, f"instantiations without a row: {missing}; rows naming no kernel: {stale}"
    for name, rows in REGISTRY.items():
        assert rows, name
        if name.startswith(("step_kernel<", "step_kernel64<")):
            assert any(r.startswith(ORACLE_TESTS) for r in rows), f"{name}: no oracle row"


def test_kernel_names_normalise():
    """nm -C's and the profiler's spellings of one kernel compare equal"""
    want = "step_kernel<true,128,3,false,true>"
    assert step_kernel_name("void mdg::step_kernel<true, 128, 3, false, true>(mdg::StepArgs)") == want
    assert step_kernel_name("void mdg::step_kernel<true,128,3,false,true>(mdg::StepArgs)") == want
    assert step_kernel_name("0000000000013a30 W void mdg::step_kernel64<true, false>(mdg::StepArgs)") == \
        "step_kernel64<true,false>"
    assert step_kernel_name("void mdg::step_sets_broker_kernel<false, 128, 4, true, false>(mdg::StepSetsBrokerArgs)") \
        == "step_sets_broker_kernel<false,128,4,true,false>"
    assert step_kernel_name("void mdg::reset_fill_pairs_kernel(mdg::ResetWsArgs)") is None
    if shutil.which("c++filt"):
        assert step_kernel_name("_ZN3mdg11step_kernelILb1ELi128ELi3ELb0ELb1EEEvNS_8StepArgsE") == want


def test_rows_reach_the_sizes_they_name():
    """The size classes of the rows sit on the dispatcher's edges."""
    assert BULK1 % 128 == 0 and RAGGED1 % 128 and BULK3 % 128 == 0 and RAGGED3 % 128
    assert BULK1 <= BS64_MAX and RAGGED1 <= BS64_MAX and BULK1 % 64 == 0
    assert RAGGED3 == ONE_WAVE + 1 and ONE_WAVE < BULK3 < ONE_WAVE + 1024
    assert expected_kernel(True, ONE_WAVE, False, knobs={}) == "step_kernel<true,128,4,false,true>"
    assert expected_kernel(True, BULK3, False, knobs={}) == "step_kernel<true,128,3,false,true>"


# ---------------------------------------------------------------------------------------------------- GPU: oracle rows
def step_kind(drive, t):
    if drive in ("units", "sortino"):
        return "units"
    if drive == "single_hold":
        return "hold" if t % 3 == 1 else "single"
    return drive


def make_steps(kind, env, orc, rng, P, N, t):
    """(GPU step, oracle step) on the same inputs"""
    nA = P.n_assets
    nz, uz = noise(rng, P, N)
    if kind == "units":
        u = gen_units(rng, orc, N, nA, SCALE)
        return (lambda: env.step(torch.from_numpy(u), normals=nz, uniforms=uz),
                lambda: orc.step(u, normals=nz, uniforms=uz))
    if kind == "single":
        idx = (5 * t + 3) % nA
        u = np.ascontiguousarray(gen_units(rng, orc, N, nA, SCALE)[:, idx])
        return (lambda: env.step(idx, torch.from_numpy(u), normals=nz, uniforms=uz),
                lambda: orc.step(u, asset_idx=idx, normals=nz, uniforms=uz))
    if kind == "hold":
        # a hold step writes no order response (the last order's stays in the buffers); the oracle reports an empty one
        for name in ("trans_price", "trans_units", "trans_cost", "risk", "margin_call"):
            env.t[name].zero_()
        return (lambda: env.step(normals=nz, uniforms=uz), lambda: orc.step(None, normals=nz, uniforms=uz))
    if kind == "actions":
        acts = rng.integers(0, ATOMS, size=(N, nA)).astype(np.int8)
        return (lambda: env.step_actions(torch.from_numpy(acts), action_atoms=ATOMS, unit_size=UNIT, normals=nz,
                                         uniforms=uz),
                lambda: orc.step_actions(acts, ATOMS, UNIT, normals=nz, uniforms=uz))
    assert kind == "weights"
    w = rng.random((N, nA + 1)).astype(np.float32)
    w[rng.random(N) < .05] = 0.                              # zero-sum rows
    w[:, 0] += rng.random(N).astype(np.float32) * 3          # mostly cash
    return (lambda: env.step_weights(torch.from_numpy(w), normals=nz, uniforms=uz),
            lambda: orc.step_weights(w, normals=nz, uniforms=uz))


def start_pair(case, N, reward, gate, seed=7):
    """Env + oracle from the same constructor state, then a full reset with history fill on injected noise"""
    env, orc, P = make_pair(case, N, WINDOW, reward, MARGINS, COSTS, seed=seed)
    orc.threads = ORACLE_THREADS
    env.flags = A.FLAG_FORCE_EXACT_GATE if gate == "exact" else 0
    orc.reset(fill_ticks=1, clear_nstep=False)
    close(cpu(env.t["price"]), orc.state()["price"], rtol=1e-9)
    sync_state_from_oracle(env, orc)
    return env, orc, P


@pytest.mark.gpu
@pytest.mark.parametrize("case,N,drive,gate", PLAIN_ROWS, ids=[row_id(r) for r in PLAIN_ROWS])
def test_plain_oracle(case, N, drive, gate, launched):
    """One plain instantiation against the oracle: multi-asset units (DSR n=1, or sortino n=6), single-asset and hold
    steps, discrete actions or target weights; masked resets with history fill whenever envs finish."""
    multi = N > ONE_WAVE
    T = 8 if multi else 30
    env, orc, P = start_pair(case, N, SORTINO if drive == "sortino" else DSR, gate)
    exact = not CASES[case][2]
    rng = np.random.default_rng(N + 7 * len(drive))
    nz, uz = noise(rng, P, N, ticks=WINDOW)
    env.reset(fill_history=True, normals=nz, uniforms=uz)
    orc.reset(fill_ticks=WINDOW, normals=nz, uniforms=uz)
    compare_windows(env, orc, exact)
    want = expected_kernel(case in PAIRS_CASES, N, drive in ACT_DRIVES)
    for kind in {step_kind(drive, t) for t in range(3)}:
        assert_launched(launched[f"plain:{row_id((case, N, drive, gate))}:{kind}"], want, kind)
    seen, n_done, traded = set(), 0, 0
    for t in range(T):
        kind = step_kind(drive, t)
        gpu_step, orc_step = make_steps(kind, env, orc, rng, P, N, t)
        gpu_step()
        orc_step()
        compare_step(env, orc, exact, t, shaped=True)
        if kind != "hold":
            seen |= set(np.unique(orc.risk).tolist())
            traded += int(np.count_nonzero(orc.trans_units))
        if orc.done.any():
            n_done += int(orc.done.sum())
            nz, uz = noise(rng, P, N, ticks=WINDOW)
            env.reset(mask=torch.from_numpy(orc.done.copy()), fill_history=True, normals=nz, uniforms=uz)
            orc.reset(mask=orc.done.copy(), fill_ticks=WINDOW, normals=nz, uniforms=uz)
            if not multi:
                compare_windows(env, orc, exact)
    compare_windows(env, orc, exact)
    d_o, d_g = orc.derived(), env._derived()
    for name, ref in d_o.items():
        if name == "risk":
            assert np.array_equal(cpu(d_g[name]), ref)
        elif exact:
            assert same_bits(cpu(d_g[name]), ref), name
        else:
            close(cpu(d_g[name]), ref, atol=1e-9)
    assert traded > N, traded
    if drive in ("units", "sortino"):  # both gates' refusals happened, and finished envs were refilled
        assert A.RISK_INSUFF_MARGIN in seen and A.RISK_MARGIN_CALL in seen, seen
        assert n_done > 0


@pytest.mark.gpu
def test_one_wave_boundary(launched):
    """151,552 envs (exactly two waves at four blocks per SM) still take the one-wave kernel"""
    from madigan_b200.environments import Env
    env = Env("Composite", 1e6, {"data_source_config": CASES["pairs8"][1]}, n_envs=ONE_WAVE, window=4, seed=3)
    assert_launched(launched["boundary"], expected_kernel(True, ONE_WAVE, False), "boundary")


@pytest.mark.gpu
@pytest.mark.parametrize("knob", list(KNOB_ROWS))
def test_knob_rows(knob):
    """Oracle rows under MDG_BS64 (all four 64-thread kernels), MDG_NO_TMA (the row-copy ring with actions and
    weights) and MDG_NO_BULK (plain loads with actions and weights), each in a child process: the knobs are read
    once per process.  The probe runs inside the child and names the kernel the knob selects."""
    rows = KNOB_ROWS[knob]
    ids = [f"{os.path.abspath(__file__)}::test_plain_oracle[{row_id(r)}]" for r in rows]
    env = dict(os.environ, **{knob: "1", "MDG_PROBE_ROWS": repr([list(r) for r in rows])})
    r = subprocess.run([sys.executable, "-m", "pytest", *ids, "-q", "-m", "gpu", "-p", "no:cacheprovider"], env=env,
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert f"{len(rows)} passed" in r.stdout, r.stdout[-2000:]


# ---------------------------------------------------------------------------------------------------- GPU: TX2 knife edges
DELTAS = [0., 1e-16, -1e-16, 2.3e-16, -2.3e-16, 1e-14, -1e-14, 1e-13, -1e-13, 1e-12, -1e-12, 1e-10, -1e-10, 1e-8, -1e-8]
N_PROBE = 16 * len(DELTAS)  # 240 lanes: every asset position x every distance from the threshold


@pytest.mark.gpu
@pytest.mark.parametrize("case,N,gate", KNIFE_ROWS, ids=[row_id(r) for r in KNIFE_ROWS])
def test_knife_edge_multi_wave(case, N, gate, launched):
    """test_gpu_ledger_kat's knife edge on later assets, in the first and the last 240 envs of a multi-wave slab (the
    rest trade random orders): each probe order sits at the exact availableMargin its gate will see, after the same
    step's trades of the assets before it, +- 1e-16 ... 1e-8 relative.  This is where the TX2 gate's predicated
    `certain` / `r_fast` could disagree with exact_gate."""
    from madigan_b200.environments import Env
    from madigan_b200.environments.data_source import make_params
    from oracle.oracle import OracleBatch, OrcEnv, lib as olib
    import ctypes as C
    cfg = CASES["pairs8"][1] if case == "pairs8" else OU_MIX
    nA, reqM, init_cash = 16, .2, 1e6
    P, _ = make_params("Composite", cfg, required_margin=reqM, maintenance_margin=.25, transaction_cost_rel=.002,
                       transaction_cost_abs=.5, slippage_rel=.001, slippage_abs=.002)
    assert P.n_assets == nA
    env = Env("Composite", init_cash, {"data_source_config": cfg}, n_envs=N, window=4, seed=5)
    env.setRequiredMargin(reqM); env.setMaintenanceMargin(.25)
    env.setTransactionCost(.002, .5); env.setSlippage(.001, .002)
    env.flags = A.FLAG_FORCE_EXACT_GATE if gate == "exact" else 0
    orc = OracleBatch(N, P, None, window=4, seed=5, threads=ORACLE_THREADS)
    orc.reset(fill_ticks=1, clear_nstep=False)
    st = orc.state()
    for name in ("price", "gstate", "timestamp"):
        env.t[name].copy_(torch.from_numpy(st[name]))
    env.invalidate()
    lanes = np.r_[np.arange(N_PROBE), np.arange(N - N_PROBE, N)]
    local = np.r_[np.arange(N_PROBE), np.arange(N_PROBE)]
    rng = np.random.default_rng(17)
    L = olib()
    nU = max(P.n_uniforms, 1)
    assert_launched(launched[f"knife:{row_id((case, N, gate))}"], expected_kernel(case in PAIRS_CASES, N, False), "step")
    n_insuff = n_green = 0
    for t in range(8):
        st = orc.state()
        price, led = st["price"].T, st["ledger"].T  # (N, nA)
        units = rng.integers(-1, 2, size=(N, nA)) * (20_000. / price) * rng.uniform(.2, 1.5, size=(N, nA))
        for e_, l_ in zip(lanes, local):
            i, delta = l_ % nA, DELTAS[l_ // nA]
            scratch = OrcEnv()  # the oracle's portfolio after the trades of assets < i
            C.memmove(C.byref(scratch), L.orc_batch_env(orc.h, int(e_)), C.sizeof(OrcEnv))
            tp, tu, tc = C.c_double(), C.c_double(), C.c_double()
            for j in range(i):
                L.orc_broker_transaction(C.byref(scratch), j, float(units[e_, j]), C.byref(tp), C.byref(tu), C.byref(tc))
            am = L.orc_available_margin(C.byref(scratch))
            sign = 1. if led[e_, i] >= 0 else -1.  # same side as the position: not an offsetting order
            units[e_, i] = sign * (am / price[e_, i]) * (1. + delta)
        units = np.ascontiguousarray(units)
        z = rng.standard_normal((P.n_normals, N))
        u = np.zeros((nU, N))
        env.step(torch.from_numpy(units), normals=z, uniforms=u)
        orc.step(units, normals=z, uniforms=u)
        assert np.array_equal(cpu(env.t["risk"]), orc.risk), f"step {t}: riskInfo"
        assert np.array_equal(cpu(env.t["trans_units"]), orc.trans_units), f"step {t}: transactionUnits"
        s2 = orc.state()
        for name in ("ledger", "mean_entry", "borrowed", "cash", "price"):
            assert np.array_equal(cpu(env.t[name]), s2[name]), f"step {t}: {name}"
        assert np.array_equal(cpu(env.t["done"]), orc.done), f"step {t}: done"
        probe = orc.risk[local % nA, lanes]
        n_insuff += int((probe == A.RISK_INSUFF_MARGIN).sum())
        n_green += int((probe == A.RISK_GREEN).sum())
        if orc.done.any():
            zz = rng.standard_normal((1, P.n_normals, N))
            env.reset(mask=torch.from_numpy(orc.done.copy()), normals=zz, uniforms=np.zeros((1, nU, N)))
            orc.reset(mask=orc.done.copy(), fill_ticks=1, normals=zz, uniforms=np.zeros((1, nU, N)))
    assert n_insuff > 200 and n_green > 200, (n_insuff, n_green)  # both sides of the threshold were hit


# ---------------------------------------------------------------------------------------------------- GPU: free running
@pytest.mark.gpu
@pytest.mark.parametrize("case,N", FREE_ROWS, ids=[row_id(r) for r in FREE_ROWS])
def test_free_running_multi_wave(case, N, launched):
    """Philox normals drawn in the kernel, no injection: the multi-wave kernels against the oracle's Philox
    (test_free_running_philox_matches_oracle at multi-wave sizes).  Ledgers exact; prices 1e-9 (CUDA's and glibc's
    log/sincos in Box-Muller differ in the last ulp)."""
    env, orc, P = make_pair(case, N, WINDOW, None, MARGINS, COSTS, seed=1234, env_offset=1000)
    orc.threads = ORACLE_THREADS
    orc.reset(fill_ticks=1, clear_nstep=False)
    rng = np.random.default_rng(2)
    assert_launched(launched[f"free:{row_id((case, N))}"], expected_kernel(case in PAIRS_CASES, N, False), "step")
    for t in range(8):
        units = gen_units(rng, orc, N, P.n_assets, 20_000.)
        env.step(torch.from_numpy(units))
        orc.step(units)
        st = orc.state()
        close(cpu(env.t["price"]), st["price"], rtol=1e-9)
        assert np.array_equal(cpu(env.t["ledger"]), st["ledger"]), f"step {t}: ledger"
        assert np.array_equal(cpu(env.t["risk"]), orc.risk), f"step {t}: riskInfo"
        assert np.array_equal(cpu(env.t["done"]), orc.done), f"step {t}: done"


# ---------------------------------------------------------------------------------------------------- GPU: sets rows
@pytest.mark.gpu
@pytest.mark.parametrize("cfg,N,drive", SET_SHAPES, ids=[row_id(r) for r in SET_SHAPES])
def test_sets_rows(cfg, N, drive, launched):
    """Each of the 12 shapes of the sets kernels: a param_sets Env (S = 2, random assignment) and a broker_sets Env
    (S = 2), each bit for bit against plain Envs of its sets, 40 steps with auto-reset.  The probe names the sets, the
    broker-sets and the plain kernel of the same shape (the plain one is pinned to the oracle above)."""
    from test_broker_sets import BROKER, broker_env, check_derived, plain_env
    from test_param_sets import COMPOSITE, COMPOSITE_SETS, PAIR_SETS, check_sets, make_env
    sets = PAIR_SETS[:2] if cfg == "pairs8" else COMPOSITE_SETS[:2]
    base = PAIR_SETS[0] if cfg == "pairs8" else COMPOSITE
    pairs, acts = cfg == "pairs8", drive == "acts"
    g = torch.Generator(device="cuda").manual_seed(N)
    assign = torch.randint(0, 2, (N,), generator=g, device="cuda", dtype=torch.int32)
    multi = make_env(base, N, sets, assign, reward=DSR, window=WINDOW)
    plains = [make_env(c, N, reward=DSR, window=WINDOW) for c in sets]
    broker = broker_env(base, N, sets, BROKER[:2], assign, reward=DSR, window=WINDOW)
    bplains = [plain_env(c, N, b, reward=DSR, window=WINDOW) for c, b in zip(sets, BROKER[:2])]
    envs = [multi, broker] + plains + bplains
    for family in ("step_sets_kernel", "step_sets_broker_kernel", "step_kernel"):
        assert_launched(launched[f"sets:{row_id((cfg, N, drive))}:{family}"], expected_kernel(pairs, N, acts, family),
                        family)
    nA = multi.nA
    for t in range(40):
        if not acts:
            x = torch.randint(-1, 2, (N, nA), generator=g, device="cuda").double() * 40_000.
            step = lambda e: e.step(x, auto_reset=True)
        elif t % 2 == 0:
            x = torch.randint(0, 3, (N, nA), generator=g, device="cuda", dtype=torch.int8)
            step = lambda e: e.step_actions(x, action_atoms=3, unit_size=.05, auto_reset=True)
        else:
            x = torch.rand((N, nA + 1), generator=g, device="cuda", dtype=torch.float32)
            step = lambda e: e.step_weights(x, auto_reset=True)
        for e in envs:
            step(e)
        if t % 10 == 9:
            check_sets(multi, plains, f"sets step {t}")
            check_sets(broker, bplains, f"broker sets step {t}")
    check_derived(broker, bplains, "end")
    assert not torch.equal(plains[0].t["price"], plains[1].t["price"])  # two different markets


# ---------------------------------------------------------------------------------------------------- GPU: episode stats
STATS_SIZES = [1, 31, 33, 65_543, 1_048_589]  # the last is above the 592 x 256-thread grid: the grid-stride loop runs


def stats_env(N, nA, seed=4):
    from madigan_b200.environments import Env
    cfg = {f"pair{i}": {"data_source_type": "OUPair", "data_source_config": {"theta": .015, "phi": .01, "noise": .03}}
           for i in range(nA // 2)}
    env = Env("Composite", 1e6, {"data_source_config": cfg}, n_envs=N, window=4, seed=seed)
    env.setRequiredMargin(.1); env.setMaintenanceMargin(.25)
    env.setTransactionCost(.002, .5); env.setSlippage(.001, 0.)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(6):  # leveraged random orders; finished envs keep their state (no reset)
        u = torch.randint(-1, 2, (N, nA), generator=g, device="cuda").double()
        env.step(u * 80_000. * torch.rand((N, nA), generator=g, device="cuda", dtype=torch.float64))
    written = torch.rand(N, generator=g, device="cuda") < .1  # envs written flat, cash kept
    env.t["ledger"][:, written] = 0.
    env.t["borrowed"][:, written] = 0.
    env.t["done"] |= torch.rand(N, generator=g, device="cuda") < .05  # and some more finished ones
    return env


def stats_terms(env):
    """the terms of every slot of mdg_episode_stats, from the device tensors; equity folded left to right"""
    led, pr, bor = (cpu(env.t[n]) for n in ("ledger", "price", "borrowed"))
    av, bms = np.zeros(env.N), np.zeros(env.N)
    for j in range(env.nA):
        av = av + led[j] * pr[j]
        bms = bms + bor[j]
    eq = cpu(env.t["cash"]) + av - bms
    return dict(eq=eq, reward=cpu(env.t["reward"]), cost=cpu(env.t["trans_cost"]).ravel(),
                done=cpu(env.t["done"]), expo=np.abs(led * pr) / eq, held=led != 0.)


def assert_fsum(got, terms, tag):
    ref, mag = math.fsum(terms), math.fsum(np.abs(terms))
    assert abs(got - ref) <= 1e-12 * mag, f"{tag}: {got!r} against fsum {ref!r} (sum of |terms| {mag!r})"


def fmin_all(x):
    return float(np.fmin.reduce(np.r_[np.inf, x]))  # fmin skips NaN; no env: +inf


def fmax_all(x):
    return float(np.fmax.reduce(np.r_[-np.inf, x]))


@pytest.mark.gpu
@pytest.mark.parametrize("nA", [2, 16])
@pytest.mark.parametrize("N", STATS_SIZES)
def test_episode_stats_vs_fsum(N, nA):
    """stats_kernel against math.fsum of the same terms: counts, min and max exact; the sums within 1e-12 of the sum
    of their magnitudes (the atomics' order changes from run to run).  Also summarize_stats against numpy."""
    from madigan_b200.parallel import summarize_stats
    env = stats_env(N, nA)
    vec = cpu(env.episode_stats())
    ns = A.MDG_STATS_NSCALAR
    assert vec.shape == (ns + 2 * nA,)
    x = stats_terms(env)
    eq = x["eq"]
    assert np.isfinite(eq).all()
    assert vec[0] == N and vec[7] == int(x["done"].sum())
    assert vec[3] == fmin_all(eq) and vec[4] == fmax_all(eq)
    assert_fsum(vec[1], eq, "sum equity")
    assert_fsum(vec[2], eq * eq, "sum equity^2")
    assert_fsum(vec[5], x["reward"], "sum reward")
    assert_fsum(vec[6], x["cost"], "sum transaction cost")
    for j in range(nA):
        assert_fsum(vec[ns + j], x["expo"][j], f"exposure {j}")
        assert vec[ns + nA + j] == int(x["held"][j].sum()), f"held {j}"
    if N > 1000:  # the state is not trivial: positions, flat envs, finished envs, costs, negative rewards
        assert 0 < x["held"].sum() < N * nA and x["done"].any() and vec[6] > 0 and (x["reward"] < 0).any()
    s = summarize_stats(torch.from_numpy(vec), nA)
    assert s["n_envs"] == N and s["n_done"] == int(x["done"].sum())
    assert s["min_equity"] == eq.min() and s["max_equity"] == eq.max()
    assert abs(s["mean_equity"] - eq.mean()) <= 1e-12 * np.abs(eq).mean()
    assert abs(s["std_equity"] ** 2 - eq.var()) <= 1e-11 * (eq * eq).mean()
    assert abs(s["mean_reward"] - x["reward"].mean()) <= 1e-12 * np.abs(x["reward"]).mean() + 1e-300
    for j in range(nA):
        e_j = x["expo"][j]
        assert abs(s["mean_exposure"][j] - e_j.mean()) <= 1e-12 * np.abs(e_j).mean() + 1e-300, j
        assert s["frac_in_position"][j] == x["held"][j].sum() / N, j


@pytest.mark.gpu
def test_episode_stats_nan_equity():
    """An env with NaN cash: min and max skip it (fmin / fmax), the sums it enters are NaN, the counts are unchanged."""
    N, nA = 33, 2
    env = stats_env(N, nA, seed=9)
    env.t["cash"][5] = float("nan")
    vec = cpu(env.episode_stats())
    x = stats_terms(env)
    eq = x["eq"]
    assert np.isnan(eq[5]) and np.isfinite(np.delete(eq, 5)).all()
    assert vec[0] == N and vec[7] == int(x["done"].sum())
    assert vec[3] == fmin_all(eq) and vec[4] == fmax_all(eq)
    assert np.isnan(vec[1]) and np.isnan(vec[2])
    ns = A.MDG_STATS_NSCALAR
    for j in range(nA):
        assert np.isnan(vec[ns + j]) and vec[ns + nA + j] == int(x["held"][j].sum())
    assert_fsum(vec[5], x["reward"], "sum reward")
