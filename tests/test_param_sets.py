"""Generator parameter sets: one Env whose envs tick different markets.

The contract: env e of an Env with parameter sets is, bit for bit, env e of a plain Env built from its set's config
with the same n_envs, seed and env_offset (Philox keys every draw on seed, global env id and tick only).  The GPU
tests drive a multi-set Env next to one plain Env per set and compare the envs of each set with that set's plain Env
on every state, output and observation tensor.  The CPU tests cover the table builder and the launchers' argument
checks."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from madigan_b200.environments.data_source import PARAM_SLOTS, make_param_table, make_params, make_reward


def pairs_cfg(theta, phi, noise, n=8):
    """n OU pairs; theta / phi / noise: a number or one value per pair"""
    pick = lambda v, i: v[i] if isinstance(v, (list, tuple)) else v
    return {f"pair{i}": {"data_source_type": "OUPair", "data_source_config": {
        "theta": pick(theta, i), "phi": pick(phi, i), "noise": pick(noise, i)}} for i in range(n)}


PAIR_SETS = [pairs_cfg(.015, .01, .03),                      # the default OUPair set
             pairs_cfg(.03, .012, .02),
             pairs_cfg(.008, .02, .045),
             pairs_cfg([.01 + .003 * i for i in range(8)], [.006 + .002 * i for i in range(8)],
                       [.05 - .004 * i for i in range(8)])]

COMPOSITE = {  # bench.py's C4 composite: every generator type that parameter sets support except Sawtooth/Triangle/Gaussian
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


def vary(cfg, f, s):
    """Another market with the same assets: every parameter of every source moved (periods by whole ticks, phases by
    an offset, everything else by the factor f)."""
    out = {}
    for label, sub in cfg.items():
        c = {}
        for key, v in sub["data_source_config"].items():
            vec = v if isinstance(v, list) else [v]
            if key in ("min_period", "max_period"):
                new = [x + (s if key == "min_period" else 3 * s) for x in vec]
            elif key == "phase":
                new = [x + .37 * s for x in vec]
            else:
                new = [x * f for x in vec]
            c[key] = new if isinstance(v, list) else new[0]
        out[label] = {"data_source_type": sub["data_source_type"], "data_source_config": c}
    return out


COMPOSITE_SETS = [COMPOSITE, vary(COMPOSITE, 1.3, 1), vary(COMPOSITE, .7, 2)]

DSR = dict(reward_shaper_config={"reward_shaper": "DSR", "adaptation_rate": .001}, nstep_return=1, reduce_rewards=True)
PPC = dict(reward_shaper_config={"reward_shaper": "cosine_port_shaper", "desired_portfolio": [1.] + [0.] * 16,
                                 "cosine_temp": .025}, nstep_return=5, reduce_rewards=False)

STATE = ("price", "ledger", "mean_entry", "borrowed", "cash", "gstate", "timestamp", "folds", "reset_ts",
         "reward", "done", "trans_price", "trans_units", "trans_cost", "risk", "margin_call",
         "agent_reward", "shaped_reward", "n_popped", "shaper_A", "shaper_B", "pre_price")
RINGS = ("obs_price", "obs_port")
ENV_MAJOR = ("pre_price",)  # [N][k][nA]; every other tensor has the env index last


# ---------------------------------------------------------------------------------------------------- CPU
def test_param_table_layout_and_slots():
    sets = [PAIR_SETS[0], PAIR_SETS[3]]
    tab = make_param_table("Composite", PAIR_SETS[0], sets)
    assert tab.shape == (16, A.MDG_GEN_NPARAM, 2) and tab.dtype == np.float64
    th, ph, nz = (PARAM_SLOTS["OUPair"].index(k) for k in ("theta", "phi", "noise"))
    for i in range(8):
        for q in range(2):  # both assets of a pair carry the pair's values
            assert tab[2 * i + q, th, 1] == .01 + .003 * i and tab[2 * i + q, ph, 1] == .006 + .002 * i
            assert tab[2 * i + q, nz, 1] == .05 - .004 * i and tab[2 * i + q, th, 0] == .015
    # every slot of every type comes out where PARAM_SLOTS says, and the composite sets vary every one of them
    tab = make_param_table("Composite", COMPOSITE, COMPOSITE_SETS)
    from madigan_b200.environments.data_source import build_generator_table
    names, recs, *_ = build_generator_table("Composite", COMPOSITE)
    gen_name = {A.GEN_SYNTH: "Synth", A.GEN_OU: "OU", A.GEN_OUPAIR: "OUPair", A.GEN_SIMPLETREND: "SimpleTrend",
                A.GEN_TRENDOU: "TrendOU", A.GEN_TRENDYOU: "TrendyOU"}
    label_of = {"Synth": "sines", "OU": "ou", "OUPair": "pair", "SimpleTrend": "trend", "TrendOU": "trendou",
                "TrendyOU": "trendyou"}
    seen = {}
    for i, r in enumerate(recs):
        ty = gen_name[r["type"]]
        k = seen.get(ty, 0)
        seen[ty] = k + 1 if ty != "OUPair" else 0
        for j, key in enumerate(PARAM_SLOTS[ty]):
            for s, cfg in enumerate(COMPOSITE_SETS):
                v = cfg[label_of[ty]]["data_source_config"][key]
                assert tab[i, j, s] == float(v[k] if isinstance(v, list) else v), (names[i], key, s)
            assert len(set(tab[i, j, :].tolist())) == len(COMPOSITE_SETS), (names[i], key)


def test_param_table_rejects_other_structures():
    with pytest.raises(ValueError, match="asset 14"):  # one asset pair fewer
        make_param_table("Composite", PAIR_SETS[0], [PAIR_SETS[0], pairs_cfg(.01, .01, .01, n=7)])
    other = dict(PAIR_SETS[0])
    other["pair3"] = {"data_source_type": "OU", "data_source_config": {"mean": [1., 2.], "theta": [.1, .1],
                                                                       "phi": [.1, .1]}}
    with pytest.raises(ValueError, match="asset 6"):
        make_param_table("Composite", PAIR_SETS[0], [other])
    reordered = {k: COMPOSITE[k] for k in ("ou", "sines", "pair", "trend", "trendou", "trendyou")}
    with pytest.raises(ValueError, match="asset 0"):
        make_param_table("Composite", COMPOSITE, [reordered])
    for kind in ("SineAdder", "SineDynamic", "SineDynamicTrend"):
        with pytest.raises(ValueError, match="SINE"):
            make_param_table(kind, None, [None])
    with pytest.raises(ValueError):
        make_param_table("OU", None, [])


def test_sets_launchers_validate_without_gpu():
    """The _sets entry points check their arguments before touching CUDA."""
    from madigan_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from madigan_b200.build import build
        build()
    lib = _lib.lib()
    P, _ = make_params("OU")
    L = A.MdgLaunch(n_envs=4, window=8, head=0)
    S, IO = A.MdgState(), A.MdgStepIO()
    S.folds = S.reset_ts = IO.pre_price = 1  # non-null dummies: never dereferenced, validation fails first
    ok = A.MdgParamSets(p=1, set_of_env=1, n_sets=2)
    bad = [None, C.byref(A.MdgParamSets(p=1, set_of_env=1, n_sets=0)), C.byref(A.MdgParamSets(p=None, set_of_env=1,
                                                                                              n_sets=1))]
    for ps in bad:
        assert lib.mdg_step_sets(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), ps) == A.MDG_E_INVALID
        assert lib.mdg_step_autoreset_sets(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), 8, 1, 1, 1 << 20,
                                           ps) == A.MDG_E_INVALID
        assert lib.mdg_reset_ws_sets(C.byref(P), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, 1, 1 << 20,
                                     ps) == A.MDG_E_INVALID
        assert lib.mdg_init_state_sets(C.byref(P), None, C.byref(S), C.byref(L), ps) == A.MDG_E_INVALID
    # a workspace is required: no fall-back to mdg_reset
    assert lib.mdg_reset_ws_sets(C.byref(P), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, None, 0,
                                 C.byref(ok)) == A.MDG_E_INVALID
    for kind in ("SineAdder", "SineDynamic"):
        Ps, _ = make_params(kind)
        Ps.gen_ext, Ps.n_gen_ext = 1, 1 << 20
        assert lib.mdg_step_sets(C.byref(Ps), None, C.byref(S), C.byref(IO), C.byref(L), C.byref(ok)) == \
            A.MDG_E_UNSUPPORTED
        assert lib.mdg_init_state_sets(C.byref(Ps), None, C.byref(S), C.byref(L), C.byref(ok)) == A.MDG_E_UNSUPPORTED
        assert lib.mdg_reset_ws_sets(C.byref(Ps), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, 1, 1 << 20,
                                     C.byref(ok)) == A.MDG_E_UNSUPPORTED
    assert lib.mdg_sizeof(14) == C.sizeof(A.MdgParamSets) == 24


# ---------------------------------------------------------------------------------------------------- GPU helpers
def make_env(cfg, N, sets=None, assign=None, seed=11, env_offset=0, reward=None, window=64, flags=0,
             margins=(.1, .25), costs=(.02, .001)):
    from madigan_b200.environments import Env
    e = Env("Composite", 1e6, {"data_source_config": cfg}, n_envs=N, window=window, seed=seed, env_offset=env_offset,
            reward=reward, param_sets=sets, param_set=assign)
    e.setRequiredMargin(margins[0])
    e.setMaintenanceMargin(margins[1])
    e.setTransactionCost(costs[0], 0.)
    e.setSlippage(costs[1], 0.)
    e.flags = flags
    return e


def same(a, b):
    if a.dtype == torch.float64:
        return torch.equal(a.view(torch.int64), b.view(torch.int64))
    return torch.equal(a, b)


def pick(x, name, idx):
    return x[idx] if name in ENV_MAJOR else x[..., idx]


def check_sets(multi, plains, tag, names=STATE + RINGS, windows=True):
    """the envs of set s in `multi` against plain Env s, on every listed tensor and the standard_normal window"""
    assign = multi.param_set.long()
    wm = multi.window("standard_normal") if windows else None
    pm = multi.portfolio_window() if windows else None
    for s, pl in enumerate(plains):
        idx = (assign == s).nonzero().squeeze(1)
        if idx.numel() == 0:
            continue
        for name in names:
            assert same(pick(multi.t[name], name, idx), pick(pl.t[name], name, idx)), (tag, s, name)
        if windows:
            assert same(wm[idx], pl.window("standard_normal")[idx]), (tag, s, "window")
            assert same(pm[idx], pl.portfolio_window()[idx]), (tag, s, "portfolio window")


def step_all(envs, kind, g, N, nA=16):
    if kind == "actions":
        a = torch.randint(0, 3, (N, nA), generator=g, device="cuda", dtype=torch.int8)
        for e in envs:
            e.step_actions(a, action_atoms=3, unit_size=.05, auto_reset=True)
    elif kind == "weights":
        w = torch.rand((N, nA + 1), generator=g, device="cuda", dtype=torch.float32)
        for e in envs:
            e.step_weights(w, auto_reset=True)
    else:
        u = torch.randint(-1, 2, (N, nA), generator=g, device="cuda").double() * 40_000.
        for e in envs:
            e.step(u, auto_reset=True)


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["units", "actions", "weights", "generic_fill", "multi_wave"])
def test_all_pairs_equivalence(kind):
    """8 OU pairs, four sets (the default one among them) at random: with DSR and auto-reset for 300 steps, the envs
    of each set equal a plain Env of that set.  generic_fill: the generic refill kernel; multi_wave: 155,648 envs
    (the multi-wave step instantiation)."""
    N = 155_648 if kind == "multi_wave" else 65_536
    flags = A.FLAG_GENERIC_FILL if kind == "generic_fill" else 0
    g = torch.Generator(device="cuda").manual_seed(5)
    assign = torch.randint(0, len(PAIR_SETS), (N,), generator=g, device="cuda", dtype=torch.int32)
    multi = make_env(PAIR_SETS[0], N, PAIR_SETS, assign, reward=DSR, flags=flags)
    plains = [make_env(c, N, reward=DSR, flags=flags) for c in PAIR_SETS]
    assert multi.n_param_sets == 4 and torch.equal(multi.param_set, assign)
    check_sets(multi, plains, "constructor")
    envs = [multi] + plains
    n_done = 0
    step_kind = kind if kind in ("actions", "weights") else "units"
    for t in range(300):
        step_all(envs, step_kind, g, N)
        n_done += int(multi.t["done"].sum())
        if t % 10 == 9:
            check_sets(multi, plains, f"step {t}")
    if step_kind == "units":
        assert n_done > 1000
    # the sets are different markets: the same env of two plain Envs has different prices
    assert not torch.equal(plains[0].t["price"], plains[1].t["price"])


@pytest.mark.gpu
@pytest.mark.parametrize("knob", ["MDG_NO_TMA", "MDG_NO_BULK", "MDG_BS64"])
def test_all_pairs_equivalence_operand_paths(knob):
    """The step kernel's other operand paths (row copies, plain loads; MDG_BS64: the plain Envs take the 64-thread
    instantiation, the sets launch keeps 128 threads), in child processes: the knobs are read once per process."""
    import subprocess
    import sys
    env = dict(os.environ, **{knob: "1"})
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        "test_all_pairs_equivalence and units"], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


@pytest.mark.gpu
def test_generic_path_equivalence():
    """C4 composite (Synth, OU, OUPair, SimpleTrend, TrendOU, TrendyOU), sets that move every slot including the start
    values: hold, multi-asset and single-asset steps, explicit masked resets with history fill."""
    N = 4096
    g = torch.Generator(device="cuda").manual_seed(9)
    assign = torch.randint(0, len(COMPOSITE_SETS), (N,), generator=g, device="cuda", dtype=torch.int32)
    kw = dict(reward=PPC, window=16, margins=(.1, .25), costs=(.001, 0.))
    multi = make_env(COMPOSITE, N, COMPOSITE_SETS, assign, **kw)
    plains = [make_env(c, N, **kw) for c in COMPOSITE_SETS]
    envs = [multi] + plains
    check_sets(multi, plains, "constructor")
    for t in range(90):
        if t % 3 == 0:
            for e in envs:
                e.step()
        elif t % 3 == 1:
            u = torch.randint(-1, 2, (N, 16), generator=g, device="cuda").double() * 5000.
            for e in envs:
                e.step(u, auto_reset=t % 2 == 0)
        else:
            u = torch.randint(-1, 2, (N,), generator=g, device="cuda").double() * 5000.
            for e in envs:
                e.step(t % 16, u)
        if t % 15 == 14:
            mask = torch.rand(N, generator=g, device="cuda") < .3
            for e in envs:
                e.reset(mask, fill_history=True)
        check_sets(multi, plains, f"step {t}")
    # start values differ per set (OU mean, Synth phase, trend start): the constructor prices differ
    fresh = [make_env(c, 8, window=4) for c in COMPOSITE_SETS]
    assert not torch.equal(fresh[0].t["price"], fresh[1].t["price"])


@pytest.mark.gpu
def test_one_set_per_env():
    """S = N with random parameters and the identity assignment: env e equals a one-env plain Env with env_offset e."""
    N = 24
    rng = np.random.default_rng(4)
    sets = [pairs_cfg(list(rng.uniform(.005, .05, 8)), list(rng.uniform(.005, .02, 8)), list(rng.uniform(.01, .05, 8)))
            for _ in range(N)]
    multi = make_env(sets[0], N, sets, torch.arange(N, dtype=torch.int32), window=16)
    plains = [make_env(sets[e], 1, env_offset=e, window=16) for e in range(N)]
    g = torch.Generator(device="cuda").manual_seed(2)
    n_done = 0
    for t in range(120):
        u = torch.randint(-1, 2, (N, 16), generator=g, device="cuda").double() * 40_000.
        multi.step(u, auto_reset=True)
        for e in range(N):
            plains[e].step(u[e:e + 1].contiguous(), auto_reset=True)
        n_done += int(multi.t["done"].sum())
        if t % 10 == 9 or t == 119:
            wm = multi.window("standard_normal")
            for e in range(N):
                for name in STATE + RINGS:
                    a = multi.t[name][e:e + 1] if name in ENV_MAJOR else multi.t[name][..., e:e + 1]
                    assert same(a, plains[e].t[name]), (t, e, name)
                assert same(wm[e:e + 1], plains[e].window("standard_normal")), (t, e)
    assert n_done > 0


@pytest.mark.gpu
def test_reassignment_then_reset():
    """assign_param_sets(mask) + reset(mask, fill_history=True) after hold steps: from then on those envs equal a plain
    Env of their new set that reset the same envs at the same step."""
    N = 4096
    g = torch.Generator(device="cuda").manual_seed(6)
    old = torch.randint(0, 4, (N,), generator=g, device="cuda", dtype=torch.int32)
    multi = make_env(PAIR_SETS[0], N, PAIR_SETS, old, window=16)
    plains = [make_env(c, N, window=16) for c in PAIR_SETS]
    envs = [multi] + plains
    for _ in range(5):
        for e in envs:
            e.step()
    new = torch.randint(0, 4, (N,), generator=g, device="cuda", dtype=torch.int32)
    mask = torch.rand(N, generator=g, device="cuda") < .5
    multi.assign_param_sets(new, mask=mask)
    assert torch.equal(multi.param_set, torch.where(mask, new, old))
    for e in envs:
        e.reset(mask, fill_history=True)
    # the rings' rows older than a reset are not part of the window: compare the windows instead of the raw rings
    check_sets(multi, plains, "reset", names=STATE)
    n_done = 0
    for t in range(100):
        step_all(envs, "units", g, N)
        n_done += int(multi.t["done"].sum())
        if t % 10 == 9:
            check_sets(multi, plains, f"step {t}", names=STATE)
    assert n_done > 0


@pytest.mark.gpu
def test_oracle_with_injected_noise():
    """Generic path, injected noise: the envs of set s against oracle/mdg_oracle.c built from set s's MdgParams.
    Ledgers, transaction units and risk codes bit-exact; prices, rewards and windows at test_gpu_parity's 1e-9."""
    from oracle.oracle import OracleBatch
    N, k = 384, 8
    margins, costs = (1., .25), (.02, .001)
    rng = np.random.default_rng(3)
    assign = torch.from_numpy(rng.integers(0, 3, N).astype(np.int32))
    multi = make_env(COMPOSITE, N, COMPOSITE_SETS, assign, reward=DSR, window=k, seed=7, margins=margins, costs=costs)
    R = make_reward(DSR["reward_shaper_config"], 1, .99, True, n_assets=16)
    Ps = [make_params("Composite", c, required_margin=margins[0], maintenance_margin=margins[1],
                      transaction_cost_rel=costs[0], slippage_rel=costs[1])[0] for c in COMPOSITE_SETS]
    orcs = [OracleBatch(N, P, R, window=k, seed=7) for P in Ps]
    a = assign.numpy()
    idx = [np.nonzero(a == s)[0] for s in range(3)]

    def merged(get):
        out = np.array(get(orcs[0]), copy=True)
        for s in (1, 2):
            out[..., idx[s]] = get(orcs[s])[..., idx[s]]
        return out

    for o in orcs:
        o.reset(fill_ticks=1, clear_nstep=False)
    for name in ("price", "gstate", "timestamp"):  # start from the oracles' constructor state (libm sin of Synth)
        multi.t[name].copy_(torch.from_numpy(merged(lambda o: o.state()[name])))
    multi.invalidate()
    P = Ps[0]
    nz, uz = rng.standard_normal((k, P.n_normals, N)), rng.random((k, P.n_uniforms, N))
    multi.reset(fill_history=True, normals=nz, uniforms=uz)
    for o in orcs:
        o.reset(fill_ticks=k, normals=nz, uniforms=uz)
    cpu = lambda x: x.detach().cpu().numpy()
    n_done = 0
    for t in range(24):
        units = rng.integers(-1, 2, size=(N, 16)) * 9000.
        nz, uz = rng.standard_normal((P.n_normals, N)), rng.random((P.n_uniforms, N))
        multi.step(torch.from_numpy(units), normals=nz, uniforms=uz)
        for o in orcs:
            o.step(units, normals=nz, uniforms=uz)
        T = multi.t
        assert np.array_equal(cpu(T["ledger"]), merged(lambda o: o.state()["ledger"])), t
        assert np.array_equal(cpu(T["trans_units"]), merged(lambda o: o.trans_units)), t
        assert np.array_equal(cpu(T["risk"]), merged(lambda o: o.risk)), t
        done = merged(lambda o: o.done)
        assert np.array_equal(cpu(T["done"]), done), t
        np.testing.assert_allclose(cpu(T["price"]), merged(lambda o: o.state()["price"]), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(cpu(T["reward"]), merged(lambda o: o.reward), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(cpu(T["shaped_reward"]), merged(lambda o: o.shaped_reward), rtol=1e-9, atol=1e-11)
        nv = orcs[0].n_valid
        w = cpu(multi.window(None, n_valid=nv))
        ref = np.array(orcs[0].window(nv), copy=True)
        for s in (1, 2):
            ref[idx[s]] = orcs[s].window(nv)[idx[s]]
        np.testing.assert_allclose(w, ref, rtol=1e-9, atol=1e-12)
        if done.any():
            n_done += int(done.sum())
            nz, uz = rng.standard_normal((k, P.n_normals, N)), rng.random((k, P.n_uniforms, N))
            multi.reset(mask=torch.from_numpy(done.copy()), fill_history=True, normals=nz, uniforms=uz)
            for o in orcs:
                o.reset(mask=done.copy(), fill_ticks=k, normals=nz, uniforms=uz)
    assert n_done > 0


@pytest.mark.gpu
def test_sharding_with_sets():
    """A multi-set Env over 256 envs equals two 128-env halves with env_offset and the halves of the assignment."""
    g = torch.Generator(device="cuda").manual_seed(8)
    assign = torch.randint(0, 4, (256,), generator=g, device="cuda", dtype=torch.int32)
    big = make_env(PAIR_SETS[0], 256, PAIR_SETS, assign, seed=99, window=8)
    lo = make_env(PAIR_SETS[0], 128, PAIR_SETS, assign[:128], seed=99, window=8)
    hi = make_env(PAIR_SETS[0], 128, PAIR_SETS, assign[128:], seed=99, env_offset=128, window=8)
    for t in range(40):
        u = torch.randint(-1, 2, (256, 16), generator=g, device="cuda").double() * 40_000.
        big.step(u, auto_reset=True)
        lo.step(u[:128].contiguous(), auto_reset=True)
        hi.step(u[128:].contiguous(), auto_reset=True)
    for name in ("price", "ledger", "cash", "gstate", "timestamp", "obs_price"):
        assert same(big.t[name], torch.cat([lo.t[name], hi.t[name]], dim=-1)), name


@pytest.mark.gpu
def test_param_table_view_and_clamp():
    """param_table is the (S, nA, NPARAM) view the kernels read: an in-place write takes effect at the next launch.
    An index outside [0, S) written past the setter reads set S-1 (the kernels clamp it)."""
    N = 1024
    g = torch.Generator(device="cuda").manual_seed(1)
    multi = make_env(PAIR_SETS[0], N, 4, torch.full((N,), 3, dtype=torch.int32), window=8)
    ref = torch.from_numpy(make_param_table("Composite", PAIR_SETS[0], [PAIR_SETS[0]] * 4)).permute(2, 0, 1)
    assert multi.param_table.shape == (4, 16, A.MDG_GEN_NPARAM) and torch.equal(multi.param_table.cpu(), ref)
    # set 3 becomes PAIR_SETS[2]'s market, in place; the envs then follow a plain Env of that config
    multi.param_table[3] = torch.from_numpy(make_param_table("Composite", PAIR_SETS[2], [PAIR_SETS[2]])[:, :, 0])
    plain = make_env(PAIR_SETS[2], N, window=8)
    # one constructor tick ran under the base values: restart both from the same state
    for e in (multi, plain):
        e.reset(fill_history=True)
    bad = torch.randint(-5, 1000, (N,), generator=g, device="cuda", dtype=torch.int32)
    bad[bad.clamp(0, 3) == bad] = 3
    multi.param_set.copy_(bad)  # past the setter: out-of-range values clamp to set 3
    for t in range(30):
        u = torch.randint(-1, 2, (N, 16), generator=g, device="cuda").double() * 40_000.
        multi.step(u, auto_reset=True)
        plain.step(u, auto_reset=True)
    for name in STATE:
        assert same(multi.t[name], plain.t[name]), name


@pytest.mark.gpu
def test_checkpoint_round_trip():
    N = 2048
    g = torch.Generator(device="cuda").manual_seed(12)
    assign = torch.randint(0, 4, (N,), generator=g, device="cuda", dtype=torch.int32)
    a = make_env(PAIR_SETS[0], N, PAIR_SETS, assign, reward=DSR, window=16)
    for _ in range(10):
        step_all([a], "units", g, N)
    sd = a.state_dict()
    us = [torch.randint(-1, 2, (N, 16), generator=g, device="cuda").double() * 40_000. for _ in range(20)]
    for u in us:
        a.step(u, auto_reset=True)
    b = make_env(PAIR_SETS[0], N, 4, None, reward=DSR, window=16)  # other table, other assignment
    b.load_state_dict(sd)
    assert torch.equal(b.param_set, assign) and torch.equal(b.param_table, a.param_table)
    for u in us:
        b.step(u, auto_reset=True)
    for name in STATE + RINGS:
        assert same(a.t[name], b.t[name]), name
    with pytest.raises(ValueError, match="parameter sets"):
        make_env(PAIR_SETS[0], N, reward=DSR, window=16).load_state_dict(sd)
    with pytest.raises(ValueError, match="parameter sets"):
        make_env(PAIR_SETS[0], N, 3, reward=DSR, window=16).load_state_dict(sd)
    with pytest.raises(ValueError, match="parameter sets"):
        b.load_state_dict(make_env(PAIR_SETS[0], N, reward=DSR, window=16).state_dict())


@pytest.mark.gpu
def test_assign_param_sets_validation():
    from madigan_b200.environments import Env
    N = 256
    e = make_env(PAIR_SETS[0], N, 4, window=8)
    assert torch.equal(e.param_set.cpu(), (torch.arange(N) % 4).int())
    for ids in (torch.full((N,), 4), torch.full((N,), -1), torch.arange(N)):
        with pytest.raises(ValueError, match="in \\[0, 4\\)"):
            e.assign_param_sets(ids)
    with pytest.raises(ValueError, match="shape"):
        e.assign_param_sets(torch.zeros(N + 1, dtype=torch.int64))
    with pytest.raises(ValueError, match="integers"):
        e.assign_param_sets(torch.zeros(N))
    with pytest.raises(ValueError, match="shape"):
        e.assign_param_sets(torch.zeros(N, dtype=torch.int64), mask=torch.ones(3, dtype=torch.bool))
    assert torch.equal(e.param_set.cpu(), (torch.arange(N) % 4).int())  # nothing written by a rejected call
    e.assign_param_sets(2)
    assert torch.equal(e.param_set.cpu(), torch.full((N,), 2, dtype=torch.int32))
    with pytest.raises(ValueError):
        make_env(PAIR_SETS[0], N, 4, torch.full((N,), 7), window=8)
    with pytest.raises(ValueError, match="SINE"):
        Env("SineAdder", 1e6, None, n_envs=8, window=4, param_sets=2)
    with pytest.raises(RuntimeError):
        make_env(PAIR_SETS[0], N, window=8).assign_param_sets(0)
    assert make_env(PAIR_SETS[0], N, window=8).n_param_sets == 0
