"""Broker sets: the seven broker settings (starting cash, margins, slippage, costs) per parameter set.

The contract: env e of an Env with broker sets is, bit for bit, env e of a plain Env built from its set's generator
config with setRequiredMargin / setMaintenanceMargin / setSlippage / setTransactionCost and initCash at its broker
set's values, with the same n_envs, seed and env_offset.  The GPU tests drive a multi-set Env next to one plain Env per
set and compare the envs of each set with that set's plain Env on every state, output and observation tensor.  The CPU
tests cover the table builder and the launchers' argument checks."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from madigan_b200.environments.data_source import BROKER_SLOTS, make_broker_table, make_params
from test_param_sets import COMPOSITE, COMPOSITE_SETS, DSR, PAIR_SETS, PPC, RINGS, STATE, check_sets, same

# Four broker sets that differ in every field.  Set 1 has required_margin = 0 (the fast gate never decides: every gated
# order goes to the exact gate, and availableMargin is infinite); set 2 a small starting cash and a large fixed cost, so
# that episodes end through equity < 0.1 * init_cash; set 3 a required margin of 1 (no borrowing).
BROKER = [
    dict(init_cash=1e6, required_margin=.1, maintenance_margin=.25, slippage_rel=.001, slippage_abs=0.,
         transaction_cost_rel=.02, transaction_cost_abs=0.),
    dict(init_cash=2.5e6, required_margin=0., maintenance_margin=.1, slippage_rel=.003, slippage_abs=.01,
         transaction_cost_rel=.005, transaction_cost_abs=2.),
    dict(init_cash=3e5, required_margin=.5, maintenance_margin=.4, slippage_rel=0., slippage_abs=.002,
         transaction_cost_rel=.01, transaction_cost_abs=1500.),
    dict(init_cash=1.5e6, required_margin=1., maintenance_margin=.05, slippage_rel=.0005, slippage_abs=.005,
         transaction_cost_rel=0., transaction_cost_abs=1.),
]


# ---------------------------------------------------------------------------------------------------- CPU
def test_broker_table_layout_and_defaults():
    base = dict(zip(BROKER_SLOTS, [1e6, .1, .25, .001, .002, .02, .5]))
    tab = make_broker_table(base, BROKER + [{}, {"required_margin": .7, "transaction_cost_abs": float("nan")}])
    assert tab.shape == (A.MDG_BROKER_NPARAM, 6) and tab.dtype == np.float64
    for s, d in enumerate(BROKER):
        assert tab[:, s].tolist() == [d[k] for k in BROKER_SLOTS]
    assert tab[:, 4].tolist() == [base[k] for k in BROKER_SLOTS]  # an empty set: every value from the base
    assert tab[1, 5] == .7 and np.isnan(tab[6, 5])                  # NaN is a value like any other
    assert tab[[0, 2, 3, 4, 5], 5].tolist() == [base[k] for k in ("init_cash", "maintenance_margin", "slippage_rel",
                                                                     "slippage_abs", "transaction_cost_rel")]
    assert BROKER_SLOTS == ("init_cash", "required_margin", "maintenance_margin", "slippage_rel", "slippage_abs",
                            "transaction_cost_rel", "transaction_cost_abs")
    assert A.MDG_BROKER_NPARAM == len(BROKER_SLOTS)
    # out-of-range values are taken as they are (the setters do not check them either)
    assert make_broker_table(base, [{"required_margin": -3., "init_cash": 0}])[:2, 0].tolist() == [0., -3.]


def test_broker_table_rejects_bad_input():
    base = dict(zip(BROKER_SLOTS, [1e6, .1, .25, 0., 0., 0., 0.]))
    with pytest.raises(ValueError, match="unknown broker setting 'tcost_rel'"):
        make_broker_table(base, [{"tcost_rel": .1}])
    with pytest.raises(ValueError, match="required_margin must be a number"):
        make_broker_table(base, [{}, {"required_margin": "0.1"}])
    for bad in (None, True, [0.1], np.bool_(True)):
        with pytest.raises(ValueError, match="must be a number"):
            make_broker_table(base, [{"slippage_abs": bad}])
    with pytest.raises(ValueError, match="at least one set"):
        make_broker_table(base, [])
    with pytest.raises(ValueError, match="missing"):
        make_broker_table({"init_cash": 1e6}, [{}])


def _lib():
    from madigan_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from madigan_b200.build import build
        build()
    return _lib.lib()


def test_abi_version_and_sizes():
    lib = _lib()
    assert lib.mdg_abi_version() == A.MDG_ABI_VERSION == 16
    for i, st in enumerate(A.STRUCTS):
        assert lib.mdg_sizeof(i) == C.sizeof(st), st.__name__
    assert lib.mdg_sizeof(14) == 24


def test_broker_launchers_validate_without_gpu():
    """The _sets_broker entry points check their arguments before touching CUDA."""
    lib = _lib()
    P, _ = make_params("OU")
    L = A.MdgLaunch(n_envs=4, window=8, head=0)
    S, IO, D = A.MdgState(), A.MdgStepIO(), A.MdgDerived()
    S.folds = S.reset_ts = IO.pre_price = 1  # non-null dummies: never dereferenced, validation fails first
    ok = A.MdgParamSets(p=1, set_of_env=1, n_sets=2)
    broker = 1  # a non-null table: the checks must not depend on it
    bad = [None, C.byref(A.MdgParamSets(p=1, set_of_env=1, n_sets=0)), C.byref(A.MdgParamSets(p=1, set_of_env=None,
                                                                                              n_sets=1))]
    for ps in bad:
        assert lib.mdg_step_sets_broker(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), ps, broker) == \
            A.MDG_E_INVALID
        assert lib.mdg_step_autoreset_sets_broker(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), 8, 1, 1,
                                                  1 << 20, ps, broker) == A.MDG_E_INVALID
        assert lib.mdg_reset_ws_sets_broker(C.byref(P), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, 1, 1 << 20,
                                            ps, broker) == A.MDG_E_INVALID
        assert lib.mdg_init_state_sets_broker(C.byref(P), None, C.byref(S), C.byref(L), ps, broker) == A.MDG_E_INVALID
        assert lib.mdg_derived_sets_broker(C.byref(P), C.byref(S), C.byref(D), C.byref(L), ps, broker) == \
            A.MDG_E_INVALID
    # a workspace is required
    assert lib.mdg_reset_ws_sets_broker(C.byref(P), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, None, 0,
                                        C.byref(ok), broker) == A.MDG_E_INVALID
    assert lib.mdg_step_autoreset_sets_broker(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), 8, 1, None, 0,
                                              C.byref(ok), broker) == A.MDG_E_INVALID
    for kind in ("SineAdder", "SineDynamic"):
        Ps, _ = make_params(kind)
        Ps.gen_ext, Ps.n_gen_ext = 1, 1 << 20
        for b in (broker, None):
            assert lib.mdg_step_sets_broker(C.byref(Ps), None, C.byref(S), C.byref(IO), C.byref(L), C.byref(ok),
                                            b) == A.MDG_E_UNSUPPORTED
            assert lib.mdg_step_autoreset_sets_broker(C.byref(Ps), None, C.byref(S), C.byref(IO), C.byref(L), 8, 1, 1,
                                                      1 << 20, C.byref(ok), b) == A.MDG_E_UNSUPPORTED
            assert lib.mdg_init_state_sets_broker(C.byref(Ps), None, C.byref(S), C.byref(L), C.byref(ok), b) == \
                A.MDG_E_UNSUPPORTED
            assert lib.mdg_reset_ws_sets_broker(C.byref(Ps), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, 1,
                                                1 << 20, C.byref(ok), b) == A.MDG_E_UNSUPPORTED
            assert lib.mdg_derived_sets_broker(C.byref(Ps), C.byref(S), C.byref(D), C.byref(L), C.byref(ok), b) == \
                A.MDG_E_UNSUPPORTED


# ---------------------------------------------------------------------------------------------------- GPU helpers
def plain_env(cfg, N, b, seed=11, env_offset=0, reward=None, window=64, flags=0, kind="Composite"):
    """a plain Env of one generator config with broker set b applied through initCash and the setters"""
    from madigan_b200.environments import Env
    e = Env(kind, b["init_cash"], {"data_source_config": cfg}, n_envs=N, window=window, seed=seed,
            env_offset=env_offset, reward=reward)
    e.setRequiredMargin(b["required_margin"])
    e.setMaintenanceMargin(b["maintenance_margin"])
    e.setSlippage(b["slippage_rel"], b["slippage_abs"])
    e.setTransactionCost(b["transaction_cost_rel"], b["transaction_cost_abs"])
    e.flags = flags
    return e


def broker_env(cfg, N, gen_sets, broker_sets, assign=None, seed=11, env_offset=0, reward=None, window=64, flags=0,
               kind="Composite"):
    from madigan_b200.environments import Env
    e = Env(kind, 1e6, {"data_source_config": cfg}, n_envs=N, window=window, seed=seed, env_offset=env_offset,
            reward=reward, param_sets=gen_sets, param_set=assign, broker_sets=broker_sets)
    e.flags = flags
    return e


def check_derived(multi, plains, tag):
    """Portfolio's derived accounting per env: the margins come from the env's set"""
    assign = multi.param_set.long()
    multi.invalidate()
    got = dict(am=multi.availableMargin.clone(), um=multi.usedMargin.clone(), risk=multi.checkRisk().clone(),
               eq=multi.equity.clone())
    for s, pl in enumerate(plains):
        idx = (assign == s).nonzero().squeeze(1)
        if idx.numel() == 0:
            continue
        pl.invalidate()
        ref = dict(am=pl.availableMargin, um=pl.usedMargin, risk=pl.checkRisk(), eq=pl.equity)
        for k, v in ref.items():
            assert same(got[k][idx], v[idx]), (tag, s, k)


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
@pytest.mark.parametrize("exact", [False, True], ids=["fast_gate", "forced_exact_gate"])
@pytest.mark.parametrize("kind", ["units", "actions", "weights", "generic_fill", "multi_wave"])
def test_broker_all_pairs_equivalence(kind, exact):
    """8 OU pairs, four generator sets and four broker sets at random: with DSR and auto-reset for 200 steps, the envs
    of each set equal a plain Env of that set, and so does their derived accounting.  generic_fill: the generic refill
    kernel; multi_wave: 155,648 envs (the multi-wave step instantiation)."""
    N = 155_648 if kind == "multi_wave" else 65_536
    flags = (A.FLAG_GENERIC_FILL if kind == "generic_fill" else 0) | (A.FLAG_FORCE_EXACT_GATE if exact else 0)
    g = torch.Generator(device="cuda").manual_seed(5)
    assign = torch.randint(0, len(BROKER), (N,), generator=g, device="cuda", dtype=torch.int32)
    multi = broker_env(PAIR_SETS[0], N, PAIR_SETS, BROKER, assign, reward=DSR, flags=flags)
    plains = [plain_env(c, N, b, reward=DSR, flags=flags) for c, b in zip(PAIR_SETS, BROKER)]
    assert multi.n_param_sets == 4 and torch.equal(multi.broker_table.cpu(), torch.tensor(
        [[b[k] for k in BROKER_SLOTS] for b in BROKER], dtype=torch.float64))
    check_sets(multi, plains, "constructor")
    envs = [multi] + plains
    n_done = torch.zeros(len(BROKER), dtype=torch.int64, device="cuda")
    seen = torch.zeros(4, dtype=torch.bool, device="cuda")  # risk codes met by the gates
    step_kind = kind if kind in ("actions", "weights") else "units"
    for t in range(200):
        step_all(envs, step_kind, g, N)
        n_done += torch.bincount(assign[multi.t["done"]].long(), minlength=len(BROKER))
        seen |= torch.bincount(multi.t["risk"].flatten().long(), minlength=4)[:4] > 0
        if t % 10 == 9:
            check_sets(multi, plains, f"step {t}")
        if t % 50 == 49:
            check_derived(multi, plains, f"step {t}")
    if step_kind == "units":
        assert int(n_done[2]) > 0, n_done  # the small-cash set's episodes end
        assert bool(seen[A.RISK_INSUFF_MARGIN]) and bool(seen[A.RISK_MARGIN_CALL]), seen


@pytest.mark.gpu
@pytest.mark.parametrize("knob", ["MDG_NO_TMA", "MDG_NO_BULK", "MDG_BS64"])
def test_broker_equivalence_operand_paths(knob):
    """The step kernel's other operand paths (row copies, plain loads; MDG_BS64: the plain Envs take the 64-thread
    instantiation, the sets launch keeps 128 threads), in child processes: the knobs are read once per process."""
    import subprocess
    import sys
    env = dict(os.environ, **{knob: "1"})
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k",
                        "test_broker_all_pairs_equivalence and units"], env=env, capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "2 passed" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True], ids=["fast_gate", "forced_exact_gate"])
def test_broker_generic_path_equivalence(exact):
    """C4 composite (Synth, OU, OUPair, SimpleTrend, TrendOU, TrendyOU) with three generator and three broker sets: hold,
    multi-asset and single-asset steps, explicit masked resets with history fill, derived accounting."""
    N = 4096
    flags = A.FLAG_FORCE_EXACT_GATE if exact else 0
    g = torch.Generator(device="cuda").manual_seed(9)
    assign = torch.randint(0, len(COMPOSITE_SETS), (N,), generator=g, device="cuda", dtype=torch.int32)
    bsets = [dict(BROKER[0], transaction_cost_rel=.001, slippage_rel=0.), BROKER[1], dict(BROKER[2],
                                                                                          transaction_cost_abs=20.)]
    multi = broker_env(COMPOSITE, N, COMPOSITE_SETS, bsets, assign, reward=PPC, window=16, flags=flags)
    plains = [plain_env(c, N, b, reward=PPC, window=16, flags=flags) for c, b in zip(COMPOSITE_SETS, bsets)]
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
            check_derived(multi, plains, f"step {t}")
        check_sets(multi, plains, f"step {t}")


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, A.FLAG_FORCE_EXACT_GATE], ids=["fast_gate", "forced_exact_gate"])
def test_margin_call_knife_edge_per_set(flags):
    """test_gpu_ledger_kat's margin-call probe (envTest.py:527-538) with two broker sets that differ only in the
    maintenance margin: 1,000,000 units of asset 1 bought at 4 with required margin 0.1, then the price falls to 3.69.
    Portfolio::checkRisk: balance + pnl = 290,000 against maintenance_margin * 310,000, so the move calls margin in the
    set with 1.0 and not in the set with 0.93 (threshold 0.9355).  Each set equals its plain Env."""
    cfg = {'freq': [1.] * 4, 'mu': [2., 4., 2.2, 2.3], 'amp': [0.] * 4, 'phase': [0.] * 4, 'dX': 0., 'noise': 0.}
    N = 8
    bsets = [dict(BROKER[0], required_margin=.1, maintenance_margin=m, slippage_rel=0., transaction_cost_rel=0.)
             for m in (1., .93)]
    assign = torch.tensor([0, 1] * 4, dtype=torch.int32)
    multi = broker_env(cfg, N, 2, bsets, assign, window=4, flags=flags, kind="Synth")
    plains = [plain_env(cfg, N, b, window=4, flags=flags, kind="Synth") for b in bsets]
    envs = [multi] + plains

    def set_mu(mu):
        multi.param_table[:, 1, 1] = mu
        for p in plains:
            p.P.gen[1].p[1] = mu

    u = torch.zeros((N, 4), dtype=torch.float64, device="cuda")
    u[:, 1] = 1_000_000
    for e in envs:
        e.step(u)
    check_sets(multi, plains, "buy", windows=False)
    assert (multi.t["risk"][1] == A.RISK_GREEN).all()
    set_mu(3.71)
    for e in envs:
        e.step()
    assert (multi.checkRisk() == A.RISK_GREEN).all() and not multi.t["done"].any()
    set_mu(3.69)
    for e in envs:
        e.step()
    check_sets(multi, plains, "3.69", windows=False)
    check_derived(multi, plains, "3.69")
    called = assign.cuda() == 0
    assert torch.equal(multi.checkRisk() == A.RISK_MARGIN_CALL, called)
    assert torch.equal(multi.t["done"], called)  # Env::step: done on a margin call (Env.h:196-198)
    u[:, 1] = 1000.
    for e in envs:
        e.step(u)
    check_sets(multi, plains, "order after the move", windows=False)
    assert torch.equal(multi.t["risk"][1] == A.RISK_MARGIN_CALL, called)


@pytest.mark.gpu
def test_reassignment_then_reset_takes_the_new_cash():
    """assign_param_sets(mask=done) + reset(mask=done, fill_history=True): the new episodes start with the new set's
    init_cash and from then on equal a plain Env of the new set that reset the same envs at the same step."""
    N = 4096
    g = torch.Generator(device="cuda").manual_seed(6)
    old = torch.randint(0, 4, (N,), generator=g, device="cuda", dtype=torch.int32)
    multi = broker_env(PAIR_SETS[0], N, PAIR_SETS, BROKER, old, window=16)
    plains = [plain_env(c, N, b, window=16) for c, b in zip(PAIR_SETS, BROKER)]
    envs = [multi] + plains
    done = torch.zeros(N, dtype=torch.bool, device="cuda")
    for _ in range(30):  # without auto-reset: finished envs stay done
        u = torch.randint(-1, 2, (N, 16), generator=g, device="cuda").double() * 40_000.
        for e in envs:
            e.step(u)
        done |= multi.t["done"]
    assert done.any()
    new = (old + 1 + torch.randint(0, 3, (N,), generator=g, device="cuda", dtype=torch.int32)) % 4  # another set
    multi.assign_param_sets(new, mask=done)
    assert torch.equal(multi.param_set, torch.where(done, new, old))
    for e in envs:
        e.reset(done, fill_history=True)
    cash0 = torch.tensor([b["init_cash"] for b in BROKER], dtype=torch.float64, device="cuda")
    assert torch.equal(multi.cash[done], cash0[new[done].long()])
    assert torch.equal(multi.initCash, cash0[multi.param_set.long()])
    # the last step's outputs (reward, transactions, risk, done) are the old set's until the next step
    outputs = ("reward", "done", "trans_price", "trans_units", "trans_cost", "risk", "margin_call")
    check_sets(multi, plains, "reset", names=tuple(n for n in STATE if n not in outputs))
    for t in range(60):
        step_all(envs, "units", g, N)
        if t % 10 == 9:
            check_sets(multi, plains, f"step {t}", names=STATE)
    check_derived(multi, plains, "end")


@pytest.mark.gpu
def test_setters_and_make_env():
    """On an Env with broker sets a setter writes its field into every set; make_env(config, broker_sets=...) equals
    an Env built directly, with the config's broker keys as base values."""
    from madigan_b200.environments import Env, make_env
    N = 2048
    config = dict(env_type="Synth", data_source_type="Composite", data_source_config=PAIR_SETS[0], init_cash=2e6,
                  required_margin=.2, maintenance_margin=.3, transaction_cost_rel=.01, transaction_cost_abs=.5,
                  slippage_rel=.002, slippage_abs=.001, n_envs=N, seed=21, preprocessor_config={"window_length": 16})
    bsets = [{}, {"init_cash": 5e5, "maintenance_margin": .1}, BROKER[3]]
    a = make_env(config, broker_sets=bsets)
    b = Env("Composite", 2e6, config, broker_sets=bsets)
    base = [2e6, .2, .3, .002, .001, .01, .5]
    assert a.broker_table[0].tolist() == base
    assert a.broker_table[1].tolist() == [5e5, .2, .1, .002, .001, .01, .5]
    assert torch.equal(a.broker_table, b.broker_table) and a.n_param_sets == 3
    g = torch.Generator(device="cuda").manual_seed(3)
    for _ in range(40):
        step_all([a, b], "units", g, N)
    for name in STATE + RINGS:
        assert same(a.t[name], b.t[name]), name
    # per-env values, then the setters on a fresh Env: every set takes the value
    assert torch.equal(a.requiredMargin, a.broker_table[a.param_set.long(), 1])
    assert a.initCash.shape == a.maintenanceMargin.shape == (N,)
    a = make_env(config, broker_sets=bsets)
    a.setRequiredMargin(.4)
    a.setMaintenanceMargin(.15)
    a.setSlippage(.003, .004)
    a.setTransactionCost(.005, .006)
    tab = a.broker_table.cpu()
    assert (tab[:, 1] == .4).all() and (tab[:, 2] == .15).all() and (tab[:, 3] == .003).all()
    assert (tab[:, 4] == .004).all() and (tab[:, 5] == .005).all() and (tab[:, 6] == .006).all()
    assert torch.equal(tab[:, 0], torch.tensor([2e6, 5e5, BROKER[3]["init_cash"]], dtype=torch.float64))
    assert (a.requiredMargin == .4).all() and (a.maintenanceMargin == .15).all()
    # ... and the envs of set 1 now trade as a plain Env with those settings and set 1's starting cash
    p = plain_env(PAIR_SETS[0], N, dict(init_cash=5e5, required_margin=.4, maintenance_margin=.15, slippage_rel=.003,
                                         slippage_abs=.004, transaction_cost_rel=.005, transaction_cost_abs=.006),
                  seed=21, window=16)
    for _ in range(30):
        step_all([a, p], "units", g, N)
    idx = (a.param_set == 1).nonzero().squeeze(1)
    for name in STATE:
        x, y = a.t[name], p.t[name]
        assert same(x[idx] if name == "pre_price" else x[..., idx], y[idx] if name == "pre_price" else y[..., idx]), name
    with pytest.raises(ValueError, match="broker_sets has 3 sets"):
        Env("Composite", 2e6, config, broker_sets=bsets, param_sets=2)
    with pytest.raises(ValueError, match="unknown broker setting"):
        Env("Composite", 2e6, config, broker_sets=[{"margin": 1.}])


@pytest.mark.gpu
def test_broker_checkpoint_round_trip():
    N = 2048
    g = torch.Generator(device="cuda").manual_seed(12)
    assign = torch.randint(0, 4, (N,), generator=g, device="cuda", dtype=torch.int32)
    a = broker_env(PAIR_SETS[0], N, PAIR_SETS, BROKER, assign, reward=DSR, window=16)
    for _ in range(10):
        step_all([a], "units", g, N)
    sd = a.state_dict()
    us = [torch.randint(-1, 2, (N, 16), generator=g, device="cuda").double() * 40_000. for _ in range(20)]
    for u in us:
        a.step(u, auto_reset=True)
    b = broker_env(PAIR_SETS[0], N, 4, 4, None, reward=DSR, window=16)  # other tables, other assignment
    b.load_state_dict(sd)
    assert torch.equal(b.param_set, assign) and torch.equal(b.broker_table, a.broker_table)
    for u in us:
        b.step(u, auto_reset=True)
    for name in STATE + RINGS:
        assert same(a.t[name], b.t[name]), name
    check_derived(b, [a] * 4, "after load")
    # generator sets without broker sets, and the other way round
    with pytest.raises(ValueError, match="broker sets"):
        broker_env(PAIR_SETS[0], N, 4, None, reward=DSR, window=16).load_state_dict(sd)
    with pytest.raises(ValueError, match="broker sets"):
        b.load_state_dict(broker_env(PAIR_SETS[0], N, 4, None, reward=DSR, window=16).state_dict())


@pytest.mark.gpu
def test_broker_sharding():
    """An Env with broker sets over 256 envs equals two 128-env halves with env_offset and the halves of the
    assignment, env for env."""
    g = torch.Generator(device="cuda").manual_seed(8)
    assign = torch.randint(0, 4, (256,), generator=g, device="cuda", dtype=torch.int32)
    big = broker_env(PAIR_SETS[0], 256, PAIR_SETS, BROKER, assign, seed=99, window=8)
    lo = broker_env(PAIR_SETS[0], 128, PAIR_SETS, BROKER, assign[:128], seed=99, window=8)
    hi = broker_env(PAIR_SETS[0], 128, PAIR_SETS, BROKER, assign[128:], seed=99, env_offset=128, window=8)
    for t in range(60):
        u = torch.randint(-1, 2, (256, 16), generator=g, device="cuda").double() * 40_000.
        big.step(u, auto_reset=True)
        lo.step(u[:128].contiguous(), auto_reset=True)
        hi.step(u[128:].contiguous(), auto_reset=True)
    for name in STATE + RINGS:
        if name == "pre_price":
            assert same(big.t[name], torch.cat([lo.t[name], hi.t[name]], dim=0)), name
        else:
            assert same(big.t[name], torch.cat([lo.t[name], hi.t[name]], dim=-1)), name
