"""Per-set episode results (utils.metrics.EpisodeResults) on the GPU.

Env A steps with ``auto_reset=True, results=res``: the fused step records, harvests every finished episode into the
exact per-set table and re-arms the recorder.  Env B follows the manual recipe: ``step(..., tearsheet=ts)``, the
``ts.summary()`` rows of the envs that finished with their set and starting cash, ``ts.reset(done)`` and the explicit
masked reset of test_param_set_draw (restated draws when the draw is on).  The table built by
oracle/episode_results_oracle.py from B's rows must equal A's limbs exactly, and A's envs and recorders B's, bit for
bit."""
import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from madigan_b200.environments.data_source import make_set_cdf
from madigan_b200.utils.metrics import EpisodeResults, EpisodeTearsheet, carry_
from oracle import episode_results_oracle as O
from test_param_set_draw import W3, W4, draw_env, initial, manual_reset, units
from test_param_sets import COMPOSITE, COMPOSITE_SETS, DSR, PAIR_SETS, RINGS, STATE, same

pytestmark = pytest.mark.gpu


def plain_env(N, seed=11, env_offset=0, window=16):
    """an Env without parameter sets (one row), the margins and costs of draw_env"""
    from madigan_b200.environments import Env
    e = Env("Composite", 1e6, {"data_source_config": PAIR_SETS[0]}, n_envs=N, window=window, seed=seed,
            env_offset=env_offset, reward=DSR)
    e.setRequiredMargin(.1)
    e.setMaintenanceMargin(.25)
    e.setTransactionCost(.02, 0.)
    e.setSlippage(.001, 0.)
    return e


CASES = {  # name: (base config, sets (None: a plain Env), weights, broker sets, N, flags, n_offsets, stepping)
    "pairs": (PAIR_SETS[0], PAIR_SETS, None, False, 2048, 0, 6, "units"),
    "pairs_broker": (PAIR_SETS[0], PAIR_SETS, None, True, 2048, 0, 6, "units"),
    "pairs_draw_broker": (PAIR_SETS[0], PAIR_SETS, W4, True, 2048, 0, 6, "units"),
    "generic_fill_draw": (PAIR_SETS[0], PAIR_SETS, W4, False, 2048, A.FLAG_GENERIC_FILL, 6, "units"),
    "composite_draw": (COMPOSITE, COMPOSITE_SETS, W3, False, 1024, 0, 6, "units"),
    "plain": (PAIR_SETS[0], None, None, False, 2000, 0, 3, "units"),
    "plain_no_offsets": (PAIR_SETS[0], None, None, False, 1000, 0, 0, "units"),
    "S_eq_N_draw": (PAIR_SETS[0], 777, None, False, 777, 0, 6, "units"),
    "actions_draw_broker": (PAIR_SETS[0], PAIR_SETS, W4, True, 2048, 0, 6, "actions"),
    "noise_draw_broker": (COMPOSITE, COMPOSITE_SETS, W3, True, 512, 0, 4, "noise"),
}


def build(name):
    cfg, sets, w, broker, N, flags, J, how = CASES[name]
    if sets is None:
        return plain_env(N), plain_env(N), None
    if isinstance(sets, int):  # S = N sets (every slot of the base config scaled by 0.9 .. 1.1), drawn uniformly
        w = [1.] * sets
        a = draw_env(cfg, [cfg] * sets, N, w)
        cdf = make_set_cdf(w)
        b = draw_env(cfg, [cfg] * sets, N, None, initial(a, cdf))
        for e in (a, b):
            g = torch.Generator(device="cuda").manual_seed(21)
            e.param_table.mul_(0.9 + 0.2 * torch.rand(e.param_table.shape, generator=g, device="cuda",
                                                      dtype=torch.float64))
        return a, b, cdf
    a = draw_env(cfg, sets, N, w, broker=broker, flags=flags)
    cdf = make_set_cdf(w) if w is not None else None
    b = draw_env(cfg, sets, N, None, initial(a, cdf) if w is not None else None, broker=broker, flags=flags)
    return a, b, cdf


def start_cash(env):
    """(N,) starting cash of every env's current episode"""
    c = env.initCash
    return c if isinstance(c, torch.Tensor) else torch.full((env.N,), float(c), dtype=torch.float64, device="cuda")


def take_rows(b, ts, done, log):
    if not bool(done.any()):
        return
    summ = ts.summary()
    log["rows"].append(torch.stack([summ[n] for n in ts.fields()], 1)[done].cpu())
    ids = b.param_set if b.param_set is not None else torch.zeros(b.N, dtype=torch.int32, device="cuda")
    log["sets"].append(ids[done].cpu())
    log["cash"].append(start_cash(b)[done].cpu())
    log["mc"].append(b.t["margin_call"][done].cpu())


def oracle_of(log, n_sets):
    cat = lambda k: torch.cat(log[k]).numpy()
    return O.table(cat("rows"), cat("sets"), n_sets, cash=cat("cash"), margin_call=cat("mc")), cat("rows")


def assert_same_envs(a, b, tag):
    for name in STATE + RINGS:
        assert same(a.t[name], b.t[name]), (tag, name)
    if a.param_set is not None:
        assert torch.equal(a.param_set, b.param_set), (tag, "param_set")


def assert_same_recorders(x, y, tag):
    for k in x.t:
        assert same(x.t[k], y.t[k]), (tag, k)


def check_table(res, tab_o, rows, sets):
    """A's limbs equal the oracle's exactly; its statistics agree with numpy over B's rows"""
    acc, ext = O.limbs(tab_o)
    lim = res.limbs()
    assert np.array_equal(lim["acc"].cpu().numpy(), acc)
    assert np.array_equal(lim["ext"].cpu().numpy(), ext)
    tab = res.table()
    names = res.fields()
    S = res.n_sets
    assert tab["n_episodes"].tolist() == tab_o["n_episodes"]
    assert tab["n_margin_call"].tolist() == tab_o["n_margin_call"]
    for f, n in enumerate(names):
        assert tab[f"{n}_count"].tolist() == [c[f] for c in tab_o["count"]], n
        assert np.array_equal(tab[f"{n}_min"].cpu().numpy(), tab_o["min"][:, f], equal_nan=True), n
        assert np.array_equal(tab[f"{n}_max"].cpu().numpy(), tab_o["max"][:, f], equal_nan=True), n
        np.testing.assert_allclose(tab[f"{n}_std"].cpu().numpy(), tab_o["std"][:, f], rtol=1e-9, err_msg=n)
    # numpy over B's rows (money fields over the starting cash, values that are not admitted left out)
    for s in range(S):
        x = rows[sets == s]
        for f, n in enumerate(names):
            y = x[:, f]
            y = y[np.isfinite(y) & (np.abs(y) < 2. ** 31)]
            if len(y) == 0:
                assert np.isnan(tab[f"{n}_mean"][s].item())
                continue
            scale = np.abs(y).max()
            np.testing.assert_allclose(tab[f"{n}_mean"][s].item(), y.mean(), rtol=1e-12, atol=1e-14 * scale, err_msg=n)
            if len(y) > 1:  # variances to 2e-9 relative, beyond what the 2^-65 rounding of v and v*v and the fp64
                # decode of the sum of squares can move them
                k = len(y) / (len(y) - 1)
                bound = k * (2. ** -65 * (1 + 2 * abs(y.mean())) + 4e-16 * (y * y).mean())
                var, want = tab[f"{n}_std"][s].item() ** 2, y.var(ddof=1)
                assert abs(var - want) <= 2e-9 * want + bound, (n, s, var, want, bound)


@pytest.mark.parametrize("name", list(CASES))
def test_results_equal_manual_recipe(name):
    cfg, sets, w, broker, N, flags, J, how = CASES[name]
    a, b, cdf = build(name)
    res = EpisodeResults(a, J)
    ts = EpisodeTearsheet(b, J)
    assert res.n_sets == max(a.n_param_sets, 1) and res.fields() == ts.fields()
    g = torch.Generator(device="cuda").manual_seed(7)
    log = dict(rows=[], sets=[], cash=[], mc=[])
    steps = 150 if how == "noise" else 200
    for t in range(steps):
        u = units(g, N)
        n0 = a.launches
        if how == "units":
            a.step(u, auto_reset=True, results=res)
            assert a.launches - n0 == 3
            b.step(u, tearsheet=ts)
        elif how == "actions":
            acts = torch.randint(0, 3, (N, 16), generator=g, device="cuda", dtype=torch.int8)
            a.step_actions(acts, action_atoms=3, unit_size=.3, auto_reset=True, results=res)
            assert a.launches - n0 == 3
            b.step_actions(acts, action_atoms=3, unit_size=.3)
            ts.update()
        else:
            nz = torch.randn((a.P.n_normals, N), generator=g, device="cuda", dtype=torch.float64)
            uz = torch.rand((a.P.n_uniforms, N), generator=g, device="cuda", dtype=torch.float64)
            a.step(u, normals=nz, uniforms=uz, auto_reset=True, results=res)
            assert a.launches - n0 == 4  # step, record, list scan, refill
            b.step(u, normals=nz, uniforms=uz, tearsheet=ts)
        done = b.t["done"].clone()
        assert torch.equal(a.t["done"], done), t
        take_rows(b, ts, done, log)
        ts.reset(done)
        if cdf is not None:
            manual_reset(b, cdf, done)
        else:
            b.reset(mask=done, fill_history=True)
        assert_same_envs(a, b, f"step {t}")
    assert_same_recorders(res.tearsheet, ts, "recorders")
    tab_o, rows = oracle_of(log, res.n_sets)
    assert sum(tab_o["n_episodes"]) >= 200, sum(tab_o["n_episodes"])
    money = np.asarray(O.MONEY)
    rows[:, money] /= torch.cat(log["cash"]).numpy()[:, None]
    check_table(res, tab_o, rows, torch.cat(log["sets"]).numpy())


def test_results_change_nothing():
    """An Env with results has the state of the same Env without them, bit for bit, over the same steps."""
    N = 1024
    a = draw_env(PAIR_SETS[0], PAIR_SETS, N, W4, broker=True)
    b = draw_env(PAIR_SETS[0], PAIR_SETS, N, W4, broker=True)
    res = EpisodeResults(a, 6)
    g = torch.Generator(device="cuda").manual_seed(3)
    for t in range(100):
        u = units(g, N)
        a.step(u, auto_reset=True, results=res)
        b.step(u, auto_reset=True)
        assert_same_envs(a, b, f"step {t}")
        assert torch.equal(a.episode_param_set, b.episode_param_set)
    assert int(res.table()["n_episodes"].sum()) > 100


def test_shard_invariance():
    """Two Envs with env_offset over the halves of one slab, the draw on: their tables added limb-wise and carried
    equal the one-slab table exactly."""
    kw = dict(weights=W4, seed=99, window=8, broker=True)
    big = draw_env(PAIR_SETS[0], PAIR_SETS, 512, **kw)
    lo = draw_env(PAIR_SETS[0], PAIR_SETS, 256, **kw)
    hi = draw_env(PAIR_SETS[0], PAIR_SETS, 256, env_offset=256, **kw)
    rb, rl, rh = EpisodeResults(big), EpisodeResults(lo), EpisodeResults(hi)
    rl._carry_every = 7  # carries mid-run on one shard only: the sums are the same
    g = torch.Generator(device="cuda").manual_seed(8)
    for t in range(120):
        u = units(g, 512)
        big.step(u, auto_reset=True, results=rb)
        lo.step(u[:256].contiguous(), auto_reset=True, results=rl)
        hi.step(u[256:].contiguous(), auto_reset=True, results=rh)
    one, a, b = rb.limbs(), rl.limbs(), rh.limbs()
    assert int(one["acc"][:, 0].sum()) > 200
    assert torch.equal(carry_(a["acc"] + b["acc"]), one["acc"])
    assert torch.equal(torch.minimum(a["ext"][0], b["ext"][0]), one["ext"][0])
    assert torch.equal(torch.maximum(a["ext"][1], b["ext"][1]), one["ext"][1])


def test_checkpoint_round_trip():
    """state_dict mid-run, load into fresh objects, continue: exactly the uninterrupted run."""
    N = 2048
    g = torch.Generator(device="cuda").manual_seed(12)
    a = draw_env(PAIR_SETS[0], PAIR_SETS, N, W4, broker=True)
    ra = EpisodeResults(a, 5)
    for _ in range(30):
        a.step(units(g, N), auto_reset=True, results=ra)
    sd_env, sd_res = a.state_dict(), ra.state_dict()
    us = [units(g, N) for _ in range(40)]
    for u in us:
        a.step(u, auto_reset=True, results=ra)
    b = draw_env(PAIR_SETS[0], PAIR_SETS, N, W4, broker=True, seed=5)
    b.load_state_dict(sd_env)
    rb = EpisodeResults(b, 5)
    rb.load_state_dict(sd_res)
    for u in us:
        b.step(u, auto_reset=True, results=rb)
    la, lb = ra.limbs(), rb.limbs()
    assert torch.equal(la["acc"], lb["acc"]) and torch.equal(la["ext"], lb["ext"])
    assert_same_recorders(ra.tearsheet, rb.tearsheet, "resumed")
    for other in (EpisodeResults(b, 4), EpisodeResults(plain_env(N), 5), EpisodeResults(plain_env(N // 2), 5)):
        with pytest.raises(ValueError):
            other.load_state_dict(sd_res)


def test_errors_and_reset():
    N = 1000
    a = plain_env(N)
    other = plain_env(N)
    res = EpisodeResults(a, 6)
    u = torch.zeros((N, 16), dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError, match="auto_reset"):
        a.step(u, results=res)
    with pytest.raises(ValueError, match="tearsheet"):
        a.step(u, auto_reset=True, results=res, tearsheet=EpisodeTearsheet(a))
    with pytest.raises(ValueError, match="another Env"):
        other.step(u, auto_reset=True, results=res)
    with pytest.raises(ValueError, match="another Env"):
        other.step_weights(torch.ones((N, 17)), auto_reset=True, results=res)
    with pytest.raises(ValueError, match="auto_reset"):
        a.step_actions(torch.zeros((N, 16), dtype=torch.int8), action_atoms=3, unit_size=.1, results=res)
    assert int(a.t["timestamp"][0]) == int(other.t["timestamp"][0])  # nothing was launched
    g = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(60):
        a.step_weights(torch.rand((N, 17), generator=g, device="cuda"), auto_reset=True, results=res)
        a.step(units(g, N), auto_reset=True, results=res)
    tab = res.table()
    assert int(tab["n_episodes"][0]) > 0
    res.reset()
    tab = res.table()
    assert int(tab["n_episodes"][0]) == 0 and int(tab["nsteps_count"][0]) == 0
    assert torch.isnan(tab["nsteps_mean"]).all() and torch.isnan(tab["final_equity_min"]).all()
    n = 0
    for _ in range(60):
        a.step(units(g, N), auto_reset=True, results=res)
        n += int(a.t["done"].sum())
    tab = res.table()
    assert n > 0 and int(tab["n_episodes"][0]) == n and int(tab["nsteps_count"][0]) == n
    assert float(tab["nsteps_min"][0]) >= 1.
