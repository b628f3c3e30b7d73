"""The CPU oracle against the REFERENCE'S OWN C++ env, compiled unmodified from its sources
(oracle/ref_build.py -> oracle/_ref/libmadigan_ref.so: Env.h, Broker.cpp, Account.cpp, Portfolio.cpp,
DataSource.cpp, Config.cpp against a small Eigen shim with left-to-right folds, strict IEEE flags).

Both sides get the same actions; the reference's generator is re-seeded and a clone of its engine +
distribution objects yields the standard normals it is about to draw, which are injected into the oracle.
Every output of Env::step -- prices, ledgerNormedFull, reward, done, transaction price/units/cost, risk codes,
marginCall -- and the accounting properties must then agree BIT FOR BIT (same compiler, same libm).
This pins what the reference's own tests leave unpinned: OU / OUPair / noisy Synth generators, Env::step's
reward clamp and done logic, slippage and transaction-cost arithmetic, the risk gates under leverage.

Skipped when the reference build is absent: oracle/ref_build.py produces it from the madigan checkout that
MADIGAN_REFERENCE names."""
import zlib

import numpy as np
import pytest

from madigan_b200 import _abi as A
from madigan_b200.environments.data_source import make_params
from oracle import ref
from oracle.oracle import OracleEnv

pytestmark = pytest.mark.skipif(not ref.available(), reason="oracle/_ref not built (needs MADIGAN_REFERENCE)")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.array_equal(bits(a), bits(b)) or np.array_equal(a, b, equal_nan=True)


CASES = {
    "synth": (ref.SYNTH, "Synth", dict(freq=[1., 0.3, 2.], mu=[2., 2.1, 2.2], amp=[1., 1.2, 1.3], phase=[0., 1., 2.],
                                       dX=0.01, noise=0.05)),
    "ou": (ref.OU, "OU", dict(mean=[10., 5., 1., 2.], theta=[.08, .15, .15, .1], phi=[.04, .02, .01, .03])),
    "oupair": (ref.OUPAIR, "OUPair", dict(theta=.015, phi=.01, noise=.03)),
    "sawtooth": (ref.SAWTOOTH, "SawTooth", dict(freq=[1., 0.3, 2.], mu=[2., 2.1, 2.2], amp=[1., 1.2, 1.3],
                                                phase=[0., 1., 2.], dX=0.01, noise=0.05)),
    "triangle": (ref.TRIANGLE, "Triangle", dict(freq=[1., 0.3, 2.], mu=[2., 2.1, 2.2], amp=[1., 1.2, 1.3],
                                                phase=[0., 1., 2.], dX=0.01, noise=0.05)),
    "gaussian": (ref.GAUSSIAN, "Gaussian", dict(mean=[2., 5., 10.], var=[.5, 1., 2.])),
    "pairs8": (ref.MULTIPAIR, "Composite", dict(theta=.015, phi=.01, noise=.03)),
}


def build(case, margins, costs, seed):
    kind, ds_type, cfg = CASES[case]
    if kind in (ref.SYNTH, ref.SAWTOOTH, ref.TRIANGLE):
        n = len(cfg["freq"])
        p = [x for i in range(n) for x in (cfg["freq"][i], cfg["mu"][i], cfg["amp"][i], cfg["phase"][i])]
        p += [cfg["dX"], cfg["noise"]]
        ds_cfg = cfg
    elif kind == ref.OU:
        n = len(cfg["mean"])
        p = [x for i in range(n) for x in (cfg["mean"][i], cfg["theta"][i], cfg["phi"][i])]
        ds_cfg = cfg
    elif kind == ref.GAUSSIAN:
        n = len(cfg["mean"])
        p = [x for i in range(n) for x in (cfg["mean"][i], cfg["var"][i])]
        ds_cfg = cfg
    elif kind == ref.OUPAIR:
        n, p, ds_cfg = 2, [cfg["theta"], cfg["phi"], cfg["noise"]], cfg
    else:
        n, p = 16, [cfg["theta"], cfg["phi"], cfg["noise"]]
        ds_cfg = {f"pair{i}": {"data_source_type": "OUPair", "data_source_config": cfg} for i in range(8)}
    r = ref.RefEnv(kind, n, p, 1_000_000., seed)
    r.set(margins[0], margins[1], *costs)
    P, _ = make_params(ds_type, ds_cfg, required_margin=margins[0], maintenance_margin=margins[1],
                       transaction_cost_rel=costs[0], transaction_cost_abs=costs[1], slippage_rel=costs[2],
                       slippage_abs=costs[3])
    o = OracleEnv(P, construct=False)
    return r, o, P.n_assets


def gen_units(rng, o, n, scale):
    price = np.where(np.abs(o.prices) > 1e-9, o.prices, 1.0)
    led = o.ledger.copy()
    a = rng.integers(-1, 2, size=n).astype(np.float64)
    units = a * (scale / np.abs(price)) * rng.uniform(0.2, 1.5, size=n)
    r = rng.random(n)
    units = np.where(r < 0.08, -led, units)
    units = np.where((r >= 0.08) & (r < 0.14), -2. * led, units)
    units = np.where((r >= 0.14) & (r < 0.17), -0.5 * led, units)
    units = np.where((r >= 0.17) & (r < 0.20), units * 50., units)
    return units


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("margins,costs,scale", [
    ((1., .25), (0., 0., 0., 0.), 30_000.),
    ((.1, .25), (.02, 1.5, .001, .002), 400_000.),
    ((.05, 1.), (.001, 0., 0., 0.), 900_000.),
])
def test_env_step_bit_exact_vs_reference(case, margins, costs, scale):
    rng = np.random.default_rng(zlib.crc32(f"{case}/{margins}".encode()))  # stable across processes (hash() is salted)
    r, o, n = build(case, margins, costs, seed=4242)
    z = r.next_normals()
    rs, os_ = r.reset(), o.reset(normals=z)
    assert same(rs["price"], os_["price"]) and same(rs["portfolio"], os_["portfolio"])
    seen, dones = set(), 0
    for t in range(400):
        mode = t % 7
        z = r.next_normals()
        if mode == 5:
            ro, oo = r.step(), o.step(normals=z)
        elif mode == 6:
            i = int(rng.integers(0, n))
            u = float(gen_units(rng, o, n, scale)[i])
            ro, oo = r.step(u, asset_idx=i), o.step(u, asset_idx=i, normals=z)
        else:
            u = gen_units(rng, o, n, scale)
            ro, oo = r.step(u), o.step(u, normals=z)
        for k in ("price", "portfolio", "transactionPrice", "transactionUnits", "transactionCost"):
            assert same(ro[k], oo[k]), f"step {t} {k}"
        assert same(ro["reward"], oo["reward"]), f"step {t} reward {ro['reward']} {oo['reward']}"
        assert ro["done"] == oo["done"], f"step {t} done"
        assert np.array_equal(ro["riskInfo"], oo["riskInfo"]), f"step {t} riskInfo"
        if mode != 5:
            assert ro["marginCall"] == oo["marginCall"], f"step {t} marginCall"
        acc = r.accounting()
        assert same(acc["ledger"], o.ledger) and same(acc["meanEntryPrices"], o.meanEntryPrices)
        for k, v in (("equity", o.equity), ("cash", o.cash), ("pnl", o.pnl), ("balance", o.balance),
                     ("availableMargin", o.availableMargin), ("usedMargin", o.usedMargin),
                     ("borrowedMargin", o.borrowedMargin), ("borrowedAssetValue", o.borrowedAssetValue)):
            assert same(acc[k], v), f"step {t} {k}: {acc[k]!r} vs {v!r}"
        seen |= set(int(x) for x in oo["riskInfo"])
        if oo["done"]:
            dones += 1
            z = r.next_normals()
            rs, os_ = r.reset(), o.reset(normals=z)
            assert same(rs["price"], os_["price"]) and same(rs["portfolio"], os_["portfolio"])
    if margins[0] < 1.:
        assert A.RISK_INSUFF_MARGIN in seen


TREND = dict(trend_prob=[.05, .1, .02], min_period=[3, 5, 10], max_period=[9, 30, 40],
             dYMin=[.001, .02, .05], dYMax=[.01, .2, .6], start=[10., .5, 2.])
TREND_CASES = {
    "simpletrend": (ref.SIMPLETREND, "SimpleTrend", dict(TREND, noise=[.01, .05, .2])),
    "trendou": (ref.TRENDOU, "TrendOU", dict(TREND, theta=[.1, .3, .05], phi=[.02, .1, .3], noise_trend=[.01, .05, .2],
                                             ema_alpha=[.1, .2, .3])),
    "trendyou": (ref.TRENDYOU, "TrendyOU", dict(TREND, theta=[.1, .3, .05], phi=[.02, .1, .3],
                                                noise_trend=[.01, .05, .2], ema_alpha=[.1, .2, .3])),
}


def build_trend(case, seed):
    kind, ds_type, cfg = TREND_CASES[case]
    n = len(cfg["start"])
    if kind == ref.SIMPLETREND:
        keys = ("trend_prob", "min_period", "max_period", "noise", "start", "dYMin", "dYMax")
    else:
        keys = ("trend_prob", "min_period", "max_period", "dYMin", "dYMax", "start", "theta", "phi", "noise_trend",
                "ema_alpha")
    p = [float(cfg[k][i]) for i in range(n) for k in keys]
    r = ref.RefEnv(kind, n, p, 1_000_000., seed)
    r.set(.1, .25, .02, 0., .001, 0.)
    P, _ = make_params(ds_type, cfg, required_margin=.1, maintenance_margin=.25, transaction_cost_rel=.02,
                       slippage_rel=.001)
    for i in range(n):
        assert P.gen[i].nslot == i and P.gen[i].uslot == 4 * i
    return r, OracleEnv(P, construct=False), n


def oracle_trend_state(o, P_type, n):
    """(dY, direction, length, trending) from the oracle's packed generator state"""
    gs = np.ctypeslib.as_array(o.e.gstate)
    per = {ref.SIMPLETREND: (2, 0, 1), ref.TRENDOU: (3, 1, 2), ref.TRENDYOU: (4, 2, 3)}[P_type]
    dY = np.array([gs[per[0] * i + per[1]] for i in range(n)])
    f = np.array([gs[per[0] * i + per[2]] for i in range(n)]).view(np.int64)
    return dict(dY=dY, direction=np.where(f & 2, 1, -1), length=(f >> 32).astype(np.int32), trending=(f & 1) == 1)


@pytest.mark.parametrize("case", list(TREND_CASES))
@pytest.mark.parametrize("seed", [7, 4242])
def test_trend_generators_bit_exact_vs_reference(case, seed):
    """SimpleTrend / TrendOU / TrendyOU: data-dependent draw pattern (uniform test, direction, integer trend
    length, dY), floors at 0.01 / 0.1 and direction flips -- prices and the trend state machine bit for bit."""
    kind = TREND_CASES[case][0]
    rng = np.random.default_rng(seed)
    r, o, n = build_trend(case, seed)
    z, u = r.next_draws(after_reset=True)
    rs, os_ = r.reset(), o.reset(normals=z, uniforms=u)
    assert same(rs["price"], os_["price"])
    n_trending, dones, floors = 0, 0, 0
    for t in range(3000):
        z, u = r.next_draws()
        units = gen_units(rng, o, n, 60_000.) if t % 5 else None
        ro, oo = r.step(units), o.step(units, normals=z, uniforms=u)
        assert same(ro["price"], oo["price"]), f"step {t}: {ro['price']} vs {oo['price']}"
        assert same(ro["portfolio"], oo["portfolio"]) and same(ro["reward"], oo["reward"]), f"step {t}"
        assert ro["done"] == oo["done"]
        a, b = r.trend_state(), oracle_trend_state(o, kind, n)
        assert np.array_equal(a["trending"], b["trending"]), f"step {t}"
        assert same(a["dY"], b["dY"]), f"step {t}"
        live = a["trending"]
        assert np.array_equal(a["length"][live], b["length"][live]), f"step {t}"
        n_trending += int(live.sum())
        floors += int((ro["price"] <= .1001).sum())
        if oo["done"]:
            dones += 1
            z, u = r.next_draws(after_reset=True)
            rs, os_ = r.reset(), o.reset(normals=z, uniforms=u)
            assert same(rs["price"], os_["price"])
    assert n_trending > 200


def test_reference_timestamp_counts_ticks():
    """The reference leaves timestamp_ uninitialised (quirk A8); its increments are still one per getData."""
    r, o, n = build("oupair", (1., .25), (0., 0., 0., 0.), seed=1)
    t0 = r.reset()["timestamp"]
    t1 = r.step()["timestamp"]
    t2 = r.step(np.zeros(2))["timestamp"]
    assert t1 - t0 == 1 and t2 - t1 == 1


# ---------------------------------------------------------------------------------------------------------
# SineAdder / SineDynamic / SineDynamicTrend (DataSource.cpp:663-673, 802-841, 1002-1047; WaveTableOsc.h;
# randomBoolGenerator.h) -- left unpinned by the reference's own tests
# ---------------------------------------------------------------------------------------------------------
SINE_DYN = dict(freqRange=[[.1, 1., .01], [0.3, 3.0, .01], [5., 15., .1], [10., 50., .1]],
                muRange=[[1., 5., .02], [.3, 3., .05], [.2, 5., .02], [.5, 5., .02]],
                ampRange=[[1., 5., .01], [.3, 3., .02], [.2, 2., .04], [.5, 5., .05]], dX=0.01, noise=.3)
SINE_CASES = {
    "adder": (ref.SINEADDER, "SineAdder", dict(freq=[1., 0.3, 2., 0.5], mu=[2., 2.1, 2.2, 2.3], amp=[1., 1.2, 1.3, 1.],
                                                phase=[0., 1., 2., 1.], dX=0.01, noise=.05)),
    "dynamic": (ref.SINEDYNAMIC, "SineDynamic", SINE_DYN),
    "dynamic_3comp": (ref.SINEDYNAMIC, "SineDynamic",
                      dict(freqRange=[[.5, 2., .05], [1., 20., .5], [2., 4., .01]], muRange=[[1., 2., .1]] * 3,
                           ampRange=[[.1, .5, .05]] * 3, dX=0.02, noise=0.)),
    # short, likely trends so that the state machine turns over many times in a few thousand ticks
    "trend": (ref.SINEDYNAMICTREND, "SineDynamicTrend",
              dict(SINE_DYN, trendRange=[[5, 40], [10, 30]], trendIncr=[0.01, 0.02], trendProb=[.02, .05])),
    "trend_default_shape": (ref.SINEDYNAMICTREND, "SineDynamicTrend",
                            dict(SINE_DYN, trendRange=[[100, 500], [100, 300]], trendIncr=[0.1, 0.2],
                                 trendProb=[.001, .01], noise=1.)),
}


def build_sine(case, seed):
    kind, ds_type, cfg = SINE_CASES[case]
    if kind == ref.SINEADDER:
        K = len(cfg["freq"])
        p = [x for i in range(K) for x in (cfg["freq"][i], cfg["mu"][i], cfg["amp"][i], cfg["phase"][i])]
        p += [cfg["dX"], cfg["noise"]]
    else:
        K = len(cfg["freqRange"])
        p = [x for i in range(K) for x in cfg["freqRange"][i] + cfg["muRange"][i] + cfg["ampRange"][i]]
        p += [cfg["dX"], cfg["noise"]]
        if kind == ref.SINEDYNAMICTREND:
            T = len(cfg["trendProb"])
            p += [T] + [x for j in range(T) for x in (*cfg["trendRange"][j], cfg["trendIncr"][j], cfg["trendProb"][j])]
    r = ref.RefEnv(kind, K, p, seed=seed)
    r.set(.1, .25, .02, 0., .001, 0.)
    P, names = make_params(ds_type, cfg, required_margin=.1, maintenance_margin=.25, transaction_cost_rel=.02,
                           slippage_rel=.001)
    assert P.n_assets == 1 and P.gen[0].nslot == 0
    return r, OracleEnv(P, construct=False), kind, K


def oracle_sine_state(o, kind, K, T):
    gs = np.ctypeslib.as_array(o.e.gstate)
    if kind == ref.SINEADDER:
        return dict(comp=gs[:K].copy())
    out = dict(comp=gs[:4 * K].copy())
    if kind == ref.SINEDYNAMICTREND:
        f = gs[4 * K + 1: 4 * K + 1 + T].copy().view(np.int64)
        out.update(trend_component=gs[4 * K], direction=np.where(f & 2, 1, -1), length=(f >> 32).astype(np.int32),
                   trending=(f & 1) == 1)
    return out


@pytest.mark.parametrize("case", list(SINE_CASES))
@pytest.mark.parametrize("seed", [11, 909])
def test_sine_sources_bit_exact_vs_reference(case, seed):
    """SineAdder, SineDynamic, SineDynamicTrend through Env.step: prices, the bounded parameter walks, the
    wave-table oscillator phase, the trend state machine and reset()'s re-sampled (freq, mu, amp), bit for bit."""
    rng = np.random.default_rng(seed)
    r, o, kind, K = build_sine(case, seed)
    T = len(SINE_CASES[case][2].get("trendProb", []))

    def do_reset():
        z, u, cu = r.next_sine_draws(after_reset=True)
        o.set_ctor_uniforms(cu if kind != ref.SINEADDER else None)
        rs, os_ = r.reset(), o.reset(normals=z, uniforms=u)
        assert same(rs["price"], os_["price"]), (rs["price"], os_["price"])

    def compare_state(t):
        a = r.sine_state(T)
        b = oracle_sine_state(o, kind, K, T)
        na = K if kind == ref.SINEADDER else 4 * K
        assert same(a["comp"][:na], b["comp"]), f"step {t}: {a['comp'][:na]} vs {b['comp']}"
        if kind == ref.SINEDYNAMICTREND:
            assert same(a["trend_component"], b["trend_component"]), f"step {t}"
            assert np.array_equal(a["trending"], b["trending"]), f"step {t}"
            live = a["trending"]
            assert np.array_equal(a["length"][live], b["length"][live]), f"step {t}"
            assert np.array_equal(a["direction"][live], b["direction"][live]), f"step {t}"
            return int(live.sum())
        return 0

    do_reset()
    compare_state(-1)
    n_trending, resets = 0, 0
    for t in range(3000):
        z, u, _ = r.next_sine_draws()
        units = gen_units(rng, o, 1, 20_000.) if t % 5 else None
        ro, oo = r.step(units), o.step(units, normals=z, uniforms=u)
        assert same(ro["price"], oo["price"]), f"step {t}: {ro['price']} vs {oo['price']}"
        assert same(ro["portfolio"], oo["portfolio"]) and same(ro["reward"], oo["reward"]), f"step {t}"
        assert ro["done"] == oo["done"]
        n_trending += compare_state(t)
        if oo["done"] or t % 700 == 699:
            resets += 1
            do_reset()
            compare_state(t)
    assert resets >= 4
    if case == "trend":
        assert n_trending > 300
