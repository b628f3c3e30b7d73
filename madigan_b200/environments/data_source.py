"""Synthetic dataSource configuration -> per-asset generator table (``MdgParams.gen``).

Host-side mirror of the reference's config plumbing for the synthetic sources:
``makeConfigFromPyDict`` (reference: madigan/environments/cpp/Config.cpp:5-164 and
the per-type builders :166-577) and ``makeDataSource`` (DataSource.cpp:9-108).  The
Python-dict key names (``trend_prob``, ``noise_trend`` ...) are the ones the
reference's pybind boundary accepts; the C++ camelCase names are accepted too.

Deviations, all listed in SURVEY.md Appendix A:
  * Composite sub-sources keep config insertion order and may repeat a type
    (A11; the reference keys them by type name in an unordered_map).
  * ``SimpleTrend`` takes config keys, never positions (A10).
"""
import math
import numbers

import numpy as np

from .. import _abi as A


class ConfigError(RuntimeError):
    """reference: ConfigError is a std::logic_error (DataTypes.h:36-40) -> RuntimeError in Python."""


_SINE_LIKE = {"Synth": A.GEN_SYNTH, "SawTooth": A.GEN_SAWTOOTH, "Triangle": A.GEN_TRIANGLE}

# default constructors of the reference (DataSource.cpp:475-482,1079,1142,1201,1293-1295,1419-1423,1564-1568)
_DEFAULTS = {
    "Synth": dict(freq=[1., 0.3, 2., 0.5], mu=[2., 2.1, 2.2, 2.3], amp=[1., 1.2, 1.3, 1.],
                  phase=[0., 1., 2., 1.], dX=0.01, noise=0.),
    "Gaussian": dict(mean=[2., 5., 10., 15.], var=[1., 1., 2., 5.]),
    "OU": dict(mean=[2., 4.3, 3., 0.5], theta=[1., 0.3, 2., 0.5], phi=[2., 2.1, 2.2, 2.3]),
    "OUPair": dict(theta=.015, phi=.01, noise=.03),
    "SimpleTrend": dict(trend_prob=[0.001, 0.001], min_period=[100, 500], max_period=[200, 1500],
                        noise=[1., 0.1], start=[10., 15.], dYMin=[0.001, 0.01], dYMax=[0.003, 0.03]),
    "TrendOU": dict(trend_prob=[0.001, 0.001], min_period=[100, 500], max_period=[200, 1500],
                    dYMin=[0.001, 0.01], dYMax=[0.003, 0.03], start=[10., 15.], theta=[1., 0.5],
                    phi=[2., 2.1], noise_trend=[1., 1.2], ema_alpha=[0.1, 0.2]),
}
_DEFAULTS["SineAdder"] = _DEFAULTS["Synth"]  # DataSource.cpp:581-588 (one asset, four components)
# DataSource.cpp:677-687, :850-862.  The reference's default constructors pass the still-zero member dX, so
# sampleRate = (int)(1/0); its config fallback uses dX = 0.01, which is what these defaults use (noise 1).
_DEFAULTS["SineDynamic"] = dict(freqRange=[[.1, 1., .01], [0.3, 3.0, .01], [5., 15., .1], [10., 50., .1]],
                                muRange=[[1., 5., .02], [.3, 3., .05], [.2, 5., .02], [.5, 5., .02]],
                                ampRange=[[1., 5., .01], [.3, 3., .02], [.2, 2., .04], [.5, 5., .05]],
                                dX=0.01, noise=1.)
_DEFAULTS["SineDynamicTrend"] = dict(_DEFAULTS["SineDynamic"], trendRange=[[100, 500], [100, 300]],
                                     trendIncr=[0.1, 0.2], trendProb=[.001, .01])
_DEFAULTS["SawTooth"] = _DEFAULTS["Synth"]
_DEFAULTS["Triangle"] = _DEFAULTS["Synth"]
_DEFAULTS["TrendyOU"] = _DEFAULTS["TrendOU"]

_ALIASES = {"trendProb": "trend_prob", "minPeriod": "min_period", "maxPeriod": "max_period",
            "noiseTrend": "noise_trend", "emaAlpha": "ema_alpha"}

SUPPORTED = tuple(_DEFAULTS) + ("Composite",)


def _get(cfg, key):
    for k in (key,) + tuple(a for a, s in _ALIASES.items() if s == key):
        if k in cfg:
            return cfg[k]
    raise ConfigError(f"data_source_config is missing required key: {key}")


def _vec(cfg, key, n=None):
    v = _get(cfg, key)
    v = [float(x) for x in (v if isinstance(v, (list, tuple)) else list(v))]
    return v


def _same_len(kind, *vecs):
    if len({len(v) for v in vecs}) != 1:
        # std::length_error -> ValueError (DataSource.cpp:487-494,1133-1136,1279-1282)
        raise ValueError(f"parameters passed to DataSource of type {kind} need to be vectors of same length")
    return len(vecs[0])


class _Table:
    def __init__(self):
        self.assets = []   # list of dicts (type, role, nslot, nslot_aux, uslot, gslot, partner, p)
        self.names = []
        self.n_gstate = 0
        self.n_normals = 0
        self.n_uniforms = 0
        self.ext = []      # MdgParams.gen_ext: parameter / wave tables of the SINE* generators
        self._wave = {}    # table length -> offset of its samples in ext

    def wave_table(self, length):
        """offset of sin(i 2 pi / length), i = 0..length (last = first), WaveTableOsc.h:113-157"""
        if length not in self._wave:
            self._wave[length] = len(self.ext)
            tab = [math.sin(float(i) * 2. * math.pi / length) for i in range(length)]  # libm sin, as the reference
            self.ext.extend(tab + tab[:1])
        return self._wave[length]

    def add(self, name, type_, p, n_g, role=0, aux_normal=False, uniforms=False, partner=-1, normals=1):
        rec = dict(type=type_, role=role, nslot=-1, nslot_aux=-1, uslot=-1, gslot=-1,
                   partner=partner, p=list(p) + [0.] * (A.MDG_GEN_NPARAM - len(p)))
        if aux_normal:
            rec["nslot_aux"] = self.n_normals
            self.n_normals += 1
        rec["nslot"] = self.n_normals
        self.n_normals += normals
        if uniforms:
            rec["uslot"] = self.n_uniforms
            self.n_uniforms += 4 if uniforms is True else int(uniforms)
        if n_g:
            rec["gslot"] = self.n_gstate
            self.n_gstate += n_g
        # Composite: a duplicate asset code gets "_1" appended (DataSource.cpp:427-431)
        # (a third repeat would collide again in the reference; count up instead)
        base, k = name, 0
        while name in self.names:
            k += 1
            name = f"{base}_{k}"
        self.names.append(name)
        self.assets.append(rec)
        return len(self.assets) - 1


def _add_source(tab, kind, cfg):
    if cfg is None:
        if kind not in _DEFAULTS:
            raise NotImplementedError(f"Default Constructor for {kind} as dataSource is not implemented")
        cfg = _DEFAULTS[kind]
    if kind in _SINE_LIKE:  # DataSource.cpp:455-528
        freq, mu, amp, phase = (_vec(cfg, k) for k in ("freq", "mu", "amp", "phase"))
        n = _same_len(kind, freq, mu, amp, phase)
        dX = float(_get(cfg, "dX"))
        noise = float(cfg.get("noise", 0.))
        for i in range(n):
            tab.add(f"sine_{i}", _SINE_LIKE[kind], [freq[i], mu[i], amp[i], phase[i], dX, noise], 1)
    elif kind == "Gaussian":  # :1057-1104
        mean, var = _vec(cfg, "mean"), _vec(cfg, "var")
        for i in range(_same_len(kind, mean, var)):
            tab.add(f"Gaussian_{i}", A.GEN_GAUSSIAN, [mean[i], var[i]], 0)
    elif kind == "OU":  # :1118-1169
        mean, theta, phi = _vec(cfg, "mean"), _vec(cfg, "theta"), _vec(cfg, "phi")
        for i in range(_same_len(kind, mean, theta, phi)):
            tab.add(f"OU_{i}", A.GEN_OU, [mean[i], theta[i], phi[i]], 0)
    elif kind == "OUPair":  # :1183-1228
        p = [float(_get(cfg, "theta")), float(_get(cfg, "phi")), float(_get(cfg, "noise"))]
        first = tab.add("OUPair_0", A.GEN_OUPAIR, p, 1, role=0, aux_normal=True)
        tab.add("OUPair_1", A.GEN_OUPAIR, p, 0, role=1, partner=first)
    elif kind == "SimpleTrend":  # :1249-1319
        v = [_vec(cfg, k) for k in ("trend_prob", "min_period", "max_period", "noise", "start",
                                    "dYMin", "dYMax")]
        for i in range(_same_len(kind, *v)):
            tab.add(f"SimpleTrend_{i}", A.GEN_SIMPLETREND, [x[i] for x in v], 2, uniforms=True)
    elif kind in ("TrendOU", "TrendyOU"):  # :1364-1452, :1506-1597
        v = [_vec(cfg, k) for k in ("trend_prob", "min_period", "max_period", "dYMin", "dYMax",
                                    "start", "theta", "phi", "noise_trend", "ema_alpha")]
        t, ng = (A.GEN_TRENDOU, 3) if kind == "TrendOU" else (A.GEN_TRENDYOU, 4)
        for i in range(_same_len(kind, *v)):
            tab.add(f"{kind}_{i}", t, [x[i] for x in v], ng, uniforms=True)
    elif kind == "SineAdder":  # :590-661: ONE asset, the sum of the components
        freq, mu, amp, phase = (_vec(cfg, k) for k in ("freq", "mu", "amp", "phase"))
        K = _same_len(kind, freq, mu, amp, phase)
        _check_components(kind, K)
        off = len(tab.ext)
        for c in range(K):
            tab.ext.extend([freq[c], mu[c], amp[c], phase[c]])
        tab.add("multi_sine", A.GEN_SINEADDER, [K, off, float(_get(cfg, "dX")), float(cfg.get("noise", 0.))], K,
                normals=K)
    elif kind in ("SineDynamic", "SineDynamicTrend"):  # :689-780, :864-989
        _add_sine_dynamic(tab, kind, cfg)
    else:
        # NotImplemented is a std::logic_error -> RuntimeError (DataSource.cpp:101-107)
        raise NotImplementedError(f"Constructor from config for {kind} as dataSource is not implemented")


def _check_components(kind, K):
    if not 1 <= K <= A.MDG_MAX_SINE_COMPONENTS:
        raise ValueError(f"{kind}: {K} components, supported 1..{A.MDG_MAX_SINE_COMPONENTS}")


def _ranges(cfg, key, width, cast=float):
    v = _get(cfg, key)
    out = [[cast(x) for x in row] for row in v]
    if any(len(r) != width for r in out):
        raise ValueError(f"{key}: every entry needs {width} values")
    return out


def _add_sine_dynamic(tab, kind, cfg):
    """SineDynamic / SineDynamicTrend::initParams (DataSource.cpp:741-780, :938-989) and setSineOsc
    (WaveTableOsc.h:126-157): per component the (lo, hi, step) ranges and the list of wave tables."""
    trend = kind == "SineDynamicTrend"
    fr, mr, ar = (_ranges(cfg, k, 3) for k in ("freqRange", "muRange", "ampRange"))
    K = _same_len(kind, fr, mr, ar)
    _check_components(kind, K)
    dX = float(_get(cfg, "dX"))
    noise = float(_get(cfg, "noise") if trend else cfg.get("noise", 0.))
    if not dX > 0.:
        raise ValueError(f"{kind}: dX must be > 0")
    sample_rate = int(1. / dX)
    recs = []
    for c in range(K):
        lo, hi = fr[c][0], fr[c][1]
        if hi * 2 > sample_rate:  # std::logic_error -> RuntimeError (:758-765)
            raise RuntimeError("Sampling Rate as determined by 1 / dX must be at least the nyquist sampling rate "
                               f"relative to the largest frequency. freqRange entry #{c} with range of {lo} - {hi} "
                               "doesn't satisfy this constraint.")
        if not lo > 0.:
            raise ValueError(f"{kind}: freqRange low must be > 0")
        max_harms = int(sample_rate / (3.0 * lo) + 0.5)
        if max_harms < 1:
            raise ValueError(f"{kind}: freqRange low {lo} too high for sampleRate {sample_rate} (no wave table)")
        v = 1 << (max_harms - 1).bit_length()  # next power of two
        table_len, top = v * 2 * 2, lo * 2. / sample_rate  # overSample = 2
        tables = []
        while max_harms >= 1:
            tables.append((top, table_len))
            if table_len > 99999:  # constantRatioLimit
                table_len >>= 1
            top *= 2
            max_harms >>= 1
        tables = tables[:32]  # WaveTableOsc's default maxWaveTables (the oscillators are default-constructed, :756)
        recs.append(tables)
    # layout: [K component records of 12][per component: table list of 3 per table][trend list][samples ...]
    off = len(tab.ext)
    tab.ext.extend([0.] * (12 * K))
    for c in range(K):
        tl_off = len(tab.ext)
        tab.ext.extend([0.] * (3 * len(recs[c])))
        for t, (top, ln) in enumerate(recs[c]):
            tab.ext[tl_off + 3 * t: tl_off + 3 * t + 3] = [top, float(ln), float(tab.wave_table(ln))]
        tab.ext[off + 12 * c: off + 12 * c + 12] = fr[c] + mr[c] + ar[c] + [float(len(recs[c])), float(tl_off), 0.]
    p = [K, off, float(sample_rate), noise]
    n_g, n_u = 4 * K, 1
    if trend:
        tr = _ranges(cfg, "trendRange", 2, int)
        incr, prob = _vec(cfg, "trendIncr"), _vec(cfg, "trendProb")
        T = _same_len(kind, tr, incr, prob)
        if T > A.MDG_MAX_SINE_TRENDS:
            raise ValueError(f"{kind}: {T} trends, supported 0..{A.MDG_MAX_SINE_TRENDS}")
        t_off = len(tab.ext)
        for j in range(T):
            tab.ext.extend([float(tr[j][0]), float(tr[j][1]), incr[j], prob[j]])
        p += [T, t_off]
        n_g, n_u = 4 * K + 1 + T, 1 + 2 * T
    tab.add("sine_dynamic_trend" if trend else "sine_dynamic",
            A.GEN_SINEDYNAMICTREND if trend else A.GEN_SINEDYNAMIC, p, n_g, uniforms=n_u)


def build_generator_table(data_source_type, data_source_config=None, with_ext=False):
    """Returns (asset_names, list-of-asset-records, n_gstate, n_normals, n_uniforms[, gen_ext list])."""
    tab = _Table()
    if data_source_type == "Composite":  # DataSource.cpp:411-437, Config.cpp:107-126
        if not data_source_config:
            raise ConfigError("config passed but doesn't contain generator params")
        for _label, sub in data_source_config.items():
            subs = sub if isinstance(sub, (list, tuple)) else [sub]
            for s in subs:
                kind = s["data_source_type"]
                reps = int(s.get("repeat", 1))
                for _ in range(reps):
                    _add_source(tab, kind, s.get("data_source_config"))
    else:
        _add_source(tab, data_source_type, data_source_config)
    if not tab.assets:
        raise ConfigError("data source has no assets")
    if len(tab.assets) > A.MDG_MAX_ASSETS:
        raise ValueError(f"{len(tab.assets)} assets > MDG_MAX_ASSETS={A.MDG_MAX_ASSETS} "
                         "(thread-per-env kernels keep the whole portfolio in registers)")
    out = (tab.names, tab.assets, tab.n_gstate, tab.n_normals, tab.n_uniforms)
    return out + (tab.ext,) if with_ext else out


# Reference key name of every p[] slot per generator type, in the order _add_source fills them (include/madigan_b200.h
# lists the same slots).  Parameter sets (make_param_table) can vary every one of them.
PARAM_SLOTS = {
    "Synth": ("freq", "mu", "amp", "phase", "dX", "noise"),
    "SawTooth": ("freq", "mu", "amp", "phase", "dX", "noise"),
    "Triangle": ("freq", "mu", "amp", "phase", "dX", "noise"),
    "Gaussian": ("mean", "var"),
    "OU": ("mean", "theta", "phi"),
    "OUPair": ("theta", "phi", "noise"),
    "SimpleTrend": ("trend_prob", "min_period", "max_period", "noise", "start", "dYMin", "dYMax"),
    "TrendOU": ("trend_prob", "min_period", "max_period", "dYMin", "dYMax", "start", "theta", "phi", "noise_trend",
                "ema_alpha"),
    "TrendyOU": ("trend_prob", "min_period", "max_period", "dYMin", "dYMax", "start", "theta", "phi", "noise_trend",
                 "ema_alpha"),
}
_SINE_TYPES = (A.GEN_SINEADDER, A.GEN_SINEDYNAMIC, A.GEN_SINEDYNAMICTREND)
_STRUCTURE = ("type", "role", "nslot", "nslot_aux", "uslot", "gslot", "partner")


def make_param_table(data_source_type, base_config, set_configs):
    """Generator parameter table of a multi-set ``Env``: a ``(nA, MDG_GEN_NPARAM, S)`` float64 array whose
    ``[:, :, s]`` holds the ``p`` slots of every asset built from ``set_configs[s]`` (set-minor, the layout of
    ``MdgParamSets.p``).  Every set must describe the same assets as ``base_config``: same names, types, roles and
    noise / uniform / state slots; only the parameter values may differ.  SINE* sources are not supported (their slots
    are component counts and table offsets).  Raises ValueError naming the first asset that breaks either rule."""
    names, base, n_g, n_n, n_u = build_generator_table(data_source_type, base_config)
    for i, rec in enumerate(base):
        if rec["type"] in _SINE_TYPES:
            raise ValueError(f"asset {i} ({names[i]}): SINE* sources do not support parameter sets")
    set_configs = list(set_configs)
    if not set_configs:
        raise ValueError("parameter sets: need at least one set")
    table = np.empty((len(base), A.MDG_GEN_NPARAM, len(set_configs)), dtype=np.float64)
    built = {}  # one build per distinct config object (an int S passes the base config S times)
    for s, cfg in enumerate(set_configs):
        if id(cfg) not in built:
            built[id(cfg)] = build_generator_table(data_source_type, cfg)
        names_s, recs, n_g_s, n_n_s, n_u_s = built[id(cfg)]
        for i in range(max(len(base), len(recs))):
            if i >= len(recs) or i >= len(base):
                name = names[i] if i < len(base) else names_s[i]
                raise ValueError(f"parameter set {s}: asset {i} ({name}) is not in both the base and the set")
            if names_s[i] != names[i]:
                raise ValueError(f"parameter set {s}: asset {i} is {names_s[i]}, the base has {names[i]}")
            for key in _STRUCTURE:
                if recs[i][key] != base[i][key]:
                    raise ValueError(f"parameter set {s}: asset {i} ({names[i]}) differs from the base in {key}")
        if (n_g_s, n_n_s, n_u_s) != (n_g, n_n, n_u):  # implied by the slots above; kept as a guard on the builder
            raise ValueError(f"parameter set {s}: generator state / noise rows differ from the base")
        table[:, :, s] = [r["p"] for r in recs]
    return table


# The broker settings a broker set holds, in MdgParams field order (the rows of the broker table, MdgBrokerSlot); the
# names are make_env's config keys
BROKER_SLOTS = ("init_cash", "required_margin", "maintenance_margin", "slippage_rel", "slippage_abs",
                "transaction_cost_rel", "transaction_cost_abs")


def _broker_values(d, what):
    for key, v in d.items():
        if key not in BROKER_SLOTS:
            raise ValueError(f"{what}: unknown broker setting {key!r} (known: {', '.join(BROKER_SLOTS)})")
        if isinstance(v, bool) or not isinstance(v, numbers.Real):
            raise ValueError(f"{what}: {key} must be a number, got {v!r}")
    return d


def make_broker_table(base, set_dicts):
    """Broker table of an ``Env`` with broker sets: a ``(MDG_BROKER_NPARAM, S)`` float64 array whose column s holds the
    seven ``BROKER_SLOTS`` of ``set_dicts[s]`` (set-minor, the layout the ``_sets_broker`` launches read).  ``base``
    maps every slot to its base value; a key a set omits takes the base value.  An unknown key or a value that is not a
    real number raises ValueError.  Values are not range-checked (the setters do not check them either)."""
    base = _broker_values(dict(base), "base")
    missing = [k for k in BROKER_SLOTS if k not in base]
    if missing:
        raise ValueError(f"base: missing broker settings {missing}")
    set_dicts = list(set_dicts)
    if not set_dicts:
        raise ValueError("broker sets: need at least one set")
    table = np.empty((A.MDG_BROKER_NPARAM, len(set_dicts)), dtype=np.float64)
    for s, d in enumerate(set_dicts):
        d = _broker_values(dict(d or {}), f"broker set {s}")
        table[:, s] = [float(d.get(k, base[k])) for k in BROKER_SLOTS]
    return table


def make_params(data_source_type, data_source_config=None, init_cash=1_000_000.,
                required_margin=0., maintenance_margin=0., slippage_rel=0., slippage_abs=0.,
                transaction_cost_rel=0., transaction_cost_abs=0.):
    """Fill an ``MdgParams``.  Margin/cost defaults are Env's (0, Env.h:131-136), not Portfolio's."""
    names, assets, n_g, n_n, n_u, ext = build_generator_table(data_source_type, data_source_config, with_ext=True)
    P = A.MdgParams()
    # SINE* sources: parameter / wave tables.  gen_ext (a DEVICE pointer) is set by the env after the upload.
    P.ext_host = np.asarray(ext, dtype=np.float64) if ext else None
    P.gen_ext, P.n_gen_ext = None, len(ext)
    P.n_assets, P.n_gstate, P.n_normals, P.n_uniforms = len(assets), n_g, n_n, n_u
    P.init_cash = float(init_cash)
    P.required_margin = float(required_margin)
    P.maintenance_margin = float(maintenance_margin)
    P.slippage_rel, P.slippage_abs = float(slippage_rel), float(slippage_abs)
    P.tcost_rel, P.tcost_abs = float(transaction_cost_rel), float(transaction_cost_abs)
    for i, rec in enumerate(assets):
        g = P.gen[i]
        for k in ("type", "role", "nslot", "nslot_aux", "uslot", "gslot", "partner"):
            setattr(g, k, rec[k])
        for j, v in enumerate(rec["p"]):
            g.p[j] = v
    return P, names


_SHAPERS = {None: A.SHAPER_SUM, "None": A.SHAPER_SUM, "none": A.SHAPER_SUM,
            "sum_default": A.SHAPER_SUM, "DSR": A.SHAPER_DSR, "DDR": A.SHAPER_DDR,
            "cosine": A.SHAPER_COSINE, "cosine_similarity": A.SHAPER_COSINE,
            "cosine_port_shaper": A.SHAPER_COSINE, "sharpe_shaper": A.SHAPER_SHARPE,
            "sortino_shaperA": A.SHAPER_SORTINO_A, "sortino_shaperB": A.SHAPER_SORTINO_B}


def make_reward(reward_shaper_config=None, nstep_return=1, discount=0.99, reduce_rewards=False,
                n_assets=1, enabled=True):
    """``MdgReward`` from the keys ``NStepBuffer.make_reward_shaper`` reads
    (reference: utils/buffers/nstep_buffer.py:378-408) plus the agent's nstep/discount."""
    R = A.MdgReward()
    R.nstep = max(1, int(nstep_return))
    R.discount = float(discount)
    R.reduce_rewards = int(bool(reduce_rewards))
    if R.nstep > A.MDG_MAX_NSTEP:
        raise ValueError(f"nstep_return {R.nstep} > MDG_MAX_NSTEP={A.MDG_MAX_NSTEP}")
    for i in range(R.nstep):  # NStepBuffer.__init__, nstep_buffer.py:330
        R.discounts[i] = math.pow(R.discount, i)
    if not enabled:
        R.shaper = A.SHAPER_OFF
        return R
    cfg = reward_shaper_config or {"reward_shaper": None}
    kind = cfg.get("reward_shaper")
    if kind not in _SHAPERS:
        raise NotImplementedError(f"Reward Shaper type {kind} not implemented")
    R.shaper = _SHAPERS[kind]
    if R.nstep > A.MDG_MAX_NSTEP:
        raise ValueError(f"nstep_return {R.nstep} > MDG_MAX_NSTEP={A.MDG_MAX_NSTEP}")
    if R.shaper in (A.SHAPER_DSR, A.SHAPER_DDR):
        R.adaptation_rate = float(cfg["adaptation_rate"])
    if R.shaper == A.SHAPER_COSINE:
        desired = [float(x) for x in cfg["desired_portfolio"]]
        if len(desired) != n_assets + 1:
            raise ValueError("desired_portfolio must have n_assets+1 weights (cash first)")
        for j, v in enumerate(desired):
            R.desired_portfolio[j] = v
        R.cosine_temp = float(cfg["cosine_temp"])
    if R.shaper in (A.SHAPER_SORTINO_A, A.SHAPER_SORTINO_B):
        R.sortino_exp = float(cfg["sortino_exp"])
    return R
