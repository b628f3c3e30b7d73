"""The window normalisers' reductions in numpy's order, on every path that normalises a window: the register kernel,
the TMA kernel, the dilated column blocks of MultiStackerDiscrete and the replay row store's gather.

numpy sums a column of a (k, F>1) array row by row, left to right, and a (k, 1) array pairwise (``pairwise_sum``:
eight accumulators up to 128 rows, halves above).  Where the result depends on rounding -- above all a flat column,
whose mean is the constant exactly in one order and an ulp off in another -- the kernels must follow it: a flat column
normalises to 0 when numpy's mean is exact and to about +-1 when it is not.  The CPU part restates the order and finds
the flat constants that tell the orders apart; the GPU part plants them."""
import functools
import warnings

import numpy as np
import pytest
import torch

from oracle import py_oracle

NORMS = [None, "lookback", "lookback_log", "log", "standard_normal", "log_standard_normal", "expanding"]
LONG_K = (129, 136, 200, 256, 300, 513)


# ------------------------------------------------------------------------------------------------ numpy's order
def _left_to_right(v):
    s = v[0]
    for x in v[1:]:
        s = s + x
    return s


def _block8(v):
    """numpy's pairwise block: eight interleaved accumulators (any n >= 8; numpy uses it for n <= 128)."""
    n = len(v)
    if n < 8:
        return _left_to_right(v)
    r = list(v[:8])
    i = 8
    while i < n - n % 8:
        for j in range(8):
            r[j] = r[j] + v[i + j]
        i += 8
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for x in v[i:]:
        res = res + x
    return res


def _pairwise(v):
    """numpy's pairwise_sum of a 1-D float64 array."""
    n = len(v)
    if n <= 128:
        return _block8(v)
    n2 = n // 2 - (n // 2) % 8
    return _pairwise(v[:n2]) + _pairwise(v[n2:])


def _halving_walk(v):
    """The kernel's iterative form of the n > 128 case (mdg_window_norm.cuh col_sum_halving), statement for statement."""
    n, left, path, d = len(v), [0.] * 25, 0, 0
    while True:
        s, m = 0, n
        for i in range(d):
            h = m // 2 - (m // 2) % 8
            if (path >> i) & 1:
                s, m = s + h, m - h
            else:
                m = h
        while m > 128:
            m, d = m // 2 - (m // 2) % 8, d + 1
        x = _block8(v[s:s + m])
        while d > 0 and (path >> (d - 1)) & 1:
            d -= 1
            path &= ~(1 << d)
            x = left[d] + x
        if d == 0:
            return x
        left[d - 1] = x
        path |= 1 << (d - 1)


ORDERS = {"left_to_right": _left_to_right, "block8": _block8, "pairwise": _pairwise}


def numpy_order_sum(x):
    """x.sum(0) of a (n, F) float64 array, restated: rows left to right for F > 1, pairwise for F == 1."""
    x = np.asarray(x, dtype=np.float64)
    if x.shape[1] > 1:
        return _left_to_right(list(x))
    return np.array([_pairwise(list(x[:, 0]))])


def restated_stats(x):
    """(mean, std, nanmean, nanstd) over axis 0 in the restated order."""
    n = x.shape[0]
    mean = numpy_order_sum(x) / n
    std = np.sqrt(numpy_order_sum((x - mean) * (x - mean)) / n)
    ok = ~np.isnan(x)
    cnt = ok.sum(0)
    z = np.where(ok, x, 0.)
    with np.errstate(all="ignore"):
        nmean = numpy_order_sum(z) / cnt
        d = np.where(ok, z - nmean, 0.)
        nstd = np.sqrt(numpy_order_sum(d * d) / cnt)
    return mean, std, nmean, nstd


def flat_standard_normal(c, n, order):
    """standard_normal of a flat column of n values c when both of its sums run in `order`."""
    f = ORDERS[order]
    mean = f([c] * n) / n
    d = c - mean
    with np.errstate(all="ignore"):
        return np.nan_to_num(d / np.sqrt(f([d * d] * n) / n))


def discriminates(c, n, numpy_order="pairwise"):
    """c, planted as a flat column of n rows, normalises differently (by more than any test tolerance) in numpy's order
    than in every other order: left to right, eight accumulators without halving, or pairwise where numpy adds left
    to right."""
    want = flat_standard_normal(c, n, numpy_order)
    if numpy_order == "pairwise":
        wrong = ["left_to_right"] + (["block8"] if n > 128 else [])  # up to 128 rows block8 is numpy's order
    else:
        wrong = ["pairwise"]
    return all(abs(flat_standard_normal(c, n, o) - want) > .5 for o in wrong)


@functools.lru_cache(maxsize=None)
def flat_constants(n, count=3, numpy_order="pairwise"):
    """The first `count` constants of a fixed candidate list that discriminate at window length n (ValueError when
    none does: the flat-column checks would be vacuous)."""
    rng = np.random.default_rng(n)
    cands = [.1, .3, .7, 1.1, 2.3, 3.7, 10.1] + list(np.round(rng.uniform(.05, 50., 400), 3))
    out = [float(c) for c in cands if discriminates(float(c), n, numpy_order)][:count]
    if not out:
        raise ValueError(f"no discriminating constant for n={n}")
    return tuple(out)


# ------------------------------------------------------------------------------------------------ CPU
def _sampled_lengths():
    rng = np.random.default_rng(0)
    return sorted(set(range(1, 140)) | {255, 256, 257, 263, 300, 513, 1024, 1100} | set(rng.integers(140, 1100, 40)))


@pytest.mark.parametrize("F", [1, 2, 3, 16])
def test_restated_order_equals_numpy_bit_for_bit(F):
    rng = np.random.default_rng(F)
    for n in _sampled_lengths():
        x = rng.standard_normal((n, F)) * 10. ** rng.uniform(-3, 3, (n, F)) + 3.
        assert np.array_equal(numpy_order_sum(x), x.sum(0)), n
        mean, std, _, _ = restated_stats(x)
        assert np.array_equal(mean, x.mean(0)) and np.array_equal(std, x.std(0)), n
        xn = x.copy()
        xn[rng.random((n, F)) < .2] = np.nan
        if n % 5 == 0:
            xn[:, 0] = np.nan  # an all-NaN column now and then
        _, _, nmean, nstd = restated_stats(xn)
        with np.errstate(all="ignore"), warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)  # nanmean / nanstd of an all-NaN column
            np.testing.assert_array_equal(nmean, np.nanmean(xn, 0))
            np.testing.assert_array_equal(nstd, np.nanstd(xn, 0))
        if F == 1:
            assert _halving_walk(list(x[:, 0])) == _pairwise(list(x[:, 0])), n


def test_halving_walk_restates_the_recursion_up_to_large_n():
    rng = np.random.default_rng(1)
    for n in list(range(129, 1200, 7)) + [4096, 9000, 12800]:
        v = list(rng.standard_normal(n) + .1)
        assert _halving_walk(v) == _pairwise(v) == np.sum(np.asarray(v)), n


GPU_LENGTHS = sorted({7, 16, 64, 130} | set(LONG_K))


@pytest.mark.parametrize("n", GPU_LENGTHS)
def test_flat_constants_discriminate(n):
    """Every window length the GPU tests plant flat columns at (but n < 8, where every order is the same) has constants
    whose numpy result differs from the result in each wrong order; numpy itself confirms the planted outcome."""
    if n < 8:
        assert not any(discriminates(c, n) for c in (.1, .3, .7, 1.1))
        return
    for numpy_order in ("pairwise", "left_to_right"):
        cs = flat_constants(n, numpy_order=numpy_order)
        assert cs
        for c in cs:
            col = np.full((n, 1), c) if numpy_order == "pairwise" else np.stack([np.full(n, c), np.arange(n) + 1.], 1)
            want = py_oracle.normalise(col, "standard_normal")[:, 0]
            assert np.all(want == flat_standard_normal(c, n, numpy_order)), (n, c)


# ------------------------------------------------------------------------------------------------ GPU helpers
def _env(n_envs, n_feats, k, seed=3):
    from test_gpu_window import make_env
    return make_env(n_envs, n_feats, k)


def _load(env, rows):
    from test_gpu_window import load_ring
    load_ring(env, rows, rows.shape[0] - 1)


def _path(monkeypatch, path):
    monkeypatch.setenv("MDG_WIN_TMA", "1" if path == "tma" else "0")
    monkeypatch.setenv("MDG_WIN_TMA_E", "16")
    monkeypatch.setenv("MDG_WIN_TMA_FT", "1")


def _log_standard_normal_from(L):
    """log_standard_normal of windows whose logs are L (N, k, F): the reference's nanmean / nanstd in numpy."""
    with np.errstate(all="ignore"):
        return np.stack([np.nan_to_num((w - np.nanmean(w, 0)) / np.nanstd(w, 0), 0.) for w in L])


def _reference(raw, norm, kernel_logs=None, transform=None):
    """numpy of the raw windows (N, k, F); log_standard_normal from the kernel's own logs where given (fast_log and
    np.log may differ by an ulp, and a flat column's outcome hinges on its exact value)."""
    if norm == "log_standard_normal" and kernel_logs is not None:
        return _log_standard_normal_from(kernel_logs)
    return np.stack([py_oracle.stack_window(w, norm, transform) for w in raw])


def _check(got64, got32, want, tag):
    np.testing.assert_allclose(got64, want, rtol=1e-9, atol=1e-11, equal_nan=True, err_msg=str(tag))
    np.testing.assert_array_equal(got32, got64.astype(np.float32), err_msg=str(tag))  # rounded once, NaN == NaN


def _kernel_logs(env, nv, raw, transform=None, **kw):
    """The kernel's log of each window value (``log`` clamps at 1e-5; below it numpy's log stands in)."""
    from madigan_b200 import _abi as A
    xf = A.XFORM_PAIR_RATIO if transform == "pairs" else A.XFORM_NONE
    L = env.window("log", torch.float64, n_valid=nv, transform=xf, **kw).cpu().numpy()
    x = raw if transform != "pairs" else (raw[..., :1] / raw[..., 1:2])
    with np.errstate(all="ignore"):
        return np.where(x >= 1e-5, L, np.log(x))


# ------------------------------------------------------------------------------------------------ GPU: kernels
@pytest.mark.gpu
@pytest.mark.parametrize("path", ["register", "tma"])
@pytest.mark.parametrize("transform", [None, "pairs"])
@pytest.mark.parametrize("k", LONG_K)
def test_long_windows_single_column(monkeypatch, path, transform, k):
    """F = 1 (and the pair ratio, 2 features -> 1) at k > 128, full and partial windows, every normaliser, random
    columns and flat ones planted by flat_constants, including the last env of a partial block."""
    from madigan_b200 import _abi as A
    if path == "tma" and transform:
        pytest.skip("the TMA kernel takes untransformed windows only")
    N, nF = 50, (2 if transform else 1)
    rng = np.random.default_rng(k)
    rows = np.abs(10 + np.cumsum(rng.standard_normal((k + 3, nF, N)) * .2, axis=0)) + .1
    nvs = sorted({k, 130, 64, 7} - {n for n in (130,) if n >= k})
    plant = {}  # env -> constant; every length gets its own, the last env carries the full window's
    for i, nv in enumerate(n for n in nvs if n >= 8):
        for j, c in enumerate(flat_constants(nv)[:2]):
            plant[N - 1 - 2 * i - j] = c
    plant[0] = 4.0  # dyadic: exact in every order
    for e, c in plant.items():
        if transform:
            rows[:, 0, e], rows[:, 1, e] = 2. * c, 2.  # the ratio is c exactly
        else:
            rows[:, 0, e] = c
    env = _env(N, nF, k)
    _load(env, rows)
    _path(monkeypatch, path)
    xf = A.XFORM_PAIR_RATIO if transform else A.XFORM_NONE
    for nv in nvs:
        raw = rows[-nv:].transpose(2, 0, 1)
        logs = _kernel_logs(env, nv, raw, transform)
        for norm in NORMS:
            if path == "tma" and norm == "expanding":
                continue
            want = _reference(raw, norm, logs, transform)
            got64 = env.window(norm, torch.float64, n_valid=nv, transform=xf).cpu().numpy()
            got32 = env.window(norm, torch.float32, n_valid=nv, transform=xf).cpu().numpy()
            _check(got64, got32, want, (nv, norm))
            if norm == "standard_normal" and nv >= 8:  # the planted outcome is numpy's, and it is not vacuous
                for e, c in plant.items():
                    if c in flat_constants(nv):
                        assert np.all(got64[e, :, 0] == flat_standard_normal(c, nv, "pairwise")), (nv, e)


@pytest.mark.gpu
@pytest.mark.parametrize("dilations", [[1, 2], [1, 3, 5], [1]])
@pytest.mark.parametrize("norm", ["standard_normal", "log_standard_normal", "lookback", "log"])
def test_multistacker_single_feature_normalises_the_concatenation(dilations, norm):
    """One feature, several dilations: the reference normalises the (k, D) concatenation, whose columns numpy sums left
    to right; one dilation leaves a (k, 1) array, summed pairwise."""
    from madigan_b200.utils.preprocessor import MultiStackerDiscrete
    D, k = len(dilations), 200 if len(dilations) == 1 else 64
    order = "pairwise" if D == 1 else "left_to_right"
    ring = k * max(dilations) + 2
    N = 24
    rng = np.random.default_rng(D)
    rows = np.abs(10 + np.cumsum(rng.standard_normal((ring + 5, 1, N)) * .2, axis=0)) + .1
    cs = flat_constants(k, count=6, numpy_order=order)
    for i, c in enumerate(cs):
        rows[:, 0, N - 1 - i] = c
    env = _env(N, 1, ring)
    _load(env, rows)
    st = MultiStackerDiscrete(k, dilations, 1, norm=True, norm_type=norm)
    st._bind(env)
    st._count = k * max(dilations) + 7
    got = st.current_data().price.cpu().numpy()
    R = rows.shape[0]
    cols = []
    for d in dilations:
        age0 = (st._count - 1) % d
        ages = age0 + (k - 1 - np.arange(k)) * d
        cols.append(rows[R - 1 - ages, 0, :].T)  # (N, k)
    raw = np.stack(cols, axis=2)  # (N, k, D)
    logs = None
    if norm == "log_standard_normal":
        L = env.window("log", torch.float64, n_valid=ring).cpu().numpy()[:, :, 0]  # kernel logs of the ring, oldest first
        logs = np.stack([L[:, ring - 1 - ((st._count - 1) % d + (k - 1 - np.arange(k)) * d)] for d in dilations], 2)
    want = _reference(raw, norm, logs)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-11, equal_nan=True)
    if norm == "standard_normal":
        for i, c in enumerate(cs):
            assert np.all(got[N - 1 - i] == flat_standard_normal(c, k, order)), c


@pytest.mark.gpu
@pytest.mark.parametrize("nF", [1, 3])
def test_dilated_windows_after_masked_resets(nF):
    """stride > 1 and age0 > 0 on envs that reset with fill_history: the rows older than a reset come from the prefix
    buffer at pbase - age * F.  Rows are picked from the full window, which the parity tests tie to the oracle."""
    from madigan_b200.environments import Env
    k, N = 40, 36
    cfg = {"data_source_config": {"mean": [10.] * nF, "theta": [.1] * nF, "phi": [.05] * nF}}
    env = Env("OU", 1e6, cfg, n_envs=N, window=k, seed=11, device="cuda")
    env.reset(fill_history=True)
    u = torch.zeros((N, nF), dtype=torch.float64, device="cuda")
    for t in range(12):
        env.step(u)
        if t in (3, 8):
            m = torch.zeros(N, dtype=torch.bool, device="cuda")
            m[t % 3::3] = True
            env.reset(mask=m, fill_history=True)
    assert env.n_valid == k
    full = env.window(None, torch.float64, n_valid=k).cpu().numpy()
    port = env.portfolio_window(k).cpu().numpy()
    for nv, stride, age0 in ((13, 3, 1), (10, 4, 2), (20, 2, 0), (8, 5, 4), (39, 1, 1)):
        idx = k - 1 - (age0 + (nv - 1 - np.arange(nv)) * stride)
        raw = full[:, idx]
        np.testing.assert_array_equal(env.portfolio_window(nv, stride=stride, age0=age0).cpu().numpy(), port[:, idx])
        for norm in NORMS:
            got = env.window(norm, torch.float64, n_valid=nv, stride=stride, age0=age0).cpu().numpy()
            np.testing.assert_allclose(got, _reference(raw, norm), rtol=1e-9, atol=1e-11, equal_nan=True,
                                       err_msg=str((nv, stride, age0, norm)))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["register", "tma"])
@pytest.mark.parametrize("k", [64, 200])
def test_degenerate_values(monkeypatch, path, k):
    """Zero last values (inf / NaN from lookback*), zeros, negatives and values below 1e-5 (the log clamp; NaN and -inf
    in log_standard_normal), a column that is all NaN after log, flat dyadic and non-dyadic columns, 1e300: the inf and
    NaN positions and the values match numpy."""
    N = 32
    rng = np.random.default_rng(k + 1)
    rows = np.abs(10 + np.cumsum(rng.standard_normal((k + 2, 1, N)) * .2, axis=0)) + .1
    col = lambda e: rows[:, 0, e]
    col(0)[-1] = 0.                                   # last value 0
    col(1)[::7] = 0.                                  # zeros inside
    col(2)[1::5] *= -1.                               # negatives
    col(3)[::3] = rng.uniform(1e-12, 1e-5, len(col(3)[::3]))  # below the log clamp
    col(4)[:] = -np.abs(col(4))                       # every log NaN: log_standard_normal gives 0
    col(5)[:] = 0.5                                   # dyadic flat
    col(6)[:] = flat_constants(k)[0]                  # non-dyadic flat, numpy's mean decides
    col(7)[:] *= 1e300                                # near the top of the range
    col(8)[:] = 0.                                    # all zeros
    col(9)[:] = 1e-7                                  # flat below the clamp
    col(10)[-1] = -1.                                 # negative last value
    col(N - 1)[:] = flat_constants(k)[-1]
    env = _env(N, 1, k)
    _load(env, rows)
    _path(monkeypatch, path)
    raw = rows[-k:].transpose(2, 0, 1)
    logs = _kernel_logs(env, k, raw)
    for norm in NORMS:
        if path == "tma" and norm == "expanding":
            continue
        want = _reference(raw, norm, logs)
        got64 = env.window(norm, torch.float64).cpu().numpy()
        got32 = env.window(norm, torch.float32).cpu().numpy()
        for g, w in ((got64, want), (got32, want.astype(np.float32))):
            assert np.array_equal(np.isnan(g), np.isnan(w)), norm
            assert np.array_equal(np.isposinf(g), np.isposinf(w)) and np.array_equal(np.isneginf(g), np.isneginf(w))
        _check(got64, got32, want, norm)
        if norm == "log_standard_normal":
            assert np.all(got64[4] == 0.)


# ------------------------------------------------------------------------------------------------ GPU: row store
@pytest.mark.gpu
@pytest.mark.parametrize("source", ["flat", "ou"])
def test_row_store_long_single_asset_windows(source):
    """store="rows", one asset, k 200: each sampled state and next window against numpy normalising the raw window
    recorded for that record's step on the host, in fp64 and (rounded once) in fp32."""
    from madigan_b200.environments import Env
    from madigan_b200.utils.replay import DeviceReplay
    k, N, T = 200, 16, 24
    rw = dict(reward_shaper_config={"reward_shaper": "None"}, nstep_return=1, discount=.99, reduce_rewards=True)
    mu = flat_constants(k)[0]
    if source == "flat":
        env = Env("Synth", 1e6, {"data_source_config": {"freq": [1.], "mu": [mu], "amp": [0.], "phase": [0.],
                                                        "dX": .01, "noise": 0.}}, n_envs=N, window=k, seed=5, reward=rw)
    else:
        env = Env("OU", 1e6, {"data_source_config": {"mean": [10.], "theta": [.1], "phi": [.05]}}, n_envs=N, window=k,
                  seed=5, reward=rw)
    env.reset(fill_history=True)
    depth = T + 4  # no slot is reused: slot s holds step s, slot depth - 1 step -1
    norms = ("standard_normal", "log_standard_normal")
    bufs = {(nm, dt): DeviceReplay(env, depth=depth, norm_type=nm, dtype=dt, seed=9, store="rows")
            for nm in norms for dt in (torch.float64, torch.float32)}
    raw, logs = {}, {}

    def record(step):
        raw[step] = env.window(None, torch.float64).cpu().numpy()
        with np.errstate(all="ignore"):
            logs[step] = np.where(raw[step] >= 1e-5, env.window("log", torch.float64).cpu().numpy(), np.log(raw[step]))

    for b in bufs.values():
        b.observe_start()
    record(-1)
    if source == "flat":
        assert np.all(raw[-1] == mu)
    rng = np.random.default_rng(2)
    for t in range(T):
        a = torch.from_numpy(rng.integers(-1, 2, size=(N, 1)) * 1000.).double().cuda()
        env.step(a, auto_reset=True)
        for b in bufs.values():
            b.add(a)
        record(t)
    for nm in norms:
        b64, b32 = bufs[(nm, torch.float64)], bufs[(nm, torch.float32)]
        s64, _ = b64.sample(256)
        s32, _ = b32.sample(256)
        assert torch.equal(b64.last_idx, b32.last_idx) and bool(b64.last_valid.all())
        idx = b64.last_idx.cpu().numpy()
        te = b64.t["t_env"].cpu().numpy()[idx]
        st = b64.t["t_state_step"].cpu().numpy()[idx]
        nslot = b64.t["t_next_slot"].cpu().numpy()[idx]
        nxt = np.where(nslot == depth - 1, -1, nslot)
        for which, steps, g64, g32 in (("state", st, s64.state.price, s32.state.price),
                                       ("next", nxt, s64.next_state.price, s32.next_state.price)):
            src = logs if nm == "log_standard_normal" else raw
            win = np.stack([src[s][e] for s, e in zip(steps, te)])
            want = _log_standard_normal_from(win) if nm == "log_standard_normal" else \
                py_oracle.normalise_batch(win, nm)
            _check(g64.cpu().numpy(), g32.cpu().numpy(), want, (nm, which))
            if source == "flat" and nm == "standard_normal":
                assert np.all(g64.cpu().numpy() == flat_standard_normal(mu, k, "pairwise"))


# ------------------------------------------------------------------------------------------------ GPU: bench shape
@pytest.mark.gpu
def test_bench_shape_register_and_tma_against_numpy(monkeypatch):
    """65,536 envs x 16 assets x k 64, fp32 standard_normal after 50 auto-reset steps of the bench configuration: both
    kernels against numpy on 4,096 envs (the first and the last included)."""
    import bench
    dev = torch.device("cuda", 0)
    n = 65536
    env = bench.make_env(dev, 0, n_envs=n)
    acts = bench.synth_actions(4, n, 1, device=dev)
    for t in range(50):
        env.step(acts[t % 4], auto_reset=True)
    pick = np.unique(np.concatenate([[0, n - 1], np.random.default_rng(0).choice(n, 4094, replace=False)]))
    raw = env.window(None, torch.float64).cpu().numpy()[pick]
    want = py_oracle.normalise_batch(raw, "standard_normal")
    monkeypatch.setenv("MDG_WIN_TMA_E", "8")
    monkeypatch.setenv("MDG_WIN_TMA_FT", "16")
    for tma in ("0", "1"):
        monkeypatch.setenv("MDG_WIN_TMA", tma)
        got64 = env.window("standard_normal", torch.float64).cpu().numpy()[pick]
        got32 = env.window("standard_normal", torch.float32).cpu().numpy()[pick]
        _check(got64, got32, want, tma)
