"""GPU: the window materialiser (StackerDiscrete.current_data + the six normalisers) against
(a) vectors produced by the reference's own preprocessor (tests/golden/preprocessor.npz) and
(b) the numpy restatement on random rings, all layouts and dtypes.  Bar: 1e-9 relative in fp64;
fp32 output is the fp64 result rounded once (checked to 1e-6)."""
import os

import numpy as np
import pytest
import torch

from oracle import py_oracle
from test_window_numpy_order import flat_constants

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NORMS = [None, "lookback", "lookback_log", "log", "standard_normal", "log_standard_normal", "expanding"]


def make_env(n_envs, n_assets, window):
    from madigan_b200.environments import Env
    cfg = {"data_source_config": {"mean": [10.] * n_assets, "theta": [.1] * n_assets, "phi": [.02] * n_assets}}
    return Env("OU", 1e6, cfg, n_envs=n_envs, window=window, seed=3)


def load_ring(env, rows, newest_index):
    """rows: (R, nF, N) price rows with global indices 0..R-1; ring slot = index % k."""
    k = env.k
    R = rows.shape[0]
    for r in range(max(0, R - k), R):
        env.t["obs_price"][r % k].copy_(torch.from_numpy(np.ascontiguousarray(rows[r])))
    env.head = newest_index % k
    env.n_valid = min(k, R)
    # pretend the rows were written by steps: no row is older than the env's last reset
    env.t["reset_ts"].fill_(-(10 ** 9))


@pytest.mark.parametrize("norm", NORMS)
def test_window_matches_reference_preprocessor(norm):
    PP = np.load(os.path.join(GOLD, "preprocessor.npz"))
    prices, steps, lens = PP["prices"], PP["steps"], PP["lens"]
    ref = PP[f"out_{norm}"]
    k, nF = ref.shape[1], ref.shape[2]
    env = make_env(7, nF, k)
    for idx, (t, ln) in enumerate(zip(steps, lens)):
        rows = np.repeat(prices[:t + 1, :, None], 7, axis=2)
        load_ring(env, rows, t)
        got = env.window(norm, dtype=torch.float64).cpu().numpy()
        assert got.shape == (7, ln, nF)
        for e in range(7):
            np.testing.assert_allclose(got[e], ref[idx, :ln], rtol=1e-9, atol=1e-12, equal_nan=True)


@pytest.mark.parametrize("norm", NORMS)
@pytest.mark.parametrize("nF,k,N", [(1, 64, 1000), (2, 64, 333), (16, 64, 300), (5, 10, 65), (16, 7, 33)])
def test_window_matches_numpy_random(norm, nF, k, N):
    rng = np.random.default_rng(nF * 100 + k)
    env = make_env(N, nF, k)
    R = k + 11
    rows = np.abs(10 + np.cumsum(rng.standard_normal((R, nF, N)) * .2, axis=0)) + .1
    if k >= 8:  # a flat column whose standard_normal is 0 or ~+-1 depending on the summation order: the kernel's must be numpy's
        rows[:, 0, 0] = flat_constants(k, numpy_order="pairwise" if nF == 1 else "left_to_right")[0]
    else:  # below 8 rows every order is the same
        rows[:, 0, 0] = 3.0
    load_ring(env, rows, R - 1)
    ref = py_oracle.normalise_batch(rows[R - k:].transpose(2, 0, 1), norm)  # (N,k,nF)
    got = env.window(norm, dtype=torch.float64).cpu().numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-9, atol=1e-11, equal_nan=True)
    got_cf = env.window(norm, dtype=torch.float64, channels_first=True).cpu().numpy()
    np.testing.assert_allclose(got_cf, ref.transpose(0, 2, 1), rtol=1e-9, atol=1e-11, equal_nan=True)
    got32 = env.window(norm, dtype=torch.float32).cpu().numpy()
    np.testing.assert_allclose(got32, ref.astype(np.float32), rtol=2e-6, atol=1e-6, equal_nan=True)
    # partially filled window (fewer rows than k), oldest first
    nv = max(1, k // 3)
    ref_p = py_oracle.normalise_batch(rows[R - nv:].transpose(2, 0, 1), norm)
    got_p = env.window(norm, dtype=torch.float64, n_valid=nv).cpu().numpy()
    np.testing.assert_allclose(got_p, ref_p, rtol=1e-9, atol=1e-11, equal_nan=True)


@pytest.mark.parametrize("norm", [n for n in NORMS if n != "expanding"])
@pytest.mark.parametrize("nF,k,N,E,FT", [(16, 64, 300, 8, 16), (16, 64, 4098, 32, 4), (2, 64, 334, 16, 2), (16, 7, 34, 8, 16)])
def test_window_tma_variant_matches_numpy_and_register_path(monkeypatch, norm, nF, k, N, E, FT):
    """The opt-in TMA tile kernel (cp.async.bulk.tensor loads against an mbarrier, bulk stores; csrc/mdg_aux.cu
    window_tma_kernel) against numpy and against the default register-staged kernel, incl. rows older than a reset
    that come from the prefix buffer."""
    rng = np.random.default_rng(nF * 10 + k)
    env = make_env(N, nF, k)
    R = k + 5
    rows = np.abs(10 + np.cumsum(rng.standard_normal((R, nF, N)) * .2, axis=0)) + .1
    load_ring(env, rows, R - 1)
    ref = py_oracle.normalise_batch(rows[R - k:].transpose(2, 0, 1), norm)
    monkeypatch.setenv("MDG_WIN_TMA_E", str(E))
    monkeypatch.setenv("MDG_WIN_TMA_FT", str(FT))
    for dtype, tol in ((torch.float64, dict(rtol=1e-9, atol=1e-11)), (torch.float32, dict(rtol=2e-6, atol=1e-6))):
        monkeypatch.setenv("MDG_WIN_TMA", "1")
        got = env.window(norm, dtype=dtype).cpu().numpy()
        monkeypatch.setenv("MDG_WIN_TMA", "0")
        base = env.window(norm, dtype=dtype).cpu().numpy()
        np.testing.assert_allclose(got, ref.astype(got.dtype), equal_nan=True, **tol)
        np.testing.assert_array_equal(got, base)
    # after real steps and resets: pre-reset rows come from the prefix buffer; both kernels must agree bit for bit
    from madigan_b200.environments import Env
    env2 = Env("OU", 1e6, {"data_source_config": {"mean": [10.] * 4, "theta": [.1] * 4, "phi": [.05] * 4}}, n_envs=258,
               window=16, seed=3, device="cuda")
    env2.reset(fill_history=True)
    u = torch.zeros((258, 4), dtype=torch.float64, device="cuda")
    for t in range(9):
        env2.step(u)
        if t == 4:
            m = torch.zeros(258, dtype=torch.bool, device="cuda"); m[::3] = True
            env2.reset(mask=m, fill_history=True)
    monkeypatch.setenv("MDG_WIN_TMA_E", "8"); monkeypatch.setenv("MDG_WIN_TMA_FT", "4")
    monkeypatch.setenv("MDG_WIN_TMA", "1")
    a_ = env2.window(norm, dtype=torch.float64).cpu().numpy()
    monkeypatch.setenv("MDG_WIN_TMA", "0")
    b_ = env2.window(norm, dtype=torch.float64).cpu().numpy()
    np.testing.assert_array_equal(a_, b_)


def test_stacker_discrete_api_roundtrip():
    """The reference's agent loop (offpolicy_q.py:93-99): reset -> stream_state -> initialize_history -> current_data."""
    from madigan_b200.environments import Env
    from madigan_b200.utils.preprocessor import StackerDiscrete
    from madigan_b200.environments.data_source import make_params
    from oracle.oracle import OracleBatch
    cfg = {"data_source_config": {"theta": .015, "phi": .01, "noise": .03}}
    N, k = 50, 12
    env = Env("OUPair", 1e6, cfg, n_envs=N, window=k, seed=5)
    env.setRequiredMargin(1.)
    P, _ = make_params("OUPair", cfg["data_source_config"], required_margin=1.)
    orc = OracleBatch(N, P, None, window=k, seed=5)
    pre = StackerDiscrete(k, env.nFeats, norm=True, norm_type="lookback")
    rng = np.random.default_rng(0)
    nz = rng.standard_normal((1, 3, N))
    state = env.reset(normals=nz)
    orc.reset(fill_ticks=1, normals=nz)
    pre.reset_state()
    pre.stream_state(state)
    assert len(pre) == 1
    # initialize_history: k-1 no-action steps (here with an injected stream so both sides agree exactly)
    while len(pre) < k:
        nz = rng.standard_normal((3, N))
        s, r, d, info = env.step(normals=nz)
        orc.step(None, normals=nz)
        pre.stream_state(s)
    cd = pre.current_data()
    ref = py_oracle.normalise_batch(orc.window(), "lookback")
    np.testing.assert_allclose(cd.price.cpu().numpy(), ref, rtol=1e-9)
    assert cd.portfolio.shape == (N, k, 3) and cd.timestamp.shape == (N, k)
    np.testing.assert_array_equal(cd.timestamp.cpu().numpy(), np.tile(np.arange(2, k + 2), (N, 1)))
    np.testing.assert_allclose(cd.portfolio.cpu().numpy()[:, :, 0], 1.0)
    # one real step: the window slides by one row
    u = rng.integers(-1, 2, size=(N, 2)) * 1000.
    nz = rng.standard_normal((3, N))
    s, r, d, info = env.step(torch.from_numpy(u), normals=nz)
    orc.step(u, normals=nz)
    pre.stream_state(s)
    cd = pre.current_data()
    np.testing.assert_allclose(cd.price.cpu().numpy(), py_oracle.normalise_batch(orc.window(), "lookback"), rtol=1e-9)
    last_port = cd.portfolio[:, -1].cpu().numpy()
    np.testing.assert_allclose(last_port, orc.obs_port[orc.head].T, rtol=1e-9, atol=1e-12)



@pytest.mark.parametrize("norm", NORMS)
@pytest.mark.parametrize("name", ["pairs", "returns"])
def test_stacker_variants_match_reference(name, norm):
    """StackerDiscretePairs / StackerDiscreteReturns (preprocessor.py:295-333) against the reference's own classes
    (tests/golden/stackers.npz) and, at a larger shape, against the numpy restatement."""
    from madigan_b200 import _abi as A
    SK = np.load(os.path.join(GOLD, "stackers.npz"))
    prices, steps = SK[f"{name}_prices"], SK["steps"]
    ref = SK[f"{name}_out_{norm}"]
    k, nF = ref.shape[1], prices.shape[1]
    xf = A.XFORM_PAIR_RATIO if name == "pairs" else A.XFORM_RETURNS
    env = make_env(5, nF, k)
    for idx, t in enumerate(steps):
        load_ring(env, np.repeat(prices[:t + 1, :, None], 5, axis=2), t)
        got = env.window(norm, dtype=torch.float64, transform=xf).cpu().numpy()
        assert got.shape == (5,) + ref[idx].shape
        for e in range(5):
            np.testing.assert_allclose(got[e], ref[idx], rtol=1e-9, atol=1e-12, equal_nan=True)
    # random ring, channels-first and fp32 too
    rng = np.random.default_rng(31)
    N, k2, nF2 = 130, 64, (2 if name == "pairs" else 16)
    env = make_env(N, nF2, k2)
    R = k2 + 5
    rows = np.abs(10 + np.cumsum(rng.standard_normal((R, nF2, N)) * .2, axis=0)) + .1
    load_ring(env, rows, R - 1)
    want = np.stack([py_oracle.stack_window(w, norm, name) for w in rows[R - k2:].transpose(2, 0, 1)])
    got = env.window(norm, dtype=torch.float64, transform=xf).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-11, equal_nan=True)
    got_cf = env.window(norm, dtype=torch.float32, channels_first=True, transform=xf).cpu().numpy()
    np.testing.assert_allclose(got_cf, want.transpose(0, 2, 1).astype(np.float32), rtol=2e-6, atol=1e-6, equal_nan=True)


def test_stacker_variant_classes():
    from madigan_b200.utils.preprocessor import StackerDiscretePairs, StackerDiscreteReturns, make_preprocessor
    env = make_env(9, 2, 8)
    env.reset(fill_history=True)
    pre = make_preprocessor({"preprocessor_type": "StackerDiscretePairs",
                             "preprocessor_config": {"window_length": 8, "norm": True, "norm_type": "lookback"}}, 2)
    assert isinstance(pre, StackerDiscretePairs) and pre.feature_output_shape == (8, 1)
    pre.sync(env)
    st = pre.current_data()
    assert st.price.shape == (9, 8, 1) and st.portfolio.shape == (9, 8, 3) and st.timestamp.shape == (9, 8)
    ret = StackerDiscreteReturns(8, 2, norm=False)
    ret.sync(env)
    st = ret.current_data()
    assert st.price.shape == (9, 8, 1) and st.portfolio.shape == (9, 7, 3) and st.timestamp.shape == (9, 7)
