"""The all-OU-pairs refill (reset_fill_pairs_kernel, one lane per (env, pair)) against the generic refill
(reset_fill_kernel, forced with MDG_FLAG_GENERIC_FILL) -- bit for bit on every state and IO tensor -- and, with
free-running Philox and auto-reset, against the CPU oracle."""
import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from madigan_b200.environments.data_source import make_params, make_reward

pytestmark = pytest.mark.gpu

REWARD = dict(reward_shaper_config={"reward_shaper": "DSR", "adaptation_rate": .001}, nstep_return=1,
              discount=0.99, reduce_rewards=True)
UNIT = 5000.


def pairs(n):
    return {f"pair{i}": {"data_source_type": "OUPair",
                         "data_source_config": {"theta": .015, "phi": .01, "noise": .03}} for i in range(n)}


def make_env(n_pairs, N, k, seed, margin, env_offset=0):
    from madigan_b200.environments import Env
    env = Env("Composite", 1_000_000., {"data_source_config": pairs(n_pairs)}, n_envs=N, window=k, seed=seed,
              env_offset=env_offset, reward=REWARD)
    env.setRequiredMargin(margin)
    env.setMaintenanceMargin(.25)
    env.setTransactionCost(.02, 0.)
    env.setSlippage(.001, 0.)
    return env


def assert_same(a, b, what):
    for name, x in a.t.items():
        assert torch.equal(x, b.t[name]), f"{what}: {name} differs"


# (pairs, envs, window, required margin, units scale): the bench's shape; five pairs (no shared Philox block between
# lanes; 25 envs x 5 lanes per block, so envs straddle warps) at an env count that is not a multiple of the 25 envs of
# a block; four pairs
SHAPES = {"bench_nA16": (8, 65536, 64, .2, UNIT), "nA10_odd_n": (5, 4099, 8, .1, 20000.),
          "nA8": (4, 1000, 16, .1, 20000.)}


@pytest.mark.parametrize("shape", list(SHAPES))
def test_pairs_refill_equals_generic(shape):
    n_pairs, N, k, margin, scale = SHAPES[shape]
    fast = make_env(n_pairs, N, k, 11, margin, env_offset=3)
    ref = make_env(n_pairs, N, k, 11, margin, env_offset=3)
    ref.flags |= A.FLAG_GENERIC_FILL
    assert_same(fast, ref, "constructor")
    fast.reset(fill_history=True)  # count = N
    ref.reset(fill_history=True)
    torch.cuda.synchronize()
    assert_same(fast, ref, "full reset")
    g = torch.Generator().manual_seed(5)
    n_done = 0

    def steps(n):
        nonlocal n_done
        for t in range(n):
            u = (torch.randint(-1, 2, (N, 2 * n_pairs), generator=g).double() * scale).to(fast.device)
            fast.step(u, auto_reset=True)
            ref.step(u, auto_reset=True)
            n_done += int(ref.t["done"].sum())
            assert_same(fast, ref, f"step {t}")

    steps(25)
    mask = torch.from_numpy(np.random.default_rng(3).random(N) < .1)
    fast.reset(mask=mask, fill_history=False)  # fill 1
    ref.reset(mask=mask, fill_history=False)
    assert_same(fast, ref, "masked reset, fill 1")
    none = torch.zeros(N, dtype=torch.bool)
    fast.reset(mask=none, fill_history=True)  # count = 0: the header must come back clean
    ref.reset(mask=none, fill_history=True)
    assert_same(fast, ref, "empty reset")
    steps(25)
    assert n_done > 0, "no env finished: the auto-reset refill was not exercised"


def test_free_running_pairs_autoreset_matches_oracle():
    """The bench's configuration (8 OU pairs, DSR n=1, window 64) with Philox noise and auto-reset for 200 steps:
    ledger, risk, done and timestamps bit-exact, prices and the refilled history (pre_price, through the window)
    within 1e-9 (the normals pass through CUDA's and glibc's log / sincos)."""
    from oracle.oracle import OracleBatch
    N, k, seed, off = 4096, 64, 21, 70_000
    env = make_env(8, N, k, seed, 1., env_offset=off)
    P, _ = make_params("Composite", pairs(8), required_margin=1., maintenance_margin=.25,
                       transaction_cost_rel=.02, slippage_rel=.001)
    R = make_reward(REWARD["reward_shaper_config"], 1, .99, True, n_assets=16)
    orc = OracleBatch(N, P, R, window=k, seed=seed, env_offset=off)
    orc.reset(fill_ticks=1, clear_nstep=False)  # the constructor's tick
    env.reset(fill_history=True)
    orc.reset(fill_ticks=k)
    rng = np.random.default_rng(9)
    n_done = 0
    for t in range(200):
        units = rng.integers(-1, 2, size=(N, 16)).astype(np.float64) * UNIT
        ts_before = env.t["reset_ts"].cpu().numpy()
        env.step(torch.from_numpy(units), auto_reset=True)
        orc.step(units)
        done = orc.done.astype(bool)
        assert np.array_equal(env.t["done"].cpu().numpy(), done), f"step {t} done"
        assert np.array_equal(env.t["risk"].cpu().numpy(), orc.risk), f"step {t} risk"
        if done.any():  # the CUDA side has already refilled these envs
            orc.reset(mask=orc.done.copy(), fill_ticks=k)
        n_done += int(done.sum())
        st = orc.state()
        assert np.array_equal(env.t["ledger"].cpu().numpy(), st["ledger"]), f"step {t} ledger"
        ts = env.t["timestamp"].cpu().numpy()
        assert np.array_equal(ts, st["timestamp"]), f"step {t} timestamp"
        rts = env.t["reset_ts"].cpu().numpy()
        assert np.array_equal(rts[done], ts[done]) and np.array_equal(rts[~done], ts_before[~done]), f"step {t} reset_ts"
        np.testing.assert_allclose(env.t["price"].cpu().numpy(), st["price"], rtol=1e-9, atol=0)
        if t % 20 == 19 or t == 199:
            w = env.window(None, dtype=torch.float64).cpu().numpy()
            np.testing.assert_allclose(w, orc.window(), rtol=1e-9, atol=0, err_msg=f"step {t} window")
    assert n_done > 50, f"only {n_done} envs finished in 200 steps"
