"""Per-episode set draw: every reset of an env draws its parameter set on the device (param_set_weights).

The contract: the draw of env e at a reset is a function of (seed, global env id, the env's timestamp before the refill,
cdf) only -- oracle/set_draw_oracle.py restates it -- and the new episode then runs exactly as if the set had been
assigned on the host before a masked reset.  The GPU tests drive an Env with the draw and auto-reset next to an Env
without it that follows the manual recipe (step, assign_param_sets(restated ids, mask=done), reset(mask=done,
fill_history=True)) and compare them bit for bit.  The CPU tests cover the cdf builder, the restatement and the
launchers' argument checks."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from madigan_b200.environments.data_source import make_params, make_set_cdf
from oracle.set_draw_oracle import draw_sets, draw_uniform
from test_broker_sets import BROKER, plain_env
from test_param_sets import COMPOSITE, COMPOSITE_SETS, DSR, PAIR_SETS, RINGS, STATE, check_sets, same
from test_param_sets import make_env as plain_sets_env

SEED = 11
W4 = [3., 1., 0., 2.]  # over PAIR_SETS: set 2 is never drawn
W3 = [2., 1., 1.]      # over COMPOSITE_SETS


# ---------------------------------------------------------------------------------------------------- CPU
def test_make_set_cdf():
    cdf = make_set_cdf([4, 2, 1, 1, 0])
    assert cdf.dtype == np.float64 and cdf.tolist() == [.5, .75, .875, 1., 1.]
    cdf = make_set_cdf([0., .1, 0., .2, 0., .3, 0.])  # zero weights repeat their predecessor, the first one 0
    assert cdf[0] == 0. and cdf[2] == cdf[1] and cdf[4] == cdf[3] and cdf[6] == cdf[5] == 1.
    w = np.random.default_rng(1).random(1000) * 1e-3
    cdf = make_set_cdf(w)
    assert cdf[-1] == 1.0 and np.all(np.diff(cdf) >= 0)
    assert np.array_equal(cdf[:-1], (np.cumsum(w) / np.cumsum(w)[-1])[:-1])
    assert make_set_cdf([7.]).tolist() == [1.]
    assert make_set_cdf([1, 1, 1], n_sets=3).tolist() == [1 / 3, 2 / 3, 1.]
    for bad in ([], [[1., 2.]], [1., -1e-300], [1., float("nan")], [float("inf"), 1.], [0., 0.], [1e308, 1e308],
                ["a", 1.], None):
        with pytest.raises(ValueError):
            make_set_cdf(bad)
    with pytest.raises(ValueError, match="3 weights"):
        make_set_cdf([1., 2.], n_sets=3)


def test_restatement_golden():
    """Fixed ids for a fixed seed: the draw rule (Philox stream 4, u = (x0 >> 11) 2^-53, upper bound in the cdf) must
    not move."""
    cdf = make_set_cdf([4, 2, 1, 1, 0])
    got = draw_sets(cdf, 0x6d61646967616e00, range(24), [0] * 12 + [65] * 12)
    assert got.tolist() == [3, 0, 0, 1, 2, 1, 3, 1, 3, 1, 0, 3, 0, 2, 3, 3, 3, 3, 0, 0, 0, 1, 3, 0]
    got = draw_sets(make_set_cdf([1] * 7), 12345, range(100, 116), range(1000, 1016))
    assert got.tolist() == [3, 2, 2, 6, 2, 2, 6, 1, 5, 0, 3, 4, 2, 6, 0, 4]
    assert draw_sets(make_set_cdf([0, 0, 1, 0]), 3, range(50), range(50)).tolist() == [2] * 50
    assert draw_uniform(5, 7, 2 ** 40 + 3) != draw_uniform(5, 7, 3)  # the tick's high word is in the counter
    assert draw_uniform(5, 7 + 2 ** 32, 3) == draw_uniform(5, 7, 3)  # the env id is 32-bit, as in the kernels


def _lib():
    from madigan_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from madigan_b200.build import build
        build()
    return _lib.lib()


def test_draw_launchers_validate_without_gpu():
    """The _sets_draw entry points check their arguments before touching CUDA."""
    lib = _lib()
    P, _ = make_params("OU")
    L = A.MdgLaunch(n_envs=4, window=8, head=0)
    S, IO = A.MdgState(), A.MdgStepIO()
    S.folds = S.reset_ts = IO.pre_price = 1  # non-null dummies: never dereferenced, validation fails first
    ok = C.byref(A.MdgParamSets(p=1, set_of_env=1, n_sets=2))
    bad = [C.byref(A.MdgSetDraw(cdf=None, episode_set=1)), C.byref(A.MdgSetDraw(cdf=1, episode_set=None)),
           C.byref(A.MdgSetDraw())]
    for broker in (None, 1):
        for d in bad:
            assert lib.mdg_step_autoreset_sets_draw(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), 8, 1, 1,
                                                    1 << 20, ok, broker, d) == A.MDG_E_INVALID
            assert lib.mdg_reset_ws_sets_draw(C.byref(P), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, 1, 1 << 20,
                                              ok, broker, d) == A.MDG_E_INVALID
            assert lib.mdg_init_state_sets_draw(C.byref(P), None, C.byref(S), C.byref(L), ok, broker, d) == \
                A.MDG_E_INVALID
        good = C.byref(A.MdgSetDraw(cdf=1, episode_set=1))
        # no sets, or no workspace: refused as the _sets_broker launches refuse them
        assert lib.mdg_step_autoreset_sets_draw(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), 8, 1, 1,
                                                1 << 20, None, broker, good) == A.MDG_E_INVALID
        assert lib.mdg_reset_ws_sets_draw(C.byref(P), C.byref(S), C.byref(IO), C.byref(L), None, 8, 1, None, 0, ok,
                                          broker, good) == A.MDG_E_INVALID
        assert lib.mdg_init_state_sets_draw(C.byref(P), None, C.byref(S), C.byref(L), None, broker, good) == \
            A.MDG_E_INVALID
        Ps, _ = make_params("SineAdder")
        Ps.gen_ext, Ps.n_gen_ext = 1, 1 << 20
        assert lib.mdg_init_state_sets_draw(C.byref(Ps), None, C.byref(S), C.byref(L), ok, broker, good) == \
            A.MDG_E_UNSUPPORTED
    assert lib.mdg_sizeof(15) == C.sizeof(A.MdgSetDraw) == 16


# ---------------------------------------------------------------------------------------------------- GPU helpers
KINDS = {  # base config, sets, weights, flags: the all-pairs refill, the generic refill, the C4 composite
    "pairs": (PAIR_SETS[0], PAIR_SETS, W4, 0),
    "generic_fill": (PAIR_SETS[0], PAIR_SETS, W4, A.FLAG_GENERIC_FILL),
    "composite": (COMPOSITE, COMPOSITE_SETS, W3, 0),
}


def draw_env(cfg, sets, N, weights=None, assign=None, broker=False, seed=SEED, env_offset=0, window=16, flags=0,
             reward=DSR):
    """an Env with parameter sets (and broker sets), margins .1 / .25 and costs .02 / .001 without broker sets"""
    from madigan_b200.environments import Env
    e = Env("Composite", 1e6, {"data_source_config": cfg}, n_envs=N, window=window, seed=seed, env_offset=env_offset,
            reward=reward, param_sets=sets if isinstance(sets, int) else list(sets), param_set=assign,
            broker_sets=BROKER[:len(sets)] if broker else None, param_set_weights=weights)
    if not broker:
        e.setRequiredMargin(.1)
        e.setMaintenanceMargin(.25)
        e.setTransactionCost(.02, 0.)
        e.setSlippage(.001, 0.)
    e.flags = flags
    return e


def units(g, N, scale=40_000.):
    return torch.randint(-1, 2, (N, 16), generator=g, device="cuda").double() * scale


def restated(env, cdf, mask):
    """(N,) int32 ids: the restated draw for the envs where mask is true (at their timestamps now), 0 elsewhere"""
    idx = mask.nonzero().squeeze(1).cpu().numpy()
    ids = np.zeros(env.N, dtype=np.int32)
    ids[idx] = draw_sets(cdf, env.seed, idx + env.env_offset, env.t["timestamp"].cpu().numpy()[idx])
    return torch.from_numpy(ids).cuda()


def initial(env, cdf):
    """(N,) int32 ids of the constructor's draw (tick 0)"""
    gids = np.arange(env.N) + env.env_offset
    return torch.from_numpy(draw_sets(cdf, env.seed, gids, np.zeros(env.N, dtype=np.int64))).cuda()


def manual_reset(env, cdf, mask, normals=None, uniforms=None):
    """the recipe without the draw: restated ids for the masked envs, then a masked reset with history fill"""
    if bool(mask.any()):
        env.assign_param_sets(restated(env, cdf, mask), mask=mask)
    env.reset(mask=mask, fill_history=True, normals=normals, uniforms=uniforms)


def assert_same_envs(a, b, tag, names=STATE + RINGS):
    for name in names:
        assert same(a.t[name], b.t[name]), (tag, name)
    assert torch.equal(a.param_set, b.param_set), (tag, "param_set")


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("broker", [False, True], ids=["gen_sets", "broker_sets"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_fused_equals_manual(kind, broker):
    """Env A draws in the fused auto-reset; Env B (no weights) steps, assigns the restated ids to the envs that finished
    and resets them.  Every state and ring tensor and the assignment agree bit for bit after every step, through
    explicit masked resets too; episode_param_set holds the finished episode's set."""
    cfg, sets, weights, flags = KINDS[kind]
    N = 2048 if kind != "composite" else 1024
    cdf = make_set_cdf(weights)
    a = draw_env(cfg, sets, N, weights, broker=broker, flags=flags)
    b = draw_env(cfg, sets, N, None, initial(a, cdf), broker=broker, flags=flags)
    assert (a.episode_param_set == -1).all()
    assert_same_envs(a, b, "constructor")
    g = torch.Generator(device="cuda").manual_seed(7)
    resets = torch.zeros(N, dtype=torch.int64, device="cuda")
    for t in range(200):
        u = units(g, N)
        before, ep_before = a.param_set.clone(), a.episode_param_set.clone()
        a.step(u, auto_reset=True)
        b.step(u)
        done = b.t["done"].clone()
        assert torch.equal(a.t["done"], done), t
        manual_reset(b, cdf, done)
        assert_same_envs(a, b, f"step {t}")
        assert torch.equal(a.episode_param_set, torch.where(done, before, ep_before)), t
        resets += done
        if t % 25 == 24:  # an explicit reset draws for the masked envs only
            mask = torch.rand(N, generator=g, device="cuda") < .3
            before = a.param_set.clone()
            a.reset(mask, fill_history=True)
            manual_reset(b, cdf, mask)
            assert_same_envs(a, b, f"reset {t}")
            assert torch.equal(a.episode_param_set[mask], before[mask])
            resets += mask
    assert int((resets >= 3).sum()) > N // 2, f"too few resets: {resets.float().mean().item()} per env"
    if weights[2] == 0.:
        assert not (a.param_set == 2).any()


@pytest.mark.gpu
@pytest.mark.parametrize("broker", [False, True], ids=["gen_sets", "broker_sets"])
def test_injected_noise_resets(broker):
    """C4 composite with injected normals / uniforms: the step's separate reset and explicit masked resets with injected
    noise draw with Philox all the same, and equal the manual recipe with the same noise."""
    N, k = 512, 8
    cdf = make_set_cdf(W3)
    a = draw_env(COMPOSITE, COMPOSITE_SETS, N, W3, broker=broker, window=k)
    b = draw_env(COMPOSITE, COMPOSITE_SETS, N, None, a.param_set.clone(), broker=broker, window=k)
    assert torch.equal(a.param_set, initial(a, cdf))
    g = torch.Generator(device="cuda").manual_seed(3)
    nn_, nu = a.P.n_normals, a.P.n_uniforms
    n_reset = 0
    for t in range(60):
        u = units(g, N)
        nz = torch.randn((nn_, N), generator=g, device="cuda", dtype=torch.float64)
        uz = torch.rand((nu, N), generator=g, device="cuda", dtype=torch.float64)
        a.step(u, normals=nz, uniforms=uz, auto_reset=True)
        b.step(u, normals=nz, uniforms=uz)
        done = b.t["done"].clone()
        manual_reset(b, cdf, done)
        n_reset += int(done.sum())
        assert_same_envs(a, b, f"step {t}")
        if t % 6 == 5:
            mask = torch.rand(N, generator=g, device="cuda") < .4
            nz = torch.randn((k, nn_, N), generator=g, device="cuda", dtype=torch.float64)
            uz = torch.rand((k, nu, N), generator=g, device="cuda", dtype=torch.float64)
            a.reset(mask, fill_history=True, normals=nz, uniforms=uz)
            manual_reset(b, cdf, mask, nz, uz)
            n_reset += int(mask.sum())
            assert_same_envs(a, b, f"reset {t}")
    assert n_reset > N


@pytest.mark.gpu
@pytest.mark.parametrize("kind,broker", [("pairs", False), ("pairs", True), ("composite", False)])
def test_initial_draw_first_episode(kind, broker):
    """Without param_set the first episode's set is the tick-0 draw, and each env's first episode equals a plain Env of
    its drawn set (test_param_sets' contract and comparison)."""
    cfg, sets, weights, _ = KINDS[kind]
    N = 4096
    multi = draw_env(cfg, sets, N, weights, broker=broker)
    ids = initial(multi, make_set_cdf(weights))
    assert torch.equal(multi.param_set, ids)
    assert (multi.episode_param_set == -1).all()
    assert np.allclose(multi.param_set_weights, np.asarray(weights) / sum(weights))
    if broker:
        plains = [plain_env(c, N, BROKER[s], seed=SEED, reward=DSR, window=16) for s, c in enumerate(sets)]
    else:
        plains = [plain_sets_env(c, N, seed=SEED, reward=DSR, window=16) for c in sets]
    check_sets(multi, plains, "constructor")
    g = torch.Generator(device="cuda").manual_seed(4)
    for t in range(20):  # no auto-reset: every env stays in its first episode
        u = units(g, N, 5000.)
        for e in [multi] + plains:
            e.step(u)
        check_sets(multi, plains, f"step {t}")
    assert torch.equal(multi.param_set, ids) and (multi.episode_param_set == -1).all()


@pytest.mark.gpu
def test_shard_invariance():
    """One Env of 256 envs draws the same sets and runs the same states as two Envs of 128 with env_offset."""
    kw = dict(weights=W4, seed=99, window=8)
    big = draw_env(PAIR_SETS[0], PAIR_SETS, 256, **kw)
    lo = draw_env(PAIR_SETS[0], PAIR_SETS, 128, **kw)
    hi = draw_env(PAIR_SETS[0], PAIR_SETS, 128, env_offset=128, **kw)
    cat = lambda x, y: torch.cat([x, y], dim=-1)
    assert torch.equal(big.param_set, cat(lo.param_set, hi.param_set))
    assert torch.equal(big.param_set, initial(big, make_set_cdf(W4)))
    assert torch.equal(hi.param_set, initial(hi, make_set_cdf(W4)))
    g = torch.Generator(device="cuda").manual_seed(8)
    n_done = 0
    for t in range(60):
        u = units(g, 256)
        big.step(u, auto_reset=True)
        lo.step(u[:128].contiguous(), auto_reset=True)
        hi.step(u[128:].contiguous(), auto_reset=True)
        n_done += int(big.t["done"].sum())
        if t == 30:
            mask = torch.rand(256, generator=g, device="cuda") < .5
            big.reset(mask, fill_history=True)
            lo.reset(mask[:128], fill_history=True)
            hi.reset(mask[128:], fill_history=True)
    assert n_done > 0
    assert torch.equal(big.param_set, cat(lo.param_set, hi.param_set))
    assert torch.equal(big.episode_param_set, cat(lo.episode_param_set, hi.episode_param_set))
    for name in STATE + RINGS:
        if name == "pre_price":
            assert same(big.t[name], torch.cat([lo.t[name], hi.t[name]])), name
        else:
            assert same(big.t[name], cat(lo.t[name], hi.t[name])), name


@pytest.mark.gpu
def test_weights_distribution_and_changes():
    """Weights [4, 2, 1, 1, 0] over 65,536 envs: set 4 is never drawn and the counts fit the weights (chi-square, a
    fixed seed); a one-hot change mid-run sends every later reset to that set and leaves the other envs' sets alone;
    None keeps the sets through resets."""
    from scipy.stats import chisquare
    N = 65_536
    w = [4., 2., 1., 1., 0.]
    cdf = make_set_cdf(w)
    env = draw_env(PAIR_SETS[0], 5, N, w)
    assert torch.equal(env.param_set, initial(env, cdf))
    counts = torch.bincount(env.param_set.long(), minlength=5).cpu().numpy()
    g = torch.Generator(device="cuda").manual_seed(2)
    for t in range(10):
        env.step(units(g, N), auto_reset=True)
        done = env.t["done"]
        counts += torch.bincount(env.param_set[done].long(), minlength=5).cpu().numpy()
    assert counts[4] == 0 and counts.sum() >= 10_000
    p = np.array(w[:4]) / sum(w)
    assert chisquare(counts[:4], counts.sum() * p).pvalue > 1e-3, counts
    # one-hot mid-run: the next resets all draw set 3; the envs that do not reset keep their sets
    env.set_param_set_weights([0, 0, 0, 1, 0])
    assert env.param_set_weights.tolist() == [0., 0., 0., 1., 0.]
    n_done = 0
    for t in range(10):
        before = env.param_set.clone()
        env.step(units(g, N), auto_reset=True)
        done = env.t["done"]
        n_done += int(done.sum())
        assert (env.param_set[done] == 3).all() and torch.equal(env.param_set[~done], before[~done]), t
    mask = torch.rand(N, generator=g, device="cuda") < .5
    before = env.param_set.clone()
    env.reset(mask)
    assert (env.param_set[mask] == 3).all() and torch.equal(env.param_set[~mask], before[~mask])
    assert n_done > 0
    # None: the sets stay through resets, and episode_param_set is no longer written
    env.set_param_set_weights(None)
    assert env.param_set_weights is None
    before, ep = env.param_set.clone(), env.episode_param_set.clone()
    for t in range(10):
        env.step(units(g, N), auto_reset=True)
    env.reset(mask, fill_history=True)
    assert torch.equal(env.param_set, before) and torch.equal(env.episode_param_set, ep)


@pytest.mark.gpu
def test_set_param_set_weights_turns_the_draw_on():
    """An Env built with sets and no weights: set_param_set_weights turns the draw on at the next reset; an Env without
    sets refuses weights; make_env passes the keyword through."""
    from madigan_b200.environments import Env, make_env
    N = 1024
    env = draw_env(PAIR_SETS[0], PAIR_SETS, N, None)
    assert env.param_set_weights is None and torch.equal(env.param_set.cpu(), (torch.arange(N) % 4).int())
    env.set_param_set_weights([0, 1, 0, 0])
    mask = torch.arange(N, device="cuda") < N // 2
    env.reset(mask, fill_history=True)
    assert (env.param_set[mask] == 1).all()
    assert torch.equal(env.param_set[~mask].cpu(), (torch.arange(N // 2, N) % 4).int())
    assert torch.equal(env.episode_param_set[mask].cpu(), (torch.arange(N // 2) % 4).int())
    assert (env.episode_param_set[~mask] == -1).all()
    with pytest.raises(ValueError):
        env.set_param_set_weights([1., 1.])  # wrong length
    with pytest.raises(ValueError):
        env.set_param_set_weights([1., -1., 1., 1.])
    assert env.param_set_weights.tolist() == [0., 1., 0., 0.]  # a rejected call changes nothing
    with pytest.raises(ValueError, match="param_sets or broker_sets"):
        Env("Composite", 1e6, {"data_source_config": PAIR_SETS[0]}, n_envs=8, window=4, param_set_weights=[1.])
    with pytest.raises(RuntimeError):
        Env("Composite", 1e6, {"data_source_config": PAIR_SETS[0]}, n_envs=8, window=4).set_param_set_weights([1.])
    config = dict(env_type="Synth", data_source_type="Composite", data_source_config=PAIR_SETS[0], init_cash=1e6,
                  required_margin=.1, maintenance_margin=.25, transaction_cost_rel=.02, transaction_cost_abs=0.,
                  slippage_rel=.001, slippage_abs=0., n_envs=N, seed=SEED, preprocessor_config={"window_length": 16})
    m = make_env(config, param_sets=PAIR_SETS, param_set_weights=W4)
    assert torch.equal(m.param_set, initial(m, make_set_cdf(W4)))


@pytest.mark.gpu
@pytest.mark.parametrize("broker", [False, True], ids=["gen_sets", "broker_sets"])
def test_checkpoint_round_trip(broker):
    """state_dict mid-run, load_state_dict into a fresh Env with other weights, continue: bit for bit the uninterrupted
    run, the assignment, episode_param_set and the weights included.  Loading across the draw being on and off raises."""
    N = 2048
    g = torch.Generator(device="cuda").manual_seed(12)
    a = draw_env(PAIR_SETS[0], PAIR_SETS, N, W4, broker=broker)
    for _ in range(10):
        a.step(units(g, N), auto_reset=True)
    sd = a.state_dict()
    us = [units(g, N) for _ in range(20)]
    for u in us:
        a.step(u, auto_reset=True)
    b = draw_env(PAIR_SETS[0], PAIR_SETS, N, [1., 1., 1., 1.], broker=broker, seed=5)
    b.load_state_dict(sd)
    assert np.array_equal(b.param_set_weights, np.asarray(W4) / sum(W4))
    for u in us:
        b.step(u, auto_reset=True)
    assert_same_envs(a, b, "resumed")
    assert torch.equal(a.episode_param_set, b.episode_param_set)
    with pytest.raises(ValueError, match="set draw"):
        draw_env(PAIR_SETS[0], PAIR_SETS, N, None, broker=broker).load_state_dict(sd)
    with pytest.raises(ValueError, match="set draw"):
        b.load_state_dict(draw_env(PAIR_SETS[0], PAIR_SETS, N, None, broker=broker).state_dict())
