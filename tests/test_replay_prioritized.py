"""Device-side prioritized replay (DevicePrioritizedReplay, csrc/mdg_per.cu) against the sequential oracle
(oracle/per_oracle.py), on the seeded golden episode of tests/test_replay.py."""
import functools

import numpy as np
import pytest
import torch

from oracle import per_oracle as po
from test_replay import N, run_episode

pytestmark = pytest.mark.gpu
ALPHA = .6
POW_RTOL = 5e-16  # CUDA's pow: at most 2 ulp (CUDA C++ Programming Guide, mathematical functions)


def prioritized_episode(name, depth=128, alpha=ALPHA):
    """run_episode of tests/test_replay.py with the buffer it builds replaced by a DevicePrioritizedReplay."""
    from madigan_b200.utils import replay as R
    plain = R.DeviceReplay
    R.DeviceReplay = functools.partial(R.DevicePrioritizedReplay, alpha=alpha)
    try:
        return run_episode(name, depth=depth)
    finally:
        R.DeviceReplay = plain


def snapshot(rp):
    """The GPU buffer's state as an oracle (leaves, positions, max_priority, count) plus its two trees."""
    s = {k: v.cpu().numpy() for k, v in rp.per.items()}
    T = rp.tree_size
    orc = po.PerOracle(rp.capacity, rp.alpha)
    orc.sum_leaves, orc.min_leaves = s["sum_tree"][T:].copy(), s["min_tree"][T:].copy()
    orc.leaf_pos, orc.max_priority = s["leaf_pos"].copy(), float(s["max_priority"][0])
    orc.n_rejected, orc.seen = int(s["n_rejected"][0]), int(s["seen"][0])
    return orc, s["sum_tree"], s["min_tree"]


def assert_trees_pairwise(st, mt):
    """Every internal node is bit-equal to numpy's left + right / min(left, right) of the GPU's own leaves."""
    T = len(st) // 2
    np.testing.assert_array_equal(st[1:], po.build_tree(st[T:], np.add)[1:])
    np.testing.assert_array_equal(mt[1:], po.build_tree(mt[T:], np.minimum)[1:])


def assert_same_leaves(rp, orc):
    got, st, mt = snapshot(rp)
    np.testing.assert_allclose(got.sum_leaves, orc.sum_leaves, rtol=POW_RTOL, atol=0)
    np.testing.assert_allclose(got.min_leaves, orc.min_leaves, rtol=POW_RTOL, atol=0)
    assert np.array_equal(got.leaf_pos, orc.leaf_pos)
    assert got.max_priority == orc.max_priority and got.n_rejected == orc.n_rejected
    assert_trees_pairwise(st, mt)


def oracle_sample(rp, st, mt, batch, beta):
    """The oracle's descent on the given trees with the draw the next rp.sample(batch, beta) uses."""
    cur = int(rp.t["cursor"].item())
    return po.sample(st, mt, rp.per["leaf_pos"].cpu().numpy(), rp.t["t_state_step"].cpu().numpy(),
                     min(cur, rp.capacity), rp.step_count, rp.depth, batch, beta, rp.seed, rp.draws + 1)


def bad_priorities(rng, n):
    """|TD|-like priorities with a few rows that must be rejected (nan, inf, 0, negative)."""
    p = rng.gamma(2., .5, size=n)
    p[rng.choice(n, 4, replace=False)] = [np.nan, np.inf, 0., -1.]
    return p


def test_leaves_and_trees_after_ingest_and_updates():
    env, rp, _ = prioritized_episode("dsr_n5")
    n = len(rp)
    orc = po.PerOracle(rp.capacity, ALPHA)
    orc.ingest(n)
    assert_same_leaves(rp, orc)
    assert (orc.sum_leaves[:n] == 1.).all() and n < rp.capacity  # max_priority 1 ** alpha
    rng = np.random.default_rng(5)
    for r in range(4):
        rp.sample(256, .4)
        idx, pos = rp.last_idx.cpu().numpy(), rp.last_pos.cpu().numpy()
        pr = bad_priorities(rng, 256) * (r + 1)
        rp.update_priorities(torch.from_numpy(pr if r % 2 else pr.astype(np.float32)))
        orc.update(idx, pos, pr if r % 2 else pr.astype(np.float32).astype(np.float64))
        assert_same_leaves(rp, orc)
    assert orc.max_priority > 1. and orc.n_rejected == 16
    # records appended after the updates enter at the new max_priority ** alpha
    env.step(torch.zeros((N, 2), dtype=torch.float64))
    rp.add(torch.zeros((N, 2), dtype=torch.float64))
    orc.ingest(int(rp.t["cursor"].item()))
    assert_same_leaves(rp, orc)


def test_sample_matches_oracle_and_gathers_stored_records():
    env, rp, _ = prioritized_episode("dsr_n5")
    rng = np.random.default_rng(6)
    for _ in range(3):  # uneven priorities first
        rp.sample(128, .4)
        rp.update_priorities(torch.from_numpy(rng.gamma(1., 1., size=128)))
    for batch, beta in ((512, .5), (4096, 1.)):
        _, st, mt = snapshot(rp)
        idx_o, pos_o, w_o = oracle_sample(rp, st, mt, batch, beta)
        sarsd, w = rp.sample(batch, beta)
        idx = rp.last_idx.cpu().numpy()
        assert np.array_equal(idx, idx_o) and (idx >= 0).all()
        assert np.array_equal(rp.last_pos.cpu().numpy(), pos_o)
        assert w.dtype == torch.float64 and w.shape == (batch,)
        np.testing.assert_allclose(w.cpu().numpy(), w_o, rtol=1e-12, atol=0)
        assert rp.last_valid.all()
        te, ss, sn = (rp.t[k_].cpu().numpy()[idx] for k_ in ("t_env", "t_state_slot", "t_next_slot"))
        op, opt = rp.obs_price.cpu().numpy(), rp.obs_port.cpu().numpy()
        np.testing.assert_array_equal(sarsd.state.price.cpu().numpy(), op[ss, te])
        np.testing.assert_array_equal(sarsd.next_state.price.cpu().numpy(), op[sn, te])
        np.testing.assert_array_equal(sarsd.state.portfolio.cpu().numpy(), opt[ss, te])
        np.testing.assert_array_equal(sarsd.next_state.portfolio.cpu().numpy(), opt[sn, te])
        np.testing.assert_array_equal(sarsd.action.cpu().numpy(), rp.t["t_action"].cpu().numpy()[idx])
        np.testing.assert_array_equal(sarsd.reward.cpu().numpy(), rp.t["t_reward"].cpu().numpy()[idx])
        np.testing.assert_array_equal(sarsd.done.cpu().numpy(), rp.t["t_done"].cpu().numpy()[idx].astype(bool))


def test_never_samples_overwritten_observations_and_matches_oracle():
    """depth 16 < episode length: stale leaves keep their mass and are rejected and redrawn."""
    env, rp, _ = prioritized_episode("sum_n3", depth=16)
    steps_all = rp.t["t_state_step"].cpu().numpy()
    _, st, mt = snapshot(rp)
    for ahead in (0, 8):  # sampling as if `ahead` more steps had overwritten observation slots: most leaves stale
        rp.step_count += ahead
        try:
            idx_o, _, w_o = oracle_sample(rp, st, mt, 1024, .7)
            _, w = rp.sample(1024, .7)
            idx = rp.last_idx.cpu().numpy()
            stale = steps_all[:len(rp)] <= rp.step_count - rp.depth
            if ahead:
                assert stale.mean() > .25
            assert np.array_equal(idx, idx_o) and (idx >= 0).all()
            np.testing.assert_allclose(w.cpu().numpy(), w_o, rtol=1e-12, atol=0)
            assert (steps_all[idx] > rp.step_count - rp.depth).all()
        finally:
            rp.step_count -= ahead


def test_empirical_frequencies_follow_priorities():
    """A few thousand envs: the sampled frequencies pass a chi-square test against p_i / sum(p_resident)."""
    from scipy.stats import chisquare
    from madigan_b200.environments import Env
    from madigan_b200.utils.replay import DevicePrioritizedReplay
    n_envs = 2048
    env = Env("OUPair", 1e6, {"data_source_config": {"theta": .015, "phi": .01, "noise": .03}}, n_envs=n_envs,
              window=8, seed=11, reward=dict(reward_shaper_config={"reward_shaper": "None"}, nstep_return=1,
                                             discount=.99, reduce_rewards=True))
    rp = DevicePrioritizedReplay(env, alpha=.7, depth=8, norm_type="lookback", seed=4)
    env.reset(fill_history=True)
    rp.observe_start()
    hold = torch.zeros((n_envs, 2), dtype=torch.float64, device=env.device)
    for _ in range(10):
        env.step(hold, auto_reset=True)
        rp.add(hold)
    gen = torch.Generator(env.device).manual_seed(3)
    for _ in range(6):  # spread the priorities over two orders of magnitude
        rp.sample(4096, 0.)
        rp.update_priorities(torch.exp(torch.randn(4096, dtype=torch.float64, device=env.device, generator=gen) * 1.5))
    T, cap = rp.tree_size, rp.capacity
    leaves = rp.per["sum_tree"][T:T + cap].cpu().numpy()
    resident = (rp.per["leaf_pos"].cpu().numpy() >= 0) & \
        (rp.t["t_state_step"].cpu().numpy() > rp.step_count - rp.depth)
    counts = torch.zeros(cap, dtype=torch.int64, device=env.device)
    draws = 0
    for _ in range(48):
        rp.sample(32768, .5)
        counts += torch.bincount(rp.last_idx, minlength=cap)
        draws += 32768
    counts = counts.cpu().numpy()
    assert counts[~resident].sum() == 0
    p = leaves[resident] / leaves[resident].sum()
    assert resident.sum() > 10000
    assert chisquare(counts[resident], p * draws).pvalue > 1e-3


def test_update_semantics_with_duplicates_drops_and_overwrites():
    env, rp, _ = prioritized_episode("sum_n3", depth=16)
    rp.sample(64, .4)
    idx, pos = rp.last_idx, rp.last_pos
    idx[7], pos[7] = idx[3], pos[3]     # the same record three times: the last occurrence wins
    idx[40], pos[40] = idx[3], pos[3]
    idx[11], pos[11] = -1, -1           # a row without a record
    hold = torch.zeros((N, 2), dtype=torch.float64)
    for _ in range(6):                  # the ring (72 records) turns over about halfway
        env.step(hold)
        rp.add(hold)
    orc, _, _ = snapshot(rp)
    idx_h, pos_h = idx.cpu().numpy(), pos.cpu().numpy()
    overwritten = (idx_h >= 0) & (orc.leaf_pos[np.maximum(idx_h, 0)] != pos_h)
    assert overwritten.any() and (~overwritten & (idx_h >= 0)).sum() > 10
    pr = np.random.default_rng(9).gamma(2., 1., size=64)
    pr[[5, 9, 20]] = [np.nan, -2., 0.]
    pr[40] = 7.5
    rp.update_priorities(torch.from_numpy(pr).to(env.device))
    orc.update(idx_h, pos_h, pr)
    assert_same_leaves(rp, orc)
    assert int(rp.n_rejected.item()) == orc.n_rejected
    assert float(rp.max_priority.item()) == orc.max_priority


def test_cuda_graph_capture_matches_eager():
    """add, sample and update_priorities captured in one CUDA graph give the eager calls' trees, indices, weights."""
    runs = [prioritized_episode("dsr_n5") for _ in range(2)]
    pr = torch.from_numpy(np.random.default_rng(2).gamma(2., 1., size=256)).cuda()
    act = torch.ones((N, 2), dtype=torch.float64, device="cuda") * 1000.
    for env, rp, _ in runs:  # warm-up: same calls on both, so that both are in the same state
        rp.sample(256, .3)
        rp.update_priorities(pr)
        env.step(act)
    torch.cuda.synchronize()
    (_, eager, _), (_, graphed, _) = runs
    eager.add(act)
    _, w_e = eager.sample(256, .3)
    eager.update_priorities(pr * 2)
    g = torch.cuda.CUDAGraph()
    pr2 = pr * 2
    with torch.cuda.graph(g):
        graphed.add(act)
        _, w_g = graphed.sample(256, .3)
        graphed.update_priorities(pr2)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(eager.last_idx.cpu().numpy(), graphed.last_idx.cpu().numpy())
    assert np.array_equal(w_e.cpu().numpy(), w_g.cpu().numpy())
    for k in ("sum_tree", "min_tree", "leaf_pos", "max_priority", "seen", "ctl", "dirty"):
        assert np.array_equal(eager.per[k].cpu().numpy(), graphed.per[k].cpu().numpy()), k
    assert (eager.per["ctl"].cpu().numpy() == 0).all() and (eager.per["dirty"].cpu().numpy() == 0).all()
