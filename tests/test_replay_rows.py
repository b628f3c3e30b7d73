"""The replay row store (DeviceReplay / DevicePrioritizedReplay with store="rows", include/madigan_b200.h "Replay row
store"): the ingest invariant against env.window, bit-identical samples against the window store, the rows'
residency rule, CUDA-graph capture and argument validation."""
import ctypes as C

import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from oracle import per_oracle as po
from test_replay import CASES, K, N, SCALE, SEED, T

NORMS = [None, "lookback", "lookback_log", "log", "standard_normal", "log_standard_normal", "expanding"]


def golden_run(name, make_buffers, steps=T, on_step=None):
    """The seeded episode of tests/test_replay.py (explicit env.reset(mask, fill_history=True) of finished envs between
    step and add), feeding every buffer make_buffers(env) returns; on_step(env, t) after each step's adds."""
    from madigan_b200.environments import Env
    rw = dict(CASES[name], discount=.99, reduce_rewards=True)
    env = Env("OUPair", 1e6, {"data_source_config": {"theta": .015, "phi": .01, "noise": .03}}, n_envs=N, window=K,
              seed=7, reward=rw)
    env.setRequiredMargin(.1); env.setMaintenanceMargin(.25)
    env.setTransactionCost(.02, 0.); env.setSlippage(.001, 0.)
    nn = env.P.n_normals
    rng = np.random.default_rng(SEED)
    env.reset(fill_history=True, normals=rng.standard_normal((K, nn, N)), uniforms=rng.random((K, 1, N)))
    bufs = make_buffers(env)
    for b in bufs:
        b.observe_start()
    if on_step:
        on_step(env, -1)
    for t in range(steps):
        price = env.t["price"].cpu().numpy().T
        price = np.where(np.abs(price) > 1e-9, price, 1.)
        a = rng.integers(-1, 2, size=(N, 2)).astype(np.float64)
        units = np.ascontiguousarray(a * (SCALE / np.abs(price)) * rng.uniform(.2, 1.5, size=(N, 2)))
        env.step(torch.from_numpy(units), normals=rng.standard_normal((nn, N)), uniforms=rng.random((1, N)))
        done = env.t["done"].cpu().numpy().astype(bool)
        if done.any():
            env.reset(mask=torch.from_numpy(done), fill_history=True, normals=rng.standard_normal((K, nn, N)),
                      uniforms=rng.random((K, 1, N)))
        for b in bufs:
            b.add(torch.from_numpy(units))
        if on_step:
            on_step(env, t)
    return env, bufs


def stored_window(rp, step):
    """(N, k, nF) raw window the row store keeps for the observation of `step`, gathered on the device."""
    end = rp.row_end[step % rp.depth]                                    # (N,)
    c = end[:, None] + torch.arange(-rp.k + 1, 1, device=end.device)     # (N, k) row numbers, oldest first
    return torch.gather(rp.rows, 1, (c % rp.n_rows)[:, :, None].expand(-1, -1, rp.nF))


def resident_rows(rp, idx):
    """numpy restatement of the row store's residency rule for records idx."""
    te, ss = (rp.t[k_].cpu().numpy()[idx] for k_ in ("t_env", "t_state_slot"))
    end = rp.row_end.cpu().numpy()[ss, te]
    return (end >= rp.k) & (end - rp.k + 1 > rp.row_count.cpu().numpy()[te] - rp.n_rows)


def assert_same_sample(a, b):
    for x, y in zip((a.state.price, a.state.portfolio, a.action, a.reward, a.next_state.price,
                     a.next_state.portfolio, a.done), (b.state.price, b.state.portfolio, b.action, b.reward,
                                                       b.next_state.price, b.next_state.portfolio, b.done)):
        assert x.dtype == y.dtype and x.shape == y.shape
        assert torch.equal(x.view(torch.uint8) if x.dtype != torch.bool else x,
                           y.view(torch.uint8) if y.dtype != torch.bool else y)  # bit-identical, NaN included


# ---------------------------------------------------------------------------------------------------- CPU
def test_rows_abi_validation_without_gpu():
    """The rows launchers validate their arguments before touching CUDA."""
    import os
    from madigan_b200 import _lib
    from madigan_b200._lib import check
    if not os.path.exists(_lib.LIB_PATH):
        from madigan_b200.build import build
        build()
    cdll = _lib.lib()
    rr = A.MdgReplayRows(rows=1, row_end=1, row_count=1, last_ts=1, n_rows=64 + 8 - 1, n_feats=2, window=8)
    w = A.MdgWindow(ring=1, prefix=1, timestamp=1, reset_ts=1, n_envs=4, n_feats=2, window=8, head=0, n_valid=8)
    rp = A.MdgReplay(**{n: 1 for n in ("t_env", "t_state_slot", "t_next_slot", "t_state_step", "t_done", "t_reward",
                                       "t_action", "cursor", "act_ring")}, capacity=10, depth=64, nstep=1, ra=1,
                     n_action=2)
    out = A.MdgReplayBatch(**{n: 1 for n in ("idx", "state_price", "next_price", "state_port", "next_port", "action",
                                             "reward", "done")})
    pr = A.MdgPrioritized(**{n: 1 for n in ("sum_tree", "min_tree", "leaf_pos", "batch_pos", "dirty", "dirty_list",
                                            "ctl", "seen", "max_priority", "n_rejected")}, capacity=10,
                          tree_size=1024, alpha=.6)

    def ingest(rr_, w_, slot=0):
        return cdll.mdg_replay_rows_ingest(C.byref(rr_) if rr_ is not None else None, C.byref(w_), slot, 0)

    def sample(rr_, norm=A.NORM_NONE, dt=A.DTYPE_F32, port=1):
        return cdll.mdg_replay_sample_rows(C.byref(rp), C.byref(rr_), 4, 10, port, 3, norm, dt, 16, 0, 1,
                                           C.byref(out), None)

    def per_sample(rr_, norm=A.NORM_NONE):
        return cdll.mdg_per_sample_rows(C.byref(pr), C.byref(rp), C.byref(rr_), 4, 10, 1, 3, norm, A.DTYPE_F32, 16,
                                        .4, 0, 1, C.byref(out), 1, 1, None)

    with pytest.raises(ValueError):
        check(ingest(None, w))
    with pytest.raises(ValueError):
        check(ingest(A.MdgReplayRows(rows=None, row_end=1, row_count=1, last_ts=1, n_rows=70, n_feats=2, window=8), w))
    with pytest.raises(ValueError):  # a window shorter than k
        check(ingest(rr, A.MdgWindow(ring=1, prefix=1, timestamp=1, reset_ts=1, n_envs=4, n_feats=2, window=8,
                                     head=0, n_valid=5)))
    with pytest.raises(ValueError):  # no prefix buffer
        check(ingest(rr, A.MdgWindow(ring=1, prefix=None, timestamp=1, reset_ts=1, n_envs=4, n_feats=2, window=8,
                                     head=0, n_valid=8)))
    with pytest.raises(ValueError):
        check(ingest(rr, w, slot=-1))
    small = A.MdgReplayRows(rows=1, row_end=1, row_count=1, last_ts=1, n_rows=64 + 8 - 2, n_feats=2, window=8)
    for f in (sample, per_sample):
        with pytest.raises(ValueError):
            check(f(small))
        with pytest.raises(ValueError):
            check(f(rr, norm=7))
    with pytest.raises(ValueError):
        check(sample(rr, dt=5))
    with pytest.raises(ValueError):
        check(sample(rr, port=0))  # null obs_port


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_ingest_invariant_golden_episode(name):
    from madigan_b200.utils.replay import DeviceReplay
    seen = []

    def check_step(env, t):
        rp = seen[0]
        assert torch.equal(stored_window(rp, t), env.window(None, torch.float64)), t
        seen.append(t)

    def make(env):
        seen.append(DeviceReplay(env, depth=16, rows=16 + 3 * (K - 1), store="rows"))
        return seen[:1]

    golden_run(name, make, on_step=check_step)
    assert len(seen) == T + 2


@pytest.mark.gpu
def test_ingest_invariant_bench_shaped_auto_reset():
    """8 OU pairs x 16 assets, k 64, DSR n=1, 2,048 envs, 300 auto-reset steps: the all-pairs refill path."""
    import bench
    from madigan_b200.utils.replay import DeviceReplay
    dev = torch.device("cuda", 0)
    env = bench.make_env(dev, 0, n_envs=2048)
    acts = bench.synth_actions(4, 2048, 1, device=dev)
    rp = DeviceReplay(env, depth=16, store="rows", norm_type="standard_normal")
    rp.observe_start()
    assert torch.equal(stored_window(rp, -1), env.window(None, torch.float64))
    resets = 0
    for t in range(300):
        env.step(acts[t % 4], auto_reset=True)
        rp.add(acts[t % 4])
        resets += int(env.t["done"].sum().item())
        assert torch.equal(stored_window(rp, t), env.window(None, torch.float64)), t
    assert resets > 100
    rec = int(rp.row_count.sum().item())
    assert rec == 2048 * (64 + 300) + (64 - 1) * resets  # one row per env-step, k - 1 more per reset


def _fed_pair(name, norm, dtype, depth, prioritized=False):
    from madigan_b200.utils.replay import DevicePrioritizedReplay, DeviceReplay
    cls = DevicePrioritizedReplay if prioritized else DeviceReplay
    kw = dict(alpha=.6) if prioritized else {}

    def make(env):
        return [cls(env, depth=depth, norm_type=norm, dtype=dtype, seed=3, **kw),
                cls(env, depth=depth, norm_type=norm, dtype=dtype, seed=3, store="rows", rows=depth * K, **kw)]

    return golden_run(name, make)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("norm", NORMS)
def test_uniform_samples_match_window_store(norm, dtype):
    env, (win, rows) = _fed_pair("dsr_n5", norm, dtype, depth=32)
    assert rows.obs_price is None
    for k_ in win.t:
        assert torch.equal(win.t[k_], rows.t[k_]), k_
    assert torch.equal(win.obs_port, rows.obs_port)
    for n in (512, 4096):
        a, _ = win.sample(n)
        b, _ = rows.sample(n)
        assert torch.equal(win.last_idx, rows.last_idx) and bool(win.last_valid.all())
        assert_same_sample(a, b)
    assert len(win) == len(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("norm", NORMS)
def test_prioritized_samples_match_window_store(norm, dtype):
    env, (win, rows) = _fed_pair("sum_n3", norm, dtype, depth=32, prioritized=True)
    rng = np.random.default_rng(4)
    for n, beta in ((512, .4), (4096, 1.)):
        T_ = rows.tree_size
        st, mt = rows.per["sum_tree"].cpu().numpy(), rows.per["min_tree"].cpu().numpy()
        cur = int(rows.t["cursor"].item())
        idx_o, pos_o, w_o = po.sample(st, mt, rows.per["leaf_pos"].cpu().numpy(),
                                      rows.t["t_state_step"].cpu().numpy(), min(cur, rows.capacity),
                                      rows.step_count, rows.depth, n, beta, rows.seed, rows.draws + 1)
        a, wa = win.sample(n, beta)
        b, wb = rows.sample(n, beta)
        assert torch.equal(win.last_idx, rows.last_idx) and torch.equal(win.last_pos, rows.last_pos)
        assert np.array_equal(rows.last_idx.cpu().numpy(), idx_o)
        assert torch.equal(wa, wb)
        assert_same_sample(a, b)
        p = torch.from_numpy(rng.gamma(2., 1., size=n)).cuda()
        win.update_priorities(p)
        rows.update_priorities(p)
        for k_ in ("sum_tree", "min_tree", "leaf_pos", "max_priority", "n_rejected"):
            assert torch.equal(win.per[k_], rows.per[k_]), k_
        assert T_ == win.tree_size


@pytest.mark.gpu
def test_records_stale_through_rows_are_not_drawn():
    """depth 16 and rows = depth + k - 1 on an episode with resets: some records lose their rows; none is drawn."""
    from madigan_b200.utils.replay import DevicePrioritizedReplay, DeviceReplay

    def make(env):
        return [DeviceReplay(env, depth=16, store="rows", rows=16 + K - 1, norm_type="lookback"),
                DevicePrioritizedReplay(env, depth=16, store="rows", rows=16 + K - 1, norm_type="lookback")]

    env, (uni, per) = golden_run("ddr_n1", make)
    hold = torch.zeros((N, 2), dtype=torch.float64)
    for _ in range(2):  # two resets of every env within the last `depth` steps: k - 1 extra rows each
        env.step(hold)
        env.reset(fill_history=True)
        uni.add(hold)
        per.add(hold)
    for _ in range(3):
        env.step(hold)
        uni.add(hold)
        per.add(hold)
    n = len(uni)
    all_idx = np.arange(n)
    steps = uni.t["t_state_step"].cpu().numpy()[:n]
    slot_ok = steps > uni.step_count - uni.depth
    rows_ok = resident_rows(uni, all_idx)
    assert (slot_ok & ~rows_ok).any(), "the episode must make some records stale through their rows"
    assert (slot_ok & rows_ok).any()
    for rp, draw in ((uni, lambda: uni.sample(4096)), (per, lambda: per.sample(4096, .5))):
        draw()
        idx = rp.last_idx.cpu().numpy()
        assert bool(rp.last_valid.all())
        assert resident_rows(rp, idx).all()
        assert (rp.t["t_state_step"].cpu().numpy()[idx] > rp.step_count - rp.depth).all()
        assert len(np.unique(idx)) > 1


@pytest.mark.gpu
@pytest.mark.parametrize("prioritized", [False, True])
def test_cuda_graph_capture_matches_eager(prioritized):
    from madigan_b200.utils.replay import DevicePrioritizedReplay, DeviceReplay
    cls = DevicePrioritizedReplay if prioritized else DeviceReplay
    runs = [golden_run("dsr_n5", lambda env: [cls(env, depth=32, store="rows", norm_type="standard_normal")])
            for _ in range(2)]
    act = torch.ones((N, 2), dtype=torch.float64, device="cuda") * 1000.
    pr = torch.from_numpy(np.random.default_rng(2).gamma(2., 1., size=256)).cuda()
    sample = (lambda rp: rp.sample(256, .3)) if prioritized else (lambda rp: rp.sample(256))
    for env, (rp,) in runs:  # warm-up: the same calls on both
        sample(rp)
        if prioritized:
            rp.update_priorities(pr)
        env.step(act)
    torch.cuda.synchronize()
    (_, (eager,)), (_, (graphed,)) = runs
    eager.add(act)
    s_e, w_e = sample(eager)
    if prioritized:
        eager.update_priorities(pr)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        graphed.add(act)
        s_g, w_g = sample(graphed)
        if prioritized:
            graphed.update_priorities(pr)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager.last_idx, graphed.last_idx)
    assert_same_sample(s_e, s_g)
    for k_ in ("rows", "row_end", "row_count", "last_ts"):
        assert torch.equal(getattr(eager, k_), getattr(graphed, k_)), k_
    if prioritized:
        assert torch.equal(w_e, w_g)
        for k_ in ("sum_tree", "min_tree", "leaf_pos", "max_priority"):
            assert torch.equal(eager.per[k_], graphed.per[k_]), k_


@pytest.mark.gpu
def test_rows_store_value_errors():
    from madigan_b200.environments import Env
    from madigan_b200.utils.replay import DevicePrioritizedReplay, DeviceReplay
    rw = dict(reward_shaper_config={"reward_shaper": "None"}, nstep_return=1, discount=.99, reduce_rewards=True)
    env = Env("OUPair", 1e6, {"data_source_config": {"theta": .015, "phi": .01, "noise": .03}}, n_envs=8, window=8,
              seed=1, reward=rw)
    with pytest.raises(ValueError):
        DeviceReplay(env, depth=16, store="frames")
    for cls in (DeviceReplay, DevicePrioritizedReplay):
        with pytest.raises(ValueError):
            cls(env, depth=16, store="rows", rows=16 + 8 - 2)
        cls(env, depth=16, store="rows", rows=16 + 8 - 1)
    rp = DeviceReplay(env, depth=16, store="rows")
    assert rp.n_rows == 16 + 3 * 7 and rp.obs_price is None
    assert env.n_valid < env.k  # a fresh env holds one row
    with pytest.raises(ValueError):
        rp.observe_start()
    env.step()
    with pytest.raises(ValueError):
        rp.add(torch.zeros((8, 2), dtype=torch.float64))
