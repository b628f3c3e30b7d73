"""INTEGRATION.md made executable (VERDICT round 1, item 10).

* `prep_state_tensors` (reference: modelling/algorithm/dqn.py:188-199, with `abs_port_norm`,
  modelling/algorithm/utils.py:31-41) is restated below in the reference's words.  CPU test (runs where
  MADIGAN_REFERENCE names a madigan checkout): the restatement equals the reference's own functions, cut
  out of the reference files with `ast` (the modules themselves import the compiled C++ env), on random States.
* GPU tests: the restated function consumes the States produced by `madigan_b200.Env` + `StackerDiscrete` --
  batch=False for a single-env view, batch=True for N envs -- and the reference's agent-loop body
  (modelling/algorithm/offpolicy_q.py:136-205), restated statement for statement on the `SingleEnv` view, computes
  from `env.equity / positionValues / brokerResponse` the same reward as the batched Env's step kernel (1e-9),
  for 100 steps with resets."""
import ast
import os

import numpy as np
import pytest

REF = os.path.join(os.environ["MADIGAN_REFERENCE"], "madigan", "modelling", "algorithm") \
    if os.environ.get("MADIGAN_REFERENCE") else None


def abs_port_norm(port):
    """restated: modelling/algorithm/utils.py:31-41"""
    return port / port.abs().sum(-1, keepdim=True)


def prep_state_tensors(self, state, batch=False, device=None):
    """restated: modelling/algorithm/dqn.py:188-199"""
    import torch
    from madigan_b200.utils.data import State
    if not batch:
        price = torch.as_tensor(state.price[None, ...], dtype=torch.float32).to(self.device)
        port = torch.as_tensor(state.portfolio[None, -1], dtype=torch.float32).to(self.device)
    else:
        price = torch.as_tensor(state.price, dtype=torch.float32).to(self.device)
        port = torch.as_tensor(state.portfolio[:, -1], dtype=torch.float32).to(self.device)
    return State(price, abs_port_norm(port), state.timestamp)


def _reference_functions():
    import torch
    from madigan_b200.utils.data import State
    ns = {"torch": torch, "np": np, "State": State}
    tree = ast.parse(open(os.path.join(REF, "utils.py")).read())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "abs_port_norm")
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "utils.py", "exec"), ns)
    tree = ast.parse(open(os.path.join(REF, "dqn.py")).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "DQN")
    fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "prep_state_tensors")
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "dqn.py", "exec"), ns)
    return ns["prep_state_tensors"], ns["abs_port_norm"]


@pytest.mark.skipif(not REF or not os.path.isdir(REF), reason="needs MADIGAN_REFERENCE (a madigan checkout)")
def test_restated_prep_state_tensors_equals_the_reference_function():
    import types
    import torch
    from madigan_b200.utils.data import State
    ref_prep, ref_norm = _reference_functions()
    agent = types.SimpleNamespace(device="cpu")
    rng = np.random.default_rng(0)
    for batch, shape_p, shape_q in ((False, (16, 4), (16, 5)), (True, (8, 16, 4), (8, 16, 5))):
        st = State(rng.standard_normal(shape_p), rng.standard_normal(shape_q), np.arange(16))
        a, b = ref_prep(agent, st, batch=batch), prep_state_tensors(agent, st, batch=batch)
        assert torch.equal(a.price, b.price) and torch.equal(a.portfolio, b.portfolio)
    x = torch.randn(7, 5)
    assert torch.equal(ref_norm(x), abs_port_norm(x))


CFG = {"data_source_config": {f"pair{i}": {"data_source_type": "OUPair",
                                           "data_source_config": {"theta": .015, "phi": .01, "noise": .03}}
                              for i in range(2)}}
REWARD = dict(reward_shaper_config={"reward_shaper": None}, nstep_return=1, reduce_rewards=True)


@pytest.mark.gpu
def test_prep_state_tensors_consumes_our_states():
    import types
    import torch
    from madigan_b200.environments import Env, SingleEnv
    from madigan_b200.utils.preprocessor import StackerDiscrete
    prep = prep_state_tensors
    agent = types.SimpleNamespace(device="cuda")
    k = 16
    # N envs, batch=True
    env = Env("Composite", 1e6, CFG, n_envs=8, window=k, seed=1, device="cuda")
    st = StackerDiscrete(k, env.nFeats, norm=True, norm_type="lookback")
    env.reset(fill_history=True); st.sync(env)
    out = prep(agent, st.current_data(), batch=True)
    assert out.price.shape == (8, k, 4) and out.price.dtype == torch.float32 and out.price.is_cuda
    assert out.portfolio.shape == (8, 5)
    assert torch.allclose(out.portfolio.abs().sum(-1), torch.ones(8, device="cuda"))
    # one env, batch=False, through the single-env view (numpy in, as the reference's preprocessor hands it over)
    env1 = Env("Composite", 1e6, CFG, n_envs=1, window=k, seed=1, device="cuda")
    st1 = StackerDiscrete(k, env1.nFeats, norm=True, norm_type="lookback")
    env1.reset(fill_history=True); st1.sync(env1)
    cur = st1.current_data()
    from madigan_b200.utils.data import State
    single = State(cur.price[0].cpu().numpy(), cur.portfolio[0].cpu().numpy(), cur.timestamp[0].cpu().numpy())
    out1 = prep(agent, single, batch=False)
    assert out1.price.shape == (1, k, 4) and out1.portfolio.shape == (1, 5)
    # same seed, same generator stream: env 0 of the batch is the single env
    assert torch.allclose(out1.price[0], out.price[0]) and torch.allclose(out1.portfolio[0], out.portfolio[0])
    assert isinstance(SingleEnv(env1).equity, float)


@pytest.mark.gpu
def test_reference_agent_loop_body_on_single_env_matches_in_kernel_reward():
    import torch
    from madigan_b200.environments import Env, SingleEnv
    k = 8
    fast = Env("Composite", 1e6, CFG, n_envs=1, window=k, seed=4, device="cuda", reward=REWARD)  # in-kernel rewards
    slow = Env("Composite", 1e6, CFG, n_envs=1, window=k, seed=4, device="cuda")                 # the reference's way
    for e in (fast, slow):
        e.setTransactionCost(.002, 0.); e.setSlippage(.001, 0.); e.setRequiredMargin(.5)
        e.reset(fill_history=True)
    env = SingleEnv(slow)
    rng = np.random.default_rng(0)
    n_done = 0
    for t in range(100):
        transaction = rng.integers(-1, 2, size=4) * 40_000.
        # ---- offpolicy_q.py:140-164, on the single-env view
        prev_eq = env.equity
        prev_val = env.positionValues
        _next_state, reward, done, info = env.step(transaction)
        info = info.brokerResponse
        curr_val = env.positionValues
        mar_diff = (info.transactionUnits * info.transactionPrice + info.transactionCost)
        reward = (curr_val - prev_val - mar_diff) / prev_eq
        reward += 1
        reward = np.log(np.maximum(reward, .35))
        reward = reward.sum(keepdims=True)  # reduce_rewards
        # ---- the batched env computes the same thing inside the step kernel
        fast.step(torch.from_numpy(transaction).reshape(1, 4).cuda())
        got = fast.agent_reward[0].cpu().numpy()
        np.testing.assert_allclose(got, reward, rtol=1e-9, atol=1e-12)
        assert bool(fast.t["done"][0]) == done
        if done:  # offpolicy_q.py:199-201 reset_state(): env.reset() + initialize_history
            n_done += 1
            slow.reset(fill_history=True)
            fast.reset(fill_history=True)
    assert _next_state.price.shape == (4,) and isinstance(done, bool)
