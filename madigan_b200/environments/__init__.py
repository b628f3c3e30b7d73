"""reference: madigan/environments/__init__.py (make_env :9-22, get_env_info :41-56)."""
import copy

from .env import Asset, Env  # noqa: F401
from .data_source import ConfigError, make_params, make_reward  # noqa: F401


def _get(cfg, key, default=None):
    try:
        return cfg[key] if key in cfg else default
    except TypeError:
        return getattr(cfg, key, default)


def make_env(config, test=False, **batched):
    """Same keys as the reference; the batched ones (``n_envs``, ``seed``, ``device``) may be in
    ``config`` or passed as keywords, and every other keyword goes to ``Env``.  With ``broker_sets`` the config's
    margins, costs and slippage are the base values of the broker sets, and no setter is called.  ``param_set_weights``
    (with ``param_sets`` or ``broker_sets``) turns on the per-episode set draw, as for ``Env``."""
    config = copy.deepcopy(config)
    if test and "data_source_config_test" in config.keys():
        config["data_source_config"] = config["data_source_config_test"]
    if _get(config, "env_type") in ("Synth",):
        env = Env(_get(config, "data_source_type"), _get(config, "init_cash"), config, **batched)
        if batched.get("broker_sets") is not None:
            return env
        env.setRequiredMargin(_get(config, "required_margin"))
        env.setMaintenanceMargin(_get(config, "maintenance_margin"))
        env.setTransactionCost(_get(config, "transaction_cost_rel"), _get(config, "transaction_cost_abs"))
        env.setSlippage(_get(config, "slippage_rel"), _get(config, "slippage_abs"))
        return env
    raise NotImplementedError(f"Env type {_get(config, 'env_type')} not implemented")


def get_env_info(env):
    """The 13 accounting fields of the reference, as batched tensors (copies)."""
    return {
        "timestamp": env.timestamp.clone(),
        "riskInfo": env.checkRisk().clone(),
        "prices": env.currentPrices.clone(),
        "equity": env.equity.clone(),
        "cash": env.cash.clone(),
        "pnl": env.pnl.clone(),
        "balance": env.portfolio.balance.clone(),
        "availableMargin": env.availableMargin.clone(),
        "usedMargin": env.usedMargin.clone(),
        "borrowedAssetValue": env.borrowedAssetValue.clone(),
        "borrowedMargin": env.borrowedMargin.clone(),
        "ledger": env.ledger.clone(),
        "ledgerNormed": env.ledgerNormed.clone(),
    }


class SingleEnv:
    """A one-env view of a batched ``Env(n_envs=1)`` that speaks the reference's single-env dialect: numpy arrays
    without the leading batch axis and Python scalars, so that the reference's agent loop (``offpolicy_q.py:136-205``:
    ``prev_eq = env.equity``, ``env.step(transaction)``, ``info.brokerResponse.transactionUnits`` ...) runs on it
    unmodified.  Every read is a device-to-host copy: this is the compatibility path, not the fast one -- the batched
    ``Env`` with in-kernel rewards and ``DeviceReplay`` is."""
    _ARRAYS = ("currentPrices", "currentData", "ledger", "meanEntryPrices", "borrowedMarginLedger", "positionValues",
               "positionValuesFull", "pnlPositions", "ledgerFull", "ledgerNormed", "ledgerNormedFull",
               "ledgerAbsNormed", "ledgerAbsNormedFull")
    _SCALARS = ("cash", "equity", "assetValue", "pnl", "balance", "availableMargin", "usedMargin", "borrowedMargin",
                "borrowedAssetValue")

    def __init__(self, env):
        if env.N != 1:
            raise ValueError("SingleEnv wraps an Env built with n_envs=1")
        self._env = env

    def __getattr__(self, name):
        env = self.__dict__["_env"]
        if name in SingleEnv._ARRAYS:
            return getattr(env, name)[0].cpu().numpy()
        if name in SingleEnv._SCALARS:
            return float(getattr(env, name)[0])
        if name in ("timestamp", "currentTime"):
            return int(env.timestamp[0])
        return getattr(env, name)

    @staticmethod
    def _state(st):
        from ..utils.data import State
        return State(st.price[0].cpu().numpy(), st.portfolio[0].cpu().numpy(), int(st.timestamp[0]), _ring=st._ring)

    def _out(self, out):
        from ..utils.data import BrokerResponse, EnvInfo
        st, reward, done, info = out
        br = info.brokerResponse
        resp = BrokerResponse(br.event, int(br.timestamp[0]), br.transactionPrice[0].cpu().numpy(),
                              br.transactionUnits[0].cpu().numpy(), br.transactionCost[0].cpu().numpy(),
                              br.riskInfo[0].cpu().numpy(), bool(br.marginCall[0]))
        return self._state(st), float(reward[0]), bool(done[0]), EnvInfo(resp, info.dataEnd)

    def step(self, *args):
        import numpy as np
        import torch
        conv = [a if isinstance(a, (str, int)) and i == 0 and len(args) == 2
                else torch.as_tensor(np.asarray(a, dtype=np.float64)).reshape(1, -1) if len(args) == 1
                else torch.as_tensor(np.asarray(a, dtype=np.float64)).reshape(1) for i, a in enumerate(args)]
        return self._out(self._env.step(*conv))

    def reset(self):
        return self._state(self._env.reset())

    def checkRisk(self):
        return int(self._env.checkRisk()[0])
