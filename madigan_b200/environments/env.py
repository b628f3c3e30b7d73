"""Batched drop-in for Madigan's C++ ``Env`` (reference: madigan/environments/cpp/Env.h:17-256,
bound to Python in madigan/environments/cpp/env.cpp:843-1005).

Same member names as the reference; every scalar becomes an ``(N,)`` CUDA tensor, every
per-asset vector an ``(N,nA)`` tensor.  torch owns all state (structure-of-arrays,
``[rows][N]`` storage, fp64); every operation is one launch of a hand-written sm_100a
kernel through the C-ABI in ``include/madigan_b200.h``.  There is no CPU path.
"""
import ctypes as C

import numpy as np
import torch

from .. import _abi as A
from .._lib import check, lib
from ..utils.data import BrokerResponse, EnvInfo, State
from .data_source import BROKER_SLOTS, make_broker_table, make_param_table, make_params, make_reward, make_set_cdf


def _cfg_get(cfg, key, default=None):
    if cfg is None:
        return default
    try:
        if key in cfg:
            v = cfg[key]
            return default if v is None else v
    except TypeError:
        pass
    return getattr(cfg, key, default)


# MdgParams field of each broker setting (data_source.BROKER_SLOTS)
_P_FIELD = dict(init_cash="init_cash", required_margin="required_margin", maintenance_margin="maintenance_margin",
                slippage_rel="slippage_rel", slippage_abs="slippage_abs", transaction_cost_rel="tcost_rel",
                transaction_cost_abs="tcost_abs")


class Asset:
    """reference: environments/cpp/Assets.h:10-30."""

    def __init__(self, code):
        self.code = code
        self.name = code

    def __repr__(self):
        return f"Asset({self.code})"

    def __eq__(self, other):
        return getattr(other, "code", other) == self.code


class _View:
    """`env.portfolio` / `env.account` / `env.broker` / `env.dataSource`: the reference returns the
    C++ sub-objects (Env.h:51-55); with one account and one portfolio per env they all read the same
    ledger, so they are views of the env."""

    def __init__(self, env):
        self._env = env

    def __getattr__(self, name):
        return getattr(self._env, name)

    def currentData(self):
        return self._env.currentData

    def checkRisk(self, *a):
        return self._env.checkRisk(*a)


import contextlib

_NULL_CTX = contextlib.nullcontext()
# raw cudaStream_t of torch's current stream on a device: the C accessor is ~10x cheaper than building a Stream object
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None) or \
    (lambda idx: torch.cuda.current_stream(idx).cuda_stream)

# reset workspaces are scratch (no state between calls): one per (device, stream), shared by all Envs
_RESET_WS = {}


_RESET_NEED = {}


def _reset_workspace(lib_, P, n_envs, fill_ticks, device, stream_ptr=None, stream=None):
    nk = (P.n_normals, n_envs, fill_ticks)
    need = _RESET_NEED.get(nk)
    if need is None:
        need = _RESET_NEED[nk] = int(lib_.mdg_reset_workspace_bytes(C.byref(P), n_envs, fill_ticks))
    key = (device.index, _raw_stream(device.index) if stream_ptr is None else stream_ptr)
    ws = _RESET_WS.get(key)
    if ws is None or ws.numel() < need:
        # the 256-byte header {list length, exit ticket} must be zero before the first use; the kernels leave it zero
        ws = torch.zeros(need, dtype=torch.uint8, device=device)
        if stream is not None:  # zeroed on torch's current stream, used on the bound one
            stream.wait_stream(torch.cuda.current_stream(device))
            ws.record_stream(stream)
        _RESET_WS[key] = ws
    return ws


class Env:
    def __init__(self, dataSourceType, initCash=1_000_000., config=None, *, n_envs=None, device=None,
                 window=None, seed=None, env_offset=0, reward=None, param_sets=None, param_set=None,
                 broker_sets=None, param_set_weights=None):
        """``Env(data_source_type, init_cash, config)`` as the reference (env.cpp:843-849); the batched
        keys ``n_envs``, ``seed``, ``device``, ``window_length`` may come from ``config`` or keywords.
        ``reward``: None (env reward only) or a dict with ``reward_shaper_config``, ``nstep_return``,
        ``discount``, ``reduce_rewards`` to also compute the agent + shaped rewards in the step kernel.
        ``param_sets``: generator parameter sets, so that the envs of the slab tick different markets -- a list of
        ``data_source_config`` dicts for ``dataSourceType`` (same assets as the base config, other values), or an int
        ``S`` for S copies of the base config (to be edited through ``param_table``).  ``param_set``: the ``(N,)``
        integer set of every env, ``arange(N) % S`` by default.  Env e then equals, bit for bit, env e of a plain Env
        built from its set's config with the same ``n_envs``, ``seed`` and ``env_offset``
        (see ``make_param_table``, ``assign_param_sets``).
        ``broker_sets``: broker settings per parameter set, so that the envs also trade under different frictions -- a
        list of dicts over ``data_source.BROKER_SLOTS`` (a key a set omits takes the base value), or an int ``S`` for S
        copies of the base values (to be edited through ``broker_table``).  The base values are ``initCash`` and the
        same keys in ``config`` (0 when absent).  With ``param_sets`` its length must be S; without, the generator
        table is S copies of the base config.  One index per env selects both tables: env e then equals, bit for bit,
        env e of a plain Env of its set's config with ``setRequiredMargin / setMaintenanceMargin / setSlippage /
        setTransactionCost`` and ``initCash`` at its broker set's values (see ``make_broker_table``).
        ``param_set_weights``: S weights (finite, >= 0, positive sum) of a per-episode set draw, so that every episode
        runs in a market drawn anew (training that is robust to the market); needs ``param_sets`` or ``broker_sets``.
        Every reset of an env -- the fused auto-reset of ``step`` / ``step_actions`` / ``step_weights``, the separate
        one after a tearsheet or injected noise, and ``reset(mask)`` -- then draws the env's set with probability
        ``w[s] / sum(w)`` on the device, from Philox keyed on seed, global env id and the env's timestamp (see
        ``data_source.make_set_cdf``, ``set_param_set_weights``, ``episode_param_set``).  The first episode's set is
        ``param_set`` when given, else the draw at tick 0."""
        self._lib = lib()
        if not torch.cuda.is_available():
            raise RuntimeError("madigan_b200.Env needs a CUDA device (sm_100a); there is no CPU fallback")
        ds_cfg = _cfg_get(config, "data_source_config")
        self.N = int(n_envs if n_envs is not None else _cfg_get(config, "n_envs", 1))
        self.device = torch.device(device if device is not None else _cfg_get(config, "device", "cuda"))
        if self.device.type != "cuda":
            raise RuntimeError("madigan_b200.Env runs on CUDA devices only")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        pre = _cfg_get(config, "preprocessor_config")
        self.k = int(window if window is not None else _cfg_get(pre, "window_length", 64))
        self.seed = int(seed if seed is not None else _cfg_get(config, "seed", 0x6d61646967616e00))
        self.env_offset = int(env_offset)
        self._dataSourceType = dataSourceType
        self._initCash = float(initCash)
        self.P, self._asset_names = make_params(dataSourceType, ds_cfg, init_cash=initCash)
        self.nA = self.P.n_assets
        if self.P.ext_host is not None:  # SINE* sources: parameter / wave tables in device memory
            self._gen_ext = torch.from_numpy(self.P.ext_host).to(self.device)
            self.P.gen_ext, self.P.n_gen_ext = self._gen_ext.data_ptr(), self._gen_ext.numel()
        if reward is None and _cfg_get(config, "reward_shaper_config") is not None and _cfg_get(config, "in_kernel_rewards", False):
            ac = _cfg_get(config, "agent_config")
            reward = dict(reward_shaper_config=_cfg_get(config, "reward_shaper_config"),
                          nstep_return=_cfg_get(ac, "nstep_return", 1), discount=_cfg_get(ac, "discount", 0.99),
                          reduce_rewards=_cfg_get(ac, "reduce_rewards", False))
        if reward is None:
            self.R = make_reward(enabled=False)
        else:
            self.R = make_reward(reward.get("reward_shaper_config"), reward.get("nstep_return", 1),
                                 reward.get("discount", 0.99), reward.get("reduce_rewards", False),
                                 n_assets=self.nA)
        self.ra = 1 if self.R.reduce_rewards else self.nA
        self._alloc()
        self._PS = None  # MdgParamSets of an env with parameter sets
        self._btab, self._bptr = None, None  # broker table [MDG_BROKER_NPARAM][S] and its address (broker sets)
        if broker_sets is not None:
            btab = self._broker_table(config, broker_sets)
            S = btab.shape[1]
            if param_sets is None:
                param_sets = S
            elif (param_sets if isinstance(param_sets, int) else len(param_sets)) != S:
                raise ValueError(f"broker_sets has {S} sets, param_sets has "
                                 f"{param_sets if isinstance(param_sets, int) else len(param_sets)}")
        if param_set_weights is not None and param_sets is None:
            raise ValueError("param_set_weights needs param_sets or broker_sets")
        if param_sets is not None:
            self._init_param_sets(dataSourceType, ds_cfg, param_sets, param_set)
        self._cdf, self._weights, self._DRAW, self._pDRAW = None, None, None, None  # per-episode set draw
        if param_set_weights is not None:
            self.set_param_set_weights(param_set_weights)
        if broker_sets is not None:
            self._btab = torch.from_numpy(btab).to(self.device).contiguous()
            self._bptr = self._btab.data_ptr()
            for k_, v in self._broker_base.items():  # MdgParams holds the base values, as a plain Env's would
                setattr(self.P, _P_FIELD[k_], v)
        self.head = 0
        self.n_valid = 0
        self._gstep = 0
        self._version = 0
        self._derived_version = -1
        self.launches = 0  # kernels launched so far (bench.py's gpu_launches)
        self.flags = 0     # MdgLaunch.flags (validation: A.FLAG_FORCE_EXACT_GATE, A.FLAG_GENERIC_FILL)
        with torch.cuda.device(self.device):
            if self._PS is None:
                check(self._lib.mdg_init_state(C.byref(self.P), C.byref(self.R), C.byref(self._S),
                                               C.byref(self._launch())))
            else:  # with weights and no param_set, the first episode's set is the draw at tick 0
                check(self._lib.mdg_init_state_sets_draw(C.byref(self.P), C.byref(self.R), C.byref(self._S),
                                                         C.byref(self._launch()), self._pPS, self._bptr,
                                                         self._pDRAW if param_set is None else None))
            self.launches += 1
            # the constructor consumes one generator tick (Env.h:160); it is not a reset: it draws no set
            self._reset_launch(None, 1, False, None, None, draw=False)
        self.n_valid = 1

    # ------------------------------------------------------------------ allocation
    def _alloc(self):
        N, nA, k, dev = self.N, self.nA, self.k, self.device
        f8 = dict(dtype=torch.float64, device=dev)
        z = torch.zeros
        # price, ledger, mean_entry, borrowed are equally spaced views of ONE slab: the step kernel then fetches a
        # pair's eight state rows with a single 3-D TMA tensor copy (csrc/mdg_step_kernel.cuh, tm_state)
        slab = z((4, nA, N), **f8)
        self.t = dict(
            price=slab[0], ledger=slab[1], mean_entry=slab[2],
            borrowed=slab[3], cash=z((N,), **f8), gstate=z((max(1, self.P.n_gstate), N), **f8),
            timestamp=z((N,), dtype=torch.int64, device=dev), folds=z((5, N), **f8),
            reset_ts=z((N,), dtype=torch.int64, device=dev),
            shaper_A=z((self.ra, N), **f8), shaper_B=z((self.ra, N), **f8),
            nstep_ring=z((self.R.nstep, self.ra, N), **f8), nstep_len=z((N,), dtype=torch.int32, device=dev),
            obs_price=z((k, nA, N), **f8), obs_port=z((k, nA + 1, N), **f8),
            pre_price=z((N, k, nA), **f8),
            reward=z((N,), **f8), done=z((N,), dtype=torch.bool, device=dev),
            trans_price=z((nA, N), **f8), trans_units=z((nA, N), **f8), trans_cost=z((nA, N), **f8),
            risk=z((nA, N), dtype=torch.uint8, device=dev), margin_call=z((N,), dtype=torch.bool, device=dev),
            agent_reward=z((self.ra, N), **f8), shaped_reward=z((self.R.nstep, self.ra, N), **f8),
            n_popped=z((N,), dtype=torch.int32, device=dev),
            units=z((N, nA), **f8),
        )
        S = A.MdgState()
        for name in ("price", "ledger", "mean_entry", "borrowed", "cash", "gstate", "timestamp", "shaper_A",
                     "shaper_B", "nstep_ring", "nstep_len", "reset_ts", "folds"):
            setattr(S, name, self.t[name].data_ptr())
        self._S = S
        IO = A.MdgStepIO()
        for name in ("obs_price", "obs_port", "pre_price", "reward", "done", "trans_price", "trans_units",
                     "trans_cost", "risk", "margin_call", "agent_reward", "shaped_reward", "n_popped"):
            setattr(IO, name, self.t[name].data_ptr())
        self._IO = IO
        self._d = None
        self._stream, self._stream_ptr = None, None
        self._L = A.MdgLaunch(n_envs=N, env_offset=self.env_offset, seed=self.seed, window=k)
        # byref() objects of the persistent descriptors, built once (each byref() call costs ~0.3 us)
        self._pP, self._pR, self._pS = C.byref(self.P), C.byref(self.R), C.byref(self._S)
        self._pIO, self._pL = C.byref(self._IO), C.byref(self._L)
        # zero-copy (N, nA) views of the [nA][N] output tensors, built once
        t = self.t
        self._resp = BrokerResponse("", t["timestamp"], t["trans_price"].t(), t["trans_units"].t(),
                                    t["trans_cost"].t(), t["risk"].t(), t["margin_call"])
        self._info = EnvInfo(self._resp, False)
        self._states = [None] * k
        self._want_multi, self._want_single = torch.Size((N, nA)), torch.Size((N,))
        self._done_u8 = t["done"].view(torch.uint8)

    # ------------------------------------------------------------------ generator parameter sets
    def _init_param_sets(self, ds_type, ds_cfg, param_sets, param_set):
        if isinstance(param_sets, bool) or not isinstance(param_sets, (int, list, tuple)):
            raise TypeError("param_sets must be a list of data_source_config dicts or an int")
        if isinstance(param_sets, int):
            if param_sets < 1:
                raise ValueError("param_sets must be >= 1")
            param_sets = [ds_cfg] * param_sets
        table = make_param_table(ds_type, ds_cfg, param_sets)  # (nA, NPARAM, S), set-minor
        S = table.shape[2]
        # [nA][NPARAM][S] storage, as MdgParamSets.p reads it
        self._ptab = torch.from_numpy(table).to(self.device).contiguous()
        self._pset = torch.arange(self.N, device=self.device, dtype=torch.int32) % S
        if param_set is not None:
            self.assign_param_sets(param_set)
        self._PS = A.MdgParamSets(p=self._ptab.data_ptr(), set_of_env=self._pset.data_ptr(), n_sets=S)
        self._pPS = C.byref(self._PS)
        # set of the episode that each env's last drawing reset finished (-1: none yet)
        self._epset = torch.full((self.N,), -1, dtype=torch.int32, device=self.device)

    def _broker_table(self, config, broker_sets):
        """(MDG_BROKER_NPARAM, S) numpy table of ``broker_sets``; resolves the base values"""
        if isinstance(broker_sets, bool) or not isinstance(broker_sets, (int, list, tuple)):
            raise TypeError("broker_sets must be a list of dicts over data_source.BROKER_SLOTS or an int")
        if isinstance(broker_sets, int):
            if broker_sets < 1:
                raise ValueError("broker_sets must be >= 1")
            broker_sets = [{}] * broker_sets
        base = {k: float(_cfg_get(config, k, 0.)) for k in BROKER_SLOTS[1:]}
        self._broker_base = dict(init_cash=self._initCash, **base)
        return make_broker_table(self._broker_base, broker_sets)

    @property
    def broker_table(self):
        """``(S, MDG_BROKER_NPARAM)`` fp64 device view of the broker sets: ``broker_table[s, k]`` is setting k
        (``data_source.BROKER_SLOTS``) of set s.  Writable in place, with ``param_table``'s semantics: every launch reads
        it as it stands on the env's stream, so a change takes effect at the next step or reset.  After an in-place
        write, call ``invalidate()`` before reading derived properties (``availableMargin``, ``usedMargin``,
        ``checkRisk()``), which are cached per step.  None without broker sets."""
        return None if self._btab is None else self._btab.t()

    def _per_env(self, k):
        """(N,) broker setting k of every env's set (out-of-range set indices clamp as in the kernels)"""
        S = self._btab.shape[1]
        with self._copy_ctx():
            s = self._pset.long()
            return self._btab[k][torch.where((s < 0) | (s >= S), S - 1, s)]

    def _set_broker(self, **values):
        """the setters of an Env with broker sets: the field of every set, on the env's stream"""
        if self._stream is not None:
            self._stream.wait_stream(torch.cuda.current_stream(self.device))
        with self._device_ctx(), self._copy_ctx():
            for k_, v in values.items():
                self._btab[BROKER_SLOTS.index(k_)].fill_(v)

    @property
    def n_param_sets(self):
        """Number of generator parameter sets (0: the env was built without ``param_sets``)."""
        return 0 if self._PS is None else int(self._PS.n_sets)

    @property
    def param_table(self):
        """``(S, nA, MDG_GEN_NPARAM)`` fp64 device view of the parameter sets: ``param_table[s, i, j]`` is slot j
        (``data_source.PARAM_SLOTS``) of asset i in set s.  Writable in place; every launch reads the table as it
        stands on the env's stream, so a change takes effect at the next step or reset and an episode in progress
        continues under the new values.  None without parameter sets."""
        return None if self._PS is None else self._ptab.permute(2, 0, 1)

    @property
    def param_set(self):
        """``(N,)`` int32: the parameter set of every env (read it; change it with ``assign_param_sets``)."""
        return None if self._PS is None else self._pset

    @property
    def param_set_weights(self):
        """The normalised weights ``w / sum(w)`` of the per-episode set draw (a float64 numpy array of S), or None when
        the draw is off."""
        return None if self._weights is None else self._weights.copy()

    @property
    def episode_param_set(self):
        """``(N,)`` int32 device view: for the envs that reset in the last call with the set draw on, the set of the
        episode that just finished; the other entries are unchanged, and -1 until an env's first such reset.  With
        ``torch.bincount`` over ``episode_param_set[done]`` it attributes finished episodes to markets.  None without
        parameter sets."""
        return None if self._PS is None else self._epset

    def set_param_set_weights(self, weights):
        """Turn the per-episode set draw on with ``weights`` (S numbers: finite, >= 0, positive sum; see
        ``data_source.make_set_cdf``), change its weights, or turn it off with None (the sets then stay as they are
        through resets).  Validates on the host, then writes the draw's table on the env's stream: the change takes
        effect at the next reset (a curriculum over markets), and episodes in progress keep their sets."""
        if self._PS is None:
            raise RuntimeError("this Env was built without param_sets / broker_sets")
        if weights is None:
            self._cdf, self._weights, self._DRAW, self._pDRAW = None, None, None, None
            return
        S = int(self._PS.n_sets)
        cdf = make_set_cdf(weights, S)
        w = np.asarray(weights, dtype=np.float64)
        if self._stream is not None:
            self._stream.wait_stream(torch.cuda.current_stream(self.device))
        with self._device_ctx(), self._copy_ctx():
            if self._cdf is None:
                self._cdf = torch.empty((S,), dtype=torch.float64, device=self.device)
            self._cdf.copy_(torch.from_numpy(cdf))
        self._weights = w / w.sum()
        self._DRAW = A.MdgSetDraw(cdf=self._cdf.data_ptr(), episode_set=self._epset.data_ptr())
        self._pDRAW = C.byref(self._DRAW)

    def assign_param_sets(self, ids, mask=None):
        """Set the parameter set of every env (``mask=None``) or of the envs where ``mask`` (N,) is true to ``ids``
        (an (N,) integer tensor/array, or one int).  Checks the range with one host synchronisation (a setup call, not
        one for the hot loop), then writes on the env's stream.  The change takes effect at the next launch: an episode
        in progress continues under the new values.  For a new market per episode, use ``param_set_weights`` (or
        ``set_param_set_weights``): every reset then draws the env's set on the device, inside the fused auto-reset.
        This method stays a manual override; with the draw on, the next reset of an env replaces what it wrote."""
        if self._PS is None and not hasattr(self, "_pset"):
            raise RuntimeError("this Env was built without param_sets")
        S = self._ptab.shape[2]
        with self._device_ctx():
            ids = torch.as_tensor(ids, device=self.device)
            if ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool:
                raise ValueError(f"parameter set ids must be integers, got {ids.dtype}")
            if ids.dim() == 0:
                ids = ids.expand(self.N)
            if tuple(ids.shape) != (self.N,):
                raise ValueError(f"parameter set ids must have shape ({self.N},), got {tuple(ids.shape)}")
            lo, hi = (int(v) for v in torch.aminmax(ids))
            if lo < 0 or hi >= S:
                raise ValueError(f"parameter set ids must be in [0, {S}), got [{lo}, {hi}]")
            m = None
            if mask is not None:
                m = torch.as_tensor(mask, device=self.device)
                if tuple(m.shape) != (self.N,):
                    raise ValueError(f"mask must have shape ({self.N},)")
                m = m.to(torch.bool)
            if self._stream is not None:
                self._stream.wait_stream(torch.cuda.current_stream(self.device))
            with self._copy_ctx():
                if m is None:
                    self._pset.copy_(ids)
                else:
                    self._pset.copy_(torch.where(m, ids.to(torch.int32), self._pset))

    def _launch(self, mode=A.MODE_HOLD, asset_idx=0):
        """The (persistent) launch descriptor, refreshed for this call: the host path of a step is a handful of
        attribute writes and one ctypes call, so that Python can enqueue steps faster than the GPU retires them."""
        L = self._L
        L.head = self.head
        L.mode = mode
        L.asset_idx = asset_idx
        L.nstep_pos = self._gstep % self.R.nstep
        L.seed = self.seed
        L.env_offset = self.env_offset
        L.stream = self._sptr()
        L.flags = self.flags
        return L

    def _sptr(self):
        """cudaStream_t every launch of this env goes to: the bound stream, else torch's current stream."""
        return self._stream_ptr if self._stream_ptr is not None else _raw_stream(self.device.index)

    def _copy_ctx(self):
        """`with` context for torch ops that must run on this env's stream (staging copies)."""
        if self._stream is None or _raw_stream(self.device.index) == self._stream_ptr:
            return _NULL_CTX  # torch's current stream already is the env's stream
        return torch.cuda.stream(self._stream)

    def bind_stream(self, stream):
        """Pin this env's launches to ``stream`` (a torch.cuda.Stream; None = torch's current stream again).
        A driver that steps several slabs round-robin, one stream per slab, then needs no stream context manager
        per call (which costs more host time than the step itself).  EVERY launch of the env follows the binding --
        step, reset, derived accounting, window / time materialisation, episode statistics, and the kernels of a
        DeviceReplay built on it -- and so do the staging copies of host inputs.  Tensors the env returns are
        produced on that stream: a consumer on another stream must wait for it (``other.wait_stream(stream)``)."""
        self._stream = stream
        self._stream_ptr = None if stream is None else stream.cuda_stream

    def _device_ctx(self):
        """`with` context selecting this env's device only when it is not already current (saves ~5 us per call)."""
        if torch.cuda.current_device() == self.device.index:
            return _NULL_CTX
        return torch.cuda.device(self.device)

    def _noise(self, normals, uniforms):
        keep = []
        ptrs = []
        for x in (normals, uniforms):
            if x is None:
                ptrs.append(None)
                continue
            x = torch.as_tensor(x, dtype=torch.float64).to(self.device).contiguous()
            keep.append(x)
            ptrs.append(x.data_ptr())
        return ptrs[0], ptrs[1], keep

    # ------------------------------------------------------------------ setters (Env.h:94-111)
    # With broker sets, each setter writes its field into every set: the Env's envs all take the value.
    def setRequiredMargin(self, reqM):
        self.P.required_margin = float(reqM)
        if self._btab is not None:
            self._set_broker(required_margin=float(reqM))
        self._version += 1

    def setMaintenanceMargin(self, mainM):
        self.P.maintenance_margin = float(mainM)
        if self._btab is not None:
            self._set_broker(maintenance_margin=float(mainM))
        self._version += 1

    def setSlippage(self, slippagePct=0., slippageAbs=0.):
        self.P.slippage_rel, self.P.slippage_abs = float(slippagePct), float(slippageAbs)
        if self._btab is not None:
            self._set_broker(slippage_rel=float(slippagePct), slippage_abs=float(slippageAbs))

    def setTransactionCost(self, transactionPct=0., transactionAbs=0.):
        self.P.tcost_rel, self.P.tcost_abs = float(transactionPct), float(transactionAbs)
        if self._btab is not None:
            self._set_broker(transaction_cost_rel=float(transactionPct), transaction_cost_abs=float(transactionAbs))

    # ------------------------------------------------------------------ reset / step
    def _reset_launch(self, mask, fill_ticks, clear_nstep, normals, uniforms, draw=True):
        io = self._IO
        if normals is None and uniforms is None:
            io.normals = io.uniforms = None
            keep = None
        else:
            io.normals, io.uniforms, keep = self._noise(normals, uniforms)
        io.units = None
        m = None
        if mask is self.t["done"]:
            m = self._done_u8
        elif mask is not None:
            m = torch.as_tensor(mask)
            if m.dtype == torch.bool:
                m = m.view(torch.uint8)  # same bytes, no conversion kernel
            m = m.to(device=self.device, dtype=torch.uint8).contiguous()
            if tuple(m.shape) != (self.N,):
                raise ValueError(f"mask must have shape ({self.N},)")
        ws = _reset_workspace(self._lib, self.P, self.N, int(fill_ticks), self.device, self._stream_ptr, self._stream)
        if self._PS is None:
            check(self._lib.mdg_reset_ws(C.byref(self.P), C.byref(self._S), C.byref(io), C.byref(self._launch()),
                                         None if m is None else m.data_ptr(), int(fill_ticks), int(clear_nstep),
                                         ws.data_ptr(), ws.numel()))
        else:
            check(self._lib.mdg_reset_ws_sets_draw(C.byref(self.P), C.byref(self._S), C.byref(io),
                                                   C.byref(self._launch()), None if m is None else m.data_ptr(),
                                                   int(fill_ticks), int(clear_nstep), ws.data_ptr(), ws.numel(),
                                                   self._pPS, self._bptr, self._pDRAW if draw else None))
        self.launches += 2  # list scan + refill kernel
        self._version += 1
        del keep

    def _state(self):
        st = self._states[self.head]
        if st is None:  # one State (views of ring slot `head`) per slot, built on first use
            t = self.t
            st = State(t["obs_price"][self.head].t(), t["obs_port"][self.head].t(), t["timestamp"], _ring=(self, 0))
            self._states[self.head] = st
        return st

    def reset(self, mask=None, fill_history=False, normals=None, uniforms=None):
        """Env::reset (Env.h:181-187).  ``mask``: (N,) bool/uint8, only those envs (None = all).
        ``fill_history``: also run the k-1 no-action ticks of ``initialize_history``
        (reference: utils/preprocessor.py:191-194) so the whole window belongs to the new episode.
        Returns the newest State row."""
        fill = self.k if fill_history else 1
        with self._device_ctx():
            self._reset_launch(mask, fill, True, normals, uniforms)
        if mask is None:
            self.n_valid = fill
        return self._state()

    def step(self, *args, normals=None, uniforms=None, auto_reset=False, tearsheet=None, results=None):
        """``step()`` hold (Env.h:189-204); ``step(units)`` with units (N,nA) (Env.h:206-230);
        ``step(assetIdx|assetCode, units)`` with units (N,) (Env.h:232-256, env.cpp:995-1005).
        Returns ``(State, reward (N,), done (N,) bool, EnvInfo)``; the tensors are views of live
        buffers that the next call overwrites (same aliasing as the reference's Eigen maps).
        ``tearsheet``: a ``utils.metrics.EpisodeTearsheet`` that records the step before any auto-reset.
        ``results``: a ``utils.metrics.EpisodeResults`` of this Env (needs ``auto_reset=True``, excludes ``tearsheet``)
        that records the step and harvests every finished episode into its per-set table before the refill."""
        self._check_results(results, auto_reset, tearsheet)
        asset_idx = 0
        if len(args) == 0:
            mode, units = A.MODE_HOLD, None
        elif len(args) == 1:
            mode, units = A.MODE_MULTI, args[0]
        elif len(args) == 2:
            mode, units = A.MODE_SINGLE, args[1]
            a = args[0]
            asset_idx = self._asset_names.index(a) if isinstance(a, str) else int(a)
            if not 0 <= asset_idx < self.nA:
                raise IndexError("asset index out of range")
        else:
            raise TypeError("step() takes at most (assetIdx, units)")
        io = self._IO
        with self._device_ctx():
            if units is not None:
                u = units if (isinstance(units, torch.Tensor) and units.dtype == torch.float64) \
                    else torch.as_tensor(units, dtype=torch.float64)
                want = self._want_multi if mode == A.MODE_MULTI else self._want_single
                if u.shape != want:
                    if self.N == 1 and u.dim() == len(want) - 1:
                        u = u.unsqueeze(0)
                    if u.shape != want:
                        raise ValueError(f"units must have shape {tuple(want)}, got {tuple(u.shape)}")
                if not u.is_cuda or u.device != self.device or not u.is_contiguous():
                    dst = self.t["units"] if mode == A.MODE_MULTI else self.t["units"].view(-1)[:self.N]
                    with self._copy_ctx():
                        dst.copy_(u, non_blocking=True)  # H2D from (pinned) host memory, async on the env's stream
                    u = dst
                io.units = u.data_ptr()
            else:
                io.units = None
            if normals is None and uniforms is None:
                io.normals = io.uniforms = None
                keep = None
            else:
                io.normals, io.uniforms, keep = self._noise(normals, uniforms)
            head0 = self.head
            self.head = (self.head + 1) % self.k
            L = self._launch(mode, asset_idx)
            self.head = head0  # the ring head moves only once the launch has been accepted
            if auto_reset and keep is None and tearsheet is None:  # step + masked reset + history fill in one trip through the binding
                ws = _reset_workspace(self._lib, self.P, self.N, self.k, self.device, self._stream_ptr, self._stream)
                if self._PS is None and results is None:
                    check(self._lib.mdg_step_autoreset(self._pP, self._pR, self._pS, self._pIO, self._pL, self.k, 1,
                                                       ws.data_ptr(), ws.numel()))
                else:
                    self._step_autoreset_call(ws, results)
                # step kernel (appends the finished envs to the list) [+ results record] + refill kernel
                self.launches += 2 if results is None else 3
                auto_reset = False
            else:
                if self._PS is None:
                    check(self._lib.mdg_step(self._pP, self._pR, self._pS, self._pIO, self._pL))
                else:
                    self._step_call()
                self.launches += 1
            self.head = L.head
            self.n_valid = min(self.k, self.n_valid + 1)
            if mode != A.MODE_HOLD and self.R.shaper != A.SHAPER_OFF:
                self._gstep += 1
            self._version += 1
            if tearsheet is not None:
                tearsheet.update()
            if auto_reset:
                self._record_results(results)
                self._reset_launch(self.t["done"], self.k, True, None, None)
        t = self.t
        return self._state(), t["reward"], t["done"], self._info

    def _check_results(self, results, auto_reset, tearsheet=None):
        if results is None:
            return
        if getattr(results, "env", None) is not self:
            raise ValueError("results were built on another Env")
        if not auto_reset:
            raise ValueError("results= needs auto_reset=True: an episode's row is harvested as the env resets")
        if tearsheet is not None:
            raise ValueError("results= and tearsheet= cannot be combined: the results own their recorder")

    def _record_results(self, results):
        """the record + harvest kernel alone, between a step and a separate reset of the finished envs"""
        if results is None:
            return
        check(self._lib.mdg_episode_results_record(self._pP, self._pS, self._pIO,
                                                   self._pPS if self._PS is not None else None, self._bptr,
                                                   results._pR, self._sptr()))
        results._recorded()
        self.launches += 1

    def _step_call(self):
        if self._PS is None:
            check(self._lib.mdg_step(self._pP, self._pR, self._pS, self._pIO, self._pL))
        else:
            check(self._lib.mdg_step_sets_broker(self._pP, self._pR, self._pS, self._pIO, self._pL, self._pPS,
                                                 self._bptr))

    def _step_autoreset_call(self, ws, results=None):
        if results is not None:  # step, record + harvest, refill
            check(self._lib.mdg_step_autoreset_results(self._pP, self._pR, self._pS, self._pIO, self._pL, self.k, 1,
                                                       ws.data_ptr(), ws.numel(),
                                                       self._pPS if self._PS is not None else None, self._bptr,
                                                       self._pDRAW, results._pR))
            results._recorded()
        elif self._PS is None:
            check(self._lib.mdg_step_autoreset(self._pP, self._pR, self._pS, self._pIO, self._pL, self.k, 1,
                                               ws.data_ptr(), ws.numel()))
        else:
            check(self._lib.mdg_step_autoreset_sets_draw(self._pP, self._pR, self._pS, self._pIO, self._pL, self.k,
                                                         1, ws.data_ptr(), ws.numel(), self._pPS, self._bptr,
                                                         self._pDRAW))

    def step_actions(self, actions, *, action_atoms, unit_size, normals=None, uniforms=None, auto_reset=False, results=None):
        """``env.step(agent.action_to_transaction(actions))`` in one launch: ``actions`` is an (N, nA) integer tensor
        of discrete actions in [0, action_atoms); the kernel converts them to transaction units exactly as
        ``DQN.action_to_transaction`` does (modelling/algorithm/dqn.py:160-179 -- ``(a - atoms//2) * unit_size *
        availableMargin / price``, action 0 closes an open position) and steps.  The action matrix is 1 byte per
        asset instead of the 8 of a units matrix.  ``results``: as in ``step``.  Returns what ``step(units)`` returns."""
        self._check_results(results, auto_reset)
        io = self._IO
        with self._device_ctx():
            a = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(actions)
            if a.dtype != torch.int8:
                a = a.to(torch.int8)
            if a.shape != self._want_multi:
                if self.N == 1 and a.dim() == 1:
                    a = a.unsqueeze(0)
                if a.shape != self._want_multi:
                    raise ValueError(f"actions must have shape {tuple(self._want_multi)}, got {tuple(a.shape)}")
            if not a.is_cuda or a.device != self.device or not a.is_contiguous():
                if "actions" not in self.t:
                    self.t["actions"] = torch.empty((self.N, self.nA), dtype=torch.int8, device=self.device)
                with self._copy_ctx():
                    self.t["actions"].copy_(a, non_blocking=True)
                a = self.t["actions"]
            io.units = None
            io.actions = a.data_ptr()
            try:
                if normals is None and uniforms is None:
                    io.normals = io.uniforms = None
                    keep = None
                else:
                    io.normals, io.uniforms, keep = self._noise(normals, uniforms)
                head0 = self.head
                self.head = (self.head + 1) % self.k
                L = self._launch(A.MODE_MULTI, 0)
                self.head = head0
                L.action_atoms, L.unit_size = int(action_atoms), float(unit_size)
                if auto_reset and keep is None:
                    ws = _reset_workspace(self._lib, self.P, self.N, self.k, self.device, self._stream_ptr, self._stream)
                    self._step_autoreset_call(ws, results)
                    self.launches += 1 if results is None else 2  # + [the results record and] the refill kernel
                    auto_reset = False
                else:
                    self._step_call()
            finally:
                io.actions = None
            self.head = L.head
            self.n_valid = min(self.k, self.n_valid + 1)
            self.launches += 1
            if self.R.shaper != A.SHAPER_OFF:
                self._gstep += 1
            self._version += 1
            if auto_reset:
                self._record_results(results)
                self._reset_launch(self.t["done"], self.k, True, None, None)
        t = self.t
        return self._state(), t["reward"], t["done"], self._info

    def step_weights(self, weights, *, normals=None, uniforms=None, auto_reset=False, results=None):
        """``env.step(agent.action_to_transaction(weights))`` in one launch for a DDPG-style actor: ``weights`` is an
        (N, nA+1) real tensor of target portfolio weights, cash first; the kernel converts them to transaction units
        exactly as ``DDPG.action_to_transaction`` does (modelling/algorithm/ddpg.py:182-207 -- ``desired = w / w.sum()``
        in fp32, ``units = (desired - ledgerNormedFull)[1:] * equity / currentPrices``) and steps.  4 bytes per weight
        cross to the device instead of 8 per unit.  ``results``: as in ``step``.  Returns what ``step(units)`` returns."""
        self._check_results(results, auto_reset)
        io = self._IO
        with self._device_ctx():
            w = weights if isinstance(weights, torch.Tensor) else torch.as_tensor(weights)
            if w.dtype != torch.float32:
                w = w.to(torch.float32)
            want = torch.Size((self.N, self.nA + 1))
            if w.shape != want:
                if self.N == 1 and w.dim() == 1:
                    w = w.unsqueeze(0)
                if w.shape != want:
                    raise ValueError(f"weights must have shape {tuple(want)}, got {tuple(w.shape)}")
            if not w.is_cuda or w.device != self.device or not w.is_contiguous():
                if "weights" not in self.t:
                    self.t["weights"] = torch.empty((self.N, self.nA + 1), dtype=torch.float32, device=self.device)
                with self._copy_ctx():
                    self.t["weights"].copy_(w, non_blocking=True)
                w = self.t["weights"]
            io.units = None
            io.weights = w.data_ptr()
            try:
                if normals is None and uniforms is None:
                    io.normals = io.uniforms = None
                    keep = None
                else:
                    io.normals, io.uniforms, keep = self._noise(normals, uniforms)
                head0 = self.head
                self.head = (self.head + 1) % self.k
                L = self._launch(A.MODE_MULTI, 0)
                self.head = head0
                if auto_reset and keep is None:
                    ws = _reset_workspace(self._lib, self.P, self.N, self.k, self.device, self._stream_ptr, self._stream)
                    self._step_autoreset_call(ws, results)
                    self.launches += 1 if results is None else 2  # + [the results record and] the refill kernel
                    auto_reset = False
                else:
                    self._step_call()
            finally:
                io.weights = None
            self.head = L.head
            self.n_valid = min(self.k, self.n_valid + 1)
            self.launches += 1
            if self.R.shaper != A.SHAPER_OFF:
                self._gstep += 1
            self._version += 1
            if auto_reset:
                self._record_results(results)
                self._reset_launch(self.t["done"], self.k, True, None, None)
        t = self.t
        return self._state(), t["reward"], t["done"], self._info

    # ------------------------------------------------------------------ in-kernel rewards
    @property
    def agent_reward(self):
        """(N, ra) per-asset (or reduced) log-return reward of the last step (offpolicy_q.py:152-164)."""
        return self.t["agent_reward"].t()

    @property
    def shaped_reward(self):
        """(nstep, N, ra): rewards popped from the n-step buffer by the last step, row j = j-th pop;
        ``n_popped`` (N,) says how many rows are valid (nstep_buffer.py:342-361, replay_buffer.py:68-80)."""
        return self.t["shaped_reward"].transpose(1, 2)

    @property
    def n_popped(self):
        return self.t["n_popped"]

    def reset_shaper_state(self):
        """Zero the DSR/DDR moments (they persist across episode resets in the reference, A18)."""
        self.t["shaper_A"].zero_()
        self.t["shaper_B"].zero_()

    # ------------------------------------------------------------------ derived accounting
    def _derived(self):
        if self._derived_version == self._version and self._d is not None:
            return self._d
        N, nA, dev = self.N, self.nA, self.device
        if self._d is None:
            f8 = dict(dtype=torch.float64, device=dev)
            d = {n: torch.empty((N,), **f8) for n in ("equity", "asset_value", "pnl", "balance", "available_margin",
                                                      "used_margin", "borrowed_margin", "borrowed_asset_value")}
            d["risk"] = torch.empty((N,), dtype=torch.uint8, device=dev)
            for n in ("position_values", "pnl_positions", "ledger_normed", "ledger_abs_normed"):
                d[n] = torch.empty((nA, N), **f8)
            for n in ("ledger_normed_full", "ledger_abs_normed_full", "position_values_full", "ledger_full"):
                d[n] = torch.empty((nA + 1, N), **f8)
            self._d = d
            D = A.MdgDerived()
            for n, v in d.items():
                setattr(D, n, v.data_ptr())
            self._D = D
        with torch.cuda.device(self.device):
            if self._PS is None:
                check(self._lib.mdg_derived(C.byref(self.P), C.byref(self._S), C.byref(self._D),
                                            C.byref(self._launch())))
            else:
                check(self._lib.mdg_derived_sets_broker(C.byref(self.P), C.byref(self._S), C.byref(self._D),
                                                        C.byref(self._launch()), self._pPS, self._bptr))
        self.launches += 1
        self._derived_version = self._version
        return self._d

    def invalidate(self):
        """Call after writing into a live state view (e.g. ``env.currentPrices[:, 1] = 4``): drops the
        cached derived accounting and recomputes the portfolio folds the step kernel carries in state."""
        self._version += 1
        with torch.cuda.device(self.device):
            check(self._lib.mdg_refresh_folds(C.byref(self.P), C.byref(self._S), C.byref(self._launch())))
        self.launches += 1

    # live views of state (reference: return_value_policy::reference, env.cpp:897-913)
    @property
    def currentPrices(self): return self.t["price"].t()
    @property
    def currentData(self): return self.t["price"].t()
    @property
    def ledger(self): return self.t["ledger"].t()
    @property
    def meanEntryPrices(self): return self.t["mean_entry"].t()
    @property
    def borrowedMarginLedger(self): return self.t["borrowed"].t()
    @property
    def cash(self): return self.t["cash"]
    @property
    def timestamp(self): return self.t["timestamp"]
    @property
    def currentTime(self): return self.t["timestamp"]
    # derived (Portfolio.cpp:140-235)
    @property
    def equity(self): return self._derived()["equity"]
    @property
    def assetValue(self): return self._derived()["asset_value"]
    @property
    def pnl(self): return self._derived()["pnl"]
    @property
    def balance(self): return self._derived()["balance"]
    @property
    def availableMargin(self): return self._derived()["available_margin"]
    @property
    def usedMargin(self): return self._derived()["used_margin"]
    @property
    def borrowedMargin(self): return self._derived()["borrowed_margin"]
    @property
    def borrowedAssetValue(self): return self._derived()["borrowed_asset_value"]
    @property
    def positionValues(self): return self._derived()["position_values"].t()
    @property
    def positionValuesFull(self): return self._derived()["position_values_full"].t()
    @property
    def pnlPositions(self): return self._derived()["pnl_positions"].t()
    @property
    def ledgerFull(self): return self._derived()["ledger_full"].t()
    @property
    def ledgerNormed(self): return self._derived()["ledger_normed"].t()
    @property
    def ledgerNormedFull(self): return self._derived()["ledger_normed_full"].t()
    @property
    def ledgerAbsNormed(self): return self._derived()["ledger_abs_normed"].t()
    @property
    def ledgerAbsNormedFull(self): return self._derived()["ledger_abs_normed_full"].t()

    def checkRisk(self):
        """Portfolio::checkRisk() per env -> (N,) uint8 RiskInfo (Portfolio.cpp:243-252)."""
        return self._derived()["risk"]

    def dataEnd(self):
        return False  # synthetic sources never end (DataSource.h)

    # static info
    @property
    def nAssets(self): return self.nA
    @property
    def nFeats(self): return self.nA  # nFeats()==nAssets() for every synthetic source (DataSource.h:231)
    @property
    def n_envs(self): return self.N
    @property
    def assets(self): return [Asset(n) for n in self._asset_names]
    @property
    def isDateTime(self): return False
    # with broker sets: the (N,) values of every env's set
    @property
    def initCash(self): return self._initCash if self._btab is None else self._per_env(0)
    @property
    def requiredMargin(self): return self.P.required_margin if self._btab is None else self._per_env(1)
    @property
    def maintenanceMargin(self): return self.P.maintenance_margin if self._btab is None else self._per_env(2)
    @property
    def dataSourceType(self): return self._dataSourceType
    @property
    def dataSource(self): return _View(self)
    @property
    def portfolio(self): return _View(self)
    @property
    def account(self): return _View(self)
    @property
    def broker(self): return _View(self)

    # ------------------------------------------------------------------ window / stats / checkpoint
    def window(self, norm_type=None, dtype=torch.float64, channels_first=False, n_valid=None, out=None,
               transform=A.XFORM_NONE, stride=1, age0=0, out_feat_offset=None):
        """Materialise the price window ``(N, n_valid, nF)`` (or ``(N, nF, n_valid)``) from the observation
        ring, normalised as ``make_normalizer(norm_type)`` (reference: utils/preprocessor.py:53-107,183-189).
        ``transform``: ``XFORM_PAIR_RATIO`` (StackerDiscretePairs, nF 2 -> 1) or ``XFORM_RETURNS``
        (StackerDiscreteReturns, nF -> nF-1).  ``stride`` / ``age0``: a dilated window -- row s is the ring row of age
        ``age0 + (n_valid-1-s)*stride`` (MultiStackerDiscrete); with ``out_feat_offset`` the window is written into
        the column block ``[offset, offset + nF)`` of a wider ``out`` (the concatenation over dilations)."""
        from ..utils.preprocessor import NORM_TYPES
        nv = self.n_valid if n_valid is None else int(n_valid)
        norm = NORM_TYPES[norm_type]
        f_out = 1 if transform == A.XFORM_PAIR_RATIO else (self.nA - 1 if transform == A.XFORM_RETURNS else self.nA)
        shape = (self.N, f_out, nv) if channels_first else (self.N, nv, f_out)
        if out is None:
            out = torch.empty(shape, dtype=dtype, device=self.device)
        dt = A.DTYPE_F32 if out.dtype == torch.float32 else A.DTYPE_F64
        ftot = 0
        if out_feat_offset is not None:
            ftot = out.shape[1] if channels_first else out.shape[2]
        self._window_launch(self.t["obs_price"], self.t["pre_price"], 0, self.nA, nv, norm, out, dt,
                            A.LAYOUT_NFK if channels_first else A.LAYOUT_NKF, transform, stride, age0, ftot,
                            out_feat_offset or 0)
        return out

    def _window_launch(self, ring, prefix, flat_prefix, n_feats, nv, norm, out, dt, layout, transform=A.XFORM_NONE,
                       stride=1, age0=0, ftot=0, foff=0):
        w = A.MdgWindow(ring=ring.data_ptr(), prefix=None if prefix is None else prefix.data_ptr(),
                        timestamp=self.t["timestamp"].data_ptr(), reset_ts=self.t["reset_ts"].data_ptr(),
                        n_envs=self.N, n_feats=n_feats, window=self.k, head=self.head, n_valid=nv, norm_type=norm,
                        flat_prefix=flat_prefix, out_dtype=dt, out_layout=layout, out=out.data_ptr(),
                        stream=self._sptr(), transform=transform, stride=int(stride), age0=int(age0),
                        out_feats_total=int(ftot), out_feat_offset=int(foff))
        with torch.cuda.device(self.device):
            check(self._lib.mdg_materialise_window(C.byref(w)))
        self.launches += 1

    def portfolio_window(self, n_valid=None, stride=1, age0=0):
        """(N, n_valid, nA+1) window of ledgerNormedFull rows, oldest first (rows older than the env's last
        reset are the flat portfolio [1,0,...,0] of its history fill)."""
        nv = self.n_valid if n_valid is None else int(n_valid)
        out = torch.empty((self.N, nv, self.nA + 1), dtype=torch.float64, device=self.device)
        self._window_launch(self.t["obs_port"], None, 1, self.nA + 1, nv, A.NORM_NONE, out, A.DTYPE_F64, A.LAYOUT_NKF,
                            A.XFORM_NONE, stride, age0)
        return out

    def time_window(self, n_valid=None, stride=1, age0=0):
        nv = self.n_valid if n_valid is None else int(n_valid)
        out = torch.empty((self.N, nv), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.mdg_materialise_time(self.t["timestamp"].data_ptr(), self.N, nv, out.data_ptr(),
                                                 self._sptr()))
        self.launches += 1
        if stride != 1 or age0 != 0:  # timestamp[e] - (age0 + (nv-1-s)*stride): every ring row is one generator tick
            with self._copy_ctx():
                ages = age0 + (nv - 1 - torch.arange(nv, device=self.device)) * stride
                out = self.t["timestamp"][:, None] - ages[None, :]
        return out

    def episode_stats(self):
        """Per-slab statistics vector (device, fp64): [count, sum_equity, sum_sq_equity, min_equity,
        max_equity, sum_reward, sum_cost, n_done, exposure[nA], held[nA]] -- the only data that ever
        crosses GPUs (all-reduced by ``madigan_b200.parallel``)."""
        out = torch.empty((A.MDG_STATS_NSCALAR + 2 * self.nA,), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.mdg_episode_stats(C.byref(self.P), C.byref(self._S), C.byref(self._IO),
                                              C.byref(self._launch()), out.data_ptr()))
        self.launches += 2
        return out

    _STAGING = ("units", "actions", "weights")  # host-input staging buffers: not state

    def state_dict(self):
        """Checkpoint of the env (the reference cannot checkpoint its env: wall-clock seeded RNG)."""
        sd = {k_: v.clone() for k_, v in self.t.items() if k_ not in self._STAGING}
        if self._PS is not None:
            sd["param_table"] = self._ptab.clone()  # [nA][NPARAM][S] storage
            sd["param_set"] = self._pset.clone()
        if self._btab is not None:
            sd["broker_table"] = self._btab.clone()  # [MDG_BROKER_NPARAM][S] storage
        if self._PS is not None:
            sd["episode_param_set"] = self._epset.clone()
        if self._cdf is not None:
            sd["set_cdf"] = self._cdf.clone()
        sd["_meta"] = dict(head=self.head, n_valid=self.n_valid, gstep=self._gstep, seed=self.seed,
                           env_offset=self.env_offset, n_envs=self.N, n_assets=self.nA, window=self.k,
                           nstep=int(self.R.nstep), ra=self.ra, shaper=int(self.R.shaper),
                           margins=(self.P.required_margin, self.P.maintenance_margin),
                           costs=(self.P.tcost_rel, self.P.tcost_abs, self.P.slippage_rel, self.P.slippage_abs),
                           n_sets=self.n_param_sets, broker_sets=self._btab is not None,
                           set_draw=self._cdf is not None,
                           set_weights=None if self._weights is None else self._weights.tolist())
        return sd

    def load_state_dict(self, sd):
        m = sd["_meta"]
        mine = dict(n_envs=self.N, n_assets=self.nA, window=self.k, nstep=int(self.R.nstep), ra=self.ra,
                    shaper=int(self.R.shaper))
        for k_, v in mine.items():
            if k_ in m and m[k_] != v:
                raise ValueError(f"checkpoint was taken from an Env with {k_}={m[k_]}, this one has {k_}={v}")
        if m.get("n_sets", 0) != self.n_param_sets:
            raise ValueError(f"checkpoint was taken from an Env with {m.get('n_sets', 0)} parameter sets, this one has "
                             f"{self.n_param_sets}")
        if m.get("broker_sets", False) != (self._btab is not None):
            has = lambda b: "with" if b else "without"
            raise ValueError(f"checkpoint was taken from an Env {has(m.get('broker_sets', False))} broker sets, this one "
                             f"is {has(self._btab is not None)}")
        if m.get("set_draw", False) != (self._cdf is not None):
            has = lambda b: "with" if b else "without"
            raise ValueError(f"checkpoint was taken from an Env {has(m.get('set_draw', False))} the per-episode set "
                             f"draw, this one is {has(self._cdf is not None)}")
        if self._PS is not None:
            self._ptab.copy_(sd["param_table"])
            self._pset.copy_(sd["param_set"])
            if "episode_param_set" in sd:
                self._epset.copy_(sd["episode_param_set"])
        if self._cdf is not None:
            self._cdf.copy_(sd["set_cdf"])
            self._weights = np.asarray(m["set_weights"], dtype=np.float64)
        if self._btab is not None:
            self._btab.copy_(sd["broker_table"])
        for k_, v in sd.items():
            if k_ == "_meta" or k_ in self._STAGING or k_ not in self.t:
                continue
            self.t[k_].copy_(v)
        self.head, self.n_valid, self._gstep = m["head"], m["n_valid"], m["gstep"]
        self.seed, self.env_offset = m["seed"], m["env_offset"]
        if "margins" in m:
            self.P.required_margin, self.P.maintenance_margin = m["margins"]
            self.P.tcost_rel, self.P.tcost_abs, self.P.slippage_rel, self.P.slippage_abs = m["costs"]
        self.invalidate()
