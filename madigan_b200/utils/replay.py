"""Device-side n-step replay buffer (reference: madigan/utils/buffers/replay_buffer.py + nstep_buffer.py:315-361).

``ReplayBuffer.add`` appends a Python SARSD per env-step and ``_sample`` ``np.stack``s Python objects per sample;
here the transitions of all N envs of a slab are ingested by one kernel per step and sampled by one gather kernel,
so observations never leave HBM between env and agent.  The n-step pops themselves (full-buffer pop, drain on done,
DSR/DDR/... shaping) were already produced by the step kernel (``env.shaped_reward`` / ``env.n_popped``).

Observations are stored once per step (slot ``t % depth``): the price window the agents' nets consume
(``(N, k, nF)``, normalised, fp32 by default) and the newest portfolio row -- the agents read ``portfolio[:, -1]`` only
(dqn.py:188-199).  See include/madigan_b200.h for the record layout and the one documented deviation (the
next_state of a terminal transition).

``store="rows"`` keeps the price observations as raw rows instead: one new row per env-step (k rows when the env
reset) in a per-env row ring, and the windows of the sampled records are built and normalised at sample time
(include/madigan_b200.h, "Replay row store").  That writes ~272 B per env-step instead of ~4.2 KB (16 assets, k 64,
fp32), so the ingest is cheap and a deep replay fits on the device; a sample reads and normalises the raw rows."""
import ctypes as C

import torch

from .. import _abi as A
from .._lib import check, lib
from .data import SARSD, State


class DeviceReplay:
    def __init__(self, env, depth=64, capacity=None, n_action=None, norm_type=None, dtype=torch.float32, seed=0,
                 store="windows", rows=None):
        """``depth``: observation slots (steps of history kept); ``capacity``: transitions in the ring (default
        N * (depth - nstep - 1), so that a stored transition's state is normally still resident).
        ``store``: ``"windows"`` stores each step's normalised windows (``obs_price``); ``"rows"`` stores raw price
        rows (``rows``, ``row_end``, ``row_count``, ``last_ts``; ``obs_price`` is None) and normalises the sampled
        windows at sample time.  ``rows``: rows kept per env by the row store, at least ``depth + k - 1``; the default
        ``depth + 3 (k - 1)`` keeps every record of an env that reset at most twice in ``depth`` steps."""
        self.env, self._lib = env, lib()
        N, k, nA = env.N, env.k, env.nA
        self.N, self.k, self.nF, self.n_port = N, k, nA, nA + 1
        self.depth = int(depth)
        self.nstep, self.ra = int(env.R.nstep), int(env.ra)
        if env.R.shaper == A.SHAPER_OFF:
            raise ValueError("DeviceReplay needs an Env built with reward=... (the step kernel makes the n-step rewards)")
        if self.depth <= self.nstep + 1:
            raise ValueError("depth must exceed nstep + 1")
        cap_max = N * (self.depth - self.nstep - 1)
        self.capacity = int(capacity) if capacity else cap_max
        if self.capacity > cap_max:  # older records would point at overwritten observation slots
            raise ValueError(f"capacity {self.capacity} exceeds N * (depth - nstep - 1) = {cap_max}")
        self.n_action = int(n_action) if n_action else nA
        self.norm_type, self.dtype, self.seed = norm_type, dtype, int(seed)
        if store not in ("windows", "rows"):
            raise ValueError(f"store must be 'windows' or 'rows', not {store!r}")
        self.store = store
        dev = env.device
        z = lambda *s, dt: torch.zeros(s, dtype=dt, device=dev)
        if store == "windows":
            self.obs_price = torch.empty((self.depth, N, k, nA), dtype=dtype, device=dev)
        else:
            from .preprocessor import NORM_TYPES
            self._norm = NORM_TYPES[norm_type]
            self.n_rows = int(rows) if rows is not None else self.depth + 3 * (k - 1)
            if self.n_rows < self.depth + k - 1:
                raise ValueError(f"rows {self.n_rows} < depth + k - 1 = {self.depth + k - 1}")
            self.obs_price = None
            self.rows = torch.zeros((N, self.n_rows, nA), dtype=torch.float64, device=dev)
            self.row_end = z(self.depth, N, dt=torch.int64)
            self.row_count = z(N, dt=torch.int64)
            self.last_ts = z(N, dt=torch.int64)
            self._rr = A.MdgReplayRows(rows=self.rows.data_ptr(), row_end=self.row_end.data_ptr(),
                                       row_count=self.row_count.data_ptr(), last_ts=self.last_ts.data_ptr(),
                                       n_rows=self.n_rows, n_feats=nA, window=k)
        self.obs_port = torch.empty((self.depth, N, nA + 1), dtype=torch.float64, device=dev)
        self.t = dict(t_env=z(self.capacity, dt=torch.int32), t_state_slot=z(self.capacity, dt=torch.int32),
                      t_next_slot=z(self.capacity, dt=torch.int32),
                      t_state_step=torch.full((self.capacity,), -2 ** 63, dtype=torch.int64, device=dev),  # INT64_MIN = empty
                      t_done=z(self.capacity, dt=torch.uint8), t_reward=z(self.capacity, self.ra, dt=torch.float64),
                      t_action=z(self.capacity, self.n_action, dt=torch.float64),
                      cursor=z(1, dt=torch.int64), act_ring=z(self.nstep, N, self.n_action, dt=torch.float64))
        self._rp = A.MdgReplay(capacity=self.capacity, depth=self.depth, nstep=self.nstep, ra=self.ra,
                               n_action=self.n_action, **{k_: v.data_ptr() for k_, v in self.t.items()})
        self._out = {}
        self.step_count = -1  # index of the last ingested step; observe_start() stores slot -1 % depth
        self.draws = 0

    # ------------------------------------------------------------------ ingest
    def _store_obs(self, step, whole_window=False):
        slot = step % self.depth
        env = self.env
        if self.obs_price is not None:
            env.window(self.norm_type, dtype=self.dtype, out=self.obs_price[slot])
        else:
            if env.n_valid < self.k:
                raise ValueError(f"the row store needs a full window: env.n_valid {env.n_valid} < k {self.k}")
            T = env.t
            w = A.MdgWindow(ring=T["obs_price"].data_ptr(), prefix=T["pre_price"].data_ptr(),
                            timestamp=T["timestamp"].data_ptr(), reset_ts=T["reset_ts"].data_ptr(), n_envs=self.N,
                            n_feats=self.nF, window=self.k, head=env.head, n_valid=env.n_valid, stream=env._sptr())
            with torch.cuda.device(env.device):
                check(self._lib.mdg_replay_rows_ingest(C.byref(self._rr), C.byref(w), slot, int(whole_window)))
        self.obs_port[slot].copy_(env.t["obs_port"][env.head].t())

    def observe_start(self):
        """Store the observation the first action is taken from (after ``env.reset(fill_history=True)``)."""
        with self.env._copy_ctx():
            self._store_obs(self.step_count, whole_window=True)

    def add(self, action):
        """Call after ``env.step(..., auto_reset=True)`` / ``env.step_actions(...)`` with the action that was taken
        ((N, n_action), any real dtype): stores the new observation and appends the transitions that step popped."""
        env = self.env
        t = self.step_count + 1
        a = action if (isinstance(action, torch.Tensor) and action.dtype == torch.float64 and action.is_cuda
                       and action.is_contiguous()) else \
            torch.as_tensor(action).to(device=env.device, dtype=torch.float64).contiguous()
        if a.shape != (self.N, self.n_action):
            raise ValueError(f"action must have shape {(self.N, self.n_action)}")
        with env._copy_ctx():
            self._store_obs(t)
        self.step_count = t
        T = env.t
        with torch.cuda.device(env.device):
            check(self._lib.mdg_replay_append(
                C.byref(self._rp), self.N, t, a.data_ptr(), T["shaped_reward"].data_ptr(), T["n_popped"].data_ptr(),
                T["nstep_len"].data_ptr() if self.nstep > 1 else None, env._done_u8.data_ptr(), env._sptr()))

    def __len__(self):
        return min(int(self.t["cursor"].item()), self.capacity)

    # ------------------------------------------------------------------ sample
    def _batch_out(self, n):
        """Output tensors of a batch of n and the MdgReplayBatch pointing at them."""
        dev = self.env.device
        out = self._out.get(n)
        if out is None:  # output buffers are allocated once per batch size and reused (a sample is consumed by the
            # agent's training step before the next one is drawn; clone() what must outlive that)
            out = self._out[n] = dict(
                idx=torch.empty(n, dtype=torch.int64, device=dev),
                state_price=torch.empty((n, self.k, self.nF), dtype=self.dtype, device=dev),
                next_price=torch.empty((n, self.k, self.nF), dtype=self.dtype, device=dev),
                state_port=torch.empty((n, self.n_port), dtype=torch.float64, device=dev),
                next_port=torch.empty((n, self.n_port), dtype=torch.float64, device=dev),
                action=torch.empty((n, self.n_action), dtype=torch.float64, device=dev),
                reward=torch.empty((n, self.ra), dtype=torch.float64, device=dev),
                done=torch.empty(n, dtype=torch.uint8, device=dev))
        return out, A.MdgReplayBatch(**{k_: v.data_ptr() for k_, v in out.items()})

    def _sarsd(self, out):
        self.last_idx = out["idx"]
        # (batch,) bool: False where 64 draws found no resident transition (the row is zero-filled with done = True)
        with self.env._copy_ctx():
            self.last_valid = out["idx"] >= 0
        return SARSD(State(out["state_price"], out["state_port"], None), out["action"], out["reward"],
                     State(out["next_price"], out["next_port"], None), out["done"].bool())

    def sample(self, n):
        """``ReplayBuffer.sample`` (replay_buffer.py:94-103): (SARSD of batched tensors, None).  Runs on the env's
        stream (``Env.bind_stream``).  ``self.last_valid`` flags the rows that hold a real transition (all of them
        unless the ring is nearly empty or mostly stale)."""
        out, b = self._batch_out(n)
        self.draws += 1
        dt = A.DTYPE_F32 if self.dtype == torch.float32 else A.DTYPE_F64
        with torch.cuda.device(self.env.device):
            if self.obs_price is not None:
                check(self._lib.mdg_replay_sample(
                    C.byref(self._rp), self.N, self.step_count, self.obs_price.data_ptr(), self.obs_port.data_ptr(),
                    self.k * self.nF, self.n_port, dt, n, self.seed, self.draws, C.byref(b), self.env._sptr()))
            else:
                check(self._lib.mdg_replay_sample_rows(
                    C.byref(self._rp), C.byref(self._rr), self.N, self.step_count, self.obs_port.data_ptr(),
                    self.n_port, self._norm, dt, n, self.seed, self.draws, C.byref(b), self.env._sptr()))
        return self._sarsd(out), None


class DevicePrioritizedReplay(DeviceReplay):
    """Proportional prioritized replay (Schaul et al. 2016; the reference's PrioritizedReplayBuffer over sum/min
    segment trees, utils/buffers/prioritized_replay_buffer.py + segment_tree.py) on the device ring of DeviceReplay.

    A record enters with priority ``max_priority ** alpha``; ``sample(n, beta)`` draws records with probability
    proportional to their priority among the resident ones and returns importance weights beside the batch;
    ``update_priorities`` sets the priorities of the last sample's records (|TD| + eps, made by the caller).  Trees,
    draws and updates stay on the device and on the env's stream, with no host synchronisation: ``add``, ``sample``
    and ``update_priorities`` can be captured in a CUDA graph.  Semantics and the one documented deviation (stale
    records count in the weights' normalisers): include/madigan_b200.h, "Proportional prioritized replay"."""

    def __init__(self, env, alpha=0.6, depth=64, capacity=None, n_action=None, norm_type=None, dtype=torch.float32,
                 seed=0, store="windows", rows=None):
        super().__init__(env, depth=depth, capacity=capacity, n_action=n_action, norm_type=norm_type, dtype=dtype,
                         seed=seed, store=store, rows=rows)
        self.alpha = float(alpha)
        if not self.alpha >= 0:
            raise ValueError("alpha must be >= 0")
        cap = self.capacity
        T = max(1024, 1 << (cap - 1).bit_length())
        self.tree_size = T
        dev = env.device
        S = T // 1024
        self.per = dict(sum_tree=torch.zeros(2 * T, dtype=torch.float64, device=dev),
                        min_tree=torch.full((2 * T,), float("inf"), dtype=torch.float64, device=dev),
                        leaf_pos=torch.full((cap,), -1, dtype=torch.int64, device=dev),
                        batch_pos=torch.full((cap,), -1, dtype=torch.int32, device=dev),
                        dirty=torch.zeros(S, dtype=torch.int32, device=dev),
                        dirty_list=torch.zeros(S, dtype=torch.int32, device=dev),
                        ctl=torch.zeros(4, dtype=torch.int32, device=dev),
                        seen=torch.zeros(1, dtype=torch.int64, device=dev),
                        max_priority=torch.ones(1, dtype=torch.float64, device=dev),
                        n_rejected=torch.zeros(1, dtype=torch.int64, device=dev))
        self._pr = A.MdgPrioritized(capacity=cap, tree_size=T, alpha=self.alpha,
                                    **{k_: v.data_ptr() for k_, v in self.per.items()})
        self._pout = {}

    def add(self, action):
        """``DeviceReplay.add``, then the new records' leaves enter the trees at ``max_priority ** alpha``."""
        super().add(action)
        with torch.cuda.device(self.env.device):
            check(self._lib.mdg_per_ingest(C.byref(self._pr), C.byref(self._rp), self.N * self.nstep,
                                           self.env._sptr()))

    def sample(self, n, beta):
        """``PrioritizedReplayBuffer.sample``: (SARSD of batched tensors, importance weights (n,) float64, 1 for the
        record of least priority).  ``last_idx`` / ``last_valid`` as for DeviceReplay; ``last_pos`` holds the
        sampled records' append positions, which ``update_priorities`` uses to skip records overwritten since."""
        out, b = self._batch_out(n)
        pout = self._pout.get(n)
        if pout is None:
            dev = self.env.device
            pout = self._pout[n] = dict(weights=torch.empty(n, dtype=torch.float64, device=dev),
                                        pos=torch.empty(n, dtype=torch.int64, device=dev))
        self.draws += 1
        dt = A.DTYPE_F32 if self.dtype == torch.float32 else A.DTYPE_F64
        with torch.cuda.device(self.env.device):
            if self.obs_price is not None:
                check(self._lib.mdg_per_sample(
                    C.byref(self._pr), C.byref(self._rp), self.N, self.step_count, self.obs_price.data_ptr(),
                    self.obs_port.data_ptr(), self.k * self.nF, self.n_port, dt, n, float(beta), self.seed,
                    self.draws, C.byref(b), pout["weights"].data_ptr(), pout["pos"].data_ptr(), self.env._sptr()))
            else:
                check(self._lib.mdg_per_sample_rows(
                    C.byref(self._pr), C.byref(self._rp), C.byref(self._rr), self.N, self.step_count,
                    self.obs_port.data_ptr(), self.n_port, self._norm, dt, n, float(beta), self.seed, self.draws,
                    C.byref(b), pout["weights"].data_ptr(), pout["pos"].data_ptr(), self.env._sptr()))
        self.last_pos = pout["pos"]
        return self._sarsd(out), pout["weights"]

    def update_priorities(self, priorities):
        """``PrioritizedReplayBuffer.update_priorities`` for the records of the last ``sample``: ``priorities`` is a
        float32 or float64 tensor of shape (n,).  Rows with idx -1, records overwritten since the sample, and
        priorities that are not finite or not > 0 are skipped (the last counted in ``n_rejected``); of an index
        drawn twice the last row wins."""
        idx = getattr(self, "last_idx", None)
        if idx is None:
            raise RuntimeError("update_priorities needs a sample() first")
        p = priorities if isinstance(priorities, torch.Tensor) else torch.as_tensor(priorities)
        if p.dtype not in (torch.float32, torch.float64):
            raise ValueError("priorities must be float32 or float64")
        if p.shape != idx.shape:
            raise ValueError(f"priorities must have shape {tuple(idx.shape)}")
        with self.env._copy_ctx():
            p = p.to(device=self.env.device, dtype=torch.float64).contiguous()
        with torch.cuda.device(self.env.device):
            check(self._lib.mdg_per_update(C.byref(self._pr), idx.numel(), idx.data_ptr(), self.last_pos.data_ptr(),
                                           p.data_ptr(), self.env._sptr()))

    @property
    def n_rejected(self):
        """(1,) int64 device tensor: priorities ``update_priorities`` skipped as not finite or not > 0 (reading it
        on the host synchronises; keep it on the device inside a training loop)."""
        return self.per["n_rejected"]

    @property
    def max_priority(self):
        """(1,) float64 device tensor: the largest priority applied so far (1 at first)."""
        return self.per["max_priority"]
