"""On-device episode tearsheet: the batched counterpart of ``madigan/utils/metrics.py`` ``test_summary`` (:83-171).

The reference appends every step of a test episode to Python lists (equity, reward, ledger, transaction cost) and reduces
them with pandas/numba when the episode is over.  Here every env of a slab streams its episode into a few accumulators
in HBM -- one kernel per step -- and ``summary()`` turns them into the same tearsheet fields, per env, without the
episode ever leaving the device.  Field names follow the reference's columns:

    nsteps, mean_equity, final_equity, mean_reward, max_drawdown, mean_transaction_cost, total_transaction_cost,
    equity_returns_offset_<tf>, equity_sharpe_offset_<tf>, equity_sortino_offset_<tf>   (tf = 1, 2, 4, ...),
    time_spent_in_pos_<asset>

(beta coefficients and Q-value means need the agent's outputs / price history and stay on the host side.)

``EpisodeResults`` harvests the same recorder into one exact table per run: a row per parameter set, with the number of
episodes and, for every tearsheet field, count / mean / std / min / max over every episode the run ends.
"""
import ctypes as C

import torch

from .. import _abi as A
from .._lib import check, lib


class EpisodeTearsheet:
    def __init__(self, env, n_offsets=6):
        """``n_offsets``: return offsets 1, 2, ..., 2^(n_offsets-1) steps (the reference's integer timeframes,
        metrics.py:71-78)."""
        if not 0 <= int(n_offsets) <= A.MDG_TS_MAX_OFFSETS:
            raise ValueError(f"n_offsets must be in 0..{A.MDG_TS_MAX_OFFSETS}")
        self.env, self._lib = env, lib()
        self.N, self.nA, self.J = env.N, env.nA, int(n_offsets)
        dev = env.device
        z = lambda *s, dt=torch.float64: torch.zeros(s, dtype=dt, device=dev)
        N, nA, J = self.N, self.nA, self.J
        R = 1 << (J - 1) if J else 1
        self.t = dict(nsteps=z(N, dt=torch.int64), active=z(N, dt=torch.uint8), sum_equity=z(N), last_equity=z(N),
                      sum_reward=z(N), peak=z(N), min_valley=z(N), sum_cost=z(N), in_pos=z(nA, N), eq_ring=z(R, N),
                      ret_n=z(max(J, 1), N, dt=torch.int32), ret_mean=z(max(J, 1), N), ret_m2=z(max(J, 1), N),
                      ret_down=z(max(J, 1), N))
        self._ts = A.MdgTearsheet(n_envs=N, n_assets=nA, n_offsets=J, **{k: v.data_ptr() for k, v in self.t.items()})
        self.reset()

    def reset(self, mask=None):
        """Re-arm the envs with ``mask[e]`` set (None: all): empty accumulators, recording from the next update."""
        m = None
        if mask is not None:
            m = torch.as_tensor(mask)
            m = (m.view(torch.uint8) if m.dtype == torch.bool and m.is_cuda else m.to(torch.uint8))
            m = m.to(device=self.env.device, dtype=torch.uint8).contiguous()
        with torch.cuda.device(self.env.device):
            check(self._lib.mdg_tearsheet_reset(C.byref(self._ts), None if m is None else m.data_ptr(), self.env._sptr()))

    def update(self):
        """Record the step the env has just taken.  Call after ``env.step(...)`` and BEFORE the finished envs are reset
        (``env.step(..., auto_reset=True, tearsheet=self)`` does exactly that); an env whose step reported ``done`` is
        recorded one last time and then frozen until ``reset``."""
        env = self.env
        with torch.cuda.device(env.device):
            check(self._lib.mdg_tearsheet_update(C.byref(env.P), C.byref(env._S), C.byref(env._IO), C.byref(self._ts),
                                                 env._sptr()))
        env.launches += 1

    @property
    def active(self):
        return self.t["active"].bool()

    def fields(self):
        names = ["nsteps", "mean_equity", "final_equity", "mean_reward", "max_drawdown", "mean_transaction_cost",
                 "total_transaction_cost"]
        for j in range(self.J):
            tf = 1 << j
            names += [f"equity_returns_offset_{tf}", f"equity_sharpe_offset_{tf}", f"equity_sortino_offset_{tf}"]
        names += [f"time_spent_in_pos_{a}" for a in self.env._asset_names]
        return names

    def summary(self):
        """dict field -> (N,) fp64 tensor, the per-env tearsheet of the episodes recorded so far."""
        names = self.fields()
        out = torch.empty((len(names), self.N), dtype=torch.float64, device=self.env.device)
        with torch.cuda.device(self.env.device):
            check(self._lib.mdg_tearsheet_summary(C.byref(self._ts), out.data_ptr(), self.env._sptr()))
        return {n: out[i] for i, n in enumerate(names)}


_BITS, _DIGITS = 30, A.MDG_RES_DIGITS
_STRIDE = 1 + 2 * _DIGITS  # count, sum digits, sum-of-squares digits of one field
_I64_MAX, _I64_MIN = (1 << 63) - 1, -(1 << 63)


def _digit_view(acc):
    """(S, F, 2, 5) view of the sum and sum-of-squares digits of an (S, 2 + 11 F) limb table"""
    return acc[:, 2:].unflatten(-1, (-1, _STRIDE))[..., 1:].unflatten(-1, (2, _DIGITS))


def carry_(acc):
    """The carry pass, in place: every digit but the top one back to [0, 2^30), the carries into the next digit, the top
    digit signed.  Exact (int64; a limb may hold up to 2^63 - 2^34 before the pass).  Returns ``acc``."""
    d = _digit_view(acc)
    for k in range(_DIGITS - 1):
        c = d[..., k] >> _BITS
        d[..., k] -= c << _BITS
        d[..., k + 1] += c
    return acc


def _decode(d):
    """fp64 Horner of carried digits (..., 5): sum_k d_k 2^(30k - 64)"""
    h = d[..., _DIGITS - 1].double()
    for k in range(_DIGITS - 2, -1, -1):
        h = h * float(1 << _BITS) + d[..., k].double()
    return h * 2.0 ** -64


def _from_image(i):
    return torch.where(i < 0, i ^ _I64_MAX, i).view(torch.float64)


def decode_table(acc, ext, names):
    """The statistics of a limb table (``acc`` (S, 2 + 11 F), ``ext`` (2, S, F), int64): dict of (S,) tensors
    ``n_episodes``, ``n_margin_call`` and, per field f, ``f_count``, ``f_mean``, ``f_std`` (ddof 1; NaN below 2),
    ``f_min``, ``f_max`` (NaN when the count is 0).  The sums are decoded with fp64 Horner after a carry pass on a copy;
    the std comes from the decoded sums, (sumsq - sum * mean) / (count - 1)."""
    S, F = acc.shape[0], len(names)
    acc = carry_(acc.clone())
    cnt = acc[:, 2:].view(S, F, _STRIDE)[..., 0]
    d = _digit_view(acc)
    s1, s2 = _decode(d[..., 0, :]), _decode(d[..., 1, :])
    n = cnt.double()
    nan = torch.full_like(s1, float("nan"))
    mean = torch.where(cnt > 0, s1 / n, nan)
    std = torch.where(cnt > 1, ((s2 - s1 * mean) / (n - 1)).clamp(min=0.).sqrt(), nan)
    lo = torch.where(cnt > 0, _from_image(ext[0].contiguous()), nan)
    hi = torch.where(cnt > 0, _from_image(ext[1].contiguous()), nan)
    out = dict(n_episodes=acc[:, 0].clone(), n_margin_call=acc[:, 1].clone())
    for f, name in enumerate(names):
        out[f"{name}_count"] = cnt[:, f].clone()
        out[f"{name}_mean"], out[f"{name}_std"] = mean[:, f], std[:, f]
        out[f"{name}_min"], out[f"{name}_max"] = lo[:, f], hi[:, f]
    return out


class EpisodeResults:
    """Per-set episode results of an Env: pass it to ``env.step(..., auto_reset=True, results=res)`` (or
    ``step_actions`` / ``step_weights``).  Every such step records into the owned tearsheet; each env whose step ends an
    episode adds its tearsheet row (the money fields over the episode's starting cash) into the row of the episode's
    parameter set (0 on an Env without sets) and is re-armed, all on the device inside the fused auto-reset.

    Sums are exact: each admitted value (finite, |v| < 2^31) is quantised to rint(v 2^64) and added as integer digits
    (include/madigan_b200.h, MdgEpisodeResults), so the table does not depend on the order in which envs finish or on
    how a run is sharded (``parallel.reduce_episode_results``).  NaN values -- e.g. the Sharpe ratio at offsets too long
    for a short episode -- are left out of their field's count.  The Env's own state is exactly that of the same Env
    stepped without results."""

    def __init__(self, env, n_offsets=6):
        self.env = env
        self.tearsheet = EpisodeTearsheet(env, n_offsets)  # arms every env: recording from the next step
        self.n_sets = max(int(env.n_param_sets), 1)
        self._names = self.tearsheet.fields()
        S, F = self.n_sets, len(self._names)
        with torch.cuda.device(env.device), env._copy_ctx():
            self.acc = torch.zeros((S, 2 + _STRIDE * F), dtype=torch.int64, device=env.device)
            self.ext = torch.empty((2, S, F), dtype=torch.int64, device=env.device)
        self._R = A.MdgEpisodeResults(ts=self.tearsheet._ts, acc=self.acc.data_ptr(), ext=self.ext.data_ptr(),
                                      n_sets=S, n_fields=F)
        self._pR = C.byref(self._R)
        # a limb grows by < 2^30 per episode and at most N episodes end per step: carried every 2^32 / N steps, no limb
        # passes 2^62
        self._carry_every = max(1, (1 << 32) // max(env.N, 1))
        self.reset()

    def fields(self):
        return list(self._names)

    def reset(self):
        """Empty the table; the recorders keep running (an episode in progress is counted when it ends)."""
        with torch.cuda.device(self.env.device), self.env._copy_ctx():
            self.acc.zero_()
            self.ext[0].fill_(_I64_MAX)
            self.ext[1].fill_(_I64_MIN)
        self._since_carry = 0

    def _recorded(self):
        """after every recording step"""
        self._since_carry += 1
        if self._since_carry >= self._carry_every:
            self._carry()

    def _carry(self):
        with torch.cuda.device(self.env.device), self.env._copy_ctx():
            carry_(self.acc)
        self._since_carry = 0

    def limbs(self):
        """dict ``acc``, ``ext``: a copy of the carried limb table (``parallel.reduce_episode_results`` takes it)."""
        self._carry()
        with torch.cuda.device(self.env.device), self.env._copy_ctx():
            return dict(acc=self.acc.clone(), ext=self.ext.clone())

    def table(self, limbs=None):
        """dict of (S,) device tensors: ``n_episodes``, ``n_margin_call``, and per field f ``f_count``, ``f_mean``,
        ``f_std``, ``f_min``, ``f_max`` -- of this object's table, or of ``limbs`` (e.g. a reduction over shards)."""
        if limbs is None:
            limbs = self.limbs()
        with torch.cuda.device(self.env.device), self.env._copy_ctx():
            return decode_table(limbs["acc"], limbs["ext"], self._names)

    def state_dict(self):
        """The limbs, the recorders and the carry counter (after a carry pass)."""
        self._carry()
        with torch.cuda.device(self.env.device), self.env._copy_ctx():
            return dict(acc=self.acc.clone(), ext=self.ext.clone(), since_carry=self._since_carry,
                        tearsheet={k: v.clone() for k, v in self.tearsheet.t.items()})

    def load_state_dict(self, sd):
        """Restore a ``state_dict``; a results object of another shape (envs, sets, offsets, assets) raises ValueError."""
        shapes = [(self.acc, sd["acc"], "acc"), (self.ext, sd["ext"], "ext")]
        ts = sd["tearsheet"]
        if set(ts) != set(self.tearsheet.t):
            raise ValueError("state_dict: tearsheet accumulators differ")
        shapes += [(v, ts[k], k) for k, v in self.tearsheet.t.items()]
        for mine, theirs, name in shapes:
            if tuple(mine.shape) != tuple(theirs.shape) or mine.dtype != theirs.dtype:
                raise ValueError(f"state_dict: {name} has shape {tuple(theirs.shape)} {theirs.dtype}, this results "
                                 f"object {tuple(mine.shape)} {mine.dtype}")
        with torch.cuda.device(self.env.device), self.env._copy_ctx():
            for mine, theirs, _ in shapes:
                mine.copy_(theirs)
        self._since_carry = int(sd["since_carry"])
