"""Episode results on the CPU: the quantisation rule and its digits against Python ints, the kernel's fp64 digit
extraction against the rule, the torch carry pass and decoder against Python ints and exact rationals, and the
launchers' argument checks.  (The GPU tests are in test_episode_results.py.)"""
import ctypes as C
import math
import os
from fractions import Fraction

import numpy as np
import pytest
import torch

from madigan_b200 import _abi as A
from madigan_b200.utils.metrics import carry_, decode_table
from oracle import episode_results_oracle as O

M30 = (1 << 30) - 1


def exact_digits(v):
    """digits of rint(v 2^64) from the binary expansion of v, with Python ints only (no Fraction)"""
    num, den = float(v).as_integer_ratio()  # den is a power of two
    x = num << 64
    q, r = divmod(x, den)
    if 2 * r > den or (2 * r == den and q & 1):  # ties to even
        q += 1
    return [(q >> (30 * k)) & M30 for k in range(4)] + [q >> 120], q


EDGES = [0., -0., 1., -1., 0.5, -0.5, 3.25, -3.25, 1e-300, -1e-300, 2. ** -11, -(2. ** -11), 2. ** -11 * 1.5,
         2. ** -12 * 3, 2. ** -64, 2. ** -65, 3 * 2. ** -66, 2. ** -65 * 3, -(2. ** -65 * 3), 5 * 2. ** -66,
         -(5 * 2. ** -66), 2. ** -70, 7 * 2. ** -67, 1e-20, -1e-20, 1e-5, -7e-3, 123456.789, -98765.4321,
         2. ** 31 - 2. ** -21, -(2. ** 31 - 2. ** -21), 2. ** 31 - 1, 2. ** 30, -(2. ** 30), 2. ** 31 * (1 - 2. ** -53),
         2. ** 31 * (1 - 2. ** -52), -(2. ** 31 * (1 - 2. ** -52)), 1.999999999 * 2. ** 30]


@pytest.mark.parametrize("v", EDGES)
def test_quantisation_and_digits(v):
    want, x = exact_digits(v)
    assert O.quantise(v) == x
    assert O.digits(x) == want
    assert O.from_digits(want) == x
    assert O.digits_fp64(v) == want, (v, O.digits_fp64(v), want)
    vv = v * v  # one fp64 multiply, then the same rule (v*v near 2^62 at the largest admitted values)
    want2, x2 = exact_digits(vv)
    assert O.rint64(vv) == x2 and O.digits_fp64(vv) == want2
    assert 0 <= x2 < 1 << 126
    if v < 0 and x != 0:
        assert want[4] == -1 and O.from_digits(want) < 0  # the top digit is signed


def test_ties_of_rint():
    """rint(v 2^64) rounds halves to even: v = (2k + 1) 2^-65 -> the even neighbour"""
    for k in range(-6, 7):
        v = (2 * k + 1) * 2. ** -65
        x = O.quantise(v)
        assert abs(Fraction(v) * 2 ** 64 - x) == Fraction(1, 2) and x % 2 == 0
        assert O.digits_fp64(v) == O.digits(x)


def test_random_values_fp64_extraction():
    rng = np.random.default_rng(5)
    vals = np.concatenate([rng.standard_normal(2000) * 10. ** rng.integers(-25, 9, 2000),
                           rng.uniform(-2. ** 31, 2. ** 31, 500), rng.integers(-2 ** 31 + 1, 2 ** 31, 200) * 1.])
    for v in vals:
        if not O.admitted(v):
            continue
        want, x = exact_digits(v)
        assert O.digits_fp64(v) == want, v
        want2, _ = exact_digits(v * v)
        assert O.digits_fp64(v * v) == want2, v


@pytest.mark.parametrize("v", [2. ** 31, -(2. ** 31), 2. ** 31 * (1 + 2. ** -52), 1e300, float("inf"),
                               float("-inf"), float("nan")])
def test_not_admitted(v):
    assert O.quantise(v) is None
    t = O.table([[v, 1.]], [0], 1)
    assert t["count"][0] == [0, 1] and t["n_episodes"] == [1]
    assert np.isnan(t["mean"][0, 0]) and np.isnan(t["min"][0, 0]) and t["mean"][0, 1] == 1.


def test_oracle_table_statistics():
    rng = np.random.default_rng(2)
    rows = rng.standard_normal((300, 4)) * [1., 1e4, 1e-6, 3.]
    rows[::7, 3] = np.nan
    sets = rng.integers(0, 3, 300)
    cash = rng.choice([1e6, 2.5e6, 3e5], 300)
    t = O.table(rows, sets, 3, cash=None, margin_call=rows[:, 0] > 1.)
    for s in range(3):
        x = rows[sets == s]
        assert t["n_episodes"][s] == len(x) and t["n_margin_call"][s] == int((x[:, 0] > 1.).sum())
        for f in range(4):
            y = x[:, f][~np.isnan(x[:, f])]
            assert t["count"][s][f] == len(y)
            np.testing.assert_allclose(t["mean"][s, f], y.mean(), rtol=1e-13, atol=1e-14 * np.abs(y).max())
            np.testing.assert_allclose(t["std"][s, f], y.std(ddof=1), rtol=1e-9)
            assert t["min"][s, f] == y.min() and t["max"][s, f] == y.max()
    # starting cash divides the four money fields only
    rows = rng.standard_normal((10, 8)) + 2.
    t = O.table(rows, [0] * 10, 1, cash=cash[:10])
    for f in range(8):
        y = rows[:, f] / cash[:10] if f in O.MONEY else rows[:, f]
        assert t["min"][0, f] == y.min() and t["max"][0, f] == y.max()


def random_limbs(rng, S, F, big):
    """an (S, 2 + 11 F) limb table: digits anywhere in [-big, big]"""
    acc = rng.integers(-big, big, (S, 2 + 11 * F), dtype=np.int64, endpoint=True)
    acc[:, :2] = np.abs(acc[:, :2])
    acc[:, 2::11] = rng.integers(2, 1 << 40, (S, F))  # counts
    return acc


def ints_of(acc, S, F):
    """the exact sums held by a limb table, with Python ints"""
    out = []
    for s in range(S):
        for f in range(F):
            o = 2 + 11 * f
            out.append((O.from_digits(acc[s, o + 1:o + 6].tolist()), O.from_digits(acc[s, o + 6:o + 11].tolist())))
    return out


@pytest.mark.parametrize("big", [1 << 30, 1 << 45, (1 << 63) - (1 << 34)])
def test_carry_pass_and_decoder(big):
    rng = np.random.default_rng(big & 0xffff)
    S, F = 3, 7
    acc = random_limbs(rng, S, F, big)
    sums = ints_of(acc, S, F)
    t = torch.from_numpy(acc.copy())
    carry_(t)
    got = t.numpy()
    assert np.array_equal(got[:, :2], acc[:, :2]) and np.array_equal(got[:, 2::11], acc[:, 2::11])
    for (s1, s2), (c1, c2) in zip(sums, ints_of(got, S, F)):
        assert (s1, s2) == (c1, c2)
    for s in range(S):
        for f in range(F):
            o = 2 + 11 * f
            assert got[s, o + 1:o + 6].tolist() == O.digits(sums[s * F + f][0])
            assert got[s, o + 6:o + 11].tolist() == O.digits(sums[s * F + f][1])
    assert np.array_equal(carry_(torch.from_numpy(got.copy())).numpy(), got)  # a carried table is a fixed point
    # the decoder: sums to 1e-15 relative of the exact rationals
    ext = torch.stack([torch.full((S, F), O.image(-1.5)), torch.full((S, F), O.image(2.5))])
    names = [f"f{i}" for i in range(F)]
    tab = decode_table(torch.from_numpy(acc), ext, names)
    for s in range(S):
        for f in range(F):
            n = int(acc[s, 2 + 11 * f])
            s1, s2 = Fraction(sums[s * F + f][0], 1 << 64), Fraction(sums[s * F + f][1], 1 << 64)
            mean = float(s1 / n)
            assert abs(tab[f"f{f}_mean"][s].item() - mean) <= 1e-15 * abs(mean) + 1e-300
            assert tab[f"f{f}_count"][s].item() == n
            assert tab[f"f{f}_min"][s].item() == -1.5 and tab[f"f{f}_max"][s].item() == 2.5
    assert torch.equal(tab["n_episodes"], torch.from_numpy(acc[:, 0]))


def test_decoder_matches_oracle_statistics():
    rng = np.random.default_rng(9)
    F = 5
    rows = rng.standard_normal((500, F)) * [1., 40., 1e-3, 1e5, 1.] + [1., 80., 0., 0., -3.]
    rows[:3, 4] = [np.nan, np.inf, -0.]
    sets = rng.integers(0, 4, 500)
    t = O.table(rows, sets, 4, margin_call=rng.random(500) < .1)
    acc, ext = O.limbs(t)
    tab = decode_table(torch.from_numpy(acc), torch.from_numpy(ext), [f"f{i}" for i in range(F)])
    for f in range(F):
        np.testing.assert_allclose(tab[f"f{f}_mean"].numpy(), t["mean"][:, f], rtol=1e-15)
        np.testing.assert_allclose(tab[f"f{f}_std"].numpy(), t["std"][:, f], rtol=1e-9)
        assert np.array_equal(tab[f"f{f}_min"].numpy(), t["min"][:, f])
        assert np.array_equal(tab[f"f{f}_max"].numpy(), t["max"][:, f])
        assert tab[f"f{f}_count"].tolist() == [c[f] for c in t["count"]]
    assert tab["n_margin_call"].tolist() == t["n_margin_call"]
    # an empty table: counts 0, statistics NaN
    S = 2
    e = O.table(np.zeros((0, F)), [], S)
    acc, ext = O.limbs(e)
    tab = decode_table(torch.from_numpy(acc), torch.from_numpy(ext), [f"f{i}" for i in range(F)])
    assert tab["n_episodes"].tolist() == [0, 0]
    assert all(torch.isnan(tab[f"f0_{k}"]).all() for k in ("mean", "std", "min", "max"))


def _lib():
    from madigan_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        from madigan_b200.build import build
        build()
    return _lib.lib()


def test_results_launchers_validate_without_gpu():
    """The results entry points check their arguments before touching CUDA."""
    lib = _lib()
    from madigan_b200.environments.data_source import make_params
    P, _ = make_params("OU", {"mean": [1., 2.], "theta": [.1, .1], "phi": [.1, .1]})
    L = A.MdgLaunch(n_envs=4, window=8, head=0)
    S, IO = A.MdgState(), A.MdgStepIO()
    S.folds = S.reset_ts = S.cash = S.ledger = 1  # non-null dummies: never dereferenced, validation fails first
    IO.pre_price = IO.reward = IO.trans_cost = IO.done = IO.margin_call = 1
    names = [n for n, _ in A.MdgTearsheet._fields_[3:]]
    ts = A.MdgTearsheet(n_envs=4, n_assets=2, n_offsets=1, **{n: 1 for n in names})

    def res(**kw):
        r = A.MdgEpisodeResults(ts=ts, acc=1, ext=1, n_sets=1, n_fields=A.MDG_TS_NFIXED + 3 + 2)
        for k, v in kw.items():
            setattr(r, k, v)
        return C.byref(r)

    def fused(r, sets=None, broker=None, draw=None):
        return lib.mdg_step_autoreset_results(C.byref(P), None, C.byref(S), C.byref(IO), C.byref(L), 8, 1, 1, 1 << 20,
                                              sets, broker, draw, r)

    def record(r, sets=None, broker=None):
        return lib.mdg_episode_results_record(C.byref(P), C.byref(S), C.byref(IO), sets, broker, r, None)

    sets2 = C.byref(A.MdgParamSets(p=1, set_of_env=1, n_sets=2))
    for call in (fused, record):
        assert call(None) == A.MDG_E_INVALID
        assert call(res(acc=None)) == A.MDG_E_INVALID
        assert call(res(ext=None)) == A.MDG_E_INVALID
        assert call(res(n_fields=99)) == A.MDG_E_INVALID
        assert call(res(n_sets=2)) == A.MDG_E_INVALID          # no sets: one row
        assert call(res(), sets=sets2) == A.MDG_E_INVALID      # two sets, one row
        assert call(res(), broker=1) == A.MDG_E_INVALID        # a broker table without sets
        bad_ts = A.MdgTearsheet.from_buffer_copy(ts)
        bad_ts.nsteps = None
        assert call(res(ts=bad_ts)) == A.MDG_E_INVALID
        bad_ts = A.MdgTearsheet.from_buffer_copy(ts)
        bad_ts.n_assets = 3
        assert call(res(ts=bad_ts, n_fields=A.MDG_TS_NFIXED + 3 + 3)) == A.MDG_E_INVALID
    assert fused(res(), draw=C.byref(A.MdgSetDraw(cdf=1, episode_set=1))) == A.MDG_E_INVALID  # a draw without sets
    assert fused(res(n_sets=2), sets=sets2, draw=C.byref(A.MdgSetDraw())) == A.MDG_E_INVALID
    IO.margin_call = None
    assert record(res()) == A.MDG_E_INVALID
    assert lib.mdg_sizeof(16) == C.sizeof(A.MdgEpisodeResults)
