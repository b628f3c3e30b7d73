"""Episode results (include/madigan_b200.h, MdgEpisodeResults) restated with Python integers and exact rationals.

``table(rows, sets, n_sets, cash, margin_call)`` builds, from per-episode tearsheet rows and their set ids, what the
device table holds after a carry pass: the quantised sums as Python ints, their canonical digits, the counts, the
order-preserving min / max images, and the statistics decoded from exact rationals.  ``limbs(tab)`` lays it out as the
device tensors ``acc`` and ``ext``.  ``digits_fp64`` restates the kernel's fp64 digit extraction, so that the CPU tests
can hold it against the integer rule."""
import math
import struct
from fractions import Fraction

import numpy as np

DIGITS, BITS = 5, 30
MASK = (1 << BITS) - 1
SCALE = 1 << 64        # X = rint(v 2^64)
LIMIT = 2.0 ** 31      # admitted: finite and |v| < 2^31
MONEY = (1, 2, 5, 6)   # mean_equity, final_equity, mean_transaction_cost, total_transaction_cost: over starting cash
STRIDE = 1 + 2 * DIGITS
HEAD = 2
I64_MAX, I64_MIN = (1 << 63) - 1, -(1 << 63)


def admitted(v):
    return math.isfinite(v) and abs(v) < LIMIT


def rint64(v):
    """rint(v 2^64) (ties to even) of a finite v as a Python int"""
    return round(Fraction(float(v)) * SCALE)


def quantise(v):
    """X = rint(v 2^64) as a Python int, or None when v is not admitted."""
    return rint64(v) if admitted(float(v)) else None


def digits(x):
    """canonical digits of the integer x: four in [0, 2^30), then the signed top digit"""
    return [(x >> (BITS * k)) & MASK for k in range(DIGITS - 1)] + [x >> (BITS * (DIGITS - 1))]


def from_digits(ds):
    return sum(int(d) << (BITS * k) for k, d in enumerate(ds))


def digits_fp64(v):
    """the kernel's extraction (csrc/mdg_tearsheet.cu, res_digits) in fp64 numpy arithmetic: floor and power-of-two
    scalings of |rint(v 2^64)|, then the two's-complement negation of the digits for a negative value"""
    x = np.rint(np.float64(v) * np.float64(2.0 ** 64))
    r = np.abs(x)
    d = [0] * DIGITS
    for k in range(DIGITS - 1, 0, -1):
        q = np.floor(r * np.float64(2.0 ** (-BITS * k)))
        r = r - q * np.float64(2.0 ** (BITS * k))
        d[k] = int(q)
    d[0] = int(r)
    if x < 0:
        carry = 1
        for k in range(DIGITS - 1):
            c = (MASK - d[k]) + carry
            d[k], carry = c & MASK, c >> BITS
        d[DIGITS - 1] = ~d[DIGITS - 1] + carry
    return d


def image(v):
    """order-preserving int64 image of an fp64 value"""
    b = struct.unpack("<q", struct.pack("<d", float(v)))[0]
    return b ^ I64_MAX if b < 0 else b


def from_image(i):
    b = i ^ I64_MAX if i < 0 else i
    return struct.unpack("<d", struct.pack("<q", int(b)))[0]


def table(rows, sets, n_sets, cash=None, margin_call=None):
    """rows: (E, F) fp64 tearsheet rows of E episodes; sets: (E,) set ids in [0, n_sets); cash: (E,) starting cash
    (the money fields are divided by it in fp64) or None; margin_call: (E,) bools or None."""
    rows = np.array(rows, dtype=np.float64, copy=True)
    E, F = rows.shape
    assert len(sets) == E
    if cash is not None:
        for f in MONEY:
            rows[:, f] = rows[:, f] / np.asarray(cash, dtype=np.float64)
    S = int(n_sets)
    t = dict(n_episodes=[0] * S, n_margin_call=[0] * S, count=[[0] * F for _ in range(S)],
             sum=[[0] * F for _ in range(S)], sumsq=[[0] * F for _ in range(S)],
             lo=[[I64_MAX] * F for _ in range(S)], hi=[[I64_MIN] * F for _ in range(S)])
    for i in range(E):
        s = int(sets[i])
        t["n_episodes"][s] += 1
        t["n_margin_call"][s] += int(bool(margin_call[i])) if margin_call is not None else 0
        for f in range(F):
            v = float(rows[i, f])
            x = quantise(v)
            if x is None:
                continue
            t["count"][s][f] += 1
            t["sum"][s][f] += x
            t["sumsq"][s][f] += rint64(v * v)  # one fp64 multiply, as the kernel
            t["lo"][s][f] = min(t["lo"][s][f], image(v))
            t["hi"][s][f] = max(t["hi"][s][f], image(v))
    mean = np.full((S, F), np.nan)
    std = np.full((S, F), np.nan)
    for s in range(S):
        for f in range(F):
            n = t["count"][s][f]
            if n == 0:
                continue
            s1, s2 = Fraction(t["sum"][s][f], SCALE), Fraction(t["sumsq"][s][f], SCALE)
            mean[s, f] = float(s1 / n)
            if n > 1:
                std[s, f] = math.sqrt(max(float((s2 - s1 * s1 / n) / (n - 1)), 0.))
    t["mean"], t["std"] = mean, std
    t["min"] = np.array([[from_image(x) if n else np.nan for x, n in zip(lo, c)] for lo, c in zip(t["lo"], t["count"])])
    t["max"] = np.array([[from_image(x) if n else np.nan for x, n in zip(hi, c)] for hi, c in zip(t["hi"], t["count"])])
    return t


def limbs(t):
    """the device layout of table t after a carry pass: acc (S, 2 + 11 F) and ext (2, S, F), int64"""
    S, F = len(t["count"]), len(t["count"][0])
    acc = np.zeros((S, HEAD + STRIDE * F), dtype=np.int64)
    for s in range(S):
        acc[s, 0], acc[s, 1] = t["n_episodes"][s], t["n_margin_call"][s]
        for f in range(F):
            o = HEAD + STRIDE * f
            acc[s, o] = t["count"][s][f]
            acc[s, o + 1:o + 1 + DIGITS] = digits(t["sum"][s][f])
            acc[s, o + 1 + DIGITS:o + STRIDE] = digits(t["sumsq"][s][f])
    ext = np.array([t["lo"], t["hi"]], dtype=np.int64).reshape(2, S, F)
    return acc, ext
