"""TEST INFRASTRUCTURE, NOT PRODUCT CODE: numpy restatement of the per-episode set draw of include/madigan_b200.h
("Per-episode set draw", MdgSetDraw), one env at a time, over the Philox of ``orc_philox4x32_10``.

The draw of env ``gid`` (global env id: env_offset + e) at tick ``tick`` takes Philox4x32-10 with key (seed lo, seed hi)
and counter (gid, 4 << 16, tick lo, tick hi), u = (x0 >> 11) 2^-53 with x0 = (out[1] << 32) | out[0], and yields
``searchsorted(cdf, u, side="right")``: the number of cdf entries <= u.  At a refill the tick is the env's timestamp
before the refill; at the constructor it is 0."""
import ctypes as C

import numpy as np

from oracle.oracle import lib

STREAM = 4  # Philox stream of the set draw (0 normals, 1 uniforms, 2 reset(), 3 constructor)
_M32 = 0xFFFFFFFF


def draw_uniform(seed, gid, tick):
    """u in [0, 1) of the set draw of global env id ``gid`` at ``tick``."""
    ctr = (C.c_uint32 * 4)(gid & _M32, STREAM << 16, tick & _M32, (tick >> 32) & _M32)
    key = (C.c_uint32 * 2)(seed & _M32, (seed >> 32) & _M32)
    out = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(ctr, key, out)
    x0 = (out[1] << 32) | out[0]
    return (x0 >> 11) * 2.0 ** -53


def draw_set(cdf, seed, gid, tick):
    """The set drawn for global env id ``gid`` at ``tick`` from the table ``cdf`` (data_source.make_set_cdf)."""
    s = int(np.searchsorted(np.asarray(cdf, dtype=np.float64), draw_uniform(seed, gid, tick), side="right"))
    return min(s, len(cdf) - 1)


def draw_sets(cdf, seed, gids, ticks):
    """int32 array of the sets drawn for every (gid, tick) pair of the two sequences."""
    return np.array([draw_set(cdf, seed, int(g), int(t)) for g, t in zip(gids, ticks)], dtype=np.int32)
