"""reduce_episode_results over two processes (world size 2, gloo, CPU): two shards' limb tables reduce, digit for digit,
to the oracle table of the union of their episodes, identically on both ranks."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from madigan_b200 import parallel
from oracle import episode_results_oracle as O

S, F, E = 4, 9, 400


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def episodes():
    """E synthetic episode rows (NaN, -0.0, values past 2^31 and tiny values included), set ids and margin calls"""
    rng = np.random.default_rng(17)
    rows = rng.standard_normal((E, F)) * 10. ** rng.integers(-14, 8, F)
    rows[::11, 3] = np.nan
    rows[5, 4], rows[6, 4], rows[7, 5] = -0., 2. ** 31, np.inf
    return rows, rng.integers(0, S, E), rng.random(E) < .2


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    parallel.init_from_env("gloo")
    rows, sets, mc = episodes()
    off, cnt = parallel.shard_envs(E, world, rank)
    acc, ext = O.limbs(O.table(rows[off:off + cnt], sets[off:off + cnt], S, margin_call=mc[off:off + cnt]))
    acc = torch.from_numpy(acc)
    if rank == 1:  # an uncarried shard table: limbs far from canonical, the same sums
        d = acc[:, 2:].view(S, F, 11)
        d[..., 1] += 5 << 30
        d[..., 2] -= 5
        d[..., 7] -= 3 << 40
        d[..., 8] += 3 << 10
    red = parallel.reduce_episode_results(dict(acc=acc, ext=torch.from_numpy(ext)))
    q.put((rank, red["acc"].numpy().copy(), red["ext"].numpy().copy()))
    dist.barrier()
    dist.destroy_process_group()


def test_reduce_episode_results_world2():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        r, acc, ext = q.get(timeout=120)
        res[r] = (acc, ext)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    rows, sets, mc = episodes()
    want_acc, want_ext = O.limbs(O.table(rows, sets, S, margin_call=mc))
    for r in range(world):
        assert np.array_equal(res[r][0], want_acc), r
        assert np.array_equal(res[r][1], want_ext), r
