"""Multi-GPU plumbing: one process per GPU, envs sharded as contiguous slabs, no step-path collective.

Every env is independent (reference: Env::step touches only its own Broker/DataSource, Env.h:206-230),
so the only data that crosses GPUs is the small episode-statistics vector (or an episode-results table), all-reduced with
``torch.distributed`` (NCCL over NVLink on GPUs; gloo in the CPU tests).
"""
import os

import torch
import torch.distributed as dist

from . import _abi as A


def shard_envs(total_envs, world_size, rank):
    """Contiguous slab [offset, offset+count) of `total_envs` for `rank`; remainders go to low ranks.
    The Philox counter uses the GLOBAL env id, so results do not depend on world_size."""
    base, rem = divmod(int(total_envs), int(world_size))
    count = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return offset, count


def init_from_env(backend=None):
    """torchrun-style rendezvous (RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT)."""
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    return rank, world, local


def reduce_episode_stats(vec, n_assets):
    """All-reduce one per-slab statistics vector (layout of ``mdg_episode_stats``): sums are summed,
    min/max slots reduced with MIN/MAX.  Works on CUDA (NCCL) and CPU (gloo) tensors."""
    vec = vec.clone()
    if dist.is_initialized() and dist.get_world_size() > 1:
        mn, mx = vec[3:4].clone(), vec[4:5].clone()
        dist.all_reduce(vec, op=dist.ReduceOp.SUM)
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        vec[3:4], vec[4:5] = mn, mx
    return vec


def reduce_episode_results(results_or_tables):
    """All-reduce an episode-results limb table over the ranks: a ``utils.metrics.EpisodeResults`` or its
    ``limbs()`` dict (``acc``, ``ext``).  Carry pass, SUM of ``acc``, MIN / MAX of the min / max images, carry pass:
    integer sums, so the table is identical on every rank and equals, digit for digit, the table one slab would have
    filled.  Returns a new ``limbs`` dict (decode it with ``EpisodeResults.table(limbs)``).  Works on CUDA (NCCL) and
    CPU (gloo) tensors."""
    from .utils.metrics import carry_
    t = results_or_tables.limbs() if hasattr(results_or_tables, "limbs") else results_or_tables
    acc, ext = carry_(t["acc"].clone()), t["ext"].clone()
    if dist.is_initialized() and dist.get_world_size() > 1:
        mn, mx = ext[0].contiguous(), ext[1].contiguous()
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        ext = torch.stack([mn, mx])
        carry_(acc)
    return dict(acc=acc, ext=ext)


def summarize_stats(vec, n_assets):
    v = vec.detach().cpu().double()
    cnt = max(float(v[0]), 1.0)
    mean = float(v[1]) / cnt
    var = max(float(v[2]) / cnt - mean * mean, 0.0)
    ns = A.MDG_STATS_NSCALAR
    return dict(n_envs=int(v[0]), mean_equity=mean, std_equity=var ** 0.5, min_equity=float(v[3]),
                max_equity=float(v[4]), mean_reward=float(v[5]) / cnt, sum_cost=float(v[6]),
                n_done=int(v[7]), mean_exposure=[float(x) / cnt for x in v[ns:ns + n_assets]],
                frac_in_position=[float(x) / cnt for x in v[ns + n_assets:ns + 2 * n_assets]])
