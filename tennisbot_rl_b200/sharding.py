"""Multi-GPU layout of an env batch: contiguous shards, no data-path collective.

Envs are independent, so rank g of G steps envs [g*N/G, (g+1)*N/G) on its own GPU.  RNG streams are keyed by the
GLOBAL env id (tb_config.env_id_offset), which makes the union of the shards identical to the single-GPU batch.
The only exchange is the reduction of the int64[10] episode-statistics vector once per training iteration:
`torch.distributed.all_reduce` (NCCL over NVLink on GPUs, gloo in the CPU tests).  The sums are integers
(fixed-point for the returns), so the result does not depend on G or on the reduction order.
"""
import torch


def shard_range(total_envs, rank, world):
    """[lo, hi) of rank's contiguous shard; shards differ by at most one env."""
    lo = total_envs * rank // world
    hi = total_envs * (rank + 1) // world
    return lo, hi


def all_reduce_stats(stats, group=None):
    """Sum the per-rank statistics vectors in place. `stats`: int64 tensor (CUDA under NCCL, CPU under gloo).
    Pass a SNAPSHOT (`batch.stats_tensor().clone()`): the live vector keeps accumulating inside the kernels, and
    reducing it in place would fold the other ranks' counts into this rank's accumulator."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def all_gather(t, group=None):
    """Concatenate every rank's `t` along dim 0 in rank order (EsTrainer's `gather`: each rank evaluates an equal, contiguous
    shard of the directions).  Identity without an initialised process group of more than one rank."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return t
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size(group))]
    dist.all_gather(parts, t.contiguous(), group=group)
    return torch.cat(parts)


def make_shard(env_id, total_envs, rank, world, device=None, seed=0, precision="f64"):
    """TennisBatch for this rank's shard of a `total_envs` batch."""
    from .batch import TennisBatch

    lo, hi = shard_range(total_envs, rank, world)
    dev = rank % max(torch.cuda.device_count(), 1) if device is None else device
    return TennisBatch(env_id, hi - lo, device=dev, seed=seed, precision=precision, env_id_offset=lo)
