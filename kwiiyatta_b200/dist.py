"""Multi-GPU plumbing: one process per GPU, torch.distributed (NCCL on GPUs, gloo in CPU tests).

The hot path has exactly one exchange: the all-reduce (sum, float64) of the EM sufficient
statistics per iteration, K*(1+D+D*D)+2 values (SURVEY.md section 8e).  DTW and conversion
shard by utterance (pair) with no data-path collective."""
import numpy as np


def shard_indices(sizes, world_size):
    """Longest-processing-time assignment of items (cost = sizes[i], e.g. tx*ty of a pair) to
    ranks.  Deterministic; returns a list of index arrays, one per rank."""
    sizes = np.asarray(sizes, dtype=np.float64)
    order = np.argsort(-sizes, kind='stable')
    loads = np.zeros(world_size)
    shards = [[] for _ in range(world_size)]
    for i in order:
        r = int(np.argmin(loads))
        shards[r].append(int(i))
        loads[r] += sizes[i]
    return [np.array(sorted(s), dtype=np.int64) for s in shards]


def allreduce_stats(stats, group=None):
    """In-place sum of a statistics vector over the ranks of ``group`` (no-op when
    torch.distributed is not initialised or the world has one rank)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, group=group)
    return stats


def init_from_env(backend='nccl'):
    """torchrun-style initialisation: RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* from the
    environment; binds this process to its GPU."""
    import os

    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if backend == 'nccl':
        torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        kwargs = {}
        if backend == 'nccl':
            kwargs['device_id'] = torch.device('cuda', local_rank)
        dist.init_process_group(backend, **kwargs)
    return int(os.environ.get('RANK', '0')), world, local_rank
