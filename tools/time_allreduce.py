#!/usr/bin/env python
"""CUDA-event time of the EM statistics exchange (NCCL all-reduce of the full vector, K = 64,
D = 144) and of a 16-double all-reduce.  Launch with torch.distributed.run."""
import os, sys
import torch
import torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kwiiyatta_b200 import _lib, dist as kdist
rank, world, local_rank = kdist.init_from_env()
dev = torch.device('cuda', local_rank)
k, d = 64, 144
n = _lib.lib().kw_gmm_stats_len(k, d)
stats = torch.randn(n, dtype=torch.float64, device=dev)


def timed(fn, reps=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


t_full = timed(lambda: kdist.allreduce_stats(stats))
small = torch.zeros(16, dtype=torch.float64, device=dev)
t_small = timed(lambda: dist.all_reduce(small))
if rank == 0:
    print(f'world {dist.get_world_size()}: full vector {t_full:.1f} us, 16 doubles {t_small:.1f} us')
dist.destroy_process_group()
