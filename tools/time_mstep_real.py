#!/usr/bin/env python
"""M-step statistics kernel on the bench's EM workload (real posterior sparsity, unlike
tools/time_mstep.py's dense one): the number of (component, tile) pairs carrying weight per
threshold, the makespan of the work items, and the CUDA-event time of kw_gmm_mstep_accumulate.
ITERS = EM iterations first."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
import kwiiyatta_b200 as kw
from kwiiyatta_b200 import synth
dev = torch.device('cuda', 0)
kw.hooks.bind(pad_silence=lambda f, n: f, feature=synth.feature, resample=synth.resample)
padded = [synth.make_padded_pair(i) for i in range(503)]
xj = kw.joint_array_from_pairs(padded, pad_silence=True, pad_len=synth.PAD_LEN)
n = xj.shape[0]
lab = bench.lloyd_labels(xj, 64, seed=0)
resp0 = torch.zeros((n, 64), dtype=torch.float64, device=dev)
resp0[torch.arange(n, device=dev), torch.from_numpy(lab).to(dev)] = 1.0
gm = kw.GaussianMixture(n_components=64, max_iter=1, tol=0.0, resp_init=resp0, precision='tc', device=dev)
xd = gm.initialize(xj)
for _ in range(int(os.environ.get('ITERS', '14'))):
    gm.em_iteration(xd)
cen = gm._means[gm._cur]
gm._estep(torch, xd)
r = gm._resp[:, :n]
tmax = r[:, :n // 64 * 64].reshape(64, -1, 64).amax(dim=2)
for thr in (1e-16, 1e-12, 1e-10, 1e-8, 1e-6):
    m = tmax > thr
    dropped = r[:, :n // 64 * 64].reshape(64, -1, 64).sum(dim=2)[~m].sum().item()
    print(f'(component, tile) pairs with max r > {thr:g}: {m.sum().item()} of {tmax.numel()}; '
          f'total weight in the others {dropped:.3e}')


def makespan(costs, workers=148):
    import heapq
    h = [0.0] * workers
    for c in costs:
        heapq.heappush(h, heapq.heappop(h) + c)
    return max(h)


flag = (tmax > 1e-16).cpu().numpy()                      # (K, tiles)
for chunks in (16, 32, 64):
    per = -(-flag.shape[1] // chunks)
    cost = np.array([[flag[k, c * per:(c + 1) * per].sum() for k in range(64)]
                     for c in range(chunks)], dtype=float).ravel() + 2.0     # item = chunk * K + k
    print(f'{chunks} chunks: pairs per CTA if balanced {cost.sum() / 148:.0f}; list-scheduled in '
          f'item order {makespan(cost):.0f}; longest first {makespan(np.sort(cost)[::-1]):.0f}; '
          f'largest item {cost.max():.0f}')


def timed(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / reps


print(f'mstep_accumulate {timed(lambda: gm._accumulate(torch, xd, cen)):.3f} ms')
