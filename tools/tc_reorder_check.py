"""Does re-sorting the frames change the tensor-core fit beyond rounding?  Per-iteration error
against the FP64 oracle for several re-sort periods, and the M-step statistics of one iteration
computed on sorted and unsorted frames from identical responsibilities (debug aid)."""
import os
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from kwiiyatta_b200.gmm import GaussianMixture  # noqa: E402
from oracle import gmm_ref  # noqa: E402
from util import rel_err  # noqa: E402
from tc_trace import blobs  # noqa: E402

rng = np.random.default_rng(11)
x = blobs(rng, 20000, 48, 16, 0.6)
k, iters = 16, 8
resp0 = gmm_ref.kmeans_like_resp(x, k, 1)
refs = [gmm_ref.numpy_em(x, resp0, max_iter=i, tol=0.0) for i in range(1, iters + 1)]
for reorder in (0, 1, 3):
    gm = GaussianMixture(n_components=k, max_iter=iters, tol=0.0, resp_init=resp0,
                         precision='tc', reorder_every=reorder)
    rows = []

    def cb(g, it, lb):
        r = refs[it - 1]
        rows.append((rel_err(g._means[g._cur].cpu().numpy(), r['means']),
                     rel_err(g._cov.cpu().numpy(), r['covariances'])))
    gm.iter_callback = cb
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        gm.fit(x)
    print(f'reorder_every={reorder}: mu err per iteration', ' '.join(f'{m:.1e}' for m, _ in rows))
