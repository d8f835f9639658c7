"""Per-iteration parameter error of the tensor-core EM against the FP64 oracle (debug aid)."""
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from kwiiyatta_b200.gmm import GaussianMixture  # noqa: E402
from oracle import gmm_ref  # noqa: E402
from util import rel_err  # noqa: E402


def blobs(rng, n, d, k, sep):
    centres = rng.standard_normal((k, d)) * sep
    lab = rng.integers(0, k, n)
    a = rng.standard_normal((k, d, d)) * 0.3 + np.eye(d)
    return centres[lab] + np.einsum('nij,nj->ni', a[lab], rng.standard_normal((n, d)))


if __name__ == '__main__':
    rng = np.random.default_rng(4097 * 3 + 48)
    x = blobs(rng, 4097, 48, 5, 2.0)
    k, iters = 5, 8
    resp0 = gmm_ref.kmeans_like_resp(x, k, 0)
    refs = [gmm_ref.numpy_em(x, resp0, max_iter=i, tol=0.0) for i in range(1, iters + 1)]
    gm = GaussianMixture(n_components=k, max_iter=iters, tol=0.0, resp_init=resp0, precision='tc',
                         reorder_every=0)
    rows = []

    def cb(g, it, lb):
        mu = g._means[g._cur].cpu().numpy()
        cov = g._cov.cpu().numpy()
        w = g._weights.cpu().numpy()
        r = refs[it - 1]
        rows.append((it, rel_err(w, r['weights']), rel_err(mu, r['means']),
                     rel_err(cov, r['covariances']),
                     np.abs(mu - r['means']).max(axis=1)))
    gm.iter_callback = cb
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        gm.fit(x)
    for it, w, mu, cov, per in rows:
        print(f'  it {it}: w {w:.2e} mu {mu:.2e} cov {cov:.2e}  per-comp mu err', np.array2string(per, precision=1))
    # how much do the oracle's own iterates move?
    for i in range(1, iters):
        print('oracle step', i, '->', i + 1, 'mu change', rel_err(refs[i]['means'], refs[i - 1]['means']),
              'n_k', np.round(refs[i]['weights'] * len(x), 1))
