"""Two ranks over NCCL: EM with all-reduced sufficient statistics equals the single-GPU fit.
Runs only on a box with >= 2 GPUs (skipped otherwise; the host logic is covered on CPU by
tests/test_dist_gloo.py)."""
import os
import socket
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, x, resp0, precision, out):
    import torch
    import torch.distributed as dist
    from kwiiyatta_b200.gmm import GaussianMixture
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    cut = int(len(x) * 0.37)                  # unequal shards
    lo, hi = (0, cut) if rank == 0 else (cut, len(x))
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        gm = GaussianMixture(n_components=resp0.shape[1], max_iter=5, tol=0.0,
                             resp_init=resp0[lo:hi], precision=precision,
                             device=torch.device('cuda', rank)).fit(x[lo:hi])
    out.put((rank, gm.weights_, gm.means_, gm.covariances_, gm.lower_bounds_))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('precision', ['fp64', 'tc'])
def test_two_rank_fit_equals_single(cuda, precision):
    if cuda.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    from kwiiyatta_b200.gmm import GaussianMixture
    from oracle import gmm_ref
    rng = np.random.default_rng(3)
    n, d, k = 6000, 24, 4
    x = rng.standard_normal((n, d)) + rng.integers(0, k, n)[:, None] * 1.5
    resp0 = gmm_ref.kmeans_like_resp(x, k, 0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        single = GaussianMixture(n_components=k, max_iter=5, tol=0.0, resp_init=resp0,
                                 precision=precision).fit(x)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, x, resp0, precision, q))
             for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=240) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    tol = 1e-10 if precision == 'fp64' else 1e-5
    for _, w, m, c, lbs in res:
        assert np.abs(w - single.weights_).max() <= tol
        assert np.abs(m - single.means_).max() <= tol * max(1.0, np.abs(single.means_).max())
        assert np.abs(c - single.covariances_).max() <= tol * max(1.0, np.abs(single.covariances_).max())
        assert np.abs(np.array(lbs) - np.array(single.lower_bounds_)).max() <= tol * 100
    # both ranks hold bit-identical parameters
    assert np.array_equal(res[0][2], res[1][2]) and np.array_equal(res[0][3], res[1][3])
