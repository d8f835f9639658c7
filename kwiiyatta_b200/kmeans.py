"""K-means initial labels for the EM (sklearn ``init_params='kmeans'``,
sklearn/mixture/_base.py:119-128) -- SURVEY.md section 8f rank 1.

The assignment step of every Lloyd pass is this library's ``kw_gmm_hard_labels`` with identity
precisions and equal weights (argmin of the squared distance; tcgen05 contraction with fp64
re-check of near-ties when ``precision='tc'``); the centre update is one (K x N)(N x D) product of
the one-hot responsibilities with the frames, all-reduced across ranks.  Only
the k-means++ seeding (K sequential D^2-weighted draws, all on the device) uses stock torch ops.  The result is not
bit-compatible with any sklearn KMeans version (their seeding consumes the RNG differently
across versions); parity tests inject ``resp_init`` instead."""
import numpy as np

from . import _lib


def _dist2(x, c):
    return (x * x).sum(1, keepdim=True) - 2.0 * (x @ c.t()) + (c * c).sum(1)[None, :]


def _seed_centres(x, k, seed, group):
    import torch
    import torch.distributed as dist
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    rank = dist.get_rank(group) if multi else 0
    n, d = x.shape
    rs = np.random.RandomState(seed)
    centres = torch.empty((k, d), dtype=x.dtype, device=x.device)
    if rank == 0:
        if n < k:
            raise ValueError(f'need at least {k} frames on rank 0 to seed k-means, got {n}')
        # k-means++: every draw (D^2-weighted, by inverting the cumulative sum at a uniform
        # number drawn on the host beforehand) stays on the device -- no read-back per centre
        first = int(rs.randint(n))
        uniform = torch.from_numpy(rs.random_sample(k)).to(x.device)
        centres[0] = x[first]
        closest = _dist2(x, centres[0:1]).squeeze(1).clamp_min_(0.0)
        for j in range(1, k):
            cum = torch.cumsum(closest, dim=0)
            idx = torch.searchsorted(cum, uniform[j] * cum[-1]).clamp_(max=n - 1)
            centres[j] = x.index_select(0, idx.reshape(1))[0]
            closest = torch.minimum(closest,
                                    _dist2(x, centres[j:j + 1]).squeeze(1).clamp_min_(0.0))
    if multi:
        dist.broadcast(centres, src=dist.get_global_rank(group, 0) if group is not None else 0,
                       group=group)
    return centres


def kmeans_labels(x, k, seed=None, group=None, n_lloyd=300, precision=0, tol=1e-4):
    """Hard labels (int64 CUDA tensor) of the device-resident frames ``x`` (N, D) float64.
    Lloyd passes stop as sklearn's KMeans does (max_iter = 300, tol = 1e-4): when no label
    changes, or when the squared centre shift falls below ``tol`` times the mean per-feature
    variance of the data."""
    import torch
    import torch.distributed as dist
    lib = _lib.lib()
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    n, d = x.shape
    x = x.contiguous()
    centres = _seed_centres(x, k, seed, group).contiguous()
    f64 = dict(dtype=torch.float64, device=x.device)
    eye = torch.eye(d, **f64).expand(k, d, d).contiguous()      # prec_chol = I
    aux = torch.zeros((k, d + 2), **f64)                         # [b = mu, log|L| = 0, log w = 0]
    labels = torch.empty(n, dtype=torch.int32, device=x.device)
    ws_bytes = lib.kw_gmm_workspace_bytes(n, k, d, precision)
    ws = _lib.workspace(ws_bytes, x.device)
    npad = lib.kw_gmm_resp_len(n, k) // k
    resp = torch.zeros((k, npad), **f64)
    stream = _lib.stream_ptr(torch)
    _lib.call('kw_gmm_pack_frames', n, x, k, d, precision, ws, ws_bytes, stream)
    rows = torch.arange(n, device=x.device)
    prev = None
    # tolerance on the squared centre shift, relative to the data's mean variance (all ranks)
    mom = torch.stack((x.sum(dim=0), (x * x).sum(dim=0)))
    cnt = torch.tensor([float(n)], **f64)
    if multi:
        dist.all_reduce(mom, group=group)
        dist.all_reduce(cnt, group=group)
    var_mean = (mom[1] / cnt - (mom[0] / cnt) ** 2).mean()
    shift_tol = tol * var_mean
    for it in range(max(n_lloyd, 0) + 1):
        aux[:, :d] = centres
        _lib.call('kw_gmm_hard_labels', n, x, k, d, centres, eye, aux, labels, precision, ws,
                  ws_bytes, stream)
        lab = labels.long()
        if it == n_lloyd:
            break
        if prev is not None:
            changed = (lab != prev).sum().to(torch.float64)
            if multi:
                dist.all_reduce(changed, group=group)
            if changed.item() == 0:
                break
        prev = lab
        # centre update = first moments of the one-hot responsibilities: a (K x N)(N x D) product
        # (the full M-step statistics would also form K D^2 second moments nobody reads)
        resp.zero_()
        resp[lab, rows] = 1.0
        moments = torch.empty((k, d + 1), **f64)
        moments[:, :d] = resp[:, :n] @ x
        moments[:, d] = resp[:, :n].sum(dim=1)
        if multi:
            dist.all_reduce(moments, group=group)
        counts = moments[:, d]
        nz = counts > 0
        moved = centres.clone()
        moved[nz] = moments[nz, :d] / counts[nz][:, None]
        shift = ((moved - centres) ** 2).sum()
        centres = moved.contiguous()
        if n_lloyd > 0 and bool(shift <= shift_tol):
            # converged: one more assignment with the final centres, as sklearn does
            aux[:, :d] = centres
            _lib.call('kw_gmm_hard_labels', n, x, k, d, centres, eye, aux, labels, precision, ws,
                      ws_bytes, stream)
            break
    return labels.long()
