"""Drop-in for the third-party ``fastdtw`` module on the B200.

The reference imports ``fastdtw`` at module scope (kwiiyatta/vocoder/align.py:3) and calls
``fastdtw.fastdtw(x_feature, y_feature, dist=2, radius=radius)`` once (:71); its tests also
call ``fastdtw.fastdtw(a, b, radius=1, dist=2)`` (tests/kwiiyatta/test_vocoder.py:281-286).
This module keeps those signatures and return types ``(float, list[tuple[int, int]])`` and
adds the batched entry points the GPU needs (``fastdtw_batch``); the single-pair functions are
the batch-of-one case.  All arithmetic runs in kw_dtw_batch (csrc/dtw.cu).
"""
import numbers

import numpy as np

from . import _lib


def _norm_from_dist(dist, ndim):
    if dist is None:
        return 1                       # fastdtw default: |a-b| (1-D) or the 1-norm (2-D)
    if callable(dist):
        raise NotImplementedError('callable dist is not supported on the GPU path; use 1 or 2')
    if isinstance(dist, numbers.Number):
        if dist <= 0:
            raise ValueError('dist cannot be a negative integer')
        if dist in (1, 2):
            return int(dist)
        raise NotImplementedError(f'dist={dist!r}: only the 1- and 2-norm are built')
    raise TypeError(f'unsupported dist {dist!r}')


def _prep(x):
    x = np.asanyarray(x, dtype='float')
    if x.ndim == 1:
        x = x[:, None]
    if x.ndim != 2:
        raise ValueError('x and y must be 1-D or 2-D')
    return np.ascontiguousarray(x, dtype=np.float64)


class DtwBatchResult:
    """Device-resident result of a batched alignment."""

    def __init__(self, cost, path, path_begin, path_len, cells, tx, ty, margin=None):
        self.cost, self.path, self.path_begin, self.path_len, self.cells = (
            cost, path, path_begin, path_len, cells)
        # (n, 2) smallest decision margin on the path: finest level, all levels (or None)
        self.margin = margin
        self.tx, self.ty = tx, ty
        region = (tx.astype(np.int64) + ty.astype(np.int64))
        self.region_off = np.concatenate(([0], np.cumsum(region)))

    def to_host(self):
        """list of (distance: float, path: (L, 2) int32 ndarray)."""
        cost = self.cost.cpu().tolist()
        path = self.path.cpu().numpy()
        first = (self.region_off[:-1] + self.path_begin.cpu().numpy()).tolist()
        length = self.path_len.cpu().tolist()
        return [(cost[p], path[first[p]:first[p] + length[p]]) for p in range(len(cost))]


TIE_MODES = {'python': 0, 'cython': 1, 0: 0, 1: 1}


@_lib.device_guard(lambda x_dev, *a: x_dev.device)
def fastdtw_batch_device(x_dev, y_dev, tx, ty, radius=1, dist=2, precision=0, tie_mode='python',
                         with_margin=False):
    """Batched FastDTW on device-resident, row-concatenated float64 inputs.

    x_dev (sum tx, F), y_dev (sum ty, F) CUDA tensors; tx / ty host int arrays.
    ``radius < 0`` = exhaustive DTW.  ``tie_mode``: which fastdtw back-end's tie order to follow
    ('python', the default and what the oracle restates, or 'cython').  ``with_margin``: also
    return the smallest decision margin on each path (``result.margin``, (n, 2): the returned
    path, all resolution levels).  Returns a DtwBatchResult (device tensors)."""
    torch = _lib.require_cuda()
    tx = np.ascontiguousarray(tx, dtype=np.int32)
    ty = np.ascontiguousarray(ty, dtype=np.int32)
    n = len(tx)
    f = x_dev.shape[1]
    if y_dev.shape[1] != f:
        raise ValueError('second dimension of x and y must be the same')
    p_norm = _norm_from_dist(dist, 2)
    dev = x_dev.device
    ws_bytes = _lib.lib().kw_dtw_workspace_bytes(n, _lib.ptr(tx), _lib.ptr(ty), f, int(radius))
    total_pts = int(tx.astype(np.int64).sum() + ty.astype(np.int64).sum())
    cost = torch.empty(n, dtype=torch.float64, device=dev)
    path = torch.empty((total_pts, 2), dtype=torch.int32, device=dev)
    begin = torch.empty(n, dtype=torch.int32, device=dev)
    length = torch.empty(n, dtype=torch.int32, device=dev)
    cells = torch.empty(n, dtype=torch.int64, device=dev)
    margin = torch.empty((n, 2), dtype=torch.float64, device=dev) if with_margin else None
    _lib.call('kw_dtw_batch', n, x_dev, y_dev, tx, ty, f, int(radius), p_norm, int(precision),
              TIE_MODES[tie_mode], cost, path, begin, length, cells, margin,
              _lib.workspace(ws_bytes, dev), ws_bytes, _lib.stream_ptr(torch))
    return DtwBatchResult(cost, path, begin, length, cells, tx, ty, margin)


def fastdtw_batch(pairs, radius=1, dist=2, precision=0, device=None, tie_mode='python',
                  with_margin=False):
    """``pairs``: sequence of (x, y) host arrays.  Returns a list of
    ``(distance, path ndarray (L, 2))`` in the same order; with ``with_margin`` a pair
    ``(that list, margins ndarray (n, 2))``."""
    torch = _lib.require_cuda()
    if len(pairs) == 0:
        return []
    xs = [_prep(x) for x, _ in pairs]
    ys = [_prep(y) for _, y in pairs]
    for x, y in zip(xs, ys):
        if x.shape[1] != y.shape[1]:
            raise ValueError('second dimension of x and y must be the same')
        if len(x) == 0 or len(y) == 0:
            raise ValueError('x and y must not be empty')
    if any(x.shape[1] != xs[0].shape[1] for x in xs):
        raise ValueError('all pairs of a batch must have the same number of features')
    _norm_from_dist(dist, 2)
    dev = torch.device('cuda' if device is None else device)
    tx = np.array([len(x) for x in xs], dtype=np.int32)
    ty = np.array([len(y) for y in ys], dtype=np.int32)
    x_dev = _lib.gather_to_device(torch, xs, dev, 'dtw_x')
    y_dev = _lib.gather_to_device(torch, ys, dev, 'dtw_y')
    res = fastdtw_batch_device(x_dev, y_dev, tx, ty, radius, dist, precision, tie_mode,
                               with_margin)
    if with_margin:
        return res.to_host(), res.margin.cpu().numpy()
    return res.to_host()


def fastdtw_batch_packed(x_host, y_host, tx, ty, radius=1, dist=2, precision=0,
                         tie_mode='python', device=None, n_chunks=None):
    """Batched FastDTW from two host tensors holding all x (sum tx, F) and all y (sum ty, F)
    rows -- pinned memory for full speed.  The pairs are split into chunks that go through
    copy-in / kernels / copy-out on separate streams, so the upload of one chunk overlaps the
    kernels of the previous one.  Returns the list ``fastdtw_batch`` returns."""
    torch = _lib.require_cuda()
    dev = torch.device('cuda' if device is None else device)
    tx = np.ascontiguousarray(tx, dtype=np.int32)
    ty = np.ascontiguousarray(ty, dtype=np.int32)
    n = len(tx)
    if n == 0:
        return []
    if x_host.shape[1] != y_host.shape[1]:
        raise ValueError('second dimension of x and y must be the same')
    if n_chunks is None:
        n_chunks = 2 if n >= 296 else 1          # keep >= one wave of CTAs (148 SMs) per chunk
    xrow = np.concatenate(([0], np.cumsum(tx.astype(np.int64))))
    yrow = np.concatenate(([0], np.cumsum(ty.astype(np.int64))))
    bounds = [n * c // n_chunks for c in range(n_chunks + 1)]
    results = []
    with torch.cuda.device(dev):
        main = torch.cuda.current_stream(dev)
        streams = _lib.staging('dtw_packed', dev).setdefault('streams', [])
        while len(streams) < n_chunks:
            streams.append(torch.cuda.Stream(dev))
        streams = streams[:n_chunks] if n_chunks > 1 else [main]
        start = torch.cuda.Event()
        start.record(main)
        parts = []
        for c in range(n_chunks):
            a, b = bounds[c], bounds[c + 1]
            st = streams[c]
            with torch.cuda.stream(st):
                st.wait_event(start)
                xd = x_host[int(xrow[a]):int(xrow[b])].to(dev, non_blocking=True)
                yd = y_host[int(yrow[a]):int(yrow[b])].to(dev, non_blocking=True)
                res = fastdtw_batch_device(xd, yd, tx[a:b], ty[a:b], radius, dist, precision,
                                           tie_mode)
                host = {k: _lib.pinned(('dtw_packed', c, k), dev, t.shape, t.dtype)
                        for k, t in (('cost', res.cost), ('path', res.path),
                                     ('begin', res.path_begin), ('len', res.path_len))}
                host['cost'].copy_(res.cost, non_blocking=True)
                host['path'].copy_(res.path, non_blocking=True)
                host['begin'].copy_(res.path_begin, non_blocking=True)
                host['len'].copy_(res.path_len, non_blocking=True)
                done = torch.cuda.Event()
                done.record(st)
            parts.append((res, host, done, (xd, yd)))
        for res, host, done, _ in parts:
            done.synchronize()
            main.wait_event(done)
            cost = host['cost'].tolist()
            path = host['path'].numpy().copy()
            first = (res.region_off[:-1] + host['begin'].numpy()).tolist()
            length = host['len'].tolist()
            results.extend((cost[p], path[first[p]:first[p] + length[p]])
                           for p in range(len(cost)))
    return results


def fastdtw(x, y, radius=1, dist=None):
    """``fastdtw.fastdtw``: approximate DTW distance and path ``[(i, j), ...]``."""
    cost, path = fastdtw_batch([(x, y)], radius=radius, dist=dist)[0]
    return cost, [tuple(p) for p in path.tolist()]


def dtw(x, y, dist=None):
    """``fastdtw.dtw``: exhaustive DTW."""
    cost, path = fastdtw_batch([(x, y)], radius=-1, dist=dist)[0]
    return cost, [tuple(p) for p in path.tolist()]
