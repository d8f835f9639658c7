"""Global-variance (GV) statistics for GV-considered conversion (Toda, Black & Tokuda, IEEE
TASLP 15(8), 2007).

The GV of an utterance is the variance over time of each static feature dimension.  GMM
conversion by MLPG under-shoots it (the output is over-smoothed); ``MLPG(..., gv=...)`` and
``B200GMMFeatureConverter(gv=True)`` pull it back towards the statistics estimated here:
mu_v, the mean of the per-utterance variances, and sigma^2_v, their population variance (floored
at 1e-12), per dimension.  The estimate runs on the device (kw_gv_estimate, fixed summation
order); with ``torch.distributed`` initialised the per-rank sums [sum v | sum v^2 | count] are
all-reduced first, so every rank holds the same statistics."""
import numpy as np

from . import _lib


class GlobalVariance:
    """mu_v (``mean``) and sigma^2_v (``var``) per static dimension, float64 numpy arrays."""

    def __init__(self, mean, var):
        self.mean = np.ascontiguousarray(mean, dtype=np.float64).reshape(-1)
        self.var = np.ascontiguousarray(var, dtype=np.float64).reshape(-1)
        if self.mean.shape != self.var.shape:
            raise ValueError('GV mean and var must have the same length')
        if not (np.all(np.isfinite(self.mean)) and np.all(self.mean >= 0)
                and np.all(self.var > 0)):
            raise ValueError('GV statistics need mean >= 0 and var > 0')

    def __len__(self):
        return len(self.mean)

    def __repr__(self):
        return f'GlobalVariance(dim={len(self)})'


def as_gv(gv):
    """A ``GlobalVariance`` from one, from a dict with ``mean`` / ``var`` or a (mean, var) pair."""
    if isinstance(gv, GlobalVariance):
        return gv
    if isinstance(gv, dict):
        return GlobalVariance(gv['mean'], gv['var'])
    mean, var = gv
    return GlobalVariance(mean, var)


def estimate_gv(features, columns=None, process_group=None, device=None):
    """GV statistics of a set of utterances.

    ``features``: a list of (T_i, F) arrays, or ``(x, offsets)`` with ``x`` a (N, F) float64 CUDA
    tensor holding the utterances row after row and ``offsets`` their int64 row offsets
    (n + 1 values, numpy or tensor).  ``columns``: ``(first, count)``, the feature columns to
    take (default: all).  Utterances without frames are left out."""
    torch = _lib.require_cuda()
    if isinstance(features, tuple) and len(features) == 2 and hasattr(features[0], 'data_ptr'):
        x, offsets = features
        dev = x.device
        if not x.is_cuda or x.dtype != torch.float64 or x.dim() != 2:
            raise ValueError('x must be a 2-D float64 CUDA tensor')
        x = x.contiguous()
        if hasattr(offsets, 'data_ptr'):
            off = offsets.to(device=dev, dtype=torch.int64).contiguous()
        else:
            off = torch.from_numpy(np.asarray(offsets, dtype=np.int64)).to(dev)
    else:
        feats = [np.ascontiguousarray(f, dtype=np.float64) for f in features]
        if not feats or any(f.ndim != 2 or f.shape[1] != feats[0].shape[1] for f in feats):
            raise ValueError('features must be a non-empty list of (T, F) arrays of equal F')
        dev = torch.device('cuda' if device is None else device)
        lens = np.array([len(f) for f in feats], dtype=np.int64)
        off = torch.from_numpy(np.concatenate(([0], np.cumsum(lens)))).to(dev)
        x = torch.from_numpy(np.concatenate(feats)).to(dev)
    n_utts = int(off.numel()) - 1
    width = int(x.shape[1])
    col0, ncols = (0, width) if columns is None else (int(columns[0]), int(columns[1]))
    if n_utts < 1 or not (0 <= col0 and ncols > 0 and col0 + ncols <= width):
        raise ValueError(f'bad utterance offsets or columns {columns} for width {width}')
    if int(off[-1].item()) != x.shape[0]:
        raise ValueError('offsets do not cover the rows of x')
    f64 = dict(dtype=torch.float64, device=dev)
    utt_var = torch.empty((n_utts, ncols), **f64)
    sums = torch.empty(2 * ncols + 1, **f64)
    mean = torch.empty(ncols, **f64)
    var = torch.empty(ncols, **f64)
    with torch.cuda.device(dev):
        stream = _lib.stream_ptr(torch)
        _lib.call('kw_gv_estimate', n_utts, off, int(x.shape[0]), width, col0, ncols, x, utt_var,
                  sums, mean, var, stream)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and \
                dist.get_world_size(process_group) > 1:
            from . import dist as kdist
            kdist.allreduce_stats(sums, process_group)
            _lib.call('kw_gv_from_sums', ncols, sums, mean, var, stream)
        if float(sums[-1].item()) < 1:
            raise ValueError('no utterance with frames to estimate the GV from')
    return GlobalVariance(mean.cpu().numpy(), var.cpu().numpy())
