"""Delta features on the device (kwiiyatta/converter/delta.py:8-12,30,46)."""
import numpy as np

from . import _lib

# kwiiyatta/converter/delta.py:8-12 -- the only windows the kernels implement
DELTA_WINDOWS = [
    (0, 0, np.array([1.0])),
    (1, 1, np.array([-0.5, 0.0, 0.5])),
    (1, 1, np.array([1.0, -2.0, 1.0])),
]


def check_windows(windows):
    if len(windows) != len(DELTA_WINDOWS) or any(
            (a[0], a[1]) != (b[0], b[1]) or not np.array_equal(a[2], b[2])
            for a, b in zip(windows, DELTA_WINDOWS)):
        raise NotImplementedError('only kwiiyatta DELTA_WINDOWS are built into the kernels')


@_lib.device_guard(lambda x_dev, *a: x_dev.device)
def delta_features_device(x_dev, offsets_dev, n_utts):
    """x_dev (sum T, dim) float64 CUDA tensor, offsets (n_utts + 1) int64 -> (sum T, 3 dim)."""
    torch = _lib.require_cuda()
    total, dim = x_dev.shape
    out = torch.empty((total, 3 * dim), dtype=torch.float64, device=x_dev.device)
    _lib.call('kw_delta_features', n_utts, offsets_dev, total, dim, x_dev, out,
              _lib.stream_ptr(torch))
    return out


def delta_features(x, windows=DELTA_WINDOWS):
    """``nnmnkwii.preprocessing.delta_features(x, DELTA_WINDOWS)`` for one utterance."""
    torch = _lib.require_cuda()
    check_windows(windows)
    x = np.ascontiguousarray(x, dtype=np.float64)
    x_dev = torch.from_numpy(x).cuda()
    off = torch.tensor([0, len(x)], dtype=torch.int64, device='cuda')
    return delta_features_device(x_dev, off, 1).cpu().numpy()
