"""ctypes binding of libkwiiyatta_b200.so (the C ABI in include/kwiiyatta_b200.h).

There is no CPU fallback: if the library is missing or a call fails, this raises."""
import ctypes

import numpy as np
import os

from . import build as _build

_c = ctypes
_lib = None

KW_ERR_INVALID = -1
KW_ERR_WORKSPACE = -2
KW_ERR_UNSUPPORTED = -3
KW_ERR_CUDA = -4

_vp, _i, _i64, _sz, _dbl = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_size_t, _c.c_double

SIGNATURES = {
    'kw_abi_version': (_i, []),
    'kw_last_error': (_c.c_char_p, []),
    'kw_device_info': (_i, [_i, _vp, _vp, _vp, _vp]),
    'kw_dtw_workspace_bytes': (_sz, [_i, _vp, _vp, _i, _i]),
    'kw_dtw_batch': (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp,
                          _vp, _vp, _sz, _vp]),
    'kw_delta_features': (_i, [_i, _vp, _i64, _i, _vp, _vp, _vp]),
    'kw_gmm_stats_len': (_sz, [_i, _i]),
    'kw_gmm_resp_len': (_sz, [_i64, _i]),
    'kw_gmm_workspace_bytes': (_sz, [_i64, _i, _i, _i]),
    'kw_gmm_pack_frames': (_i, [_i64, _vp, _i, _i, _i, _vp, _sz, _vp]),
    'kw_gmm_estep': (_i, [_i64, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _sz, _vp]),
    'kw_gmm_normalize_resp': (_i, [_i64, _i, _i, _vp, _vp, _sz, _vp]),
    'kw_gmm_hard_labels': (_i, [_i64, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp]),
    'kw_gmm_mstep_accumulate': (_i, [_i64, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _sz, _vp]),
    'kw_gmm_mstep_finalize': (_i, [_i, _i, _dbl, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                   _vp]),
    'kw_gmm_precision_cholesky': (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'kw_convert_prepared_len': (_sz, [_i, _i]),
    'kw_convert_prepare': (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    'kw_convert_soft_workspace_bytes': (_sz, [_i64, _i, _i]),
    'kw_convert_soft_batch': (_i, [_i64, _vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'kw_mc2b': (_i, [_i64, _i, _dbl, _i, _vp, _vp, _vp]),
    'kw_dtw_features': (_i, [_i, _vp, _i64, _i, _vp, _vp, _vp, _i, _dbl, _dbl, _vp, _vp]),
    'kw_path_select': (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i,
                            _i, _vp, _vp, _vp]),
    'kw_joint_frames': (_i, [_i, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    'kw_convert_workspace_bytes': (_sz, [_i64, _i, _i, _i]),
    'kw_convert_batch': (_i, [_i, _vp, _i64, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _vp, _sz,
                              _vp]),
    'kw_gv_estimate': (_i, [_i, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    'kw_gv_from_sums': (_i, [_i, _vp, _vp, _vp, _vp]),
    'kw_convert_gv_workspace_bytes': (_sz, [_i64, _i, _i, _i]),
    'kw_convert_gv_batch': (_i, [_i, _vp, _i64, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _dbl, _dbl,
                                 _vp, _i, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp]),
}


class KwError(RuntimeError):
    pass


def lib():
    """The loaded library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        path = _build.LIB_PATH
        if not os.path.exists(path):
            raise KwError(
                f'{path} is missing: build it with `python -m kwiiyatta_b200.build` '
                '(nvcc, sm_100a). kwiiyatta_b200 has no CPU fallback.')
        handle = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what):
    if rc == 0:
        return
    msg = lib().kw_last_error().decode('utf-8', 'replace')
    text = f'{what} failed ({rc}): {msg}'
    if rc == KW_ERR_INVALID:
        raise ValueError(text)
    if rc == KW_ERR_UNSUPPORTED:
        raise NotImplementedError(text)
    raise KwError(text)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise KwError('kwiiyatta_b200 needs a CUDA device (B200, sm_100a); there is no CPU '
                      'fallback')
    return torch


def ptr(t):
    """Device (or host numpy) pointer as an int for ctypes."""
    if t is None:
        return None
    if hasattr(t, 'data_ptr'):
        return t.data_ptr()
    return t.ctypes.data


def stream_ptr(torch):
    return torch.cuda.current_stream().cuda_stream


def device_guard(device_of):
    """Decorator: run the call with the CUDA device of its data current, so the C-ABI launches
    (which go to ``torch.cuda.current_stream()`` of the CURRENT device) land on the GPU that
    owns the pointers.  ``device_of(self_or_first_arg, *args)`` returns a torch device or None
    (= leave the current device alone)."""
    import functools

    def wrap(fn):
        @functools.wraps(fn)
        def guarded(*args, **kwargs):
            dev = device_of(*args)
            if dev is None:
                return fn(*args, **kwargs)
            torch = require_cuda()
            dev = torch.device(dev)
            if dev.type != 'cuda' or dev.index is None:
                return fn(*args, **kwargs)
            with torch.cuda.device(dev):
                return fn(*args, **kwargs)
        return guarded
    return wrap


# Pinned staging buffers (and the side streams of the packed host APIs) kept between calls: pinning
# is far more expensive than the copy, and the caching allocator keeps one pool per stream.  This
# is a per-process cache of the Python host layer (the C ABI itself keeps no state); calls that
# share a slot must not run concurrently from several host threads.
# slot -> (tensor, event of the last copy that read it) or a dict of buffers
_STAGING = {}
_GATHER_THREADS = max(4, min(32, os.cpu_count() or 8))
_POOL = None


def copy_pool():
    """Threads for host-side copies into / out of pinned memory (numpy releases the GIL)."""
    global _POOL
    if _POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _POOL = ThreadPoolExecutor(_GATHER_THREADS)
    return _POOL


def parallel_copy(jobs):
    """``jobs``: list of (dst_view, src_array) pairs, copied by the pool; blocks until done."""
    if not jobs:
        return
    total = sum(src.nbytes for _, src in jobs)
    if total < (1 << 21) or len(jobs) == 1:
        for dst, src in jobs:
            dst[...] = src
        return
    step = max(1, (len(jobs) + 4 * _GATHER_THREADS - 1) // (4 * _GATHER_THREADS))

    def run(lo):
        for dst, src in jobs[lo:lo + step]:
            dst[...] = src
    list(copy_pool().map(run, range(0, len(jobs), step)))


def gather_to_device(torch, arrays, dev, slot):
    """Row-concatenate ``arrays`` into a pinned buffer (several threads; numpy releases the
    GIL while copying) and start one asynchronous copy to ``dev``."""
    from concurrent.futures import ThreadPoolExecutor
    rows = np.array([len(a) for a in arrays], dtype=np.int64)
    f = arrays[0].shape[1]
    total = int(rows.sum())
    key = (slot, str(dev))
    buf, ev = _STAGING.get(key, (None, None))
    if buf is None or buf.numel() < total * f:
        buf = torch.empty(max(total * f, 1), dtype=torch.float64).pin_memory()
        ev = None
    if ev is not None:
        ev.synchronize()            # the previous batch's copy has left the buffer
    view = buf[:total * f].view(total, f)
    host = view.numpy()
    off = np.concatenate(([0], np.cumsum(rows)))
    n = len(arrays)
    step = max(1, (n + 4 * _GATHER_THREADS - 1) // (4 * _GATHER_THREADS))

    def copy(lo):
        for i in range(lo, min(n, lo + step)):
            host[off[i]:off[i + 1]] = arrays[i]

    if total * f * 8 < (1 << 22) or n == 1:
        copy(0) if n == 1 else [copy(lo) for lo in range(0, n, step)]
    else:
        list(copy_pool().map(copy, range(0, n, step)))
    out = view.to(dev, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(dev))
    _STAGING[key] = (buf, ev)
    return out


def scatter_to_host(torch, tensor, offsets, slot):
    """Device (rows, F) tensor -> list of freshly allocated host arrays, rows
    ``offsets[i]:offsets[i + 1]`` each: one copy into a pinned buffer kept between calls, then
    the per-segment copies on several threads."""
    from concurrent.futures import ThreadPoolExecutor
    total, f = tensor.shape
    key = (slot, str(tensor.device))
    buf, _ = _STAGING.get(key, (None, None))
    if buf is None or buf.numel() < total * f or buf.dtype != tensor.dtype:
        buf = torch.empty(max(total * f, 1), dtype=tensor.dtype).pin_memory()
    _STAGING[key] = (buf, None)
    view = buf[:total * f].view(total, f)
    view.copy_(tensor, non_blocking=True)
    torch.cuda.current_stream(tensor.device).synchronize()
    host = view.numpy()
    n = len(offsets) - 1
    out = [None] * n
    step = max(1, (n + _GATHER_THREADS - 1) // _GATHER_THREADS)

    def copy(lo):
        for i in range(lo, min(n, lo + step)):
            out[i] = host[offsets[i]:offsets[i + 1]].copy()

    if total * f * tensor.element_size() < (1 << 22) or n == 1:
        for lo in range(0, n, step):
            copy(lo)
    else:
        list(copy_pool().map(copy, range(0, n, step)))
    return out
