"""ctypes binding of libkwiiyatta_b200.so (the C ABI in include/kwiiyatta_b200.h).

There is no CPU fallback: if the library is missing or a call fails, this raises."""
import ctypes
import math
import os

import numpy as np

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
    'kw_gmm_db_stats_len': (_sz, [_i, _i]),
    'kw_gmm_db_workspace_bytes': (_sz, [_i64, _i, _i]),
    'kw_gmm_db_estep': (_i, [_i64, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'kw_gmm_db_mstep_accumulate': (_i, [_i64, _vp, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'kw_gmm_db_mstep_finalize': (_i, [_i, _i, _dbl, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                      _vp, _vp]),
    'kw_gmm_db_precision_cholesky': (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
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
    'kw_convert_em_workspace_bytes': (_sz, [_i64, _i, _i, _i]),
    'kw_convert_em_batch': (_i, [_i, _vp, _i64, _vp, _i, _i, _vp, _i, _vp, _vp, _i, _vp, _sz,
                                 _vp]),
    'kw_convert_fullcov_prepared_len': (_sz, [_i, _i]),
    'kw_convert_fullcov_prepare_workspace_bytes': (_sz, [_i, _i]),
    'kw_convert_fullcov_prepare': (_i, [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'kw_convert_fullcov_workspace_bytes': (_sz, [_i64, _i, _i, _i]),
    'kw_convert_fullcov_batch': (_i, [_i, _vp, _i64, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _i,
                                      _vp, _sz, _vp]),
    'kw_convert_stream_state_len': (_sz, [_i, _i, _i]),
    'kw_convert_stream_init': (_i, [_i, _i, _i, _vp, _vp]),
    'kw_convert_stream_workspace_bytes': (_sz, [_i, _i, _i, _i, _i]),
    'kw_convert_stream_push': (_i, [_i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp,
                                    _sz, _vp]),
    'kw_convert_stream_end': (_i, [_i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _sz,
                                   _vp]),
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


def call(name, *args):
    """``lib().<name>(*args)`` for an entry point that returns a status: torch tensors, numpy
    arrays and None go in as pointers (``ptr``), everything else as it is, for ctypes to convert
    and range-check; a non-zero status raises (``check``).  The size queries
    (``kw_*_len``, ``kw_*_workspace_bytes``) return sizes and are called on ``lib()``."""
    rc = getattr(lib(), name)(*[
        ptr(a) if a is None or isinstance(a, np.ndarray) or hasattr(a, 'data_ptr') else a
        for a in args])
    check(rc, name)


def workspace(nbytes, device):
    """Device workspace of ``nbytes`` bytes (at least one, so that it has an address)."""
    import torch
    return torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)


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


# Host buffers and side streams of the host APIs, kept between calls per (slot, device): pinning
# costs far more than the copies, and the caching allocator keeps one pool per stream.  This is a
# per-process cache of the Python host layer (the C ABI itself keeps no state); calls that share
# a slot must not run concurrently from several host threads.
# (slot, device) -> (pinned tensor, event of the last copy that read it) or a dict (``staging``)
_STAGING = {}
_GATHER_THREADS = max(4, min(32, os.cpu_count() or 8))
_POOL = None


def pinned(slot, dev, shape, dtype):
    """Pinned host tensor of ``shape`` and ``dtype``, kept for (``slot``, ``dev``) between calls
    and reallocated only when too small.  The next call for the slot hands out the same memory,
    so every caller keeps one of these rules:

    * an asynchronous copy that may still read the buffer when the caller returns is recorded
      with ``pinned_in_flight``; the next call for the slot waits for it (``gather_to_device``);
    * what the caller returns from the buffer is copied out of it, never a view of it
      (``fastdtw_batch_packed``);
    * the caller synchronises before it returns (``MLPG.transform_many``, whose
      ``transform_packed`` does)."""
    key = (slot, str(dev))
    numel = math.prod(shape)
    buf, ev = _STAGING.get(key, (None, None))
    if buf is None or buf.numel() < numel or buf.dtype != dtype:
        import torch
        buf, ev = torch.empty(max(numel, 1), dtype=dtype).pin_memory(), None
    if ev is not None:
        ev.synchronize()
    _STAGING[key] = (buf, None)
    return buf[:numel].view(shape)


def pinned_in_flight(slot, dev, stream):
    """Record that the work queued so far on ``stream`` reads the ``pinned`` buffer of
    (``slot``, ``dev``)."""
    import torch
    key = (slot, str(dev))
    ev = torch.cuda.Event()
    ev.record(stream)
    _STAGING[key] = (_STAGING[key][0], ev)


def staging(slot, dev):
    """The dict kept for (``slot``, ``dev``) between calls, for the device buffers and side
    streams of the packed host APIs."""
    return _STAGING.setdefault((slot, str(dev)), {})


def copy_pool():
    """Threads for host-side copies into / out of pinned memory (numpy releases the GIL)."""
    global _POOL
    if _POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _POOL = ThreadPoolExecutor(_GATHER_THREADS)
    return _POOL


def parallel_copy(jobs):
    """``jobs``: list of (dst_view, src_array) pairs, copied by the pool; blocks until done.
    Below 2 MB in all, or for a single pair, the calling thread copies alone."""
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
    """Row-concatenate ``arrays`` into the pinned buffer of ``slot`` (``parallel_copy``) and start
    one asynchronous copy to ``dev``."""
    off = np.concatenate(([0], np.cumsum([len(a) for a in arrays])))
    buf = pinned(slot, dev, (int(off[-1]), arrays[0].shape[1]), torch.float64)
    host = buf.numpy()
    parallel_copy([(host[off[i]:off[i + 1]], a) for i, a in enumerate(arrays)])
    out = buf.to(dev, non_blocking=True)
    pinned_in_flight(slot, dev, torch.cuda.current_stream(dev))
    return out
