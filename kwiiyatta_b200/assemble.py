"""Device-resident training-array assembly (SURVEY.md section 8f row 2).

``joint_frames_device(pairs, ...)`` = ``align_even`` -> mel-cepstra without c0 -> delta features
-> hstack -> zero-frame removal for a list of (source, target) features, computed where the
reference computes it per pair on the host (kwiiyatta/vocoder/align.py:61-96,134-146,
kwiiyatta/converter/{mcep,delta,dataset}.py), but as five launches over the whole batch on the
device; the (N, 144) result stays in HBM for GaussianMixture.fit.  Only the mel-cepstra, one
voicing byte per frame and one threshold per utterance go up, and one int per pair comes back
(the aligned lengths, for the row offsets)."""
import numpy as np

from . import _lib
from . import alignment as _align
from . import hooks
from .fastdtw import fastdtw_batch_device

_POWER_MODES = {'binalize': 0, 'raw': 1, None: 2}


def joint_frames_device(pairs, use_delta=True, pad_silence=True, pad_len=100, vuv='voiced',
                        power='binalize', strict=True, radius=32, vuv_weight=9.0,
                        power_weight=9.4, power_pivot='max', power_threshold=1.636, device=None,
                        return_paths=False, return_offsets=False):
    """(N, 2 * (3 or 1) * order) float64 CUDA tensor of joint frames for ``pairs``.
    ``return_offsets``: also the int64 CUDA tensor of row offsets (n + 1) of each pair's rows
    after the zero-frame removal."""
    torch = _lib.require_cuda()
    dev = torch.device('cuda' if device is None else device)
    if power not in _POWER_MODES:
        raise ValueError(f'Unknown power parameter: {power!r}')
    if vuv not in ('voiced', 'f0', None):
        raise ValueError(f'Unknown vuv parameter: {vuv!r}')
    if power == 'binalize' and power_pivot not in _align._POWER_PIVOTS:
        raise ValueError(f'Unknown power_pivot parameter: {power_pivot!r}')
    if pad_silence:
        pad = hooks.get('pad_silence')
        pairs = [(pad(a, pad_len), pad(b, pad_len)) for a, b in pairs]
    n = len(pairs)
    if n == 0:
        empty = torch.zeros((0, 0), dtype=torch.float64, device=dev)
        return (empty, torch.zeros(1, dtype=torch.int64, device=dev)) if return_offsets else empty
    sides = []
    for which in (0, 1):
        mceps, flags, thr = [], [], []
        for pair in pairs:
            f = pair[which]
            fs = min(pair[0].fs, pair[1].fs)
            data = np.ascontiguousarray(f.resample_mel_cepstrum(fs).data, dtype=np.float64)
            mceps.append(data)
            if vuv == 'voiced':
                flags.append(np.asarray(f.is_voiced, dtype=np.uint8))
            elif vuv == 'f0':
                flags.append((np.asarray(f.f0) > 0).astype(np.uint8))
            if power == 'binalize':
                thr.append(_align._POWER_PIVOTS[power_pivot](data[:, 0], power_threshold))
        lens = np.array([len(m) for m in mceps], dtype=np.int64)
        sides.append((mceps, flags, np.array(thr, dtype=np.float64), lens))
    width = sides[0][0][0].shape[1]
    with torch.cuda.device(dev):
        stream = _lib.stream_ptr(torch)
        dev_side = []
        for mceps, flags, thr, lens in sides:
            off = np.concatenate(([0], np.cumsum(lens)))
            m_dev = _lib.gather_to_device(torch, mceps, dev, f'asm_m{len(dev_side)}')
            v_dev = torch.from_numpy(np.concatenate(flags)).to(dev) if flags else None
            t_dev = torch.from_numpy(thr).to(dev) if len(thr) else None
            off_dev = torch.from_numpy(off).to(dev)
            feat = torch.empty((int(off[-1]), width + 1), dtype=torch.float64, device=dev)
            _lib.call('kw_dtw_features', n, off_dev, int(off[-1]), width, m_dev, v_dev, t_dev,
                      _POWER_MODES[power], float(power_weight), float(vuv_weight), feat, stream)
            dev_side.append((m_dev, feat, off_dev, lens))
        (xm, xf, xoff, tx), (ym, yf, yoff, ty) = dev_side
        res = fastdtw_batch_device(xf, yf, tx.astype(np.int32), ty.astype(np.int32),
                                   radius=radius, dist=2)
        region_off = torch.from_numpy(res.region_off).to(dev)
        tx_dev = torch.from_numpy(tx.astype(np.int32)).to(dev)
        ty_dev = torch.from_numpy(ty.astype(np.int32)).to(dev)
        sel_len = torch.empty(n, dtype=torch.int32, device=dev)
        _lib.call('kw_path_select', n, region_off, res.path_begin, res.path_len, tx_dev, ty_dev,
                  xoff, yoff, xf, yf, width + 1, int(bool(strict)), int(power == 'binalize'),
                  int(vuv is not None), int(bool(pad_silence)), int(pad_len), res.path, sel_len,
                  stream)
        out_off = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        out_off[1:] = torch.cumsum(sel_len.long(), dim=0)
        total = int(out_off[-1].item())             # the one read-back: N, for the allocation
        cols = 2 * (3 if use_delta else 1) * (width - 1)
        out = torch.empty((total, cols), dtype=torch.float64, device=dev)
        if total:
            zero = torch.empty(total, dtype=torch.uint8, device=dev)
            _lib.call('kw_joint_frames', n, out_off, total, region_off, res.path, xoff, yoff, xm,
                      ym, width, int(bool(use_delta)), out, zero, stream)
            row_off = out_off
            if bool(zero.any()):                    # rare: silent frames inside an utterance
                out = out[~zero.bool()].contiguous()
                dropped = torch.zeros(total + 1, dtype=torch.int64, device=dev)
                dropped[1:] = torch.cumsum(zero.long(), dim=0)
                row_off = out_off - dropped[out_off]
        else:
            row_off = out_off
    if return_paths:
        return out, (res, sel_len, out_off)
    if return_offsets:
        return out, row_off
    return out
