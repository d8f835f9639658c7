"""Hand-off from the converter to the MLSA differential filter (kwiiyatta/filter/mlsa.py:9-30).

The filter itself (pysptk.synthesis.MLSADF over the waveform) is waveform synthesis and stays
with the reference; what sits directly behind the converter's output is the per-frame
mel-cepstrum -> filter-coefficient recursion ``pysptk.mc2b``, which this module runs on the
device for whole batches of converted utterances."""
import numpy as np

from . import _lib


def mc2b_many(mceps, alpha, zero_power=True):
    """``pysptk.mc2b(mc, alpha)`` for a list of (T_i, order + 1) mel-cepstrum arrays; with
    ``zero_power`` column 0 is zeroed first, as ``apply_mlsa_filter`` does (mlsa.py:23)."""
    torch = _lib.require_cuda()
    mceps = [np.ascontiguousarray(m, dtype=np.float64) for m in mceps]
    lens = [len(m) for m in mceps]
    if sum(lens) == 0:
        return [np.zeros_like(m) for m in mceps]
    width = mceps[0].shape[1]
    if any(m.ndim != 2 or m.shape[1] != width for m in mceps):
        raise ValueError('all mel-cepstra must be (T, order + 1) with the same order')
    x = torch.from_numpy(np.concatenate(mceps)).cuda()
    _lib.call('kw_mc2b', x.shape[0], width, float(alpha), int(bool(zero_power)), x, x,
              _lib.stream_ptr(torch))
    out = x.cpu().numpy()
    off = np.concatenate(([0], np.cumsum(lens)))
    return [out[off[i]:off[i + 1]] for i in range(len(mceps))]


def mc2b(mcep, alpha, zero_power=True):
    return mc2b_many([mcep], alpha, zero_power)[0]
