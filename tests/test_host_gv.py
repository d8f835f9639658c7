"""Host-side plumbing of GV conversion (CPU only)."""
import numpy as np
import pytest

import kwiiyatta_b200 as kw
from kwiiyatta_b200 import synth
from kwiiyatta_b200.dataset import _dataset_to_array_with_offsets
from kwiiyatta_b200.gv import GlobalVariance, as_gv


def test_gv_keywords_reach_the_backend():
    """MelCepstrumConverter(..., gv=True) hands gv to the back-end's constructor and
    convert(..., gv=True) to its convert, through the layers' keyword pass-through."""
    class Recorder(kw.FeatureConverter):
        def __init__(self, gv=False):
            self.gv_flag = gv
            self.seen = []

        def _train(self, dataarray, **kwargs):
            pass

        def convert(self, feature, **kwargs):
            self.seen.append(kwargs)
            return feature

    conv = kw.MelCepstrumConverter(use_delta=False, Converter=Recorder, gv=True)
    assert conv.base.gv_flag is True
    conv.order, conv.fs = synth.ORDER, synth.FS
    mcep = synth.make_pair(0)[0].mel_cepstrum
    out = conv.convert(mcep, diff=True, gv=True)
    assert conv.base.seen[-1] == {'diff': True, 'gv': True}
    assert np.array_equal(out.data, mcep.data)


def test_global_variance_forms():
    mean, var = np.arange(3.0), np.full(3, 0.5)
    for form in (GlobalVariance(mean, var), {'mean': mean, 'var': var}, (mean, var)):
        gv = as_gv(form)
        assert np.array_equal(gv.mean, mean) and np.array_equal(gv.var, var) and len(gv) == 3
    for bad in ((mean, var[:2]), (mean, np.zeros(3)), (-mean - 1, var)):
        with pytest.raises(ValueError):
            as_gv(bad)


def test_dataset_array_offsets_host_path():
    rng = np.random.default_rng(0)
    a = rng.normal(0, 1, (6, 4))
    a[2] = 0.0                                   # a zero frame, dropped
    b = rng.normal(0, 1, (3, 4))
    data = {'k1': (a, 2 * a), 'k2': (b, b), 'k3': (np.zeros((2, 4)), np.zeros((2, 4)))}
    keys = ['k2', 'k1', 'k3']
    x, off = _dataset_to_array_with_offsets(data, keys)
    assert np.array_equal(x, kw.make_dataset_to_array(data, keys))
    assert off.tolist() == [0, 3, 8, 8]
    assert np.array_equal(x[3:8], np.delete(np.hstack((a, 2 * a)), 2, axis=0))
    assert _dataset_to_array_with_offsets({}, [])[0] is None
