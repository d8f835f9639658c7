"""The converter chain of the reference around the B200 back-end
(kwiiyatta/converter/abc/converter.py:4-34, converter/delta.py:33-50, converter/mcep.py:36-61,
converter/__init__.py:9-14).

``MelCepstrumConverter(...)`` here builds the same three-layer object the reference's factory
builds -- mel-cepstrum layer (drops c0, re-attaches the SOURCE c0 after conversion, checks order
and sampling rate) around the delta layer (static -> static + deltas before, first ``dim``
columns after, frame-period check) around the GMM back-end -- with
``B200GMMFeatureConverter`` as the default back-end.  Inside kwiiyatta the reference's own
wrappers can be kept and only ``Converter=B200GMMFeatureConverter`` passed (INTEGRATION.md);
these classes are for callers that replace the chain as a whole, and add ``convert_many``."""
import copy

import numpy as np

from . import dataset as _ds
from . import hooks
from .gmm import B200GMMFeatureConverter, FeatureConverter


class MapFeatureConverter(FeatureConverter):
    """A layer around ``base``; unknown attributes fall through to it
    (kwiiyatta/converter/abc/converter.py:18-34)."""

    def __init__(self, base_converter):
        self.base = base_converter

    def __getattr__(self, name):
        return getattr(self.base, name)

    def _train(self, dataarray, **kwargs):
        return self.base._train(dataarray, **kwargs)

    def convert(self, feature, raw=None, **kwargs):
        """Hands ``raw`` (the caller's original object) down through mapped layers only."""
        if raw is None:
            raw = feature
        if isinstance(self.base, MapFeatureConverter):
            return self.base.convert(feature, raw, **kwargs)
        return self.base.convert(feature, **kwargs)


class DeltaFeatureConverter(MapFeatureConverter):
    """kwiiyatta/converter/delta.py:33-50."""

    def train(self, dataset, keys, **kwargs):
        expanded = _ds.DeltaFeatureDataset(dataset)
        self.base.train(expanded, keys, **kwargs)
        self.frame_period = expanded.frame_period

    def convert(self, feature, raw, **kwargs):
        if self.frame_period != raw.frame_period:
            raise ValueError(f'frame_period is expected to {self.frame_period!s}'
                             f' but {raw.frame_period!s}')
        width = feature.shape[-1]
        out = super().convert(_ds.delta_many([feature])[0], **kwargs)
        return out[:, :width] if out.shape[-1] > width else out


class MelCepstrumFeatureConverter(MapFeatureConverter):
    """kwiiyatta/converter/mcep.py:36-61."""

    def __init__(self, base, mcep_fs=None):
        super().__init__(base)
        self.mcep_fs = mcep_fs

    def train(self, dataset, keys, **kwargs):
        cepstra = _ds.MelCepstrumDataset(dataset, mcep_fs=self.mcep_fs)
        self.base.train(cepstra, keys, **kwargs)
        self.order = cepstra.order
        self.fs = cepstra.fs

    def convert(self, mel_cepstrum, **kwargs):
        if self.order != mel_cepstrum.order:
            raise ValueError(f'order is expected to {self.order!s}'
                             f' but {mel_cepstrum.order!s}')
        if self.fs != mel_cepstrum.fs:
            result = hooks.get('resample')(mel_cepstrum, self.fs)
        else:
            result = copy.copy(mel_cepstrum)
        power = result.data[:, :1]
        shape = super().convert(result.data[:, 1:], raw=mel_cepstrum, **kwargs)
        result.data = np.hstack((power, shape))
        return result


def MelCepstrumConverter(use_delta=True, mcep_fs=None, Converter=B200GMMFeatureConverter,
                         **kwargs):
    """kwiiyatta/converter/__init__.py:9-14 with the B200 back-end as the default."""
    converter = Converter(**kwargs)
    if use_delta:
        converter = DeltaFeatureConverter(converter)
    return MelCepstrumFeatureConverter(converter, mcep_fs=mcep_fs)


def save_converter(converter, path):
    """Persist a trained ``MelCepstrumConverter(...)`` chain: the back-end's model plus what the
    layers learned while training (order, sampling rate, frame period)."""
    layers = {'use_delta': False}
    node = converter
    while isinstance(node, MapFeatureConverter):
        if isinstance(node, MelCepstrumFeatureConverter):
            layers.update(order=node.order, fs=node.fs,
                          mcep_fs=-1 if node.mcep_fs is None else node.mcep_fs)
        if isinstance(node, DeltaFeatureConverter):
            layers.update(use_delta=True, frame_period=node.frame_period)
        node = node.base
    np.savez(path, **node.state_dict(), **{'layer_' + k: v for k, v in layers.items()})


def load_converter(path, Converter=B200GMMFeatureConverter, **kwargs):
    with np.load(path) as data:
        state = {k: data[k] for k in data.files}
    layers = {k[6:]: state.pop(k) for k in list(state) if k.startswith('layer_')}
    kind = str(state.get('covariance_type', 'full'))
    if kind != 'full':
        kwargs.setdefault('covariance_type', kind)
    backend = Converter(components=int(state['n_components']), verbose=0, **kwargs)
    backend.load_state_dict(state)
    node = backend
    if bool(layers['use_delta']):
        node = DeltaFeatureConverter(node)
        node.frame_period = layers['frame_period'].item()
    mcep_fs = int(layers['mcep_fs'])
    node = MelCepstrumFeatureConverter(node, mcep_fs=None if mcep_fs < 0 else mcep_fs)
    node.order, node.fs = int(layers['order']), int(layers['fs'])
    return node
