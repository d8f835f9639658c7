"""The dataset chain of the reference, batched (kwiiyatta/converter/abc/dataset.py:5-82,
kwiiyatta/converter/dataset.py:35-77, converter/mcep.py:10-33, converter/delta.py:15-30).

The reference's datasets are lazy mappings evaluated one key at a time: every ``dataset[key]``
re-runs the chain below it, so training walks  pair -> trim -> DTW -> mcep -> delta  once per
utterance, in Python.  Here every link also answers ``get_many(keys)``: the keys travel down
the chain TOGETHER, the alignment link runs one batched FastDTW for all of them and the delta
link one kernel launch over all utterances.  ``dataset[key]`` stays available and is the batch of
one.  Class names, constructor arguments, the ``function`` / ``with_key`` / ``with_raw`` /
``expand_tuple`` protocol and the error texts are the reference's, so its own subclasses
(``map_dataset`` decorated functions included) keep working on top of these.
"""
import collections.abc

import numpy as np

from . import _lib
from . import alignment as _align
from . import hooks
from .delta import delta_features_device

ZERO_FRAME_EPS = 1e-7      # nnmnkwii.preprocessing's threshold on a frame's absolute sum


def remove_zeros_frames(x, eps=ZERO_FRAME_EPS):
    """Rows whose absolute sum exceeds ``eps`` (nnmnkwii.preprocessing.remove_zeros_frames as
    called at kwiiyatta/converter/dataset.py:70)."""
    return x[np.abs(x).sum(axis=1) > eps]


def trim_zeros_frames(x, eps=ZERO_FRAME_EPS):
    """``x`` without its trailing run of rows whose absolute sum is below ``eps``
    (nnmnkwii.preprocessing.trim_zeros_frames, trim='b', as called at
    kwiiyatta/converter/dataset.py:51)."""
    loud = np.flatnonzero(np.abs(x).sum(axis=1) >= eps)
    return x[:loud[-1] + 1] if len(loud) else x[:0]


class Dataset(collections.abc.Mapping):
    """A keyed collection of utterances (kwiiyatta/converter/abc/dataset.py:5-21)."""

    def keys(self):
        raise NotImplementedError

    def get_data(self, key):
        raise NotImplementedError

    def get_many(self, keys):
        return [self.get_data(key) for key in keys]

    def __getitem__(self, key):
        return self.get_data(key)

    def __iter__(self):
        return ((key, self[key]) for key in self.keys())

    def __len__(self):
        return len(self.keys())


def _fetch(base, keys):
    """Items of ``base`` for ``keys`` plus the matching items of the bottom (non-mapped) dataset,
    which the reference hands to ``with_raw`` functions."""
    if isinstance(base, MapDataset):
        return base._evaluate(keys)
    if hasattr(base, 'get_many'):
        items = base.get_many(keys)
    else:
        items = [base[key] for key in keys]
    return items, items


class MapDataset(Dataset):
    """``function`` applied to every item of ``base`` (kwiiyatta/converter/abc/dataset.py:24-69).
    Subclasses either define ``function(item, **kwargs)`` like the reference's, or override
    ``map_many`` to process all items of a request at once."""
    expand_tuple = True
    with_key = False
    with_raw = False

    def __init__(self, base_dataset, **kwargs):
        super().__init__()
        self.base = base_dataset
        self.kwargs = kwargs

    def keys(self):
        return self.base.keys()

    def __getattr__(self, name):
        return getattr(self.base, name)

    @staticmethod
    def function(data):
        raise NotImplementedError

    def map_many(self, items, raws, keys):
        """Default: the reference's per-item call protocol."""
        out = []
        for item, raw, key in zip(items, raws, keys):
            args = dict(self.kwargs)
            if self.with_key:
                args['key'] = key
            if self.expand_tuple and isinstance(item, tuple):
                if self.with_raw:
                    out.append(tuple(self.function(d, raw=r, **args) for d, r in zip(item, raw)))
                else:
                    out.append(tuple(self.function(d, **args) for d in item))
            else:
                if self.with_raw:
                    args['raw'] = raw
                out.append(self.function(item, **args))
        return out

    def _evaluate(self, keys):
        keys = list(keys)
        items, raws = _fetch(self.base, keys)
        return self.map_many(items, raws, keys), raws

    def get_many(self, keys):
        return self._evaluate(keys)[0]

    def get_data(self, key, with_raw=False):
        items, raws = self._evaluate([key])
        return (items[0], raws[0]) if with_raw else items[0]


def map_dataset(expand_tuple=True, with_key=False, with_raw=False):
    """Class decorator of the reference (kwiiyatta/converter/abc/dataset.py:72-82)."""
    def build(func):
        return type(func.__name__, (MapDataset,), {
            '__module__': func.__module__, '__doc__': func.__doc__,
            'function': staticmethod(func), 'expand_tuple': expand_tuple,
            'with_key': with_key, 'with_raw': with_raw})
    return build


class ParallelDataset(Dataset):
    """(source, target) per key present in both (kwiiyatta/converter/dataset.py:35-46)."""

    def __init__(self, dataset1, dataset2):
        super().__init__()
        self.dataset1 = dataset1
        self.dataset2 = dataset2
        self.common_keys = self.dataset1.keys() & self.dataset2.keys()

    def keys(self):
        return self.common_keys

    def get_data(self, key):
        return self.dataset1[key], self.dataset2[key]


class TrimmedDataset(MapDataset):
    """Each feature cut after its last frame with spectral energy
    (kwiiyatta/converter/dataset.py:49-52)."""

    @staticmethod
    def function(feature):
        return feature[:len(trim_zeros_frames(feature.spectrum_envelope))]


class AlignedDataset(MapDataset):
    """``align_even`` of every (a, b) pair; constructor keywords go to it
    (kwiiyatta/converter/dataset.py:55-58).  All pairs of a request share one batched FastDTW."""
    expand_tuple = False

    @staticmethod
    def function(features, **kwargs):
        a, b = features
        return _align.align_even(a, b, **kwargs)

    def map_many(self, items, raws, keys):
        return _align.align_even_many(items, **self.kwargs)


def align_dataset(parallel_dataset):
    """kwiiyatta/converter/__init__.py:17-18."""
    return AlignedDataset(TrimmedDataset(parallel_dataset))


class MelCepstrumDataset(MapDataset):
    """Mel-cepstra without c0, brought to one order and sampling rate -- those of the first
    utterance seen unless given (kwiiyatta/converter/mcep.py:10-33)."""
    with_key = True

    def __init__(self, base, mcep_fs=None):
        super().__init__(base)
        self.fs = mcep_fs
        self.order = None

    def function(self, feature, key):
        f = hooks.get('feature')(feature)
        if self.order is None:
            self.order = f.mel_cepstrum_order
        elif self.order != feature.mel_cepstrum_order:
            f.mel_cepstrum_order = self.order
        data = f.mel_cepstrum.data
        if self.fs is None:
            self.fs = f.fs
        elif self.fs != f.fs:
            data = f.resample_mel_cepstrum(self.fs).data
        return data[:, 1:]


class DeltaFeatureDataset(MapDataset):
    """static -> [static, delta, delta-delta] (kwiiyatta/converter/delta.py:15-30); all
    utterances of a request go through ONE kw_delta_features launch."""
    with_key = True
    with_raw = True

    def __init__(self, base):
        super().__init__(base)
        self.frame_period = None

    def _check_period(self, raw, key):
        if self.frame_period is None:
            self.frame_period = raw.frame_period
        elif self.frame_period != raw.frame_period:
            raise ValueError(f'frame_period of "{key}" is {raw.frame_period!r}'
                             f' but others are {self.frame_period!r}')

    def function(self, feature, raw, key):
        self._check_period(raw, key)
        return delta_many([feature])[0]

    def map_many(self, items, raws, keys):
        flat = []
        for item, raw, key in zip(items, raws, keys):
            members = zip(item, raw) if isinstance(item, tuple) else ((item, raw),)
            for feature, r in members:
                self._check_period(r, key)
                flat.append(feature)
        deltas = iter(delta_many(flat))
        return [tuple(next(deltas) for _ in item) if isinstance(item, tuple) else next(deltas)
                for item in items]


def delta_many(features):
    """``delta_features(f, DELTA_WINDOWS)`` of every (T_i, dim) array in one launch."""
    torch = _lib.require_cuda()
    features = [np.ascontiguousarray(f, dtype=np.float64) for f in features]
    lens = np.array([len(f) for f in features], dtype=np.int64)
    if len(features) == 0 or lens.sum() == 0:
        return [np.zeros((len(f), 3 * f.shape[1])) for f in features]
    off = np.concatenate(([0], np.cumsum(lens)))
    x = torch.from_numpy(np.concatenate(features)).cuda()
    out = delta_features_device(x, torch.from_numpy(off).cuda(), len(features)).cpu().numpy()
    return [out[off[i]:off[i + 1]] for i in range(len(features))]


def _device_chain(dataset):
    """(delta or None, mcep, aligned) when ``dataset`` is the standard training chain
    [DeltaFeatureDataset(] MelCepstrumDataset(AlignedDataset(...)) [)], else None."""
    delta = dataset if type(dataset) is DeltaFeatureDataset else None
    mcep = dataset.base if delta is not None else dataset
    if type(mcep) is not MelCepstrumDataset or type(mcep.base) is not AlignedDataset:
        return None
    return delta, mcep, mcep.base


def _assemble_on_device(chain, keys):
    """The standard chain evaluated by kwiiyatta_b200.assemble on the device; None when the
    request needs a per-item code path (mixed orders / sampling rates / frame periods, which the
    host path resolves or reports exactly as the reference does)."""
    from . import assemble
    delta, mcep, aligned = chain
    pairs, raws = _fetch(aligned.base, keys)
    if not pairs or any(not isinstance(p, tuple) or len(p) != 2 for p in pairs):
        return None
    feats = [f for pair in pairs for f in pair]
    order = mcep.order if mcep.order is not None else feats[0].mel_cepstrum_order
    fs = mcep.fs if mcep.fs is not None else feats[0].fs
    if any(f.mel_cepstrum_order != order or f.fs != fs for f in feats):
        return None
    periods = {r.frame_period for raw in raws for r in raw}
    if delta is not None:
        if len(periods) != 1 or delta.frame_period not in (None, next(iter(periods))):
            return None
    known = ('pad_silence', 'pad_len', 'vuv', 'power', 'strict', 'radius', 'vuv_weight',
             'power_weight', 'power_pivot', 'power_threshold')
    if any(k not in known for k in aligned.kwargs):
        return None
    x, offsets = assemble.joint_frames_device(pairs, use_delta=delta is not None,
                                              return_offsets=True, **aligned.kwargs)
    mcep.order, mcep.fs = order, fs               # what the per-item path would have recorded
    if delta is not None:
        delta.frame_period = next(iter(periods))
    return x, offsets


def _dataset_to_array_with_offsets(dataset, keys=None, device_resident=False):
    """``make_dataset_to_array`` plus the int64 row offsets (n_keys + 1) of each key's rows in
    it: a numpy array with the host matrix, a CUDA tensor with the device-assembled one."""
    if keys is None:
        keys = sorted(dataset.keys())
    keys = list(keys)
    if device_resident and keys:
        chain = _device_chain(dataset)
        if chain is not None:
            res = _assemble_on_device(chain, keys)
            if res is not None:
                return res
    if hasattr(dataset, 'get_many'):
        items = dataset.get_many(keys)
    else:
        items = [dataset[key] for key in keys]
    rows = [remove_zeros_frames(np.hstack(d) if isinstance(d, tuple) else d) for d in items]
    offsets = np.concatenate(([0], np.cumsum([len(r) for r in rows]))).astype(np.int64)
    return (np.concatenate(rows) if rows else None), offsets


def make_dataset_to_array(dataset, keys=None, device_resident=False):
    """(N, dim) training matrix: per key the horizontally stacked tuple without its zero frames,
    keys in the given (default: sorted) order (kwiiyatta/converter/dataset.py:61-77).  The whole
    key list goes down the chain in one request.  ``device_resident``: for the standard training
    chain return the matrix as a CUDA tensor assembled on the device
    (kwiiyatta_b200.assemble), bit-identical to the host result."""
    return _dataset_to_array_with_offsets(dataset, keys, device_resident)[0]


def joint_array_from_pairs(pairs, use_delta=True, pad_silence=True, pad_len=100,
                           device_resident=False, **align_kwargs):
    """The training-array pipeline for a list of (source, target) features without the dataset
    objects: align_even (batched DTW) -> mcep without c0 (kwiiyatta/converter/mcep.py:33) ->
    delta features (kwiiyatta/converter/delta.py:30) -> hstack -> remove zero frames.
    ``device_resident``: the same array as a CUDA tensor, assembled on the device."""
    if device_resident:
        from . import assemble
        return assemble.joint_frames_device(pairs, use_delta=use_delta, pad_silence=pad_silence,
                                            pad_len=pad_len, **align_kwargs)
    aligned = _align.align_even_many(pairs, pad_silence=pad_silence, pad_len=pad_len,
                                     **align_kwargs)
    sides = [a.mel_cepstrum.data[:, 1:] for a, _ in aligned] + \
            [b.mel_cepstrum.data[:, 1:] for _, b in aligned]
    if sum(len(s) for s in sides) == 0:
        return np.zeros((0, 0))
    if use_delta:
        sides = delta_many(sides)
    n = len(aligned)
    return np.concatenate([remove_zeros_frames(np.hstack((sides[i], sides[n + i])))
                           for i in range(n)])
