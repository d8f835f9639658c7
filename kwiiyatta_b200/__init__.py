"""kwiiyatta_b200: B200-native alignment + spectral-mapping hot path behind kwiiyatta's API.

Public surface mirrors the reference's (kwiiyatta/__init__.py:1-22) for this path: ``align`` (the
type-dispatching one, kwiiyatta/align.py:7-19), ``align_even``, the dataset chain
(``ParallelDataset`` ... ``align_dataset``), ``MelCepstrumConverter`` with the converter back-end
``B200GMMFeatureConverter``, a ``fastdtw`` module and ``MLPG``, plus global-variance
(GV) conversion: ``estimate_gv`` and the ``gv`` options of ``MLPG`` and the converter.  See INTEGRATION.md.
"""
import collections.abc

from . import alignment, fastdtw, hooks
from .alignment import (align_even, align_even_many, align_many, dtw_feature, dtw_feature_many,
                        make_feature, project_path, project_path_iter, set_pad_silence)
from .converter import (DeltaFeatureConverter, MapFeatureConverter, MelCepstrumConverter,
                        MelCepstrumFeatureConverter, load_converter, save_converter)
from .mlsa import mc2b, mc2b_many
from .dataset import (AlignedDataset, Dataset, DeltaFeatureDataset, MapDataset,
                      MelCepstrumDataset, ParallelDataset, TrimmedDataset, align_dataset,
                      joint_array_from_pairs, make_dataset_to_array, map_dataset)
from .delta import DELTA_WINDOWS, delta_features
from .gmm import B200GMMFeatureConverter, FeatureConverter, GaussianMixture
from .gv import GlobalVariance, estimate_gv
from .mlpg import MLPG

name = 'kwiiyatta_b200'


def _is_feature(obj):
    return hasattr(obj, 'f0') and hasattr(obj, 'mel_cepstrum') and hasattr(obj, 'frame_len')


def align(a, b, **kwargs):
    """``kwiiyatta.align`` (kwiiyatta/align.py:7-19): two features -> the first warped onto the
    second's time axis (kwiiyatta/vocoder/align.py:123-131); two datasets -> the aligned
    parallel dataset (trim -> align_even per key, batched)."""
    if _is_feature(a):
        if not _is_feature(b):
            raise TypeError(f'argument type mismatch: {type(a)!r}'
                            f' and {type(b)!r}')
        return alignment.align(a, b, **kwargs)
    if isinstance(a, collections.abc.Mapping):
        if not isinstance(b, collections.abc.Mapping):
            raise TypeError(f'argument type mismatch: {type(a)!r}'
                            f' and {type(b)!r}')
        return align_dataset(ParallelDataset(a, b))
    raise TypeError('argument should be Feature or Dataset')


__all__ = ['fastdtw', 'hooks', 'align', 'align_even', 'align_even_many', 'align_many',
           'dtw_feature', 'dtw_feature_many', 'make_feature', 'project_path',
           'project_path_iter', 'set_pad_silence',
           'Dataset', 'MapDataset', 'map_dataset', 'ParallelDataset', 'TrimmedDataset',
           'AlignedDataset', 'MelCepstrumDataset', 'DeltaFeatureDataset', 'align_dataset',
           'make_dataset_to_array', 'joint_array_from_pairs',
           'MelCepstrumConverter', 'MelCepstrumFeatureConverter', 'DeltaFeatureConverter',
           'MapFeatureConverter', 'B200GMMFeatureConverter', 'FeatureConverter',
           'save_converter', 'load_converter', 'mc2b', 'mc2b_many',
           'GaussianMixture', 'MLPG', 'DELTA_WINDOWS', 'delta_features',
           'GlobalVariance', 'estimate_gv']
