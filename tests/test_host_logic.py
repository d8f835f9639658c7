"""CPU: host-side mirrors of the reference's Python (no kernels involved)."""
import re
import os

import numpy as np
import pytest

import kwiiyatta_b200 as kw
from kwiiyatta_b200 import _lib, synth
from kwiiyatta_b200.alignment import _strict_filter, _trim_even, make_feature, project_path_iter
from kwiiyatta_b200.dataset import make_dataset_to_array, remove_zeros_frames
from oracle import align_ref, delta_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, 'include', 'kwiiyatta_b200.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    declared = set(re.findall(r'\b(kw_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations found'
    lib = _lib.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), f'{name} declared in the header but not exported'
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.kw_abi_version() == 3
    assert lib.kw_gmm_stats_len(64, 144) == 64 * (1 + 144 + 144 * 144) + 2


def test_no_fallback_without_cuda(monkeypatch):
    import torch
    # on a machine with a GPU, the host API must see none
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: False)
    with pytest.raises(_lib.KwError, match='no CPU fallback'):
        kw.fastdtw.fastdtw(np.zeros((4, 2)), np.zeros((5, 2)), dist=2)
    with pytest.raises(_lib.KwError, match='no CPU fallback'):
        kw.GaussianMixture(n_components=2).fit(np.zeros((10, 2)))


def test_make_feature_matches_reference_restatement():
    a, _ = synth.make_padded_pair(1)
    for kwargs in ({}, {'vuv': 'f0'}, {'power': 'raw', 'vuv': None},
                   {'power_pivot': 'median'}, {'power_pivot': 'min'}, {'power_pivot': 'fix'},
                   {'power': None}):
        got = make_feature(a, a.fs, **kwargs)
        exp = align_ref.make_feature(a.mel_cepstrum.data, a.f0, a.is_voiced, **kwargs)
        assert got.shape == (a.frame_len, 26) and np.array_equal(got, exp)
    assert set(np.unique(make_feature(a, a.fs)[:, 0])) <= {0.0, 9.4}
    assert set(np.unique(make_feature(a, a.fs)[:, 1])) <= {0.0, 9.0}
    with pytest.raises(ValueError, match='Unknown power parameter'):
        make_feature(a, a.fs, power='x')
    with pytest.raises(ValueError, match='Unknown vuv parameter'):
        make_feature(a, a.fs, vuv='x')
    with pytest.raises(ValueError, match='Unknown power_pivot parameter'):
        make_feature(a, a.fs, power_pivot='x')


def test_strict_filter_including_quirk():
    rng = np.random.default_rng(0)
    xf = np.zeros((30, 4))
    yf = np.zeros((30, 4))
    xf[:, 0] = rng.integers(0, 2, 30) * 9.4
    xf[:, 1] = rng.integers(0, 2, 30) * 9.0
    yf[:, 0] = rng.integers(0, 2, 30) * 9.4
    yf[:, 1] = rng.integers(0, 2, 30) * 9.0
    path = np.stack([np.arange(30), np.arange(30)], axis=1)
    for vuv, power in (('voiced', 'binalize'), (None, 'binalize'), ('f0', 'raw'), (None, None)):
        got = _strict_filter(path, xf, yf, vuv, power)
        exp = align_ref.strict_filter(path, xf, yf, vuv=vuv, power=power)
        assert np.array_equal(got, exp)
    # the quirk: x's V/UV flag is compared with y's POWER flag (align.py:78)
    xf[:] = 0
    yf[:] = 0
    xf[5, 1] = 9.0
    yf[5, 1] = 9.0        # both voiced, y power flag 0 -> dropped by the reference
    got = _strict_filter(path, xf, yf, 'voiced', None)
    assert 5 not in got[:, 0]
    assert np.array_equal(_strict_filter(path[:1], xf, yf, 'voiced', 'binalize'),
                          np.array([[0, 0], [0, 0]]))


def test_project_path_iter_matches_reference_restatement():
    rng = np.random.default_rng(1)
    for _ in range(20):
        steps = rng.integers(0, 3, 120)
        i = j = 0
        path = [(0, 0)]
        for s in steps:
            i, j = (i + 1, j) if s == 0 else ((i, j + 1) if s == 1 else (i + 1, j + 1))
            path.append((i, j))
        for trim, tl in ((True, 3), (False, 1), (True, 10)):
            assert list(project_path_iter(path, trim, tl)) == \
                list(align_ref.project_path_iter(path, trim, tl))
        idx = list(project_path_iter(path, trim=False))
        assert len(idx) == path[-1][1] + 1       # one source index per target frame


def test_trim_even_path():
    path = np.stack([np.arange(50), np.arange(50)], axis=1)
    got = _trim_even(path, 50, 50, 10)
    assert np.array_equal(got, align_ref.trim_even_path(path, 50, 50, 10))
    assert got[0, 0] == 10 and got[0, -1] == 39
    # never reaching the un-padded region: np.argmax of all-False is 0 -> empty result
    assert _trim_even(path[:5], 50, 50, 10).shape[1] == 0


def test_make_dataset_to_array_semantics():
    rng = np.random.default_rng(2)
    a = rng.standard_normal((5, 3))
    b = rng.standard_normal((4, 3))
    b[2] = 0
    ds = {'k2': b, 'k1': (a, a + 1)}
    out = make_dataset_to_array({'k1': (a, a + 1)}, ['k1'])
    assert np.array_equal(out, np.hstack((a, a + 1)))
    out = make_dataset_to_array({'k2': b})
    assert np.array_equal(out, delta_ref.remove_zeros_frames(b)) and len(out) == 3
    assert np.array_equal(remove_zeros_frames(b), delta_ref.remove_zeros_frames(b))
    assert make_dataset_to_array({}, []) is None
    assert ds  # silence linters


def test_converter_plugin_surface():
    conv = kw.B200GMMFeatureConverter(components=4, random_state=0)
    assert isinstance(conv, kw.FeatureConverter)
    assert conv.gmm.n_components == 4 and conv.gmm.max_iter == 100
    assert conv.gmm.verbose == 1 and conv.gmm.covariance_type == 'full'
    assert conv.gmm.tol == 1e-3 and conv.gmm.reg_covar == 1e-6
    with pytest.raises(NotImplementedError):
        kw.GaussianMixture(covariance_type='diag')


def test_synthetic_corpus_is_seeded_and_tie_free():
    a1, b1 = synth.make_pair(7)
    a2, b2 = synth.make_pair(7)
    assert np.array_equal(a1.mel_cepstrum.data, a2.mel_cepstrum.data)
    assert np.array_equal(b1.mel_cepstrum.data, b2.mel_cepstrum.data)
    assert 450 <= a1.frame_len <= 750 and a1.mel_cepstrum.data.shape[1] == 25
    assert 0.79 * a1.frame_len <= b1.frame_len <= 1.26 * a1.frame_len
    p, q = synth.make_padded_pair(7)
    assert p.frame_len == a1.frame_len + 200 and not p.is_voiced[:100].any()
    f = make_feature(p, p.fs)
    assert (f[:100, 0] == 0).all() and (f[-100:, 1] == 0).all()
