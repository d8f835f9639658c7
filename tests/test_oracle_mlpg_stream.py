"""oracle/mlpg_stream_ref.py against its definition (CPU): the prefix system, the recursion the
device runs, the offline limit and the accuracy against the delay."""
import numpy as np
import pytest

from kwiiyatta_b200 import synth
from oracle import mlpg_ref, mlpg_stream_ref as ref

W, M, C = synth.make_joint_gmm(32, seed=3)


def _internals(t):
    statics = synth.make_source_utterances(1, frames=max(t, 1), order=24)[0][:t]
    return ref.internals(statics, W, M, C)


@pytest.fixture(scope='module')
def long_utt():
    return _internals(700)


def test_band_is_mlpg_refs_system(long_utt):
    _, _, e, dv = long_utt
    assert np.abs(ref.solve(*ref.band(e[:60], dv[:60])) -
                  mlpg_ref.mlpg_banded(e[:60], dv[:60])).max() <= 1e-12


@pytest.mark.parametrize('n', [1, 2, 3, 57, 699])
def test_prefix_system(long_utt, n):
    """Rows below n-1 of the system of [0, n) are the whole utterance's; row n-1 lacks frame n's
    terms on its diagonal and right-hand side, and nothing else."""
    _, _, e, dv = long_utt
    ab, rhs = ref.band(e, dv)
    abn, rhsn = ref.band(e[:n], dv[:n])
    assert np.array_equal(abn[0, :n - 1], ab[0, :n - 1])
    assert np.array_equal(abn[1, :n - 1], ab[1, :n - 1])
    assert np.array_equal(abn[2, :max(n - 2, 0)], ab[2, :max(n - 2, 0)])
    assert np.array_equal(rhsn[:n - 1], rhs[:n - 1])
    assert not abn[1, n - 1:].any() and not abn[2, max(n - 2, 0):].any()
    # frame n's terms: window offset -1 puts c[w][0]^2 / D and c[w][0] E / D on row n-1
    sd = e.shape[1] // 3
    cm = ref._coeff()[:, 0]
    p = 1.0 / dv[n].reshape(3, sd)
    q = p * e[n].reshape(3, sd)
    scale = np.abs(ab[0, n - 1]).max() + np.abs(rhs[n - 1]).max()
    assert np.abs(ab[0, n - 1] - abn[0, n - 1] - (cm[:, None] ** 2 * p).sum(0)).max() <= 1e-13 * scale
    assert np.abs(rhs[n - 1] - rhsn[n - 1] - (cm[:, None] * q).sum(0)).max() <= 1e-13 * scale


@pytest.mark.parametrize('delay', [0, 1, 5, 40])
def test_recursion_equals_definition(long_utt, delay):
    _, _, e, dv = long_utt
    lengths = sorted({1, 2, 3, delay, delay + 1, delay + 2, 700} - {0})
    for t in lengths:
        got = ref.stream_recursive(e[:t], dv[:t], delay)
        exp = ref.stream_prefix(e[:t], dv[:t], delay)
        assert got.shape == (t, e.shape[1] // 3)
        assert np.abs(got - exp).max() <= 1e-12, (delay, t)


@pytest.mark.parametrize('t', [1, 2, 3, 41, 150])
def test_long_delay_is_offline(t):
    statics = synth.make_source_utterances(1, frames=150, order=24)[0][:t]
    exp = mlpg_ref.transform(ref.delta_features(statics), W, M, C)
    for delay in (t - 1, t + 5):
        for recursive in (False, True):
            got = ref.convert_stream(statics, W, M, C, delay, recursive=recursive)
            assert np.abs(got - exp).max() <= 1e-12


def test_empty_stream():
    assert ref.convert_stream(np.zeros((0, 24)), W, M, C, 3).shape == (0, 24)


def test_error_shrinks_with_delay():
    errs = []
    utts = [ref.internals(synth.make_pair(u)[0].mel_cepstrum.data[:, 1:], W, M, C)
            for u in range(2)]
    for delay in (5, 10, 20, 40):
        errs.append(max(np.abs(ref.stream_recursive(e, dv, delay) - y).max()
                        for y, _, e, dv in utts))
    assert all(a > b for a, b in zip(errs, errs[1:])), errs
    assert errs[-1] <= 1e-6
