"""oracle/mlpg_full_ref.py against its own definition (CPU)."""
import numpy as np
import pytest

from kwiiyatta_b200 import synth
from oracle import delta_ref, mlpg_full_ref, mlpg_ref


def _utterance(frames, seed=0, order=24):
    return delta_ref.delta_features(
        synth.make_source_utterances(1, frames=frames, seed0=seed, order=order)[0])


def _small_model(seed=3):
    """4 mixtures, dim_half 12 (static_dim 4): small enough for dense checks."""
    return synth.make_joint_gmm(4, dim_half=12, seed=seed, static_dim=4)


def _diagonal_blocks(c):
    """Keep only the diagonals of the S_xx, S_xy, S_yx and S_yy blocks."""
    dh = c.shape[1] // 2
    out = np.zeros_like(c)
    idx = np.arange(dh)
    for r0 in (0, dh):
        for c0 in (0, dh):
            out[:, r0 + idx, c0 + idx] = c[:, r0 + idx, c0 + idx]
    return out


@pytest.mark.parametrize('diff', [False, True])
@pytest.mark.parametrize('frames', [1, 2, 3, 40])
def test_banded_equals_dense(diff, frames):
    w, m, c = _small_model()
    src = _utterance(frames, order=4)
    y_band = mlpg_full_ref.transform(src, w, m, c, diff=diff, banded=True)
    y_dense = mlpg_full_ref.transform(src, w, m, c, diff=diff, banded=False)
    assert y_band.shape == (frames, 4)
    assert np.abs(y_band - y_dense).max() <= 1e-10 * max(np.abs(y_dense).max(), 1.0)


@pytest.mark.parametrize('diff', [False, True])
def test_diagonal_blocks_reduce_to_the_diagonal_path(diff):
    w, m, c = synth.make_joint_gmm(4, seed=5)
    c = _diagonal_blocks(c)
    cond = mlpg_full_ref.conditional_full(w, m, c, diff)
    split = mlpg_ref.split_joint(w, m, c, diff)
    dv = (np.diagonal(split['cyy'], axis1=1, axis2=2)
          - np.diagonal(split['cyx'], axis1=1, axis2=2) / np.diagonal(split['cxx'], axis1=1, axis2=2)
          * np.diagonal(split['cxy'], axis1=1, axis2=2))
    assert np.abs(cond['sigma'] - np.stack([np.diag(d) for d in dv])).max() <= 1e-15
    for frames in (1, 2, 3, 120):
        src = _utterance(frames, seed=synth.SEED0 + frames)
        got = mlpg_full_ref.transform(src, w, m, c, diff=diff, cond=cond)
        exp = mlpg_ref.transform(src, w, m, c, diff=diff)
        assert np.abs(got - exp).max() <= 1e-10, frames


@pytest.mark.parametrize('diff', [False, True])
def test_gradient_vanishes_and_matches_central_differences(diff):
    w, m, c = _small_model(seed=7)
    src = _utterance(12, order=4, seed=11)
    y, _, e, prec = mlpg_full_ref.transform(src, w, m, c, diff=diff, return_internals=True)
    g = mlpg_full_ref.gradient(y, e, prec)
    assert np.abs(g).max() <= 1e-9 * max(np.abs(mlpg_full_ref.gradient(0 * y, e, prec)).max(), 1)
    rng = np.random.default_rng(0)
    y1 = y + rng.standard_normal(y.shape)                 # away from the optimum
    g1 = mlpg_full_ref.gradient(y1, e, prec)
    h = 1e-5
    num = np.empty_like(y1)
    for idx in np.ndindex(*y1.shape):
        yp, ym = y1.copy(), y1.copy()
        yp[idx] += h
        ym[idx] -= h
        num[idx] = (mlpg_full_ref.objective(yp, e, prec) - mlpg_full_ref.objective(ym, e, prec)) / (2 * h)
    assert np.abs(num - g1).max() <= 1e-6 * np.abs(g1).max()


@pytest.mark.parametrize('diff', [False, True])
def test_full_solution_is_at_least_as_likely_as_the_diagonal_one(diff):
    w, m, c = synth.make_joint_gmm(8, seed=1)
    for frames in (1, 3, 150):
        src = _utterance(frames, seed=synth.SEED0 + 2 * frames)
        y, _, e, prec = mlpg_full_ref.transform(src, w, m, c, diff=diff, return_internals=True)
        y_diag = mlpg_ref.transform(src, w, m, c, diff=diff)
        f_full = mlpg_full_ref.objective(y, e, prec)
        f_diag = mlpg_full_ref.objective(y_diag, e, prec)
        assert f_full >= f_diag - 1e-9 * abs(f_diag), (frames, f_full, f_diag)


def test_diff_sigma_is_the_schur_complement_of_the_transformed_joint():
    w, m, c = synth.make_joint_gmm(3, seed=4)
    dh = m.shape[1] // 2
    t = np.block([[np.eye(dh), np.zeros((dh, dh))], [-np.eye(dh), np.eye(dh)]])   # [x ; y - x]
    cond = mlpg_full_ref.conditional_full(w, m, c, diff=True)
    for k in range(len(w)):
        cz = t @ c[k] @ t.T
        sxx, sxy, syx, syy = cz[:dh, :dh], cz[:dh, dh:], cz[dh:, :dh], cz[dh:, dh:]
        schur = syy - syx @ np.linalg.solve(sxx, sxy)
        assert np.abs(cond['sigma'][k] - schur).max() <= 1e-12 * np.abs(schur).max()


@pytest.mark.parametrize('frames', [1, 2, 3])
def test_short_utterances(frames):
    w, m, c = synth.make_joint_gmm(4, seed=2)
    src = _utterance(frames, seed=synth.SEED0 + 9)
    y = mlpg_full_ref.transform(src, w, m, c)
    assert y.shape == (frames, 24) and np.all(np.isfinite(y))
    y_dense = mlpg_full_ref.transform(src, w, m, c, banded=False)
    assert np.abs(y - y_dense).max() <= 1e-10 * max(np.abs(y_dense).max(), 1.0)
