"""oracle/mlpg_em_ref.py (EM trajectory estimation) checked against its own definition."""
import numpy as np
import pytest
from scipy.stats import multivariate_normal, norm

from kwiiyatta_b200 import synth
from oracle import delta_ref, gmm_ref, mlpg_em_ref as em, mlpg_ref

DH, SD = 12, 4


def _model(k=4, seed=3):
    return synth.make_joint_gmm(k, dim_half=DH, seed=seed, static_dim=SD)


def _src(t, seed=0):
    rng = np.random.default_rng(seed)
    s = np.cumsum(rng.normal(0, 0.3, (t, SD)), axis=0) / (1.0 + np.arange(SD))
    return delta_ref.delta_features(s)


def _gradient(src, y, cond, joint):
    """Analytic gradient of L: W^T (q - P W y), without the posterior floor."""
    gamma, _ = em.e_step(src, y, cond, joint)
    prec, q = em.precision_terms(src, gamma, cond, floor=0.0)
    r = q - prec * em.window_apply(y)
    g = np.zeros_like(y)
    for wi, w in enumerate(delta_ref.DELTA_WINDOWS):
        g += mlpg_ref.window_matrix(w, len(y)).T @ r[:, wi * SD:(wi + 1) * SD]
    return g


def test_joint_density_factorises():
    w, m, c = _model()
    cond = em.conditional(w, m, c)
    joint = em.joint_model(cond)
    rng = np.random.default_rng(1)
    z = rng.normal(0, 0.5, (20, 2 * DH))
    got = gmm_ref.weighted_log_prob(z, w, *joint)
    x, yy = z[:, :DH], z[:, DH:]
    for k in range(len(w)):
        e = cond['offset'][k] + x @ cond['a'][k].T
        want = (np.log(w[k]) + multivariate_normal(cond['src_means'][k], cond['cxx'][k]).logpdf(x)
                + norm.logpdf(yy, e, np.sqrt(cond['var'][k])).sum(axis=1))
        assert np.abs(got[:, k] - want).max() <= 1e-10 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize('diff', [False, True])
def test_gradient_matches_central_differences(diff):
    w, m, c = _model()
    src = _src(12)
    cond = em.conditional(w, m, c, diff)
    joint = em.joint_model(cond)
    y = mlpg_ref.transform(src, w, m, c, diff=diff) + 0.05
    g = _gradient(src, y, cond, joint)
    h = 1e-5
    for t, d in [(0, 0), (5, 2), (11, 3), (6, 1)]:
        yp, ym = y.copy(), y.copy()
        yp[t, d] += h
        ym[t, d] -= h
        fd = (em.objective(src, yp, cond, joint) - em.objective(src, ym, cond, joint)) / (2 * h)
        assert abs(fd - g[t, d]) <= 1e-5 * max(1.0, abs(g[t, d])), (t, d, fd, g[t, d])


@pytest.mark.parametrize('diff', [False, True])
@pytest.mark.parametrize('t', [1, 2, 3, 40, 150])
def test_objective_non_decreasing(diff, t):
    w, m, c = _model()
    _, trace = em.convert(_src(t, seed=t), w, m, c, diff=diff, em_iter=10)
    assert len(trace) == 11
    steps = np.diff(trace)
    assert np.all(steps >= -1e-9 * np.abs(trace).max()), steps


def test_single_mixture_keeps_hard_solution():
    w, m, c = _model(k=1)
    src = _src(40)
    y0 = mlpg_ref.transform(src, w, m, c)
    y1, _ = em.convert(src, w, m, c, em_iter=1)
    assert np.abs(y1 - y0).max() <= 1e-12 * max(1.0, np.abs(y0).max())


def test_m_step_is_weighted_least_squares():
    """The M-step trajectory minimises sum_t sum_m g (W y - E)^T D^-1 (W y - E), solved here as
    one dense least-squares problem per static dimension."""
    w, m, c = _model()
    src = _src(40)
    cond = em.conditional(w, m, c)
    joint = em.joint_model(cond)
    y0 = mlpg_ref.transform(src, w, m, c)
    gamma, _ = em.e_step(src, y0, cond, joint)
    got = em.m_step(src, gamma, cond, floor=0.0)
    e = em.cond_means(src, cond)
    mats = [mlpg_ref.window_matrix(win, len(src)) for win in delta_ref.DELTA_WINDOWS]
    for d in range(SD):
        rows, rhs = [], []
        for k in range(len(w)):
            for wi, mat in enumerate(mats):
                col = wi * SD + d
                s = np.sqrt(gamma[:, k] / cond['var'][k, col])
                rows.append(s[:, None] * mat)
                rhs.append(s * e[k, :, col])
        want = np.linalg.lstsq(np.concatenate(rows), np.concatenate(rhs), rcond=None)[0]
        assert np.abs(got[:, d] - want).max() <= 1e-10 * max(1.0, np.abs(want).max())


def test_floor_is_negligible():
    w, m, c = _model()
    src = _src(150)
    cond = em.conditional(w, m, c)
    joint = em.joint_model(cond)
    gamma, _ = em.e_step(src, mlpg_ref.transform(src, w, m, c), cond, joint)
    assert np.any((gamma > 0) & (gamma <= em.FLOOR))        # the floor drops some terms here
    a = em.m_step(src, gamma, cond)
    b = em.m_step(src, gamma, cond, floor=0.0)
    assert np.abs(a - b).max() < 1e-10
