"""The global-variance oracle against its own definition (CPU only)."""
import numpy as np
import pytest
import scipy.linalg

from oracle import gv_ref, mlpg_ref


def _system(t, seed=0, sd=3):
    """Normal equations of a random MLPG problem: sd static dims, T frames."""
    rng = np.random.default_rng(seed)
    e = rng.normal(0, 1, (t, 3 * sd)) * np.repeat([1.0, 0.3, 0.1], sd)
    dv = rng.uniform(0.05, 0.5, (t, 3 * sd))
    return gv_ref.normal_equations(e, dv), e, dv


def _objective_of(ab, r, mu, var, w):
    return lambda y: gv_ref.objective(ab, r, y, mu, var, w)


def test_normal_equations_are_mlpg_ref():
    (ab, r), e, dv = _system(40)
    y = mlpg_ref.mlpg_dense(e, dv)
    for k in range(3):
        assert np.allclose(scipy.linalg.solveh_banded(ab[k], r[k], lower=True), y[:, k],
                           rtol=0, atol=1e-10)
        dense = np.linalg.solve(np.diag(ab[k][0]) + np.diag(ab[k][1, :-1], -1)
                                + np.diag(ab[k][1, :-1], 1) + np.diag(ab[k][2, :-2], -2)
                                + np.diag(ab[k][2, :-2], 2), r[k])
        assert np.allclose(dense, y[:, k], rtol=0, atol=1e-10)


@pytest.mark.parametrize('weights', [(1.0, 1.0), (0.7, 2.5)])
def test_gradient_matches_finite_differences(weights):
    (ab, r), _, _ = _system(25, seed=1)
    rng = np.random.default_rng(2)
    y = rng.normal(0, 1, 25)
    mu, var = 0.4, 0.02
    f = _objective_of(ab[0], r[0], mu, var, weights)
    g = gv_ref.gradient(ab[0], r[0], y, mu, var, weights)
    h = 1e-5
    num = np.array([(f(y + h * np.eye(25)[t]) - f(y - h * np.eye(25)[t])) / (2 * h)
                    for t in range(25)])
    assert np.abs(num - g).max() <= 1e-6 * np.abs(g).max()


def test_curvature_bounds_and_exact_hessian_diagonal():
    (ab, r), _, _ = _system(30, seed=3)
    rng = np.random.default_rng(4)
    for mu in (0.01, 1.0, 5.0):
        y = rng.normal(0, 1, 30)
        w = (1.3, 0.8)
        d = gv_ref.curvature(ab[0], y, mu, 0.05, w)
        assert np.all(d >= w[0] * ab[0][0])
        # where the clip is inactive it is the diagonal of -Hessian(F)
        f = _objective_of(ab[0], r[0], mu, 0.05, w)
        h = 1e-4
        for t in (0, 7, 29):
            u = np.eye(30)[t]
            hess = (f(y + h * u) - 2 * f(y) + f(y - h * u)) / h ** 2
            e = y - y.mean()
            if (29 * (np.var(y) - mu) + 2 * e[t] ** 2) > 0:
                assert abs(-hess - d[t]) <= 1e-4 * abs(d[t])


def test_ml_trajectory_is_a_fixed_point_without_gv():
    (ab, r), _, _ = _system(50, seed=5)
    y0 = scipy.linalg.solveh_banded(ab[1], r[1], lower=True)
    y, f, acc = gv_ref.generate(ab[1], r[1], 0.3, 0.01, gv_iter=20, weights=(1.0, 0.0),
                                scale=False)
    assert np.abs(y - y0).max() <= 1e-12 * np.abs(y0).max()


@pytest.mark.parametrize('t', [1, 2, 3, 64, 300])
def test_objective_never_decreases(t):
    (ab, r), _, _ = _system(t, seed=6)
    for k, (mu, var) in enumerate([(0.5, 0.01), (2.0, 1.0), (0.01, 1e-6)]):
        y, f, acc, hist = gv_ref.generate(ab[k], r[k], mu, var, gv_iter=30, history=True)
        assert np.all(np.diff(hist) >= -1e-12 * np.abs(hist).max())
        assert hist[-1] == f
        if t >= 3:
            assert acc > 0


def test_postfilter_is_closed_form_scaling():
    (ab, r), _, _ = _system(80, seed=7)
    for k, mu in enumerate((0.05, 1.0, 3.0)):
        y0 = scipy.linalg.solveh_banded(ab[k], r[k], lower=True)
        y, _, acc = gv_ref.generate(ab[k], r[k], mu, 0.1, gv_iter=0)
        expect = y0.mean() + np.sqrt(mu / np.var(y0)) * (y0 - y0.mean())
        assert acc == 0
        assert np.abs(y - expect).max() <= 1e-12 * np.abs(expect).max()
        assert abs(np.var(y) - mu) <= 1e-12 * mu
        assert abs(y.mean() - y0.mean()) <= 1e-12 * max(1.0, abs(y0.mean()))
    # T < 2 and constant trajectories are left as they are
    one = gv_ref.scale_variance(np.array([1.5]), 2.0)
    assert np.array_equal(one, [1.5])
    assert np.array_equal(gv_ref.scale_variance(np.full(5, 0.25), 2.0), np.full(5, 0.25))


def test_diff_mode_is_the_shifted_problem():
    """Diff mode: F_diff(y) = F(s + y; r + R s) + const, so the diff-mode output is the
    solution of the shifted problem minus s."""
    (ab, r), _, _ = _system(60, seed=8)
    rng = np.random.default_rng(9)
    s = np.cumsum(rng.normal(0, 0.2, 60))
    mu, var, w = 0.8, 0.05, (1.0, 1.0)
    a, rk = ab[0], r[0]
    rs = rk + gv_ref.band_matvec(a, s)

    def f_diff(y):      # trajectory term of the difference, GV of what is heard
        return w[0] * (-0.5 * y @ gv_ref.band_matvec(a, y) + y @ rk) \
            - 0.5 * w[1] / var * (np.var(s + y) - mu) ** 2

    consts = [f_diff(y) - gv_ref.objective(a, rs, s + y, mu, var, w)
              for y in rng.normal(0, 1, (4, 60))]
    assert np.ptp(consts) <= 1e-10 * np.abs(consts).max()
    # the ML start point: R^-1 (r + R s) = s + R^-1 r
    z0 = scipy.linalg.solveh_banded(a, rs, lower=True)
    y0 = scipy.linalg.solveh_banded(a, rk, lower=True)
    assert np.abs(z0 - (s + y0)).max() <= 1e-10 * np.abs(z0).max()
    # generate_utterance in diff mode returns z - s of the shifted problem, and its gradient
    # in y is that of the shifted problem in z
    e = np.random.default_rng(10).normal(0, 1, (60, 3))
    dv = np.full((60, 3), 0.2)
    ab1, r1 = gv_ref.normal_equations(e, dv)
    y, f, acc = gv_ref.generate_utterance(e, dv, [mu], [var], 5, w, source_static=s[:, None])
    z, fz, accz = gv_ref.generate(ab1[0], r1[0] + gv_ref.band_matvec(ab1[0], s), mu, var, 5, w)
    assert np.array_equal(y[:, 0], z - s) and f[0] == fz and acc[0] == accz
    def f_d(v):
        return w[0] * (-0.5 * v @ gv_ref.band_matvec(ab1[0], v) + v @ r1[0]) \
            - 0.5 * w[1] / var * (np.var(s + v) - mu) ** 2

    gy = np.array([f_d(y[:, 0] + 1e-6 * u) - f_d(y[:, 0] - 1e-6 * u)
                   for u in np.eye(60)[:5]]) / 2e-6
    gz = gv_ref.gradient(ab1[0], r1[0] + gv_ref.band_matvec(ab1[0], s), z, mu, var, w)[:5]
    assert np.abs(gy - gz).max() <= 1e-6 * max(1.0, np.abs(gz).max())


def test_estimate_gv_is_numpy_var():
    rng = np.random.default_rng(11)
    feats = [rng.normal(0, 1 + i, (t, 4)) for i, t in enumerate((5, 1, 40, 0, 17))]
    mean, var, v = gv_ref.estimate_gv(feats)
    used = [f for f in feats if len(f)]
    expect_v = np.array([np.var(f, axis=0) for f in used])
    assert np.array_equal(v, expect_v)
    assert np.array_equal(mean, expect_v.mean(axis=0))
    assert np.array_equal(var, np.maximum(expect_v.var(axis=0), gv_ref.VAR_FLOOR))
    # one utterance: sigma^2_v is the floor
    _, var1, _ = gv_ref.estimate_gv(feats[:1])
    assert np.all(var1 == gv_ref.VAR_FLOOR)
