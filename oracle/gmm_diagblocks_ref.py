"""EM oracle for the joint GMM with diagonal covariance blocks (TEST INFRASTRUCTURE - see
oracle/__init__.py).

The joint vector is z = [x, y] with D = 2 Dh.  Each of the four Dh x Dh blocks Sxx, Sxy, Syx, Syy
of a component's covariance is diagonal, so the only coupling is between x_d and y_d: the model is
Dh independent 2 x 2 Gaussians per component.  The likelihood factorises over the pairs, so each
pair's weighted 2 x 2 empirical covariance (+ reg_covar I) is the exact constrained
maximum-likelihood estimate.

``numpy_em`` restates sklearn's EM loop as ``gmm_ref.numpy_em`` does (BaseMixture.fit_predict,
_initialize from injected responsibilities, n_k + 10 eps, weights n_k / sum n_k, the lower bound
and the stopping rule) with the per-pair M-step and an E-step that applies each pair's 2 x 2 upper
precision Cholesky factor to the direct differences z - mu.  tests/test_oracle_gmm_diagblocks.py
pins it to sklearn's full model (D = 2, where the two models coincide) and to ``gmm_ref`` on the
expanded matrices.

Compact arrays, as the device keeps them (include/kwiiyatta_b200.h):
  covariances (K, Dh, 3): [S_xx, S_xy, S_yy] per pair;
  factors (K, Dh, 3): [a, b, c] of U = [[a, b], [0, c]] with Sigma_d^-1 = U U^T.
"""
import numpy as np
from scipy.special import logsumexp


def pair_indices(d):
    """(rows, cols) of the upper pattern: (i, i), (i, Dh + i), (Dh + i, Dh + i) for every pair."""
    dh = d // 2
    i = np.arange(dh)
    return (np.concatenate([i, i, dh + i]), np.concatenate([i, dh + i, dh + i]))


def pattern_mask(d):
    """(D, D) boolean: the entries a diagonal-blocks covariance may hold (symmetric)."""
    rows, cols = pair_indices(d)
    m = np.zeros((d, d), dtype=bool)
    m[rows, cols] = True
    m[cols, rows] = True
    return m


def expand(compact, symmetric):
    """(K, Dh, 3) -> (K, D, D): covariances (``symmetric``) or the upper precision factor."""
    k, dh, _ = compact.shape
    d = 2 * dh
    out = np.zeros((k, d, d))
    i = np.arange(dh)
    out[:, i, i] = compact[:, :, 0]
    out[:, i, dh + i] = compact[:, :, 1]
    out[:, dh + i, dh + i] = compact[:, :, 2]
    if symmetric:
        out[:, dh + i, i] = compact[:, :, 1]
    return out


def compact(full):
    """(K, D, D) covariances -> (K, Dh, 3), reading the lower triangle as sklearn's Cholesky does."""
    d = full.shape[1]
    dh = d // 2
    i = np.arange(dh)
    return np.stack([full[:, i, i], full[:, dh + i, i], full[:, dh + i, dh + i]], axis=-1)


def precision_cholesky(cov):
    """Per pair: Sigma = L L^T (lower), U = L^-T = [[1/l11, -l21/(l11 l22)], [0, 1/l22]]."""
    sxx, sxy, syy = cov[..., 0], cov[..., 1], cov[..., 2]
    if not np.all(sxx > 0):
        raise ValueError('ill-defined empirical covariance')
    a = 1.0 / np.sqrt(sxx)
    l21 = sxy * a
    t = syy - l21 * l21
    if not np.all(t > 0):
        raise ValueError('ill-defined empirical covariance')
    c = 1.0 / np.sqrt(t)
    return np.stack([a, -l21 * a * c, c], axis=-1)


def estimate_parameters(x, resp, reg_covar):
    """The constrained M-step: n_k, means, per-pair weighted covariances + reg_covar I."""
    nk = resp.sum(axis=0) + 10 * np.finfo(resp.dtype).eps
    means = resp.T @ x / nk[:, None]
    k, d = means.shape
    dh = d // 2
    cov = np.empty((k, dh, 3))
    for i in range(k):
        diff = x - means[i]
        u, v = diff[:, :dh], diff[:, dh:]
        r = resp[:, i:i + 1]
        cov[i, :, 0] = (r * u * u).sum(axis=0) / nk[i] + reg_covar
        cov[i, :, 1] = (r * u * v).sum(axis=0) / nk[i]
        cov[i, :, 2] = (r * v * v).sum(axis=0) / nk[i] + reg_covar
    return nk, means, cov


def weighted_log_prob(x, weights, means, factors):
    """log N(z | mu_k, Sigma_k) + log w_k, shape (N, K), from the direct differences z - mu_k."""
    n, d = x.shape
    dh = d // 2
    k = means.shape[0]
    log_det = np.log(factors[:, :, 0]).sum(axis=1) + np.log(factors[:, :, 2]).sum(axis=1)
    out = np.empty((n, k))
    for i in range(k):
        u = x[:, :dh] - means[i, :dh]
        v = x[:, dh:] - means[i, dh:]
        a, b, c = factors[i, :, 0], factors[i, :, 1], factors[i, :, 2]
        y0 = a * u
        y1 = b * u + c * v
        out[:, i] = np.sum(y0 * y0 + y1 * y1, axis=1)
    return -0.5 * (d * np.log(2 * np.pi) + out) + log_det + np.log(weights)


def e_step(x, weights, means, factors):
    wlp = weighted_log_prob(x, weights, means, factors)
    log_prob_norm = logsumexp(wlp, axis=1)
    with np.errstate(under='ignore'):
        log_resp = wlp - log_prob_norm[:, None]
    return np.mean(log_prob_norm), log_resp


def initialize(x, resp, reg_covar):
    """GaussianMixture._initialize: one M-step from responsibilities, weights / n_samples."""
    nk, means, cov = estimate_parameters(x, resp, reg_covar)
    return nk / x.shape[0], means, cov, precision_cholesky(cov)


def numpy_em(x, resp0, max_iter=100, tol=1e-3, reg_covar=1e-6):
    """Returns dict(weights, means, covariances, precisions_cholesky, lower_bound, lower_bounds,
    n_iter, converged) like ``gmm_ref.numpy_em``; covariances and precisions_cholesky are the
    expanded (K, D, D) arrays, ``cov`` and ``factors`` the compact ones."""
    x = np.asarray(x, dtype=np.float64)
    weights, means, cov, fac = initialize(x, resp0, reg_covar)
    lower_bound = -np.inf
    bounds = []
    converged = False
    n_iter = 0
    for n_iter in range(1, max_iter + 1):
        prev = lower_bound
        lower_bound, log_resp = e_step(x, weights, means, fac)
        nk, means, cov = estimate_parameters(x, np.exp(log_resp), reg_covar)
        weights = nk / nk.sum()
        fac = precision_cholesky(cov)
        bounds.append(lower_bound)
        if abs(lower_bound - prev) < tol:
            converged = True
            break
    return dict(weights=weights, means=means, covariances=expand(cov, True),
                precisions_cholesky=expand(fac, False), cov=cov, factors=fac,
                lower_bound=lower_bound, lower_bounds=bounds, n_iter=n_iter, converged=converged)


def paired_blobs(rng, n, d, k):
    """Frames from k clusters whose covariances have diagonal blocks (x_d correlated with y_d)."""
    dh = d // 2
    centres = rng.standard_normal((k, d)) * 2.0
    lab = rng.integers(0, k, n)
    scale = rng.uniform(0.5, 1.5, (k, d))
    rho = rng.uniform(-0.8, 0.8, (k, dh))
    e = rng.standard_normal((n, d))
    u = e[:, :dh]
    v = rho[lab] * u + np.sqrt(1 - rho[lab] ** 2) * e[:, dh:]
    return centres[lab] + scale[lab] * np.hstack([u, v])
