"""Global-variance (GV) oracle (TEST INFRASTRUCTURE - see oracle/__init__.py).

GV statistics and GV-considered ML trajectory generation (Toda, Black & Tokuda, "Voice
conversion based on maximum-likelihood estimation of spectral parameter trajectory", IEEE TASLP
15(8), 2007) in the form kwiiyatta_b200 builds it, per utterance and static dimension:

* normal equations R y = r of MLPG (R = W^T D^-1 W pentadiagonal, r = W^T D^-1 E), assembled as
  in mlpg_ref.mlpg_banded; y0 = R^-1 r by ``scipy.linalg.solveh_banded``;
* F(y) = w_traj (-1/2 y^T R y + y^T r) - w_gv 1/2 p (v(y) - mu_v)^2, p = 1 / sigma^2_v, with
  v(y) the population variance of y over time;
* variance scaling of y0 to mu_v (the GV postfilter; skipped for T < 2 or v(y0) = 0), then
  ``gv_iter`` steps of diagonal-Newton ascent with step control (start 0.1, x1.2 on accept,
  x0.5 on reject).  A step d is accepted when F(y + d) >= F(y): the change is evaluated in
  closed form from d (``delta_objective``), not as the difference of two rounded values of F,
  and compared with minus the bound of what the rounding of the gradient can contribute to it
  (``rounding_bound``), so that steps from a point that is stationary to rounding (T = 1: y0 is
  the optimum and r - R y0 is noise) are F-neutral and accepted by any correct implementation.
* diff mode: GV of z = s + y (s the source statics): the same problem in z with r' = r + R s.

PARITY UNPINNED: the defaults (w_traj = w_gv = 1, 20 iterations, step rule) follow HTS-style GV
generation as recalled; no external package was available to pin them, so this file is the pin.
"""
import numpy as np
import scipy.linalg

from .delta_ref import DELTA_WINDOWS

VAR_FLOOR = 1e-12          # sigma^2_v floor, as kw_gv_estimate


def estimate_gv(features, var_floor=VAR_FLOOR):
    """Per-utterance variances v (n, dim) over time (np.var), mu_v = their mean and sigma^2_v =
    their population variance (floored) over the utterances with at least one frame."""
    v = np.array([np.var(f, axis=0) for f in features if len(f) > 0])
    return v.mean(axis=0), np.maximum(v.var(axis=0), var_floor), v


def normal_equations(mean_frames, variance_frames, windows=DELTA_WINDOWS):
    """(ab, r): ab (sd, 3, T) lower banded R (ab[k, j, i] = R[i + j, i]), r (sd, T)."""
    t, d = mean_frames.shape
    sd = d // len(windows)
    ab = np.zeros((sd, 3, t))
    r = np.zeros((sd, t))
    for k in range(sd):
        for wi, (l, _, coeff) in enumerate(windows):
            prec = 1 / variance_frames[:, wi * sd + k]
            bs = prec * mean_frames[:, wi * sd + k]
            for row in range(t):
                for ka, ca in enumerate(coeff):
                    i = row + ka - l
                    if not 0 <= i < t:
                        continue
                    r[k, i] += ca * bs[row]
                    for kb, cb in enumerate(coeff):
                        j = row + kb - l
                        if 0 <= j < t and j >= i:
                            ab[k, j - i, i] += ca * prec[row] * cb
    return ab, r


def band_matvec(ab, y):
    """R y for one dimension: ab (3, T) lower banded, y (T,)."""
    out = ab[0] * y
    for j in (1, 2):
        if len(y) > j:
            out[j:] += ab[j, :-j] * y[:-j]          # R[i + j, i] y_i
            out[:-j] += ab[j, :-j] * y[j:]          # R[i, i + j] y_{i + j}
    return out


def objective(ab, r, y, mu, var, weights=(1.0, 1.0)):
    wt, wg = weights
    v = np.var(y)
    return wt * (-0.5 * y @ band_matvec(ab, y) + y @ r) - 0.5 * wg / var * (v - mu) ** 2


def gradient(ab, r, y, mu, var, weights=(1.0, 1.0)):
    wt, wg = weights
    t = len(y)
    return wt * (r - band_matvec(ab, y)) - wg / var * (np.var(y) - mu) * (2.0 / t) * (y - y.mean())


def curvature(ab, y, mu, var, weights=(1.0, 1.0)):
    """Diagonal of -Hessian(F) with the GV part clipped at zero: >= w_traj R_tt > 0."""
    wt, wg = weights
    t = len(y)
    e = y - y.mean()
    return wt * ab[0] + wg * (2.0 / var / t ** 2) * np.maximum(
        0.0, (t - 1) * (np.var(y) - mu) + 2.0 * e * e)


def delta_objective(ab, r, y, d, mu, var, weights=(1.0, 1.0)):
    """F(y + d) - F(y), in closed form."""
    wt, wg = weights
    t = len(y)
    v = np.var(y)
    dv = (2.0 / t) * ((y - y.mean()) @ d) + np.var(d)
    traj = d @ (r - band_matvec(ab, y)) - 0.5 * d @ band_matvec(ab, d)
    return wt * traj - 0.5 * wg / var * dv * (2.0 * (v - mu) + dv)


def rounding_bound(ab, r, y, d, mu, var, weights=(1.0, 1.0)):
    """What the rounding of the gradient can contribute to ``delta_objective``: 8 eps x
    (w_traj sum |d| (|r| + |R| |y|) + w_gv p (v + mu_v) (2/T) sum |d| |y - ybar|)."""
    wt, wg = weights
    t = len(y)
    absr = np.abs(ab)
    mag = band_matvec(absr, np.abs(y))
    return 8 * np.finfo(float).eps * (
        wt * (np.abs(d) @ (np.abs(r) + mag))
        + wg / var * (np.var(y) + mu) * (2.0 / t) * (np.abs(d) @ np.abs(y - y.mean())))


def scale_variance(y, mu):
    """The GV postfilter: y scaled about its mean to variance mu (unchanged if T < 2 or v = 0)."""
    v = np.var(y)
    if len(y) < 2 or v == 0.0:
        return y.copy()
    return y.mean() + np.sqrt(mu / v) * (y - y.mean())


def generate(ab, r, mu, var, gv_iter=20, weights=(1.0, 1.0), y0=None, scale=True,
             history=False):
    """GV-considered generation for one dimension.  Returns (y, F, accepted[, F per step])."""
    y = scipy.linalg.solveh_banded(ab, r, lower=True) if y0 is None else np.asarray(y0, float)
    if scale:
        y = scale_variance(y, mu)
    step, accepted = 0.1, 0
    hist = [objective(ab, r, y, mu, var, weights)]
    for _ in range(gv_iter):
        d = step * gradient(ab, r, y, mu, var, weights) / curvature(ab, y, mu, var, weights)
        if delta_objective(ab, r, y, d, mu, var, weights) >= \
                -rounding_bound(ab, r, y, d, mu, var, weights):
            y = y + d
            step *= 1.2
            accepted += 1
        else:
            step *= 0.5
        hist.append(objective(ab, r, y, mu, var, weights))
    out = (y, hist[-1], accepted)
    return out + (np.array(hist),) if history else out


def generate_utterance(e, dv, mu, var, gv_iter=20, weights=(1.0, 1.0), source_static=None,
                       windows=DELTA_WINDOWS):
    """All static dimensions of one utterance from the conditional means / variances E, D.
    ``source_static`` (T, sd): diff mode, GV of source + output.  Returns (y (T, sd),
    F (sd,), accepted (sd,))."""
    ab, r = normal_equations(e, dv, windows)
    sd, t = r.shape
    y = np.empty((t, sd))
    f = np.empty(sd)
    acc = np.empty(sd, dtype=np.int64)
    for k in range(sd):
        rk = r[k]
        if source_static is not None:
            rk = rk + band_matvec(ab[k], source_static[:, k])     # r' = r + R s
        z, f[k], acc[k] = generate(ab[k], rk, mu[k], var[k], gv_iter, weights)
        y[:, k] = z - source_static[:, k] if source_static is not None else z
    return y, f, acc


def transform(src, weights, means, covariances, gv_mean, gv_var, diff=False, gv_iter=20,
              gv_weights=(1.0, 1.0)):
    """MLPG conversion with GV (mlpg_ref.transform's posterior and conditional Gaussian)."""
    from . import mlpg_ref
    src = np.asarray(src, dtype=np.float64)
    _, _, e, dv = mlpg_ref.transform(src, weights, means, covariances, diff=diff,
                                     return_internals=True)
    sd = src.shape[1] // 3
    return generate_utterance(e, dv, gv_mean, gv_var, gv_iter, gv_weights,
                              source_static=src[:, :sd] if diff else None)
