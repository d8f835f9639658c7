"""Full-conditional-covariance MLPG oracle (TEST INFRASTRUCTURE - see oracle/__init__.py).

The maximum-likelihood trajectory of Toda, Black & Tokuda (IEEE TASLP 15(8), 2007) for the hard
mixture sequence with the FULL conditional covariance of each mixture, the algorithm of
kw_convert_fullcov_batch, restated in numpy/scipy.  nnmnkwii's MLPG.transform (oracle/mlpg_ref.py)
keeps only the element-wise diagonal D_m, so PARITY UNPINNED; this oracle is the pin, and
tests/test_oracle_mlpg_full.py checks it against its own definition.

Per mixture m of the split (and, in diff mode, rewritten) joint model:
    A_m = S_yx S_xx^-1,  offset_m = mu_y - A_m mu_x,  Sigma_m = S_yy - A_m S_xy,  P_m = Sigma_m^-1
and per utterance, with m_t = argmax_k P(k | x_t) and E_t = offset_{m_t} + A_{m_t} x_t,
    y = argmax_y  sum_t log N((W y)_t; E_t, Sigma_{m_t})   <=>   (W^T P W) y = W^T P E,
W the (3 sd T) x (sd T) delta-window matrix with zero-padded edges.  The system is
block-pentadiagonal SPD with sd x sd blocks: frame t adds
    G[a][b] = sum_{w,v} c[w][a+1] c[v][b+1] P^(w,v)       to block (t+a, t+b),
    sum_w c[w][a+1] g_t^(w),  g_t = P_{m_t} E_t           to block row t+a,
for a, b in {-1, 0, 1}, dropping blocks outside [0, T).
"""
import numpy as np
import scipy.linalg

from . import mlpg_ref
from .delta_ref import DELTA_WINDOWS


def window_coefficients(windows=DELTA_WINDOWS):
    """c[w][o + 1], the coefficient of window w at offset o in {-1, 0, 1}."""
    c = np.zeros((len(windows), 3))
    for w, (l, _, coeff) in enumerate(windows):
        c[w, 1 - l:1 - l + len(coeff)] = coeff
    return c


def conditional_full(weights, means, covariances, diff=False):
    """The split model plus A (K, Dh, Dh), offset (K, Dh) and Sigma (K, Dh, Dh)."""
    model = mlpg_ref.split_joint(weights, means, covariances, diff)
    a = np.stack([np.linalg.solve(cxx, cyx.T).T
                  for cxx, cyx in zip(model['cxx'], model['cyx'])])
    offset = model['tgt_means'] - np.einsum('krc,kc->kr', a, model['src_means'])
    sigma = model['cyy'] - a @ model['cxy']
    return dict(model, a=a, offset=offset, sigma=sigma)


def system(src, cond, windows=DELTA_WINDOWS):
    """Hard labels, conditional means E (T, Dh) and per-frame precisions P (T, Dh, Dh)."""
    src = np.asarray(src, dtype=np.float64)
    mix, _ = mlpg_ref.predict(src, cond)
    e = cond['offset'][mix] + np.einsum('trc,tc->tr', cond['a'][mix], src)
    prec = np.linalg.inv(cond['sigma'])[mix]
    return mix, e, prec


def window_matrix_full(t, sd, windows=DELTA_WINDOWS):
    """W (T * 3 sd, T * sd), frame-major rows [t][w][d] and columns [t][d]."""
    c = window_coefficients(windows)
    nw = len(windows)
    w = np.zeros((t * nw * sd, t * sd))
    eye = np.eye(sd)
    for i in range(t):
        for wi in range(nw):
            for o in (-1, 0, 1):
                if 0 <= i + o < t and c[wi, o + 1] != 0.0:
                    w[(i * nw + wi) * sd:(i * nw + wi + 1) * sd,
                      (i + o) * sd:(i + o + 1) * sd] = c[wi, o + 1] * eye
    return w


def solve_dense(e, prec, windows=DELTA_WINDOWS):
    """(W^T P W) y = W^T P E densely, (T sd)^2: for short utterances."""
    t, dh = e.shape
    sd = dh // len(windows)
    w = window_matrix_full(t, sd, windows)
    p = scipy.linalg.block_diag(*prec) if t else np.zeros((0, 0))
    r = w.T @ p @ w
    b = w.T @ (p @ e.reshape(-1))
    return np.linalg.solve(r, b).reshape(t, sd)


def solve_banded(e, prec, windows=DELTA_WINDOWS):
    """The same system assembled block by block from the G blocks and solved with scipy's banded
    Cholesky in frame-major order (bandwidth 3 sd - 1)."""
    t, dh = e.shape
    sd = dh // len(windows)
    c = window_coefficients(windows)
    nw = len(windows)
    n = t * sd
    bw = 3 * sd - 1
    ab = np.zeros((bw + 1, n))                 # lower form: ab[j - i, i] = R[j, i], j >= i
    rhs = np.zeros(n)
    ii, jj = np.meshgrid(np.arange(sd), np.arange(sd), indexing='ij')
    for f in range(t):
        pf = prec[f].reshape(nw, sd, nw, sd)
        g = prec[f] @ e[f]
        for a in (-1, 0, 1):
            if not 0 <= f + a < t:
                continue
            rhs[(f + a) * sd:(f + a + 1) * sd] += np.einsum('w,wd->d', c[:, a + 1],
                                                            g.reshape(nw, sd))
            for b in (-1, 0, 1):
                if not 0 <= f + b < t or b > a:
                    continue
                blk = np.einsum('w,v,wivj->ij', c[:, a + 1], c[:, b + 1], pf)  # block (f+a, f+b)
                row, col = (f + a) * sd + ii, (f + b) * sd + jj
                low = row >= col
                ab[(row - col)[low], col[low]] += blk[low]
    return scipy.linalg.solveh_banded(ab, rhs, lower=True).reshape(t, sd)


def objective(y, e, prec, windows=DELTA_WINDOWS):
    """sum_t -1/2 ((W y)_t - E_t)^T P_t ((W y)_t - E_t), the trajectory log-likelihood up to a
    constant."""
    t, sd = y.shape
    d = (window_matrix_full(t, sd, windows) @ y.reshape(-1)).reshape(t, -1) - e
    return -0.5 * np.einsum('ti,tij,tj->', d, prec, d)


def gradient(y, e, prec, windows=DELTA_WINDOWS):
    """W^T P (E - W y), (T, sd)."""
    t, sd = y.shape
    w = window_matrix_full(t, sd, windows)
    d = e - (w @ y.reshape(-1)).reshape(t, -1)
    return (w.T @ np.einsum('tij,tj->ti', prec, d).reshape(-1)).reshape(t, sd)


def transform(src, weights, means, covariances, diff=False, windows=DELTA_WINDOWS, banded=True,
              cond=None, return_internals=False):
    """The full-covariance ML trajectory of one utterance (T, sd); ``cond`` =
    conditional_full(...) to amortise the model over utterances."""
    if cond is None:
        cond = conditional_full(weights, means, covariances, diff)
    mix, e, prec = system(src, cond, windows)
    y = (solve_banded if banded else solve_dense)(e, prec, windows)
    if return_internals:
        return y, mix, e, prec
    return y
