"""EM trajectory-estimation oracle (TEST INFRASTRUCTURE - see oracle/__init__.py).

Maximum-likelihood conversion over all mixture sequences (Toda, Black & Tokuda, IEEE TASLP
15(8), 2007), the algorithm of kw_convert_em_batch, restated densely in numpy/scipy.  The reference
(nnmnkwii's MLPG.transform, oracle/mlpg_ref.py) only has the hard-sequence approximation, so
PARITY UNPINNED; this oracle is the pin, and tests/test_oracle_mlpg_em.py checks it against its
own definition.

Model, per mixture m of the split (and, in diff mode, rewritten) joint model:
    P(Y_t | x_t, m) = N(Y_t; E_{m,t}, diag D_m),  E_{m,t} = mu_y + A_m (x_t - mu_x),
    A_m = S_yx S_xx^-1,  D_m = diag(S_yy) - diag(S_yx) / diag(S_xx) * diag(S_xy)
(the diagonal conditional variance the hard-sequence MLPG uses) and the objective per utterance
    L(y) = sum_t log sum_m w_m N(x_t; mu_x, S_xx) N((W y)_t; E_{m,t}, diag D_m).
The summand is one Gaussian in z_t = [x_t ; (W y)_t] (``joint_model``), so the E-step is the GMM
E-step on z.  M-step: P_t = sum_m g D_m^-1, q_t = sum_m g D_m^-1 E_{m,t} with g = gamma where
gamma > FLOOR and 0 elsewhere, then (W^T P W) y = W^T q per static dimension.  Because E-step
and M-step use the same model, no iteration decreases L.
"""
import numpy as np
from scipy.special import logsumexp

from . import gmm_ref, mlpg_ref
from .delta_ref import DELTA_WINDOWS

FLOOR = 1e-14   # posteriors at or below this contribute nothing to the M-step


def conditional(weights, means, covariances, diff=False):
    """The split model plus A (K, Dh, Dh), offset = mu_y - A mu_x (K, Dh) and D (K, Dh)."""
    model = mlpg_ref.split_joint(weights, means, covariances, diff)
    a = np.stack([np.linalg.solve(cxx, cyx.T).T
                  for cxx, cyx in zip(model['cxx'], model['cyx'])])
    offset = model['tgt_means'] - np.einsum('krc,kc->kr', a, model['src_means'])
    var = (np.diagonal(model['cyy'], axis1=1, axis2=2)
           - np.diagonal(model['cyx'], axis1=1, axis2=2)
           / np.diagonal(model['cxx'], axis1=1, axis2=2)
           * np.diagonal(model['cxy'], axis1=1, axis2=2))
    return dict(model, a=a, offset=offset, var=var)


def joint_model(cond):
    """Means (K, 2Dh) and upper precision Cholesky factors L~ (K, 2Dh, 2Dh) of the Gaussian in
    z = [x ; Y]:  L~ = [[Lx, -A^T D^-1/2], [0, D^-1/2]]."""
    k, dh = cond['offset'].shape
    means = np.concatenate([cond['src_means'], cond['tgt_means']], axis=1)
    pc = np.zeros((k, 2 * dh, 2 * dh))
    isd = 1.0 / np.sqrt(cond['var'])
    for m in range(k):
        pc[m, :dh, :dh] = cond['px_prec_chol'][m]
        pc[m, :dh, dh:] = -cond['a'][m].T * isd[m][None, :]
        pc[m, dh:, dh:] = np.diag(isd[m])
    return means, pc


def window_apply(y, windows=DELTA_WINDOWS):
    """W y: (T, sd) -> (T, len(windows) * sd), zero padded at the edges."""
    t = len(y)
    return np.concatenate([mlpg_ref.window_matrix(w, t) @ y for w in windows], axis=1)


def e_step(src, y, cond, joint):
    """Posteriors gamma (T, K) and per-frame log-normalisers (T,) at trajectory y."""
    z = np.concatenate([src, window_apply(y)], axis=1)
    wlp = gmm_ref.weighted_log_prob(z, cond['weights'], joint[0], joint[1])
    lse = logsumexp(wlp, axis=1)
    return np.exp(wlp - lse[:, None]), lse


def cond_means(src, cond):
    """E_{m,t}: (K, T, Dh)."""
    return cond['offset'][:, None, :] + np.einsum('krc,tc->ktr', cond['a'], src)


def precision_terms(src, gamma, cond, floor=FLOOR):
    """P (T, Dh) and q (T, Dh) from the posteriors, terms with gamma <= floor dropped."""
    g = np.where(gamma > floor, gamma, 0.0)
    prec = g @ (1.0 / cond['var'])
    q = np.einsum('tk,kr,ktr->tr', g, 1.0 / cond['var'], cond_means(src, cond))
    return prec, q


def m_step(src, gamma, cond, floor=FLOOR):
    """The trajectory maximising sum_t sum_m g (W y - E)^T D^-1 (W y - E): the MLPG system with
    per-frame precision P_t and mean q_t / P_t, solved by banded Cholesky."""
    prec, q = precision_terms(src, gamma, cond, floor)
    return mlpg_ref.mlpg_banded(q / prec, 1.0 / prec)


def objective(src, y, cond, joint):
    return float(e_step(src, y, cond, joint)[1].sum())


def convert(src, weights, means, covariances, diff=False, em_iter=1, floor=FLOOR):
    """(y, trace): y after em_iter iterations from the hard-sequence MLPG output, and the
    objective L(y_k) for k = 0 .. em_iter."""
    src = np.asarray(src, dtype=np.float64)
    sd = src.shape[1] // len(DELTA_WINDOWS)
    if len(src) == 0:
        return np.zeros((0, sd)), np.zeros(em_iter + 1)
    cond = conditional(weights, means, covariances, diff)
    joint = joint_model(cond)
    y = mlpg_ref.transform(src, weights, means, covariances, diff=diff)
    trace = []
    for _ in range(em_iter):
        gamma, lse = e_step(src, y, cond, joint)
        trace.append(lse.sum())
        y = m_step(src, gamma, cond, floor)
    trace.append(objective(src, y, cond, joint))
    return y, np.array(trace)
