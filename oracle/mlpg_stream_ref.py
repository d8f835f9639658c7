"""Low-delay (fixed-lag) MLPG oracle (TEST INFRASTRUCTURE - see oracle/__init__.py).

Low-delay conversion (Muramatsu, Ohtani, Toda, Saruwatari & Shikano, Interspeech 2008) of one
stream of static frames x~_0, x~_1, ... with a delay of L frames.  x_t = [x~_t, dx~_t, ddx~_t]
under DELTA_WINDOWS is complete once x~_{t+1} has arrived (or the stream has ended: zero padding);
its hard mixture m_t, conditional mean E_t and diagonal variance D_t are those of
``mlpg_ref.transform``.  y^(n) is the MLPG solution of the frames [0, n) alone, and

    out[s] = y^(n)[s],   n = min(s + L + 1, T).

``stream_prefix`` is that definition, one banded solve per prefix; ``stream_recursive`` restates
the recursion the device runs: the banded Cholesky factor carried forward one row per frame, a
provisional last row, and L + 1 steps of back substitution.
"""
import numpy as np
import scipy.linalg

from . import mlpg_ref
from .delta_ref import DELTA_WINDOWS, delta_features


def _coeff(windows=DELTA_WINDOWS):
    """(n_windows, 3): coefficient of window w at offsets -1, 0, +1."""
    coeff = np.zeros((len(windows), 3))
    for w, (l, _, c) in enumerate(windows):
        coeff[w, 1 - l:1 - l + len(c)] = c
    return coeff


def band(e, dv, windows=DELTA_WINDOWS):
    """The pentadiagonal systems of the frames [0, T) for all static dimensions at once, the
    assembly of ``mlpg_ref.mlpg_banded`` with array operations: ``ab`` (3, T, sd) in lower form
    (ab[k, i] = P[i + k, i], zero outside the matrix) and ``rhs`` (T, sd)."""
    t, fd = e.shape
    sd = fd // len(windows)
    coeff = _coeff(windows)
    prec = 1.0 / dv
    pm = prec * e
    ab = np.zeros((3, t, sd))
    rhs = np.zeros((t, sd))
    for w in range(len(windows)):
        p = prec[:, w * sd:(w + 1) * sd]
        q = pm[:, w * sd:(w + 1) * sd]
        for oa in (-1, 0, 1):                  # frame r adds to row r + oa
            ca = coeff[w, oa + 1]
            if ca == 0.0:
                continue
            r = np.arange(max(0, -oa), min(t, t - oa))
            np.add.at(rhs, r + oa, ca * q[r])
            for ob in (-1, 0, 1):
                cb = coeff[w, ob + 1]
                if cb == 0.0 or ob < oa:
                    continue
                rr = r[(r + ob >= 0) & (r + ob < t)]
                np.add.at(ab[ob - oa], rr + oa, ca * cb * p[rr])
    return ab, rhs


def solve(ab, rhs):
    return np.stack([scipy.linalg.solveh_banded(ab[:, :, k], rhs[:, k], lower=True)
                     for k in range(rhs.shape[1])], axis=1)


def stream_prefix(e, dv, delay, windows=DELTA_WINDOWS):
    """The definition: out[s] = y^(n)[s] with n = min(s + delay + 1, T), y^(n) the MLPG solution
    of e[:n], dv[:n]."""
    t, fd = e.shape
    out = np.zeros((t, fd // len(windows)))
    for n in sorted({min(s + delay + 1, t) for s in range(t)}):
        y = solve(*band(e[:n], dv[:n], windows))
        rows = [s for s in range(t) if min(s + delay + 1, t) == n]
        out[rows] = y[rows]
    return out


def stream_recursive(e, dv, delay, windows=DELTA_WINDOWS):
    """The device's recursion, frame by frame.  Step j (static j arrives; j = T: the stream
    ends) completes frame j-1 and
      * finalises row j-2 of the banded Cholesky factor of the whole utterance's system
        (r = 1 / L_ii, e = L_{i,i-1}, f = L_{i,i-2} = c_{i-2} r_{i-2}, z = L^-1 rhs),
      * forms row j-1 from frames j-2 and j-1 only (the prefix system's last row),
      * back-substitutes rows j-1 down to max(0, j-1-delay) and emits frame j-1-delay
        (at the end: all of them)."""
    t, fd = e.shape
    sd = fd // len(windows)
    coeff = _coeff(windows)
    prec = 1.0 / dv
    terms = np.stack([prec.reshape(t, 3, sd), (prec * e).reshape(t, 3, sd)], axis=1)
    zero = np.zeros((2, 3, sd))

    def frame(i):
        return terms[i] if 0 <= i < t else zero

    def band_row(fm, fc, fx):
        """a = R[i][i], b = R[i][i+1], c = R[i][i+2], rhs_i from frames i-1, i, i+1."""
        cm, c0, cp = coeff[:, 0:1], coeff[:, 1:2], coeff[:, 2:3]
        a = (cp * cp * fm[0] + c0 * c0 * fc[0] + cm * cm * fx[0]).sum(0)
        b = (c0 * cp * fc[0] + cm * c0 * fx[0]).sum(0)
        c = (cm * cp * fx[0]).sum(0)
        rhs = (cp * fm[1] + c0 * fc[1] + cm * fx[1]).sum(0)
        return a, b, c, rhs

    init = (np.ones(sd), np.zeros(sd), np.zeros(sd), np.zeros(sd))   # row < 0: r, e, z, c
    rows = {}

    def row(i):
        return rows.get(i, init)

    def step(i, a, b_prev, rhs):
        r2, _, z2, c2 = row(i - 2)
        r1, e1, z1, _ = row(i - 1)
        f = c2 * r2
        ee = (b_prev - f * e1) * r1
        r = 1.0 / np.sqrt(a - f * f - ee * ee)
        z = (rhs - ee * z1 - f * z2) * r
        return r, ee, z

    out = np.zeros((t, sd))
    for j in range(1, t + 1):
        if j >= 2:
            a, _, c, rhs = band_row(frame(j - 3), frame(j - 2), frame(j - 1))
            b_prev = band_row(zero, frame(j - 3), frame(j - 2))[1] if j >= 3 else np.zeros(sd)
            r, ee, z = step(j - 2, a, b_prev, rhs)
            rows[j - 2] = (r, ee, z, c)
            rows.pop(j - 4 - delay, None)      # the device keeps a ring of delay + 2 rows
        a, _, c, rhs = band_row(frame(j - 2), frame(j - 1), zero)
        b_prev = band_row(zero, frame(j - 2), frame(j - 1))[1] if j >= 2 else np.zeros(sd)
        r, ee, z = step(j - 1, a, b_prev, rhs)
        lo = max(0, j - 1 - delay)
        ys = {j - 1: z * r}
        e_n1, y1, y2 = ee, ys[j - 1], np.zeros(sd)
        for i in range(j - 2, lo - 1, -1):
            ri, ei, zi, ci = rows[i]
            ys[i] = (zi - e_n1 * y1 - (ci * ri) * y2) * ri
            e_n1, y2, y1 = ei, y1, ys[i]
        if j == t:
            for i in range(lo, j):
                out[i] = ys[i]
        elif j - 1 - delay >= 0:
            out[j - 1 - delay] = ys[j - 1 - delay]
    return out


def internals(statics, weights, means, covariances, diff=False):
    """Source vectors of a whole stream and their (mix, E, D) as ``mlpg_ref.transform`` makes
    them, with its offline solution: (y, mix, e, dv)."""
    x = delta_features(np.asarray(statics, dtype=np.float64))
    return mlpg_ref.transform(x, weights, means, covariances, diff=diff, return_internals=True)


def convert_stream(statics, weights, means, covariances, delay, diff=False, recursive=False):
    """Low-delay conversion of one stream of (T, sd) statics: (T, sd)."""
    statics = np.asarray(statics, dtype=np.float64)
    if len(statics) == 0:
        return np.zeros((0, statics.shape[1]))
    _, _, e, dv = internals(statics, weights, means, covariances, diff)
    return (stream_recursive if recursive else stream_prefix)(e, dv, delay)
