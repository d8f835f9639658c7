"""Error bounds of the tensor-core GMM kernels, element by element, with a numpy witness
(TEST INFRASTRUCTURE - see oracle/__init__.py).

``estep_bound`` bounds |wlp_tc - wlp_fp64| for every (frame, component) of the tensor-core E-step
(gmm_tc.cu: pack_x_kernel, pack_l_kernel, estep_tc_kernel); ``mstats_bound`` bounds every element
of the statistics vector the tensor-core M-step (mstats_tc2_kernel and its prep / post kernels)
writes through ``kw_gmm_mstep_accumulate``.  ``emulate_estep`` / ``emulate_mstats`` compute what
those kernels compute, with fp16 operands from ``np.float16`` and fp32 products and sums rounded
to nearest; their ``defect`` argument reproduces a named kernel bug, so tests can show that the
bounds are tight enough to catch it (tests/test_oracle_tc_bound.py).

Units: u = 2^-23 is one fp32 ulp at 1 (the tensor core's accumulator TRUNCATES, so an
accumulation step errs by up to u relative, twice round-to-nearest's u / 2); fp16 operands are
split v = hi + lo 2^-11, hi = fp16(v), lo = fp16((v - hi) 2^11), which leaves |v - hi - lo 2^-11|
<= 2^-22 |v| for normal values (fp16 rounds to 2^-11 relative, twice) and 2^-36 absolute below
fp16's normal range.
"""
import numpy as np

TILE_E = 128                # frames per E-step tile
TILE_M = 64                 # frames per M-step tile
TILE_FLOOR = np.float32(1e-8)   # an M-step (component, tile) pair enters only above this
U = 2.0 ** -23
LOG2PI = np.log(2 * np.pi)
SMS = 148


def dp_of(d):
    return (d + 15) // 16 * 16


def _pow2_above(a):
    """2^e with a = m 2^e, m in [0.5, 1) (frexp), i.e. the power of two just above |a|; 1 for 0."""
    m, e = np.frexp(a)
    return np.where((a > 0) & np.isfinite(a), np.ldexp(1.0, e), 1.0)


def column_stats(x):
    """Centre c and power-of-two scale sigma of the frames (colstats_final_kernel)."""
    c = x.mean(axis=0)
    amax = np.maximum(x.max(axis=0) - c, c - x.min(axis=0))
    return c, _pow2_above(amax)


def packed_operands(x, means, prec_chol):
    """The E-step's operands before the fp16 split: x' = (x - c) / sigma, and per component
    B_k = diag(sigma) L_k 2^-t_k and the bias b'_k 2^-t_k, b'_k = (mu_k - c) L_k, with 2^t_k the
    power of two above the largest |entry| of both (pack_l_kernel).  Returns (x', B, bias, 4^t)."""
    c, sig = column_stats(x)
    xs = (x - c) / sig
    lp = prec_chol * sig[None, :, None]
    bp = np.einsum('kd,kdj->kj', means - c, prec_chol)
    amax = np.maximum(np.abs(lp).max(axis=(1, 2)), np.abs(bp).max(axis=1))
    scale = _pow2_above(amax)
    return xs, lp / scale[:, None, None], bp / scale[:, None], scale * scale


def estep_epsilon(d):
    """Relative error of one y_j = sum_d x'_d B_dj - b_j of the E-step, per unit of
    sum_d |x'_d B_dj| + |b_j| (all in the scaled units of the packed operands):

      operands  3 * 2^-22   x' and B each split to 2^-22 (module docstring), and the dropped
                            x_lo l_lo 2^-22 term (|x_lo 2^-11| <= 2^-11 |x|, same for l);
      main pass 2u per MMA  the ksteps + 1 MMAs of x_hi l_hi and of the bias each truncate their
                            result (u of the partial sum, which is <= the sum of |terms|) and align
                            their 16 products to the largest one (another u of that sum);
      cross     u           x_hi l_lo + x_lo l_hi run first and enter at 2^-11: their 2 ksteps
                            truncations are 2^-11 of the above, u covers them and the bias split.

    eps = (6 + 2 (ksteps + 1) + 1) u; at D = 144 (9 k-steps) 27 u = 3.2e-6, at D = 72 19 u.
    Round-to-nearest would need half of the accumulation terms: the constant covers truncation by
    a factor 2 over the rounding the witness (emulate_estep) does."""
    ks = dp_of(d) // 16
    return (6 + 2 * (ks + 1) + 1) * U


def _split(v):
    hi = v.astype(np.float16)
    lo = ((v - hi.astype(np.float64)) * 2048.0).astype(np.float16)
    return hi.astype(np.float32), lo.astype(np.float32)


def estep_reference(x, weights, means, prec_chol):
    """FP64 y (scaled as in the kernel, (K, N, D)) and wlp (N, K)."""
    xs, b, bias, s4 = packed_operands(x, means, prec_chol)
    y = np.matmul(xs[None], b) - bias[:, None, :]
    log_det = np.log(np.diagonal(prec_chol, axis1=1, axis2=2)).sum(axis=1)
    q = (y * y).sum(axis=2) * s4[:, None]
    wlp = (-0.5 * (x.shape[1] * LOG2PI + q) + log_det[:, None] + np.log(weights)[:, None]).T
    return y, wlp


def estep_bound(x, weights, means, prec_chol, return_y=False):
    """Per-element bound on |wlp_tc - wlp_fp64|, shape (N, K).

    With e_j = eps (sum_d |x'_d B_dj| + |b_j|) + D 2^-35 (estep_epsilon; the last term covers
    fp16's subnormal range) the accumulator holds y_j + d_j, |d_j| <= e_j, so
    |q~ - q| <= sum_j (2 |y_j| e_j + e_j^2) + 2^-21 sum_j (|y_j| + e_j)^2, the last term for the
    epilogue's fp32 sums of squares (at most 7 roundings to nearest per 16 columns), and
    |wlp~ - wlp| <= 4^t |q~ - q| / 2 plus the fp64 rounding of both sides (1e-13 (|wlp| + D)).
    ``return_y``: also (y, e) of the k-th component as (K, N, D) arrays."""
    x = np.asarray(x, dtype=np.float64)
    d = x.shape[1]
    xs, b, bias, s4 = packed_operands(x, means, prec_chol)
    y, wlp = estep_reference(x, weights, means, prec_chol)
    mag = np.matmul(np.abs(xs)[None], np.abs(b)) + np.abs(bias)[:, None, :]
    e = estep_epsilon(d) * mag + d * 2.0 ** -35
    ay = np.abs(y)
    qerr = (2 * ay * e + e * e).sum(axis=2) + 2.0 ** -21 * ((ay + e) ** 2).sum(axis=2)
    bound = (0.5 * s4[:, None] * qerr).T + 1e-13 * (np.abs(wlp) + d)
    return (bound, y, e) if return_y else bound


def emulate_estep(x, weights, means, prec_chol, defect=None):
    """What estep_tc_kernel computes, in numpy: split fp16 operands, fp32 products, fp32 sums
    rounded to nearest in the kernel's pass order (x_hi l_lo, x_lo l_hi, * 2^-11, x_hi l_hi,
    bias), fp32 squares summed per 16 columns, the rest in fp64.  Returns (wlp (N, K), y (K, N, D)).

    defect: None (faithful), 'drop_lo_pass' (the x_lo l_hi pass is skipped), or 'drop_tail'
    (the real columns of a partial last k-step, 16 floor(D/16) .. D - 1, are treated as padding)."""
    x = np.asarray(x, dtype=np.float64)
    n, d = x.shape
    xs, b, bias, s4 = packed_operands(x, means, prec_chol)
    if defect == 'drop_tail':
        xs = xs.copy()
        xs[:, 16 * (d // 16):] = 0.0
    xh, xl = _split(xs)
    k = means.shape[0]
    f32 = np.float32
    ys = np.empty((k, n, d))
    for c in range(k):
        bh, bl = _split(b[c])
        acc = np.zeros((n, d), dtype=f32)
        for dd in range(d):
            acc = (acc + (xh[:, dd, None] * bl[None, dd, :])).astype(f32)
        if defect != 'drop_lo_pass':
            for dd in range(d):
                acc = (acc + (xl[:, dd, None] * bh[None, dd, :])).astype(f32)
        acc = (acc * f32(2.0 ** -11)).astype(f32)
        for dd in range(d):
            acc = (acc + (xh[:, dd, None] * bh[None, dd, :])).astype(f32)
        nb = -bias[c]
        nbh = nb.astype(np.float16).astype(np.float64)
        nbl = ((nb - nbh) * 2048.0).astype(np.float16).astype(np.float64)
        acc = (acc + nbh.astype(f32)).astype(f32)
        acc = (acc + (nbl * 2.0 ** -11).astype(f32)).astype(f32)
        ys[c] = acc
    sq = (ys.astype(f32) ** 2).astype(f32)
    pad = (-d) % 16
    sq = np.concatenate([sq, np.zeros((k, n, pad), dtype=f32)], axis=2)
    q = sq.reshape(k, n, -1, 16).sum(axis=3, dtype=f32).astype(np.float64).sum(axis=2)
    log_det = np.log(np.diagonal(prec_chol, axis1=1, axis2=2)).sum(axis=1)
    wlp = (-0.5 * (d * LOG2PI + q * s4[:, None]) + log_det[:, None] +
           np.log(weights)[:, None]).T
    return wlp, ys


# ------------------------------------------------------------------------------------------
# M-step statistics
# ------------------------------------------------------------------------------------------
def m_chunks(k, n_mtiles):
    """tc_m_chunks (gmm_tc.cu): frame chunks per component of the tensor-core M-step."""
    best, best_eff = 1, 0.0
    for c in range(1, 65):
        if c > n_mtiles:
            break
        items = k * c
        if items < SMS and c < 64 and c + 1 <= n_mtiles:
            continue
        waves = (items + SMS - 1) // SMS
        eff = items / (waves * SMS)
        if eff > best_eff + 1e-9:
            best_eff, best = eff, c
        if items >= 8 * SMS:
            break
    return best


def tile_mask(resp):
    """(K, N) bool: frames of the (component, 64-frame tile) pairs the M-step keeps -- those with
    a weight above the floor as fp32 (mstats_tc_prep_kernel / lse_prep_kernel)."""
    n, k = resp.shape
    nt = (n + TILE_M - 1) // TILE_M
    r = np.zeros((nt * TILE_M, k), dtype=np.float32)
    r[:n] = resp.astype(np.float32)
    on = r.reshape(nt, TILE_M, k).max(axis=1) > TILE_FLOOR          # (tiles, K)
    return np.repeat(on, TILE_M, axis=0)[:n].T


def mstats_reference(x, resp, centres):
    """FP64 statistics over the kept tiles, shape (K, 1 + D + D^2): n_k, sum r (x - c_k),
    sum r (x - c_k)(x - c_k)^T -- the layout kw_gmm_mstep_accumulate writes."""
    x = np.asarray(x, dtype=np.float64)
    n, d = x.shape
    keep = tile_mask(resp)
    out = np.empty((resp.shape[1], 1 + d + d * d))
    for k in range(resp.shape[1]):
        r = np.where(keep[k], resp[:, k], 0.0)
        u = x - centres[k]
        out[k, 0] = r.sum()
        out[k, 1:1 + d] = r @ u
        out[k, 1 + d:] = ((u * r[:, None]).T @ u).ravel()
    return out


def _mstep_scaled(x, centres):
    """x' (packed as for the E-step), mu'_k = fp32((c_k - c) / sigma) and the effective-centre
    offsets e_k = c + sigma mu'_k - c_k of the post kernel, in original units."""
    c, sig = column_stats(x)
    xs = (x - c) / sig
    mu = ((centres - c) / sig).astype(np.float32).astype(np.float64)
    return xs, mu, sig, (c + sig * mu) - centres


def mstats_epsilon():
    """Relative error per unit of sum_n r |u_ni| |x'_nj| of one tensor-core M-step element (u =
    x' - mu', x' the scaled frames): the operands z = r u (fp32: r, x_hi + x_lo, - mu, * r, then the
    fp16 split) and x' (split, the dropped lo x lo term), 2^-22 each as for the E-step, with z's
    fp32 steps another 4 * 2^-24 of |r| (|x'| + |u|) -- see mstats_bound; per 64-frame tile the
    4 MMAs of the main pass at 2u each (truncation and alignment), the 8 cross-pass MMAs at
    2^-11 of that, and the post kernel's truncation gain 1 + 0.65 u: (8 + 1 + 1) u."""
    return 10 * U


def mstats_bound(x, resp, centres):
    """Per-element bound on |stats_tc - stats_fp64| (mstats_reference), shape (K, 1 + D + D^2).

    In the scaled units of the kernel (x', mu', u = x' - mu', a = |x'|, r the weight of frame n):
      z error      ez_ni <= r (2.5 2^-22 (a_i + |u_i|) + 2^-24) + 2^-24 m_t     (m_t: tile maximum;
                   the last term is fp16's subnormal step 2^-25 at the tile's weight scale)
      x' error     2^-22 a_j + 2^-25                       (lo is stored unscaled: subnormal step)
      S_ij = sum_n z_ni x'_nj:   E_S <= sum_n [ez_ni a_j + r |u_i| (2^-21 a_j + 2^-25)]
                                        + sum_n w_n r |u_i| a_j,
      w_n = mstats_epsilon() + T_c 2^-24 for a frame of chunk c with T_c kept tiles (the fp32
      flush of each tile into the item's accumulator rounds to nearest at most T_c times);
      mc_i = sum_n z_ni (the ones column, a = 1 exact) likewise, and V_ij = S_ij - mc_i mu'_j:
      E_V <= E_S + |mu'_j| E_mc, taken as max(E_V_ij, E_V_ji) for the symmetrised element.
    In original units (post kernel): s_i s_j E_V + s_i E_mc_i |e_j| + |e_i| s_j E_mc_j for the
    second moments, s_i E_mc_i for the first, plus 1e-12 of each element's fp64 scale; n_k is
    fp64 from the start (1e-12 relative)."""
    x = np.asarray(x, dtype=np.float64)
    n, d = x.shape
    kk = resp.shape[1]
    xs, mu, sig, eoff = _mstep_scaled(x, centres)
    keep = tile_mask(resp)
    nt = (n + TILE_M - 1) // TILE_M
    chunks = m_chunks(kk, nt)
    tpc = (nt + chunks - 1) // chunks
    tile_of = np.arange(n) // TILE_M
    a = np.abs(xs)
    out = np.empty((kk, 1 + d + d * d))
    for k in range(kk):
        r = np.where(keep[k], resp[:, k], 0.0)
        rt = np.zeros(nt * TILE_M)
        rt[:n] = r
        mt = np.repeat(rt.reshape(nt, TILE_M).max(axis=1), TILE_M)[:n]
        on_tile = rt.reshape(nt, TILE_M).max(axis=1) > 0
        kept_in_chunk = np.add.reduceat(on_tile.astype(float), np.arange(0, nt, tpc))
        w = mstats_epsilon() + kept_in_chunk[tile_of // tpc] * 2.0 ** -24
        au = np.abs(xs - mu[k])
        ez = r[:, None] * (2.5 * 2.0 ** -22 * (a + au) + 2.0 ** -24) + \
            2.0 ** -24 * mt[:, None] * (r > 0)[:, None]
        rau = r[:, None] * au
        e_s = ez.T @ a + rau.T @ (2.0 ** -21 * a + 2.0 ** -25) + (rau * w[:, None]).T @ a
        e_mc = ez.sum(axis=0) + 2.0 ** -22 * rau.sum(axis=0) + (rau * w[:, None]).sum(axis=0)
        e_v = e_s + e_mc[:, None] * np.abs(mu[k])[None, :]
        e_v = np.maximum(e_v, e_v.T)
        ek = np.abs(eoff[k])
        e2 = np.outer(sig, sig) * e_v + np.outer(sig * e_mc, ek) + np.outer(ek, sig * e_mc)
        out[k, 0] = 1e-12 * r.sum()
        out[k, 1:1 + d] = sig * e_mc
        out[k, 1 + d:] = e2.ravel()
    ref = mstats_reference(x, resp, centres)
    m1 = np.abs(ref[:, 1:1 + d])
    m2 = np.abs(ref[:, 1 + d:]).reshape(kk, d, d)
    out[:, 1:1 + d] += 1e-12 * (m1 + 1.0)
    diag = np.sqrt(np.abs(np.diagonal(m2, axis1=1, axis2=2)))
    out[:, 1 + d:] += 1e-12 * (np.einsum('ki,kj->kij', diag, diag).reshape(kk, -1) + 1.0)
    return out


def emulate_mstats(x, resp, centres, defect=None):
    """What the tensor-core M-step computes, in numpy, rounded to nearest: per kept (component,
    64-frame tile) z = r' ((x_hi + x_lo) - mu') in fp32 (r' the tile's weights scaled by a power
    of two into [0.5, 1) at the maximum), split into fp16 hi / lo, the three passes (z_hi x_lo,
    z_lo x_hi, z_hi x_hi, frame by frame in fp32), the tile flushed into the chunk's fp32
    accumulator times the inverse scale, chunks summed in fp64, and the post kernel's centring
    and gain.  defect: None or 'drop_lo_pass' (the z_lo x_hi pass is skipped)."""
    x = np.asarray(x, dtype=np.float64)
    n, d = x.shape
    kk = resp.shape[1]
    f32 = np.float32
    xs, mu, sig, eoff = _mstep_scaled(x, centres)
    nt = (n + TILE_M - 1) // TILE_M
    chunks = m_chunks(kk, nt)
    tpc = (nt + chunks - 1) // chunks
    npad = nt * TILE_M
    xp = np.zeros((npad, d + 1))
    xp[:n, :d] = xs
    xp[:n, d] = 1.0                                # the ones column (first moments)
    xh = xp.astype(np.float16)
    xl = (xp - xh.astype(np.float64)).astype(np.float16)
    xh32, xl32 = xh.astype(f32), xl.astype(f32)
    xr = (xh32[:, :d] + xl32[:, :d]).astype(f32)  # the generators' x' in fp32
    out = np.empty((kk, 1 + d + d * d))
    gain = 1.0 + 0.65 * U
    for k in range(kk):
        rr = np.zeros(npad, dtype=f32)
        rr[:n] = resp[:, k].astype(f32)
        rt = rr.reshape(nt, TILE_M)
        m = rt.max(axis=1)
        on = m > TILE_FLOOR
        _, ex = np.frexp(m.astype(np.float64))
        up = np.ldexp(1.0, -ex).astype(f32)
        inv = np.ldexp(1.0, ex).astype(f32)
        rs = (rt * up[:, None]).astype(f32).reshape(-1)
        z = (rs[:, None] * (xr - f32(0) - mu[k].astype(f32)).astype(f32)).astype(f32)
        zh = z.astype(np.float16).astype(f32)
        zl = (z - zh).astype(f32).astype(np.float16).astype(f32)
        tot = np.zeros((d, d + 1))
        for c0 in range(0, nt, tpc):
            acc = np.zeros((d, d + 1), dtype=f32)
            for t in range(c0, min(nt, c0 + tpc)):
                if not on[t]:
                    continue
                sl = slice(t * TILE_M, (t + 1) * TILE_M)
                tile = np.zeros((d, d + 1), dtype=f32)
                passes = [(zh, xl32), (zh, xh32)] if defect == 'drop_lo_pass' else \
                    [(zh, xl32), (zl, xh32), (zh, xh32)]
                for za, xb in passes:
                    for f in range(sl.start, sl.stop):
                        tile = (tile + np.outer(za[f], xb[f]).astype(f32)).astype(f32)
                acc = (acc + tile * inv[t]).astype(f32)
            tot += acc.astype(np.float64)
        tot *= gain
        mc = tot[:, d]
        v = tot[:, :d] - np.outer(mc, mu[k])
        v = 0.5 * (v + v.T)
        e = eoff[k]
        mi = sig * mc
        rk = np.where(np.repeat(on, TILE_M)[:n], resp[:, k], 0.0)
        nk = rk.sum()
        out[k, 0] = nk
        out[k, 1:1 + d] = sig * mc + nk * e
        out[k, 1 + d:] = (np.outer(sig, sig) * v + np.outer(mi, e) + np.outer(e, mi) +
                          nk * np.outer(e, e)).ravel()
    return out
