"""The tensor-core GMM kernels (gmm_tc.cu) element by element against FP64 references, at the
operand geometries where they branch: DP = round_up(D, 16) (the number of k-steps), two
components per MMA (DP <= 96 and K >= 2) or one, odd K padded to a pair, the mma.sync corner of
the M-step (D > 128), partial last E-tiles (128 frames) and M-tiles (64 frames), the persistent
grid looping (more than 148 E-tiles), the M-step's chunking regimes, components without a tile
above the floor, and frames re-sorted by dominant component.

Tolerances are the bounds of oracle/tc_bound.py; tests/test_oracle_tc_bound.py shows on the CPU
that a kernel which lost the lo operand on one pass, or the real columns of a partial last
k-step, breaks them on most elements.  The hard labels must equal the FP64 argmax, including on
frames whose three or four best components lie within 1e-6 nat of each other."""
import numpy as np
import pytest

from kwiiyatta_b200 import _lib
from kwiiyatta_b200.gmm import GaussianMixture
from oracle import gmm_ref, tc_bound

pytestmark = pytest.mark.gpu

DIMS = [1, 3, 15, 16, 17, 31, 32, 33, 47, 48, 63, 72, 80, 81, 95, 96, 97, 111, 112, 113, 127,
        128, 129, 143, 144]
N_LOOP = 148 * 128 + 77          # 149 E-tiles: the persistent grid loops, the last tile partial
N_EDGES = [1, 127, 128, 129, N_LOOP]
K_ODD, K_EVEN = [1, 3, 63, 65, 129], [2, 64, 384]
WORK = 4e8                       # N K D^2 per case: the numpy reference in about a second


def _estep_cases():
    cases = []
    for i, d in enumerate(DIMS):
        for ks in (K_ODD, K_EVEN):
            k = ks[i % len(ks)]
            n = N_EDGES[(i + len(cases)) % len(N_EDGES)]
            while n * k * d * d > WORK and n > 129:
                n = 129
            cases.append((d, k, n))
    # every N edge with two components per MMA (DP 48) and with one (DP 144, and K = 1)
    cases += [(48, 3, n) for n in N_EDGES] + [(144, 2, n) for n in N_EDGES]
    cases += [(40, 1, n) for n in N_EDGES]
    return sorted(set(cases))


def _model(d, k, n, seed):
    rng = np.random.default_rng(seed)
    centres = rng.standard_normal((k, d)) * 2.0
    a = rng.standard_normal((k, d, d)) * (0.3 / np.sqrt(max(d, 16) / 16.0)) + np.eye(d)
    cov = np.einsum('kij,klj->kil', a, a) + 0.05 * np.eye(d)
    lab = rng.integers(0, k, n)
    x = centres[lab] + np.einsum('nij,nj->ni', a[lab], rng.standard_normal((n, d)))
    w = rng.uniform(0.5, 1.5, k)
    return x, w / w.sum(), centres, cov


def _device_model(torch, x, w, m, cov):
    """A tensor-core GaussianMixture with the given parameters, its buffers and workspace sized
    for x, and x packed.  Returns (gm, x on the device)."""
    n, d = x.shape
    gm = GaussianMixture(n_components=len(w), precision='tc', reorder_every=0)
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    gm._alloc(torch, n, d, xd.device)
    gm.set_parameters(w, m, cov)
    gm._x_src, gm._x_used = xd, None
    gm._pack(torch, xd)
    return gm, xd


def _labels(torch, gm, xd, precision):
    n, d = xd.shape
    k = gm.n_components
    lab = torch.empty(n, dtype=torch.int32, device=xd.device)
    _lib.call('kw_gmm_hard_labels', n, xd, k, d, gm._means[gm._cur], gm._pc, gm._aux, lab,
              precision, gm._ws, gm._ws_bytes, _lib.stream_ptr(torch))
    return lab.cpu().numpy()


def _fp64_argmax_checkable(wlp):
    """np.argmax (lowest index on equal values, as refine_argmax_kernel) and the frames whose
    gap to the runner-up is above 1e-11, where summation order cannot decide."""
    top = wlp.argmax(axis=1)
    if wlp.shape[1] == 1:
        return top, np.ones(len(top), dtype=bool)
    srt = np.sort(wlp, axis=1)
    return top, (srt[:, -1] - srt[:, -2]) > 1e-11


@pytest.mark.parametrize('d,k,n', _estep_cases())
def test_estep_wlp_loglik_and_labels(cuda, d, k, n):
    """Every weighted log-probability of the tensor-core E-step within estep_bound, the
    log-likelihood sum of the statistics tail within the bound propagated to it (logsumexp is
    1-Lipschitz in the max norm), and the hard labels of both precisions equal to the FP64 argmax."""
    torch = cuda
    x, w, m, cov = _model(d, k, n, 1000 * d + k + n)
    gm, xd = _device_model(torch, x, w, m, cov)
    gm._estep(torch, xd, for_mstep=True)
    assert gm._resp_log
    got = gm._resp[:, :n].t().cpu().numpy()
    pc = gm.precisions_cholesky_
    bound = tc_bound.estep_bound(x, gm.weights_, gm.means_, pc)
    _, ref = tc_bound.estep_reference(x, gm.weights_, gm.means_, pc)
    ratio = np.abs(got - ref) / bound
    print(f'D = {d} (DP {tc_bound.dp_of(d)}), K = {k}, N = {n}: max |wlp error| / bound = '
          f'{ratio.max():.3g}, max |wlp error| = {np.abs(got - ref).max():.3g}')
    assert ratio.max() <= 1.0
    lse = np.logaddexp.reduce(ref, axis=1)
    tail = gm._stats[-2:].cpu().numpy()
    assert tail[1] == n
    assert abs(tail[0] - lse.sum()) <= bound.max(axis=1).sum() + 1e-12 * np.abs(lse).sum()
    top, ok = _fp64_argmax_checkable(ref)
    for precision in (1, 0):
        lab = _labels(torch, gm, xd, precision)
        assert np.array_equal(lab[ok], top[ok]), \
            f'precision {precision}: {(lab[ok] != top[ok]).sum()} labels differ'


@pytest.mark.parametrize('n', [64 * 40 + 37, 64 * 301])
def test_estep_for_mstep_tail_at_384_components(cuda, n):
    """resp_form 1 at its largest K: the tile flags, fp32 weights and tile sums lse_prep_kernel
    leaves behind give the M-step statistics of a resp_form-0 M-step on the normalised
    responsibilities, to 1e-12 (also with a partial last 64-frame tile)."""
    torch = cuda
    d, k = 24, 384
    x, w, m, cov = _model(d, k, n, n)
    gm, xd = _device_model(torch, x, w, m, cov)
    centres = gm._means[gm._cur].clone()
    gm._estep(torch, xd, for_mstep=True)
    gm._stats.zero_()
    gm._accumulate(torch, xd, centres)
    stats_log = gm._stats[:-2].clone()
    gm._normalize_resp(torch, xd)
    gm._stats.zero_()
    gm._accumulate(torch, xd, centres)
    stats_plain = gm._stats[:-2].clone()
    scale = stats_plain.abs().max().item()
    assert (stats_log - stats_plain).abs().max().item() <= 1e-12 * scale


def _mstep_cases():
    cases = [(d, 3 if d % 2 else 2, 700, d % 3 == 0, d % 4 == 1) for d in DIMS]
    cases += [
        (16, 2, 300, False, False),      # K m_chunks < 148: one tile per chunk
        (16, 2, 300, True, False),
        (16, 300, 2000, False, False),   # K m_chunks > 8 x 148
        (16, 300, 2000, True, False),
        (40, 5, 64 * 150 + 17, False, True),   # re-sorted frames, many tiles per chunk
        (144, 4, 64 * 60 + 3, True, True),
    ]
    return cases


@pytest.mark.parametrize('d,k,n,form1,reorder', _mstep_cases())
def test_mstep_statistics_within_bound(cuda, d, k, n, form1, reorder):
    """Every element of the statistics vector of kw_gmm_mstep_accumulate (precision 1) within
    mstats_bound of the FP64 statistics over the kept tiles.  resp_form 0 takes posteriors with
    widely mixed weights inside a tile and a last component below the tile floor (its statistics
    must be exactly 0); resp_form 1 takes the tensor-core E-step's own."""
    torch = cuda
    x, w, m, cov = _model(d, k, n, 7 * d + k + n)
    gm, xd = _device_model(torch, x, w, m, cov)
    rng = np.random.default_rng(d + n)
    centres = torch.from_numpy(m + 0.1 * rng.standard_normal(m.shape)).cuda()
    if form1:
        gm._estep(torch, xd, for_mstep=True)
        gm._stats.zero_()
        gm._accumulate(torch, xd, centres)
        gm._normalize_resp(torch, xd)           # the weights the M-step saw, for the reference
        resp = gm._resp[:, :n].t().cpu().numpy()
    else:
        resp = rng.dirichlet(np.full(k, 0.3), n)
        if k > 1:
            resp[:, -1] = 5e-9
        gm._resp[:, :n].copy_(torch.from_numpy(resp.T.copy()))
        if reorder:
            gm._reorder(torch, n, permute_resp=True)
            resp = gm._resp[:, :n].t().cpu().numpy()
            x = gm._x_used.cpu().numpy()
            assert not np.array_equal(x, xd.cpu().numpy())
        gm._stats.zero_()
        gm._accumulate(torch, xd, centres)
    got = gm._stats[:-2].view(k, -1).cpu().numpy()
    c = centres.cpu().numpy()
    ref = tc_bound.mstats_reference(x, resp, c)
    bound = tc_bound.mstats_bound(x, resp, c)
    err = np.abs(got - ref)
    ratio = np.where(err == 0, 0.0, err / np.where(bound > 0, bound, np.inf))
    print(f'D = {d} (DP {tc_bound.dp_of(d)}), K = {k}, N = {n}, resp_form {int(form1)}: '
          f'max |stats error| / bound = {ratio.max():.3g}')
    assert ratio.max() <= 1.0
    if not form1 and k > 1:
        assert np.all(got[-1] == 0.0)


@pytest.mark.parametrize('d', [3, 31, 47, 72, 113])
def test_fp64_mstep_statistics_per_tile_class(cuda, d):
    """gmm_mstats_kernel<TM> (precision 0) at each TM class (D <= 16, 32, 48, 80, 144): every
    element within 1e-12 of sum_n r |x_ni - c_i| |x_nj - c_j|."""
    torch = cuda
    k, n = 3, 1500
    x, w, m, cov = _model(d, k, n, d)
    resp = np.random.default_rng(d).dirichlet(np.full(k, 0.5), n)
    gm = GaussianMixture(n_components=k, precision='fp64')
    xd = torch.from_numpy(x).cuda()
    gm._alloc(torch, n, d, xd.device)
    gm._x_src, gm._x_used = xd, None
    gm._resp[:, :n].copy_(torch.from_numpy(resp.T.copy()))
    centres = torch.from_numpy(m).cuda()
    gm._stats.zero_()
    gm._accumulate(torch, xd, centres)
    got = gm._stats[:-2].view(k, -1).cpu().numpy()
    for j in range(k):
        r = np.where(resp[:, j] > 1e-16, resp[:, j], 0.0)
        u = x - m[j]
        au = np.abs(u)
        assert abs(got[j, 0] - r.sum()) <= 1e-12 * r.sum()
        assert np.all(np.abs(got[j, 1:1 + d] - r @ u) <= 1e-12 * (r @ au))
        scale = (au * r[:, None]).T @ au
        assert np.all(np.abs(got[j, 1 + d:].reshape(d, d) - (u * r[:, None]).T @ u) <=
                      1e-12 * scale)


# ------------------------------------------------------------------------------------------
# Three-way near-ties
# ------------------------------------------------------------------------------------------
def _tie_model(d, k, seed, m=3):
    """m components near the origin with different covariances; the other k - m far away."""
    rng = np.random.default_rng(seed)
    means = np.empty((k, d))
    covs = np.empty((k, d, d))
    means[:m] = rng.standard_normal((m, d)) * 0.6
    for c in range(m):
        a = rng.standard_normal((d, d)) * (0.4 / np.sqrt(d)) + np.eye(d) * (0.7 + 0.3 * c)
        covs[c] = a @ a.T
    far = rng.standard_normal((k - m, d))
    means[m:] = 40.0 * far / np.linalg.norm(far, axis=1, keepdims=True)
    covs[m:] = np.eye(d)
    w = rng.uniform(0.5, 1.5, k)
    return w / w.sum(), means, covs


def _tie_frames(w, means, covs, n, seed, m=3):
    """n frames at which components 0 .. m-1 have FP64 weighted log-probabilities within 1e-6
    nat of each other (the gaps to component 0 uniform in +-1e-6), solved by Newton on the slice
    x0 + sum_i s_i u_i (m - 1 directions).  Returns the frames that converged with every other
    component more than 0.05 nat below, and their FP64 weighted log-probabilities."""
    rng = np.random.default_rng(seed)
    d = means.shape[1]
    pc = gmm_ref.precision_cholesky(covs[:m])
    prec = np.einsum('kij,klj->kil', pc, pc)
    const = np.log(np.diagonal(pc, axis1=1, axis2=2)).sum(axis=1) + np.log(w[:m])
    mu_l = np.einsum('kd,kdj->kj', means[:m], pc)

    def fm(x):                         # (n, m) weighted log-probabilities of the m
        y = np.einsum('nd,kdj->nkj', x, pc) - mu_l
        return -0.5 * (y * y).sum(axis=2) + const

    x0 = means[:m].mean(axis=0) + 0.3 * rng.standard_normal((n, d))
    dirs = np.stack([(means[i] - means[0]) + 0.3 * rng.standard_normal((n, d))
                     for i in range(1, m)], axis=1)                      # (n, m-1, d)
    delta = rng.uniform(-1e-6, 1e-6, (n, m - 1))
    st = np.zeros((n, m - 1))
    for _ in range(40):
        x = x0 + np.einsum('ni,nid->nd', st, dirs)
        f = fm(x)
        r = (f[:, :1] - f[:, 1:]) - delta
        g = -np.einsum('kij,nkj->nki', prec, x[:, None, :] - means[None, :m])   # gradients
        jac = np.einsum('nid,njd->nij', g[:, :1] - g[:, 1:], dirs)
        step = np.linalg.solve(jac, r[:, :, None])[:, :, 0]
        st = st - np.clip(step, -1.0, 1.0)
    x = x0 + np.einsum('ni,nid->nd', st, dirs)
    wlp = gmm_ref.weighted_log_prob(x, w, means, gmm_ref.precision_cholesky(covs))
    gaps = wlp[:, :1] - wlp[:, 1:m]
    good = np.isfinite(wlp).all(axis=1) & (np.abs(gaps - delta) < 1e-9).all(axis=1)
    if means.shape[0] > m:
        good &= wlp[:, :m].max(axis=1) - wlp[:, m:].max(axis=1) > 0.05
    return x[good], wlp[good]


@pytest.mark.parametrize('d,k,m', [(72, 128, 3), (144, 3, 3), (72, 128, 4), (144, 5, 4)])
def test_hard_labels_on_near_ties(cuda, d, k, m):
    """Frames whose m best components lie within 1e-6 nat -- far below the tensor-core error,
    far above FP64 rounding: the labels of precision 1 must be the FP64 argmax (and those of
    precision 0 too).  Comparing only the best and the runner-up of the tensor cores leaves the
    FP64 best unchecked whenever the tensor cores ranked it third or lower."""
    torch = cuda
    w, means, covs = _tie_model(d, k, d + k, m)
    x, wlp = _tie_frames(w, means, covs, 4096, d, m)
    assert len(x) >= 3000
    gm, xd = _device_model(torch, x, w, means, covs)
    top = wlp.argmax(axis=1)
    assert set(np.unique(top)) == set(range(m))
    for precision in (1, 0):
        lab = _labels(torch, gm, xd, precision)
        wrong = int((lab != top).sum())
        assert wrong == 0, f'precision {precision}: {wrong} of {len(x)} labels are not the ' \
            'FP64 argmax'


def test_conversion_mixture_sequence_on_three_way_near_ties(cuda):
    """The same construction in the source marginal of a K = 128, Dh = 72 joint model: MLPG
    conversion with tensor-core labels takes the FP64 mixture sequence and gives the FP64
    output."""
    import torch
    from kwiiyatta_b200.mlpg import MLPG
    d, k = 72, 128
    w, mx, sxx = _tie_model(d, k, 11)
    x, wlp = _tie_frames(w, mx, sxx, 4096, 3)
    rng = np.random.default_rng(4)
    b = rng.standard_normal((d, d)) * (0.3 / np.sqrt(d))
    means = np.concatenate((mx, mx @ b.T + 0.1 * rng.standard_normal((k, d))), axis=1)
    covs = np.empty((k, 2 * d, 2 * d))
    for c in range(k):
        covs[c, :d, :d] = sxx[c]
        covs[c, :d, d:] = sxx[c] @ b.T
        covs[c, d:, :d] = b @ sxx[c]
        covs[c, d:, d:] = b @ sxx[c] @ b.T + 0.2 * np.eye(d)
    model = type('M', (), dict(weights_=w, means_=means, covariances_=covs,
                               covariance_type='full'))
    src = torch.from_numpy(x).cuda()
    n = len(x)
    off = torch.tensor([0, n // 3, 2 * n // 3, n], dtype=torch.int64).cuda()
    maxf = int((off[1:] - off[:-1]).max())
    out = {}
    for precision in ('fp64', 'tc'):
        y, mix = MLPG(model, precision=precision).transform_device(src, off, 3, maxf,
                                                                   return_mix=True)
        out[precision] = (y.cpu().numpy(), mix.cpu().numpy())
    assert np.array_equal(out['fp64'][1], wlp.argmax(axis=1))
    wrong = int((out['tc'][1] != out['fp64'][1]).sum())
    assert wrong == 0, f'{wrong} of {n} tensor-core mixture labels differ from FP64'
    assert np.abs(out['tc'][0] - out['fp64'][0]).max() <= 1e-8
