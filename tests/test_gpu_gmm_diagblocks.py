"""The diagonal-blocks GMM (csrc/gmm_diagblocks.cu, GaussianMixture(covariance_type=
'diagonal_blocks')) against oracle/gmm_diagblocks_ref.py, and conversion from such a model."""
import os
import socket
import warnings

import numpy as np
import pytest

import kwiiyatta_b200 as kw
from kwiiyatta_b200 import _lib, synth
from kwiiyatta_b200.gmm import GaussianMixture
from kwiiyatta_b200.mlpg import MLPG
from oracle import delta_ref, gmm_diagblocks_ref as dbr, gmm_ref, mlpg_ref
from util import oracle_joint_array, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-9      # FP64 against FP64
DB = 'diagonal_blocks'


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _model(rng, k, d):
    dh = d // 2
    w = rng.dirichlet(np.ones(k) * 2.0)
    m = rng.standard_normal((k, d)) * 2.0
    sxx, syy = rng.uniform(0.5, 2.0, (k, dh)), rng.uniform(0.5, 2.0, (k, dh))
    rho = rng.uniform(-0.8, 0.8, (k, dh))
    return w, m, np.stack([sxx, rho * np.sqrt(sxx * syy), syy], axis=-1)


def _soft_resp(rng, n, k):
    r = rng.uniform(size=(n, k)) ** 4 + 1e-3
    r /= r.sum(axis=1, keepdims=True)
    drop = rng.uniform(size=(n, k)) < 0.2
    drop[0] = False                                  # every component keeps some weight
    r[drop] = 1e-18                                  # below the M-step's floor: skipped
    return r


@pytest.mark.parametrize('d', [2, 12, 144])
@pytest.mark.parametrize('k', [1, 4, 64])
@pytest.mark.parametrize('n', [1, 127, 128, 129, 50000])
def test_entries_match_oracle(cuda, n, k, d):
    """Each kw_gmm_db_* entry against the oracle, statistics around centres other than the
    means; two runs of every entry are bitwise equal."""
    torch = cuda
    lib = _lib.lib()
    st = _lib.stream_ptr(torch)
    rng = np.random.default_rng(n + 7 * k + d)
    x = dbr.paired_blobs(rng, n, d, max(k, 2))
    w, m, cov = _model(rng, k, d)
    xd, wd, md, cd = _dev(torch, x), _dev(torch, w), _dev(torch, m), _dev(torch, cov)
    fac = torch.empty((k, d // 2, 3), dtype=torch.float64, device='cuda')
    aux = torch.empty((k, 2), dtype=torch.float64, device='cuda')
    info = torch.full((k,), 7, dtype=torch.int32, device='cuda')
    nbytes = lib.kw_gmm_db_workspace_bytes(n, k, d)
    ws = _lib.workspace(nbytes, 'cuda')
    npad = lib.kw_gmm_resp_len(n, k) // k
    resp = torch.zeros((k, npad), dtype=torch.float64, device='cuda')
    stats = torch.zeros(lib.kw_gmm_db_stats_len(k, d), dtype=torch.float64, device='cuda')
    assert stats.numel() == k * (1 + d + 3 * (d // 2)) + 2
    lse = torch.zeros(n, dtype=torch.float64, device='cuda')

    # precision Cholesky of given covariances
    _lib.call('kw_gmm_db_precision_cholesky', k, d, wd, cd, fac, aux, info, st)
    ref_fac = dbr.precision_cholesky(cov)
    assert not info.cpu().numpy().any()
    assert rel_err(fac.cpu().numpy(), ref_fac) <= 1e-12
    ref_logdet = np.log(ref_fac[:, :, 0]).sum(1) + np.log(ref_fac[:, :, 2]).sum(1)
    assert np.abs(aux.cpu().numpy() - np.stack([ref_logdet, np.log(w)], 1)).max() \
        <= 1e-12 * max(1.0, np.abs(ref_logdet).max())

    # E-step
    def estep():
        _lib.call('kw_gmm_db_estep', n, xd, k, d, md, fac, aux, resp, stats, lse, ws, nbytes, st)
        return resp[:, :n].clone(), stats[-2:].clone(), lse.clone()
    r1, tail1, lse1 = estep()
    r2, tail2, lse2 = estep()
    assert torch.equal(r1, r2) and torch.equal(tail1, tail2) and torch.equal(lse1, lse2)
    lb, log_resp = dbr.e_step(x, w, m, ref_fac)
    ref_lse = dbr.weighted_log_prob(x, w, m, ref_fac)
    ref_lse = np.log(np.exp(ref_lse - ref_lse.max(1, keepdims=True)).sum(1)) + ref_lse.max(1)
    assert np.abs(r1.cpu().numpy().T - np.exp(log_resp)).max() <= TOL
    assert abs(tail1[0].item() - lb * n) <= TOL * abs(lb * n) and tail1[1].item() == n
    assert rel_err(lse1.cpu().numpy(), ref_lse) <= TOL

    # statistics around centres other than the means, on soft responsibilities
    rs = _soft_resp(rng, n, k)
    resp.zero_()
    resp[:, :n].copy_(_dev(torch, rs.T))
    centres = m + 0.3 * rng.standard_normal((k, d))
    cen = _dev(torch, centres)

    def accumulate():
        _lib.call('kw_gmm_db_mstep_accumulate', n, xd, k, d, resp, cen, stats, ws, nbytes, st)
        return stats.clone()
    s1 = accumulate()
    assert torch.equal(s1[:-2], accumulate()[:-2])
    kept = np.where(rs > 1e-16, rs, 0.0)
    dh = d // 2
    got = s1[:-2].view(k, -1).cpu().numpy()
    for j in range(k):
        u = x[:, :dh] - centres[j, :dh]
        v = x[:, dh:] - centres[j, dh:]
        r = kept[:, j:j + 1]
        ref = np.concatenate([[r.sum()], (r * (x - centres[j])).sum(0),
                              np.stack([(r * u * u).sum(0), (r * u * v).sum(0),
                                        (r * v * v).sum(0)], 1).ravel()])
        assert rel_err(got[j], ref) <= TOL, j

    # finalise from those statistics: the oracle's M-step on the kept responsibilities
    nk, ref_means, ref_cov = dbr.estimate_parameters(x, kept, 1e-6)
    means_out = torch.empty((k, d), dtype=torch.float64, device='cuda')
    cov_out = torch.empty((k, dh, 3), dtype=torch.float64, device='cuda')
    stats[-1] = float(n)
    for weight_norm, ref_w in ((0, nk / nk.sum()), (1, nk / n)):
        _lib.call('kw_gmm_db_mstep_finalize', k, d, 1e-6, weight_norm, stats, cen, wd, means_out,
                  cov_out, fac, aux, info, st)
        assert not info.cpu().numpy().any()
        assert rel_err(wd.cpu().numpy(), ref_w) <= TOL
        assert rel_err(means_out.cpu().numpy(), ref_means) <= TOL
        # the finaliser undoes the centring (S / n_k - delta^2, as the full model's does); that
        # form and the oracle's direct one differ by about u^2 10 eps / n_k, which shows when a
        # component holds only a fraction of one frame: bound on the scale of the second moments
        got_cov = cov_out.cpu().numpy()
        second = max(np.abs(got[j, 1 + d:]).max() / nk[j] for j in range(k))
        assert np.abs(got_cov - ref_cov).max() <= TOL * max(1.0, second)
        assert rel_err(fac.cpu().numpy(), dbr.precision_cholesky(got_cov)) <= 1e-12


def _fit_pair(x, resp0, **kw_args):
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        return GaussianMixture(n_components=resp0.shape[1], covariance_type=DB,
                               resp_init=resp0, **kw_args).fit(x)


def _compare(gm, ref):
    errs = {key: rel_err(getattr(gm, key + '_'), ref[key])
            for key in ('weights', 'means', 'covariances', 'precisions_cholesky')}
    errs['lower_bounds'] = float(np.abs(np.array(gm.lower_bounds_) - ref['lower_bounds']).max()
                                 / abs(ref['lower_bound']))
    print('worst relative differences', errs)
    assert max(errs.values()) <= TOL, errs


@pytest.mark.parametrize('n,d,k', [(3000, 12, 4), (2000, 2, 3), (4097, 144, 5), (257, 48, 1)])
def test_fit_matches_oracle(cuda, n, d, k):
    """Seeds whose initial responsibilities leave no component empty: an empty component keeps
    its centre as its mean here (as in the full model's finaliser), where sklearn's gives 0."""
    rng = np.random.default_rng(n + d + k + 1)
    x = dbr.paired_blobs(rng, n, d, k)
    resp0 = gmm_ref.kmeans_like_resp(x, k, 0)
    ref = dbr.numpy_em(x, resp0, max_iter=12, tol=0.0)
    gm = _fit_pair(x, resp0, max_iter=12, tol=0.0)
    assert gm.n_iter_ == 12 and gm.covariance_type == DB
    _compare(gm, ref)
    ref = dbr.numpy_em(x, resp0, max_iter=200, tol=1e-3)
    gm = _fit_pair(x, resp0, max_iter=200, tol=1e-3)
    assert gm.n_iter_ == ref['n_iter'] and gm.converged_ == ref['converged']
    _compare(gm, ref)


def test_kmeans_fit_on_the_corpus_is_monotone_and_repeats(cuda):
    x, _ = oracle_joint_array(4)
    fits = [_fit_one(x) for _ in range(2)]
    lbs = np.array(fits[0].lower_bounds_)
    assert len(lbs) >= 3
    assert np.all(np.diff(lbs) >= -1e-12 * np.abs(lbs).max())
    assert np.array_equal(lbs, np.array(fits[1].lower_bounds_))
    for key in ('weights_', 'means_', 'covariances_', 'precisions_cholesky_'):
        assert np.array_equal(getattr(fits[0], key), getattr(fits[1], key)), key
    mask = dbr.pattern_mask(x.shape[1])
    assert not fits[0].covariances_[:, ~mask].any()


def _fit_one(x):
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        return GaussianMixture(n_components=8, covariance_type=DB, random_state=0,
                               max_iter=30).fit(x)


def test_init_variants_run(cuda):
    rng = np.random.default_rng(4)
    x = dbr.paired_blobs(rng, 3000, 10, 4)
    resp0 = gmm_ref.kmeans_like_resp(x, 4, 1)
    base = _fit_pair(x, resp0, max_iter=3, tol=0.0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        rnd = GaussianMixture(n_components=4, covariance_type=DB, init_params='random_from_data',
                              random_state=1, max_iter=3).fit(x)
        over = GaussianMixture(n_components=4, covariance_type=DB, resp_init=resp0,
                               means_init=base.means_, weights_init=base.weights_,
                               max_iter=3, tol=0.0).fit(x)
    assert np.isfinite(rnd.lower_bound_) and np.isfinite(over.lower_bound_)
    # em_iteration / em_iteration_async step the same iteration as fit
    gm = GaussianMixture(n_components=4, covariance_type=DB, resp_init=resp0, max_iter=3)
    xd = gm.initialize(x)
    bounds = [gm.em_iteration(xd) for _ in range(2)]
    gm.em_iteration_async(xd)
    bounds.append(gm.last_lower_bound())
    assert np.abs(np.array(bounds) - np.array(base.lower_bounds_)).max() \
        <= 1e-12 * abs(base.lower_bound_)


def test_collapsed_component_raises(cuda):
    x = np.zeros((50, 4))
    x[:, 0] = np.arange(50)
    resp0 = np.zeros((50, 2))
    resp0[:25, 0] = 1
    resp0[25:, 1] = 1
    with pytest.raises(ValueError, match='ill-defined empirical covariance'):
        GaussianMixture(n_components=2, covariance_type=DB, reg_covar=0.0,
                        resp_init=resp0).fit(x)


def test_posteriors_match_oracle(cuda):
    rng = np.random.default_rng(6)
    x = dbr.paired_blobs(rng, 1000, 14, 4)
    ref = dbr.numpy_em(x, gmm_ref.kmeans_like_resp(x, 4, 1), max_iter=8)
    gm = GaussianMixture(n_components=4, covariance_type=DB).set_parameters(
        ref['weights'], ref['means'], ref['covariances'])
    assert np.array_equal(gm.covariances_, ref['covariances'])
    assert rel_err(gm.precisions_cholesky_, ref['precisions_cholesky']) <= 1e-12
    lb, log_resp = dbr.e_step(x, ref['weights'], ref['means'], ref['factors'])
    assert np.abs(gm.predict_proba(x) - np.exp(log_resp)).max() <= 1e-10
    assert abs(gm.score(x) - lb) <= 1e-10 * abs(lb)
    assert np.array_equal(gm.predict(x), log_resp.argmax(axis=1))


def test_set_parameters_rejects_entries_outside_the_pattern(cuda):
    rng = np.random.default_rng(8)
    w, m, cov = _model(rng, 3, 6)
    full = dbr.expand(cov, True)
    gm = GaussianMixture(n_components=3, covariance_type=DB).set_parameters(w, m, full)
    assert np.array_equal(gm.covariances_, full)
    bad = full.copy()
    bad[1, 0, 1] = bad[1, 1, 0] = 1e-3
    with pytest.raises(ValueError, match='outside the diagonal blocks'):
        GaussianMixture(n_components=3, covariance_type=DB).set_parameters(w, m, bad)
    with pytest.raises(ValueError, match='even dimension'):
        GaussianMixture(n_components=3, covariance_type=DB).set_parameters(
            w, m[:, :5], full[:, :5, :5])


def test_tensor_core_precision_is_rejected(cuda):
    with pytest.raises(ValueError, match='FP64 only'):
        GaussianMixture(covariance_type=DB, precision='tc')
    assert GaussianMixture(covariance_type=DB).precision == 0


@pytest.mark.parametrize('entry,bad', [
    ('estep', dict(d=5)), ('estep', dict(d=0)), ('estep', dict(d=146)), ('estep', dict(k=0)),
    ('estep', dict(n=-1)), ('estep', dict(null='x')), ('estep', dict(ws=-256)),
    ('mstep', dict(d=7)), ('mstep', dict(k=0)), ('mstep', dict(null='resp')),
    ('mstep', dict(ws=-256)),
    ('finalize', dict(reg=-1e-6)), ('finalize', dict(weight_norm=2)), ('finalize', dict(d=3)),
    ('finalize', dict(null='info')),
    ('cholesky', dict(d=148)), ('cholesky', dict(k=0)), ('cholesky', dict(null='factors')),
])
def test_rejected_call_enqueues_nothing(cuda, entry, bad):
    torch = cuda
    lib = _lib.lib()
    n, k, d = 1000, 3, 8
    bn, bk, bd = bad.get('n', n), bad.get('k', k), bad.get('d', d)
    dev = 'cuda'

    def pattern(count):
        return torch.full((count,), 0xA5, dtype=torch.uint8, device=dev)
    bufs = {'x': torch.from_numpy(np.random.default_rng(3).standard_normal((n, d))).cuda(),
            'means': torch.zeros((k, d), dtype=torch.float64, device=dev),
            'weights': torch.full((k,), 1.0 / k, dtype=torch.float64, device=dev),
            'cov': torch.ones((k, d // 2, 3), dtype=torch.float64, device=dev),
            'factors': pattern(8 * k * d * 3), 'aux': pattern(16 * k),
            'resp': pattern(8 * lib.kw_gmm_resp_len(n, k)),
            'stats': pattern(8 * lib.kw_gmm_db_stats_len(k, 160)), 'info': pattern(4 * k)}
    nbytes = lib.kw_gmm_db_workspace_bytes(n, k, d) + bad.get('ws', 0)
    bufs['ws'] = pattern(lib.kw_gmm_db_workspace_bytes(n, k, d))
    watched = [bufs[b] for b in ('factors', 'aux', 'resp', 'stats', 'info', 'ws')]
    if 'null' in bad:
        bufs[bad['null']] = None
    b, st = bufs, _lib.stream_ptr(torch)
    args = {'estep': ('kw_gmm_db_estep', bn, b['x'], bk, bd, b['means'], b['factors'], b['aux'],
                      b['resp'], b['stats'], None, b['ws'], nbytes, st),
            'mstep': ('kw_gmm_db_mstep_accumulate', bn, b['x'], bk, bd, b['resp'], b['means'],
                      b['stats'], b['ws'], nbytes, st),
            'finalize': ('kw_gmm_db_mstep_finalize', bk, bd, bad.get('reg', 1e-6),
                         bad.get('weight_norm', 0), b['stats'], b['means'], b['weights'],
                         b['means'], b['cov'], b['factors'], b['aux'], b['info'], st),
            'cholesky': ('kw_gmm_db_precision_cholesky', bk, bd, b['weights'], b['cov'],
                         b['factors'], b['aux'], b['info'], st)}[entry]
    exc = _lib.KwError if 'ws' in bad else ValueError
    with pytest.raises(exc, match='workspace too small' if 'ws' in bad else args[0]):
        _lib.call(*args)
    torch.cuda.synchronize()
    for buf in watched:
        assert bool((buf == 0xA5).all())


# ---- conversion from a diagonal-blocks model ------------------------------------------------

_TRAINED = {}


def _trained():
    if 'gm' not in _TRAINED:
        x, _ = oracle_joint_array(4)
        _TRAINED['gm'] = _fit_one(x)
    return _TRAINED['gm']


def test_conversion_from_a_diagonal_blocks_model(cuda):
    gm = _trained()
    feats = [delta_ref.delta_features(s) for s in synth.make_source_utterances(3, frames=300)]
    for diff in (False, True):
        diag = MLPG(gm, diff=diff).transform_many(feats)
        full = MLPG(gm, diff=diff, conditional_covariance='full').transform_many(feats)
        for a, b, f in zip(diag, full, feats):
            assert np.abs(a - b).max() <= 1e-10
            exp = mlpg_ref.transform(f, gm.weights_, gm.means_, gm.covariances_, diff=diff)
            assert np.abs(a - exp).max() <= 1e-4
    em = MLPG(gm, em_iter=2).transform(feats[0])
    gv = MLPG(gm, gv=(np.full(24, 0.1), np.full(24, 0.01))).transform(feats[0])
    assert em.shape == gv.shape == (len(feats[0]), 24)
    assert np.isfinite(em).all() and np.isfinite(gv).all()


@pytest.fixture()
def padded_hook():
    kw.hooks.bind(pad_silence=lambda f, n: f, feature=synth.feature, resample=synth.resample)
    yield
    kw.hooks.bind(pad_silence=None, feature=None, resample=None)


def test_converter_chain_keeps_its_type(cuda, padded_hook, tmp_path):
    src = {f'u{i}': synth.make_padded_pair(i)[0] for i in range(6)}
    tgt = {f'u{i}': synth.make_padded_pair(i)[1] for i in range(6)}
    keys = sorted(src)
    conv = kw.MelCepstrumConverter(components=4, verbose=0, max_iter=5, tol=0.0, random_state=0,
                                   covariance_type=DB)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        conv.train(kw.align(src, tgt), keys)
    assert conv.gmm.covariance_type == DB
    mcep = synth.make_pair(20)[0].mel_cepstrum
    out = conv.convert(mcep).data
    assert out.shape == mcep.data.shape and np.isfinite(out).all()
    path = str(tmp_path / 'db.npz')
    kw.save_converter(conv, path)
    again = kw.load_converter(path)
    assert again.gmm.covariance_type == DB
    assert np.array_equal(again.convert(mcep).data, out)
    backend = conv.base.base
    backend.save(str(tmp_path / 'b.npz'))
    loaded = kw.B200GMMFeatureConverter.load(str(tmp_path / 'b.npz'))
    assert loaded.gmm.covariance_type == DB
    with pytest.raises(ValueError, match='covariance_type'):
        kw.B200GMMFeatureConverter(components=4).load_state_dict(backend.state_dict())


# ---- two ranks ------------------------------------------------------------------------------

def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, x, resp0, out):
    import torch
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    cut = int(len(x) * 0.37)
    lo, hi = (0, cut) if rank == 0 else (cut, len(x))
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        gm = GaussianMixture(n_components=resp0.shape[1], covariance_type=DB, max_iter=5,
                             tol=0.0, resp_init=resp0[lo:hi],
                             device=torch.device('cuda', rank)).fit(x[lo:hi])
    out.put((rank, gm.weights_, gm.means_, gm.covariances_, gm.lower_bounds_))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_fit_equals_single(cuda):
    if cuda.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    rng = np.random.default_rng(3)
    x = dbr.paired_blobs(rng, 6000, 24, 4)
    resp0 = gmm_ref.kmeans_like_resp(x, 4, 0)
    single = _fit_pair(x, resp0, max_iter=5, tol=0.0)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, x, resp0, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=240) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, w, m, c, lbs in res:
        assert rel_err(w, single.weights_) <= 1e-10
        assert rel_err(m, single.means_) <= 1e-10
        assert rel_err(c, single.covariances_) <= 1e-10
        assert np.abs(np.array(lbs) - np.array(single.lower_bounds_)).max() <= 1e-8
    assert np.array_equal(res[0][2], res[1][2]) and np.array_equal(res[0][3], res[1][3])
