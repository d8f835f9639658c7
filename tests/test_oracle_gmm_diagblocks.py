"""CPU: the diagonal-blocks EM oracle (oracle/gmm_diagblocks_ref.py) against sklearn's full model
at D = 2 and against gmm_ref on the expanded matrices at any D."""
import numpy as np
import pytest

from oracle import gmm_diagblocks_ref as dbr, gmm_ref


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def _soft_resp(rng, n, k):
    r = rng.uniform(size=(n, k)) ** 4
    return r / r.sum(axis=1, keepdims=True)


@pytest.mark.parametrize('n,k,seed', [(600, 3, 0), (1500, 5, 1), (400, 1, 2)])
def test_one_pair_is_the_full_model(n, k, seed):
    """D = 2: the constrained model is the full model, so the oracle is sklearn's EM."""
    rng = np.random.default_rng(seed)
    x = dbr.paired_blobs(rng, n, 2, k)
    resp0 = gmm_ref.kmeans_like_resp(x, k, seed)
    ref = gmm_ref.sklearn_em(x, resp0, max_iter=40, tol=1e-6)
    got = dbr.numpy_em(x, resp0, max_iter=40, tol=1e-6)
    assert got['n_iter'] == ref['n_iter'] and got['converged'] == ref['converged']
    assert np.abs(np.array(got['lower_bounds']) - np.array(ref['lower_bounds'])).max() \
        <= 1e-12 * abs(ref['lower_bound'])
    for key in ('weights', 'means', 'covariances', 'precisions_cholesky'):
        assert _rel(got[key], ref[key]) <= 1e-12, key


@pytest.mark.parametrize('d,k', [(2, 2), (12, 4), (36, 3), (144, 2)])
def test_mstep_is_the_masked_full_mstep(d, k):
    rng = np.random.default_rng(d + k)
    x = dbr.paired_blobs(rng, 900, d, k)
    resp = _soft_resp(rng, 900, k)
    nk, means, cov = dbr.estimate_parameters(x, resp, 1e-6)
    nk_f, means_f, cov_f = gmm_ref.estimate_parameters(x, resp, 1e-6)
    assert _rel(nk, nk_f) <= 1e-12 and _rel(means, means_f) <= 1e-12
    full = dbr.expand(cov, True)
    assert _rel(full, np.where(dbr.pattern_mask(d), cov_f, 0.0)) <= 1e-12
    assert np.array_equal(dbr.compact(full), cov)


@pytest.mark.parametrize('d,k', [(2, 3), (12, 4), (144, 3)])
def test_estep_is_the_full_estep_on_the_expanded_model(d, k):
    rng = np.random.default_rng(7 * d + k)
    x = dbr.paired_blobs(rng, 700, d, k)
    weights, means, cov, fac = dbr.initialize(x, _soft_resp(rng, 700, k), 1e-6)
    got = dbr.weighted_log_prob(x, weights, means, fac)
    ref = gmm_ref.weighted_log_prob(x, weights, means, dbr.expand(fac, False))
    assert _rel(got, ref) <= 1e-12
    lb, log_resp = dbr.e_step(x, weights, means, fac)
    lb_f, log_resp_f = gmm_ref.e_step(x, weights, means, dbr.expand(fac, False))
    assert abs(lb - lb_f) <= 1e-12 * abs(lb_f)
    assert np.abs(np.exp(log_resp) - np.exp(log_resp_f)).max() <= 1e-12


@pytest.mark.parametrize('d', [2, 10, 144])
def test_precision_cholesky_is_sklearns_on_the_expanded_covariances(d):
    rng = np.random.default_rng(d)
    x = dbr.paired_blobs(rng, 500, d, 3)
    _, _, cov = dbr.estimate_parameters(x, _soft_resp(rng, 500, 3), 1e-6)
    fac = dbr.precision_cholesky(cov)
    got = dbr.expand(fac, False)
    ref = gmm_ref.precision_cholesky(dbr.expand(cov, True))
    assert _rel(got, ref) <= 1e-12
    upper = np.zeros((d, d), dtype=bool)
    upper[dbr.pair_indices(d)] = True
    assert np.all(np.triu(upper) == upper)
    assert np.array_equal(np.abs(ref) > 1e-13 * np.abs(ref).max(), np.broadcast_to(upper, ref.shape))


def test_precision_cholesky_rejects_a_singular_pair():
    cov = np.array([[[1.0, 1.0, 1.0], [2.0, 0.5, 1.0]]])
    with pytest.raises(ValueError, match='ill-defined'):
        dbr.precision_cholesky(cov)


def test_lower_bound_does_not_decrease():
    rng = np.random.default_rng(3)
    x = dbr.paired_blobs(rng, 3000, 16, 6)
    resp0 = gmm_ref.kmeans_like_resp(x, 6, 3)
    got = dbr.numpy_em(x, resp0, max_iter=20, tol=0.0)
    assert got['n_iter'] == 20
    assert np.all(np.diff(got['lower_bounds']) >= -1e-12 * abs(got['lower_bound']))
