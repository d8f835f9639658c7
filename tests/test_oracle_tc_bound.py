"""oracle/tc_bound.py: the per-element error bounds of the tensor-core E-step and M-step hold for
a numpy emulation of what the kernels compute, and are tight enough that a kernel which loses the
lo operand on one pass, or the real columns of a partial last k-step, breaks them on most
elements.  That is what gives the device tests of tests/test_gpu_gmm_tc_kernels.py their meaning."""
import numpy as np
import pytest

from oracle import gmm_ref, tc_bound

# every DP class of the kernels and both sides of each 16-column boundary and of the switch from
# two components per MMA to one (DP 96 / 112)
DIMS = [1, 3, 15, 16, 17, 31, 32, 33, 47, 48, 63, 72, 80, 81, 95, 96, 97, 111, 112, 113, 127,
        128, 129, 143, 144]


def _model(d, k, n, seed):
    rng = np.random.default_rng(seed)
    centres = rng.standard_normal((k, d)) * 2.0
    a = rng.standard_normal((k, d, d)) * (0.3 / np.sqrt(max(d, 1) / 16.0)) + np.eye(d)
    cov = np.einsum('kij,klj->kil', a, a) + 0.05 * np.eye(d)
    lab = rng.integers(0, k, n)
    x = centres[lab] + np.einsum('nij,nj->ni', a[lab], rng.standard_normal((n, d)))
    w = rng.uniform(0.5, 1.5, k)
    return x, w / w.sum(), centres, cov


def _ratio(got, ref, bound):
    err = np.abs(got - ref)
    return np.where(err == 0, 0.0, err / np.where(bound > 0, bound, np.inf))


def _resp(n, k, seed):
    """Posteriors with widely mixed weights, and one component whose weights all lie below the
    M-step's tile floor."""
    rng = np.random.default_rng(seed)
    r = rng.dirichlet(np.full(k, 0.3), n)
    r[:, -1] = 5e-9 if k > 1 else r[:, -1]
    return r


def test_references_restate_the_oracle():
    x, w, m, cov = _model(20, 3, 300, 1)
    pc = gmm_ref.precision_cholesky(cov)
    _, wlp = tc_bound.estep_reference(x, w, m, pc)
    assert np.abs(wlp - gmm_ref.weighted_log_prob(x, w, m, pc)).max() <= 1e-10
    resp = np.random.default_rng(2).dirichlet(np.ones(3), 300)
    st = tc_bound.mstats_reference(x, resp, m)
    for k in range(3):
        u = x - m[k]
        assert np.allclose(st[k, 0], resp[:, k].sum(), rtol=1e-14)
        assert np.allclose(st[k, 1:21], resp[:, k] @ u, rtol=1e-12)
        assert np.allclose(st[k, 21:].reshape(20, 20), (u * resp[:, k, None]).T @ u, rtol=1e-12)


def test_tile_floor_and_chunking_follow_the_kernel():
    resp = np.zeros((64 * 5 + 3, 2))
    resp[:, 0] = 1.0
    resp[64:128, 1] = 5e-9
    resp[130, 1] = 2e-8
    keep = tc_bound.tile_mask(resp)
    assert keep[0].all()
    assert not keep[1, 64:128].any() and keep[1, 128:192].all() and not keep[1, :64].any()
    # tc_m_chunks: enough items for full waves of the 148 SMs
    assert tc_bound.m_chunks(1, 298) == 64
    assert tc_bound.m_chunks(64, 2000) * 64 >= 148
    assert tc_bound.m_chunks(384, 298) == 3


@pytest.mark.parametrize('d', DIMS)
def test_faithful_emulation_within_both_bounds(d):
    k = 3 if d % 2 else 2
    x, w, m, cov = _model(d, k, 129, d)
    pc = gmm_ref.precision_cholesky(cov)
    _, ref = tc_bound.estep_reference(x, w, m, pc)
    got, _ = tc_bound.emulate_estep(x, w, m, pc)
    ratio = _ratio(got, ref, tc_bound.estep_bound(x, w, m, pc))
    assert ratio.max() <= 1.0, ratio.max()
    xm, _, cm, _ = _model(d, k, 200, d + 1)
    resp = _resp(200, k, d)
    cen = cm + 0.05
    ref = tc_bound.mstats_reference(xm, resp, cen)
    got = tc_bound.emulate_mstats(xm, resp, cen)
    ratio = _ratio(got, ref, tc_bound.mstats_bound(xm, resp, cen))
    assert ratio.max() <= 1.0, ratio.max()
    if k > 1:
        assert np.all(got[-1] == 0.0) and np.all(ref[-1] == 0.0)     # below the floor


@pytest.mark.parametrize('d', [3, 17, 48, 72, 97, 144])
def test_dropping_the_lo_operand_on_one_pass_breaks_the_bounds(d):
    """Losing the lo half of one operand on one pass is a 2^-11 relative error per product: the
    E-step's weighted log-probabilities and the M-step's statistics then leave their bounds on
    most elements."""
    x, w, m, cov = _model(d, 3, 129, d)
    pc = gmm_ref.precision_cholesky(cov)
    _, ref = tc_bound.estep_reference(x, w, m, pc)
    bad, _ = tc_bound.emulate_estep(x, w, m, pc, defect='drop_lo_pass')
    broken = np.abs(bad - ref) > tc_bound.estep_bound(x, w, m, pc)
    print(f'D = {d}: E-step, lo dropped on one pass, {broken.mean():.0%} outside the bound')
    assert broken.mean() > 0.5
    xm, _, cm, _ = _model(d, 2, 700, d + 1)
    resp = np.random.default_rng(d).dirichlet(np.full(2, 0.3), 700)
    cen = cm + 0.05
    ref = tc_bound.mstats_reference(xm, resp, cen)
    bad = tc_bound.emulate_mstats(xm, resp, cen, defect='drop_lo_pass')
    broken = np.abs(bad - ref) > tc_bound.mstats_bound(xm, resp, cen)
    first, second = broken[:, 1:1 + d], broken[:, 1 + d:]
    print(f'D = {d}: M-step, lo dropped on one pass, {first.mean():.0%} of the first and '
          f'{second.mean():.0%} of the second moments outside the bound')
    assert first.mean() > 0.5 and second.mean() > 0.5


@pytest.mark.parametrize('d', [d for d in DIMS if d % 16 and d > 16])
def test_dropping_the_partial_last_kstep_breaks_the_estep_bound(d):
    x, w, m, cov = _model(d, 3, 129, d)
    pc = gmm_ref.precision_cholesky(cov)
    _, ref = tc_bound.estep_reference(x, w, m, pc)
    bad, _ = tc_bound.emulate_estep(x, w, m, pc, defect='drop_tail')
    broken = np.abs(bad - ref) > tc_bound.estep_bound(x, w, m, pc)
    assert broken.mean() > 0.9
