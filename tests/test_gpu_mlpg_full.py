"""MLPG with the full conditional covariance (kw_convert_fullcov_batch,
MLPG(conditional_covariance='full')) on the device vs oracle/mlpg_full_ref.py."""
import numpy as np
import pytest

import kwiiyatta_b200 as kw
from kwiiyatta_b200 import _lib, synth
from kwiiyatta_b200.delta import DELTA_WINDOWS
from kwiiyatta_b200.mlpg import MLPG
from oracle import delta_ref, mlpg_full_ref

pytestmark = pytest.mark.gpu

TOL_ABS = 1e-4   # the project's MLPG gate; both sides are FP64 direct solves


class _Model:
    covariance_type = 'full'

    def __init__(self, w, m, c):
        self.weights_, self.means_, self.covariances_ = w, m, c


def _corpus(order=24):
    """Lengths 0, 1, 2, 3, 150 and 2100."""
    base = [delta_ref.delta_features(s)
            for s in synth.make_source_utterances(3, frames=2100, order=order)]
    return [base[0][:0], base[1][:1], base[2][:2], base[0][:3], base[1][:150], base[2]]


def _diagonal_blocks(c):
    """Keep only the diagonals of the S_xx, S_xy, S_yx and S_yy blocks."""
    dh = c.shape[1] // 2
    out = np.zeros_like(c)
    idx = np.arange(dh)
    for r0 in (0, dh):
        for c0 in (0, dh):
            out[:, r0 + idx, c0 + idx] = c[:, r0 + idx, c0 + idx]
    return out


def _run(torch, paramgen, src, return_mix=False):
    lens = [len(s) for s in src]
    off = np.concatenate(([0], np.cumsum(lens)))
    res = paramgen.transform_device(torch.from_numpy(np.concatenate(src)).cuda(),
                                    torch.from_numpy(off).cuda(), len(src), max(lens),
                                    return_mix=return_mix)
    if return_mix:
        return res[0].cpu().numpy(), res[1].cpu().numpy(), off
    return res.cpu().numpy(), off


_ORACLE = {}


def _oracle(src, w, m, c, diff, key):
    if (key, diff) not in _ORACLE:
        cond = mlpg_full_ref.conditional_full(w, m, c, diff)
        _ORACLE[key, diff] = [mlpg_full_ref.transform(s, w, m, c, diff=diff, cond=cond)
                              for s in src]
    return _ORACLE[key, diff]


@pytest.mark.parametrize('precision', ['fp64', 'tc'])
@pytest.mark.parametrize('diff', [False, True])
@pytest.mark.parametrize('shape', ['dh72', 'dh30'])
def test_fullcov_matches_oracle(cuda, shape, diff, precision):
    """dh72: the configs[4] dimensions (static_dim 24, the exact instantiation of the block
    solve); dh30: static_dim 10 (the general one)."""
    torch = cuda
    if shape == 'dh72':
        w, m, c = synth.make_joint_gmm(8, seed=1)
        src = _corpus()
    else:
        w, m, c = synth.make_joint_gmm(6, dim_half=30, seed=2, static_dim=10)
        src = _corpus(order=10)
    paramgen = MLPG(_Model(w, m, c), diff=diff, precision=precision,
                    conditional_covariance='full')
    out, off = _run(torch, paramgen, src)
    errs = []
    for i, y in enumerate(_oracle(src, w, m, c, diff, shape)):
        got = out[off[i]:off[i + 1]]
        assert got.shape == y.shape
        errs.append(float(np.abs(got - y).max(initial=0.0)))
    print(f'fullcov {shape} diff={diff} {precision}: max |device - oracle| per utterance {errs}')
    assert max(errs) <= TOL_ABS, errs
    again, _ = _run(torch, paramgen, src)
    assert np.array_equal(again, out)


@pytest.mark.parametrize('precision', ['fp64', 'tc'])
@pytest.mark.parametrize('diff', [False, True])
def test_diagonal_block_model_equals_the_diagonal_path(cuda, diff, precision):
    torch = cuda
    w, m, c = synth.make_joint_gmm(8, seed=3)
    model = _Model(w, m, _diagonal_blocks(c))
    src = _corpus()
    full, mix_full, _ = _run(torch, MLPG(model, diff=diff, precision=precision,
                                         conditional_covariance='full'), src, return_mix=True)
    diag, mix_diag, _ = _run(torch, MLPG(model, diff=diff, precision=precision), src,
                             return_mix=True)
    assert np.abs(full - diag).max() <= 1e-9
    assert np.array_equal(mix_full, mix_diag)


def test_return_mix_is_the_diagonal_paths(cuda):
    torch = cuda
    w, m, c = synth.make_joint_gmm(8, seed=1)
    src = _corpus()
    _, mix_full, _ = _run(torch, MLPG(_Model(w, m, c), conditional_covariance='full'), src,
                          return_mix=True)
    _, mix_diag, _ = _run(torch, MLPG(_Model(w, m, c)), src, return_mix=True)
    assert np.array_equal(mix_full, mix_diag)


def test_host_apis_match_device(cuda):
    torch = cuda
    w, m, c = synth.make_joint_gmm(8, seed=1)
    src = _corpus()
    lens = [len(s) for s in src]
    paramgen = MLPG(_Model(w, m, c), conditional_covariance='full')
    out, off = _run(torch, paramgen, src)
    many = paramgen.transform_many(src)
    assert all(np.array_equal(many[i], out[off[i]:off[i + 1]]) for i in range(len(src)))
    assert np.array_equal(paramgen.transform(src[4]), out[off[4]:off[5]])
    paramgen.CHUNK_FRAMES = 100                            # several chunks of whole utterances
    packed = paramgen.transform_packed(torch.from_numpy(np.concatenate(src)), lens)
    assert np.array_equal(packed.numpy(), out)


def test_converter_conditional_covariance(cuda):
    w, m, c = synth.make_joint_gmm(4, seed=2)
    conv = kw.B200GMMFeatureConverter(components=4, verbose=0)
    conv.gmm.set_parameters(w, m, c)
    src = _corpus()[1:5]
    for diff in (False, True):
        ref = MLPG(conv.gmm, diff=diff, conditional_covariance='full')
        got = conv.convert(src[3], diff=diff, conditional_covariance='full')
        assert np.array_equal(got, ref.transform(src[3]))
        many = conv.convert_many(src, diff=diff, conditional_covariance='full')
        assert all(np.array_equal(a, b) for a, b in zip(many, ref.transform_many(src)))
        diag = conv.convert(src[3], diff=diff)
        assert np.array_equal(diag, MLPG(conv.gmm, diff=diff).transform(src[3]))
        assert not np.array_equal(diag, got)
    with pytest.raises(ValueError):
        conv.convert(src[3][:, :24], mlpg=False, conditional_covariance='full')


def test_error_cases(cuda):
    w, m, c = synth.make_joint_gmm(2, seed=1)
    model = _Model(w, m, c)
    with pytest.raises(ValueError):
        MLPG(model, conditional_covariance='dense')
    with pytest.raises(ValueError):
        MLPG(model, windows=DELTA_WINDOWS[0:1], conditional_covariance='full')
    with pytest.raises(NotImplementedError):
        MLPG(model, gv=(np.ones(24), np.ones(24)), conditional_covariance='full')
    with pytest.raises(NotImplementedError):
        MLPG(model, em_iter=2, conditional_covariance='full')
    bad = c.copy()
    dh = c.shape[1] // 2
    bad[1, dh:, dh:] = bad[1, dh:, :dh] @ np.linalg.solve(bad[1, :dh, :dh], bad[1, :dh, dh:])
    bad[1, dh:, dh:] -= 1e-3 * np.eye(dh)                  # S_yy - S_yx S_xx^-1 S_xy = -1e-3 I
    with pytest.raises(np.linalg.LinAlgError):
        MLPG(_Model(w, m, bad), conditional_covariance='full')


def _abi_args(torch, precision, k, dh, sd, total):
    w, m, c = synth.make_joint_gmm(k, dim_half=dh, seed=5, static_dim=sd)
    paramgen = MLPG(_Model(w, m, c), precision=precision)
    x = torch.from_numpy(np.random.default_rng(5).standard_normal((total, dh))).cuda()
    off = torch.tensor([0, 15, total], dtype=torch.int64, device='cuda')
    out = torch.zeros((total, sd), dtype=torch.float64, device='cuda')
    return paramgen, x, off, out


@pytest.mark.parametrize('precision', [0, 1])
def test_rejected_call_enqueues_nothing(cuda, precision):
    """dim_half 84 is past what the conditional-mean kernel holds (80): the call raises before
    it queues any work, so the workspace keeps its bytes."""
    torch = cuda
    k, dh, sd, total = 4, 84, 28, 40
    paramgen, x, off, out = _abi_args(torch, precision, k, dh, sd, total)
    fullcov = torch.zeros(16, dtype=torch.float64, device='cuda')
    nbytes = _lib.lib().kw_convert_fullcov_workspace_bytes(total, k, dh, precision)
    ws = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device='cuda')
    with pytest.raises(ValueError, match='dim_half 84 > 80'):
        _lib.call('kw_convert_fullcov_batch', 2, off, total, 25, x, k, dh, paramgen._prepared,
                  fullcov, out, None, precision, ws, nbytes, _lib.stream_ptr(torch))
    torch.cuda.synchronize()
    assert bool((ws == 0xA5).all())
    with pytest.raises(ValueError, match='dim_half 84 > 80'):
        _lib.call('kw_convert_fullcov_prepare', k, dh, 0, x, paramgen._prepared, fullcov, None,
                  ws, nbytes, _lib.stream_ptr(torch))


def test_small_workspace_is_reported(cuda):
    torch = cuda
    k, dh, sd, total = 4, 72, 24, 40
    w, m, c = synth.make_joint_gmm(k, seed=5)
    paramgen = MLPG(_Model(w, m, c), precision=0, conditional_covariance='full')
    x = torch.from_numpy(np.random.default_rng(5).standard_normal((total, dh))).cuda()
    off = torch.tensor([0, 15, total], dtype=torch.int64, device='cuda')
    out = torch.zeros((total, sd), dtype=torch.float64, device='cuda')
    nbytes = _lib.lib().kw_convert_fullcov_workspace_bytes(total, k, dh, 0)
    assert nbytes >= 8 * total * (3 * sd * sd + sd)
    ws = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device='cuda')
    with pytest.raises(_lib.KwError, match='workspace too small'):
        _lib.call('kw_convert_fullcov_batch', 2, off, total, 25, x, k, dh, paramgen._prepared,
                  paramgen._fullcov, out, None, 0, ws, nbytes - 1, _lib.stream_ptr(torch))
    torch.cuda.synchronize()
    assert bool((ws == 0xA5).all())
    pbytes = _lib.lib().kw_convert_fullcov_prepare_workspace_bytes(k, dh)
    assert pbytes >= 8 * 2 * k * dh * dh
    pws = _lib.workspace(pbytes, x.device)
    with pytest.raises(_lib.KwError, match='workspace too small'):
        _lib.call('kw_convert_fullcov_prepare', k, dh, 0, torch.from_numpy(c).cuda(),
                  paramgen._prepared, paramgen._fullcov, None, pws, pbytes - 1,
                  _lib.stream_ptr(torch))
