"""EM conversion over all mixture sequences (kw_convert_em_batch, MLPG(em_iter=)) on the device
vs oracle/mlpg_em_ref.py."""
import numpy as np
import pytest

import kwiiyatta_b200 as kw
from kwiiyatta_b200 import _lib, synth
from kwiiyatta_b200.mlpg import MLPG
from oracle import delta_ref, mlpg_em_ref

pytestmark = pytest.mark.gpu


class _Model:
    covariance_type = 'full'

    def __init__(self, w, m, c):
        self.weights_, self.means_, self.covariances_ = w, m, c


def _corpus():
    """Lengths 0, 1, 2, 150 and 1100."""
    base = [delta_ref.delta_features(s) for s in synth.make_source_utterances(3, frames=1100)]
    return [base[0][:0], base[1][:1], base[2][:2], base[1][:150], base[0]]


_ORACLE = {}


def _oracle(src, w, m, c, diff, em_iter):
    key = (diff, em_iter)
    if key not in _ORACLE:
        _ORACLE[key] = [mlpg_em_ref.convert(s, w, m, c, diff=diff, em_iter=em_iter) for s in src]
    return _ORACLE[key]


def _run(torch, paramgen, src):
    lens = [len(s) for s in src]
    off = np.concatenate(([0], np.cumsum(lens)))
    out, trace = paramgen.transform_device(
        torch.from_numpy(np.concatenate(src)).cuda(), torch.from_numpy(off).cuda(), len(src),
        max(lens), return_em_info=True)
    return out.cpu().numpy(), trace.cpu().numpy(), off


@pytest.mark.parametrize('precision', ['fp64', 'tc'])
@pytest.mark.parametrize('em_iter', [1, 5])
@pytest.mark.parametrize('diff', [False, True])
def test_convert_em_batch_matches_oracle(cuda, diff, em_iter, precision):
    torch = cuda
    w, m, c = synth.make_joint_gmm(8, seed=1)
    src = _corpus()
    paramgen = MLPG(_Model(w, m, c), diff=diff, precision=precision, em_iter=em_iter)
    out, trace, off = _run(torch, paramgen, src)
    assert trace.shape == (len(src), em_iter + 1)
    for i, (y, etrace) in enumerate(_oracle(src, w, m, c, diff, em_iter)):
        got = out[off[i]:off[i + 1]]
        err = np.abs(got - y).max(initial=0.0)
        terr = np.abs(trace[i] - etrace).max() / max(np.abs(etrace).max(), 1e-300)
        if precision == 'fp64':
            assert err <= 1e-9 * max(np.abs(y).max(initial=0.0), 1e-300) or len(y) == 0, (i, err)
            assert terr <= 1e-10, (i, terr)
            steps = np.diff(trace[i])
            assert np.all(steps >= -1e-12 * np.abs(trace[i]).max()), (i, steps)
        else:
            assert err <= 1e-4, (i, err)
            assert terr <= 1e-6, (i, terr)
    assert np.all(trace[0] == 0.0)                        # the empty utterance
    again, trace2, _ = _run(torch, paramgen, src)
    assert np.array_equal(again, out) and np.array_equal(trace2, trace)


def test_host_apis_match_device(cuda):
    torch = cuda
    w, m, c = synth.make_joint_gmm(8, seed=1)
    src = _corpus()
    lens = [len(s) for s in src]
    paramgen = MLPG(_Model(w, m, c), em_iter=3)
    out, _, off = _run(torch, paramgen, src)
    many = paramgen.transform_many(src)
    assert all(np.array_equal(many[i], out[off[i]:off[i + 1]]) for i in range(len(src)))
    assert np.array_equal(paramgen.transform(src[3]), out[off[3]:off[4]])
    paramgen.CHUNK_FRAMES = 100                            # several chunks of whole utterances
    packed = paramgen.transform_packed(torch.from_numpy(np.concatenate(src)), lens)
    assert np.array_equal(packed.numpy(), out)


def test_em_iter_zero_is_the_hard_path(cuda):
    w, m, c = synth.make_joint_gmm(8, seed=1)
    src = _corpus()
    for diff in (False, True):
        a = MLPG(_Model(w, m, c), diff=diff).transform_many(src)
        b = MLPG(_Model(w, m, c), diff=diff, em_iter=0).transform_many(src)
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_abi_rejects_bad_arguments(cuda):
    torch = cuda
    w, m, c = synth.make_joint_gmm(2, seed=1)
    paramgen = MLPG(_Model(w, m, c))
    x = torch.zeros((4, 72), dtype=torch.float64, device='cuda')
    off = torch.tensor([0, 4], dtype=torch.int64, device='cuda')
    out = torch.empty((4, 24), dtype=torch.float64, device='cuda')
    ws_bytes = _lib.lib().kw_convert_em_workspace_bytes(4, 2, 72, 0)
    ws = _lib.workspace(ws_bytes, x.device)
    stream = _lib.stream_ptr(torch)
    for em_iter, dh in ((0, 72), (-1, 72), (1, 71)):
        with pytest.raises(ValueError):
            _lib.call('kw_convert_em_batch', 1, off, 4, x, 2, dh, paramgen._prepared, em_iter,
                      out, None, 0, ws, ws_bytes, stream)


def test_converter_em_iter(cuda):
    w, m, c = synth.make_joint_gmm(4, seed=2)
    conv = kw.B200GMMFeatureConverter(components=4, verbose=0)
    conv.gmm.set_parameters(w, m, c)
    src = _corpus()[1:4]
    ref = MLPG(conv.gmm, em_iter=3)
    assert np.array_equal(conv.convert(src[2], em_iter=3), ref.transform(src[2]))
    many = conv.convert_many(src, em_iter=3)
    assert all(np.array_equal(a, b) for a, b in zip(many, ref.transform_many(src)))
    with pytest.raises(ValueError):
        conv.convert(src[2], em_iter=-1)
    with pytest.raises(ValueError):
        conv.convert(src[2][:, :24], mlpg=False, em_iter=3)
    conv.gv = (np.ones(24), np.ones(24))
    with pytest.raises(NotImplementedError):
        conv.convert(src[2], gv=True, em_iter=3)
    torch = cuda
    x = torch.from_numpy(src[2]).cuda()
    off = torch.tensor([0, len(src[2])], dtype=torch.int64, device='cuda')
    with pytest.raises(ValueError):
        ref.transform_device(x, off, 1, len(src[2]), return_mix=True)
    with pytest.raises(ValueError):
        MLPG(conv.gmm).transform_device(x, off, 1, len(src[2]), return_em_info=True)
