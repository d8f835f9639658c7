"""Global-variance statistics and GV-considered conversion on the device vs oracle/gv_ref.py."""
import os
import socket
import warnings

import numpy as np
import pytest

import kwiiyatta_b200 as kw
from kwiiyatta_b200 import synth
from kwiiyatta_b200.mlpg import MLPG
from oracle import delta_ref, gv_ref, mlpg_ref

pytestmark = pytest.mark.gpu


class _Model:
    covariance_type = 'full'

    def __init__(self, w, m, c):
        self.weights_, self.means_, self.covariances_ = w, m, c


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def test_gv_estimate_matches_oracle(cuda):
    torch = cuda
    rng = np.random.default_rng(0)
    lens = [5, 1, 0, 333, 40, 2, 1200]
    feats = [rng.normal(0.3 * i, 1 + 0.1 * i, (t, 30)) for i, t in enumerate(lens)]
    mean, var, _ = gv_ref.estimate_gv([f[:, 7:19] for f in feats])
    off = np.concatenate(([0], np.cumsum(lens)))
    x = torch.from_numpy(np.concatenate(feats)).cuda()
    for got in (kw.estimate_gv((x, off), columns=(7, 12)),
                kw.estimate_gv((x, torch.from_numpy(off).cuda()), columns=(7, 12)),
                kw.estimate_gv([f[:, 7:19] for f in feats])):
        assert _rel(got.mean, mean) <= 1e-12 and _rel(got.var, var) <= 1e-12
    # bitwise reproducible
    again = kw.estimate_gv((x, off), columns=(7, 12))
    assert np.array_equal(again.mean, got.mean) and np.array_equal(again.var, got.var)
    # a single utterance: sigma^2_v is the floor
    assert np.all(kw.estimate_gv(feats[:1]).var == gv_ref.VAR_FLOOR)


def _corpus():
    """Synthetic source utterances: T = 1 and 2, ordinary lengths, and one longer than the
    shared-memory staging limit (1024 frames) that the kernel iterates in global memory."""
    base = [delta_ref.delta_features(s) for s in synth.make_source_utterances(3, frames=1100)]
    return [base[0][:1], base[1][:2], base[2][:150], base[0], base[1][:333]]


_ORACLE = {}


def _oracle(src, w, m, c, diff):
    key = diff
    if key not in _ORACLE:
        _ORACLE[key] = [mlpg_ref.transform(s, w, m, c, diff=diff, return_internals=True)
                        for s in src]
    return _ORACLE[key]


def _stats(src, w, m, c):
    y0 = [r[0] for r in _oracle(src, w, m, c, False)]
    v = np.array([np.var(y, axis=0) for y in y0 if len(y) > 1])
    mu = 1.8 * v.mean(axis=0)
    return mu, (0.4 * mu) ** 2


@pytest.mark.parametrize('diff', [False, True])
@pytest.mark.parametrize('gv_iter', [0, 1, 20])
def test_convert_gv_batch_matches_oracle(cuda, diff, gv_iter):
    torch = cuda
    w, m, c = synth.make_joint_gmm(8, seed=1)
    src = _corpus()
    mu, var = _stats(src, w, m, c)
    lens = [len(s) for s in src]
    off = np.concatenate(([0], np.cumsum(lens)))
    paramgen = MLPG(_Model(w, m, c), diff=diff, gv=(mu, var), gv_iter=gv_iter)
    out, (f, acc) = paramgen.transform_device(
        torch.from_numpy(np.concatenate(src)).cuda(), torch.from_numpy(off).cuda(), len(src),
        max(lens), return_gv_info=True)
    out, f, acc = out.cpu().numpy(), f.cpu().numpy(), acc.cpu().numpy()
    for i, s in enumerate(src):
        _, _, e, dv = _oracle(src, w, m, c, diff)[i]
        y, ef, eacc = gv_ref.generate_utterance(e, dv, mu, var, gv_iter,
                                                source_static=s[:, :24] if diff else None)
        assert np.array_equal(acc[i], eacc), (i, acc[i], eacc)
        assert np.abs(f[i] - ef).max() <= 1e-10 * np.abs(ef).max()
        assert np.abs(out[off[i]:off[i + 1]] - y).max() <= 1e-8
        if gv_iter == 0 and len(s) >= 2:
            z = y + (s[:, :24] if diff else 0.0)
            assert np.abs(np.var(z, axis=0) - mu).max() <= 1e-10 * mu.max()
    # the host APIs give the same result as the device one
    many = paramgen.transform_many(src)
    assert all(np.array_equal(many[i], out[off[i]:off[i + 1]]) for i in range(len(src)))
    paramgen.CHUNK_FRAMES = 500
    packed = paramgen.transform_packed(torch.from_numpy(np.concatenate(src)), lens)
    assert np.array_equal(packed.numpy(), out)


def _train_chain(gv=True, n=8):
    src = {f'u{i}': synth.make_padded_pair(i)[0] for i in range(n)}
    tgt = {f'u{i}': synth.make_padded_pair(i)[1] for i in range(n)}
    keys = sorted(src)
    conv = kw.MelCepstrumConverter(components=4, verbose=0, max_iter=5, tol=0.0, random_state=0,
                                   gv=gv)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        conv.train(kw.align(src, tgt), keys)
    return conv, src, tgt, keys


@pytest.fixture()
def padded_hook():
    kw.hooks.bind(pad_silence=lambda f, n: f, feature=synth.feature, resample=synth.resample)
    yield
    kw.hooks.bind(pad_silence=None, feature=None, resample=None)


def test_converter_chain_with_gv(cuda, padded_hook, tmp_path):
    """MelCepstrumConverter(gv=True).train -> convert(..., gv=True) against the oracle: GV of
    the target statics of the training matrix per key, GV-considered MLPG, source c0."""
    from kwiiyatta_b200.dataset import _dataset_to_array_with_offsets
    conv, src, tgt, keys = _train_chain()
    x, off = _dataset_to_array_with_offsets(
        kw.DeltaFeatureDataset(kw.MelCepstrumDataset(kw.align(src, tgt))), keys)
    mean, var, _ = gv_ref.estimate_gv([x[off[i]:off[i + 1], 72:96] for i in range(len(keys))])
    gv = conv.base.base.gv
    assert _rel(gv.mean, mean) <= 1e-12 and _rel(gv.var, var) <= 1e-12
    g = conv.gmm
    tests = [synth.make_pair(20 + i)[0].mel_cepstrum for i in range(4)]
    v_gv, v_plain = [], []
    for diff in (False, True):
        for mcep in tests:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                got = conv.convert(mcep, diff=diff, gv=True).data
                plain = conv.convert(mcep, diff=diff).data
            s72 = delta_ref.delta_features(mcep.data[:, 1:])
            y, _, _ = gv_ref.transform(s72, g.weights_, g.means_, g.covariances_, mean, var,
                                       diff=diff)
            assert np.array_equal(got[:, 0], mcep.data[:, 0])
            assert np.abs(got[:, 1:] - y).max() <= 1e-8
            # gv=False is the plain conversion of the same model, bit for bit
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                assert np.array_equal(conv.convert(mcep, diff=diff, gv=False).data, plain)
            assert np.array_equal(plain[:, 1:], MLPG(g, diff=diff).transform(s72))
            heard = (lambda d: d + mcep.data[:, 1:]) if diff else (lambda d: d)
            v_gv.append(np.var(heard(got[:, 1:]), axis=0))
            v_plain.append(np.var(heard(plain[:, 1:]), axis=0))
    gap = lambda v: np.mean(np.abs(np.log(np.array(v) / mean)))   # noqa: E731
    assert gap(v_gv) < gap(v_plain)
    # save / load keeps the statistics; a file without them loads as before
    path = str(tmp_path / 'gv.npz')
    kw.save_converter(conv, path)
    again = kw.load_converter(path)
    assert np.array_equal(again.gv.mean, gv.mean) and np.array_equal(again.gv.var, gv.var)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        assert np.array_equal(again.convert(tests[0], gv=True).data,
                              conv.convert(tests[0], gv=True).data)
    backend = conv.base.base
    backend.save(str(tmp_path / 'b.npz'))
    assert np.array_equal(kw.B200GMMFeatureConverter.load(str(tmp_path / 'b.npz')).gv.var, gv.var)
    backend.gv = None
    kw.save_converter(conv, str(tmp_path / 'plain.npz'))
    plain = kw.load_converter(str(tmp_path / 'plain.npz'))
    assert plain.base.base.gv is None
    with pytest.raises(ValueError):
        plain.convert(tests[0], gv=True)


def test_gv_errors(cuda):
    w, m, c = synth.make_joint_gmm(2, seed=4)
    mu, var = np.full(24, 0.1), np.full(24, 0.01)
    with pytest.raises(ValueError):
        MLPG(_Model(w, m, c), gv=(mu[:5], var[:5]))
    with pytest.raises(ValueError):
        MLPG(_Model(w, m, c), gv=(mu, var), gv_weights=(0.0, 1.0))
    w1, m1, c1 = synth.make_joint_gmm(2, dim_half=24, seed=8, static_dim=24)
    with pytest.raises(ValueError):
        MLPG(_Model(w1, m1, c1), windows=delta_ref.DELTA_WINDOWS[0:1], gv=(mu, var))
    conv = kw.B200GMMFeatureConverter(components=2, verbose=0)
    conv.gmm.set_parameters(w, m, c)
    src = delta_ref.delta_features(synth.make_source_utterances(1, frames=30)[0])
    with pytest.raises(ValueError):
        conv.convert(src, gv=True)                      # no statistics
    conv.gv = {'mean': mu, 'var': var}
    assert conv.convert(src, gv=True).shape == (30, 24)
    with pytest.raises(ValueError):
        conv.convert(src, mlpg=False, gv=True)          # soft branch: not defined


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, feats, out):
    import torch
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    from kwiiyatta_b200.gv import estimate_gv
    gv = estimate_gv(feats[rank::world], device=torch.device('cuda', rank))
    out.put((rank, gv.mean, gv.var))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_gv_statistics(cuda):
    if cuda.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    rng = np.random.default_rng(5)
    feats = [rng.normal(0, 1 + 0.05 * i, (int(t), 24))
             for i, t in enumerate(rng.integers(50, 400, 21))]
    single = kw.estimate_gv(feats)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, feats, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=240) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert np.array_equal(res[0][1], res[1][1]) and np.array_equal(res[0][2], res[1][2])
    assert _rel(res[0][1], single.mean) <= 1e-12 and _rel(res[0][2], single.var) <= 1e-9
