"""CUDA posterior + MLPG and delta features vs the oracle."""
import numpy as np
import pytest

from kwiiyatta_b200 import delta as kdelta
from kwiiyatta_b200 import synth
from kwiiyatta_b200.mlpg import MLPG
from oracle import delta_ref, mlpg_ref

pytestmark = pytest.mark.gpu

TOL_ABS = 1e-4   # north_star: MLPG output within 1e-4 absolute on the mcep


class _Model:
    covariance_type = 'full'

    def __init__(self, w, m, c):
        self.weights_, self.means_, self.covariances_ = w, m, c


def _sources(n, frames):
    return [delta_ref.delta_features(s) for s in
            (synth.make_source_utterances(n, frames=frames))]


@pytest.mark.parametrize('diff', [False, True])
def test_transform_matches_oracle(cuda, diff):
    w, m, c = synth.make_joint_gmm(8, seed=1)
    src = _sources(2, 150)
    paramgen = MLPG(_Model(w, m, c), diff=diff)
    for s in src:
        exp, mix, _, _ = mlpg_ref.transform(s, w, m, c, diff=diff, return_internals=True)
        got = paramgen.transform(s)
        assert got.shape == exp.shape == (150, 24)
        assert np.abs(got - exp).max() <= 1e-8 < TOL_ABS


def test_mixture_sequence_and_batching(cuda):
    import torch
    w, m, c = synth.make_joint_gmm(16, seed=2)
    lens = [1, 2, 3, 17, 64, 65, 200]
    src = [delta_ref.delta_features(synth.make_source_utterances(1, frames=max(t, 2))[0][:t])
           for t in lens]
    paramgen = MLPG(_Model(w, m, c))
    outs = paramgen.transform_many(src)
    off = np.concatenate(([0], np.cumsum(lens)))
    _, mix = paramgen.transform_device(torch.from_numpy(np.concatenate(src)).cuda(),
                                       torch.from_numpy(off).cuda(), len(src), max(lens),
                                       return_mix=True)
    mix = mix.cpu().numpy()
    for i, s in enumerate(src):
        exp, emix, _, _ = mlpg_ref.transform(s, w, m, c, return_internals=True)
        assert np.array_equal(mix[off[i]:off[i + 1]], emix)
        assert np.abs(outs[i] - exp).max() <= 1e-8
    assert [len(o) for o in paramgen.transform_many([])] == []


def test_tensor_core_posterior_gives_the_same_mixture_sequence(cuda):
    """precision='tc': tcgen05 posterior + FP64 re-check of near-ties => identical hard labels,
    hence identical (FP64) MLPG output."""
    import torch
    w, m, c = synth.make_joint_gmm(32, seed=6)
    src = _sources(6, 300)
    paramgen = MLPG(_Model(w, m, c), precision='tc')
    lens = [len(s) for s in src]
    off = np.concatenate(([0], np.cumsum(lens)))
    out, mix = paramgen.transform_device(torch.from_numpy(np.concatenate(src)).cuda(),
                                         torch.from_numpy(off).cuda(), len(src), max(lens),
                                         return_mix=True)
    out, mix = out.cpu().numpy(), mix.cpu().numpy()
    for i, s in enumerate(src):
        exp, emix, _, _ = mlpg_ref.transform(s, w, m, c, return_internals=True)
        assert np.array_equal(mix[off[i]:off[i + 1]], emix)
        assert np.abs(out[off[i]:off[i + 1]] - exp).max() <= 1e-8


def test_dense_oracle_agrees(cuda):
    w, m, c = synth.make_joint_gmm(4, seed=3)
    s = _sources(1, 40)[0]
    exp = mlpg_ref.transform(s, w, m, c, banded=False)
    assert np.abs(MLPG(_Model(w, m, c)).transform(s) - exp).max() <= 1e-8


def test_delta_features_exact(cuda):
    rng = np.random.default_rng(0)
    for t in (1, 2, 3, 50, 333):
        x = rng.standard_normal((t, 24))
        assert np.array_equal(kdelta.delta_features(x), delta_ref.delta_features(x))


@pytest.mark.parametrize('diff', [False, True])
def test_soft_posterior_mapping_without_mlpg(cuda, diff):
    """mlpg=False (kwiiyatta/converter/gmm.py:30-31): windows[0:1] -> per-frame soft mapping."""
    w, m, c = synth.make_joint_gmm(6, dim_half=24, seed=8, static_dim=24)
    rng = np.random.default_rng(8)
    src = rng.standard_normal((77, 24)) * (1.0 / (1.0 + np.arange(24)))
    exp = mlpg_ref.transform_frames_soft(src, w, m, c, diff=diff)
    got = MLPG(_Model(w, m, c), windows=delta_ref.DELTA_WINDOWS[0:1], diff=diff).transform(src)
    assert got.shape == exp.shape == (77, 24)
    assert np.abs(got - exp).max() <= 1e-9


def test_errors(cuda):
    w, m, c = synth.make_joint_gmm(2, seed=4)
    paramgen = MLPG(_Model(w, m, c))
    with pytest.raises(ValueError):
        paramgen.transform(np.zeros((5, 71)))
    with pytest.raises(NotImplementedError):
        MLPG(_Model(w, m, c), windows=delta_ref.DELTA_WINDOWS[:2])
    with pytest.raises(ValueError):
        MLPG(_Model(w, m, c)).transform(np.zeros((5, 71)))


@pytest.mark.parametrize('precision', [0, 1])
@pytest.mark.parametrize('entry', ['kw_convert_batch', 'kw_convert_gv_batch'])
def test_rejected_call_enqueues_nothing(cuda, entry, precision):
    """dim_half 84 is past what the conditional-mean kernel holds (80) but within the E-step's
    limit (144): the call raises before it queues any work, so the workspace keeps its bytes."""
    from kwiiyatta_b200 import _lib
    torch = cuda
    k, dh, sd, total = 4, 84, 28, 40
    w, m, c = synth.make_joint_gmm(k, dim_half=dh, seed=5, static_dim=sd)
    paramgen = MLPG(_Model(w, m, c), precision=precision)
    x = torch.from_numpy(np.random.default_rng(5).standard_normal((total, dh))).cuda()
    off = torch.tensor([0, 15, total], dtype=torch.int64, device='cuda')
    out = torch.zeros((total, sd), dtype=torch.float64, device='cuda')
    ones = torch.ones(sd, dtype=torch.float64, device='cuda')
    nbytes = getattr(_lib.lib(), entry.replace('_batch', '_workspace_bytes'))(total, k, dh,
                                                                             precision)
    ws = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device='cuda')
    head = (2, off, total, 25, x, k, dh, paramgen._prepared)
    tail = (precision, ws, nbytes, _lib.stream_ptr(torch))
    args = {'kw_convert_batch': head + (out, None) + tail,
            'kw_convert_gv_batch': head + (ones, ones, 20, 1.0, 1.0, None, dh, out, None, None,
                                           None) + tail}[entry]
    with pytest.raises(ValueError, match='dim_half 84 > 80'):
        _lib.call(entry, *args)
    torch.cuda.synchronize()
    assert bool((ws == 0xA5).all())


def test_mc2b_hand_off_to_the_mlsa_filter(cuda):
    """pysptk.mc2b as called at kwiiyatta/filter/mlsa.py:23-29 (power coefficient zeroed first)."""
    import kwiiyatta_b200 as kw
    from oracle import mlsa_ref
    rng = np.random.default_rng(9)
    mceps = [rng.standard_normal((t, 25)) for t in (1, 7, 300)] + [np.zeros((0, 25))]
    got = kw.mc2b_many(mceps, alpha=0.41)
    for m, g in zip(mceps, got):
        zeroed = np.hstack((np.zeros((len(m), 1)), m[:, 1:]))
        assert np.array_equal(g, mlsa_ref.mc2b(zeroed, 0.41))
    assert np.array_equal(kw.mc2b(mceps[1], 0.55, zero_power=False),
                          mlsa_ref.mc2b(mceps[1], 0.55))


def test_converter_persistence_round_trip(cuda, tmp_path):
    """save_converter / load_converter: the reloaded chain converts identically (the reference
    keeps its model in memory only, kwiiyatta/convert_voice.py:15-20)."""
    import warnings
    import kwiiyatta_b200 as kw
    w, m, c = synth.make_joint_gmm(4, seed=8)
    conv = kw.MelCepstrumConverter(components=4, verbose=0)
    conv.base.base.gmm.set_parameters(w, m, c)
    conv.order, conv.fs, conv.base.frame_period = synth.ORDER, synth.FS, synth.FRAME_PERIOD
    path = str(tmp_path / 'model.npz')
    kw.save_converter(conv, path)
    again = kw.load_converter(path)
    assert (again.order, again.fs, again.frame_period) == (conv.order, conv.fs, conv.frame_period)
    assert np.array_equal(again.gmm.covariances_, c)
    mcep = synth.make_pair(4)[0].mel_cepstrum
    for kwargs in ({}, {'diff': True}, {'mlpg': False}):
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            assert np.array_equal(conv.convert(mcep, **kwargs).data,
                                  again.convert(mcep, **kwargs).data)


def test_pipelined_transform_packed_equals_single_shot(cuda):
    """transform_packed (chunks of utterances through copy-in / kernels / copy-out on three
    streams, from one pinned block to one pinned block) returns what one launch over the whole
    batch returns, and transform_many is the same thing from and to lists."""
    import torch
    w, m, c = synth.make_joint_gmm(8, seed=11)
    rng = np.random.default_rng(4)
    base = _sources(4, 400)
    src = [base[i % 4][:int(t)] + rng.normal(0, 0.01, (int(t), 72))
           for i, t in enumerate(rng.integers(1, 400, 60))]
    lens = [len(s) for s in src]
    off = np.concatenate(([0], np.cumsum(lens)))
    packed = torch.from_numpy(np.concatenate(src)).pin_memory()
    for precision in ('fp64', 'tc'):
        paramgen = MLPG(_Model(w, m, c), precision=precision)
        single = paramgen.transform_device(packed.cuda(), torch.from_numpy(off).cuda(), len(src),
                                           max(lens)).cpu().numpy()
        for chunk in (1500, 4000, 10 ** 9):
            paramgen.CHUNK_FRAMES = chunk
            out = paramgen.transform_packed(packed, lens)
            assert np.array_equal(out.numpy(), single)
            many = paramgen.transform_many(src)
            assert all(np.array_equal(many[i], single[off[i]:off[i + 1]])
                       for i in range(len(src)))
        # into a caller-provided pinned buffer, twice in a row (buffers and streams are reused)
        buf = torch.empty((int(off[-1]), 24), dtype=torch.float64).pin_memory()
        for _ in range(2):
            assert paramgen.transform_packed(packed, lens, out=buf) is buf
            assert np.array_equal(buf.numpy(), single)
    with pytest.raises(ValueError):
        paramgen.transform_packed(packed[:, :10], lens)
