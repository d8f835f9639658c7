"""Low-delay conversion (kw_convert_stream_*, MLPG.stream) on the device vs
oracle/mlpg_stream_ref.py and the offline conversion."""
import numpy as np
import pytest

from kwiiyatta_b200 import _lib, synth
from kwiiyatta_b200.converter import MelCepstrumConverter
from kwiiyatta_b200.mlpg import MLPG
from oracle import delta_ref, mlpg_stream_ref

pytestmark = pytest.mark.gpu

TOL_ORACLE = 1e-9
TOL_OFFLINE = 1e-12


class _Model:
    covariance_type = 'full'

    def __init__(self, w, m, c):
        self.weights_, self.means_, self.covariances_ = w, m, c


MODELS = {24: synth.make_joint_gmm(32, seed=3),
          10: synth.make_joint_gmm(16, dim_half=30, seed=4, static_dim=10)}


def _statics(n, frames, order, seed=0):
    return synth.make_source_utterances(n, frames=frames, order=order, seed0=1000 + seed)


def run_streams(stream, utts, starts, slots, device=False):
    """Runs utterance u (statics (T_u, sd)) in slot slots[u] from tick starts[u] on: one push per
    tick while it lasts, ended at tick starts[u] + T_u (after that tick's push).  Checks that every
    frame is emitted once, in order, and returns the outputs."""
    torch = _lib.require_cuda()
    outs = [np.full((len(s), s.shape[1]), np.nan) for s in utts]
    nxt = [0] * len(utts)
    last = max(st + len(u) for st, u in zip(starts, utts))
    for tick in range(last + 1):
        live = [u for u in range(len(utts)) if starts[u] <= tick < starts[u] + len(utts[u])]
        if live:
            frames = np.stack([utts[u][tick - starts[u]] for u in live])
            sl = [slots[u] for u in live]
            if device:
                o, idx = stream.push_device(sl, torch.from_numpy(frames).cuda())
                o, idx = o.cpu().numpy(), idx.cpu().numpy()
            else:
                o, idx = stream.push(sl, frames)
            for row, u in enumerate(live):
                if idx[row] >= 0:
                    assert idx[row] == nxt[u]
                    outs[u][idx[row]] = o[row]
                    nxt[u] += 1
                else:
                    assert not o[row].any()
        done = [u for u in range(len(utts)) if starts[u] + len(utts[u]) == tick]
        if done:
            for u, tail in zip(done, stream.end([slots[u] for u in done])):
                assert len(tail) == min(len(utts[u]), stream.delay + 1)
                assert nxt[u] + len(tail) == len(utts[u])
                outs[u][nxt[u]:] = tail
                nxt[u] = len(utts[u])
    assert all(not np.isnan(o).any() for o in outs)
    return outs


_INTERNALS = {}


def _oracle(sd, diff, utts, delay):
    w, m, c = MODELS[sd]
    res = []
    for s in utts:
        key = (sd, diff, s.tobytes())
        if key not in _INTERNALS:
            _INTERNALS[key] = mlpg_stream_ref.internals(s, w, m, c, diff)
        _, _, e, dv = _INTERNALS[key]
        res.append(mlpg_stream_ref.stream_prefix(e, dv, delay))
    return res


@pytest.mark.parametrize('sd', [24, 10])
@pytest.mark.parametrize('precision', ['fp64', 'tc'])
@pytest.mark.parametrize('diff', [False, True])
@pytest.mark.parametrize('delay', [0, 1, 5, 40])
def test_parity_with_oracle(cuda, sd, precision, diff, delay):
    """Several utterances of the lengths 1, 2, 3, L, L+1, L+2 and ~700 interleaved in one stream
    object, with staggered starts and slots idle on some calls."""
    lengths = sorted({1, 2, 3, delay, delay + 1, delay + 2, 700} - {0})
    base = _statics(2, 700, sd)
    utts = [base[i % 2][:t] for i, t in enumerate(lengths)]
    n_slots = len(utts) + 3
    slots = list(np.random.default_rng(delay).permutation(n_slots)[:len(utts)])
    starts = [3 * i for i in range(len(utts))]
    stream = MLPG(_Model(*MODELS[sd]), diff=diff, precision=precision).stream(n_slots, delay)
    got = run_streams(stream, utts, starts, slots, device=delay % 2 == 1)
    for g, e, s in zip(got, _oracle(sd, diff, utts, delay), utts):
        assert g.shape == (len(s), sd)
        assert np.abs(g - e).max() <= TOL_ORACLE, len(s)


@pytest.mark.parametrize('precision', ['fp64', 'tc'])
@pytest.mark.parametrize('diff', [False, True])
def test_long_delay_is_offline(cuda, precision, diff):
    utts = [s[:t] for s, t in zip(_statics(4, 300, 24, seed=1), (1, 2, 57, 300))]
    paramgen = MLPG(_Model(*MODELS[24]), diff=diff, precision=precision)
    exp = paramgen.transform_many([delta_ref.delta_features(s) for s in utts])
    for delay in (299, 310):
        got = run_streams(paramgen.stream(5, delay), utts, [0, 0, 4, 1], [4, 0, 2, 1])
        for g, e in zip(got, exp):
            assert np.abs(g - e).max() <= TOL_OFFLINE


def test_slot_lifecycle(cuda):
    paramgen = MLPG(_Model(*MODELS[24]))
    stream = paramgen.stream(3, 4)
    a, b = _statics(2, 40, 24, seed=2)
    assert [len(t) for t in stream.end([0, 2])] == [0, 0]       # ending empty slots
    first = run_streams(stream, [a, b[:9]], [0, 2], [1, 2])
    again = run_streams(stream, [b[:9], a], [0, 0], [1, 2])     # both slots reused
    assert np.abs(first[0] - again[1]).max() <= TOL_OFFLINE
    assert np.abs(first[1] - again[0]).max() <= TOL_OFFLINE
    assert [len(t) for t in stream.end([1, 2, 0])] == [0, 0, 0]
    exp = _oracle(24, False, [a, b[:9]], 4)
    assert np.abs(first[0] - exp[0]).max() <= TOL_ORACLE
    assert np.abs(first[1] - exp[1]).max() <= TOL_ORACLE


def test_converter(cuda):
    w, m, c = MODELS[24]
    chain = MelCepstrumConverter(components=32, verbose=0)
    backend = chain.base.base
    backend.gmm.set_parameters(w, m, c)
    utts = _statics(3, 60, 24, seed=3)
    for diff in (False, True):
        exp = run_streams(MLPG(backend.gmm, diff=diff, precision=backend.gmm.precision_request)
                          .stream(4, 6), utts, [0, 5, 9], [3, 1, 0])
        for conv in (backend, chain):
            got = run_streams(conv.stream(4, 6, diff=diff), utts, [0, 5, 9], [3, 1, 0])
            assert all(np.array_equal(g, e) for g, e in zip(got, exp))


def test_error_cases(cuda):
    model = _Model(*MODELS[24])
    stream = MLPG(model).stream(4, 2)
    with pytest.raises(ValueError):
        MLPG(model).stream(4, -1)
    with pytest.raises(ValueError):
        MLPG(model, windows=delta_ref.DELTA_WINDOWS[:1]).stream(4, 2)
    with pytest.raises(ValueError):
        MLPG(model, em_iter=1).stream(4, 2)
    with pytest.raises(ValueError):
        MLPG(model, conditional_covariance='full').stream(4, 2)
    with pytest.raises(ValueError):
        MLPG(model, gv=(np.ones(24), np.ones(24))).stream(4, 2)
    frames = np.zeros((2, 24))
    for slots in ([0, 0], [0, 4], [-1, 1]):
        with pytest.raises(ValueError):
            stream.push(slots, frames)
        with pytest.raises(ValueError):
            stream.end(slots)
    with pytest.raises(ValueError):
        stream.push([0, 1], np.zeros((2, 25)))
    with pytest.raises(ValueError):
        stream.push([0, 1, 2], frames)


@pytest.mark.parametrize('precision', [0, 1])
def test_rejected_call_changes_nothing(cuda, precision):
    """Every argument is checked before the first launch: a rejected push or end leaves the
    byte-patterned workspace and state as they were."""
    torch = _lib.require_cuda()
    lib = _lib.lib()
    w, m, c = MODELS[24]
    paramgen = MLPG(_Model(w, m, c), precision=precision)
    n_slots, delay, k, dh = 4, 3, 32, 72
    stream = paramgen.stream(n_slots, delay)
    state = stream._state.view(torch.uint8)
    state.fill_(0x5A)
    nbytes = lib.kw_convert_stream_workspace_bytes(n_slots, k, dh, delay, precision)
    ws = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device='cuda')
    x = torch.zeros((n_slots, 24), dtype=torch.float64, device='cuda')
    out = torch.zeros((n_slots, delay + 1, 24), dtype=torch.float64, device='cuda')
    idx = torch.zeros(n_slots, dtype=torch.int64, device='cuda')
    st = _lib.stream_ptr(torch)

    def push(slots, nsl=n_slots, dl=delay, m_=None, dh_=dh, prec=precision, wsb=nbytes):
        s = np.asarray(slots, dtype=np.int32)
        _lib.call('kw_convert_stream_push', nsl, dl, len(s) if m_ is None else m_, s, x, k, dh_,
                  paramgen._prepared, stream._state, out, idx, prec, ws, wsb, st)

    def end(slots, nsl=n_slots, dl=delay, m_=None, dh_=dh, prec=precision, wsb=nbytes):
        s = np.asarray(slots, dtype=np.int32)
        _lib.call('kw_convert_stream_end', nsl, dl, len(s) if m_ is None else m_, s, k, dh_,
                  paramgen._prepared, stream._state, out, idx, prec, ws, wsb, st)

    bad = [dict(slots=[0, 0]), dict(slots=[0, 4]), dict(slots=[-1]), dict(slots=[0], dl=-1),
           dict(slots=[0], dl=9000), dict(slots=[0, 1, 2, 3], nsl=3),
           dict(slots=[0, 1], m_=-1), dict(slots=[0], dh_=84), dict(slots=[0], dh_=71),
           dict(slots=[0], prec=2), dict(slots=[0], nsl=0)]
    for fn in (push, end):
        for kwargs in bad:
            with pytest.raises(ValueError):
                fn(**kwargs)
        with pytest.raises(_lib.KwError, match='workspace too small'):
            fn([0, 1], wsb=lib.kw_convert_stream_workspace_bytes(2, k, dh, delay, precision) - 1)
    torch.cuda.synchronize()
    assert bool((ws == 0xA5).all()) and bool((state == 0x5A).all())


def test_large_batch(cuda):
    """4096 streams of random lengths: all against offline with L >= T-1, a sample against the
    oracle at L = 20."""
    rng = np.random.default_rng(7)
    n = 4096
    lens = rng.integers(1, 161, n)
    pool = _statics(8, 160, 24, seed=5)
    utts = [pool[i % 8][rng.integers(0, 161 - t):][:t] for i, t in enumerate(lens)]
    starts = list(rng.integers(0, 40, n))
    slots = list(rng.permutation(n))
    paramgen = MLPG(_Model(*MODELS[24]))
    exp = paramgen.transform_many([delta_ref.delta_features(s) for s in utts])
    got = run_streams(paramgen.stream(n, int(lens.max()) - 1), utts, starts, slots, device=True)
    assert max(np.abs(g - e).max() for g, e in zip(got, exp)) <= TOL_OFFLINE
    got = run_streams(paramgen.stream(n, 20), utts, starts, slots, device=True)
    sample = rng.choice(n, 12, replace=False)
    for u, e in zip(sample, _oracle(24, False, [utts[u] for u in sample], 20)):
        assert np.abs(got[u] - e).max() <= TOL_ORACLE
