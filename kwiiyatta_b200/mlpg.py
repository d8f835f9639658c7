"""Posterior + MLPG on the B200 (nnmnkwii.baseline.gmm.MLPG as used at
kwiiyatta/converter/gmm.py:28-34), optionally with global variance (``gv=``; kwiiyatta_b200.gv),
maximum-likelihood conversion over all mixture sequences (``em_iter=``) or the full conditional
covariance (``conditional_covariance='full'``), and low-delay conversion of many concurrent streams
(``MLPG.stream``)."""
import numpy as np

from . import _lib
from .delta import DELTA_WINDOWS, check_windows


_on_own_device = _lib.device_guard(lambda self, *a: getattr(self, '_dev', None))


class MLPG:
    """``MLPG(gmm, windows, diff).transform(src)``.  ``gmm`` is anything with ``weights_``,
    ``means_`` and ``covariances_`` (our GaussianMixture or sklearn's).  The sliced model
    (marginal precision Cholesky, regression matrices, variance table) is prepared once
    here; the reference rebuilds it on every convert call (kwiiyatta/converter/gmm.py:32)."""

    def __init__(self, gmm, windows=None, swap=False, diff=False, precision='auto',
                 device=None, gv=None, gv_iter=20, gv_weights=(1.0, 1.0), em_iter=0,
                 conditional_covariance='diagonal'):
        torch = _lib.require_cuda()
        self._dev = torch.device('cuda' if device is None else device)
        with torch.cuda.device(self._dev):      # 'cuda' without an index: the current device
            self._setup(torch, gmm, windows, swap, diff, precision)
            self._setup_gv(torch, gv, gv_iter, gv_weights)
            self._setup_em(precision, em_iter)
            self._setup_fullcov(torch, gmm, conditional_covariance)

    def _setup_fullcov(self, torch, gmm, conditional_covariance):
        """``conditional_covariance='full'``: the ML trajectory under the full conditional
        covariance S_yy - A S_xy of each mixture (Toda, Black & Tokuda 2007), which couples the
        static dimensions, instead of nnmnkwii's element-wise diagonal (``'diagonal'``)."""
        if conditional_covariance not in ('diagonal', 'full'):
            raise ValueError("conditional_covariance must be 'diagonal' or 'full', got "
                             f'{conditional_covariance!r}')
        self.conditional_covariance = conditional_covariance
        self._fullcov = None
        if conditional_covariance == 'diagonal':
            return
        if len(self.windows) == 1:
            raise ValueError('the full conditional covariance is defined for MLPG trajectories '
                             'only (not with a single static window)')
        if self.gv is not None or self.em_iter:
            raise NotImplementedError("conditional_covariance='full' together with GV or EM "
                                      'conversion is not built')
        lib = _lib.lib()
        k, dh = self.num_mixtures, self.dim_half
        c = torch.from_numpy(np.ascontiguousarray(gmm.covariances_, dtype=np.float64)).to(self._dev)
        self._fullcov = torch.empty(lib.kw_convert_fullcov_prepared_len(k, dh),
                                    dtype=torch.float64, device=self._dev)
        info = torch.zeros(k, dtype=torch.int32, device=self._dev)
        ws_bytes = lib.kw_convert_fullcov_prepare_workspace_bytes(k, dh)
        _lib.call('kw_convert_fullcov_prepare', k, dh, int(self.diff), c, self._prepared,
                  self._fullcov, info, _lib.workspace(ws_bytes, self._dev), ws_bytes,
                  _lib.stream_ptr(torch))
        if info.cpu().numpy().any():
            raise np.linalg.LinAlgError('conditional covariance of some mixture is not positive '
                                        'definite')

    def _setup_em(self, precision, em_iter):
        """``em_iter > 0``: every transform runs ``em_iter`` EM iterations of maximum-likelihood
        conversion over all mixture sequences (Toda, Black & Tokuda 2007), started from the
        hard-sequence trajectory: E-step = posteriors of the joint model of [x_t ; (W y)_t],
        M-step = MLPG with per-frame precisions.  ``em_iter = 0`` is the hard-sequence path."""
        em_iter = int(em_iter)
        if em_iter < 0:
            raise ValueError(f'em_iter must be >= 0, got {em_iter}')
        if em_iter and len(self.windows) == 1:
            raise ValueError('EM conversion is defined for MLPG trajectories only (not with a '
                             'single static window)')
        if em_iter and self.gv is not None:
            raise NotImplementedError('EM conversion together with GV is not built')
        self.em_iter = em_iter
        # 'auto' = the FP64 E-step for EM: soft posteriors feel the tensor-core E-step's error
        # directly, with no FP64 re-check as the hard labels have (DESIGN.md, "Numerics")
        self._em_precision = 0 if precision == 'auto' else self.precision

    def _setup_gv(self, torch, gv, gv_iter, gv_weights):
        """``gv``: GV statistics (a kwiiyatta_b200.gv.GlobalVariance, a dict with ``mean`` /
        ``var`` or a (mean, var) pair, one value per static dimension) -> every transform
        generates the GV-considered trajectory: the ML trajectory scaled to the GV mean, then
        ``gv_iter`` ascent steps on w_traj * (trajectory log-likelihood) + w_gv * (GV
        log-likelihood), ``gv_weights = (w_traj, w_gv)``.  ``gv_iter = 0`` is the
        variance-scaling postfilter.  In diff mode the GV is that of source + output."""
        self.gv = None
        if gv is None:
            return
        from .gv import as_gv
        if len(self.windows) == 1:
            raise ValueError('GV is defined for MLPG trajectories only (not with a single '
                             'static window)')
        gv = as_gv(gv)
        if len(gv) != self.static_dim:
            raise ValueError(f'GV statistics have {len(gv)} dimensions, expected '
                             f'{self.static_dim}')
        w_traj, w_gv = (float(w) for w in gv_weights)
        if int(gv_iter) < 0 or not w_traj > 0 or not w_gv >= 0:
            raise ValueError('need gv_iter >= 0, w_traj > 0 and w_gv >= 0')
        self.gv, self.gv_iter, self.gv_weights = gv, int(gv_iter), (w_traj, w_gv)
        self._gv_mean = torch.from_numpy(gv.mean).to(self._dev)
        self._gv_var = torch.from_numpy(gv.var).to(self._dev)

    def _setup(self, torch, gmm, windows, swap, diff, precision):
        if windows is None:
            windows = DELTA_WINDOWS
        if len(windows) > 1:
            check_windows(windows)
        elif not (windows[0][0] == 0 and windows[0][1] == 0 and
                  np.array_equal(windows[0][2], [1.0])):
            raise NotImplementedError('a single window must be the static window (0, 0, [1.0])')
        if swap:
            raise NotImplementedError('swap=True is not built')
        # a diagonal-blocks model publishes its expanded (K, D, D) covariances: the kernels of the
        # full model convert it unchanged
        if getattr(gmm, 'covariance_type', 'full') not in ('full', 'diagonal_blocks'):
            raise AssertionError("covariance_type must be 'full' or 'diagonal_blocks'")
        self.windows = windows
        self.diff = bool(diff)
        dev = self._dev
        means = np.ascontiguousarray(gmm.means_, dtype=np.float64)
        self.num_mixtures, d = means.shape
        self.dim_half = d // 2
        self.static_dim = d // 2 // len(windows)
        # 'auto' = the tcgen05 posterior whenever the kernels hold the frame width: its hard
        # labels are re-checked in FP64 where the best mixtures are close, so the mixture
        # sequence and the (FP64) MLPG output are those of the FP64 path
        self.precision = {'fp64': 0, 'tc': 1, 0: 0, 1: 1,
                          'auto': 1 if self.dim_half <= 144 else 0}[precision]
        lib = _lib.lib()
        k, dh = self.num_mixtures, self.dim_half
        w = torch.from_numpy(np.ascontiguousarray(gmm.weights_, dtype=np.float64)).to(dev)
        m = torch.from_numpy(means).to(dev)
        c = torch.from_numpy(np.ascontiguousarray(gmm.covariances_, dtype=np.float64)).to(dev)
        self._prepared = torch.empty(lib.kw_convert_prepared_len(k, dh), dtype=torch.float64,
                                     device=dev)
        info = torch.zeros(k, dtype=torch.int32, device=dev)
        _lib.call('kw_convert_prepare', k, dh, int(self.diff), w, m, c, self._prepared, info,
                  _lib.stream_ptr(torch))
        if info.cpu().numpy().any():
            raise np.linalg.LinAlgError('source covariance of some mixture is not positive '
                                        'definite')

    def _launch(self, n_utts, off_dev, total, max_frames, src, out, mix, stream,
                gv_f=None, gv_accepted=None, em_loglik=None):
        """kw_convert_batch, kw_convert_gv_batch when GV statistics are set,
        kw_convert_em_batch when ``em_iter > 0``, or kw_convert_fullcov_batch with the full
        conditional covariance, on device tensors (``src`` (total, dim_half), ``out`` (total,
        static_dim))."""
        lib = _lib.lib()
        k, dh = self.num_mixtures, self.dim_half
        if self._fullcov is not None:
            ws_bytes = lib.kw_convert_fullcov_workspace_bytes(total, k, dh, self.precision)
            _lib.call('kw_convert_fullcov_batch', n_utts, off_dev, total, int(max_frames), src, k,
                      dh, self._prepared, self._fullcov, out, mix, self.precision,
                      _lib.workspace(ws_bytes, src.device), ws_bytes, stream)
            return
        if self.em_iter:
            ws_bytes = lib.kw_convert_em_workspace_bytes(total, k, dh, self._em_precision)
            _lib.call('kw_convert_em_batch', n_utts, off_dev, total, src, k, dh, self._prepared,
                      self.em_iter, out, em_loglik, self._em_precision,
                      _lib.workspace(ws_bytes, src.device), ws_bytes, stream)
            return
        if self.gv is None:
            ws_bytes = lib.kw_convert_workspace_bytes(total, k, dh, self.precision)
            _lib.call('kw_convert_batch', n_utts, off_dev, total, int(max_frames), src, k, dh,
                      self._prepared, out, mix, self.precision,
                      _lib.workspace(ws_bytes, src.device), ws_bytes, stream)
            return
        ws_bytes = lib.kw_convert_gv_workspace_bytes(total, k, dh, self.precision)
        _lib.call('kw_convert_gv_batch', n_utts, off_dev, total, int(max_frames), src, k, dh,
                  self._prepared, self._gv_mean, self._gv_var, self.gv_iter, self.gv_weights[0],
                  self.gv_weights[1], src if self.diff else None, dh, out, mix, gv_f,
                  gv_accepted, self.precision, _lib.workspace(ws_bytes, src.device), ws_bytes,
                  stream)

    @_on_own_device
    def transform_device(self, src_dev, offsets_dev, n_utts, max_frames, return_mix=False,
                         return_gv_info=False, return_em_info=False):
        """src_dev (sum T, dim_half) float64 CUDA tensor, offsets int64 (n_utts + 1).
        ``return_gv_info`` (with GV): also the final objective F and the number of accepted
        ascent steps per (utterance, static dim), as (n_utts, static_dim) tensors.
        ``return_em_info`` (with ``em_iter > 0``): also the (n_utts, em_iter + 1) trace of the
        objective L(y_k), k = 0 (the hard-sequence start) .. em_iter."""
        torch = _lib.require_cuda()
        if return_mix and self.em_iter:
            raise ValueError('return_mix: EM conversion has no single mixture sequence')
        if return_em_info and not self.em_iter:
            raise ValueError('return_em_info needs em_iter > 0')
        total = src_dev.shape[0]
        dev = src_dev.device
        out = torch.empty((total, self.static_dim), dtype=torch.float64, device=dev)
        mix = torch.empty(total, dtype=torch.int32, device=dev) if return_mix else None
        info = None
        if return_gv_info:
            if self.gv is None:
                raise ValueError('return_gv_info needs GV statistics')
            info = (torch.zeros((n_utts, self.static_dim), dtype=torch.float64, device=dev),
                    torch.zeros((n_utts, self.static_dim), dtype=torch.int32, device=dev))
        loglik = (torch.zeros((n_utts, self.em_iter + 1), dtype=torch.float64, device=dev)
                  if return_em_info else None)
        self._launch(n_utts, offsets_dev, total, max_frames, src_dev, out, mix,
                     _lib.stream_ptr(torch), *(info or (None, None)), em_loglik=loglik)
        res = (out,) + ((mix,) if return_mix else ()) + ((info,) if return_gv_info else ()) + \
            ((loglik,) if return_em_info else ())
        return res if len(res) > 1 else out

    CHUNK_FRAMES = 65536       # frames per pipeline chunk (36 MB in, 12 MB out at Dh = 72)

    @_on_own_device
    def transform_many(self, features):
        """Batched ``transform`` from a list of host arrays to a list of host arrays: one
        multi-threaded gather into pinned memory, ``transform_packed``, one scatter.  (With
        separate pageable arrays on both sides the host copies bound this call; callers that
        keep their frames in one pinned block use ``transform_packed`` directly.)"""
        torch = _lib.require_cuda()
        feats = [np.ascontiguousarray(f, dtype=np.float64) for f in features]
        for f in feats:
            if f.ndim != 2 or f.shape[1] != self.dim_half:
                raise ValueError(f'expected (T, {self.dim_half}) features, got {f.shape}')
        lens = np.array([len(f) for f in feats], dtype=np.int64)
        total = int(lens.sum())
        if total == 0:
            return [np.zeros((0, self.static_dim)) for _ in feats]
        off = np.concatenate(([0], np.cumsum(lens)))
        hin = _lib.pinned('mlpg_in', self._dev, (total, self.dim_half), torch.float64)
        hout = _lib.pinned('mlpg_out', self._dev, (total, self.static_dim), torch.float64)
        host = hin.numpy()
        _lib.parallel_copy([(host[off[i]:off[i + 1]], feats[i]) for i in range(len(feats))])
        self.transform_packed(hin, lens, out=hout)
        res = hout.numpy()
        outputs = [np.empty((int(t), self.static_dim)) for t in lens]
        _lib.parallel_copy([(outputs[i], res[off[i]:off[i + 1]]) for i in range(len(feats))])
        return outputs

    @_on_own_device
    def transform_packed(self, src, lens, out=None):
        """Conversion of utterances packed row-wise in ONE host tensor ``src`` (sum T, dim_half)
        float64 -- pinned memory for full speed -- with lengths ``lens``; returns (and, when
        given, fills) the host tensor ``out`` (sum T, static_dim).  Runs as a three-stage
        pipeline over chunks of whole utterances: while the kernels of chunk i run, chunk i + 1
        is copied up and the result of chunk i - 1 is copied down (a copy-in and a copy-out
        stream beside the compute stream, two device buffers per direction); synchronised on
        return."""
        torch = _lib.require_cuda()
        dev, dh, sd = self._dev, self.dim_half, self.static_dim
        lens = np.asarray(lens, dtype=np.int64)
        total = int(lens.sum())
        if tuple(src.shape) != (total, dh) or src.dtype != torch.float64 or src.is_cuda:
            raise ValueError(f'src must be a host float64 tensor of shape ({total}, {dh})')
        if out is None:
            out = torch.empty((total, sd), dtype=torch.float64).pin_memory()
        elif tuple(out.shape) != (total, sd) or out.dtype != torch.float64 or out.is_cuda:
            raise ValueError(f'out must be a host float64 tensor of shape ({total}, {sd})')
        if total == 0:
            return out
        rows = np.concatenate(([0], np.cumsum(lens)))
        chunks, lo, acc = [], 0, 0
        for i, t in enumerate(lens):
            acc += int(t)
            if acc >= self.CHUNK_FRAMES or i == len(lens) - 1:
                chunks.append((lo, i + 1))
                lo, acc = i + 1, 0
        cap = max(int(rows[b] - rows[a]) for a, b in chunks)
        bufs = _lib.staging(('mlpg_pipe', dh, sd), dev)
        if bufs.get('cap', 0) < cap:
            bufs.update(cap=cap,
                        din=[torch.empty((cap, dh), dtype=torch.float64, device=dev)
                             for _ in range(2)],
                        dout=[torch.empty((cap, sd), dtype=torch.float64, device=dev)
                              for _ in range(2)],
                        streams=(torch.cuda.Stream(dev), torch.cuda.Stream(dev)))
        s_in, s_out = bufs['streams']
        compute = torch.cuda.current_stream(dev)
        start = torch.cuda.Event()
        start.record(compute)
        s_in.wait_event(start)            # buffers may still be in use by the previous call
        s_out.wait_event(start)
        ev_comp, ev_d2h = {}, {}
        keep = []
        for c, (a, b) in enumerate(chunks):
            r0, r1 = int(rows[a]), int(rows[b])
            n_c = r1 - r0
            off = rows[a:b + 1] - r0
            with torch.cuda.stream(s_in):
                if c >= 2:
                    s_in.wait_event(ev_comp[c - 2])      # device input buffer consumed
                bufs['din'][c & 1][:n_c].copy_(src[r0:r1], non_blocking=True)
                off_dev = torch.from_numpy(off).to(dev, non_blocking=True)
                ev_in = torch.cuda.Event()
                ev_in.record(s_in)
            compute.wait_event(ev_in)
            if c >= 2:
                compute.wait_event(ev_d2h[c - 2])        # device output buffer copied down
            chunk_in, chunk_out = bufs['din'][c & 1][:n_c], bufs['dout'][c & 1][:n_c]
            self._launch(b - a, off_dev, n_c, int(lens[a:b].max()), chunk_in, chunk_out,
                         None, compute.cuda_stream)
            off_dev.record_stream(compute)
            keep.append(off)
            ev_comp[c] = torch.cuda.Event()
            ev_comp[c].record(compute)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_comp[c])
                out[r0:r1].copy_(chunk_out, non_blocking=True)
                ev_d2h[c] = torch.cuda.Event()
                ev_d2h[c].record(s_out)
        ev_d2h[len(chunks) - 1].synchronize()
        compute.wait_event(ev_d2h[len(chunks) - 1])
        return out

    @_on_own_device
    def transform_soft(self, src):
        """MLPGBase.transform: per-frame soft-posterior conditional mean, (T, dim_half)."""
        torch = _lib.require_cuda()
        src = np.ascontiguousarray(src, dtype=np.float64)
        if src.ndim != 2 or src.shape[1] != self.dim_half:
            raise ValueError(f'expected (T, {self.dim_half}) features, got {src.shape}')
        total = len(src)
        if total == 0:
            return np.zeros((0, self.dim_half))
        x = torch.from_numpy(src).to(self._dev)
        out = torch.empty((total, self.dim_half), dtype=torch.float64, device=self._dev)
        ws_bytes = _lib.lib().kw_convert_soft_workspace_bytes(total, self.num_mixtures,
                                                              self.dim_half)
        _lib.call('kw_convert_soft_batch', total, x, self.num_mixtures, self.dim_half,
                  self._prepared, out, _lib.workspace(ws_bytes, self._dev), ws_bytes,
                  _lib.stream_ptr(torch))
        return out.cpu().numpy()

    def stream(self, n_slots, delay):
        """Low-delay conversion of up to ``n_slots`` concurrent streams (``MLPGStream``): the frame
        emitted for static frame ``j`` of a stream is frame ``j - 1 - delay`` of the MLPG solution
        of the frames known so far (fixed-lag MLPG, Muramatsu et al., Interspeech 2008), so a
        frame comes out ``delay + 1`` frames after its static went in.  With
        ``delay >= T - 1`` a stream of ``T`` frames gets exactly ``transform``'s output."""
        if self.gv is not None or self.em_iter or self._fullcov is not None:
            raise ValueError('low-delay conversion is built for the hard-sequence MLPG with the '
                             'diagonal conditional covariance only (no GV, EM or full covariance)')
        if len(self.windows) == 1:
            raise ValueError('low-delay conversion is defined for MLPG trajectories only (not '
                             'with a single static window)')
        return MLPGStream(self, n_slots, delay)

    def transform(self, src):
        src = np.asarray(src, dtype=np.float64)
        if src.ndim != 2:
            raise ValueError('MLPG.transform expects a (T, dim) array')
        if src.shape[1] == self.static_dim:
            # nnmnkwii: feature_dim == static_dim -> MLPGBase.transform (no trajectory smoothing)
            return self.transform_soft(src)
        return self.transform_many([src])[0]


class MLPGStream:
    """Low-delay conversion state of ``n_slots`` streams on an ``MLPG``'s device
    (kw_convert_stream_*).  Each call delivers one static frame (``static_dim`` values: the
    mel-cepstrum without c0) to each of a set of distinct slots; a slot holds one stream from its
    first ``push`` to its ``end``."""

    def __init__(self, mlpg, n_slots, delay):
        torch = _lib.require_cuda()
        self.mlpg, self.n_slots, self.delay = mlpg, int(n_slots), int(delay)
        if self.n_slots < 1:
            raise ValueError(f'n_slots must be >= 1, got {n_slots}')
        if self.delay < 0:
            raise ValueError(f'delay must be >= 0, got {delay}')
        self._dev = mlpg._dev
        with torch.cuda.device(self._dev):
            n = _lib.lib().kw_convert_stream_state_len(self.n_slots, mlpg.dim_half, self.delay)
            self._state = torch.empty(n, dtype=torch.float64, device=self._dev)
            _lib.call('kw_convert_stream_init', self.n_slots, mlpg.dim_half, self.delay,
                      self._state, _lib.stream_ptr(torch))

    def _slots(self, slots):
        s = np.asarray(slots)
        if s.ndim != 1 or (s.size and s.dtype.kind not in 'iu'):
            raise ValueError('slots must be a 1-D array of integers')
        if s.size and (s.min() < 0 or s.max() >= self.n_slots):
            raise ValueError(f'slots must be in [0, {self.n_slots})')
        if len(np.unique(s)) != len(s):
            raise ValueError('slots must be distinct')
        return np.ascontiguousarray(s, dtype=np.int32)

    def _workspace(self, m):
        g = self.mlpg
        ws_bytes = _lib.lib().kw_convert_stream_workspace_bytes(m, g.num_mixtures, g.dim_half,
                                                               self.delay, g.precision)
        return _lib.workspace(ws_bytes, self._dev), ws_bytes

    @_on_own_device
    def push_device(self, slots, frames):
        """``frames`` (m, static_dim) float64 CUDA tensor, one static frame for each slot of the
        host array ``slots``.  Returns CUDA tensors ``out`` (m, static_dim), the emitted frames,
        and ``frame_index`` (m,) int64, their frame numbers in their streams (-1 and a zero row
        where a stream has not yet emitted).  Queued on the current stream, no synchronisation."""
        torch = _lib.require_cuda()
        g = self.mlpg
        s = self._slots(slots)
        m = len(s)
        if (tuple(frames.shape) != (m, g.static_dim) or frames.dtype != torch.float64
                or not frames.is_cuda or frames.device.index != torch.cuda.current_device()):
            raise ValueError(f'frames must be a float64 tensor of shape ({m}, {g.static_dim}) '
                             f'on the MLPG\'s device {self._dev}')
        frames = frames.contiguous()
        out = torch.empty((m, g.static_dim), dtype=torch.float64, device=frames.device)
        index = torch.empty(m, dtype=torch.int64, device=frames.device)
        ws, ws_bytes = self._workspace(m)
        _lib.call('kw_convert_stream_push', self.n_slots, self.delay, m, s, frames,
                  g.num_mixtures, g.dim_half, g._prepared, self._state, out, index, g.precision,
                  ws, ws_bytes, _lib.stream_ptr(torch))
        return out, index

    @_on_own_device
    def push(self, slots, frames):
        """``push_device`` from and to host arrays: ``frames`` (m, static_dim) -> (``out``
        (m, static_dim), ``frame_index`` (m,)) as numpy arrays."""
        torch = _lib.require_cuda()
        f = np.ascontiguousarray(frames, dtype=np.float64)
        if f.ndim != 2 or f.shape[1] != self.mlpg.static_dim:
            raise ValueError(f'expected (m, {self.mlpg.static_dim}) static frames, got {f.shape}')
        out, index = self.push_device(slots, torch.from_numpy(f).to(self._dev))
        return out.cpu().numpy(), index.cpu().numpy()

    @_on_own_device
    def end(self, slots):
        """End the streams of ``slots`` (which are then empty): a list with, per slot, the
        (k, static_dim) array of its last k = min(T, delay + 1) frames (none for an empty
        slot)."""
        torch = _lib.require_cuda()
        g = self.mlpg
        s = self._slots(slots)
        m = len(s)
        out = torch.empty((m, self.delay + 1, g.static_dim), dtype=torch.float64,
                          device=self._dev)
        count = torch.empty(m, dtype=torch.int64, device=self._dev)
        ws, ws_bytes = self._workspace(m)
        _lib.call('kw_convert_stream_end', self.n_slots, self.delay, m, s, g.num_mixtures,
                  g.dim_half, g._prepared, self._state, out, count, g.precision, ws, ws_bytes,
                  _lib.stream_ptr(torch))
        out, count = out.cpu().numpy(), count.cpu().numpy()
        return [out[i, :int(count[i])].copy() for i in range(m)]
