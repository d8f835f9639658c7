"""Joint GMM on the B200: the back-end behind kwiiyatta's converter seam.

* ``GaussianMixture`` keeps the slice of ``sklearn.mixture.GaussianMixture`` the reference
  uses (kwiiyatta/converter/gmm.py:13-26; nnmnkwii's MLPG reads ``weights_``, ``means_``,
  ``covariances_``, ``covariance_type``): same constructor keywords, same fitted attributes,
  same stopping rule (sklearn/mixture/_base.py fit_predict loop).
* ``B200GMMFeatureConverter`` mirrors ``GMMFeatureConverter`` (kwiiyatta/converter/gmm.py:8-34)
  and is what ``MelCepstrumConverter(Converter=...)`` / ``Config.create_converter(Converter=...)``
  (kwiiyatta/converter/__init__.py:9-14, kwiiyatta/config.py:59-69) receive.

Two model types: ``covariance_type='full'`` (sklearn's, the default) and
``'diagonal_blocks'``, a joint model whose four D/2 x D/2 covariance blocks are diagonal (each
x_d is coupled to y_d only).  Every E-step / M-step / finalisation runs in csrc/gmm.cu,
csrc/gmm_tc.cu or csrc/gmm_diagblocks.cu through the C ABI; the only host-side arithmetic is the
scalar convergence test.  With ``torch.distributed`` initialised
the per-iteration sufficient statistics are summed over ranks (one all-reduce per iteration);
every rank then finalises identical parameters.
"""
import abc
import warnings

import numpy as np

from . import _lib
from .delta import DELTA_WINDOWS, check_windows

PRECISIONS = {'fp64': 0, 'tc': 1, 0: 0, 1: 1, 'auto': -1}
TC_MAX_DIM = 144          # the tcgen05 kernels hold one frame row of <= 144 features
TC_MIN_FRAMES_PER_DIM = 8
RESP_FORM1_MAX_COMPONENTS = 384   # kw_gmm_estep resp_form 1: K x 64 doubles of shared memory
TC_MIN_WORK = 2e10        # N K D^2 below which the FP64 kernels take about a millisecond anyway


def resolve_precision(precision, n_frames, n_components, dim):
    """'auto' -> the tensor-core path when the fit is large enough to need it and well enough
    determined for it.  The split-fp16 statistics carry a relative error of about 1e-7 of
    ||Sigma_k||; what the next E-step sees is that error times the condition number of Sigma_k,
    and a component estimated from only a few frames per dimension is ill-conditioned by
    construction.  With at least TC_MIN_FRAMES_PER_DIM frames per component and dimension on
    average (configs[1]: 176 k frames, K = 64, D = 144 -> 19) the fit stays within the 1e-5
    tolerance; below that the problem is also small enough for the FP64 CUDA-core kernels
    (N < 8 K D frames), and so is anything under TC_MIN_WORK."""
    code = PRECISIONS[precision]
    if code >= 0:
        return code
    if dim > TC_MAX_DIM:
        return 0
    enough_frames = n_frames >= TC_MIN_FRAMES_PER_DIM * n_components * dim
    enough_work = float(n_frames) * n_components * dim * dim >= TC_MIN_WORK
    return 1 if enough_frames and enough_work else 0


class ConvergenceWarning(UserWarning):
    pass


def _as_device(x, torch, device):
    if hasattr(x, 'data_ptr'):
        t = x.to(device=device, dtype=torch.float64)
    else:
        t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(device)
    return t.contiguous()


_on_own_device = _lib.device_guard(lambda self, *a: self.device)


def _pair_index(d, device, torch):
    """Rows and columns of the (D, D) entries a diagonal-blocks model keeps: per pair d the
    upper-pattern entries (d, d), (d, Dh + d), (Dh + d, Dh + d)."""
    i = torch.arange(d // 2, device=device)
    return i, i + d // 2


def _expand_pairs(torch, compact, symmetric):
    """(K, Dh, 3) compact covariances (``symmetric``) or precision factors -> (K, D, D)."""
    k, dh, _ = compact.shape
    i, j = _pair_index(2 * dh, compact.device, torch)
    out = torch.zeros((k, 2 * dh, 2 * dh), dtype=compact.dtype, device=compact.device)
    out[:, i, i] = compact[:, :, 0]
    out[:, i, j] = compact[:, :, 1]
    out[:, j, j] = compact[:, :, 2]
    if symmetric:
        out[:, j, i] = compact[:, :, 1]
    return out


class GaussianMixture:
    covariance_type = 'full'

    def __init__(self, n_components=1, covariance_type='full', tol=1e-3, reg_covar=1e-6,
                 max_iter=100, n_init=1, init_params='kmeans', weights_init=None,
                 means_init=None, precisions_init=None, random_state=None, warm_start=False,
                 verbose=0, verbose_interval=10, precision='auto', resp_init=None,
                 process_group=None, device=None, reorder_every=10):
        if covariance_type not in ('full', 'diagonal_blocks'):
            raise NotImplementedError("only covariance_type='full' (kwiiyatta/converter/gmm.py:"
                                      "17-18) and 'diagonal_blocks' are built")
        if covariance_type == 'diagonal_blocks' and PRECISIONS[precision] == 1:
            raise ValueError("covariance_type='diagonal_blocks' runs in FP64 only: use "
                             "precision='fp64' or 'auto'")
        if n_init != 1 or warm_start:
            raise NotImplementedError('n_init > 1 / warm_start are not built')
        if precisions_init is not None:
            raise NotImplementedError('precisions_init is not built; pass resp_init or '
                                      'means_init + weights_init')
        self.n_components = n_components
        self.covariance_type = covariance_type
        self._db = covariance_type == 'diagonal_blocks'
        self.tol = tol
        self.reg_covar = reg_covar
        self.max_iter = max_iter
        self.n_init = n_init
        self.init_params = init_params
        self.weights_init = weights_init
        self.means_init = means_init
        self.random_state = random_state
        self.verbose = verbose
        self.verbose_interval = verbose_interval
        self.precision_request = precision
        # -1 ('auto') until the frames are seen; the diagonal-blocks model has the FP64 path only
        self.precision = 0 if self._db else PRECISIONS[precision]
        self.resp_init = resp_init
        self.process_group = process_group
        self.device = device
        self.iter_callback = None
        # Tensor-core path only: the M-step skips (64-frame tile, component) pairs without
        # responsibility mass, so the frames are kept sorted by their dominant component
        # (at initialisation and again every `reorder_every` iterations; 0 = never).  EM sums
        # over frames, the order only changes the rounding of those sums.
        self.reorder_every = int(reorder_every)
        self._x_src = None
        self._x_used = None
        self._iters_done = 0
        self._resp_log = False      # `_resp` holds log-probabilities (see _estep)

    # ------------------------------------------------------------------ device plumbing
    def _alloc(self, torch, n, d, dev):
        k = self.n_components
        lib = _lib.lib()
        f64 = dict(dtype=torch.float64, device=dev)
        self._weights = torch.empty(k, **f64)
        self._means = [torch.empty((k, d), **f64), torch.empty((k, d), **f64)]
        self._cur = 0
        self._alloc_model(torch, k, d, dev)
        self._info = torch.zeros(k, dtype=torch.int32, device=dev)
        self._stats = torch.zeros(self._stats_len(k, d), **f64)
        self._npad = lib.kw_gmm_resp_len(n, k) // k
        self._resp = torch.zeros((k, self._npad), **f64)   # component-major
        self._ws_bytes = self._workspace_bytes(n, k, d)
        self._ws = _lib.workspace(self._ws_bytes, dev)
        # two slots of pinned host memory for the per-iteration scalars (sum log p, n) and the
        # finalisation flags: copied asynchronously, read half an iteration later
        self._host_tail = torch.empty((2, 2), dtype=torch.float64).pin_memory()
        self._host_info = torch.empty((2, k), dtype=torch.int32).pin_memory()
        self._tickets = 0

    def _alloc_model(self, torch, k, d, dev):
        """Covariances, precision factors and aux: (K, D, D), (K, D, D), (K, D + 2) for the full
        model; the compact (K, D/2, 3), (K, D/2, 3), (K, 2) of include/kwiiyatta_b200.h for
        diagonal blocks."""
        f64 = dict(dtype=torch.float64, device=dev)
        if self._db:
            if d % 2:
                raise ValueError(f"covariance_type='diagonal_blocks' needs an even dimension, "
                                 f'got {d}')
            self._pc = torch.empty((k, d // 2, 3), **f64)
            self._aux = torch.empty((k, 2), **f64)
        else:
            self._pc = torch.empty((k, d, d), **f64)
            self._aux = torch.empty((k, d + 2), **f64)
        self._cov = torch.empty(self._pc.shape, **f64)

    def _stats_len(self, k, d):
        lib = _lib.lib()
        return lib.kw_gmm_db_stats_len(k, d) if self._db else lib.kw_gmm_stats_len(k, d)

    def _workspace_bytes(self, n, k, d):
        lib = _lib.lib()
        if self._db:
            return lib.kw_gmm_db_workspace_bytes(n, k, d)
        return lib.kw_gmm_workspace_bytes(n, k, d, self.precision)

    def _pack(self, torch, x):
        if self._db:
            return
        n, d = x.shape
        _lib.call('kw_gmm_pack_frames', n, x, self.n_components, d, self.precision, self._ws,
                  self._ws_bytes, _lib.stream_ptr(torch))

    def _frames(self, x):
        """The tensor the kernels read for the caller's ``x``: its reordered copy if one is
        in use."""
        if self._x_used is not None and self._x_src is not None and \
                x.data_ptr() == self._x_src.data_ptr():
            return self._x_used
        return x

    def _reorder(self, torch, n, permute_resp):
        """Sort the frames by dominant component (the argmax of ``_resp``, responsibilities or
        log-probabilities alike) and re-pack them.  ``permute_resp``: carry the responsibilities
        along (the initial ones); between iterations the next E-step rewrites them instead."""
        labels = self._resp[:, :n].argmax(dim=0)
        perm = torch.argsort(labels, stable=True)
        base = self._x_used if self._x_used is not None else self._x_src
        self._x_used = base.index_select(0, perm)
        if permute_resp:
            self._resp[:, :n] = self._resp[:, :n].index_select(1, perm)
        self._pack(torch, self._x_used)

    def _wants_reorder(self, n):
        return self.precision == 1 and self.reorder_every > 0 and n >= 8192

    def _estep(self, torch, x, for_mstep=False):
        """E-step into ``_resp``.  ``for_mstep`` (tensor-core E-step followed by the
        tensor-core M-step only): ``_resp`` keeps the weighted log-probabilities and the M-step's
        inputs (tile flags, fp32 weights, tile sums) go straight to the workspace -- the
        responsibilities themselves are never written (kw_gmm_estep resp_form 1)."""
        x = self._frames(x)
        n, d = x.shape
        if self._db:
            _lib.call('kw_gmm_db_estep', n, x, self.n_components, d, self._means[self._cur],
                      self._pc, self._aux, self._resp, self._stats, None, self._ws,
                      self._ws_bytes, _lib.stream_ptr(torch))
            return
        self._resp_log = (bool(for_mstep) and self.precision == 1
                          and self.n_components <= RESP_FORM1_MAX_COMPONENTS)
        _lib.call('kw_gmm_estep', n, x, self.n_components, d, self._means[self._cur], self._pc,
                  self._aux, self._resp, self._stats, self.precision, int(self._resp_log),
                  self._ws, self._ws_bytes, _lib.stream_ptr(torch))

    def _normalize_resp(self, torch, x):
        """``_resp`` from log-probabilities to responsibilities, in place (no-op otherwise)."""
        if not self._resp_log:
            return
        n, d = self._frames(x).shape
        _lib.call('kw_gmm_normalize_resp', n, self.n_components, d, self._resp, self._ws,
                  self._ws_bytes, _lib.stream_ptr(torch))
        self._resp_log = False

    def _accumulate(self, torch, x, centres):
        x = self._frames(x)
        n, d = x.shape
        if self._db:
            _lib.call('kw_gmm_db_mstep_accumulate', n, x, self.n_components, d, self._resp,
                      centres, self._stats, self._ws, self._ws_bytes, _lib.stream_ptr(torch))
            return
        _lib.call('kw_gmm_mstep_accumulate', n, x, self.n_components, d, self._resp, centres,
                  self._stats, self.precision, int(self._resp_log), self._ws, self._ws_bytes,
                  _lib.stream_ptr(torch))

    def _allreduce(self, torch):
        """The path's one exchange: sum of the statistics vector over the ranks."""
        from . import dist as kdist
        kdist.allreduce_stats(self._stats, self.process_group)

    def _finalize(self, torch, centres, weight_norm):
        k, d = centres.shape
        new = self._means[self._cur ^ 1]
        entry = 'kw_gmm_db_mstep_finalize' if self._db else 'kw_gmm_mstep_finalize'
        _lib.call(entry, k, d, float(self.reg_covar), weight_norm, self._stats, centres, self._weights, new, self._cov, self._pc, self._aux, self._info,
                  _lib.stream_ptr(torch))
        self._cur ^= 1

    @staticmethod
    def _raise_ill_defined():
        raise ValueError(
            'Fitting the mixture model failed because some components have ill-defined '
            'empirical covariance (for instance caused by singleton or collapsed '
            'samples). Try to decrease the number of components, or increase reg_covar.')

    def _check_info(self):
        if self._info.cpu().numpy().any():
            self._raise_ill_defined()

    # ------------------------------------------------------------------ initialisation
    def _initial_resp(self, torch, x):
        n, _ = x.shape
        k = self.n_components
        if self.resp_init is not None:
            r = _as_device(self.resp_init, torch, x.device)
            if tuple(r.shape) != (n, k):
                raise ValueError(f'resp_init must have shape {(n, k)}, got {tuple(r.shape)}')
            return r.t()
        from . import kmeans
        seed = self.random_state
        if self.init_params == 'kmeans':
            labels = kmeans.kmeans_labels(x, k, seed, self.process_group,
                                          precision=self.precision)
        elif self.init_params == 'random_from_data':
            labels = kmeans.kmeans_labels(x, k, seed, self.process_group, n_lloyd=0,
                                          precision=self.precision)
        else:
            raise NotImplementedError(f'init_params={self.init_params!r} is not built')
        r = torch.zeros((k, n), dtype=torch.float64, device=x.device)
        r[labels, torch.arange(n, device=x.device)] = 1.0
        return r

    # ------------------------------------------------------------------ public API
    @_on_own_device
    def initialize(self, X):
        """Move the frames to the device, allocate the model and run the initial M-step
        (GaussianMixture._initialize).  Returns the device tensor of frames."""
        torch = _lib.require_cuda()
        dev = torch.device('cuda' if self.device is None else self.device)
        x = _as_device(X, torch, dev)
        if x.dim() != 2:
            raise ValueError('Expected 2D array')
        n, d = x.shape
        k = self.n_components
        if self.process_group is None and n < k:
            raise ValueError('Expected n_samples >= n_components '
                             f'but got n_components = {k}, n_samples = {n}')
        import torch.distributed as dist
        multi = dist.is_available() and dist.is_initialized() and \
            dist.get_world_size(self.process_group) > 1
        count = torch.tensor([float(n)], dtype=torch.float64, device=dev)
        if multi:
            dist.all_reduce(count, group=self.process_group)
        if self.precision_request == 'auto' and not self._db:
            self.precision = resolve_precision('auto', int(count.item()), k, d)
        self._alloc(torch, n, d, dev)
        self._x_src, self._x_used, self._iters_done = x, None, 0
        if self.verbose:
            print('Initialization 0')
        # GaussianMixture._initialize: one M-step from the initial responsibilities
        self._resp[:, :n].copy_(self._initial_resp(torch, x))
        self._resp_log = False
        if self._wants_reorder(n):
            self._reorder(torch, n, permute_resp=True)
        else:
            self._pack(torch, x)
        centre = x.sum(dim=0, keepdim=True)
        if multi:
            dist.all_reduce(centre, group=self.process_group)
        centres0 = (centre / count).expand(k, d).contiguous()
        self._stats.zero_()
        self._stats[-1] = float(n)
        self._accumulate(torch, x, centres0)
        self._allreduce(torch)
        self._finalize(torch, centres0, weight_norm=1)
        if self.means_init is not None or self.weights_init is not None:
            self._override_init(torch)
        self._check_info()
        return x

    @_on_own_device
    def fit(self, X, y=None):
        """sklearn's fit loop (sklearn/mixture/_base.py:265-278: E-step, M-step, stop when the
        lower bound of the E-step moved by less than ``tol``), without a host synchronisation on
        the critical path: the statistics of iteration i + 1 are enqueued BEFORE the host reads
        iteration i's lower bound, and iteration i + 1 is finalised (the only step that changes
        the parameters) only once iteration i is known not to have converged.  ``n_iter_``,
        ``converged_``, ``lower_bounds_`` and the parameters are those of the plain loop."""
        torch = _lib.require_cuda()
        x = self.initialize(X)
        self.lower_bounds_ = []
        self.converged_ = False
        state = {'prev': -np.inf, 'n_iter': 0}

        def conclude(n_iter, ticket):
            """Read iteration ``n_iter``'s lower bound; True when the fit stops there."""
            lower_bound = self._resolve(ticket)
            self.lower_bounds_.append(lower_bound)
            change = lower_bound - state['prev']
            state['prev'] = lower_bound
            state['n_iter'] = n_iter
            if self.verbose and n_iter % self.verbose_interval == 0:
                print(f'  Iteration {n_iter}')
            if self.iter_callback is not None:
                self.iter_callback(self, n_iter, lower_bound)
            if abs(change) < self.tol:
                self.converged_ = True
            return self.converged_

        pending = None
        for n_iter in range(1, self.max_iter + 1):
            centres, ticket = self._enqueue_statistics(torch, x)
            if pending is not None and conclude(*pending):
                pending = None
                break           # this iteration's statistics are dropped, nothing was changed
            self._finalize(torch, centres, weight_norm=0)
            pending = (n_iter, ticket)
        if pending is not None:
            conclude(*pending)
        self._check_info()
        if self.verbose:
            print(f'Initialization converged: {self.converged_}')
        if not self.converged_ and self.max_iter > 0:
            warnings.warn('Best performing initialization did not converge. Try different '
                          'init parameters, or increase max_iter, tol, or check for '
                          'degenerate data.', ConvergenceWarning)
        self.n_iter_ = state['n_iter']
        self.lower_bound_ = state['prev']
        self._publish()
        self._resp = None
        self._ws = None
        self._x_src = self._x_used = None
        return self

    def _enqueue_statistics(self, torch, x):
        """E-step, sufficient statistics and their all-reduce for the current parameters, all
        enqueued; the iteration's scalars travel to pinned host memory behind them.  Returns the
        centres the statistics are taken around and a ticket for ``_resolve``."""
        centres = self._means[self._cur]
        self._iters_done += 1
        if self._wants_reorder(x.shape[0]) and self._iters_done % self.reorder_every == 0:
            # by the dominant components of the previous E-step; this one rewrites `_resp`
            self._reorder(torch, x.shape[0], permute_resp=False)
        self._estep(torch, x, for_mstep=True)
        self._accumulate(torch, x, centres)
        self._allreduce(torch)
        slot = self._tickets & 1
        self._tickets += 1
        self._host_tail[slot].copy_(self._stats[-2:], non_blocking=True)
        self._host_info[slot].copy_(self._info, non_blocking=True)   # of the LAST finalisation
        event = torch.cuda.Event()
        event.record(torch.cuda.current_stream(x.device))
        return centres, (slot, event)

    def _resolve(self, ticket):
        slot, event = ticket
        event.synchronize()
        if self._host_info[slot].numpy().any():
            self._raise_ill_defined()
        tail = self._host_tail[slot].numpy()
        return float(tail[0] / tail[1])

    @_on_own_device
    def em_iteration(self, x):
        """One EM iteration on device-resident frames ``x`` (E-step, sufficient statistics,
        all-reduce across ranks, finalisation).  Returns the lower bound of the E-step."""
        torch = _lib.require_cuda()
        centres, ticket = self._enqueue_statistics(torch, x)
        self._finalize(torch, centres, weight_norm=0)
        return self._resolve(ticket)

    @_on_own_device
    def em_iteration_async(self, x):
        """``em_iteration`` without reading anything back: the caller synchronises (and may call
        ``last_lower_bound``) when it needs to."""
        torch = _lib.require_cuda()
        centres, self._last_ticket = self._enqueue_statistics(torch, x)
        self._finalize(torch, centres, weight_norm=0)

    def last_lower_bound(self):
        return self._resolve(self._last_ticket)

    def _override_init(self, torch):
        """means_init / weights_init replace the initial M-step's values (sklearn
        _initialize); the precision Cholesky stays that of the estimated covariances."""
        dev = self._weights.device
        if self.weights_init is not None:
            self._weights.copy_(_as_device(self.weights_init, torch, dev))
        if self.means_init is not None:
            self._means[self._cur].copy_(_as_device(self.means_init, torch, dev))
        self._precision_cholesky(torch)

    def _precision_cholesky(self, torch):
        """Precision factors and aux of ``_cov`` and ``_weights`` (and, for the full model, of the
        current means)."""
        k, d = self._means[self._cur].shape
        if self._db:
            _lib.call('kw_gmm_db_precision_cholesky', k, d, self._weights, self._cov, self._pc,
                      self._aux, self._info, _lib.stream_ptr(torch))
            return
        _lib.call('kw_gmm_precision_cholesky', k, d, self._weights, self._means[self._cur],
                  self._cov, self._pc, self._aux, self._info, _lib.stream_ptr(torch))

    def _publish(self):
        """The fitted attributes.  A diagonal-blocks model publishes full (K, D, D) covariances
        and precision Cholesky factors, zero outside its pattern, so that every consumer of a
        full model (MLPG conversion, sklearn-style code) takes it as it is."""
        self.weights_ = self._weights.cpu().numpy()
        self.means_ = self._means[self._cur].cpu().numpy()
        if self._db:
            import torch
            self.covariances_ = _expand_pairs(torch, self._cov, True).cpu().numpy()
            self.precisions_cholesky_ = _expand_pairs(torch, self._pc, False).cpu().numpy()
            return
        self.covariances_ = self._cov.cpu().numpy()
        self.precisions_cholesky_ = self._pc.cpu().numpy()

    @property
    def precisions_(self):
        pc = self.precisions_cholesky_
        return np.einsum('kij,klj->kil', pc, pc)

    @_on_own_device
    def set_parameters(self, weights, means, covariances):
        """Load an existing model (e.g. a fitted sklearn GaussianMixture's attributes).  With
        ``covariance_type='diagonal_blocks'`` the (K, D, D) covariances must be zero outside the
        pattern of diagonal blocks (ValueError otherwise)."""
        torch = _lib.require_cuda()
        dev = torch.device('cuda' if self.device is None else self.device)
        means = np.asarray(means, dtype=np.float64)
        k, d = means.shape
        self.n_components = k
        f64 = dict(dtype=torch.float64, device=dev)
        self._weights = _as_device(weights, torch, dev)
        self._means = [_as_device(means, torch, dev), torch.empty((k, d), **f64)]
        self._cur = 0
        self._alloc_model(torch, k, d, dev)
        cov = _as_device(covariances, torch, dev)
        if self._db:
            if tuple(cov.shape) != (k, d, d):
                raise ValueError(f'covariances must have shape {(k, d, d)}, got '
                                 f'{tuple(cov.shape)}')
            keep = _expand_pairs(torch, torch.ones((1, d // 2, 3), **f64), True)[0] != 0
            if bool((cov[:, ~keep] != 0).any()):
                raise ValueError("covariance_type='diagonal_blocks': a covariance has a non-zero "
                                 'entry outside the diagonal blocks')
            i, j = _pair_index(d, dev, torch)
            # the lower triangle, as sklearn's Cholesky reads it
            self._cov = torch.stack([cov[:, i, i], cov[:, j, i], cov[:, j, j]], dim=-1)
        else:
            self._cov = cov
        self._info = torch.zeros(k, dtype=torch.int32, device=dev)
        self._precision_cholesky(torch)
        self._check_info()
        self._publish()
        return self

    @_on_own_device
    def _posterior(self, X):
        torch = _lib.require_cuda()
        x = _as_device(X, torch, self._weights.device)
        n, d = x.shape
        k = self.n_components
        lib = _lib.lib()
        self._npad = lib.kw_gmm_resp_len(n, k) // k
        self._resp = torch.empty((k, self._npad), dtype=torch.float64, device=x.device)
        self._stats = torch.zeros(self._stats_len(k, d), dtype=torch.float64, device=x.device)
        if self.precision < 0:      # 'auto' on a model that was loaded, not fitted: FP64 posteriors
            self.precision = 0
        self._ws_bytes = self._workspace_bytes(n, k, d)
        self._ws = _lib.workspace(self._ws_bytes, x.device)
        self._pack(torch, x)
        self._estep(torch, x)
        resp, self._resp, self._ws = self._resp[:, :n].t(), None, None
        return resp, float(self._stats[-2].item()) / n

    def predict_proba(self, X):
        return self._posterior(X)[0].cpu().numpy()

    def predict(self, X):
        return self._posterior(X)[0].argmax(dim=1).cpu().numpy()

    def score(self, X, y=None):
        return self._posterior(X)[1]


class FeatureConverter(abc.ABC):
    """kwiiyatta/converter/abc/converter.py:4-15."""

    @abc.abstractmethod
    def _train(self, dataarray, **kwargs):
        raise NotImplementedError

    # a back-end that takes the training matrix as a CUDA tensor gets it assembled on the device
    accepts_device_array = False

    def train(self, dataset, keys, **kwargs):
        from . import dataset as ds
        self._train(ds.make_dataset_to_array(dataset, keys,
                                             device_resident=self.accepts_device_array),
                    **kwargs)

    @abc.abstractmethod
    def convert(self, feature, **kwargs):
        raise NotImplementedError


class B200GMMFeatureConverter(FeatureConverter):
    """Drop-in for GMMFeatureConverter (kwiiyatta/converter/gmm.py:8-34)."""
    accepts_device_array = True

    def __init__(self, components=64, max_iter=100, random_state=None, gv=False, **kwargs):
        """``gv=True``: ``train`` also estimates the global-variance (GV) statistics that
        ``convert(..., gv=True)`` uses (see ``train``)."""
        super().__init__()
        self.train_gv = bool(gv)
        self._gv = None
        self.init_gmm(components, max_iter, random_state, **kwargs)

    @property
    def gv(self):
        """GV statistics (kwiiyatta_b200.gv.GlobalVariance) or None.  Assign the result of
        ``kwiiyatta_b200.estimate_gv`` to use statistics of other data, e.g. of natural target
        utterances."""
        return self._gv

    @gv.setter
    def gv(self, value):
        from .gv import as_gv
        self._gv = None if value is None else as_gv(value)
        self._paramgen = {k: p for k, p in self._paramgen.items() if not k[2]}

    def train(self, dataset, keys, **kwargs):
        """With ``gv=True`` at construction, the GV statistics come from the TARGET static
        columns [Dh, Dh + static_dim) of each key's rows of the training matrix: the aligned
        target frames without zero frames, exactly what the model is trained on (estimated on the
        device before the fit)."""
        if not self.train_gv:
            return super().train(dataset, keys, **kwargs)
        from . import dataset as ds
        from .gv import estimate_gv
        x, offsets = ds._dataset_to_array_with_offsets(dataset, keys, device_resident=True)
        if x is None:
            raise ValueError('no training data')
        dh = x.shape[1] // 2
        gv = estimate_gv((_as_device(x, _lib.require_cuda(), self._gv_device()), offsets),
                         columns=(dh, dh // len(DELTA_WINDOWS)),
                         process_group=self.gmm.process_group)
        self._train(x, **kwargs)
        self.gv = gv

    def _gv_device(self):
        torch = _lib.require_cuda()
        return torch.device('cuda' if self.gmm.device is None else self.gmm.device)

    def init_gmm(self, components, max_iter=100, random_state=None, **kwargs):
        if 'verbose' not in kwargs:
            kwargs['verbose'] = 1
        if 'covariance_type' not in kwargs:
            kwargs['covariance_type'] = 'full'
        self.gmm = GaussianMixture(n_components=components, max_iter=max_iter,
                                   random_state=random_state, **kwargs)
        self._paramgen = {}

    def _train(self, dataarray, **kwargs):
        self._paramgen = {}
        self.gmm.fit(dataarray, **kwargs)

    # ---- model persistence (the reference keeps the trained model in memory only,
    # kwiiyatta/convert_voice.py:15-20; SURVEY.md section 8f row 4)
    def state_dict(self):
        """The fitted model and its hyper-parameters as plain numpy arrays / scalars."""
        g = self.gmm
        return {'weights': g.weights_, 'means': g.means_, 'covariances': g.covariances_,
                'covariance_type': g.covariance_type, 'n_components': g.n_components, 'max_iter': g.max_iter, 'tol': g.tol,
                'reg_covar': g.reg_covar,
                'random_state': -1 if g.random_state is None else g.random_state,
                'n_iter': getattr(g, 'n_iter_', 0), 'converged': getattr(g, 'converged_', False),
                'lower_bound': getattr(g, 'lower_bound_', float('nan')),
                **({} if self._gv is None else {'gv_mean': self._gv.mean, 'gv_var': self._gv.var})}

    def load_state_dict(self, state):
        """``state`` as ``state_dict`` gives it; one without 'covariance_type' is a full model."""
        g = self.gmm
        kind = str(state.get('covariance_type', 'full'))
        if kind != g.covariance_type:
            raise ValueError(f'the state holds a covariance_type={kind!r} model, this converter '
                             f'was built for {g.covariance_type!r}')
        g.set_parameters(np.asarray(state['weights']), np.asarray(state['means']),
                         np.asarray(state['covariances']))
        g.max_iter, g.tol, g.reg_covar = int(state['max_iter']), float(state['tol']), \
            float(state['reg_covar'])
        rs = int(state['random_state'])
        g.random_state = None if rs < 0 else rs
        g.n_iter_, g.converged_ = int(state['n_iter']), bool(state['converged'])
        g.lower_bound_ = float(state['lower_bound'])
        self._paramgen = {}
        self.gv = (state['gv_mean'], state['gv_var']) if 'gv_mean' in state else None
        return self

    def save(self, path):
        np.savez(path, **self.state_dict())

    @classmethod
    def load(cls, path, **kwargs):
        with np.load(path) as state:
            state = {k: state[k] for k in state.files}
        kind = str(state.get('covariance_type', 'full'))
        if kind != 'full':
            kwargs.setdefault('covariance_type', kind)
        conv = cls(components=int(state['n_components']), verbose=0, **kwargs)
        return conv.load_state_dict(state)

    def _mlpg(self, diff, mlpg=True, gv=False, em_iter=0, conditional_covariance='diagonal'):
        from .mlpg import MLPG
        key = (bool(diff), bool(mlpg), bool(gv), int(em_iter), conditional_covariance)
        if gv and not mlpg:
            raise ValueError('GV is defined for MLPG conversion only (mlpg=True)')
        if conditional_covariance != 'diagonal' and not mlpg:
            raise ValueError('conditional_covariance is defined for MLPG conversion only '
                             '(mlpg=True)')
        if gv and self._gv is None:
            raise ValueError('gv=True needs GV statistics: construct with gv=True and train, '
                             'or assign estimate_gv(...) to .gv')
        if key not in self._paramgen:
            windows = DELTA_WINDOWS if mlpg else DELTA_WINDOWS[0:1]   # gmm.py:29-31
            # 'auto': the tensor-core posterior re-checks near-ties in FP64, so the mixture
            # sequence (and with it the FP64 MLPG output) is the FP64 one at any size
            self._paramgen[key] = MLPG(self.gmm, windows=windows, diff=diff,
                                       precision=self.gmm.precision_request,
                                       gv=self._gv if gv else None, em_iter=em_iter,
                                       conditional_covariance=conditional_covariance)
        return self._paramgen[key]

    def convert(self, feature, mlpg=True, diff=False, gv=False, em_iter=0,
                conditional_covariance='diagonal'):
        """``gv=True``: GV-considered MLPG with the statistics in ``.gv`` (in diff mode the GV
        is that of source + output, which is what the MLSA filter makes heard).
        ``em_iter > 0``: maximum-likelihood conversion over all mixture sequences, ``em_iter``
        EM iterations from the hard-sequence trajectory (``MLPG(em_iter=)``).
        ``conditional_covariance='full'``: the ML trajectory under each mixture's full
        conditional covariance (``MLPG(conditional_covariance=)``)."""
        return self._mlpg(diff, mlpg, gv, em_iter, conditional_covariance).transform(feature)

    def stream(self, n_slots, delay, diff=False):
        """Low-delay conversion of up to ``n_slots`` concurrent streams with a lag of ``delay``
        frames (``MLPG.stream``).  The streams take (m, 24) frames, the mel-cepstrum without c0:
        the caller re-attaches c0, as the mel-cepstrum layer does offline."""
        return self._mlpg(diff).stream(n_slots, delay)

    def convert_many(self, features, diff=False, gv=False, em_iter=0,
                     conditional_covariance='diagonal'):
        """Batched ``convert`` over a list of (T_i, 72) arrays."""
        return self._mlpg(diff, True, gv, em_iter,
                          conditional_covariance).transform_many(features)
