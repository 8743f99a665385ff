"""
`transport_map` -- drop-in class for the hot path of the Triangular Transport Toolbox, backed by
hand-written sm_100a CUDA kernels behind the C ABI of libttm.so (include/ttm.h).

Mirrors the reference class (`/root/reference/transport_map.py`, "tm.py"): constructor signature and
defaults tm.py:12-39, public attributes, `optimize`, `map`, `inverse_map`, `reset`, `s`,
`objective_function`, `objective_function_jacobian`, `evaluate_pullback_density`,
`evaluate_pushforward_density`; beyond the reference, `evaluate_log_pullback_density` and
`evaluate_log_pushforward_density` (log densities of the fitted map, both monotonicity modes).  What stays on the host is what the reference's callers own: the
scipy optimizer steps (BFGS / L-BFGS-B, tm.py:3252-3257 / :3108-3114), the m x m linear algebra of
the separable fit, quantile look-ups for special-term placement, and option/error handling.

Map adaptation (`adapt_map`, `adaptation_cross_terms`) runs on top of this path (adaptation.py).
Out of scope (SURVEY.md section 2): adaptive quadrature order, the
generated-source strings (`fun_mon_strings` ...), `projectedNewton`, progress bars.

PyTorch is used for device buffers, streams and (multi-GPU) torch.distributed only.
"""

import copy
import os

import numpy as np

from . import binding as B
from . import hostopt
from .plan import ComponentPlan, resolve_family

_RECT = {'exponential': 0, 'softplus': 1, 'squared': 2, 'expneg': 3, 'explinearunit': 4}

# grid of the table root finder: the reference's start_distance = 10 and resolution = 1001 of
# vectorized_root_search_alternate (tm.py:4047), which inverse_map never overrides
_TABLE_HALF_WIDTH, _TABLE_NTAB = 10, 1001


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise B.TTMError('no CUDA device visible: this package runs on B200 (sm_100a) only and has no CPU fallback')
    return torch


_SHAPE_MSG = ('X should be a two-dimensional array of shape (N,D), N = number of samples, '
              'D = number of dimensions. Current shape of X is ')


class _DevSamples:
    """A CUDA-tensor sample argument as the *_ld kernels read it in place: n rows of d values, row stride `ld`
    elements, float64 or float32 (`code`: B.TTM_DTYPE_*).  `t` is the tensor (it keeps the storage alive)."""
    __slots__ = ('t', 'n', 'd', 'ld', 'code')

    def __init__(self, t, n, d, ld, code):
        self.t, self.n, self.d, self.ld, self.code = t, n, d, ld, code

    ndim = 2

    @property
    def shape(self):
        return (self.n, self.d)


class _LazyList:
    """List-like view whose items are computed on first access (Psi_mon, Psi_nonmon, der_Psi_mon)."""

    def __init__(self, n, compute):
        self._n, self._compute, self._cache = n, compute, {}

    def __len__(self):
        return self._n

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [self[i] for i in range(*k.indices(self._n))]
        k = int(k)
        if k < 0:
            k += self._n
        if not 0 <= k < self._n:
            raise IndexError(k)
        if k not in self._cache:
            self._cache[k] = self._compute(k)
        return self._cache[k]

    def __setitem__(self, k, v):
        self._cache[int(k)] = v

    def __iter__(self):
        return (self[k] for k in range(self._n))


class transport_map():

    def __init__(self,
                 X,
                 monotone=None,
                 nonmonotone=None,
                 polynomial_type='hermite function',
                 monotonicity='integrated rectifier',
                 standardize_samples=True,
                 standardization='standard',
                 workers=1,
                 ST_scale_factor=1.0,
                 ST_scale_mode='dynamic',
                 coeffs_init=0.,
                 alternate_root_finding=True,
                 root_search_truncation=True,
                 verbose=True,
                 linearization=None,
                 linearization_specified_as_quantiles=True,
                 linearization_increment=1E-6,
                 regularization=None,
                 regularization_lambda=0.1,
                 quadrature_input={},
                 rectifier_type='exponential',
                 delta=1E-8,
                 adaptation=False,
                 adaptation_map_type="cross-terms",
                 adaptation_max_order=10,
                 adaptation_skip_dimensions=0,
                 adaptation_max_iterations=25,
                 device=None,
                 sample_sharded=False,
                 fit_threads=None):
        """Same arguments as the reference constructor (tm.py:12-168).  `device` (extra, optional)
        selects the CUDA device index; default: torch's current device.  `sample_sharded` (extra, optional):
        with torch.distributed initialised, X is this rank's shard of the ensemble; statistics, objective,
        gradient and Gram matrices are all-reduced so that every rank fits every component in lockstep
        (the K < #GPUs case of SURVEY.md 8(e)); default: components are sharded instead.  `fit_threads`
        (extra, optional; default 2, env TTM_FIT_THREADS): host threads of optimize() in integrated-rectifier mode;
        each fits its own components on its own CUDA stream so that kernels of different components overlap."""
        torch = _torch()
        self._torch = torch
        self._dev_index = torch.cuda.current_device() if device is None else int(device)
        self._device = torch.device('cuda', self._dev_index)
        self._lib = B.lib()
        from .parallel import world
        self._rank, self._world = world()
        self._sharded = bool(sample_sharded) and self._world > 1
        if self._world > 1:
            # create the communicator now (the first NCCL collective costs ~3 s) instead of inside optimize()
            from .parallel import warm_up
            warm_up(self._device)
        import os as _os
        self.fit_threads = int(fit_threads if fit_threads is not None else _os.environ.get('TTM_FIT_THREADS', 2))
        if fit_threads is None and isinstance(workers, int) and workers > 1:
            self.fit_threads = min(int(workers), 4)     # the reference's process pool becomes host threads + streams
        # Gram mode of K-objgrad (dJ/da = G a + h, one sweep over x_<c per evaluation): on whenever the component is
        # in the tile kernel's class; TTM_GRAM=0/1 forces it off/on
        _g = _os.environ.get('TTM_GRAM')
        self._use_gram = None if _g is None else (_g != '0')
        import threading as _threading
        self._gram_lock = _threading.Lock()

        self.monotone = copy.deepcopy(monotone)
        self.nonmonotone = copy.deepcopy(nonmonotone)
        self.workers = workers
        self.rectifier_type = rectifier_type
        self.delta = delta
        if rectifier_type not in _RECT:
            raise ValueError("rectifier_type " + str(rectifier_type) + " not understood.")

        # Gauss-Legendre rule, computed exactly as tm.py:199-225 (legroots + closed-form weights)
        self.quadrature_input = quadrature_input
        if 'xis' not in self.quadrature_input and 'Ws' not in self.quadrature_input:
            order = self.quadrature_input.get('order', 100)
            coefs = [0] * order + [1]
            LegendreDer = np.polynomial.legendre.Legendre(np.polynomial.legendre.legder(coefs))
            xis = np.polynomial.legendre.legroots(coefs)
            Ws = 2.0 / ((1.0 - xis ** 2) * (LegendreDer(xis) ** 2))
            self.quadrature_input['xis'] = copy.copy(xis)
            self.quadrature_input['Ws'] = copy.copy(Ws)
        if self.quadrature_input.get('adaptive', False):
            raise NotImplementedError("adaptive quadrature order is out of scope of the CUDA path (SURVEY.md section 2)")

        self.ST_scale_factor = ST_scale_factor
        self.ST_scale_mode = ST_scale_mode
        if self.ST_scale_mode not in ['dynamic', 'static']:
            raise ValueError("'ST_scale_mode' must be either 'dynamic' or 'static'.")
        self.standardization = standardization
        self.coeffs_init = coeffs_init
        self.alternate_root_finding = alternate_root_finding
        self.root_search_truncation = root_search_truncation
        self.verbose = verbose
        self.regularization = regularization
        self.regularization_lambda = regularization_lambda
        self.linearization = linearization
        self.linearization_specified_as_quantiles = linearization_specified_as_quantiles
        self.linearization_increment = linearization_increment
        self.monotonicity = monotonicity
        if self.monotonicity.lower() not in ['integrated rectifier', 'separable monotonicity']:
            raise ValueError("'monotonicity' type " + str(self.monotonicity) + " not understood. " +
                             "Must be either 'integrated rectifier' or 'separable monotonicity'.")
        self._family, self.polyfunc, self.polyfunc_der, self.polynomial_type = resolve_family(polynomial_type)
        self.polyfunc_str = "np.polynomial." + self.polyfunc.__name__

        self.adaptation = adaptation
        self.adaptation_map_type = adaptation_map_type.lower()
        self.adaptation_max_order = adaptation_max_order
        self.adaptation_skip_dimensions = adaptation_skip_dimensions
        self.adaptation_max_iterations = adaptation_max_iterations

        # ---- device context
        ctx = B.c_void_p()
        B.check(self._lib.ttm_ctx_create(self._dev_index, B.ctypes.byref(ctx)))
        self._ctx = ctx
        xis = np.ascontiguousarray(self.quadrature_input['xis'], dtype=np.float64)
        Ws = np.ascontiguousarray(self.quadrature_input['Ws'], dtype=np.float64)
        B.check(self._lib.ttm_ctx_set_quadrature(ctx, B.dptr(xis), B.dptr(Ws), len(xis)))
        B.check(self._lib.ttm_ctx_set_rectifier(ctx, _RECT[rectifier_type], float(delta)))
        sm = B.c_int()
        B.check(self._lib.ttm_device_sm_count(self._dev_index, B.ctypes.byref(sm)))
        self._sm_count = sm.value
        self._scratch = torch.empty(max(4 * self._sm_count * 256, 1 << 16), dtype=torch.float64, device=self._device)

        # ---- samples (tm.py:311-314, 327-328)
        self.standardize_samples = standardize_samples
        if not self.adaptation:
            self.D = len(monotone)
            self.skip_dimensions = X.shape[-1] - self.D
        else:
            # adaptation starts from a dummy map, one constant term per list (tm.py:331-345)
            self.D = X.shape[-1] - self.adaptation_skip_dimensions
            self.skip_dimensions = self.adaptation_skip_dimensions
            self.monotone = [[[]] for _ in range(self.D)]
            self.nonmonotone = [[[]] for _ in range(self.D)]
        self._plans = None
        self._fit_info = {}
        self.chronicle = None       # set to persistence.Chronicle() to log every fit (tm.py:4647-4660 layout)
        self._load_samples(X)

        # ---- term tables (replaces function_constructor_alternative, tm.py:358)
        self.check_for_special_terms()
        self.determine_special_term_locations()
        self._compile_plans()
        self.coeffs_mon = [np.ones(p.m_mon) * self.coeffs_init for p in self._host_plans]
        self.coeffs_nonmon = [np.ones(len(self.nonmonotone[k])) * self.coeffs_init for k in range(self.D)]
        if self.monotonicity.lower() == 'separable monotonicity':
            self.optimization_constraints_lb = [p.lb.copy() for p in self._host_plans]
            self.optimization_constraints_ub = [p.ub.copy() for p in self._host_plans]
        self._make_callables()
        self._reset_lazy()          # precalculate() without re-placing the special terms a second time

    # ================================================================== plumbing
    def _stream(self):
        return B.c_void_p(self._torch.cuda.current_stream(self._device).cuda_stream)

    def _empty(self, *shape):
        return self._torch.empty(*shape, dtype=self._torch.float64, device=self._device)

    def _upload(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        return self._torch.from_numpy(a).to(self._device, non_blocking=False)

    def _samples(self, X, ncol=None):
        """Classify a sample-array argument.  numpy arrays, lists and CPU tensors -> float64 numpy array (the host path).
        A CUDA tensor -> _DevSamples, checked before any launch (2-D, `ncol` columns if given, on this map's device):
        float64 / float32 with unit column stride and a row stride >= d are read in place (column views such as
        Xe[:, skip:]); any other dtype or layout is converted once on the device, as np.asarray(X, float64) converts
        on the host."""
        torch = self._torch
        if isinstance(X, _DevSamples):
            return X
        if not (isinstance(X, torch.Tensor) and X.is_cuda):
            return np.asarray(X, dtype=np.float64)
        if X.ndim != 2:
            raise ValueError(_SHAPE_MSG + str(tuple(X.shape)))
        if X.device != self._device:
            raise ValueError('the tensor is on %s; this map runs on %s' % (X.device, self._device))
        n, d = X.shape
        if ncol is not None and d != ncol:
            raise ValueError('operands could not be broadcast together: %d columns vs %d' % (d, ncol))
        if (X.dtype not in (torch.float64, torch.float32) or (d > 1 and X.stride(1) != 1)
                or (n > 1 and X.stride(0) < d)):
            X = X.to(torch.float64).contiguous()
        return _DevSamples(X, n, d, X.stride(0) if n > 1 else max(d, 1),
                           B.TTM_DTYPE_F32 if X.dtype == torch.float32 else B.TTM_DTYPE_F64)

    def _on_device(self, X):
        """_DevSamples of a host float64 (n, d) array (uploaded contiguous) or of a _DevSamples (itself)."""
        if isinstance(X, _DevSamples):
            return X
        t = self._upload(X)
        n, d = t.shape
        return _DevSamples(t, n, d, d, B.TTM_DTYPE_F64)

    def _to_colmajor(self, X, mean=None, std=None, out=None):
        """row-major (n, d) samples (host array or _DevSamples) -> device column-major (d, n), optionally standardised
        with (mean, std); written to rows [0, d) of `out` (ld = out.shape[1]) instead of a new tensor if given."""
        S = self._on_device(X)
        Xt = self._empty(S.d, S.n) if out is None else out
        mp = B.c_void_p(mean.data_ptr()) if mean is not None else None
        sp = B.c_void_p(std.data_ptr()) if std is not None else None
        B.check(self._lib.ttm_standardize_transpose_ld(self._ctx, B.c_void_p(S.t.data_ptr()), S.code, S.ld, S.n, S.d,
                                                       mp, sp, B.c_void_p(Xt.data_ptr()), Xt.shape[1], self._stream()))
        return Xt

    def _result(self, t, dev):
        """Output step: the device tensor itself for a CUDA-tensor call (dev), else downloaded to numpy."""
        return t if dev else self._download(t)

    def _download(self, t):
        """Device tensor -> numpy.  Large results go through a pinned staging tensor from torch's caching host
        allocator (a pageable `.cpu()` runs at ~2 GB/s; pinned D2H at PCIe rate); the returned array owns it."""
        if t.numel() * 8 < (1 << 22):
            return t.cpu().numpy()
        host = self._torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        host.copy_(t, non_blocking=False)
        return host.numpy()

    def _to_rowmajor(self, Xt, n, d, mean=None, std=None, dev=False):
        """device column-major (d, ld>=n) -> row-major (n, d), optionally un-standardised: host array, or the
        device tensor if dev."""
        out = self._empty(n, d)
        mp = B.c_void_p(mean.data_ptr()) if mean is not None else None
        sp = B.c_void_p(std.data_ptr()) if std is not None else None
        B.check(self._lib.ttm_transpose_back(self._ctx, B.c_void_p(Xt.data_ptr()), Xt.shape[1], n, d, mp, sp,
                                             B.c_void_p(out.data_ptr()), d, self._stream()))
        return self._result(out, dev)

    def _load_samples(self, X):
        """Upload the training ensemble (or read a CUDA tensor in place), standardise it on the device
        (tm.py:750-787) and keep the column-major copy resident.  Quantile standardisation downloads the samples
        for numpy's order statistics (setup, once per reset)."""
        torch = self._torch
        X = self._samples(X)
        if X.ndim != 2:
            raise Exception(_SHAPE_MSG + str(X.shape))
        n, d = X.shape
        self._N, self._Dtot = n, d
        self._N_global = n
        self._X_host = None
        if self._sharded and (not self.standardize_samples or self.standardization.lower() != 'standard'):
            from .parallel import allreduce_sum
            self._N_global = int(round(allreduce_sum(np.array([float(n)]), self._device)[0]))
            if self.standardize_samples:
                raise NotImplementedError("sample_sharded supports standardization='standard' only")
        if not self.standardize_samples:
            self._Xt = self._to_colmajor(X)
            self._mean_d = self._std_d = None
            torch.cuda.current_stream(self._device).synchronize()   # worker streams of optimize() read _Xt
            return
        mode = self.standardization.lower()
        if mode == 'standard':
            Xd = self._on_device(X)
            self._mean_d, self._std_d = self._empty(d), self._empty(d)
            B.check(self._lib.ttm_colstats_ld(self._ctx, B.c_void_p(Xd.t.data_ptr()), Xd.code, Xd.ld, n, d,
                                              B.c_void_p(self._mean_d.data_ptr()), B.c_void_p(self._std_d.data_ptr()),
                                              B.c_void_p(self._scratch.data_ptr()), self._stream()))
            if self._sharded:
                # exact combination of the per-shard moments: one all-reduce of [n, n*mean, n*(var + mean^2)]
                from .parallel import allreduce_sum
                mu, sd = self._mean_d.cpu().numpy(), self._std_d.cpu().numpy()
                tot = allreduce_sum(np.concatenate(([float(n)], n * mu, n * (sd ** 2 + mu ** 2))), self._device)
                self._N_global = int(round(tot[0]))
                gmu = tot[1:1 + d] / tot[0]
                gsd = np.sqrt(np.maximum(tot[1 + d:] / tot[0] - gmu ** 2, 0.0))
                self._mean_d, self._std_d = self._upload(gmu), self._upload(gsd)
            self._Xt = self._to_colmajor(Xd, self._mean_d, self._std_d)
            self.X_mean = self._mean_d.cpu().numpy()
            self.X_std = self._std_d.cpu().numpy()
            del Xd
        elif mode in ('quantile', 'quantiles'):
            # order statistics: host numpy (setup, not hot), exactly tm.py:775-778
            Xh = X.t.to(torch.float64).cpu().numpy() if isinstance(X, _DevSamples) else X
            self.X_mean = np.quantile(Xh, q=0.5, axis=0)
            self.X_std = (np.quantile(Xh - self.X_mean, q=0.8413447460685429, axis=0) -
                          np.quantile(Xh - self.X_mean, q=0.15865525393145707, axis=0)) / 2
            self._mean_d, self._std_d = self._upload(self.X_mean), self._upload(self.X_std)
            self._Xt = self._to_colmajor(X, self._mean_d, self._std_d)
        else:
            raise ValueError("'standardization' must be either 'standard' or 'quantiles'.")
        torch.cuda.current_stream(self._device).synchronize()

    @property
    def X(self):
        """Standardised training samples (N, Dtot), downloaded on demand (the resident copy is column-major)."""
        if self._X_host is None:
            self._X_host = np.ascontiguousarray(self._Xt.cpu().numpy().T)
        return self._X_host

    @X.setter
    def X(self, value):
        value = self._samples(value)
        self._Xt = self._to_colmajor(value)
        self._torch.cuda.current_stream(self._device).synchronize()
        self._N, self._Dtot = value.shape
        self._N_global = self._N
        if self._sharded:
            from .parallel import allreduce_sum
            self._N_global = int(round(allreduce_sum(np.array([float(self._N)]), self._device)[0]))
        self._X_host = None
        self._reset_lazy()                     # memoised (J, grad), Gram matrices and lazy Psi belong to the old ensemble

    def _column(self, d):
        col = self._Xt[d].cpu().numpy()
        if self._sharded:                      # order statistics need the whole column (setup, once per reset)
            import torch.distributed as dist
            parts = [None] * self._world
            dist.all_gather_object(parts, col)
            col = np.concatenate(parts)
        return col

    # ================================================================== special terms
    def check_for_special_terms(self):
        """Counts RBF-type terms per (component, variable); tm.py:2136-2217."""
        blank = lambda: {'counter': 0, 'centers': np.asarray([]), 'scales': np.asarray([])}
        self.special_terms = {}
        for k in range(self.D):
            c = k + self.skip_dimensions
            st = self.special_terms[c] = {}
            for entry in self.nonmonotone[k]:
                if type(entry) == str:
                    st.setdefault(int(entry.split(' ')[1]), blank())['counter'] += 1
            for entry in self.monotone[k]:
                if type(entry) == str:
                    idx = int(entry.split(' ')[1])
                    if idx == c:
                        st.setdefault(idx, blank())['counter'] += 1
                    else:
                        st.setdefault('cross-terms', {}).setdefault(idx, blank())['counter'] += 1

    def determine_special_term_locations(self, k=None):
        """Centres at ensemble quantiles, scales from neighbour spacing; tm.py:2219-2361.
        Quantiles are order statistics of one standardised column: the column is downloaded and
        numpy's linear-interpolation quantile is applied (setup, not hot)."""
        cols = {}

        def column(d):
            if d not in cols:
                cols[d] = self._column(d)
            return cols[d]

        def place(dictionary):
            f = self.ST_scale_factor
            for d in [key for key in dictionary.keys() if key != 'cross-terms']:
                cnt = dictionary[d]['counter']
                if cnt == 1:
                    dictionary[d]['centers'] = np.asarray([np.quantile(column(d), q=0.5)])
                    dictionary[d]['scales'] = np.asarray([f / 2 if self.ST_scale_mode == 'dynamic' else f])
                elif cnt > 1:
                    ctr = np.quantile(a=column(d), q=np.arange(1, cnt + 1, 1) / (cnt + 1))
                    scales = np.zeros(cnt)
                    if self.ST_scale_mode == 'dynamic':
                        for i in range(cnt):
                            if i == 0:
                                scales[i] = (ctr[1] - ctr[0]) * f
                            elif i == cnt - 1:
                                scales[i] = (ctr[i] - ctr[i - 1]) * f
                            else:
                                scales[i] = (ctr[i + 1] - ctr[i - 1]) / 2 * f
                    else:
                        scales = scales + f
                    dictionary[d]['centers'], dictionary[d]['scales'] = ctr, scales
            return dictionary

        K = np.arange(self.D) + self.skip_dimensions if k is None else [k + self.skip_dimensions]
        for c in K:
            c = int(c)
            if 'cross-terms' in self.special_terms[c]:
                self.special_terms[c]['cross-terms'] = place(copy.deepcopy(self.special_terms[c]['cross-terms']))
            self.special_terms[c] = place(copy.deepcopy(self.special_terms[c]))

    # ================================================================== plans
    def _compile_plans(self):
        self._inv_pack_cache = {}
        self._donor_cache = None
        self._host_plans = []
        for k in range(self.D):
            self._host_plans.append(ComponentPlan(
                k, k + self.skip_dimensions, self._Dtot, self._family, self.polyfunc, self.polyfunc_der,
                self.monotone[k], self.nonmonotone[k], self.special_terms, self.linearization))
        self._free_plans()
        self._plans = []
        self._plan_info = []
        for p in self._host_plans:
            self._plans.append(self._create_plan(p))
            self._plan_info.append(self._query_plan(self._plans[-1]))

    def _create_plan(self, p):
        h = B.c_void_p()
        B.check(self._lib.ttm_plan_create(self._ctx, B.iptr(p.iblob), p.iblob.size, B.dptr(p.dblob), p.dblob.size,
                                          B.ctypes.byref(h)))
        return h

    def _query_plan(self, h):
        info = (B.c_int * 4)()
        B.check(self._lib.ttm_plan_info(h, info))
        return {'tile_ok': bool(info[0]), 'dense_mask': int(info[1]), 'n_out_terms': int(info[2])}

    def function_constructor_alternative(self, k=None):
        """Re-compile the term tables after `monotone` / `nonmonotone` were edited (tm.py:1263-1856): of the whole map
        (k None: special terms are re-counted and re-placed, coefficients re-initialised to coeffs_init, :1300-1301,
        :1491, :1610) or of component k only (tables only; coefficients and special-term placement untouched, as in
        the reference's partial construction).  Used by the adaptation routines."""
        if k is None:
            self.check_for_special_terms()
            self.determine_special_term_locations()
            self._compile_plans()
            self.coeffs_mon = [np.ones(p.m_mon) * self.coeffs_init for p in self._host_plans]
            self.coeffs_nonmon = [np.ones(len(self.nonmonotone[kk])) * self.coeffs_init for kk in range(self.D)]
        elif np.isscalar(k):
            k = int(k)
            p = ComponentPlan(k, k + self.skip_dimensions, self._Dtot, self._family, self.polyfunc, self.polyfunc_der,
                              self.monotone[k], self.nonmonotone[k], self.special_terms, self.linearization)
            self._host_plans[k] = p
            self._lib.ttm_plan_destroy(self._plans[k])
            self._plans[k] = self._create_plan(p)
            self._plan_info[k] = self._query_plan(self._plans[k])
            self._inv_pack_cache = {}
            self._donor_cache = None
        else:
            raise Exception("'k' for function_constructor_alternative must be either None or an integer.")
        if self.monotonicity.lower() == 'separable monotonicity':
            self.optimization_constraints_lb = [p.lb.copy() for p in self._host_plans]
            self.optimization_constraints_ub = [p.ub.copy() for p in self._host_plans]
        self._make_callables()
        self._reset_lazy()

    # ================================================================== adaptation (adaptation.py)
    def adapt_map(self, coeffs={}, maxorder_mon=10, maxorder_nonmon=10, threshold_sw=0.1, threshold_prec=0.1,
                  sequential_updates=False, map_finished=None):
        """tm.py:373-657."""
        from . import adaptation
        if self.adaptation_map_type == 'separable':
            adaptation.adapt_separable(self, maxorder_mon, maxorder_nonmon, threshold_sw, threshold_prec, map_finished)
        elif self.adaptation_map_type == 'cross-terms':
            self.adaptation_cross_terms(*coeffs)
        else:
            raise Exception("Currently, only adaptation_map_type = 'cross-terms' is implemented.")

    def adaptation_cross_terms(self, increment=1E-6, chronicle=False):
        """tm.py:4575-4950."""
        from . import adaptation
        adaptation.adapt_cross_terms(self, increment, chronicle)

    def _refresh_special_terms(self):
        """Special-term centres/scales moved (reset / precalculate): patch them into the double blobs.  The tables and
        the int blob do not depend on the data (special-term factors are identified by position, plan._Factors.add;
        tests/test_plan_compiler.py checks refresh_special against a full rebuild, tied centres included)."""
        for k, p in enumerate(self._host_plans):
            if p.has_special:
                p.refresh_special(self.special_terms)          # patches centres / scales in place (== p.build(...))
                B.check(self._lib.ttm_plan_update_doubles(self._plans[k], B.dptr(p.dblob), p.dblob.size))

    def _free_plans(self):
        if getattr(self, '_plans', None):
            for h in self._plans:
                self._lib.ttm_plan_destroy(h)
        self._plans = None

    def __del__(self):
        try:
            self._free_plans()
            if getattr(self, '_ctx', None):
                self._lib.ttm_ctx_destroy(self._ctx)
                self._ctx = None
        except Exception:
            pass

    # ================================================================== basis matrices
    def _basis(self, k, which, Xt, n):
        p = self._host_plans[k]
        m = (p.m_non, p.m_mon, p.m_dmon)[which]
        if m == 0:
            return None
        Psi = self._empty(n, m)
        B.check(self._lib.ttm_basis_eval(self._plans[k], which, B.c_void_p(Xt.data_ptr()), Xt.shape[1], n,
                                         B.c_void_p(Psi.data_ptr()), self._stream()))
        return self._download(Psi)

    def _make_callables(self):
        """fun_mon[k](x, self), fun_nonmon[k](x, self), der_fun_mon[k](x, self): same call signature as the
        reference's exec'd functions (tm.py:1588-1589, 1804-1805, 2131-2132), evaluated by K-basis."""
        def make(k, which):
            def fun(x, _self=None):
                x = np.asarray(x, dtype=np.float64)
                return self._basis(k, which, self._to_colmajor(x), x.shape[0])
            return fun
        self.fun_nonmon = [make(k, 0) for k in range(self.D)]
        self.fun_mon = [make(k, 1) for k in range(self.D)]
        if self.monotonicity.lower() == 'separable monotonicity':
            self.der_fun_mon = [make(k, 2) for k in range(self.D)]

    def precalculate(self):
        """tm.py:789-821: re-place the special terms; the Psi matrices are evaluated lazily on first
        access (the fused kernels never read them)."""
        self.determine_special_term_locations()
        self._refresh_special_terms()
        self._reset_lazy()

    def _reset_lazy(self):
        self._ensemble_version = getattr(self, '_ensemble_version', 0) + 1   # invalidates cached inverse operands
        self._inv_fused_cache = None
        self.Psi_nonmon = _LazyList(self.D, lambda k: self._basis(k, 0, self._Xt, self._N))
        self.Psi_mon = _LazyList(self.D, lambda k: self._basis(k, 1, self._Xt, self._N))
        if self.monotonicity.lower() == 'separable monotonicity':
            self.der_Psi_mon = _LazyList(self.D, lambda k: self._basis(k, 2, self._Xt, self._N))
        self._fg_cache = {}
        self._gram_nn = {}
        self._gram_donor_G = {}
        self._sep_donor = {}

    def reset(self, X):
        """tm.py:710-748."""
        X = self._samples(X)                       # a CUDA tensor of the wrong shape raises ValueError here
        if len(X.shape) != 2:
            raise Exception(_SHAPE_MSG + str(X.shape))
        self._load_samples(X)
        for k in range(self.D):
            self.coeffs_mon[k] = self.coeffs_mon[k] * 0 + self.coeffs_init
            self.coeffs_nonmon[k] = self.coeffs_nonmon[k] * 0 + self.coeffs_init
        self.precalculate()

    def standardize(self):
        """tm.py:750-787: standardise the stored samples in place (mean/std or median/quantile spread) and record
        X_mean / X_std.  The constructor and reset() do this on the way in (K-std); calling it again treats the
        currently stored samples as raw, exactly like the reference."""
        raw = np.array(self.X)
        keep = self.standardize_samples
        self.standardize_samples = True
        try:
            self._load_samples(raw)
        finally:
            self.standardize_samples = keep
        self._reset_lazy()

    # ================================================================== forward map
    def _set_coeffs(self, k, coeffs_nonmon, coeffs_mon):
        c = np.ascontiguousarray(np.concatenate((np.asarray(coeffs_nonmon, dtype=np.float64).ravel(),
                                                 np.asarray(coeffs_mon, dtype=np.float64).ravel())))
        p = self._host_plans[k]
        if c.size != p.m_non + p.m_mon:
            raise ValueError('component %d expects %d nonmonotone + %d monotone coefficients, got %d'
                             % (k, p.m_non, p.m_mon, c.size))
        B.check(self._lib.ttm_plan_set_coeffs(self._plans[k], B.dptr(c), self._stream()))

    def _s_device(self, k, Xt, n, out):
        """S_k on the columns of Xt into the device vector `out` (coefficients already set)."""
        if self.monotonicity == "integrated rectifier":
            B.check(self._lib.ttm_eval_s_ir(self._plans[k], B.c_void_p(Xt.data_ptr()), Xt.shape[1], n,
                                            B.c_void_p(out.data_ptr()), self._stream()))
        elif self.monotonicity == "separable monotonicity":
            B.check(self._lib.ttm_sep_eval(self._plans[k], B.c_void_p(Xt.data_ptr()), Xt.shape[1], n,
                                           B.c_void_p(out.data_ptr()), None, 0, None, self._stream()))
        else:
            raise ValueError("monotonicity must be 'integrated rectifier' or 'separable monotonicity' (case-sensitive "
                             "in s(), tm.py:2516/2550)")

    def s(self, x, k, coeffs_nonmon=None, coeffs_mon=None):
        """k-th map component on (already standardised) samples x, or on the training ensemble if x is None
        (tm.py:2439-2567)."""
        if coeffs_mon is None:
            coeffs_mon = self.coeffs_mon[k]
        if coeffs_nonmon is None:
            coeffs_nonmon = self.coeffs_nonmon[k]
        dev = False
        if x is None:
            Xt, n = self._Xt, self._N
        else:
            x = self._samples(x, ncol=self._Dtot)
            dev = isinstance(x, _DevSamples)
            if dev and x.n == 0:
                return self._empty(0)
            Xt, n = self._to_colmajor(x), x.shape[0]
        self._set_coeffs(k, coeffs_nonmon, coeffs_mon)
        out = self._empty(n)
        self._s_device(k, Xt, n, out)
        return self._result(out, dev)

    # ------------------------------------------------------------------ fused small-map path (K-map-fused)
    def _fused_small(self):
        """True when the whole map goes through ttm_map_fused (all components in one launch on row-major samples):
        separable maps with a few hundred terms in total (Example 05 / 06 shapes).  TTM_MAP_FUSED=0 disables it."""
        if self.monotonicity != "separable monotonicity" or not self.standardize_samples:
            return False
        if os.environ.get('TTM_MAP_FUSED', '1') == '0':
            return False
        return self._Dtot <= 64 and sum(p.m_non + p.m_mon + p.m_dmon for p in self._host_plans) <= 512

    def _map_fused(self, X, mode, sigma=None, log_target=None, want_Z=False):
        """mode 0: pullback density (and Z), 1: pushforward density, 2: Z only; X row-major (n, Dtot): host array
        (results downloaded) or _DevSamples (results stay on the device); log_target: device vector or None."""
        dev = isinstance(X, _DevSamples)
        if X.ndim != 2 or X.shape[1] != self._Dtot:         # the kernel reads Dtot values per row
            raise ValueError('operands could not be broadcast together: X has shape %s, the map has %d columns'
                             % (tuple(X.shape), self._Dtot))
        Xd = self._on_device(X if dev else np.ascontiguousarray(X))
        n = Xd.n
        for k in range(self.D):
            self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
        Z = self._empty(n, self.D) if (want_Z or mode == 2) else None
        out = self._empty(n) if mode != 2 else None
        plans = (B.c_void_p * self.D)(*[h.value for h in self._plans])
        sg = np.ascontiguousarray(sigma, dtype=np.float64) if sigma is not None else None
        ptr = lambda t: B.c_void_p(t.data_ptr()) if t is not None else None
        B.check(self._lib.ttm_map_fused_ld(self._ctx, plans, self.D, B.dptr(sg) if sg is not None else None, ptr(Xd.t),
                                           Xd.code, Xd.ld, n, self._Dtot, ptr(self._mean_d), ptr(self._std_d),
                                           ptr(log_target), mode, ptr(Z), ptr(out), self._stream()))
        return (self._result(Z, dev) if Z is not None else None), (self._result(out, dev) if out is not None else None)

    def map(self, X=None):
        """Forward map target -> reference (tm.py:2391-2437).  X: host array, or a CUDA tensor on the map's device
        (the result is then a float64 CUDA tensor)."""
        dev = False
        if X is not None:
            X = self._samples(X, ncol=self._Dtot)
            dev = isinstance(X, _DevSamples)
            if dev and X.n == 0:
                return self._empty(0, self.D)
        if X is not None and self._fused_small():
            return self._map_fused(X, 2)[0]
        if X is not None and self.standardize_samples:
            Xt, n = self._to_colmajor(X, self._mean_d, self._std_d), X.shape[0]
        else:
            # NB the reference ignores a user-supplied X when standardize_samples is False (tm.py:2419-2422)
            Xt, n = self._Xt, self._N
        Zt = self._empty(self.D, n)
        gm = self._map_gemm_static() if n >= 4096 else None
        if gm is not None:
            # wide separable map: the nonmonotone sums of ALL components are one block-triangular FP64 GEMM (K-inv-rect
            # on DMMA); per component only the monotone terms of its own column remain
            cat = np.concatenate([np.asarray(self.coeffs_nonmon[k], dtype=np.float64) for k in range(self.D)])
            R = np.zeros(gm['r_size'])
            R[gm['rdst']] = (cat[gm['src']] * gm['sc'])[gm['rkeep']]
            cp, cs = gm['const_ptr'], gm['const_src']
            Rd = self._upload(R)
            base = self._empty(self.D, (n + 1) // 2 * 2)
            st = self._stream()
            B.check(self._lib.ttm_map_rect(self._ctx, B.c_void_p(Xt.data_ptr()), Xt.shape[1], n, self.D, gm['rows'],
                                           gm['ns'], self.skip_dimensions, B.c_void_p(Rd.data_ptr()),
                                           B.c_void_p(base.data_ptr()), base.shape[1], st))
            for k in range(self.D):
                self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
                a0 = float(sum(cat[q] for q in cs[cp[k]:cp[k + 1]]))
                B.check(self._lib.ttm_sep_eval_base(self._plans[k], B.c_void_p(Xt.data_ptr()), Xt.shape[1], n,
                                                    B.c_void_p(base[k].data_ptr()), a0, B.c_void_p(Zt[k].data_ptr()), st))
            return self._to_rowmajor(Zt, n, self.D, dev=dev)
        for k in range(self.D):
            self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
            self._s_device(k, Xt, n, Zt[k])
        return self._to_rowmajor(Zt, n, self.D, dev=dev)

    def _map_gemm_static(self):
        """Packing indices of the forward map's GEMM operand (ttm_map_rect), or None when the map is outside its class:
        separable, Hermite functions, >= 32 components, nonmonotone terms = constants + per-variable groups of order
        <= 3 on predecessor columns (the class of K-inv-fused).  Cached until the plans are recompiled.
        TTM_MAP_GEMM=0 keeps the per-component kernels."""
        if self.monotonicity != 'separable monotonicity' or self.D < 32 or os.environ.get('TTM_MAP_GEMM', '1') == '0':
            return None
        from .plan import FAM_HERMITE_E, pack_fused_operands, rect_rpack_doubles
        cache = self.__dict__.setdefault('_inv_pack_cache', {})
        if 'map_gemm' in cache:
            return cache['map_gemm']
        cache['map_gemm'] = None
        rows = self._Dtot - 1
        if self._family != FAM_HERMITE_E or rows <= 0:
            return None
        gm = pack_fused_operands(self._host_plans, self.skip_dimensions, rows, want_apack=False)
        if gm is None:
            return None
        size = B.c_int64()
        B.check(self._lib.ttm_inverse_rect_rpack_size(self.D, rows, gm['ns'], B.ctypes.byref(size)))
        assert size.value == rect_rpack_doubles(self.D, rows, gm['ns'])
        gm.update(rows=rows, r_size=size.value)
        cache['map_gemm'] = gm
        return gm

    # ================================================================== objective + gradient (IR)
    def _objgrad(self, coeffs, k):
        """(J, grad) without regularisation from ONE fused launch; memoised on the coefficient bytes because
        scipy calls `fun` and `jac` separately at the same point (tm.py:3252-3257)."""
        c = np.ascontiguousarray(coeffs, dtype=np.float64)
        key = c.tobytes()
        ent = self._fg_cache.get(k)
        if ent is None or ent[0] != key:
            p = self._host_plans[k]
            G = self._gram_nonmon(k)
            out = np.empty(1 + p.m_non + p.m_mon)
            B.check(self._lib.ttm_objgrad_ir(self._plans[k], B.c_void_p(self._Xt.data_ptr()), self._Xt.shape[1],
                                             self._N, B.dptr(c), B.dptr(out), self._stream()))
            if self._sharded:                  # sample means -> global mean: one all-reduce of (1+m) doubles
                from .parallel import allreduce_sum
                out = allreduce_sum(out * self._N, self._device) / self._N_global
            if G is not None:                  # Gram mode: the kernel returned h only, dJ/da = G a + h
                out[1:1 + p.m_non] += G @ c[:p.m_non]
            ent = self._fg_cache[k] = (key, out)
        return ent[1]

    def _gram_donor(self, k):
        """Component whose nonmonotone term list starts with component k's list (and is the longest such): its
        Gram matrix contains G_k as the leading block, so one K-gram launch serves every component of a map whose
        components share their basis (C4: nonmonotone[k] is a prefix of nonmonotone[D-1]).  Special terms are
        placed per component (tm.py:2241-2330), so lists containing them are not shared."""
        dm = getattr(self, '_donor_cache', None)
        if dm is None:
            from .plan import donor_map
            dm = self._donor_cache = donor_map(self.nonmonotone)
        return dm[k]

    def _gram_nonmon(self, k):
        """G = Psi_non^T Psi_non / N of component k (K-gram, once per ensemble -- the counterpart of the reference's
        precalculate()).  With it K-objgrad sweeps the columns x_<c once per evaluation instead of twice
        (dJ/da = G a + mean_i M_i psi_i).  None when the two-sweep form is used (TTM_GRAM=0, no nonmonotone terms,
        nonmonotone polynomial order > 3, or a component outside the tile kernel's class unless TTM_GRAM=1)."""
        if k in self._gram_nn:
            return self._gram_nn[k]
        with self._gram_lock:
            if k not in self._gram_nn:
                p = self._host_plans[k]
                use = self._plan_info[k]['tile_ok'] if self._use_gram is None else self._use_gram
                G = None
                if use and p.m_non > 0 and p.dense_maxord <= 3:
                    d = self._gram_donor(k)
                    if d not in self._gram_donor_G:
                        md = self._host_plans[d].m_non
                        self._gram_donor_G[d] = np.ascontiguousarray(self._gram(d)[:md, :md]) / self._N_global
                    G = np.ascontiguousarray(self._gram_donor_G[d][:p.m_non, :p.m_non])
                    B.check(self._lib.ttm_plan_set_gram_mode(self._plans[k], 1))
                else:
                    B.check(self._lib.ttm_plan_set_gram_mode(self._plans[k], 0))
                self._gram_nn[k] = G
        return self._gram_nn[k]

    def _reg_lambda(self, k, div):
        lam = self.regularization_lambda
        if np.isscalar(lam):
            return lam, lam
        if type(lam) == list:
            return lam[k][:div], lam[k][div:]
        raise ValueError("Data type of regularization_lambda not understood. Must be either scalar or list.")

    def _split(self, coeffs, k, div):
        if coeffs is None:
            return np.concatenate((self.coeffs_nonmon[k], self.coeffs_mon[k])), len(self.coeffs_nonmon[k])
        return np.asarray(coeffs, dtype=np.float64), div

    def objective_function(self, coeffs, k, div=0):
        """tm.py:3300-3433."""
        coeffs, div = self._split(coeffs, k, div)
        a, b = coeffs[:div], coeffs[div:]
        objective = float(self._objgrad(coeffs, k)[0])
        if self.regularization is not None:
            if type(self.regularization) != str:
                raise ValueError("The variable 'regularization' must be either None, 'l1', or 'l2'.")
            la, lb = self._reg_lambda(k, div)
            if self.regularization.lower() == 'l1':
                objective += np.sum(lb * np.abs(b)) + np.sum(la * np.abs(a))
            elif self.regularization.lower() == 'l2':
                objective += np.sum(lb * b ** 2) + np.sum(la * a ** 2)
            else:
                raise ValueError("regularization_type must be either 'l1' or 'l2'.")
        return objective

    def objective_function_jacobian(self, coeffs, k, div=0):
        """tm.py:3435-3635."""
        if self.rectifier_type in ('squared', 'explinearunit'):
            raise Exception("Not implemented yet.")            # rectifier.evaluate_dfdc, tm.py:5119-5163
        coeffs, div = self._split(coeffs, k, div)
        a, b = coeffs[:div], coeffs[div:]
        grad = np.array(self._objgrad(coeffs, k)[1:])
        if self.regularization is not None:
            if type(self.regularization) != str:
                raise ValueError("The variable 'regularization' must be either None, 'l1', or 'l2'.")
            la, lb = self._reg_lambda(k, div)
            if self.regularization.lower() == 'l1':
                grad = grad + np.concatenate((la * np.sign(a), lb * np.sign(b)))
            elif self.regularization.lower() == 'l2':
                grad = grad + np.concatenate((la * 2 * a, lb * 2 * b))
            else:
                raise ValueError("regularization_type must be either 'l1' or 'l2'.")
        return grad

    # ================================================================== fitting
    def worker_task(self, k, task_supervisor=None):
        """BFGS on the fused objective/gradient (tm.py:3174-3298)."""
        from scipy.optimize import minimize
        import time as _time
        div = len(self.coeffs_nonmon[k])
        x0 = np.concatenate((self.coeffs_nonmon[k], self.coeffs_mon[k]))
        _t0 = _time.perf_counter()
        from . import hostopt
        if os.environ.get('TTM_HOST_OPT', 'native') != 'scipy' and hostopt.available():
            # the same BFGS iteration with scipy's own line search and an O(n^2) update (hostopt.py): scipy's O(n^3)
            # update costs more than the CUDA evaluation once a component has a few hundred coefficients
            opt = hostopt.quasi_newton(lambda c: (self.objective_function(c, k, div),
                                                  self.objective_function_jacobian(c, k, div)), x0)
        else:
            opt = minimize(method='BFGS', fun=self.objective_function, jac=self.objective_function_jacobian,
                           x0=x0, args=(k, div))
        self._last_opt = opt
        self._fit_info[k] = {'nit': int(opt.nit), 'nfev': int(opt.nfev), 'fun': float(opt.fun),
                             'success': bool(opt.success), 'seconds': _time.perf_counter() - _t0}
        return (opt.x[:div].copy(), opt.x[div:].copy())

    def _gram(self, k, first_col=0):
        """[Psi_non | Psi_mon]^T [Psi_non | Psi_mon] of component k (K-gram), (M, M).  first_col > 0: only the columns
        from first_col on are computed (ttm_gram_tail) and returned, (M, M - first_col)."""
        p = self._host_plans[k]
        M = p.m_non + p.m_mon
        G = self._empty(M, M)
        Mp = (M + 7) // 8 * 8
        need = 64 * Mp * Mp + min(self._N, 1 << 18) * Mp      # split partials + one materialised Psi chunk
        if self._scratch.numel() < need:
            self._scratch = self._empty(need)
        B.check(self._lib.ttm_gram_tail(self._plans[k], B.c_void_p(self._Xt.data_ptr()), self._Xt.shape[1], self._N,
                                        int(first_col), B.c_void_p(G.data_ptr()), B.c_void_p(self._scratch.data_ptr()),
                                        self._scratch.numel(), self._stream()))
        if first_col > 0:
            G = G[:, first_col:].contiguous()                  # only the computed columns travel to the host
        G = G.cpu().numpy()
        if self._sharded:
            from .parallel import allreduce_sum
            G = allreduce_sum(G.ravel(), self._device).reshape(G.shape)
        return G

    def _separable_donor(self, k):
        """Shared pieces of the separable setup for every component whose nonmonotone list is a prefix of the donor's
        (one full K-gram and ONE factorisation per donor instead of one per component): the nonmonotone Gram block
        and the Cholesky factors of the (Jacobi-scaled) block, of Gnn + lam I and of Gnn + 2 lam I.  The Cholesky
        factor of a leading principal block is the leading block of the factor."""
        d = self._gram_donor(k)
        with self._gram_lock:
            if d not in self._sep_donor:
                from scipy.linalg import cholesky
                md = self._host_plans[d].m_non
                G = self._gram(d)
                Gnn = np.ascontiguousarray(G[:md, :md])
                ent = {'Gnn': Gnn, 'G_full': G}
                if self.regularization is None:
                    dv = 1.0 / np.sqrt(np.maximum(np.diag(Gnn), np.finfo(float).tiny))
                    ent['d'] = dv
                    ent['L'] = cholesky(Gnn * dv[:, None] * dv[None, :], lower=True, check_finite=False)
                elif type(self.regularization) == str and self.regularization.lower() == 'l2':
                    lam = self.regularization_lambda
                    ent['L1'] = cholesky(Gnn + lam * np.identity(md), lower=True, check_finite=False)
                    ent['L2'] = cholesky(Gnn + 2 * lam * np.identity(md), lower=True, check_finite=False)
                self._sep_donor[d] = ent
        return d, self._sep_donor[d]

    def _separable_setup(self, k):
        """Reduced m_mon x m_mon problem from the Gram blocks of [Psi_non | Psi_mon] (K-gram, DMMA).
        No regularisation: A = (Gmm - Gmn Gnn^-1 Gnm)/N, which equals A_sqrt^T A_sqrt / N of the reference's QR
        formulation (tm.py:2966-2975).  L2: the ridge normal equations of tm.py:3031-3050 (no 1/N there)."""
        from scipy.linalg import solve_triangular
        p = self._host_plans[k]
        mn = p.m_non
        d, ent = self._separable_donor(k)
        if d == k:
            Gt = ent['G_full'][:, mn:]
        else:
            Gt = self._gram(k, first_col=mn)                   # Psi^T Psi_mon only: the leading block is the donor's
        Gnn, Gnm, Gmm = ent['Gnn'][:mn, :mn], Gt[:mn], Gt[mn:]
        N = self._N_global
        tri = lambda L, rhs, trans=0: solve_triangular(L, rhs, lower=True, trans=trans, check_finite=False)
        if self.regularization is None:
            # scaled Cholesky solve (Jacobi preconditioning tames the squared condition number)
            dv, L = ent['d'][:mn], ent['L'][:mn, :mn]
            Y = tri(L, Gnm * dv[:, None])
            A = (Gmm - Y.T @ Y) / N
            back = lambda b: -(dv * tri(L, Y @ b, 'T'))
        elif self.regularization.lower() == 'l2':
            lam = self.regularization_lambda
            L1, L2 = ent['L1'][:mn, :mn], ent['L2'][:mn, :mn]
            Bm = tri(L1, tri(L1, Gnm), 'T')                    # (Gnn + lam I)^-1 Gnm
            # (Psi_m - Psi_n B)^T (Psi_m - Psi_n B) expanded in Gram blocks
            R = Gmm - Gnm.T @ Bm - Bm.T @ Gnm + Bm.T @ Gnn @ Bm
            A = R / 2 + lam * (Bm.T @ Bm + np.identity(Bm.shape[-1]))
            back = lambda b: -tri(L2, tri(L2, Gnm @ b), 'T')
        else:
            raise ValueError("separable monotonicity supports regularization None or 'l2'")
        return 0.5 * (A + A.T), back

    def _sep_objective(self, b, A, k):
        """(f, grad) of the reduced problem, tm.py:2978-3006; the N-long sums come from K-sepobj."""
        p = self._host_plans[k]
        b = np.ascontiguousarray(b, dtype=np.float64)
        out = np.empty(1 + p.m_dmon)
        B.check(self._lib.ttm_sep_objgrad(self._plans[k], B.c_void_p(self._Xt.data_ptr()), self._Xt.shape[1],
                                          self._N, B.dptr(b), B.dptr(out), self._stream()))
        if self._sharded:
            from .parallel import allreduce_sum
            out = allreduce_sum(out, self._device)
        N = self._N_global
        bvec = self.delta * np.sum(A, axis=-1)
        Ax = A @ b
        f = b @ Ax / 2 - out[0] / N + b @ bvec
        g = Ax - out[1:] / N + bvec
        return f, g

    def worker_task_monotone(self, k, task_supervisor=None):
        """Separable fit of component k (tm.py:2903-3172)."""
        from scipy.optimize import minimize
        if self._host_plans[k].m_non == 0:
            raise ValueError("separable monotonicity requires at least one nonmonotone term per component "
                             "(the reference's np.linalg.qr(None) fails too)")
        A, back = self._separable_setup(k)
        bounds = [[self.optimization_constraints_lb[k][i], self.optimization_constraints_ub[k][i]]
                  for i in range(len(self.optimization_constraints_lb[k]))]
        opt = minimize(fun=lambda b, A, k: self._sep_objective(b, A, k), method='L-BFGS-B',
                       x0=copy.copy(self.coeffs_mon[k]), jac=True, bounds=bounds, args=(A, k))
        self._last_opt = opt
        self._fit_info[k] = {'nit': int(opt.nit), 'nfev': int(opt.nfev), 'fun': float(opt.fun),
                             'success': bool(opt.success)}
        return (back(opt.x), opt.x)

    def _fit_separable_lockstep(self, comps):
        """Separable fits of the listed components (tm.py:2903-3172 per component), their L-BFGS-B iterations advanced
        together: every round launches K-sepobj for each component that asked for (f, g) and then collects the
        results (hostopt.lbfgsb_lockstep; the iterates are those of scipy's minimize).  With a sample-sharded
        ensemble every rank runs the same iteration on all-reduced sums."""
        setups, x0s, bnds = {}, [], []
        for k in comps:
            if self._host_plans[k].m_non == 0:
                raise ValueError("separable monotonicity requires at least one nonmonotone term per component "
                                 "(the reference's np.linalg.qr(None) fails too)")
            A, back = self._separable_setup(k)
            setups[k] = (A, back, self.delta * np.sum(A, axis=-1))
            x0s.append(np.array(self.coeffs_mon[k], dtype=np.float64))
            inf = lambda v, sgn: sgn * np.inf if v is None else float(v)
            bnds.append((np.array([inf(v, -1.0) for v in self.optimization_constraints_lb[k]]),
                         np.array([inf(v, 1.0) for v in self.optimization_constraints_ub[k]])))
        lib, Xp, ld, N, st = self._lib, B.c_void_p(self._Xt.data_ptr()), self._Xt.shape[1], self._N, self._stream()
        outs = [np.empty(1 + self._host_plans[k].m_dmon) for k in comps]
        held = {}

        def launch(i, b):
            held[i] = np.array(b, dtype=np.float64)                  # setulb updates its x in place
            B.check(lib.ttm_sep_objgrad_launch(self._plans[comps[i]], Xp, ld, N, B.dptr(held[i]), st))

        def collect(i):
            k = comps[i]
            B.check(lib.ttm_sep_objgrad_wait(self._plans[k], B.dptr(outs[i]), st))
            out = outs[i]
            if self._sharded:
                from .parallel import allreduce_sum
                out = allreduce_sum(out, self._device)
            A, _, bvec = setups[k]
            b = held[i]
            Ax = A @ b
            Ng = self._N_global
            return b @ Ax / 2 - out[0] / Ng + b @ bvec, Ax - out[1:] / Ng + bvec

        if self._sharded:
            res = hostopt.lbfgsb_lockstep(x0s, bnds, launch, collect)
        else:
            # one C call per round: queue every K-sepobj launch, collect, assemble (f, g) of the reduced problem
            ct = B.ctypes
            vp = ct.c_void_p
            Ab = [np.ascontiguousarray(setups[k][0]) for k in comps]
            cb = [np.ascontiguousarray(setups[k][2]) for k in comps]
            bb = [np.empty(len(x)) for x in x0s]
            fg = [np.empty(1 + len(x)) for x in x0s]
            addr = lambda arrs: [a.ctypes.data for a in arrs]
            pA, pc, pb, pfg = addr(Ab), addr(cb), addr(bb), addr(fg)
            pl = [self._plans[k].value if hasattr(self._plans[k], 'value') else self._plans[k] for k in comps]
            Ng = float(self._N_global)

            def batch(idx, xs):
                n = len(idx)
                for i, x in zip(idx, xs):
                    bb[i][:] = x
                arr = lambda src: (vp * n)(*[src[i] for i in idx])
                B.check(lib.ttm_sep_reduced_batch(n, arr(pl), Xp, ld, N, Ng, arr(pb), arr(pA), arr(pc), arr(pfg), st))
                return [(fg[i][0], fg[i][1:].copy()) for i in idx]

            res = hostopt.lbfgsb_lockstep(x0s, bnds, batch=batch)
        results = {}
        for k, opt in zip(comps, res):
            self._last_opt = opt
            self._fit_info[k] = {'nit': int(opt.nit), 'nfev': int(opt.nfev), 'fun': float(opt.fun),
                                 'success': bool(opt.success)}
            results[k] = (setups[k][1](opt.x), opt.x)
        return results

    def optimize(self, K=None):
        """tm.py:2714-2901.  Components are independent; with torch.distributed initialised they are sharded
        over the ranks (longest first, like the reference's Pool over np.flip(K)) and the coefficients are
        gathered with one all-gather."""
        if K is None:
            K = np.arange(self.D)
        K = [int(k) for k in K]
        fit = self.worker_task if self.monotonicity == "integrated rectifier" else self.worker_task_monotone
        from .parallel import shard_components, allgather_coeffs, world
        rank, size = world()
        if self._sharded:
            rank, size = 0, 1                  # every rank fits every component on its shard, in lockstep
        mine = shard_components(K, rank, size)
        results = {}
        import time as _time
        _t0 = _time.perf_counter()
        nthreads = self.fit_threads if (self.monotonicity == "integrated rectifier" and not self._sharded) else 1
        if nthreads > 1 and len(mine) > 1:
            # components are independent: a few host threads, each on its own stream with a reduced grid per
            # launch, so that the sweeps of one component overlap the node loop of another on every SM
            import concurrent.futures
            import threading
            torch = self._torch
            tls = threading.local()
            main_stream = torch.cuda.current_stream(self._device)
            B.check(self._lib.ttm_ctx_set_blocks_per_sm(self._ctx, 2))

            def run(k):
                if not hasattr(tls, 'stream'):
                    # a new host thread starts on device 0: bind it to this map's GPU first, or the stream context
                    # below would query (and so create a context on) device 0 from every rank
                    torch.cuda.set_device(self._device)
                    tls.stream = torch.cuda.Stream(device=self._device)
                    tls.stream.wait_stream(main_stream)      # the ensemble was produced on the caller's stream
                with torch.cuda.stream(tls.stream):
                    return k, fit(k, None)
            try:
                with concurrent.futures.ThreadPoolExecutor(max_workers=nthreads) as ex:
                    for k, r in ex.map(run, mine):
                        results[k] = r
            finally:
                B.check(self._lib.ttm_ctx_set_blocks_per_sm(self._ctx, 0))
            torch.cuda.synchronize(self._device)
        elif (self.monotonicity != "integrated rectifier" and len(mine) > 0
              and os.environ.get('TTM_HOST_OPT', '') != 'scipy' and hostopt.lbfgsb_available()):
            results = self._fit_separable_lockstep(mine)
        else:
            for k in mine:
                results[k] = fit(k, None)
                if self.verbose and size == 1:
                    print('\r' + 'Progress: |' + (K.index(k) + 1) * '█' + (len(K) - K.index(k) - 1) * ' ' + '|', end='\r')
        _t1 = _time.perf_counter()
        if size > 1:
            results = allgather_coeffs(results, K, [self._host_plans[k].m_non for k in K],
                                       [self._host_plans[k].m_mon for k in K], self._device)
        self._last_timing = {'fit_s': _t1 - _t0, 'gather_s': _time.perf_counter() - _t1, 'components': len(mine)}
        for k in K:
            self.coeffs_nonmon[k] = copy.deepcopy(results[k][0])
            self.coeffs_mon[k] = copy.deepcopy(results[k][1])
        if self.chronicle is not None:             # fit log (persistence.Chronicle), components fitted by this rank
            for k in mine:
                self.chronicle.record(self, k, **self._fit_info.get(k, {}))

    # ================================================================== persistence (examples' pickle format)
    def save_coefficients(self, path):
        """pickle {'coeffs_mon': [...], 'coeffs_nonmon': [...]} exactly as example_01.py:215-224 does."""
        from .persistence import save_coefficients
        save_coefficients(self, path)

    def load_coefficients(self, path):
        """Impose pickled coefficients (the reference examples' files load unchanged), example_01.py:226-231."""
        from .persistence import load_coefficients
        return load_coefficients(self, path)

    # ================================================================== inverse map
    def inverse_map(self, Z, X_star=None):
        """Inverse map reference -> target, optionally conditioned on X_star (tm.py:3639-3796).  Z: host array, or a
        CUDA tensor on the map's device (the result is then a float64 CUDA tensor); X_star may be either kind."""
        Z = self._samples(Z)
        dev = isinstance(Z, _DevSamples)
        N = Z.shape[0]
        skip, D = self.skip_dimensions, self.D
        if X_star is None:
            ncol, comps, E = skip + D, [(k, k) for k in range(D)], 0
        else:
            X_star = self._samples(X_star)
            if X_star.shape[-1] == skip:
                ncol, comps, E = skip + D, [(k, k) for k in range(D)], skip
            elif skip == 0:
                E = X_star.shape[-1]
                ncol, comps = E + Z.shape[-1], [(i, k) for i, k in enumerate(range(E, E + Z.shape[-1]))]
            else:
                raise UnboundLocalError("X_star has %d columns; expected skip_dimensions = %d" % (X_star.shape[-1], skip))
        if ncol != self._Dtot:
            raise ValueError("operands could not be broadcast together: %d columns vs %d" % (ncol, self._Dtot))
        if dev and Z.shape[1] != len(comps):
            raise ValueError("operands could not be broadcast together: %d columns vs %d" % (Z.shape[1], len(comps)))
        if E > 0 and X_star.shape[0] != N:
            raise ValueError("operands could not be broadcast together: %d samples in Z vs %d in X_star"
                             % (N, X_star.shape[0]))
        if dev and N == 0:
            return self._empty(0, ncol - skip)
        torch = self._torch
        table_mode = self.alternate_root_finding and self.monotonicity.lower() == 'separable monotonicity'
        # the pipeline hides host <-> device copies: device operands take the one-shot path (bit-identical)
        if (table_mode and not dev and not isinstance(X_star, _DevSamples)
                and N >= int(os.environ.get('TTM_INV_PIPELINE_MIN', 131072))):
            return self._inverse_map_pipelined(Z, X_star, E, ncol, comps)
        Xw = torch.zeros(ncol, N, dtype=torch.float64, device=self._device)
        if E > 0:
            std = self.standardize_samples
            self._to_colmajor(X_star, self._mean_d[:E].contiguous() if std else None,
                              self._std_d[:E].contiguous() if std else None, out=Xw)
        Zt = self._to_colmajor(Z)
        self._inverse_solve(self._inverse_solver(comps, table_mode), Xw, Xw.shape[1], N, Zt, Zt.shape[1], self._stream())
        if self.standardize_samples:
            Xout = self._to_rowmajor(Xw[skip:], N, ncol - skip, self._mean_d[skip:].contiguous(),
                                     self._std_d[skip:].contiguous(), dev=dev)
        else:
            Xout = self._to_rowmajor(Xw[skip:], N, ncol - skip, dev=dev)
        return Xout

    def _monotone_tables(self, comps):
        """Lookup tables of vectorized_root_search_alternate (tm.py:4047-4062) for all listed components in ONE device
        buffer [ncomp][2*_TABLE_NTAB] (values | abscissae) with ONE host round trip: scipy's interp1d sorts its
        abscissae with a stable sort (assume_sorted=False), which is the identity for a non-decreasing table -- the
        normal case (monotone coefficients >= 0); only rows that are not sorted are sorted on the host.  Sets the
        components' coefficients on their plans."""
        pts = np.linspace(-_TABLE_HALF_WIDTH, _TABLE_HALF_WIDTH, _TABLE_NTAB)
        tabs = self._empty(len(comps), 2 * _TABLE_NTAB)
        tabs[:, _TABLE_NTAB:] = self._upload(pts)
        for r, (_, k) in enumerate(comps):
            self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
            B.check(self._lib.ttm_mon_table(self._plans[k], _TABLE_NTAB, B.c_void_p(tabs[r].data_ptr()), self._stream()))
        vals = tabs[:, :_TABLE_NTAB].cpu().numpy()
        bad = np.nonzero(~np.all(vals[:, 1:] >= vals[:, :-1], axis=1))[0]
        for r in bad:
            ind = np.argsort(vals[r], kind="mergesort")
            tabs[r] = self._upload(np.concatenate((vals[r][ind], pts[ind])))
        return tabs

    def _inverse_fused_static(self, ks, mode):
        """The part of the K-inv-fused / K-inv-rect operands that depends on the term lists only (class check, slot set,
        packed destination of every coefficient: plan.pack_fused_operands), cached until the plans are recompiled: a
        conditional-sampling loop with changing coefficients (EnTF cycles, adaptation) pays one gather/scatter per call
        instead of a walk over every dense group of every component."""
        from .plan import FAM_HERMITE_E, pack_fused_operands, fused_apack_doubles, rect_rpack_doubles
        cache = self.__dict__.setdefault('_inv_pack_cache', {})
        skey = (tuple(ks), mode)
        if skey in cache:
            return cache[skey]
        cache[skey] = None
        plans = [self._host_plans[k] for k in ks]
        c0, ncomp = plans[0].c, len(ks)
        if self._family != FAM_HERMITE_E:
            return None
        # wide conditioning block: its share of the offsets is one GEMM (K-inv-rect) ahead of the sequential walk
        split = c0 > 0 and mode != '0' and (mode == '1' or (c0 >= 32 and ncomp >= 32))
        st = pack_fused_operands(plans, c0, c0 if split else 0)
        if st is None:
            return None
        size = B.c_int64()
        B.check(self._lib.ttm_inverse_fused_apack_size(ncomp, c0, st['ns'], B.ctypes.byref(size)))
        assert size.value == fused_apack_doubles(ncomp, c0, st['ns'])
        st.update(ncomp=ncomp, c0=c0, split=split, a_size=size.value, r_size=0)
        if split:
            B.check(self._lib.ttm_inverse_rect_rpack_size(ncomp, c0, st['ns'], B.ctypes.byref(size)))
            assert size.value == rect_rpack_doubles(ncomp, c0, st['ns'])
            st['r_size'] = size.value
        cache[skey] = st
        return st

    def _inverse_fused_setup(self, comps):
        """Operands of K-inv-fused (ttm_inverse_fused: the component loop of tm.py:3684-3698 in one launch), or None if
        some component is outside its class (nonmonotone terms other than constants and per-variable Hermite-function
        groups of order <= 3, components not on consecutive columns)."""
        if not comps or os.environ.get('TTM_INV_FUSED', '1') == '0':
            return None
        ks = [k for _, k in comps]
        # operands depend on the coefficients and the special-term placement only: repeated calls (sampling in batches,
        # the chunks of one call) reuse them
        import hashlib
        h = hashlib.blake2b(digest_size=16)
        for k in ks:
            h.update(np.ascontiguousarray(self.coeffs_nonmon[k], dtype=np.float64).tobytes())
            h.update(np.ascontiguousarray(self.coeffs_mon[k], dtype=np.float64).tobytes())
        mode = os.environ.get('TTM_INV_SPLIT', 'auto')
        key = (tuple(ks), self._ensemble_version, h.digest(), mode)
        hit = getattr(self, '_inv_fused_cache', None)
        if hit is not None and hit[0] == key:
            return hit[1]
        st = self._inverse_fused_static(ks, mode)
        if st is None:
            return None
        ncomp, c0, ns, split = st['ncomp'], st['c0'], st['ns'], st['split']
        # dynamic part: coefficient * scale scattered into the packed operands, all components at once
        cat = np.concatenate([np.asarray(self.coeffs_nonmon[k], dtype=np.float64) for k in ks])
        val = cat[st['src']] * st['sc']
        A = np.zeros(st['a_size'])
        A[st['dst']] = val
        cp, cs = st['const_ptr'], st['const_src']
        a0 = np.array([sum(cat[q] for q in cs[cp[j]:cp[j + 1]]) for j in range(ncomp)], dtype=np.float64)
        if split:
            R = np.zeros(st['r_size'])
            R[st['rdst']] = val[st['rkeep']]
        fused = {'ncomp': ncomp, 'c0': c0, 'ns': ns, 'A': self._upload(A), 'a0': self._upload(a0),
                 'tabs': self._monotone_tables(comps), 'ntab': _TABLE_NTAB,
                 'R': self._upload(R) if split else None}
        self._inv_fused_cache = (key, fused)
        return fused

    def _inverse_fused_launch(self, f, Xw, ld, n, Zt, ldz, stream=None, base=None):
        if f.get('R') is not None:
            # two launches: K-inv-rect (conditioning block -> base), then the walk over the solved columns
            if base is None:
                base = self._torch.empty((f['ncomp'], (n + 1) // 2 * 2), dtype=self._torch.float64, device=self._device)
            B.check(self._lib.ttm_inverse_fused_split(
                self._ctx, B.c_void_p(Xw.data_ptr()), ld, n, B.c_void_p(Zt.data_ptr()), ldz, f['ncomp'], f['c0'], f['ns'],
                B.c_void_p(f['A'].data_ptr()), B.c_void_p(f['R'].data_ptr()), B.c_void_p(f['a0'].data_ptr()),
                B.c_void_p(f['tabs'].data_ptr()), f['ntab'], 1 if self.root_search_truncation else 0,
                B.c_void_p(base.data_ptr()), base.shape[1], stream if stream is not None else self._stream()))
            return
        B.check(self._lib.ttm_inverse_fused(self._ctx, B.c_void_p(Xw.data_ptr()), ld, n, B.c_void_p(Zt.data_ptr()), ldz,
                                            f['ncomp'], f['c0'], f['ns'], B.c_void_p(f['A'].data_ptr()),
                                            B.c_void_p(f['a0'].data_ptr()), B.c_void_p(f['tabs'].data_ptr()), f['ntab'],
                                            1 if self.root_search_truncation else 0,
                                            stream if stream is not None else self._stream()))

    def _inverse_solver(self, comps, table_mode):
        """What _inverse_solve runs for the components `comps`: K-inv-fused with its operands, else one launch per
        component -- K-inv-table with its row of _monotone_tables, or K-inv-bisect.  Sets the coefficients the
        per-component launches read."""
        fused = self._inverse_fused_setup(comps) if table_mode else None
        if fused is not None:
            return {'fused': fused}
        if table_mode:
            return {'comps': comps, 'tabs': self._monotone_tables(comps)}
        for _, k in comps:
            self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
        return {'comps': comps, 'tabs': None}

    def _inverse_solve(self, solver, Xw, ld, n, Zt, ldz, stream, base=None):
        """The component loop of inverse_map (tm.py:3684-3698) on n samples: solves the columns of Xw (leading dimension
        ld) from the reference samples of component i at Zt + i*ldz.  Table mode: vectorized_root_search_alternate
        (:3987-4084); otherwise vectorized_root_search_bisection (:3798-3985), at most 100 iterations."""
        if 'fused' in solver:
            self._inverse_fused_launch(solver['fused'], Xw, ld, n, Zt, ldz, stream=stream, base=base)
            return
        xw, trunc, tabs = B.c_void_p(Xw.data_ptr()), 1 if self.root_search_truncation else 0, solver['tabs']
        sep = 1 if self.monotonicity.lower() == 'separable monotonicity' else 0
        for r, (i, k) in enumerate(solver['comps']):
            z = B.c_void_p(Zt.data_ptr() + i * ldz * 8)
            if tabs is not None:
                B.check(self._lib.ttm_inverse_table(self._plans[k], xw, ld, n, z, B.c_void_p(tabs[r].data_ptr()),
                                                    _TABLE_NTAB, trunc, stream))
                continue
            stalled = B.c_int(0)
            B.check(self._lib.ttm_inverse_bisect(self._plans[k], xw, ld, n, z, sep, 100, B.ctypes.byref(stalled), stream))
            if stalled.value and self.verbose:
                print('WARNING: root search for %d particles stopped at maximum iterations.' % stalled.value)

    def _inverse_map_pipelined(self, Z, X_star, E, ncol, comps):
        """Table-mode inverse_map for large sample counts.  Samples are independent (tm.py:3684-3698 loops over the
        components, never across samples), so the call is cut into chunks of samples that flow through four
        slots: host threads stage chunk c+1 into pinned memory (page-locked inputs are copied from directly) while
        chunk c is copied, transposed and solved and chunk c-1 is copied back.  The call is bound by the host->device
        copies (torch.profiler timeline: 16 copies of 168 MB at 52-58 GB/s back to back); four slots keep a copy from
        waiting for the slot's previous result to leave, and the last chunks are short so that little of the final
        solve + copy-back is exposed.  Bit-identical to the one-shot path."""
        from concurrent.futures import ThreadPoolExecutor
        torch, lib, dev = self._torch, self._lib, self._device
        N, nz, skip = Z.shape[0], Z.shape[1], self.skip_dimensions
        nout = ncol - skip
        std = self.standardize_samples
        solver = self._inverse_solver(comps, True)
        fused = solver.get('fused')
        mean_in = self._mean_d[:E].contiguous() if (std and E > 0) else None
        std_in = self._std_d[:E].contiguous() if (std and E > 0) else None
        mean_out = self._mean_d[skip:].contiguous() if std else None
        std_out = self._std_d[skip:].contiguous() if std else None
        torch.cuda.current_stream(dev).synchronize()
        nchunk = max(2, -(-N // int(os.environ.get('TTM_INV_CHUNK', 163840))))
        cap = -(-N // nchunk)
        # chunk boundaries: equal chunks, the last one cut into 1/2, 1/4, 1/4
        bounds = [min(N, c * cap) for c in range(nchunk + 1)]
        if nchunk >= 4 and bounds[-1] - bounds[-2] >= 64:
            lo, hi = bounds[-2], bounds[-1]
            q = (hi - lo) // 4
            bounds = bounds[:-1] + [lo + 2 * q, lo + 3 * q, hi]
        bounds = [b for i, b in enumerate(bounds) if i == 0 or b > bounds[i - 1]]
        nslot = min(4, len(bounds) - 1)
        f64 = torch.float64

        def pinned(a):                                       # caller's array already page-locked: DMA straight from it
            if a is None or not a.flags['C_CONTIGUOUS'] or a.dtype != np.float64:
                return False
            flag = B.c_int(0)
            B.check(lib.ttm_host_is_pinned(B.c_void_p(a.ctypes.data), B.ctypes.byref(flag)))
            return bool(flag.value)
        z_pinned, x_pinned = pinned(Z), pinned(X_star)
        slots = []
        for _ in range(nslot):
            slots.append({
                'stream': torch.cuda.Stream(device=dev), 'event': None,
                'hz': torch.empty((cap, nz), dtype=f64, pin_memory=True) if not z_pinned else None,
                'hx': torch.empty((cap, E), dtype=f64, pin_memory=True) if (E > 0 and not x_pinned) else None,
                'dz': torch.empty((cap, nz), dtype=f64, device=dev),
                'dx': torch.empty((cap, E), dtype=f64, device=dev) if E > 0 else None,
                'Xw': torch.empty((ncol, cap), dtype=f64, device=dev),
                'Zt': torch.empty((nz, cap), dtype=f64, device=dev),
                'base': (torch.empty((nz, (cap + 1) // 2 * 2), dtype=f64, device=dev)
                         if fused is not None and fused.get('R') is not None else None),
                'out': torch.empty((cap, nout), dtype=f64, device=dev)})
        out_host = torch.empty((N, nout), dtype=f64, pin_memory=True)
        ptr = lambda t: B.c_void_p(t.data_ptr()) if t is not None else None
        # host threads of the pageable -> pinned staging copies (memcpy-bound: ~8 GB/s per thread against 55 GB/s of PCIe)
        from .parallel import world as _world
        nthr = max(2, min(8, (os.cpu_count() or 8) // max(1, _world()[1])))

        def stage(dst, src, n):                              # pageable -> pinned, split over host threads
            edges = [n * t // nthr for t in range(nthr + 1)]
            return [pool.submit(np.copyto, dst[edges[t]:edges[t + 1]], src[edges[t]:edges[t + 1]])
                    for t in range(nthr) if edges[t + 1] > edges[t]]

        with ThreadPoolExecutor(nthr) as pool:
            for c in range(len(bounds) - 1):
                c0, c1 = bounds[c], bounds[c + 1]
                n = c1 - c0
                sl = slots[c % nslot]
                if sl['event'] is not None:
                    sl['event'].synchronize()                # the slot's previous chunk is back on the host
                futs = [] if z_pinned else stage(sl['hz'].numpy(), Z[c0:c1], n)
                if E > 0 and not x_pinned:
                    futs += stage(sl['hx'].numpy(), X_star[c0:c1], n)
                for f in futs:
                    f.result()
                src_z = torch.from_numpy(Z[c0:c1]) if z_pinned else sl['hz'][:n]
                src_x = (torch.from_numpy(X_star[c0:c1]) if x_pinned else sl['hx'][:n]) if E > 0 else None
                with torch.cuda.stream(sl['stream']):
                    st = self._stream()
                    sl['dz'][:n].copy_(src_z, non_blocking=True)
                    B.check(lib.ttm_standardize_transpose(self._ctx, ptr(sl['dz']), n, nz, None, None,
                                                          ptr(sl['Zt']), cap, st))
                    if E < skip:                             # unconditioned leading columns read as zero
                        sl['Xw'][E:skip].zero_()
                    if E > 0:
                        sl['dx'][:n].copy_(src_x, non_blocking=True)
                        B.check(lib.ttm_standardize_transpose(self._ctx, ptr(sl['dx']), n, E, ptr(mean_in), ptr(std_in),
                                                              ptr(sl['Xw']), cap, st))
                    self._inverse_solve(solver, sl['Xw'], cap, n, sl['Zt'], cap, st, base=sl['base'])
                    B.check(lib.ttm_transpose_back(self._ctx, B.c_void_p(sl['Xw'].data_ptr() + skip * cap * 8), cap, n,
                                                   nout, ptr(mean_out), ptr(std_out), ptr(sl['out']), nout, st))
                    out_host[c0:c1].copy_(sl['out'][:n], non_blocking=True)
                    sl['event'] = torch.cuda.Event()
                    sl['event'].record()
        for sl in slots:
            if sl['event'] is not None:
                sl['event'].synchronize()
        return out_host.numpy()

    # ================================================================== densities (separable only)
    def _log_det_accumulate(self, acc, Xraw_t, n, Zt, mode, std_offset):
        dS = self._empty(n)
        for k in range(self.D):
            self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
            # NB the reference evaluates the derivative basis on the UNstandardised samples (tm.py:2627, 2695)
            B.check(self._lib.ttm_sep_eval(self._plans[k], None, 0, n, None, B.c_void_p(Xraw_t.data_ptr()),
                                           Xraw_t.shape[1], B.c_void_p(dS.data_ptr()), self._stream()))
            sigma = float(self.X_std[k + std_offset]) if self.standardize_samples else None
            if sigma is None:
                sigma = float(self.X_std[k + std_offset])        # AttributeError like the reference
            B.check(self._lib.ttm_density_accumulate(self._ctx, B.c_void_p(acc.data_ptr()),
                                                     B.c_void_p(Zt[k].data_ptr()) if Zt is not None else None,
                                                     B.c_void_p(dS.data_ptr()), sigma, mode, n, self._stream()))

    def evaluate_pullback_density(self, X, X_star=None):
        """tm.py:2646-2712."""
        assert self.monotonicity == "separable monotonicity", "evaluate_pushforward_density is currently only implemented for monotonicity = 'separable monotonicity'."
        X = self._samples(X, ncol=self._Dtot if X_star is None else None)
        dev = isinstance(X, _DevSamples)
        X = self._stack(X_star, X)
        if dev and X.n == 0:
            return self._empty(0)
        if self._fused_small():
            return self._map_fused(X, 0, sigma=[float(self.X_std[k]) for k in range(self.D)])[1]   # X_std[k], tm.py:2706
        n = X.shape[0]
        torch = self._torch
        if self.standardize_samples:
            Xt = self._to_colmajor(X, self._mean_d, self._std_d)
        else:
            Xt, n = self._Xt, self._N
        Xraw_t = self._to_colmajor(X)
        Zt = self._empty(self.D, n)
        for k in range(self.D):
            self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
            self._s_device(k, Xt, n, Zt[k])
        acc = torch.zeros(n, dtype=torch.float64, device=self._device)
        self._log_det_accumulate(acc, Xraw_t, n, Zt, 0, 0)      # X_std[k] (not k+skip), tm.py:2706
        out = self._empty(n)
        B.check(self._lib.ttm_density_finish(self._ctx, B.c_void_p(acc.data_ptr()), None,
                                             B.c_void_p(out.data_ptr()), n, self._stream()))
        return self._result(out, dev)

    def _stack(self, X_star, X):
        """[X_star | X] (np.column_stack of tm.py:2614 / :2675) in the kind of X (host array or _DevSamples); with a
        CUDA X the column count is checked before the device copy."""
        if X_star is None:
            return X
        torch = self._torch
        if not isinstance(X, _DevSamples):
            if isinstance(X_star, torch.Tensor) and X_star.is_cuda:
                X_star = X_star.to(torch.float64).cpu().numpy()
            return np.column_stack((X_star, X))
        Xs = self._samples(X_star)
        if Xs.ndim != 2 or Xs.shape[1] + X.d != self._Dtot:
            raise ValueError('operands could not be broadcast together: X_star %s and X %s, the map has %d columns'
                             % (tuple(Xs.shape), tuple(X.shape), self._Dtot))
        xs = Xs.t if isinstance(Xs, _DevSamples) else self._upload(Xs)
        return self._samples(torch.cat((xs.to(torch.float64), X.t.to(torch.float64)), dim=1))

    def evaluate_pushforward_density(self, Z, log_target_pdf, X_star=None):
        """tm.py:2569-2644.  `log_target_pdf` is a user Python callback, called with the inverse-mapped samples: a
        host array, or a CUDA tensor when Z is one (it may then return a CUDA tensor or a host array of length n)."""
        assert self.monotonicity == "separable monotonicity", "evaluate_pushforward_density is currently only implemented for monotonicity = 'separable monotonicity'."
        torch = self._torch
        dev = isinstance(Z, torch.Tensor) and Z.is_cuda
        X = self.inverse_map(Z, X_star)
        n = X.shape[0]
        if dev and n == 0:
            return self._empty(0)
        log_target = log_target_pdf(X)
        if isinstance(log_target, torch.Tensor) and log_target.is_cuda:
            lt = log_target.to(self._device, torch.float64).reshape(-1).contiguous()
        else:
            lt = self._upload(np.ascontiguousarray(log_target, dtype=np.float64))
        if dev and lt.numel() != n:
            raise ValueError('log_target_pdf returned %d values for %d samples' % (lt.numel(), n))
        X = self._stack(X_star, self._samples(X) if dev else X)
        if self._fused_small():
            return self._map_fused(X, 1, sigma=[float(self.X_std[k + self.skip_dimensions]) for k in range(self.D)],
                                   log_target=lt)[1]                                  # X_std[k+skip], tm.py:2638
        Xraw_t = self._to_colmajor(X)
        acc = torch.zeros(n, dtype=torch.float64, device=self._device)
        self._log_det_accumulate(acc, Xraw_t, n, None, 1, self.skip_dimensions)   # X_std[k+skip], tm.py:2638
        out = self._empty(n)
        B.check(self._lib.ttm_density_finish(self._ctx, B.c_void_p(acc.data_ptr()), B.c_void_p(lt.data_ptr()),
                                             B.c_void_p(out.data_ptr()), n, self._stream()))
        return self._result(out, dev)

    # ================================================================== log densities (both monotonicity modes)
    def _log_sigma(self):
        """sigma_c = X_std[skip + k] per component (1 without standardisation)."""
        if not self.standardize_samples:
            return [1.0] * self.D
        return [float(self.X_std[k + self.skip_dimensions]) for k in range(self.D)]

    def _check_x_star(self, X_star, n):
        """X_star of the log-density evaluators: the conditioning columns of a partial map, (n, skip_dimensions)."""
        skip = self.skip_dimensions
        if X_star is None:
            return
        shape = tuple(X_star.shape) if hasattr(X_star, 'shape') else np.shape(X_star)
        if skip == 0 or len(shape) != 2 or shape[1] != skip or shape[0] != n:
            raise ValueError('X_star must have shape (%d, skip_dimensions = %d), got %s' % (n, skip, shape))

    def _log_det_terms(self, acc, Xt, n, mode):
        """acc += sum_k [-S_k^2/2 - log(2 pi)/2 + l_k - log sigma_c] (mode 0) or acc -= sum_k [l_k - log sigma_c]
        (mode 1) on the standardised column-major samples Xt, l_k = log d_c S_k."""
        ir = self.monotonicity == "integrated rectifier"
        S = self._empty(n) if mode == 0 else None
        dS = None if ir else self._empty(n)
        ptr = lambda t: B.c_void_p(t.data_ptr()) if t is not None else None
        st = self._stream()
        for k, sigma in enumerate(self._log_sigma()):
            self._set_coeffs(k, self.coeffs_nonmon[k], self.coeffs_mon[k])
            if S is not None:
                self._s_device(k, Xt, n, S)
            if ir:
                B.check(self._lib.ttm_ir_logdet_accumulate(self._plans[k], ptr(Xt), Xt.shape[1], n, ptr(S), sigma,
                                                           mode, ptr(acc), st))
            else:
                B.check(self._lib.ttm_sep_eval(self._plans[k], None, 0, n, None, ptr(Xt), Xt.shape[1], ptr(dS), st))
                B.check(self._lib.ttm_density_accumulate(self._ctx, ptr(acc), ptr(S), ptr(dS), sigma, mode, n, st))

    def _standardized_colmajor(self, X):
        if self.standardize_samples:
            return self._to_colmajor(X, self._mean_d, self._std_d)
        return self._to_colmajor(X)

    def evaluate_log_pullback_density(self, X, X_star=None):
        """log rho(x) = sum_k [-S_k(x~)^2/2 - log(2 pi)/2 + l_k(x~) - log sigma_c], the log density the fitted map pulls
        back from the standard Gaussian, for both monotonicity modes (DESIGN.md section 1).

        x are samples in the caller's units; x~ = (x - X_mean) / X_std with standardize_samples, else x~ = x and
        sigma = 1 (the X passed is used).  c = skip_dimensions + k, sigma_c = X_std[c], and l_k = log dS_k/dx~_c:
        integrated rectifier log(g(r_k(x~)) + delta), r_k = sum_j b_j psi^mon_j at the upper limit x~_c (r_k itself for
        the exponential rectifier with delta = 0); separable log(der_Psi_mon(x~) . b).  On the training ensemble
        -mean log rho = sum_k J_k + D/2 log(2 pi) + sum_k log sigma_c, J_k the objective optimize() minimises.
        With X_star ((n, skip_dimensions), partial maps only) the result is the conditional log density of X given
        X_star; X then has D columns, otherwise skip_dimensions + D.  X / X_star: host arrays or CUDA tensors; the
        result (n,) float64 follows X.  Unlike evaluate_pullback_density it returns the log (no underflow in high
        dimension) and differentiates the map it evaluates."""
        X = self._samples(X, ncol=self._Dtot if X_star is None else self.D)
        dev = isinstance(X, _DevSamples)
        if X.ndim != 2 or X.shape[1] != (self._Dtot if X_star is None else self.D):
            raise ValueError('X has shape %s; the map expects %d columns' %
                             (tuple(X.shape), self._Dtot if X_star is None else self.D))
        n = X.shape[0]
        self._check_x_star(X_star, n)
        if n == 0:
            return self._empty(0) if dev else np.empty(0)
        X = self._stack(X_star, X)
        if self._fused_small():
            return self._map_fused(X, 3, sigma=self._log_sigma())[1]
        Xt = self._standardized_colmajor(X)
        acc = self._torch.zeros(n, dtype=self._torch.float64, device=self._device)
        self._log_det_terms(acc, Xt, n, 0)
        return self._result(acc, dev)

    def evaluate_log_pushforward_density(self, Z, log_target_pdf, X_star=None):
        """log p(z) = log_target_pdf(x) - sum_k [l_k(x~) - log sigma_c], x = inverse_map(Z, X_star): the log density of
        the samples the map pushes forward from `log_target_pdf`, for both monotonicity modes (l_k, sigma_c and X_star
        as in evaluate_log_pullback_density).  `log_target_pdf` is called with the inverse-mapped samples (n, D) in the
        caller's units: a host array, or a CUDA tensor when Z is one; it returns n values (host array or CUDA
        tensor).  The result (n,) float64 follows Z."""
        torch = self._torch
        Z = self._samples(Z, ncol=self.D)
        dev = isinstance(Z, _DevSamples)
        if Z.ndim != 2 or Z.shape[1] != self.D:
            raise ValueError('Z has shape %s; the map has %d components' % (tuple(Z.shape), self.D))
        n = Z.shape[0]
        self._check_x_star(X_star, n)
        if n == 0:
            return self._empty(0) if dev else np.empty(0)
        X = self.inverse_map(Z, X_star)
        log_target = log_target_pdf(X)
        if isinstance(log_target, torch.Tensor) and log_target.is_cuda:
            lt = log_target.to(self._device, torch.float64).reshape(-1).contiguous()
        else:
            lt = self._upload(np.ascontiguousarray(log_target, dtype=np.float64).reshape(-1))
        if lt.numel() != n:
            raise ValueError('log_target_pdf returned %d values for %d samples' % (lt.numel(), n))
        X = self._stack(X_star, self._samples(X) if dev else X)
        if self._fused_small():
            return self._map_fused(X, 4, sigma=self._log_sigma(), log_target=lt)[1]
        Xt = self._standardized_colmajor(X)
        acc = lt.clone()
        self._log_det_terms(acc, Xt, n, 1)
        return self._result(acc, dev)

    # ================================================================== measurement helpers
    def fp64_peak_tflops(self):
        v = B.c_double(0.0)
        B.check(self._lib.ttm_fp64_peak(self._ctx, B.ctypes.byref(v)))
        return v.value
