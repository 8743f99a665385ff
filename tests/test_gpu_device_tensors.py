"""CUDA tensors as inputs and outputs of the public map API.

A call on a CUDA tensor runs the same kernels on the same operands as the call on a numpy array with the same
values, so every result must be bit-identical (np.array_equal), not merely close.  Results are float64 CUDA
tensors on the map's device; inputs are never modified; once the coefficient-sized operands are cached, a call
copies nothing sample-sized between host and device."""

import json

import numpy as np
import pytest
import torch

from cases import cases, fresh_kwargs, synthetic_samples, c4_terms, c5_terms
from harness import run_case

pytestmark = pytest.mark.gpu

CASES = cases()


def make_cuda(X, **kw):
    from transport_map import transport_map
    return transport_map(X=X, **kw)


def cuda(a):
    return torch.from_numpy(np.array(a, dtype=np.float64)).cuda()


def back(tm, r):
    """A device result -> numpy, after checking that it is what the API promises."""
    assert isinstance(r, torch.Tensor) and r.is_cuda, type(r)
    assert r.dtype == torch.float64 and r.device == tm._device and r.is_contiguous()
    return r.cpu().numpy()


class DeviceWrapped:
    """The drop-in class driven with CUDA tensors wherever it accepts samples; results come back as numpy so that
    tests/harness.py can compare them with the host-array run."""

    def __init__(self, X, **kw):
        object.__setattr__(self, '_tm', make_cuda(cuda(X), **kw))

    def __getattr__(self, name):
        return getattr(self._tm, name)

    def __setattr__(self, name, value):
        setattr(self._tm, name, value)

    def _star(self, X_star):
        return None if X_star is None else cuda(X_star)

    def reset(self, X):
        self._tm.reset(cuda(X))

    def map(self, X=None):
        return self._tm.map() if X is None else back(self._tm, self._tm.map(cuda(X)))

    def inverse_map(self, Z, X_star=None):
        return back(self._tm, self._tm.inverse_map(cuda(Z), self._star(X_star)))

    def evaluate_pullback_density(self, X, X_star=None):
        return back(self._tm, self._tm.evaluate_pullback_density(cuda(X), self._star(X_star)))

    def evaluate_pushforward_density(self, Z, log_target_pdf, X_star=None):
        def on_device(x):
            assert isinstance(x, torch.Tensor) and x.is_cuda
            return log_target_pdf(x.cpu().numpy())
        return back(self._tm, self._tm.evaluate_pushforward_density(cuda(Z), on_device, self._star(X_star)))


@pytest.mark.parametrize('name', sorted(CASES))
def test_every_case_bit_identical_through_cuda_tensors(name):
    case = CASES[name]
    ref = run_case(make_cuda, case)
    got = run_case(DeviceWrapped, case)
    assert set(got) == set(ref)
    for key in ref:
        assert np.array_equal(got[key], ref[key]), (name, key)


# ---------------------------------------------------------------------------------------------- views and float32
def _unchanged(*pairs):
    for t, before in pairs:
        assert torch.equal(t, before)


def _ex06_map():
    case = CASES['sep_ex06_cycle']
    tm = make_cuda(case['X'].copy(), **fresh_kwargs(case))
    tm.reset(case['reset_X'].copy())
    tm.optimize()
    return tm, case['reset_X']


def test_views_and_float32_ex06_cycle():
    tm, X = _ex06_map()                                  # skip_dimensions = 1, K-map-fused path
    assert tm.skip_dimensions == 1 and tm._fused_small()
    rng = np.random.default_rng(3)
    Zfull = rng.standard_normal((X.shape[0], 4))
    Xd, Zd = cuda(X), cuda(Zfull)
    Xc, Zc = Xd.clone(), Zd.clone()
    # the same elementwise operations on numpy arrays and on tensors (a reduction need not sum in the same order)
    lg = lambda x: -0.5 * (x[:, 0] * x[:, 0] + x[:, 1] * x[:, 1] + x[:, 2] * x[:, 2])

    assert np.array_equal(back(tm, tm.map(Xd)), tm.map(X))
    assert np.array_equal(back(tm, tm.inverse_map(Zd[:, 1:], Xd[:, :1])),
                          tm.inverse_map(np.ascontiguousarray(Zfull[:, 1:]), np.ascontiguousarray(X[:, :1])))
    assert np.array_equal(back(tm, tm.evaluate_pullback_density(Xd[:, 1:], X_star=Xd[:, :1])),
                          tm.evaluate_pullback_density(np.ascontiguousarray(X[:, 1:]), X_star=X[:, :1].copy()))
    host = tm.evaluate_pushforward_density(np.ascontiguousarray(Zfull[:, 1:]), lg, X_star=X[:, :1].copy())
    assert np.array_equal(back(tm, tm.evaluate_pushforward_density(Zd[:, 1:], lg, X_star=Xd[:, :1])), host)
    assert np.array_equal(back(tm, tm.evaluate_pushforward_density(Zd[:, 1:], lambda x: lg(x.cpu().numpy()),
                                                                X_star=X[:, :1].copy())), host)
    for k in range(tm.D):
        assert np.array_equal(back(tm, tm.s(Xd, k)), tm.s(X, k))

    X32 = X.astype(np.float32).astype(np.float64)
    assert np.array_equal(back(tm, tm.map(Xd.float())), tm.map(X32))
    assert np.array_equal(back(tm, tm.evaluate_pullback_density(Xd[:, 1:].float(), X_star=Xd[:, :1].float())),
                          tm.evaluate_pullback_density(np.ascontiguousarray(X32[:, 1:]), X_star=X32[:, :1].copy()))

    Xt = cuda(X.T.copy()).T                               # column stride N: read through the conversion
    assert Xt.stride(1) != 1
    assert np.array_equal(back(tm, tm.map(Xt)), tm.map(X))
    _unchanged((Xd, Xc), (Zd, Zc))


def test_views_and_float32_ir_c4():
    D, N = 4, 3000
    W = synthetic_samples(N, D + 1, seed=12)              # leading extra column: W[:, 1:] is a strided view
    X = np.ascontiguousarray(W[:, 1:])
    mon, non = c4_terms(D)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='integrated rectifier', quadrature_input={'order': 20},
              verbose=False)
    Wd = cuda(W)
    Wc = Wd.clone()
    host = make_cuda(X.copy(), **kw)
    view = make_cuda(Wd[:, 1:], **kw)
    for a in ('X', 'X_mean', 'X_std'):
        assert np.array_equal(getattr(view, a), getattr(host, a)), a
        assert isinstance(getattr(view, a), np.ndarray)
    rng = np.random.default_rng(7)
    for k in range(D):
        div = len(host.coeffs_nonmon[k])
        c = rng.standard_normal(div + len(host.coeffs_mon[k])) * 0.2
        for tm in (host, view):
            tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:div].copy(), c[div:].copy()
    assert np.array_equal(back(view, view.map(Wd[:, 1:])), host.map(X))
    Z = host.map(X[:200])
    Zw = cuda(np.column_stack((Z, np.zeros(200))))
    assert np.array_equal(back(view, view.inverse_map(Zw[:, :D])), host.inverse_map(Z))
    for k in range(D):
        assert np.array_equal(back(view, view.s(Wd[:, 1:], k)), host.s(X, k))

    X32 = X.astype(np.float32).astype(np.float64)
    h32 = make_cuda(X32.copy(), **kw)
    d32 = make_cuda(Wd[:, 1:].float(), **kw)
    for a in ('X', 'X_mean', 'X_std'):
        assert np.array_equal(getattr(d32, a), getattr(h32, a)), a
    d32.reset(Wd[:, 1:].float())
    h32.reset(X32.copy())
    assert np.array_equal(d32.X_std, h32.X_std)
    assert np.array_equal(back(view, view.map(Wd[:, 1:].float())), host.map(X32))
    h32.X = X32[:500].copy()
    d32.X = Wd[:500, 1:].float()
    assert np.array_equal(d32.X, h32.X)
    _unchanged((Wd, Wc))


# ---------------------------------------------------------------------------------------------- large / wide shapes
def _c5_map(D, ntrain, seed, fit=True):
    mon, non = c5_terms(D)
    tm = make_cuda(synthetic_samples(ntrain, D, seed=seed), monotone=mon, nonmonotone=non,
                   monotonicity='separable monotonicity', verbose=False)
    if fit:
        tm.optimize()
    else:
        rng = np.random.default_rng(seed)
        for k in range(D):
            tm.coeffs_nonmon[k] = rng.standard_normal(len(tm.coeffs_nonmon[k])) * 0.05
            tm.coeffs_mon[k] = np.abs(rng.standard_normal(len(tm.coeffs_mon[k]))) * 0.2 + 0.05
    return tm


def test_table_inverse_one_shot_matches_pipelined():
    D, E, N = 24, 12, 140_000
    tm = _c5_map(D, 2000, seed=3)
    Xs = synthetic_samples(N, D, seed=4)[:, :E].copy()
    Z = np.random.default_rng(1).standard_normal((N, D - E))
    host = tm.inverse_map(Z, X_star=Xs)                  # N >= TTM_INV_PIPELINE_MIN: the pipelined path
    assert np.array_equal(back(tm, tm.inverse_map(cuda(Z), X_star=cuda(Xs))), host)
    assert np.array_equal(back(tm, tm.inverse_map(cuda(Z), X_star=Xs)), host)


def test_wide_separable_map_rect_path():
    D, n = 34, 5000
    tm = _c5_map(D, 1000, seed=5, fit=False)
    assert tm._map_gemm_static() is not None
    X = synthetic_samples(n, D, seed=6)
    assert np.array_equal(back(tm, tm.map(cuda(X))), tm.map(X))


# ---------------------------------------------------------------------------------------------- copies
def _memcpy_bytes(prof, path):
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        ev = json.load(f)['traceEvents']
    assert any(e.get('cat') == 'kernel' for e in ev)
    return [int(e.get('args', {}).get('bytes', 0)) for e in ev if e.get('cat') == 'gpu_memcpy']


def test_no_sample_sized_copies(tmp_path):
    from torch.profiler import profile, ProfilerActivity
    wide = _c5_map(34, 1000, seed=5, fit=False)
    tm = _c5_map(24, 2000, seed=3)
    E, n = 12, 400_000
    Xw = cuda(synthetic_samples(262_144, 34, seed=8))                 # 71 MB
    Xs = cuda(synthetic_samples(n, 24, seed=9))                       # 77 MB
    Z = torch.randn(n, 12, dtype=torch.float64, device='cuda')
    calls = [('map', lambda: wide.map(Xw), Xw.numel() * 8),
             ('inverse', lambda: tm.inverse_map(Z, X_star=Xs[:, :E]), (Z.numel() + n * E) * 8),
             ('pullback', lambda: tm.evaluate_pullback_density(Xs), Xs.numel() * 8)]
    for name, fn, nbytes in calls:
        fn()                                                          # warm-up: tables, packed operands
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        sizes = _memcpy_bytes(prof, tmp_path / ('%s.json' % name))
        assert max(sizes, default=0) <= 4 << 20, (name, max(sizes))
        assert sum(sizes) < 0.1 * nbytes, (name, sum(sizes), nbytes)


# ---------------------------------------------------------------------------------------------- streams
def test_side_stream_results_equal_default_stream():
    tm = _c5_map(24, 2000, seed=3)
    X = cuda(synthetic_samples(20_000, 24, seed=10))
    Z = torch.randn(20_000, 12, dtype=torch.float64, device='cuda')
    ref = [tm.map(X), tm.inverse_map(Z, X_star=X[:, :12]), tm.evaluate_pullback_density(X)]
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = [tm.map(X), tm.inverse_map(Z, X_star=X[:, :12]), tm.evaluate_pullback_density(X)]
        got = [g * 1.0 for g in got]                                  # consumed on s, no synchronise in between
    s.synchronize()
    for g, r in zip(got, ref):
        assert torch.equal(g, r)


# ---------------------------------------------------------------------------------------------- errors, edges
def test_shape_errors_and_empty_inputs():
    tm, X = _ex06_map()
    Dtot, D = X.shape[1], tm.D
    Xd = cuda(X)
    for bad in (Xd[:, 0], Xd[:, :2]):
        with pytest.raises(ValueError):
            tm.map(bad)
        with pytest.raises(ValueError):
            tm.evaluate_pullback_density(bad)
        with pytest.raises(ValueError):
            tm.s(bad, 0)
    with pytest.raises(ValueError):
        tm.inverse_map(cuda(np.zeros((8, D + 1))), X_star=Xd[:8, :1])
    with pytest.raises(ValueError):
        tm.inverse_map(cuda(np.zeros((8, D))), X_star=Xd[:9, :1])
    with pytest.raises(ValueError, match='two-dimensional'):
        tm.reset(Xd[:, 0])
    with pytest.raises(ValueError):                       # host array on the K-map-fused path: checked, not read
        tm.map(np.zeros((8, Dtot + 3)))
    with pytest.raises(ValueError):
        tm.evaluate_pullback_density(np.zeros((8, Dtot - 2)), X_star=X[:8, :1])

    empty = torch.empty((0, Dtot), dtype=torch.float64, device='cuda')
    for r, shape in ((tm.map(empty), (0, D)), (tm.s(empty, 0), (0,)),
                     (tm.inverse_map(empty[:, 1:], X_star=empty[:, :1]), (0, D)),
                     (tm.evaluate_pullback_density(empty[:, 1:], X_star=empty[:, :1]), (0,))):
        assert isinstance(r, torch.Tensor) and r.is_cuda and tuple(r.shape) == shape
    assert tuple(tm.inverse_map(empty[:, 1:]).shape) == (0, D)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_tensor_on_another_device_is_rejected():
    tm, X = _ex06_map()
    other = torch.from_numpy(X).to('cuda:1')
    with pytest.raises(ValueError, match='device|cuda'):
        tm.map(other)
