"""evaluate_log_pullback_density / evaluate_log_pushforward_density on the GPU, both monotonicity modes: against the
restatement in tests/log_density_oracle.py of the definition (DESIGN.md section 1) and against identities that hold whatever the
quirks of the reference's evaluators -- the objective optimize() minimises, the normalisation of the density, and
pushforward(pullback) = the reference Gaussian."""

import copy
import os

import numpy as np
import pytest

from cases import c4_terms, cases, ex01_terms, ex05_terms, fresh_kwargs, synthetic_samples
from ttm_oracle import OracleMap
import log_density_oracle as LD

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
CASES = cases()
TOL_BISECT = 2e-8     # both inverses stop on a 1e-9 residual
TOL_TABLE = 1e-10


def _tm(X, **kw):
    from transport_map import transport_map
    return transport_map(X=X, **kw)


def _log_gauss(X):
    X = np.asarray(X)
    return -0.5 * np.sum(X ** 2, axis=1) - 0.5 * X.shape[1] * np.log(2 * np.pi)


def _rel(a, b):
    """max |a-b| / max(1, |b|) over the finite entries; NaN and +-inf (maps with random coefficients whose inverse
    runs off to |x| ~ 1e16, where -|x|^2/2 overflows) must sit at the same places on both sides."""
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    assert a.shape == b.shape, (a.shape, b.shape)
    fin = np.isfinite(b)
    assert np.array_equal(np.isfinite(a), fin)
    assert np.array_equal(a[~fin], b[~fin], equal_nan=True)
    if not fin.any():
        return 0.0
    return float(np.max(np.abs(a[fin] - b[fin]) / np.maximum(1.0, np.abs(b[fin]))))


def _impose(m, src):
    for k in range(m.D):
        m.coeffs_mon[k] = np.array(src['coeffs_mon_%d' % k])
        m.coeffs_nonmon[k] = np.array(src['coeffs_nonmon_%d' % k])


def _set_coeffs(m, coeffs):
    for k, (cn, cm) in enumerate(coeffs):
        m.coeffs_nonmon[k], m.coeffs_mon[k] = cn.copy(), cm.copy()


def _random_ir_coeffs(m, seed, scale=0.05):
    rng = np.random.default_rng(seed)
    out = []
    for k in range(m.D):
        c = rng.standard_normal(len(m.coeffs_nonmon[k]) + len(m.coeffs_mon[k])) * scale
        out.append((c[:len(m.coeffs_nonmon[k])], c[len(m.coeffs_nonmon[k]):]))
    return out


# ---------------------------------------------------------------------------------------------- 1. oracle parity
PARITY = [(n, '1') for n in sorted(CASES)] + \
         [(n, '0') for n in sorted(CASES) if CASES[n]['kwargs']['monotonicity'].startswith('sep')]


@pytest.mark.parametrize('name,fused', PARITY)
def test_log_densities_match_oracle(name, fused, monkeypatch):
    """Fixture coefficients imposed on both sides; separable maps through K-map-fused (fused = 1, where the map is
    small enough) and through the per-component kernels (fused = 0)."""
    case = CASES[name]
    monkeypatch.setenv('TTM_MAP_FUSED', fused)
    gold = np.load(os.path.join(GOLD, name + '.npz'))
    tm, om = _tm(copy.copy(case['X']), **fresh_kwargs(case)), OracleMap(copy.copy(case['X']), **fresh_kwargs(case))
    if 'reset_X' in case:
        tm.reset(copy.copy(case['reset_X']))
        om.reset(copy.copy(case['reset_X']))
    _impose(tm, gold)
    _impose(om, gold)
    Xref = case.get('reset_X', case['X'])
    Dtot, D = Xref.shape[1], tm.D
    skip = Dtot - D
    rng = np.random.default_rng(4321)
    Xe = Xref.mean(axis=0) + Xref.std(axis=0) * rng.standard_normal((96, Dtot))
    Xs = Xe[:, :skip].copy() if skip else None
    lp = tm.evaluate_log_pullback_density(Xe[:, skip:].copy(), X_star=Xs)
    lpo = LD.log_pullback_density(om, Xe[:, skip:].copy(), X_star=Xs)
    assert lp.shape == (96,)
    assert _rel(lp, lpo) <= 1e-10, (name, _rel(lp, lpo))
    Zd = rng.standard_normal((96, D))
    table = tm.alternate_root_finding and tm.monotonicity.startswith('sep')
    lq = tm.evaluate_log_pushforward_density(Zd.copy(), _log_gauss, X_star=Xs)
    lqo = LD.log_pushforward_density(om, Zd.copy(), _log_gauss, X_star=Xs)
    assert _rel(lq, lqo) <= (TOL_TABLE if table else TOL_BISECT), (name, _rel(lq, lqo))


# ---------------------------------------------------------------------------------------------- 2. objective identity
def _objective_identity(tm, X, coeffs):
    _set_coeffs(tm, coeffs)
    lp = tm.evaluate_log_pullback_density(X)
    c = np.arange(tm.D) + tm.skip_dimensions
    lhs = -np.mean(lp) - tm.D / 2 * np.log(2 * np.pi) - np.sum(np.log(tm.X_std[c]))
    rhs = sum(tm.objective_function(np.concatenate(coeffs[k]), k, len(coeffs[k][0])) for k in range(tm.D))
    assert abs(lhs - rhs) <= 1e-12 * abs(rhs), (lhs, rhs)


def test_objective_identity_c4_d8():
    mon, non = c4_terms(8)
    X = synthetic_samples(20000, 8, seed=41)
    tm = _tm(X.copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': 30}, verbose=False)
    _objective_identity(tm, X, _random_ir_coeffs(tm, 42))


def test_objective_identity_example01_shipped_coefficients():
    ka = np.load(os.path.join(GOLD, 'ex01_known_answer.npz'))
    mon, non = ex01_terms(10)
    tm = _tm(ka['X'].copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': 25}, verbose=False)
    coeffs = [(ka['full_coeffs_%d' % k][:int(ka['full_div_%d' % k])], ka['full_coeffs_%d' % k][int(ka['full_div_%d' % k]):])
              for k in range(2)]
    _objective_identity(tm, ka['X'], coeffs)


@pytest.mark.parametrize('name', ['ir_softplus_l1', 'ir_softplus_l2'])
def test_objective_identity_softplus(name):
    case = CASES[name]
    kw = fresh_kwargs(case)
    kw['regularization'] = None
    tm = _tm(case['X'].copy(), **kw)
    _objective_identity(tm, case['X'], _random_ir_coeffs(tm, 43, scale=0.3))


# ---------------------------------------------------------------------------------------------- 3. normalisation
def test_example01_density_integrates_to_one():
    """Example-01 spiral map (D = 2, order 10, Q = 25, shipped coefficients).  Trapezoid rule on a 1000 x 1000 grid
    (10^6 points) over the box x0 in [-3, 3.5], x1 in [-3.5, 3] (the ensemble spans [-2.3, 2.7] x [-2.4, 2.1]); the
    density is below 1e-8 on the box's edge.  Measured: 1 - 4.88e-4, the same with the box 0.5 wider on every side and
    with a 1400 x 1400 grid, so the deficit is not truncation or grid error.  It comes from Q = 25 quadrature of the
    extrapolated second component: S_1 is a 25-node sum while l_1 is the log of its exact derivative, and far from the
    ensemble the order-10 exponent makes exp(r) too peaked for 25 nodes (at x0 = -2 the conditional density of x1
    carries 7 % spurious mass near x1 = -5; over [-6, 6]^2 the integral is 1.065)."""
    ka = np.load(os.path.join(GOLD, 'ex01_known_answer.npz'))
    mon, non = ex01_terms(10)
    tm = _tm(ka['X'].copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': 25}, verbose=False)
    for k in range(2):
        c, div = ka['full_coeffs_%d' % k], int(ka['full_div_%d' % k])
        tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:div].copy(), c[div:].copy()
    g0, g1 = np.linspace(-3.0, 3.5, 1000), np.linspace(-3.5, 3.0, 1000)
    XX = np.stack(np.meshgrid(g0, g1, indexing='xy'), -1).reshape(-1, 2)
    p = np.exp(tm.evaluate_log_pullback_density(XX)).reshape(1000, 1000)          # p[i1, i0]
    assert max(p[0].max(), p[-1].max(), p[:, 0].max(), p[:, -1].max()) < 1e-8
    total = np.trapezoid(np.trapezoid(p, g0, axis=1), g1)
    print('Example-01 normalisation: 1 %+.3e' % (total - 1.0))
    assert abs(total - 1.0) <= 1e-3, total


# ---------------------------------------------------------------------------------------------- 4. push(pull) = Gaussian
def _gauss_check(tm, Z, X_star=None):
    cb = (lambda x: tm.evaluate_log_pullback_density(x, X_star))
    lq = tm.evaluate_log_pushforward_density(Z, cb, X_star=X_star)
    ref = _log_gauss(Z)
    err = float(np.max(np.abs(lq - ref)))
    assert err <= 1e-7, err


def test_pushforward_of_pullback_is_gaussian_c4():
    mon, non = c4_terms(4)
    X = synthetic_samples(50000, 4, seed=44)
    tm = _tm(X.copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': 25}, verbose=False)
    _set_coeffs(tm, _random_ir_coeffs(tm, 45))
    _gauss_check(tm, np.random.default_rng(46).standard_normal((50000, 4)))


def test_pushforward_of_pullback_is_gaussian_partial_ir():
    ka = np.load(os.path.join(GOLD, 'ex01_known_answer.npz'))
    mon, non = ex01_terms(10)
    tm = _tm(ka['X'].copy(), monotone=mon[1:], nonmonotone=non[1:], quadrature_input={'order': 25}, verbose=False)
    c, div = ka['partial_coeffs_0'], int(ka['partial_div_0'])
    tm.coeffs_nonmon[0], tm.coeffs_mon[0] = c[:div].copy(), c[div:].copy()
    n = 4000
    _gauss_check(tm, np.random.default_rng(47).standard_normal((n, 1)), X_star=ka['X'][:n, :1].copy())


def test_pushforward_of_pullback_is_gaussian_separable_bisection():
    gold = np.load(os.path.join(GOLD, 'sep_ex05.npz'))
    case = CASES['sep_ex05']
    tm = _tm(case['X'].copy(), **fresh_kwargs(case))
    _impose(tm, gold)
    tm.alternate_root_finding = False
    _gauss_check(tm, np.random.default_rng(48).standard_normal((2000, 2)))


# ---------------------------------------------------------------------------------------------- 5. existing API
def test_log_of_existing_pullback_on_standardised_ensemble():
    gold = np.load(os.path.join(GOLD, 'sep_ex05.npz'))
    X5 = CASES['sep_ex05']['X']
    Xs = (X5 - X5.mean(axis=0)) / X5.std(axis=0)
    mon, non = ex05_terms()
    tm = _tm(Xs.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity', verbose=False)
    _impose(tm, gold)
    Xe = np.random.default_rng(49).standard_normal((500, 2))
    a, b = np.log(tm.evaluate_pullback_density(Xe.copy())), tm.evaluate_log_pullback_density(Xe.copy())
    assert np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))) <= 1e-12


# ---------------------------------------------------------------------------------------------- 6. input kinds, errors
def _maps():
    mon, non = c4_terms(4)
    X = synthetic_samples(3000, 4, seed=50)
    ir = _tm(X.copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': 25}, verbose=False)
    _set_coeffs(ir, _random_ir_coeffs(ir, 51))
    gold = np.load(os.path.join(GOLD, 'sep_c5_d6.npz'))
    case = CASES['sep_c5_d6']
    sep = _tm(case['X'].copy(), **fresh_kwargs(case))
    _impose(sep, gold)
    return [ir, sep]


def test_cuda_tensors_float32_and_views():
    import torch
    for tm in _maps():
        Dt = tm.skip_dimensions + tm.D
        X = np.random.default_rng(52).standard_normal((700, Dt))
        Z = np.random.default_rng(53).standard_normal((300, tm.D))
        ref = tm.evaluate_log_pullback_density(X)
        got = tm.evaluate_log_pullback_density(torch.from_numpy(X).cuda())
        assert got.is_cuda and got.dtype == torch.float64
        assert np.array_equal(got.cpu().numpy(), ref)
        target = lambda x: 0.5 * x[:, 0] - 1.0           # elementwise: the same bits from numpy and torch
        refq = tm.evaluate_log_pushforward_density(Z, target)
        gotq = tm.evaluate_log_pushforward_density(torch.from_numpy(Z).cuda(), target)
        assert gotq.is_cuda
        assert np.array_equal(gotq.cpu().numpy(), refq)
        X32 = torch.from_numpy(X).float().cuda()
        assert np.array_equal(tm.evaluate_log_pullback_density(X32).cpu().numpy(),
                              tm.evaluate_log_pullback_density(X32.cpu().double().numpy()))
        wide = torch.from_numpy(np.random.default_rng(54).standard_normal((700, Dt + 3))).cuda()
        view = wide[:, 2:2 + Dt]
        assert np.array_equal(tm.evaluate_log_pullback_density(view).cpu().numpy(),
                              tm.evaluate_log_pullback_density(view.cpu().numpy()))


def test_empty_and_errors():
    import torch
    for tm in _maps():
        Dt = tm.skip_dimensions + tm.D
        assert tm.evaluate_log_pullback_density(np.zeros((0, Dt))).shape == (0,)
        e = tm.evaluate_log_pullback_density(torch.zeros((0, Dt), dtype=torch.float64, device='cuda'))
        assert e.is_cuda and e.shape == (0,)
        assert tm.evaluate_log_pushforward_density(np.zeros((0, tm.D)), _log_gauss).shape == (0,)
        for bad in (np.zeros((5, Dt + 1)), torch.zeros((5, Dt - 1), dtype=torch.float64, device='cuda')):
            with pytest.raises(ValueError):
                tm.evaluate_log_pullback_density(bad)
        with pytest.raises(ValueError):
            tm.evaluate_log_pushforward_density(np.zeros((5, tm.D + 1)), _log_gauss)
        with pytest.raises(ValueError):                                   # a full map takes no X_star
            tm.evaluate_log_pullback_density(np.zeros((5, tm.D)), X_star=np.zeros((5, 1)))
        with pytest.raises(ValueError):
            tm.evaluate_log_pushforward_density(np.zeros((5, tm.D)), _log_gauss, X_star=np.zeros((5, 1)))
        with pytest.raises(ValueError):                                   # callback of the wrong length
            tm.evaluate_log_pushforward_density(np.zeros((5, tm.D)), lambda x: np.zeros(4))


# ---------------------------------------------------------------------------------------------- 7. full size
def test_full_size_c4_d64():
    import torch
    D, N = 64, 1_000_000
    mon, non = c4_terms(D)
    X = torch.from_numpy(synthetic_samples(N, D, seed=55)).cuda()
    tm = _tm(X, monotone=mon, nonmonotone=non, quadrature_input={'order': 100}, verbose=False)
    rng = np.random.default_rng(56)
    for k in range(D):
        m = len(non[k]) + len(mon[k])
        c = rng.standard_normal(m) * 0.05
        tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:len(non[k])].copy(), c[len(non[k]):].copy()
    a = tm.evaluate_log_pullback_density(X)
    b = tm.evaluate_log_pullback_density(X)
    assert bool(torch.isfinite(a).all())
    assert torch.equal(a, b)
    head = tm.evaluate_log_pullback_density(X[:1000])
    assert torch.equal(head, a[:1000])
