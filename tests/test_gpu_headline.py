"""GPU parity at the HEADLINE shapes (BASELINE.json configs C4 and C5 at their real dimensions), against fixtures
produced by the unmodified reference (tests/golden/make_golden_headline.py) and against the CPU oracle.

  * C4, D=64 (m_non up to 190, 63 dense groups), N=4000: J_k and grad J_k for k in {0,1,5,31,63}, Q in {25,100},
    through every kernel form (tile kernel with and without the Gram identity, general kernel): <= 1e-10;
  * full D=64 optimize() at N=4000, Q=100 against the reference's BFGS fit: objective at the optimum, fitted
    coefficients and map() output (north_star: "fitted ... matching the reference within tolerance");
  * separable fit at D=64 and D=128 (m_non up to 382) against the reference's Householder-QR path;
  * C5 at D=256: table and bisection inverse_map with E=128 conditioning columns against the reference.
"""

import os

import numpy as np
import pytest

from cases import (synthetic_samples, c4_terms, c5_terms, headline_coeffs, headline_sep_coeffs, HEADLINE_N,
                   HEADLINE_KS, HEADLINE_QS, C5_INV)
from harness import rel_err

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TOL_OBJ = 1e-10
TOL_FIT = 1e-6


def make_cuda(X, **kw):
    from transport_map import transport_map
    return transport_map(X=X, verbose=False, **kw)


def _set_kernel(tm, general):
    from ttt_b200 import binding as B
    B.check(tm._lib.ttm_ctx_set_objgrad_kernel(tm._ctx, 1 if general else 0))
    tm._fg_cache = {}


@pytest.mark.parametrize('Q', HEADLINE_QS)
@pytest.mark.parametrize('form', ['tile_gram', 'tile_two_sweeps', 'general'])
def test_c4_objgrad_at_d64_matches_reference(Q, form, monkeypatch):
    """tm.py:3300-3635 at the real C4 shape: k = 63 has 190 nonmonotone + 4 monotone terms."""
    gold = np.load(os.path.join(GOLD, 'headline_c4_objgrad.npz'))
    if form == 'tile_two_sweeps':
        monkeypatch.setenv('TTM_GRAM', '0')
    D = 64
    mon, non = c4_terms(D)
    tm = make_cuda(synthetic_samples(HEADLINE_N, D, seed=0), monotone=mon, nonmonotone=non,
                   polynomial_type='hermite function', monotonicity='integrated rectifier',
                   quadrature_input={'order': Q})
    _set_kernel(tm, form == 'general')
    assert all(info['tile_ok'] for info in tm._plan_info)
    for k in HEADLINE_KS:
        c = headline_coeffs(mon, non, k)
        div = len(non[k])
        J = tm.objective_function(c.copy(), k, div)
        g = tm.objective_function_jacobian(c.copy(), k, div)
        assert rel_err(J, gold['J_q%d_k%d' % (Q, k)]) <= TOL_OBJ, (form, Q, k)
        assert rel_err(g, gold['grad_q%d_k%d' % (Q, k)]) <= TOL_OBJ, (form, Q, k, rel_err(g, gold['grad_q%d_k%d' % (Q, k)]))
        assert (tm._gram_nonmon(k) is not None) == (form != 'tile_two_sweeps')


def test_c4_value_kernel_at_d64_matches_oracle():
    """map() (K-S, value-only form of the tile kernel) at D=64 against the CPU oracle on 300 rows."""
    from ttm_oracle import OracleMap
    D = 64
    mon, non = c4_terms(D)
    X = synthetic_samples(300, D, seed=3)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='integrated rectifier', quadrature_input={'order': 40})
    tm = make_cuda(X.copy(), **kw)
    om = OracleMap(X=X.copy(), **kw)
    for k in range(D):
        c = headline_coeffs(mon, non, k)
        div = len(non[k])
        tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:div].copy(), c[div:].copy()
        om.coeffs_nonmon[k], om.coeffs_mon[k] = c[:div].copy(), c[div:].copy()
    assert rel_err(tm.map(X.copy()), om.map(X.copy())) <= 1e-10


def test_c4_full_fit_at_d64_matches_reference():
    """optimize() of all 64 components (scipy BFGS on the host, tm.py:3252-3257, fed by the tile kernel) against the
    reference's fit of the same ensemble.  Both sides stop on |grad|_inf <= 1e-5 (scipy gtol): the objective at the
    optimum agrees to ~1e-10, map() to <= 1e-6; individual coefficients are only determined up to gtol / curvature."""
    gold = np.load(os.path.join(GOLD, 'headline_c4_fit.npz'))
    D = 64
    mon, non = c4_terms(D)
    X = synthetic_samples(HEADLINE_N, D, seed=0)
    tm = make_cuda(X.copy(), monotone=mon, nonmonotone=non, polynomial_type='hermite function',
                   monotonicity='integrated rectifier', quadrature_input={'order': 100})
    tm.optimize()
    worst_c, worst_J = 0.0, 0.0
    for k in range(D):
        c = np.concatenate((tm.coeffs_nonmon[k], tm.coeffs_mon[k]))
        cg = np.concatenate((gold['coeffs_nonmon_%d' % k], gold['coeffs_mon_%d' % k]))
        worst_c = max(worst_c, rel_err(c, cg))
        worst_J = max(worst_J, rel_err(tm.objective_function(c, k, len(tm.coeffs_nonmon[k])), gold['J_%d' % k]))
        # the reference's optimum is stationary for OUR objective too (same function, same gtol)
        g = tm.objective_function_jacobian(cg, k, len(tm.coeffs_nonmon[k]))
        assert np.max(np.abs(g)) <= 2e-5, (k, np.max(np.abs(g)))
    err_map = rel_err(tm.map(X[:256].copy()), gold['map_head'])
    print('C4 D=64 fit vs reference: coefficients %.2e, J at optimum %.2e, map %.2e' % (worst_c, worst_J, err_map))
    assert worst_J <= 1e-8
    assert err_map <= TOL_FIT
    assert worst_c <= 1e-4          # see docstring; map() and J are the gated quantities


@pytest.mark.parametrize('D', [64, 128])
def test_separable_fit_at_d64_d128_matches_reference_qr(D):
    """worker_task_monotone (tm.py:2903-3172): the reference projects with a Householder QR of Psi_non
    (:2966-2975); m_non reaches 190 (D=64) and 382 (D=128) correlated columns here."""
    gold = np.load(os.path.join(GOLD, 'headline_sep_fit_%d.npz' % D))
    mon, non = c5_terms(D)
    X = synthetic_samples(HEADLINE_N, D, seed=0)
    tm = make_cuda(X.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    tm.optimize()
    worst_m = max(rel_err(tm.coeffs_mon[k], gold['coeffs_mon_%d' % k]) for k in range(D))
    worst_n = max(rel_err(tm.coeffs_nonmon[k], gold['coeffs_nonmon_%d' % k]) for k in range(D))
    err_map = rel_err(tm.map(X[:256].copy()), gold['map_head'])
    print('separable D=%d fit vs reference QR path: mon %.2e nonmon %.2e map %.2e' % (D, worst_m, worst_n, err_map))
    assert worst_m <= TOL_FIT and worst_n <= TOL_FIT
    assert err_map <= TOL_FIT


def test_c5_inverse_at_d256_matches_reference():
    """inverse_map (tm.py:3639-4084) at D=256 with E=128 conditioning columns, seeded coefficients: the table
    solver is a deterministic interpolation (<= 1e-10); bisection stops on a 1e-9 residual on both sides."""
    gold = np.load(os.path.join(GOLD, 'headline_c5_inverse.npz'))
    D, E = C5_INV['D'], C5_INV['E']
    mon, non = c5_terms(D)
    tm = make_cuda(synthetic_samples(C5_INV['ntrain'], D, seed=0), monotone=mon, nonmonotone=non,
                   monotonicity='separable monotonicity')
    cm, cn = headline_sep_coeffs(mon, non)
    for k in range(D):
        tm.coeffs_mon[k], tm.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
    rng = np.random.default_rng(C5_INV['seed'])
    Xstar = synthetic_samples(C5_INV['n_table'], D, seed=C5_INV['seed'] + 1)[:, :E].copy()
    Z = rng.standard_normal((C5_INV['n_table'], D - E))
    tm.alternate_root_finding = True
    Xt = tm.inverse_map(Z.copy(), X_star=Xstar.copy())
    # the fixture holds the solved columns of a fixed sample of the rows; the reference returns the conditioning
    # columns as given (to 1e-15)
    assert rel_err(Xt[:, :E], Xstar) <= 1e-10
    assert rel_err(Xt[gold['rows_table'], E:], gold['inverse_table']) <= 1e-10
    nb = C5_INV['n_bisect']
    tm.alternate_root_finding = False
    Xb = tm.inverse_map(Z[:nb].copy(), X_star=Xstar[:nb].copy())
    assert np.max(np.abs(Xb[:, :E] - Xstar[:nb])) <= 1e-6
    assert np.max(np.abs(Xb[gold['rows_bisect'], E:] - gold['inverse_bisect'])) <= 1e-6
