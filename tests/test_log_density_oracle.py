"""The log-density restatement (tests/log_density_oracle.py) against the reference's own
density evaluator where its quirks vanish, and against finite differences of the map.  CPU only."""

import copy
import os

import numpy as np
import pytest

from cases import c4_terms, ex05_terms, random_coeffs, synthetic_samples
from ttm_oracle import OracleMap
import log_density_oracle as LD

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _impose(om, gold):
    for k in range(om.D):
        om.coeffs_mon[k] = np.array(gold['coeffs_mon_%d' % k])
        om.coeffs_nonmon[k] = np.array(gold['coeffs_nonmon_%d' % k])


def test_log_pullback_equals_log_of_reference_pullback_on_standardised_ensemble():
    """skip = 0 and X_mean ~ 0, X_std ~ 1: the reference's evaluator (derivative basis on the raw samples, X_std[k])
    then computes the density of the fitted map, so its log is the new quantity."""
    gold = np.load(os.path.join(GOLD, 'sep_ex05.npz'))
    X5 = synthetic_samples(1000, 2, seed=5) * np.array([2.0, 0.5]) + np.array([1.0, -3.0])
    Xs = (X5 - X5.mean(axis=0)) / X5.std(axis=0)
    mon, non = ex05_terms()
    om = OracleMap(X=Xs.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    assert np.max(np.abs(om.X_mean)) < 1e-14 and np.max(np.abs(om.X_std - 1)) < 1e-14
    _impose(om, gold)
    rng = np.random.default_rng(1)
    Xe = rng.standard_normal((96, 2))
    ref = np.log(om.evaluate_pullback_density(Xe.copy()))
    new = LD.log_pullback_density(om, Xe.copy())
    assert np.all(np.isfinite(new))
    assert np.max(np.abs(new - ref) / np.maximum(1.0, np.abs(ref))) <= 1e-10


def _fd_check(om, X, rel_tol):
    """d Z_k / d x_c by central differences of om.map against exp(l_k(x~)) / sigma_c."""
    Xs = (X - om.X_mean) / om.X_std
    worst = 0.0
    for k in range(om.D):
        c = k + om.skip_dimensions
        h = 1e-5 * om.X_std[c]
        Xp, Xm = X.copy(), X.copy()
        Xp[:, c] += h
        Xm[:, c] -= h
        fd = (om.map(Xp)[:, k] - om.map(Xm)[:, k]) / (2 * h)
        an = np.exp(LD.log_dS(om, k, Xs)) / om.X_std[c]
        worst = max(worst, float(np.max(np.abs(fd - an) / np.abs(an))))
    assert worst <= rel_tol, worst


def test_ir_log_derivative_matches_finite_differences_q100():
    mon, non = c4_terms(3)
    X = synthetic_samples(400, 3, seed=12) * np.array([2.0, 0.5, 3.0]) + np.array([1.0, -2.0, 0.3])
    om = OracleMap(X=X.copy(), monotone=mon, nonmonotone=non, monotonicity='integrated rectifier',
                   quadrature_input={'order': 100})
    for k in range(om.D):
        div = len(om.coeffs_nonmon[k])
        cf = random_coeffs(div, len(om.coeffs_mon[k]), seed=300 + k, scale=0.2)
        om.coeffs_nonmon[k], om.coeffs_mon[k] = cf[:div].copy(), cf[div:].copy()
    _fd_check(om, X[:40].copy(), 1e-6)


def test_separable_log_derivative_matches_finite_differences():
    gold = np.load(os.path.join(GOLD, 'sep_ex05.npz'))
    X5 = synthetic_samples(1000, 2, seed=5) * np.array([2.0, 0.5]) + np.array([1.0, -3.0])
    mon, non = ex05_terms()
    om = OracleMap(X=X5.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    _impose(om, gold)
    _fd_check(om, X5[:40].copy(), 1e-6)


def test_oracle_rejects_x_star_on_a_full_map():
    mon, non = c4_terms(2)
    om = OracleMap(X=synthetic_samples(64, 2, seed=0), monotone=mon, nonmonotone=non,
                   monotonicity='integrated rectifier', quadrature_input={'order': 10})
    with pytest.raises(ValueError):
        LD.log_pullback_density(om, np.zeros((4, 2)), X_star=np.zeros((4, 1)))
