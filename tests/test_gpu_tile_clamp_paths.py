"""The tile kernel's two node-loop instances: a warp whose samples are all in the exps' range runs the clamp-free one,
any other warp the clamped one.  Both must agree with the general kernel on an ensemble that has rows with |x| ~ 70
(which send their warps down the clamped path and the sweep's exp(-x^2/4) into its clamp), at the two rule lengths
that have fully unrolled node loops, and the two instances must give the same bits on in-range samples."""
import numpy as np
import pytest

from cases import synthetic_samples, c4_terms, headline_coeffs
from harness import rel_err

pytestmark = pytest.mark.gpu

D = 64
N = 4000
KS = (0, 1, 31, 63)


def _map(X, Q):
    from transport_map import transport_map
    mon, non = c4_terms(D)
    tm = transport_map(X=X, monotone=mon, nonmonotone=non, polynomial_type='hermite function',
                       monotonicity='integrated rectifier', quadrature_input={'order': Q}, verbose=False)
    return tm, mon, non


def _set_kernel(tm, general):
    from ttt_b200 import binding as B
    B.check(tm._lib.ttm_ctx_set_objgrad_kernel(tm._ctx, 1 if general else 0))
    tm._fg_cache = {}


def _with_outliers():
    X = synthetic_samples(N, D, seed=4)
    X[7, :] = 70.0
    X[1000, ::2] = -70.0
    X[3001, 1::3] = 69.5
    return X


@pytest.mark.parametrize('Q', [100, 25])
def test_tile_kernel_matches_general_kernel_with_out_of_range_rows(Q):
    tm, mon, non = _map(_with_outliers(), Q)
    assert all(info['tile_ok'] for info in tm._plan_info)
    for k in KS:
        c = headline_coeffs(mon, non, k)
        div = len(non[k])
        res = {}
        for general in (False, True):
            _set_kernel(tm, general)
            res[general] = (tm.objective_function(c.copy(), k, div), tm.objective_function_jacobian(c.copy(), k, div))
        assert np.isfinite(res[False][0]) and np.all(np.isfinite(res[False][1])), k
        assert rel_err(res[False][0], res[True][0]) <= 1e-10, (Q, k)
        assert rel_err(res[False][1], res[True][1]) <= 1e-10, (Q, k)


def _fast_path_condition(mon, non, x, k, c_mon):
    """The kernel's per-sample vote, restated from the CPU oracle: ya = -(x_c/2)^2/4 and the bound
    |E0| + 2|E1| + 4|E2| + 8|E3| of the rectifier argument's polynomial part P(tau) = r(hx tau) e^{(hx tau)^2/4}, a cubic
    in tau whose coefficients are recovered from four evaluations of the monotone function."""
    from ttm_oracle import OracleMap
    om = OracleMap(X=synthetic_samples(200, D, seed=9), monotone=mon, nonmonotone=non,
                   polynomial_type='hermite function', monotonicity='integrated rectifier', verbose=False)
    hx = 0.5 * x[:, k]
    taus = np.array([0.5, 1.0, 1.5, 2.0])
    P = np.empty((x.shape[0], 4))
    for q, tau in enumerate(taus):
        xl = x.copy()
        xl[:, k] = hx * tau
        P[:, q] = (om.fun_mon(k, xl) @ c_mon) * np.exp(0.25 * (hx * tau) ** 2)
    E = np.linalg.solve(np.vander(taus, 4, increasing=True), P.T).T
    return -0.25 * hx ** 2, np.abs(E) @ np.array([1.0, 2.0, 4.0, 8.0])


@pytest.mark.parametrize('Q', [100, 25])
def test_clamped_and_clamp_free_node_loops_give_the_same_bits(Q):
    """S_k per sample: rows 0..31 form one warp.  With x_c = 60 in row 5 (e^{-t^2/4} at t = 30 is far below the
    clamp-free range) that warp takes the clamped instance; its other 31 samples must not change in a single bit."""
    tm, mon, non = _map(synthetic_samples(N, D, seed=5), Q)
    x = synthetic_samples(N, D, seed=6)
    for k in KS:
        c = headline_coeffs(mon, non, k)
        div = len(non[k])
        ya, rbound = _fast_path_condition(mon, non, x[:32], k, c[div:])
        assert np.all(ya >= -175.0) and np.all(rbound < 350.0), (k, ya.min(), rbound.max())   # the warp votes fast
        fast = np.asarray(tm.s(x.copy(), k, c[:div], c[div:]))
        x2 = x.copy()
        x2[5, k] = 60.0
        clamped = np.asarray(tm.s(x2, k, c[:div], c[div:]))
        keep = np.arange(N) != 5
        assert np.array_equal(fast[keep].view(np.uint64), clamped[keep].view(np.uint64)), k
        assert np.isfinite(clamped[5]), k
