"""Edge cases of the CUDA path against the oracle: ragged sample counts (not a multiple of the 128-thread
rows, fewer samples than one row, a single sample), a component without nonmonotone terms, a constant-only
nonmonotone part, higher polynomial orders (generic instantiations, order-chunked sweeps), empty conditioning,
duplicated terms, and reset() with a different ensemble size."""

import numpy as np
import pytest

from cases import synthetic_samples, c4_terms, ex05_terms
from harness import rel_err

pytestmark = pytest.mark.gpu


def make_cuda(X, **kw):
    from transport_map import transport_map
    return transport_map(X=X, verbose=False, **kw)


def make_oracle(X, **kw):
    from ttm_oracle import OracleMap
    return OracleMap(X=X, **kw)


def compare_objgrad(tm, om, seed=0, tol=1e-10, scale=0.2):
    rng = np.random.default_rng(seed)
    for k in range(tm.D):
        div = len(tm.coeffs_nonmon[k])
        c = rng.standard_normal(div + len(tm.coeffs_mon[k])) * scale
        assert abs(tm.objective_function(c, k, div) - om.objective_function(c, k, div)) <= tol * max(1, abs(om.objective_function(c, k, div)))
        assert rel_err(tm.objective_function_jacobian(c, k, div), om.objective_function_jacobian(c, k, div)) <= tol
        tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:div].copy(), c[div:].copy()
        om.coeffs_nonmon[k], om.coeffs_mon[k] = c[:div].copy(), c[div:].copy()


@pytest.mark.parametrize('n', [1, 2, 31, 127, 128, 129, 513, 1000, 4097])
def test_ragged_sample_counts(n):
    X = synthetic_samples(max(n, 2), 3, seed=n)[:n] if n > 1 else np.array([[0.3, -0.2, 0.9]])
    mon, non = c4_terms(3)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='integrated rectifier', standardize_samples=(n > 1))
    tm = make_cuda(X.copy(), quadrature_input={'order': 12}, **kw)
    om = make_oracle(X.copy(), quadrature_input={'order': 12}, **kw)
    compare_objgrad(tm, om, seed=n)
    assert rel_err(tm.map(X.copy()), om.map(X.copy())) <= 1e-9
    Z = np.random.default_rng(n).standard_normal((n, 3))
    assert np.max(np.abs(tm.inverse_map(Z.copy()) - om.inverse_map(Z.copy()))) <= 2e-8


def test_component_without_nonmonotone_terms_and_constant_only():
    X = synthetic_samples(300, 3, seed=2)
    mon = [[[0], [0, 0, 'HF']], [[1], [0, 1, 'HF']], [[2, 'HF'], [2, 2, 'HF'], [0, 1, 2, 'HF']]]
    non = [[], [[]], [[], [0, 1], [0, 'HF']]]
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='integrated rectifier')
    tm = make_cuda(X.copy(), quadrature_input={'order': 16}, **kw)
    om = make_oracle(X.copy(), quadrature_input={'order': 16}, **kw)
    assert tm.Psi_nonmon[0] is None and om.Psi_nonmon[0] is None
    compare_objgrad(tm, om)
    assert rel_err(tm.map(X.copy()), om.map(X.copy())) <= 1e-9


@pytest.mark.parametrize('family', ['hermite function', 'legendre', 'power series'])
def test_high_orders_use_generic_instantiations(family):
    """Monotone order up to 14 (generic <20, 8> instantiation), nonmonotone order 9 (order-chunked sweeps),
    duplicated nonmonotone terms (slow group), special inner terms in integrated-rectifier mode."""
    X = synthetic_samples(400, 2, seed=4) * 0.6
    kw_std = dict(standardize_samples=False)      # keep |x| < ~2 so that order-14 terms stay O(1e3)
    X = np.clip(X, -1.6, 1.6)
    mon = [[[0] * o + ['HF'] for o in range(1, 8)] + ['iRBF 0', 'RBF 0'],
           [[1] * o for o in (1, 2, 5, 9, 14)] + [[0, 1, 1, 'HF'], 'LET 1', 'iRBF 1', 'RET 1']]
    non = [[[]], [[], [0], [0], [0] * 9 + ['HF'], [0] * 9, [0] * 4, 'RBF 0']]
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='integrated rectifier', polynomial_type=family, **kw_std)
    tm = make_cuda(X.copy(), quadrature_input={'order': 20}, **kw)
    om = make_oracle(X.copy(), quadrature_input={'order': 20}, **kw)
    for k in range(2):
        assert rel_err(tm.Psi_mon[k], om.Psi_mon[k]) <= 1e-10 and rel_err(tm.Psi_nonmon[k], om.Psi_nonmon[k]) <= 1e-10
    rng = np.random.default_rng(1)
    for k in range(2):
        div = len(tm.coeffs_nonmon[k])
        # coefficients scaled by the column magnitudes so that the rectifier argument stays O(1)
        mag = np.concatenate((np.abs(om.Psi_nonmon[k]).max(axis=0), np.abs(om.Psi_mon[k]).max(axis=0)))
        c = rng.standard_normal(div + len(tm.coeffs_mon[k])) * 0.2 / np.maximum(mag, 1.0)
        J, Jo = tm.objective_function(c, k, div), om.objective_function(c, k, div)
        assert np.isfinite(Jo) and abs(J - Jo) <= 1e-9 * max(1, abs(Jo))
        g, go = tm.objective_function_jacobian(c, k, div), om.objective_function_jacobian(c, k, div)
        assert np.max(np.abs(g - go) / np.maximum(1.0, np.abs(go))) <= 1e-9
        tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:div].copy(), c[div:].copy()
        om.coeffs_nonmon[k], om.coeffs_mon[k] = c[:div].copy(), c[div:].copy()
    assert rel_err(tm.map(), om.map()) <= 1e-9


def test_order_above_compiled_limit_raises():
    X = synthetic_samples(64, 1, seed=1)
    tm = make_cuda(X, monotone=[[[0] * 21]], nonmonotone=[[[]]], monotonicity='integrated rectifier',
                   quadrature_input={'order': 8})
    with pytest.raises(RuntimeError, match='compiled limits'):
        tm.objective_function(np.zeros(2), 0, 1)


def test_reset_changes_ensemble_size_and_special_terms(monkeypatch):
    mon, non = ex05_terms()
    X1, X2 = synthetic_samples(500, 2, seed=1), synthetic_samples(1300, 2, seed=2) * 2 + 1
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    tm, om = make_cuda(X1.copy(), **kw), make_oracle(X1.copy(), **kw)
    tm.optimize(); om.optimize()
    tm.reset(X2.copy()); om.reset(X2.copy())
    assert all(np.all(c == 0) for c in tm.coeffs_mon)
    for k in range(2):
        assert rel_err(tm.Psi_mon[k], om.Psi_mon[k]) <= 1e-10
        assert rel_err(tm.der_Psi_mon[k], om.der_Psi_mon[k]) <= 1e-10
    tm.optimize(); om.optimize()
    for k in range(2):
        assert rel_err(tm.coeffs_mon[k], om.coeffs_mon[k]) <= 1e-6
        assert rel_err(tm.coeffs_nonmon[k], om.coeffs_nonmon[k]) <= 1e-6
    Xe = synthetic_samples(77, 2, seed=3)
    assert rel_err(tm.evaluate_pullback_density(Xe.copy()), om.evaluate_pullback_density(Xe.copy())) <= 1e-9
    # X_star on a full map (inverse_map's conditional branch): the stacked [X_star | inverse_map(Z, X_star)] has D + E
    # columns, which only the per-component path takes (K-map-fused reads skip_dimensions + D)
    monkeypatch.setenv('TTM_MAP_FUSED', '0')
    Zc = np.random.default_rng(4).standard_normal((77, 1))
    lg = lambda x: -0.5 * np.sum(x ** 2, axis=1)
    assert rel_err(tm.evaluate_pushforward_density(Zc.copy(), lg, X_star=Xe[:, :1].copy()),
                   om.evaluate_pushforward_density(Zc.copy(), lg, X_star=Xe[:, :1].copy())) <= 1e-9


def test_public_attributes_and_callables_match_reference_surface():
    X = synthetic_samples(200, 2, seed=6)
    mon, non = ex05_terms()
    tm = make_cuda(X.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    om = make_oracle(X.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    assert tm.D == 2 and tm.skip_dimensions == 0 and tm.X.shape == (200, 2)
    assert rel_err(tm.X, om.X) <= 1e-13 and rel_err(tm.X_mean, om.X_mean) <= 1e-13 and rel_err(tm.X_std, om.X_std) <= 1e-13
    assert set(tm.special_terms[1][1].keys()) == {'counter', 'centers', 'scales'}
    assert rel_err(tm.special_terms[1][1]['centers'], om.special_terms[1][1]['centers']) <= 1e-12
    Xq = synthetic_samples(50, 2, seed=7)
    assert rel_err(tm.fun_mon[1](Xq, tm), om.fun_mon(1, Xq)) <= 1e-10            # reference call signature f(x, self)
    assert rel_err(tm.fun_nonmon[1](Xq, tm), om.fun_nonmon(1, Xq)) <= 1e-10
    assert rel_err(tm.der_fun_mon[1](Xq, tm), om.der_fun_mon(1, Xq)) <= 1e-10
    assert rel_err(tm.s(Xq, 1), om.s(Xq, 1)) <= 1e-10
    assert np.array_equal(tm.optimization_constraints_lb[0], om.optimization_constraints_lb[0])


def test_gram_mode_equals_two_sweep_kernel_and_oracle():
    """dJ/da = G a + h (one sweep, Gram precomputed) against the two-sweep kernel and the oracle, incl. partial maps,
    ragged N and a component mixing dense, special and multivariate nonmonotone terms."""
    from cases import ex06_terms
    X = synthetic_samples(3001, 5, seed=12)
    mon, non = c4_terms(5)
    non[4] = non[4] + ['RBF 1', [0, 2], [3], [3]]            # special, multivariate, duplicate terms
    mon2 = [[[k + 1, 'HF'], [k + 1, k + 1, 'HF'], [k, k + 1, 'HF']] for k in range(4)]
    non2 = [[[]] + [[j] for j in range(k + 1)] + [[j, j, 'HF'] for j in range(k + 1)] for k in range(4)]
    for (mo, no) in ((mon, non), (mon2, non2)):
        kw = dict(monotone=mo, nonmonotone=no, monotonicity='integrated rectifier')
        tg = make_cuda(X.copy(), quadrature_input={'order': 15}, **kw)
        tg._use_gram = True
        t2 = make_cuda(X.copy(), quadrature_input={'order': 15}, **kw)
        t2._use_gram = False
        om = make_oracle(X.copy(), quadrature_input={'order': 15}, **kw)
        rng = np.random.default_rng(3)
        for k in range(tg.D):
            div = len(tg.coeffs_nonmon[k])
            c = rng.standard_normal(div + len(tg.coeffs_mon[k])) * 0.2
            Jg, J2, Jo = (t.objective_function(c, k, div) for t in (tg, t2, om))
            gg, g2, go = (t.objective_function_jacobian(c, k, div) for t in (tg, t2, om))
            assert tg._gram_nn[k] is not None and t2._gram_nn[k] is None
            assert abs(Jg - Jo) <= 1e-10 * max(1, abs(Jo)) and abs(J2 - Jo) <= 1e-10 * max(1, abs(Jo))
            assert rel_err(gg, go) <= 1e-10 and rel_err(g2, go) <= 1e-10


@pytest.mark.parametrize('conditioning', ['x_star', 'skip_dimensions', 'skip_dimensions_unconditioned', 'none'])
def test_pipelined_inverse_is_bit_identical_to_one_shot(conditioning, monkeypatch):
    """Large table-mode inverse_map calls are cut into chunks of samples that overlap staging, copies and
    solves (transport_map._inverse_map_pipelined); samples are independent, so the chunked result must equal
    the one-shot result bit for bit -- including a ragged last chunk and a slot that is reused."""
    from cases import ex06_terms
    n_train, n = 600, 2503
    if conditioning.startswith('skip_dimensions'):
        mon, non = ex06_terms(3)
        X = synthetic_samples(n_train, 4, seed=3)
        tm = make_cuda(X, monotone=mon, nonmonotone=non, monotonicity='separable monotonicity',
                       regularization='l2', regularization_lambda=0.05)
        tm.optimize()
        rng = np.random.default_rng(5)
        Z, Xs = rng.standard_normal((n, 3)), synthetic_samples(n, 4, seed=9)[:, :1].copy()
        if conditioning.endswith('unconditioned'):
            Xs = None
    else:
        mon, non = ex05_terms()
        X = synthetic_samples(n_train, 2, seed=4)
        tm = make_cuda(X, monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
        tm.optimize()
        rng = np.random.default_rng(6)
        if conditioning == 'x_star':
            Z, Xs = rng.standard_normal((n, 1)), synthetic_samples(n, 2, seed=8)[:, :1].copy()
        else:
            Z, Xs = rng.standard_normal((n, 2)), None
    monkeypatch.setenv('TTM_INV_PIPELINE_MIN', '1000000000')
    one_shot = tm.inverse_map(Z, X_star=Xs)
    monkeypatch.setenv('TTM_INV_PIPELINE_MIN', '1000')
    monkeypatch.setenv('TTM_INV_CHUNK', '600')          # 5 chunks of 501 through 4 slots, the last one (499) cut into 248 + 124 + 127
    piped = tm.inverse_map(Z, X_star=Xs)
    assert piped.shape == one_shot.shape
    assert np.array_equal(piped, one_shot)
    # the same call with the inputs in page-locked host memory: copied to the device directly, no staging
    import torch
    from ttt_b200 import binding as B
    Zp = torch.empty(Z.shape, dtype=torch.float64, pin_memory=True).numpy()
    Zp[:] = Z
    flag = B.c_int(0)
    B.check(tm._lib.ttm_host_is_pinned(B.c_void_p(Zp.ctypes.data), B.ctypes.byref(flag)))
    assert flag.value == 1
    B.check(tm._lib.ttm_host_is_pinned(B.c_void_p(Z.ctypes.data), B.ctypes.byref(flag)))
    assert flag.value == 0
    Xp = None
    if Xs is not None:
        Xp = torch.empty(Xs.shape, dtype=torch.float64, pin_memory=True).numpy()
        Xp[:] = Xs
    assert np.array_equal(tm.inverse_map(Zp, X_star=Xp), one_shot)


@pytest.mark.parametrize('D,E,n', [(20, 3, 301), (17, 0, 64), (33, 16, 1000)])
def test_fused_inverse_block_edges_match_the_oracle(D, E, n):
    """K-inv-fused walks the components in blocks of 16 and the samples in tiles of 256: component counts of 17
    (one full block + one component), 16 + 1 with an empty conditioning block, ragged sample counts."""
    from cases import c5_terms, headline_sep_coeffs
    mon, non = c5_terms(D)
    X = synthetic_samples(400, D, seed=21)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    tm = make_cuda(X.copy(), **kw)
    om = make_oracle(X.copy(), **kw)
    cm, cn = headline_sep_coeffs(mon, non)
    for k in range(D):
        tm.coeffs_mon[k], tm.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
        om.coeffs_mon[k], om.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
    rng = np.random.default_rng(5)
    Z = rng.standard_normal((n, D - E))
    Xs = synthetic_samples(n, D, seed=22)[:, :E].copy() if E else None
    assert tm._inverse_fused_setup([(i, k) for i, k in enumerate(range(E, D))]) is not None
    assert rel_err(tm.inverse_map(Z.copy(), None if Xs is None else Xs.copy()),
                   om.inverse_map(Z.copy(), None if Xs is None else Xs.copy())) <= 1e-10


@pytest.mark.parametrize('D,E,n,mixed', [(21, 9, 333, False), (40, 7, 64, False), (150, 5, 130, False),
                                         (48, 33, 1, False), (20, 6, 300, True), (14, 0, 77, True)])
def test_split_inverse_matches_the_oracle(D, E, n, mixed, monkeypatch):
    """K-inv-rect + K-inv-fused (TTM_INV_SPLIT=1: conditioning block contracted as a GEMM first): conditioning widths
    that are not multiples of the 8-variable chunk, sample counts that are not multiples of the 64-sample tile (odd,
    below one tile, a single sample), more than 128 solved components (two component tiles)."""
    from cases import c5_terms, headline_sep_coeffs
    monkeypatch.setenv('TTM_INV_SPLIT', '1')
    mon, non = c5_terms(D)
    if mixed:                                   # plain and Hermite-function terms of every order: the 6-slot operands
        non = [[[]] + [t for j in range(k) for t in ([j], [j, 'HF'], [j, j], [j, j, 'HF'], [j, j, j], [j, j, j, 'HF'])]
               for k in range(D)]
    X = synthetic_samples(400, D, seed=23)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    tm = make_cuda(X.copy(), **kw)
    om = make_oracle(X.copy(), **kw)
    cm, cn = headline_sep_coeffs(mon, non)
    for k in range(D):
        tm.coeffs_mon[k], tm.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
        om.coeffs_mon[k], om.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
    Z = np.random.default_rng(6).standard_normal((n, D - E))
    Xs = synthetic_samples(n, D, seed=24)[:, :E].copy() if E else None
    xs = lambda: None if Xs is None else Xs.copy()
    fz = tm._inverse_fused_setup([(i, k) for i, k in enumerate(range(E, D))])
    assert fz is not None and fz['ns'] == (6 if mixed else 3) and (fz['R'] is not None) == (E > 0)
    got = tm.inverse_map(Z.copy(), xs())
    assert rel_err(got, om.inverse_map(Z.copy(), xs())) <= 1e-10
    monkeypatch.setenv('TTM_INV_SPLIT', '0')                   # the one-launch walk: same numbers up to summation order
    assert tm._inverse_fused_setup([(i, k) for i, k in enumerate(range(E, D))])['R'] is None
    assert rel_err(tm.inverse_map(Z.copy(), xs()), got) <= 1e-12


def test_fused_inverse_rejects_tables_longer_than_the_limit():
    """ttm_inverse_fused and ttm_inverse_fused_split stage two tables per block in shared memory: ntab = 2049 (one past
    TTM_INVERSE_FUSED_MAX_NTAB) fails with TTM_ERR_LIMIT before any launch and leaves the output untouched; ntab = 2048
    runs and solves the column (zero offsets, identity table, z = 0 -> x = 0 up to rounding)."""
    import torch
    from cases import c5_terms
    from ttt_b200 import binding as B
    mon, non = c5_terms(2)
    tm = make_cuda(synthetic_samples(200, 2, seed=1), monotone=mon, nonmonotone=non,
                   monotonicity='separable monotonicity')
    lib, n, ns = tm._lib, 8, 3
    f64 = dict(dtype=torch.float64, device=tm._device)
    size = B.c_int64()
    B.check(lib.ttm_inverse_fused_apack_size(1, 1, ns, B.ctypes.byref(size)))
    A = torch.zeros(size.value, **f64)
    B.check(lib.ttm_inverse_rect_rpack_size(1, 1, ns, B.ctypes.byref(size)))
    R = torch.zeros(size.value, **f64)
    a0, Zt, base = torch.zeros(1, **f64), torch.zeros(1, n, **f64), torch.zeros(1, n, **f64)
    p = lambda t: B.c_void_p(t.data_ptr())
    for ntab, rc_want in ((2049, -3), (2048, 0)):
        grid = torch.linspace(-10, 10, ntab, **f64)
        tabs = torch.cat((grid, grid))
        for split in (False, True):
            Xw = torch.full((2, n), 7.0, **f64)
            if split:
                rc = lib.ttm_inverse_fused_split(tm._ctx, p(Xw), n, n, p(Zt), n, 1, 1, ns, p(A), p(R), p(a0), p(tabs), ntab,
                                                 0, p(base), n, tm._stream())
            else:
                rc = lib.ttm_inverse_fused(tm._ctx, p(Xw), n, n, p(Zt), n, 1, 1, ns, p(A), p(a0), p(tabs), ntab, 0,
                                           tm._stream())
            assert rc == rc_want, (ntab, split, lib.ttm_last_error())
            torch.cuda.synchronize(tm._device)
            if rc_want:
                assert b'TTM_INVERSE_FUSED_MAX_NTAB' in lib.ttm_last_error()
                assert torch.equal(Xw, torch.full_like(Xw, 7.0))
            else:
                assert torch.equal(Xw[0], torch.full_like(Xw[0], 7.0)) and float(Xw[1].abs().max()) <= 1e-12


@pytest.mark.parametrize('D,n,mixed', [(40, 4100, False), (34, 4097, True), (150, 4160, False)])
def test_gemm_forward_map_matches_the_oracle(D, n, mixed, monkeypatch):
    """map() of a wide separable map: nonmonotone sums of all components as one block-triangular DMMA GEMM
    (ttm_map_rect) + monotone terms per component (ttm_sep_eval_base), against the oracle and the per-component
    kernels; sample counts off the 64-sample tile, 3- and 6-slot operands, two component tiles (D = 150)."""
    from cases import c5_terms, headline_sep_coeffs
    mon, non = c5_terms(D)
    if mixed:
        non = [[[]] + [t for j in range(k) for t in ([j], [j, 'HF'], [j, j], [j, j, 'HF'], [j, j, j], [j, j, j, 'HF'])]
               for k in range(D)]
    X = synthetic_samples(400, D, seed=25)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity')
    tm = make_cuda(X.copy(), **kw)
    om = make_oracle(X.copy(), **kw)
    cm, cn = headline_sep_coeffs(mon, non)
    for k in range(D):
        tm.coeffs_mon[k], tm.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
        om.coeffs_mon[k], om.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
    Xe = synthetic_samples(n, D, seed=26)
    assert tm._map_gemm_static() is not None
    got = tm.map(Xe.copy())
    assert rel_err(got, om.map(Xe.copy())) <= 1e-10
    monkeypatch.setenv('TTM_MAP_GEMM', '0')
    tm._inv_pack_cache.pop('map_gemm', None)
    assert tm._map_gemm_static() is None
    assert rel_err(tm.map(Xe.copy()), got) <= 1e-12


@pytest.mark.parametrize('name', ['sep_ex05', 'sep_ex06_cycle', 'sep_c5_d6'])
def test_per_component_paths_match_the_fused_ones(name, monkeypatch):
    """map / inverse_map / densities through the per-component kernels (TTM_MAP_FUSED=0, TTM_INV_FUSED=0: the paths
    large or out-of-class maps take) against the reference fixtures, like the fused default."""
    import os
    from cases import cases
    from harness import run_case
    monkeypatch.setenv('TTM_MAP_FUSED', '0')
    monkeypatch.setenv('TTM_INV_FUSED', '0')
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', name + '.npz'))
    res = run_case(lambda X, **kw: make_cuda(X, **{k: v for k, v in kw.items() if k != 'verbose'}), cases()[name], fitted=gold)
    for key in ('map_X', 'map_train', 'inverse_table', 'pullback', 'pushforward'):
        if key in res:
            assert rel_err(res[key], gold[key]) <= 1e-9, (name, key)


def test_x_setter_invalidates_memoised_objective():
    """ADVICE r1: assigning tm.X must drop the memoised (J, grad), the Gram matrices and the lazy Psi."""
    X = synthetic_samples(600, 3, seed=30)
    mon, non = c4_terms(3)
    tm = make_cuda(X.copy(), monotone=mon, nonmonotone=non, monotonicity='integrated rectifier',
                   quadrature_input={'order': 12}, standardize_samples=False)
    c = np.random.default_rng(1).standard_normal(len(non[2]) + len(mon[2])) * 0.1
    f0 = tm.objective_function(c, 2, len(non[2]))
    X2 = synthetic_samples(700, 3, seed=31)
    tm.X = X2.copy()
    fresh = make_cuda(X2.copy(), monotone=mon, nonmonotone=non, monotonicity='integrated rectifier',
                      quadrature_input={'order': 12}, standardize_samples=False)
    f1 = tm.objective_function(c, 2, len(non[2]))
    assert f1 != f0 and abs(f1 - fresh.objective_function(c, 2, len(non[2]))) <= 1e-13
    assert rel_err(tm.objective_function_jacobian(c, 2, len(non[2])), fresh.objective_function_jacobian(c, 2, len(non[2]))) <= 1e-12


def test_standardize_method_matches_the_oracle():
    """tm.standardize() (tm.py:750-787) on a map built with standardize_samples=False."""
    X = synthetic_samples(500, 3, seed=40) * np.array([2.0, 0.3, 5.0]) + np.array([1.0, -2.0, 0.5])
    mon, non = c4_terms(3)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='integrated rectifier', standardize_samples=False)
    tm = make_cuda(X.copy(), quadrature_input={'order': 10}, **kw)
    om = make_oracle(X.copy(), quadrature_input={'order': 10}, **kw)
    tm.standardize()
    om.standardize()
    assert rel_err(tm.X_mean, om.X_mean) <= 1e-12 and rel_err(tm.X_std, om.X_std) <= 1e-12
    assert rel_err(tm.X, om.X) <= 1e-12
