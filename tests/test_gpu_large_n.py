"""Reducing and grid-stride kernels against the CPU oracle at sample counts where every thread block loops.

At the sizes of the parity tests each block of K-objgrad, K-gram, K-sepobj, K-sep-eval and K-std handles one tile,
chunk or pass; the code that runs only from a block's second one on (chunk carry-over of s_S / s_M / s_I, the dense
gradient sweep of a later chunk, K-gram's accumulation into the split partials, second grid-stride passes) is only
reached at production N.  decomposition.py restates each launcher's split, and every N below comes from it, so each
block makes at least three tiles / chunks / passes, the last one partial, on any SM count.

The reference is the unmodified oracle run on chunks of the ensemble and combined with math.fsum.  Each objective
test also shows that it would see one lost sample: dropping the sample that starts a block's second tile or chunk
moves J or grad J by more than 100 times the tolerance.
"""
import math

import numpy as np
import pytest

import decomposition as dec
from cases import synthetic_samples, c4_terms, c5_terms
from harness import rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-10
CHUNK = 1 << 17
IR = dict(monotonicity='integrated rectifier', polynomial_type='hermite function', verbose=False,
          standardize_samples=False)


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _ensemble(N, D, seed, bump):
    """Standardised synthetic ensemble; row `bump` (the first sample of a block's second tile or chunk) is moved to
    x = 2.5 in every column so that its J_i is far from the mean."""
    X = synthetic_samples(N, D, seed=seed)
    X = (X - X.mean(axis=0)) / X.std(axis=0)
    X[bump, :] = 2.5
    return np.ascontiguousarray(X)


def _place_from(om, Xfull):
    """Special terms are placed at quantiles of the ensemble: take the placement from all rows, not from the chunk
    the oracle was built on, and recompute its basis matrices."""
    keep, om.X = om.X, Xfull
    om._place_special_terms()
    om.X = keep
    om.Psi_mon, om.Psi_nonmon = [om.fun_mon(0, om.X)], [om.fun_nonmon(0, om.X)]
    if om.monotonicity == 'separable monotonicity':
        om.der_Psi_mon = [om.der_fun_mon(0, om.X)]
    return om


def _oracle_k(X, rows, mon, non, k, kw, Q=None):
    """Oracle of component k alone on X[rows] (columns 0..k), special terms placed on all rows of X."""
    from ttm_oracle import OracleMap
    extra = {} if Q is None else {'quadrature_input': {'order': Q}}
    om = OracleMap(X=np.array(X[rows, :k + 1]), monotone=mon[k:k + 1], nonmonotone=non[k:k + 1], **extra, **kw)
    return _place_from(om, X[:, :k + 1]) if any(isinstance(t, str) for t in mon[k] + non[k]) else om


def _reference(X, mon, non, k, Q, c, kw):
    """(J, grad J, S) of component k over all rows: oracle per chunk, chunk means weighted by their row counts and
    summed with math.fsum."""
    div = len(non[k])
    N = X.shape[0]
    Js, Gs, S = [], [], []
    for lo in range(0, N, CHUNK):
        om = _oracle_k(X, slice(lo, lo + CHUNK), mon, non, k, kw, Q)
        n = om.X.shape[0]
        Js.append(n * om.objective_function(c.copy(), 0, div))
        Gs.append(n * om.objective_function_jacobian(c.copy(), 0, div))
        S.append(om.s(None, 0, c[:div].copy(), c[div:].copy()))
    Gs = np.array(Gs)
    return (math.fsum(Js) / N, np.array([math.fsum(Gs[:, j]) for j in range(Gs.shape[1])]) / N,
            np.concatenate(S))


def _assert_sees_lost_sample(X, mon, non, k, Q, c, kw, ref, i):
    """J and grad J without sample i, from the full reference and the oracle on that row alone."""
    div = len(non[k])
    N = X.shape[0]
    om = _oracle_k(X, slice(i, i + 1), mon, non, k, kw, Q)
    Ji, gi = om.objective_function(c.copy(), 0, div), om.objective_function_jacobian(c.copy(), 0, div)
    J1, g1 = (N * ref[0] - Ji) / (N - 1), (N * ref[1] - gi) / (N - 1)
    assert max(rel_err(J1, ref[0]), rel_err(g1, ref[1])) > 100 * TOL, (i, J1, ref[0])


def _coeffs(mon, non, k, seed, scale=0.3):
    rng = np.random.default_rng(seed)
    c = rng.standard_normal(len(non[k]) + len(mon[k])) * scale
    return c


def _set(tm, general=None, gram=None, bps=None):
    from ttt_b200 import binding as B
    if general is not None:
        B.check(tm._lib.ttm_ctx_set_objgrad_kernel(tm._ctx, 1 if general else 0))
    if bps is not None:
        B.check(tm._lib.ttm_ctx_set_blocks_per_sm(tm._ctx, bps))
    if gram is not None:
        tm._use_gram = gram
        tm._gram_nn = {}
    tm._fg_cache = {}


def _kernels_run(fn):
    """Names of the CUDA kernels fn() launches (torch.profiler)."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _objgrad(tm, c, k, div):
    return tm.objective_function(c.copy(), k, div), tm.objective_function_jacobian(c.copy(), k, div)


def _s_fresh(tm, X, k, c, div):
    """S_k on every row, after the same call on a permuted ensemble (so a skipped row cannot hold a right value
    left in a recycled allocation)."""
    perm = np.random.default_rng(0).permutation(X.shape[0])
    tm.s(X[perm].copy(), k, c[:div].copy(), c[div:].copy())
    return np.asarray(tm.s(X.copy(), k, c[:div].copy(), c[div:].copy()))


# ------------------------------------------------------------------------------------------------ tile kernel
TILE_D = 6


@pytest.fixture(scope='module')
def tile_setup():
    sm = _sm_count()
    out = {}
    z = dec.sizes(sm)
    for which, N in (('ragged', z['tile']), ('exact', z['tile_exact'])):
        X = _ensemble(N, TILE_D, seed=31, bump=dec.tile(N, sm).second)
        out[which] = (N, X)
    refs = {}

    def ref(which, k, Q):
        """(coefficients, reference) of component k, computed once per (ensemble, k, Q)"""
        if (which, k, Q) not in refs:
            mon, non = c4_terms(TILE_D)
            c = _coeffs(mon, non, k, seed=10 + k)
            refs[which, k, Q] = (c, _reference(out[which][1], mon, non, k, Q, c, IR))
        return refs[which, k, Q]
    return sm, out, ref


@pytest.mark.parametrize('which,Q', [('ragged', 25), ('ragged', 100), ('ragged', 13), ('exact', 25)])
def test_tile_kernel_at_looping_n(tile_setup, which, Q):
    from transport_map import transport_map
    sm, data, tile_ref = tile_setup
    N, X = data[which]
    mon, non = c4_terms(TILE_D)
    for bps in (0, 1):
        s = dec.tile(N, sm, bps)
        assert s.loops_min >= 3 and s.partial == (which == 'ragged'), s
    tm = transport_map(X=X.copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': Q}, **IR)
    assert all(info['tile_ok'] for info in tm._plan_info)
    for k in (0, TILE_D - 1):
        c, ref = tile_ref(which, k, Q)
        div = len(non[k])
        _set(tm, gram=True, bps=0)
        names = _kernels_run(lambda: _objgrad(tm, c, k, div))      # the tile kernel ran, not its general fallback
        assert any('objgrad_tile_kernel' in n for n in names), names
        if which == 'ragged':
            _assert_sees_lost_sample(X, mon, non, k, Q, c, IR, ref, dec.tile(N, sm).second)
        for bps in (0, 1):
            for gram in (True, False):
                _set(tm, gram=gram, bps=bps)
                J, g = _objgrad(tm, c, k, div)
                assert rel_err(J, ref[0]) <= TOL, (k, bps, gram, J, ref[0])
                assert rel_err(g, ref[1]) <= TOL, (k, bps, gram, rel_err(g, ref[1]))
                print('tile N=%d Q=%d k=%d bps=%d gram=%d: J %.1e grad %.1e' % (N, Q, k, bps, gram, rel_err(J, ref[0]),
                                                                            rel_err(g, ref[1])))
            S = _s_fresh(tm, X, k, c, div)
            assert rel_err(S, ref[2]) <= TOL, (k, bps, rel_err(S, ref[2]))
            print('tile N=%d Q=%d k=%d bps=%d: S %.1e' % (N, Q, k, bps, rel_err(S, ref[2])))
        _set(tm, bps=0)


# ------------------------------------------------------------------------------------------------ general kernel
def _general_specs():
    """One map per instantiation of the general kernel (D = 2, component 1 checked; nonmonotone order 3 on x_0)."""
    non = [[[]], [[], [0], [0, 0, 'HF'], [0, 0, 0, 'HF']]]
    return {
        1: (dict(), [[[0]], [[1], [1, 1], [0, 1]]], non),                       # plain monotone terms
        2: (dict(), [[[0]], [[1, 'HF'], [1, 1, 1, 1, 1, 'HF']]], non),          # order 5
        3: (dict(), [[[0]], [[1, 'HF'], [1] * 9 + ['HF']]], non),               # order 9
        4: (dict(rectifier_type='softplus'), [[[0]], [[1, 'HF'], [1, 1, 'HF'], [0, 1, 'HF']]], non),
        5: (dict(), [[[0]], [[1], [1, 1, 'HF'], 'iRBF 1']], non),               # special term
    }


def _covers(cfg, p, rect):
    """ObjCfg::covers and the instantiation list, ttm_objgrad_impl.cuh:557-571 (RECT_EXP = 0, FAM_HERMITE_E)."""
    from ttt_b200.plan import FAM_HERMITE_E, H_HAS_PLAIN, H_HAS_HF
    maxord, plain, hf, herme, exprect, nst = {1: (3, 1, 1, 1, 1, 0), 2: (6, 1, 1, 1, 1, 0), 3: (12, 1, 1, 1, 1, 0),
                                              4: (6, 1, 1, 0, 0, 0), 5: (20, 1, 1, 0, 0, 8),
                                              6: (3, 0, 1, 1, 1, 0)}[cfg]
    return (p.maxord <= maxord and p.nst <= nst and (plain or not p.iblob[H_HAS_PLAIN]) and
            (hf or not p.iblob[H_HAS_HF]) and (not herme or p.family == FAM_HERMITE_E) and (not exprect or rect == 0))


def _instance(p, rect):
    """Dispatch order of ttm_objgrad.cu:19-25."""
    return next(cfg for cfg in (6, 1, 2, 3, 4, 5) if _covers(cfg, p, rect))


GEN_Q = 10


def _check_general(tm, X, mon, non, k, Q, kw, forms, sm, cfg):
    N = X.shape[0]
    c = _coeffs(mon, non, k, seed=50 + cfg, scale=0.2)
    div = len(non[k])
    ref = _reference(X, mon, non, k, Q, c, kw)
    _assert_sees_lost_sample(X, mon, non, k, Q, c, kw, ref, dec.general(N, sm, cfg).second)
    _set(tm, general=True)
    names = _kernels_run(lambda: _objgrad(tm, c, k, div))
    assert any('objgrad_kernel<' in n for n in names) and not any('objgrad_tile' in n for n in names), names
    worst = 0.0
    for gram, bps in forms:
        s = dec.general(N, sm, cfg, gram, bps)
        assert s.loops_min >= 3 and s.partial, (cfg, gram, bps, s)
        _set(tm, gram=gram, bps=bps)
        J, g = _objgrad(tm, c, k, div)
        assert rel_err(J, ref[0]) <= TOL, (cfg, gram, bps, J, ref[0])
        assert rel_err(g, ref[1]) <= TOL, (cfg, gram, bps, rel_err(g, ref[1]))
        worst = max(worst, rel_err(J, ref[0]), rel_err(g, ref[1]))
    _set(tm, bps=0)
    S = _s_fresh(tm, X, k, c, div)
    assert rel_err(S, ref[2]) <= TOL, (cfg, rel_err(S, ref[2]))
    print('general cfg%d N=%d: J/grad %.1e S %.1e' % (cfg, N, worst, rel_err(S, ref[2])))


@pytest.mark.parametrize('cfg', [1, 2, 3, 4, 5])
def test_general_kernel_instances_at_looping_n(cfg):
    from transport_map import transport_map
    sm = _sm_count()
    extra, mon, non = _general_specs()[cfg]
    N = dec.sizes(sm)['general'][cfg]
    X = _ensemble(N, 2, seed=40 + cfg, bump=dec.general(N, sm, cfg).second)
    kw = dict(IR, **extra)
    tm = transport_map(X=X.copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': GEN_Q}, **kw)
    from ttt_b200.transport_map import _RECT
    assert _instance(tm._host_plans[1], _RECT[tm.rectifier_type]) == cfg
    _check_general(tm, X, mon, non, 1, GEN_Q, kw, [(False, 0), (True, 0)], sm, cfg)


def test_general_kernel_cfg6_blocks_per_sm_at_looping_n():
    """The C4 class with the general kernel forced: two-sweep and Gram forms, 1, 2, 8 and the default 4 blocks per SM
    (the context setting reaches this instantiation only)."""
    from transport_map import transport_map
    sm = _sm_count()
    D, k = 3, 2
    mon, non = c4_terms(D)
    N = dec.sizes(sm)['cfg6']
    X = _ensemble(N, D, seed=46, bump=dec.general(N, sm, 6).second)
    tm = transport_map(X=X.copy(), monotone=mon, nonmonotone=non, quadrature_input={'order': GEN_Q}, **IR)
    from ttt_b200.transport_map import _RECT
    assert _instance(tm._host_plans[k], _RECT[tm.rectifier_type]) == 6
    forms = [(False, b) for b in (0, 1, 2, 8)] + [(True, b) for b in (0, 1, 8)]
    _check_general(tm, X, mon, non, k, GEN_Q, IR, forms, sm, 6)


# ------------------------------------------------------------------------------------------------ K-gram
def test_gram_accumulates_over_chunks():
    """Psi^T Psi of a C5-pattern separable component with M = 146 (three 64-column tiles) over three chunks of
    2^18 samples, the last one partial; and the tail form from column m_non = 142."""
    from transport_map import transport_map
    D = 48
    N = dec.sizes(_sm_count())['gram']
    s = dec.gram_chunks(N)
    assert s.loops_min >= 3 and s.partial
    mon, non = c5_terms(D)
    X = _ensemble(N, D, seed=60, bump=s.second)
    kw = dict(monotonicity='separable monotonicity', polynomial_type='hermite function', verbose=False,
              standardize_samples=False)
    tm = transport_map(X=X.copy(), monotone=mon, nonmonotone=non, **kw)
    k = D - 1
    p = tm._host_plans[k]
    mn, M = p.m_non, p.m_non + p.m_mon
    assert M > 128 and mn % 64 != 0
    G = np.asarray(tm._gram(k))
    tail = np.asarray(tm._gram(k, first_col=mn))
    parts = []
    for lo in range(0, N, 1 << 16):
        om = _oracle_k(X, slice(lo, lo + (1 << 16)), mon, non, k, kw)
        Psi = np.column_stack((om.Psi_nonmon[0], om.Psi_mon[0]))
        parts.append(Psi.T @ Psi)
    ref = np.sum(parts, axis=0)
    assert rel_err(G, ref) <= TOL, rel_err(G, ref)
    assert rel_err(tail, ref[:, mn:]) <= TOL, rel_err(tail, ref[:, mn:])
    print('gram N=%d: G %.1e tail %.1e' % (N, rel_err(G, ref), rel_err(tail, ref[:, mn:])))
    # one lost sample, the first of the second chunk, moves G beyond 100 times the tolerance
    om = _oracle_k(X, slice(s.second, s.second + 1), mon, non, k, kw)
    psi = np.concatenate((om.Psi_nonmon[0][0], om.Psi_mon[0][0]))
    assert rel_err(ref - np.outer(psi, psi), ref) > 100 * TOL


# ------------------------------------------------------------------------------------------------ separable kernels
SEP_D = 4


@pytest.fixture(scope='module')
def sep_setup():
    from transport_map import transport_map
    sm = _sm_count()
    N = dec.sizes(sm)['sep']
    mon, non = c5_terms(SEP_D)
    X = _ensemble(N, SEP_D, seed=70, bump=dec.sepobj(N, sm).second)
    tm = transport_map(X=X.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity',
                       polynomial_type='hermite function', verbose=False)
    rng = np.random.default_rng(71)
    for k in range(SEP_D):
        tm.coeffs_nonmon[k] = rng.standard_normal(len(non[k])) * 0.2
        tm.coeffs_mon[k] = np.abs(rng.standard_normal(len(mon[k]))) * 0.2 + 0.05
    return sm, N, X, mon, non, tm


def _sep_oracle(X, rows, mon, non, k):
    return _oracle_k(X, rows, mon, non, k, dict(monotonicity='separable monotonicity', verbose=False,
                                                 polynomial_type='hermite function', standardize_samples=False))


def test_sepobj_sums_at_looping_n(sep_setup):
    """K-sepobj's N-long sums: sum log dS and sum dPsi / dS, dS = dPsi b + delta sum_j dPsi_j."""
    sm, N, Xr, mon, non, tm = sep_setup
    s = dec.sepobj(N, sm)
    assert s.loops_min >= 3 and s.partial
    Xs = np.asarray(tm.X)                      # the standardised ensemble the kernel reads
    for k in range(SEP_D):
        A, _ = tm._separable_setup(k)
        b = np.abs(np.random.default_rng(80 + k).standard_normal(len(mon[k]))) * 0.3 + 0.1
        f, g = tm._sep_objective(b, A, k)
        # the reduced objective is affine in the sample mean: sum_c n_c f_c / N over chunks c is the whole one
        fs, gs = [], []
        for lo in range(0, N, CHUNK):
            om = _sep_oracle(Xs, slice(lo, lo + CHUNK), mon, non, k)
            fc, gc = om.separable_objective(b, A, 0)
            fs.append(om.X.shape[0] * fc)
            gs.append(om.X.shape[0] * gc)
        gs = np.array(gs)
        f_ref = math.fsum(fs) / N
        g_ref = np.array([math.fsum(gs[:, j]) for j in range(gs.shape[1])]) / N
        assert rel_err(f, f_ref) <= TOL, (k, f, f_ref)
        assert rel_err(g, g_ref) <= TOL, (k, rel_err(g, g_ref))
        print('sepobj N=%d k=%d: f %.1e g %.1e' % (N, k, rel_err(f, f_ref), rel_err(g, g_ref)))
        # one lost sample (the first of a block's second pass) is visible
        i = s.second
        fi = _sep_oracle(Xs, slice(i, i + 1), mon, non, k).separable_objective(b, A, 0)[0]
        assert rel_err((N * f_ref - fi) / (N - 1), f_ref) > 100 * TOL


def test_separable_map_per_component_at_looping_n(sep_setup, monkeypatch):
    """map() through K-sep-eval (TTM_MAP_FUSED=0), every row against the oracle on the same standardised rows."""
    sm, N, Xr, mon, non, tm = sep_setup
    s = dec.sep_eval(N, sm)
    assert s.loops_min >= 3 and s.partial
    monkeypatch.setenv('TTM_MAP_FUSED', '0')
    assert not tm._fused_small()
    perm = np.random.default_rng(1).permutation(N)
    tm.map(Xr[perm].copy())
    Z = np.asarray(tm.map(Xr.copy()))
    Xs = (Xr - tm.X_mean) / tm.X_std
    for k in range(SEP_D):
        ref = np.concatenate([_sep_oracle(Xs, slice(lo, lo + CHUNK), mon, non, k).s(None, 0, tm.coeffs_nonmon[k],
                                                                              tm.coeffs_mon[k])
                              for lo in range(0, N, CHUNK)])
        assert rel_err(Z[:, k], ref) <= TOL, (k, rel_err(Z[:, k], ref))
        print('sep-eval N=%d k=%d: %.1e' % (N, k, rel_err(Z[:, k], ref)))


def _oracle_full(Xr, Xs, mon, non, tm, **kw):
    """Oracle of the whole map that standardises with the map's X_mean / X_std and places its special terms on the
    whole standardised ensemble Xs (built on a few rows: inverse_map and s(x, k) do not read the stored ensemble)."""
    from ttm_oracle import OracleMap
    om = OracleMap(X=np.array(Xr[:4096]), monotone=mon, nonmonotone=non, polynomial_type='hermite function',
                   verbose=False, **kw)
    om.X_mean, om.X_std = np.array(tm.X_mean), np.array(tm.X_std)
    keep, om.X = om.X, Xs
    om._place_special_terms()
    om.X = keep
    for k in range(len(mon)):
        om.coeffs_nonmon[k], om.coeffs_mon[k] = np.array(tm.coeffs_nonmon[k]), np.array(tm.coeffs_mon[k])
    return om


TOL_BISECT = 2e-8        # both sides stop on a 1e-9 residual (test_gpu_parity.py)
BISECT_RESID = 1e-9      # the bisection's stopping residual (tm.py:3975)


def _inverse_checks(tm, om, Zh, N, sm, table, tag):
    """inverse_map of a CUDA-tensor Z (one launch per component over all samples) after the same call on a permuted
    Z.  Table mode: every row against the oracle's table inverse.  Bisection: every row's residual S_k(x) - z_k under
    the oracle, and the oracle's own bisection on a seeded subsample that holds the first rows of the second pass."""
    import torch
    second = dec.sep_eval(N, sm).second
    perm = np.random.default_rng(3).permutation(N)
    tm.inverse_map(torch.from_numpy(Zh[perm]).cuda())
    Xh = tm.inverse_map(torch.from_numpy(Zh).cuda()).cpu().numpy()
    sub = np.union1d(np.random.default_rng(4).choice(N, 400, replace=False), np.arange(second, second + 128))
    if table:
        ref = np.concatenate([om.inverse_map(Zh[lo:lo + CHUNK].copy()) for lo in range(0, N, CHUNK)])
        assert rel_err(Xh, ref) <= TOL, (tag, rel_err(Xh, ref))
        print('inverse %s N=%d: %.1e' % (tag, N, rel_err(Xh, ref)))
        return
    ref = om.inverse_map(Zh[sub].copy())
    assert rel_err(Xh[sub], ref) <= TOL_BISECT, (tag, rel_err(Xh[sub], ref))
    Xs = (Xh - om.X_mean) / om.X_std
    worst = 0.0
    for k in range(Zh.shape[1]):
        r = np.concatenate([om.s(Xs[lo:lo + CHUNK].copy(), k) for lo in range(0, N, CHUNK)]) - Zh[:, k]
        assert np.max(np.abs(r)) <= BISECT_RESID + 1e-12, (tag, k, np.max(np.abs(r)))   # + rounding of S
        worst = max(worst, np.max(np.abs(r)))
    print('inverse %s N=%d: subsample %.1e, residual %.2e' % (tag, N, rel_err(Xh[sub], ref), worst))


def test_separable_inverse_second_pass(sep_setup, monkeypatch):
    """Per-component table and bisection inverse kernels (TTM_INV_FUSED=0) at an N where they make a second
    grid-stride pass; Z is a CUDA tensor, so the whole ensemble goes through one launch per component."""
    sm, N, Xr, mon, non, tm = sep_setup
    s = dec.sep_eval(N, sm)
    assert s.loops_min >= 3 and s.partial
    monkeypatch.setenv('TTM_INV_FUSED', '0')
    Zh = np.asarray(tm.map(Xr.copy()))
    Xs = (Xr - tm.X_mean) / tm.X_std
    for table in (True, False):
        tm.alternate_root_finding = table
        om = _oracle_full(Xr, Xs, mon, non, tm, monotonicity='separable monotonicity', alternate_root_finding=table)
        _inverse_checks(tm, om, Zh, N, sm, table, 'table' if table else 'bisection')
    tm.alternate_root_finding = True


def test_integrated_rectifier_bisection_second_pass():
    """Bisection inverse of a C4 map (D = 2) at the same N."""
    import torch
    from transport_map import transport_map
    sm = _sm_count()
    N = dec.sizes(sm)['sep']
    mon, non = c4_terms(2)
    Xr = _ensemble(N, 2, seed=90, bump=dec.sep_eval(N, sm).second)
    kw = dict(monotonicity='integrated rectifier', quadrature_input={'order': GEN_Q})
    tm = transport_map(X=Xr.copy(), monotone=mon, nonmonotone=non, polynomial_type='hermite function',
                       verbose=False, **kw)
    for k in range(2):
        c = _coeffs(mon, non, k, seed=91 + k, scale=0.2)
        tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:len(non[k])], c[len(non[k]):]
    Zh = tm.map(torch.from_numpy(Xr).cuda()).cpu().numpy()
    om = _oracle_full(Xr, (Xr - tm.X_mean) / tm.X_std, mon, non, tm, **kw)
    _inverse_checks(tm, om, Zh, N, sm, False, 'IR bisection')


def test_separable_lockstep_fit_matches_oracle():
    """optimize() of a separable map fits its components in lockstep: one batched K-sepobj launch per L-BFGS-B round
    (grid 8 SM / active components).  Its coefficients must reach the oracle's fit to 1e-6."""
    from transport_map import transport_map
    from ttm_oracle import OracleMap
    from ttt_b200 import hostopt
    assert hostopt.lbfgsb_available()
    sm = _sm_count()
    N, D = dec.sizes(sm)['sep'], dec.SEP_FIT_D
    for nact in range(1, D + 1):
        sp = dec.sepobj(N, sm, nact)
        assert sp.loops_min >= 3 and sp.partial, (nact, sp)
    mon, non = c5_terms(D)
    Xr = _ensemble(N, D, seed=95, bump=dec.sepobj(N, sm, D).second)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity',
              polynomial_type='hermite function', verbose=False)
    tm = transport_map(X=Xr.copy(), **kw)
    tm.optimize()
    om = OracleMap(X=Xr.copy(), **kw)
    om.optimize()
    worst = 0.0
    for k in range(D):
        for mine, theirs in ((tm.coeffs_mon[k], om.coeffs_mon[k]), (tm.coeffs_nonmon[k], om.coeffs_nonmon[k])):
            assert rel_err(mine, theirs) <= 1e-6, (k, rel_err(mine, theirs))
            worst = max(worst, rel_err(mine, theirs))
    print('lockstep fit N=%d D=%d: coefficients %.1e' % (N, D, worst))


# ------------------------------------------------------------------------------------------------ K-std
@pytest.mark.parametrize('D', dec.STD_DS)
@pytest.mark.parametrize('dtype', ['float64', 'float32'])
def test_colstats_at_looping_n(D, dtype):
    """Mean and standard deviation of CUDA-tensor columns with a large offset and a small spread (1e3 + 1e-2 x)
    against a long-double two-pass computation."""
    import torch
    from transport_map import transport_map
    sm = _sm_count()
    N = dec.sizes(sm)['std'][D]
    splits = dec.colstats(N, D, sm)
    assert all(s.loops_min >= 3 and (s.partial or dec.ragged_sweep(s, N)) for s in splits), splits
    rng = np.random.default_rng(D)
    Xh = (1e3 + 1e-2 * rng.standard_normal((N, D))).astype(dtype)
    Xd = torch.from_numpy(Xh).cuda()
    tm = transport_map(X=Xd, monotone=[[[D - 1]]], nonmonotone=[[[]]], monotonicity='separable monotonicity',
                       polynomial_type='hermite function', verbose=False)
    mean, sd = np.asarray(tm.X_mean), np.asarray(tm.X_std)
    worst = 0.0
    for j in range(D):
        col = Xh[:, j].astype(np.longdouble)
        mu = col.sum() / N
        var = ((col - mu) ** 2).sum() / N
        assert abs(mean[j] - float(mu)) <= TOL * float(mu), (j, mean[j], mu)
        assert abs(sd[j] - float(np.sqrt(var))) <= TOL * float(np.sqrt(var)), (j, sd[j], np.sqrt(var))
        worst = max(worst, abs(mean[j] / float(mu) - 1), abs(sd[j] / float(np.sqrt(var)) - 1))
    print('colstats N=%d D=%d %s: %.1e' % (N, D, dtype, worst))
