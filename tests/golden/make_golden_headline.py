"""
Golden fixtures at the HEADLINE shapes (BASELINE.json configs C4 / C5), produced by the UNMODIFIED reference.

Run in the build container only (needs /root/reference, numpy 2.3.5, scipy 1.18.1):

    python tests/golden/make_golden_headline.py [c4_objgrad] [c4_fit] [sep_fit_64] [sep_fit_128] [c5_inverse]

Inputs are seeded recipes from tests/cases.py (nothing of size N is stored), outputs are what the GPU tests
compare against:

  headline_c4_objgrad.npz   C4 at D=64 on N=4000 rows: J_k and grad J_k for k in {0,1,5,31,63}, Q in {25,100}
                            (tm.py:3300-3635), at seeded coefficient vectors
  headline_c4_fit.npz       full D=64 optimize() (BFGS, tm.py:3252-3257) at N=4000, Q=100: all 6367 coefficients,
                            J_k at the optimum and map() of the first 256 training rows
  headline_sep_fit_<D>.npz  separable C5-pattern fit (QR path, tm.py:2966-2975 + L-BFGS-B :3108) at D=64 and D=128,
                            N=4000 (m_non up to 382): coefficients + map() head
  headline_c5_inverse.npz   C5 at D=256, E=128 conditioning columns: table and bisection inverse_map
                            (tm.py:3639-4084) at seeded coefficients: the solved columns X[:, E:] of a fixed
                            sample of the rows, with the row indices (all of it would pass 1 MB)

The reference's own process pool (workers = cpu_count, tm.py:2789-2845) is used for the fits.
"""

import copy
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, '..'))
sys.path.insert(0, '/root/reference')

import scipy                                                     # noqa: E402
from transport_map import transport_map                          # noqa: E402  (the reference)
from cases import (synthetic_samples, c4_terms, c5_terms, headline_coeffs, headline_sep_coeffs,  # noqa: E402
                   HEADLINE_N, HEADLINE_KS, HEADLINE_QS, C5_INV)

VERS = np.asarray('numpy %s scipy %s' % (np.__version__, scipy.__version__))
WORKERS = os.cpu_count() or 1


def save(name, out):
    out['_versions'] = VERS
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
    print('%-28s %3d arrays' % (name, len(out)), flush=True)


def c4_objgrad():
    D = 64
    mon, non = c4_terms(D)
    X = synthetic_samples(HEADLINE_N, D, seed=0)
    out = {}
    for Q in HEADLINE_QS:
        tm = transport_map(X=copy.copy(X), monotone=mon, nonmonotone=non, polynomial_type='hermite function',
                           monotonicity='integrated rectifier', quadrature_input={'order': Q}, verbose=False)
        for k in HEADLINE_KS:
            c = headline_coeffs(mon, non, k)
            div = len(non[k])
            out['J_q%d_k%d' % (Q, k)] = np.asarray(tm.objective_function(c.copy(), k, div))
            out['grad_q%d_k%d' % (Q, k)] = np.asarray(tm.objective_function_jacobian(c.copy(), k, div))
    save('headline_c4_objgrad', out)


def c4_fit():
    D = 64
    mon, non = c4_terms(D)
    X = synthetic_samples(HEADLINE_N, D, seed=0)
    tm = transport_map(X=copy.copy(X), monotone=mon, nonmonotone=non, polynomial_type='hermite function',
                       monotonicity='integrated rectifier', quadrature_input={'order': 100}, verbose=False,
                       workers=WORKERS)
    t = time.perf_counter()
    tm.optimize()
    out = {'optimize_s': np.asarray(time.perf_counter() - t), 'workers': np.asarray(WORKERS)}
    # (the pool path deletes fun_mon / fun_nonmon, tm.py:2812, and optimize() restores them, tm.py:2876-2899)
    for k in range(D):
        out['coeffs_mon_%d' % k] = np.array(tm.coeffs_mon[k])
        out['coeffs_nonmon_%d' % k] = np.array(tm.coeffs_nonmon[k])
        c = np.concatenate((tm.coeffs_nonmon[k], tm.coeffs_mon[k]))
        out['J_%d' % k] = np.asarray(tm.objective_function(c, k, len(tm.coeffs_nonmon[k])))
    out['map_head'] = tm.map(copy.copy(X[:256]))
    save('headline_c4_fit', out)
    print('  reference optimize(): %.1f s with %d workers' % (float(out['optimize_s']), WORKERS), flush=True)


def sep_fit(D):
    mon, non = c5_terms(D)
    X = synthetic_samples(HEADLINE_N, D, seed=0)
    tm = transport_map(X=copy.copy(X), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity',
                       verbose=False, workers=WORKERS)
    t = time.perf_counter()
    tm.optimize()
    out = {'optimize_s': np.asarray(time.perf_counter() - t), 'workers': np.asarray(WORKERS)}
    for k in range(D):
        out['coeffs_mon_%d' % k] = np.array(tm.coeffs_mon[k])
        out['coeffs_nonmon_%d' % k] = np.array(tm.coeffs_nonmon[k])
    out['map_head'] = tm.map(copy.copy(X[:256]))
    save('headline_sep_fit_%d' % D, out)
    print('  reference optimize(): %.1f s with %d workers' % (float(out['optimize_s']), WORKERS), flush=True)


def c5_inverse():
    D, E, ntrain, n_tab, n_bis = C5_INV['D'], C5_INV['E'], C5_INV['ntrain'], C5_INV['n_table'], C5_INV['n_bisect']
    mon, non = c5_terms(D)
    tm = transport_map(X=synthetic_samples(ntrain, D, seed=0), monotone=mon, nonmonotone=non,
                       monotonicity='separable monotonicity', verbose=False)
    cm, cn = headline_sep_coeffs(mon, non)
    tm.coeffs_mon, tm.coeffs_nonmon = copy.deepcopy(cm), copy.deepcopy(cn)
    rng = np.random.default_rng(C5_INV['seed'])
    Xstar = synthetic_samples(n_tab, D, seed=C5_INV['seed'] + 1)[:, :E].copy()
    Z = rng.standard_normal((n_tab, D - E))
    pick = np.random.default_rng(0)
    rt = np.sort(pick.choice(n_tab, 200, replace=False))
    rb = np.sort(pick.choice(n_bis, 80, replace=False))
    out = {'rows_table': rt, 'rows_bisect': rb}
    tm.alternate_root_finding = True
    out['inverse_table'] = tm.inverse_map(copy.copy(Z), X_star=copy.copy(Xstar))[rt, E:]
    tm.alternate_root_finding = False
    out['inverse_bisect'] = tm.inverse_map(copy.copy(Z[:n_bis]), X_star=copy.copy(Xstar[:n_bis]))[rb, E:]
    save('headline_c5_inverse', out)


if __name__ == '__main__':
    todo = sys.argv[1:] or ['c4_objgrad', 'c4_fit', 'sep_fit_64', 'sep_fit_128', 'c5_inverse']
    print('numpy', np.__version__, 'scipy', scipy.__version__, 'workers', WORKERS, flush=True)
    for name in todo:
        t0 = time.perf_counter()
        if name == 'c4_objgrad':
            c4_objgrad()
        elif name == 'c4_fit':
            c4_fit()
        elif name.startswith('sep_fit_'):
            sep_fit(int(name.split('_')[-1]))
        elif name == 'c5_inverse':
            c5_inverse()
        else:
            raise SystemExit('unknown fixture ' + name)
        print('  [%s: %.1f s]' % (name, time.perf_counter() - t0), flush=True)
