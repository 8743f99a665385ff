import os, sys, time, json
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
from cases import synthetic_samples, c5_terms
from transport_map import transport_map
D, E, ns = 256, 128, 1_250_000
mon, non = c5_terms(D)
tm = transport_map(X=synthetic_samples(4000, D, seed=0), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity', verbose=False)
rng = np.random.default_rng(0)
for k in range(D):
    tm.coeffs_nonmon[k] = rng.standard_normal(len(non[k])) * 0.05
    tm.coeffs_mon[k] = np.abs(rng.standard_normal(4)) + 0.2
Xstar = synthetic_samples(ns, D, seed=2)[:, :E].copy()
Z = rng.standard_normal((ns, D - E))
def T(f):
    torch.cuda.synchronize(); t = time.perf_counter(); r = f(); torch.cuda.synchronize(); return r, time.perf_counter() - t
tm.inverse_map(Z[:1000], X_star=Xstar[:1000])
_, t_all = T(lambda: tm.inverse_map(Z, X_star=Xstar))
zt, t_h2d = T(lambda: tm._to_colmajor(Z))
xs, t_h2d2 = T(lambda: tm._to_colmajor(Xstar, tm._mean_d[:E].contiguous(), tm._std_d[:E].contiguous()))
Xw = torch.zeros(D, ns, dtype=torch.float64, device='cuda'); Xw[:E] = xs
def comps():
    os.environ['TTM_INV_FUSED'] = '0'            # the per-component K-inv-table path
    tm._inverse_solve(tm._inverse_solver([(i, k) for i, k in enumerate(range(E, D))], True), Xw, ns, ns, zt, ns,
                      tm._stream())
    del os.environ['TTM_INV_FUSED']
_, t_comp = T(comps)
_, t_d2h = T(lambda: tm._to_rowmajor(Xw, ns, D, tm._mean_d, tm._std_d))
print(json.dumps({'total_s': t_all, 'h2d_Z_s': t_h2d, 'h2d_Xstar_s': t_h2d2, 'components_s': t_comp, 'd2h_s': t_d2h}))
