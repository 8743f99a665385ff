"""Device-time K-inv-fused against the per-component K-inv-table path on the C5 shape (D=256, E=128), inputs resident
in HBM; checks that both give the same samples.  Prints one JSON line."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch                                             # noqa: E402
from cases import synthetic_samples, c5_terms, headline_sep_coeffs            # noqa: E402
from transport_map import transport_map                  # noqa: E402
from ttt_b200 import binding as B                        # noqa: E402

D = int(os.environ.get('TTM_D', 256))
E = D // 2
n = int(os.environ.get('TTM_NS', 1_250_000))
mon, non = c5_terms(D)
tm = transport_map(X=synthetic_samples(2000, D, seed=0), monotone=mon, nonmonotone=non,
                   monotonicity='separable monotonicity', verbose=False)
cm, cn = headline_sep_coeffs(mon, non)
for k in range(D):
    tm.coeffs_mon[k], tm.coeffs_nonmon[k] = cm[k].copy(), cn[k].copy()
comps = [(i, k) for i, k in enumerate(range(E, D))]
t0 = time.perf_counter()
fused = tm._inverse_fused_setup(comps)
torch.cuda.synchronize()
out = {'D': D, 'E': E, 'n': n, 'setup_s': time.perf_counter() - t0, 'fused_available': fused is not None}
t0 = time.perf_counter()
fused = tm._inverse_fused_setup(comps)
torch.cuda.synchronize()
out['setup_again_s'] = time.perf_counter() - t0
g = torch.Generator(device='cuda').manual_seed(0)
Xw = torch.zeros(D, n, dtype=torch.float64, device='cuda')
Xw[:E] = torch.randn(E, n, dtype=torch.float64, device='cuda', generator=g)
Zt = torch.randn(D - E, n, dtype=torch.float64, device='cuda', generator=g)
def timed(fz):
    base = torch.empty(D - E, (n + 1) // 2 * 2, dtype=torch.float64, device='cuda') if fz.get('R') is not None else None
    ts = []
    for rep in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tm._inverse_fused_launch(fz, Xw, n, n, Zt, n, base=base)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    return ts


# one launch (walk over every column) vs K-inv-rect + walk over the solved columns
os.environ['TTM_INV_SPLIT'] = '0'
f_single = tm._inverse_fused_setup(comps)
ts = timed(f_single)
out['single_s'] = min(ts[1:])
X_single = Xw[E:].clone()
os.environ['TTM_INV_SPLIT'] = 'auto'
fused = tm._inverse_fused_setup(comps)
out['split'] = fused.get('R') is not None
ts = timed(fused)
out['split_vs_single_maxabs'] = float((Xw[E:] - X_single).abs().max())
out['fused_s'] = min(ts[1:])
out['fused_samples_per_s'] = n / out['fused_s']
out['algorithmic_bytes'] = 8 * n * (E + 2 * (D - E))
out['fused_algorithmic_gbs'] = out['algorithmic_bytes'] / out['fused_s'] / 1e9
Xf = Xw[E:].clone()
# per-component reference path on the first 200k samples
m = min(n, 200_000)
Xw2 = torch.zeros(D, m, dtype=torch.float64, device='cuda')
Xw2[:E] = Xw[:E, :m]
Zt2 = Zt[:, :m].contiguous()
torch.cuda.synchronize()
t0 = time.perf_counter()
os.environ['TTM_INV_FUSED'] = '0'
tm._inverse_solve(tm._inverse_solver(comps, True), Xw2, m, m, Zt2, m, tm._stream())
torch.cuda.synchronize()
del os.environ['TTM_INV_FUSED']
out['per_component_s_200k'] = time.perf_counter() - t0
out['max_abs_diff_vs_per_component'] = float((Xf[:, :m] - Xw2[E:]).abs().max())
print(json.dumps(out))
