"""Cost of the log-density evaluators (evaluate_log_pullback_density / evaluate_log_pushforward_density).

All inputs and outputs are CUDA tensors; every figure is the median of CUDA-event times (current stream) over >= 0.5 s
of repetitions after a warm-up, with a 512 MB buffer overwritten before every timed call so that no pass reads
the previous one's working set out of the 126 MB L2.
  * C4 (D = 64, N = 10^6, Q = 100 and 25, coefficients N(0, 0.05^2)): map(X) against evaluate_log_pullback_density(X),
    and K-logdet-IR alone (64 launches of ttm_ir_logdet_accumulate, mode 0, on a precomputed S) with its bytes,
    8 N x (x_c + outer columns + S + acc read + acc write) per component, over its time as a share of 7.7 TB/s.
  * C2 (Example-05 separable map fitted on 1000 samples, 10^6 points): evaluate_pullback_density against
    evaluate_log_pullback_density (both K-map-fused).
  * IR pushforward, C4 D = 64, N = 10^5 (Q = 100): the whole call and inverse_map alone (bisection).
The card's name, power limit and clocks are queried in the same run.

usage: python tools/time_log_density.py [--out profiles/log_density_r5.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch                                                         # noqa: E402
from cases import synthetic_samples, c4_terms, ex05_terms            # noqa: E402
from transport_map import transport_map                              # noqa: E402
from ttt_b200 import binding as B                                    # noqa: E402

MIN_MS = 500.0
HBM_BYTES_PER_S = 7.7e12
flush_buf = None


def events(fn):
    fn()
    torch.cuda.synchronize()
    ts = []
    while len(ts) < 3 or sum(ts) < MIN_MS:
        flush_buf.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), len(ts)


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm,clocks.mem,clocks.max.mem'
    r = subprocess.run(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True, text=True)
    return {'query': q, 'result': r.stdout.strip().splitlines(), 'torch_name': torch.cuda.get_device_name()}


def c4_map(X, Q, D=64):
    mon, non = c4_terms(D)
    tm = transport_map(X=X, monotone=mon, nonmonotone=non, quadrature_input={'order': Q}, verbose=False)
    rng = np.random.default_rng(56)
    for k in range(D):
        c = rng.standard_normal(len(non[k]) + len(mon[k])) * 0.05
        tm.coeffs_nonmon[k], tm.coeffs_mon[k] = c[:len(non[k])].copy(), c[len(non[k]):].copy()
    return tm


def logdet_alone(tm, X):
    """64 K-logdet-IR launches on the standardised samples and a fixed S; coefficients set once per plan."""
    Xs, n, _ = tm._density_input(X, None, tm._Dtot)
    Xt = tm._to_colmajor(Xs, tm._mean_d, tm._std_d)                 # the C4 map standardises its samples
    S = torch.zeros(n, dtype=torch.float64, device=X.device)
    acc = torch.zeros(n, dtype=torch.float64, device=X.device)
    sig = tm._sigmas(tm.skip_dimensions, log=True)
    for k in range(tm.D):
        tm._set_coeffs(k, tm.coeffs_nonmon[k], tm.coeffs_mon[k])
    ptr = lambda t: B.c_void_p(t.data_ptr())

    def run():
        st = tm._stream()
        for k in range(tm.D):
            B.check(tm._lib.ttm_ir_logdet_accumulate(tm._plans[k], ptr(Xt), Xt.shape[1], n, ptr(S), sig[k], 0,
                                                     ptr(acc), st))
    ms, reps = events(run)
    outer = [len({int(f) for term in tm.monotone[k] for f in term if not isinstance(f, str) and int(f) != k + tm.skip_dimensions})
             for k in range(tm.D)]
    nbytes = sum(8 * n * (4 + o) for o in outer)                     # x_c + outer columns + S + acc read/write
    return {'ms': ms, 'reps': reps, 'bytes': nbytes, 'TB_per_s': nbytes / ms / 1e9,
            'share_of_7.7TB_per_s': nbytes / ms / 1e9 / (HBM_BYTES_PER_S / 1e12)}


def main():
    global flush_buf
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'log_density_r5.json'))
    a = ap.parse_args()
    flush_buf = torch.empty(64 * 1024 * 1024, dtype=torch.float64, device='cuda')
    res = {'gpu': gpu_info(), 'min_ms_per_figure': MIN_MS, 'l2_flush_bytes': flush_buf.numel() * 8, 'runs': []}
    N, D = 1_000_000, 64
    X = torch.from_numpy(synthetic_samples(N, D, seed=55)).cuda()
    for Q in (100, 25):
        tm = c4_map(X, Q)
        m_ms, m_reps = events(lambda: tm.map(X))
        l_ms, l_reps = events(lambda: tm.evaluate_log_pullback_density(X))
        rec = {'workload': 'C4 D=64 N=1e6 Q=%d' % Q, 'map_ms': m_ms, 'map_reps': m_reps,
               'log_pullback_ms': l_ms, 'log_pullback_reps': l_reps, 'log_pullback_over_map': l_ms / m_ms,
               'k_logdet_ir_alone': logdet_alone(tm, X)}
        rec['k_logdet_ir_share_of_log_pullback'] = rec['k_logdet_ir_alone']['ms'] / l_ms
        res['runs'].append(rec)
        print(json.dumps(rec), flush=True)
        del tm
    mon, non = ex05_terms()
    X5 = synthetic_samples(1000, 2, seed=5) * np.array([2.0, 0.5]) + np.array([1.0, -3.0])
    tm = transport_map(X=X5.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity', verbose=False)
    tm.optimize()
    pts = torch.from_numpy(np.random.default_rng(0).uniform(-3, 3, (N, 2)) * np.array([2.0, 0.5])
                           + np.array([1.0, -3.0])).cuda()
    p_ms, p_reps = events(lambda: tm.evaluate_pullback_density(pts))
    l_ms, l_reps = events(lambda: tm.evaluate_log_pullback_density(pts))
    rec = {'workload': 'C2 Example-05 separable, 1e6 points', 'pullback_ms': p_ms, 'pullback_reps': p_reps,
           'log_pullback_ms': l_ms, 'log_pullback_reps': l_reps}
    res['runs'].append(rec)
    print(json.dumps(rec), flush=True)
    tm = c4_map(X, 100)
    n = 100_000
    Z = torch.from_numpy(np.random.default_rng(57).standard_normal((n, D))).cuda()
    target = lambda x: -0.5 * (x ** 2).sum(dim=1)
    t_ms, t_reps = events(lambda: tm.evaluate_log_pushforward_density(Z, target))
    i_ms, i_reps = events(lambda: tm.inverse_map(Z))
    rec = {'workload': 'C4 D=64 Q=100 log pushforward, 1e5 samples', 'total_ms': t_ms, 'total_reps': t_reps,
           'inverse_map_ms': i_ms, 'inverse_map_reps': i_reps, 'inverse_share': i_ms / t_ms}
    res['runs'].append(rec)
    print(json.dumps(rec), flush=True)
    res['gpu_after'] = gpu_info()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
