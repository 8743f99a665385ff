"""Host arrays against CUDA tensors through the class API (round 3).

For each workload, three figures of the same call, median per call over >= 0.5 s of repetitions after a warm-up:
  host_ms    -- numpy arrays in and out (pageable host memory), host clock around the call;
  tensor_ms  -- CUDA tensors in and out, host clock around the call ending in a device synchronise;
  device_ms  -- CUDA events recorded on the current stream around the CUDA-tensor call: the device timeline of the
                call (kernels, coefficient-sized copies and the gaps between them), without the host time before
                the first launch and after the last.
Working sets above the 126 MB L2 except C2 (24 MB), where a 512 MB buffer is overwritten before every pass.
K-std (colstats + standardise/transpose) at 10^6 x 256 is timed directly on the C ABI with CUDA events for contiguous
float64, a float64 column view X[:, 32:288] of a (10^6, 320) array and float32; bytes = 3 reads of the input + 1 write
of 8 N D (the round-2 accounting).  The card's name, clocks and power limit are queried in the same run.

usage: python tools/time_device_api.py [--out profiles/device_api_r3.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch                                                         # noqa: E402
from cases import synthetic_samples, c5_terms, ex05_terms, ex06_terms, ex06_cycle_inputs   # noqa: E402
from transport_map import transport_map                              # noqa: E402
from ttt_b200 import binding as B                                    # noqa: E402

MIN_S = 0.5
flush_buf = None


def sync():
    torch.cuda.synchronize()


def flush_l2():
    flush_buf.zero_()
    sync()


def wall(fn, flush=False):
    fn()
    sync()
    ts = []
    while len(ts) < 3 or sum(ts) < MIN_S:
        if flush:
            flush_l2()
        t = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t)
    return 1e3 * float(np.median(ts)), len(ts)


def events(fn, flush=False):
    fn()
    sync()
    ts = []
    while len(ts) < 3 or sum(ts) < 1e3 * MIN_S:
        if flush:
            flush_l2()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        sync()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), len(ts)


def three(name, host_fn, dev_fn, n, flush=False, **extra):
    h, nh = wall(host_fn, flush)
    t, nt = wall(dev_fn, flush)
    d, nd = events(dev_fn, flush)
    rec = {'workload': name, 'samples': n, 'host_ms': h, 'tensor_ms': t, 'device_ms': d,
           'host_samples_per_s': n / h * 1e3, 'tensor_samples_per_s': n / t * 1e3, 'device_samples_per_s': n / d * 1e3,
           'tensor_over_device': t / d, 'reps': [nh, nt, nd], 'l2_flushed': flush}
    rec.update(extra)
    return rec


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm,clocks.mem,clocks.max.mem'
    r = subprocess.run(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True, text=True)
    return {'query': q, 'result': r.stdout.strip().splitlines(), 'torch_name': torch.cuda.get_device_name()}


def c5(D=256, E=128):
    mon, non = c5_terms(D)
    tm = transport_map(X=synthetic_samples(10000, D, seed=0), monotone=mon, nonmonotone=non,
                       monotonicity='separable monotonicity', verbose=False)
    tm.optimize()
    return tm


def run_c5(out):
    D, E = 256, 128
    tm = c5(D, E)
    ns = 1_250_000
    Xs = synthetic_samples(ns, D, seed=2)[:, :E].copy()
    Z = np.random.default_rng(1).standard_normal((ns, D - E))
    Xs_d, Z_d = torch.from_numpy(Xs).cuda(), torch.from_numpy(Z).cuda()
    same = bool(np.array_equal(tm.inverse_map(Z_d, X_star=Xs_d).cpu().numpy(), tm.inverse_map(Z, X_star=Xs)))
    out.append(three('C5 inverse_map (table, X_star E=128), D=256', lambda: tm.inverse_map(Z, X_star=Xs),
                     lambda: tm.inverse_map(Z_d, X_star=Xs_d), ns, bit_identical=same))
    del Xs_d, Z_d
    nm = 400_000
    X = synthetic_samples(nm, D, seed=3)
    X_d = torch.from_numpy(X).cuda()
    same = bool(np.array_equal(tm.map(X_d).cpu().numpy(), tm.map(X)))
    out.append(three('C5 map (K-map-rect), D=256', lambda: tm.map(X), lambda: tm.map(X_d), nm, bit_identical=same))


def run_c2(out):
    mon, non = ex05_terms()
    X5 = synthetic_samples(1000, 2, seed=5) * np.array([2.0, 0.5]) + np.array([1.0, -3.0])
    tm = transport_map(X=X5.copy(), monotone=mon, nonmonotone=non, monotonicity='separable monotonicity', verbose=False)
    tm.optimize()
    n = 1_000_000
    pts = np.random.default_rng(0).uniform(-3, 3, (n, 2)) * np.array([2.0, 0.5]) + np.array([1.0, -3.0])
    pd = torch.from_numpy(pts).cuda()
    same = bool(np.array_equal(tm.evaluate_pullback_density(pd).cpu().numpy(), tm.evaluate_pullback_density(pts)))
    out.append(three('C2 evaluate_pullback_density (K-pullback)', lambda: tm.evaluate_pullback_density(pts),
                     lambda: tm.evaluate_pullback_density(pd), n, flush=True, bit_identical=same))


def run_c3(out):
    mon, non = ex06_terms(3)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity', regularization='l2',
              regularization_lambda=0.05, verbose=False)
    for N in (1000, 10000, 100000):
        dummy, cyc = ex06_cycle_inputs(N)
        tm = transport_map(X=dummy.copy(), **kw)
        cyc_d = torch.from_numpy(cyc).cuda()
        ys, ys_d = np.full((N, 1), 1.5), torch.full((N, 1), 1.5, dtype=torch.float64, device='cuda')

        def cycle(m, X, y):
            m.reset(X)
            m.optimize()
            return m.inverse_map(m.map(X), X_star=y)
        same = bool(np.array_equal(cycle(tm, cyc_d, ys_d).cpu().numpy(), cycle(tm, cyc.copy(), ys)))
        out.append(three('C3 EnTF cycle (reset, optimize, map, inverse_map)', lambda: cycle(tm, cyc.copy(), ys),
                         lambda: cycle(tm, cyc_d, ys_d), N, flush=N * 4 * 8 * 4 < (126 << 20), bit_identical=same))


def run_kstd(out):
    N, D = 1_000_000, 256
    tm = transport_map(X=synthetic_samples(64, 2, seed=0), monotone=[[[0]], [[1]]], nonmonotone=[[[]], [[], [0]]],
                       verbose=False)
    base = torch.from_numpy(synthetic_samples(N, D + 64, seed=1)).cuda()
    variants = [('f64 contiguous', base[:, 32:32 + D].contiguous()), ('f64 column view X[:, 32:288]', base[:, 32:32 + D]),
                ('f32 contiguous', base[:, 32:32 + D].float().contiguous())]
    mean, sd = tm._empty(D), tm._empty(D)
    Xt = tm._empty(D, N)
    ref = None
    for label, X in variants:
        S = tm._samples(X)
        P = lambda t: B.c_void_p(t.data_ptr())

        def kstd():
            B.check(tm._lib.ttm_colstats_ld(tm._ctx, P(S.t), S.code, S.ld, N, D, P(mean), P(sd), P(tm._scratch),
                                            tm._stream()))
            B.check(tm._lib.ttm_standardize_transpose_ld(tm._ctx, P(S.t), S.code, S.ld, N, D, P(mean), P(sd), P(Xt), N,
                                                         tm._stream()))
        ms, reps = events(kstd)
        es = X.element_size()
        nbytes = 3 * es * N * D + 8 * N * D
        res = torch.cat((mean, sd, Xt[:, :1000].reshape(-1))).cpu().numpy()
        if ref is None:
            ref = res
        out.append({'workload': 'K-std colstats + standardize_transpose, N=1e6, D=256, ' + label, 'device_ms': ms,
                    'reps': reps, 'bytes': nbytes, 'TBps': nbytes / ms / 1e9,
                    'same_bits_as_f64_contiguous': bool(np.array_equal(res, ref)) if es == 8 else None,
                    'round2_reference_TBps': 4.4})


def main():
    global flush_buf
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'device_api_r3.json'))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement runs on the GPU only')
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device='cuda')
    res = {'gpu': gpu_info(), 'results': []}
    for step in (run_kstd, run_c2, run_c5, run_c3):
        try:
            step(res['results'])
        except Exception as e:                                       # noqa: BLE001
            res['results'].append({'workload': step.__name__, 'error': repr(e)})
        print(json.dumps(res['results'][-1]), flush=True)
    res['gpu_after'] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['gpu']))


if __name__ == '__main__':
    main()
