"""
bench.py -- headline metric of BASELINE.json on B200:

    objective+gradient evals/sec at N = 1M, K = 64   (config C4 of SURVEY.md section 8(d):
    synthetic D = 64 map, order-3 Hermite-function integrated rectifier, Q = 100 quadrature nodes)

One *eval* = one (J_k, grad J_k) pair of ONE component over all N samples, i.e. what one
`objective_function` + `objective_function_jacobian` callback pair of scipy costs in the reference
(tm.py:3300 + :3435).  One *step* = the 64 evals of all components (one pass of the hot path over
the ensemble).  With --gpus N the 64 components are sharded over the ranks (strong scaling, no
data-path collective); value = 64 * steps / max-over-ranks device time.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`--impl reference` times the CPU port of the reference algorithm (oracle/ttm_oracle.py, component-
parallel over all host cores like the reference's multiprocessing Pool, tm.py:2789-2845) on a bounded
sample of the same workload.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from cases import synthetic_samples, c4_terms, c5_terms    # noqa: E402  (workload recipes shared with the parity tests)

D, N_FULL, Q = 64, 1_000_000, 100
METRIC = 'objective+gradient evals/sec at N=1M, K=64'
UNIT = 'evals/s'


def flops_per_eval(k, n, q=Q, m_mon=4, c_exp=30):
    """Algorithmic FP64 work of one eval, SURVEY.md 8(d): node loop Q*(8 + c_exp + m_m + 2 m_m + c_exp + 2 + 1 + 2 m_m)
    + x_<c part (c_exp + 18) k + epilogue 75 (c_log = 47), per sample.  c_exp = 30 is the survey's frozen cost of the
    CUDA library exp; c_exp = 14 re-freezes it for the exp the kernel ships (ttm_exp.cuh: 6 FMA + 1 ADD + 1 MUL)."""
    mm = 3 if k == 0 else m_mon
    node = q * (8 + c_exp + mm + 2 * mm + c_exp + 2 + 1 + 2 * mm)
    return n * (node + (c_exp + 18) * k + 75)


def flops_executed(k, n, q=Q):
    """FP64 flops the shipped tile kernel actually executes per eval (SASS instruction mix, FMA = 2): node loop 27
    instructions = 20 FMA + 7 MUL/ADD = 47 flop per node; Gram-mode sweep 21 instructions = 12 FMA + 9 = 33 flop per
    (sample, column); prologue + epilogue (two exp, log, division, slot algebra) ~300 flop per sample."""
    return n * (47 * q + 33 * k + 300)


def bytes_per_eval(k, n):
    return 8 * n * (k + 1)


def coefficients(mon, non, seed=0):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(len(non[k]) + len(mon[k])) * 0.05 for k in range(len(mon))]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.samples, self.active = gpu_index, [], False
        self.nearby = []            # samples outside the timed window (the GPU is busy before and after it as well)
        self.t_on = self.t_off = None
        self.proc = None

    def run(self):
        try:
            # -i: this rank's GPU only (every rank polling every GPU is N^2 driver queries per period)
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu_index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                p = [t.strip() for t in line.split(',')]
                if len(p) >= 8 and p[0] == str(self.gpu_index):
                    (self.samples if self.active else self.nearby).append((time.perf_counter(), p))
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self):
        use, pad = [p for _, p in self.samples], 0.0
        if len(use) < 2 and self.t_on is not None:
            # the timed window is shorter than the sampling period (multi-GPU runs: ~50 ms): take the samples within
            # 0.3 s around it -- the per-launch pass before and the fit after keep the GPU under the same load
            pad = 0.3
            use += [p for t, p in self.nearby if self.t_on - pad <= t <= (self.t_off or t) + pad]
        if not use:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        sm = sorted(float(s[1]) for s in use)
        reasons = []
        for idx, name in ((4, 'hw_slowdown'), (5, 'hw_thermal_slowdown'), (6, 'sw_thermal_slowdown'), (7, 'sw_power_cap')):
            if any(s[idx].lower().startswith('active') for s in use):
                reasons.append(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(use[0][2]),
                'power_w_max': max(float(s[3]) for s in use), 'reasons': reasons, 'samples': len(sm),
                'samples_in_window': len(self.samples), 'window_padding_s': pad}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port, component-parallel like the reference's Pool
# ------------------------------------------------------------------------------------------------
_OM = None
_CPU_VALUES = {}


def _cpu_eval(args):
    k, c = args
    div = len(_OM.coeffs_nonmon[k])
    t = time.perf_counter()
    f = _OM.objective_function(c, k, div)
    g = _OM.objective_function_jacobian(c, k, div)
    return time.perf_counter() - t, k, float(f), np.asarray(g, dtype=np.float64)


def cpu_port(n_sample, ks, workers, steps=1, warmup=0):
    """Times objective+jacobian of the listed components on an n_sample-row sample of the C4 workload.
    Returns (evals/s scaled linearly to N = 1M, seconds per step)."""
    global _OM
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    from ttm_oracle import OracleMap
    os.environ.setdefault('OPENBLAS_NUM_THREADS', '1' if workers > 1 else str(os.cpu_count()))
    X = synthetic_samples(n_sample, D, seed=0)
    mon, non = c4_terms(D)
    _OM = OracleMap(X=X, monotone=mon, nonmonotone=non, monotonicity='integrated rectifier',
                    quadrature_input={'order': Q})
    coefs = coefficients(mon, non)
    work = [(k, coefs[k]) for k in sorted(ks, reverse=True)]      # longest first (tm.py:2821)
    times, res = [], []
    if workers > 1:
        from multiprocessing import get_context
        with get_context('fork').Pool(workers) as pool:
            for s in range(warmup + steps):
                t = time.perf_counter()
                res = pool.map(_cpu_eval, work, chunksize=1)
                if s >= warmup:
                    times.append(time.perf_counter() - t)
    else:
        for s in range(warmup + steps):
            t = time.perf_counter()
            res = [_cpu_eval(w) for w in work]
            if s >= warmup:
                times.append(time.perf_counter() - t)
    per_step = float(np.mean(times))
    global _CPU_VALUES
    _CPU_VALUES = {k: (f, g) for _, k, f, g in res}               # oracle (J, grad) per component: the parity leg
    return len(ks) / per_step * (n_sample / N_FULL), per_step


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, D))
    n_sample = 4000
    t0 = time.perf_counter()
    value, per_step = cpu_port(n_sample, list(range(D)), workers, steps=args.steps, warmup=args.warmup)
    sample = ('all 64 components of C4 (D=64, Q=100) on the first %d samples, evals/s scaled linearly to N=1M '
              '(the port materialises every Psi like the reference: N=1M needs ~54 GB)' % n_sample)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': per_step * 1e3 * (N_FULL / n_sample), 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'C4: synthetic D=64 integrated-rectifier map, order-3 Hermite functions, Q=100, N=1M',
                   'sample_rows': n_sample},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': workers, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'wall_s': time.perf_counter() - t0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# secondary metric M2: conditional sampling via inverse_map (config C5)
# ------------------------------------------------------------------------------------------------
def inverse_metric(rank, world, dist, torch, with_cpu=False):
    """C5 (SURVEY.md 8(d)): D=256 separable map (LET/iRBF/iRBF/RET + order-3 nonmonotone terms), trained on 10^4
    samples (components sharded over the ranks, one all-gather), then inverse_map(Z, X_star) with E=128
    conditioning columns on 1.25M samples PER GPU (10M over 8 GPUs), through the public class API with host
    arrays in and out.  Samples shard with no collective."""
    from transport_map import transport_map
    Dm, E, ntrain, ns = 256, 128, 10000, 1_250_000
    mon, non = c5_terms(Dm)
    t = time.perf_counter()
    tm = transport_map(X=synthetic_samples(ntrain, Dm, seed=0), monotone=mon, nonmonotone=non,
                       monotonicity='separable monotonicity', verbose=False)
    ctor_s = time.perf_counter() - t
    t = time.perf_counter()
    tm.optimize()
    torch.cuda.synchronize()
    opt_s = time.perf_counter() - t
    rng = np.random.default_rng(100 + rank)
    Xstar_pg = synthetic_samples(ns, Dm, seed=200 + rank)[:, :E].copy()
    Z_pg = rng.standard_normal((ns, Dm - E))
    # the step's inputs in PINNED host memory (the bench contract's e2e definition): inverse_map copies such arrays to the
    # device directly; pageable inputs (the `table_pageable` figure) go through the library's pinned staging buffers
    Xstar = torch.empty((ns, E), dtype=torch.float64, pin_memory=True).numpy()
    Z = torch.empty((ns, Dm - E), dtype=torch.float64, pin_memory=True).numpy()
    Xstar[:], Z[:] = Xstar_pg, Z_pg
    res = {}
    for mode, alt, n_use in (('table', True, ns), ('table_pageable', True, ns), ('bisection', False, 250_000)):
        tm.alternate_root_finding = alt
        if mode == 'table_pageable':
            Z, Xstar = Z_pg, Xstar_pg
        warm = tm.inverse_map(Z[:n_use], X_star=Xstar[:n_use])   # steady state: the first full-size call also pays a
        del warm                                                 # one-off pinned staging-buffer allocation (~2 s)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t = time.perf_counter()
        Xs = tm.inverse_map(Z[:n_use], X_star=Xstar[:n_use])
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        res[mode] = {'samples_per_s': n_use * world / float(dt[0]), 'samples': n_use * world, 'seconds': float(dt[0]),
                     # bytes that cross PCIe per call (Z and X* in, the solved columns out), all ranks together
                     'host_device_gbs': 8.0 * n_use * world * (E + 2 * (Dm - E)) / float(dt[0]) / 1e9}
        if not alt:
            resid = float(np.max(np.abs(tm.map(Xs[:20000])[:, E:] - Z[:20000])))
            res[mode]['max_residual'] = resid
    # ---- device-resident rate of the fused triangular solve (K-inv-fused) and its roofline
    comps = [(i, k) for i, k in enumerate(range(E, Dm))]
    fused = tm._inverse_fused_setup(comps)
    dev = None
    if fused is not None:
        g = torch.Generator(device='cuda').manual_seed(rank)
        Xw = torch.zeros(Dm, ns, dtype=torch.float64, device='cuda')
        Xw[:E] = torch.randn(E, ns, dtype=torch.float64, device='cuda', generator=g)
        Zt = torch.randn(Dm - E, ns, dtype=torch.float64, device='cuda', generator=g)
        ts = []
        base = (torch.empty(Dm - E, (ns + 1) // 2 * 2, dtype=torch.float64, device='cuda')
                if fused.get('R') is not None else None)           # scratch of K-inv-rect
        for rep in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tm._inverse_fused_launch(fused, Xw, ns, ns, Zt, ns, base=base)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        t_dev = torch.tensor([float(np.mean(ts[1:]))], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        t_dev = float(t_dev[0])
        alg_bytes = 8 * ns * (E + 2 * (Dm - E))                         # SURVEY 8(d): X* in, Z in, X out
        pairs = sum(k for k in range(E, Dm))                            # (variable, component) pairs per sample
        fl = ns * (2 * 3 * pairs + 30 * (Dm - E))                       # 3 FMA per pair + interpolation
        peak64 = None
        traffic = None
        try:
            peak64 = json.load(open(os.path.join(ROOT, 'profiles', 'fp64_peaks_r2.json'))).get('dfma_tflops')
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_inverse_traffic_r2.json')))
            traffic = tr['bytes_per_sample_split'] * ns if fused.get('R') is not None else None
        except Exception:
            pass
        dev = {'samples_per_s': ns * world / t_dev, 'seconds': t_dev,
               'kernels': ['inverse_rect_kernel (DMMA GEMM over the conditioning block)', 'inverse_fused_kernel (walk)']
               if fused.get('R') is not None else ['inverse_fused_kernel'],
               'roofline': {'bound': 'fp64', 'achieved': fl / t_dev / 1e12, 'peak': peak64, 'unit': 'TFLOP/s',
                            'frac': (fl / t_dev / 1e12 / peak64) if peak64 else None,
                            'flops_per_sample': fl / ns, 'algorithmic_bytes': alg_bytes,
                            'algorithmic_gbs': alg_bytes / t_dev / 1e9, 'traffic': traffic,
                            'traffic_ratio': (traffic / alg_bytes) if traffic else None,
                            'traffic_source': 'profiles/ncu_inverse_traffic_r2.json (ncu dram bytes of both kernels, scaled '
                                              'per sample)',
                            'how': 'conditional inverse, inputs resident in HBM, CUDA events over both launches; flops = 3 '
                                   'FMA per (sample, variable, component) pair of the triangular contraction (exp of the '
                                   'features, table search and interpolation not counted)'}}
        del base
        del Xw, Zt
    # ---- forward map of the same C5 map (all 256 components) through map() with host arrays: GEMM form of the
    # nonmonotone sums (ttm_map_rect) against the per-component kernels
    fwd = None
    if rank == 0:
        nm = 400_000
        Xm = synthetic_samples(nm, Dm, seed=300)
        fwd = {'points': nm}
        keep = {}
        for label, flag in (('gemm', '1'), ('per_component', '0')):
            os.environ['TTM_MAP_GEMM'] = flag
            tm._inv_pack_cache.pop('map_gemm', None)
            ts = []
            for rep in range(3):                       # (the first calls pay page faults of the 0.8 GB result array)
                torch.cuda.synchronize()
                t = time.perf_counter()
                keep[label] = tm.map(Xm)
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t)
            fwd[label + '_e2e_s'] = min(ts)
        os.environ.pop('TTM_MAP_GEMM', None)
        tm._inv_pack_cache.pop('map_gemm', None)
        fwd['points_per_s_e2e'] = nm / fwd['gemm_e2e_s']
        fwd['max_rel_diff_gemm_vs_per_component'] = float(np.max(np.abs(keep['gemm'] - keep['per_component'])) /
                                                          np.max(np.abs(keep['per_component'])))
        del keep, Xm
    cpu = None
    parity = None
    if with_cpu and rank == 0 and world == 1:
        cpu, parity = inverse_cpu_port(tm, mon, non, Dm, E)
    coef_check = None
    if world > 1:
        coef_check = coefficients_identical_across_ranks(tm, dist, torch)
    out = {'metric': 'inverse_map samples/sec', 'value': res['table']['samples_per_s'], 'unit': 'samples/s',
            'config': {'workload': 'C5: D=256 separable map, conditional sampling with E=128, %d samples per GPU, '
                                   'default table root finder (alternate_root_finding=True); steady state (second full-size call)' % ns,
                       'n_train': ntrain},
            'bisection': res['bisection'], 'table': res['table'], 'table_pageable': res['table_pageable'],
            'inputs': 'pinned host arrays (value, table); pageable host arrays (table_pageable, bisection)',
            'ctor_s': ctor_s, 'optimize_s': opt_s,
            'scaling': 'weak', 'e2e': True}
    if dev is not None:
        out['device'] = dev
    if fwd is not None:
        out['forward_map'] = fwd
    if cpu is not None:
        out['cpu_baseline'] = cpu
        out['parity_max_abs'] = parity
    if coef_check is not None:
        out['coefficients_identical_across_ranks'] = coef_check
    return out


def coefficients_identical_across_ranks(tm, dist, torch):
    """After optimize() every rank must hold bit-identical coefficient lists (one all-gather of the fitted shards)."""
    import hashlib
    h = hashlib.sha256()
    for k in range(tm.D):
        h.update(np.ascontiguousarray(tm.coeffs_nonmon[k], dtype=np.float64).tobytes())
        h.update(np.ascontiguousarray(tm.coeffs_mon[k], dtype=np.float64).tobytes())
    mine = torch.tensor(list(h.digest()), dtype=torch.uint8, device='cuda')
    allh = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
    dist.all_gather(allh, mine)
    return bool(all(torch.equal(allh[0], x) for x in allh))


def inverse_cpu_port(tm, mon, non, Dm, E, ntrain=2000, n_table=2000):
    """CPU leg of M2: the oracle's inverse_map (tm.py:3639-4084 restated) of the same C5 map on a bounded sample.
    The oracle materialises every Psi of the training set like the reference (7.8 GB at 10^4 samples), so it is
    built on the first `ntrain` training samples and given the coefficients fitted on the GPU; its cost per
    conditional sample does not depend on the training set."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    from ttm_oracle import OracleMap
    os.environ.setdefault('OPENBLAS_NUM_THREADS', str(os.cpu_count()))
    om = OracleMap(X=synthetic_samples(ntrain, Dm, seed=0), monotone=mon, nonmonotone=non,
                   monotonicity='separable monotonicity')
    for k in range(Dm):
        om.coeffs_nonmon[k] = np.array(tm.coeffs_nonmon[k], dtype=np.float64)
        om.coeffs_mon[k] = np.array(tm.coeffs_mon[k], dtype=np.float64)
    rng = np.random.default_rng(300)
    Xstar = synthetic_samples(n_table, Dm, seed=301)[:, :E].copy()
    Z = rng.standard_normal((n_table, Dm - E))
    om.alternate_root_finding = True         # the default root finder (the oracle's bisection arm has ~60 s of fixed
    t = time.perf_counter()                  # cost per call at D=256 and is left to the parity tests)
    Xo = om.inverse_map(Z, X_star=Xstar)
    v = n_table / (time.perf_counter() - t)
    # parity leg: a GPU map built on the SAME training subset as the oracle (same standardisation and special-term
    # placement), same coefficients, same inputs
    from transport_map import transport_map
    tg = transport_map(X=synthetic_samples(ntrain, Dm, seed=0), monotone=mon, nonmonotone=non,
                       monotonicity='separable monotonicity', verbose=False)
    for k in range(Dm):
        tg.coeffs_nonmon[k] = np.array(tm.coeffs_nonmon[k], dtype=np.float64)
        tg.coeffs_mon[k] = np.array(tm.coeffs_mon[k], dtype=np.float64)
    Xg = tg.inverse_map(Z.copy(), X_star=Xstar.copy())
    del tg
    parity = float(np.max(np.abs(Xg - Xo)))
    return ({'value': v, 'unit': 'samples/s', 'cores': 1, 'kind': 'port',
             'sample': 'oracle inverse_map of the same C5 map (coefficients from the GPU fit, oracle built on %d training '
                       'samples): %d conditional samples, table root finder, single process' % (ntrain, n_table)}, parity)


# ------------------------------------------------------------------------------------------------
# the other BASELINE configurations (SURVEY.md 8(d)): C1 Example 01, C2 Example 05 densities at 1M points,
# C3 Example 06 EnTF cycle -- small-N / latency figures with their own parity checks, rank 0 only
# ------------------------------------------------------------------------------------------------
def extras(torch, with_cpu=True):
    from cases import ex01_terms, ex05_terms, ex06_terms, ex06_cycle_inputs
    from transport_map import transport_map
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    out = {}

    def wall(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t)
        return float(np.median(ts)), r

    # ---- C1: Example 01 (spiral, N = 1e4, order-10 map, Q = 25) with the coefficients shipped with the reference
    try:
        g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ex01_known_answer.npz'))
        mon, non = ex01_terms(10)
        tm = transport_map(X=g['X'].copy(), monotone=mon, nonmonotone=non, monotonicity='integrated rectifier',
                           quadrature_input={'order': 25}, verbose=False)
        rec = {'N': int(g['X'].shape[0])}
        for k in range(2):
            c, div = g['full_coeffs_%d' % k], int(g['full_div_%d' % k])
            state = {'i': 0}

            def ev():
                state['i'] += 1
                cc = c + 1e-9 * state['i']                     # a new point every call: nothing memoised
                return tm.objective_function(cc, k, div), tm.objective_function_jacobian(cc, k, div)
            t, _ = wall(ev, reps=9)
            J = tm.objective_function(c, k, div)
            rec['eval_ms_k%d' % k] = t * 1e3
            rec['J_%d' % k] = J
            rec['J_%d_abs_err_vs_reference' % k] = abs(J - float(g['full_J_%d' % k]))
            rec['grad_%d_max_abs_err_vs_reference' % k] = float(np.max(np.abs(
                tm.objective_function_jacobian(c, k, div) - g['full_grad_%d' % k])))
        out['C1_example01'] = rec
        del tm
    except Exception as e:                                      # noqa: BLE001
        out['C1_example01'] = {'error': repr(e)}

    # ---- C2: Example 05 map trained on 1e3 samples, densities on 1e6 points (K-pullback / K-logdet)
    mon, non = ex05_terms()
    X5 = synthetic_samples(1000, 2, seed=5) * np.array([2.0, 0.5]) + np.array([1.0, -3.0])
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity', verbose=False)
    tm = transport_map(X=X5.copy(), **kw)
    tm.optimize()
    n = 1_000_000
    pts = np.random.default_rng(0).uniform(-3, 3, (n, 2)) * np.array([2.0, 0.5]) + np.array([1.0, -3.0])
    logg = lambda x: -0.5 * np.sum(x ** 2, axis=1) - np.log(2 * np.pi)
    t_pull, dens = wall(lambda: tm.evaluate_pullback_density(pts), reps=3)
    Zr = np.random.default_rng(1).standard_normal((n, 2))
    t_push, dpush = wall(lambda: tm.evaluate_pushforward_density(Zr, logg), reps=3)
    # device time of the fused kernel alone (inputs resident)
    Xd = tm._upload(pts)
    outd = tm._empty(n)
    from ttt_b200 import binding as B
    plans = (B.c_void_p * tm.D)(*[h.value for h in tm._plans])
    sg = np.ascontiguousarray([float(tm.X_std[k]) for k in range(tm.D)])
    ts = []
    for rep in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        B.check(tm._lib.ttm_map_fused(tm._ctx, plans, tm.D, B.dptr(sg), B.c_void_p(Xd.data_ptr()), n, 2,
                                      B.c_void_p(tm._mean_d.data_ptr()), B.c_void_p(tm._std_d.data_ptr()), None, 0, None,
                                      B.c_void_p(outd.data_ptr()), tm._stream()))
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    t_dev = float(np.median(ts[1:]))
    alg = 8 * n * (2 + 1)
    hbm = 6534.1
    try:
        hbm = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs']
    except Exception:
        pass
    rec = {'points': n, 'pullback_e2e_s': t_pull, 'pullback_points_per_s_e2e': n / t_pull,
           'pushforward_e2e_s': t_push, 'pushforward_points_per_s_e2e': n / t_push,
           'pullback_device_s': t_dev,
           'roofline': {'bound': 'hbm', 'achieved': alg / t_dev / 1e9, 'peak': hbm, 'unit': 'GB/s',
                        'frac': alg / t_dev / 1e9 / hbm, 'algorithmic_bytes': alg,
                        'how': 'K-pullback (ttm_map_fused, mode 0): 8 n (Dtot + 1) bytes / CUDA-event time, inputs resident'}}
    if with_cpu:
        from ttm_oracle import OracleMap
        om = OracleMap(X=X5.copy(), **{k: v for k, v in kw.items() if k != 'verbose'})
        for k in range(2):
            om.coeffs_mon[k], om.coeffs_nonmon[k] = tm.coeffs_mon[k].copy(), tm.coeffs_nonmon[k].copy()
        t = time.perf_counter()
        do = om.evaluate_pullback_density(pts[:10000].copy())
        rec['cpu_oracle_pullback_points_per_s'] = 10000 / (time.perf_counter() - t)
        rec['pullback_max_rel_err_vs_oracle'] = float(np.max(np.abs(dens[:10000] - do) / np.maximum(1e-300, np.abs(do))))
        dpo = om.evaluate_pushforward_density(Zr[:2000].copy(), logg)
        rec['pushforward_max_rel_err_vs_oracle'] = float(np.max(np.abs(dpush[:2000] - dpo) / np.maximum(1e-300, np.abs(dpo))))
    out['C2_example05_densities'] = rec
    del tm, Xd, outd

    # ---- C3: one EnTF cycle of Example 06 (reset -> optimize -> map -> inverse_map), separable + L2
    mon, non = ex06_terms(3)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='separable monotonicity', regularization='l2',
              regularization_lambda=0.05, verbose=False)
    cyc_out = []
    for N in (500, 1000, 10000):
        dummy, cyc = ex06_cycle_inputs(N)
        tm = transport_map(X=dummy.copy(), **kw)

        def cycle(m):
            m.reset(cyc.copy())
            m.optimize()
            Z = m.map(cyc.copy())
            return m.inverse_map(X_star=np.full((N, 1), 1.5), Z=Z)
        t, post = wall(lambda: cycle(tm), reps=7)
        rec = {'N': N, 'gpu_cycle_ms': t * 1e3, 'posterior_mean': post.mean(axis=0).tolist()}
        if with_cpu:
            from ttm_oracle import OracleMap
            om = OracleMap(X=dummy.copy(), **{k: v for k, v in kw.items() if k != 'verbose'})
            cycle(om)
            t0 = time.perf_counter()
            po = cycle(om)
            rec['cpu_oracle_cycle_ms'] = (time.perf_counter() - t0) * 1e3
            rec['max_abs_diff_vs_oracle'] = float(np.max(np.abs(po - post)))
        cyc_out.append(rec)
        del tm
    out['C3_example06_entf_cycle'] = cyc_out
    return out


def step_outputs(tm, ks, coefs, world, dist, torch):
    """What the last launch of each component returned, as objective_function / objective_function_jacobian hand it to
    their caller: J_k of all components ('objective', shape (64,)) and grad J_k concatenated in component order, each in
    the coefficient layout [nonmonotone | monotone] ('gradient').  Every rank reads its own components; one all-reduce
    of the zero-padded vectors assembles the whole map."""
    from ttt_b200 import binding as B
    off = np.concatenate(([0], np.cumsum([len(c) for c in coefs])))
    J, grad = np.zeros(len(coefs)), np.zeros(int(off[-1]))
    for k in ks:
        out = np.empty(1 + len(coefs[k]))
        B.check(tm._lib.ttm_plan_get_out(tm._plans[k], B.dptr(out), out.size, tm._stream()))
        G = tm._gram_nonmon(k)
        if G is not None:                      # Gram mode: the kernel returned h, dJ/da = G a + h
            m = G.shape[0]
            out[1:1 + m] += G @ coefs[k][:m]
        J[k], grad[off[k]:off[k + 1]] = out[0], out[1:]
    if world > 1:
        both = torch.from_numpy(np.concatenate((J, grad))).cuda()
        dist.all_reduce(both)
        both = both.cpu().numpy()
        J, grad = both[:len(J)], both[len(J):]
    return {'objective': J, 'gradient': grad}


def multi_gpu_check(rank, world, dist, torch):
    """Sample-sharded evaluation (the K < #GPUs path of SURVEY 8(e): every rank holds N/world rows, (J, grad) are
    all-reduced) against the same evaluation on the whole ensemble held by one rank (the component-sharded layout)."""
    from transport_map import transport_map
    Dm, n = 8, 64 * 1024
    X = synthetic_samples(n, Dm, seed=5)
    mon, non = c4_terms(Dm)
    kw = dict(monotone=mon, nonmonotone=non, monotonicity='integrated rectifier', quadrature_input={'order': 25},
              verbose=False)
    full = transport_map(X=X.copy(), **kw)
    lo, hi = n * rank // world, n * (rank + 1) // world
    shard = transport_map(X=X[lo:hi].copy(), sample_sharded=True, **kw)
    rng = np.random.default_rng(9)
    worst = 0.0
    for k in (0, 3, 7):
        c = rng.standard_normal(len(non[k]) + len(mon[k])) * 0.1
        div = len(non[k])
        f0, g0 = full.objective_function(c, k, div), full.objective_function_jacobian(c, k, div)
        f1, g1 = shard.objective_function(c, k, div), shard.objective_function_jacobian(c, k, div)
        worst = max(worst, abs(f0 - f1) / max(1.0, abs(f0)), float(np.max(np.abs(g0 - g1) / np.maximum(1.0, np.abs(g0)))))
    w = torch.tensor([worst], dtype=torch.float64, device='cuda')
    dist.all_reduce(w, op=dist.ReduceOp.MAX)
    return {'sample_sharded_vs_whole_max_rel': float(w[0]), 'ranks': world, 'rows_per_rank': hi - lo}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_gpu(args):
    # native libraries (NCCL's version banner, ...) write to fd 1: keep stdout for the ONE JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from transport_map import transport_map
    from ttt_b200 import binding as B
    from ttt_b200.parallel import shard_components

    n = args.n
    X = synthetic_samples(n, D, seed=0)
    mon, non = c4_terms(D)
    tm = transport_map(X=X, monotone=mon, nonmonotone=non, polynomial_type='hermite function',
                       monotonicity='integrated rectifier', quadrature_input={'order': Q}, verbose=False)
    del X
    coefs = coefficients(mon, non)
    mine = shard_components(list(range(D)), rank, world)
    lib, stream = tm._lib, tm._stream()
    Xp, ld = B.c_void_p(tm._Xt.data_ptr()), tm._Xt.shape[1]
    # Gram matrix G = Psi_non^T Psi_non / N of the ensemble (K-gram, ONE launch for the map: every component's G is a
    # leading block of the last component's): once per ensemble like the reference's precalculate(); with it an
    # evaluation sweeps the columns x_<c once (dJ/da = G a + h).  Timed separately, not part of the evaluations.
    torch.cuda.synchronize()
    t_g = time.perf_counter()
    for k in mine:
        tm._gram_nonmon(k)
    torch.cuda.synchronize()
    gram_setup_s = time.perf_counter() - t_g
    for k in mine:
        tm._set_coeffs(k, coefs[k][:len(non[k])], coefs[k][len(non[k]):])
    flush = torch.empty(512 * 1024 * 1024 // 8, dtype=torch.float64, device='cuda')   # 512 MB > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    NSTREAMS = args.streams
    streams = [torch.cuda.Stream() for _ in range(NSTREAMS)]
    sptr = [B.c_void_p(st_.cuda_stream) for st_ in streams]

    def step_concurrent():
        """The step's independent evaluations are issued round-robin on two streams with 2 resident blocks per SM
        per launch, so blocks of two components share every SM and their phases overlap."""
        for i, k in enumerate(mine):
            B.check(lib.ttm_objgrad_ir_launch(tm._plans[k], Xp, ld, n, sptr[i % NSTREAMS]))

    def fork(e):
        for st_ in streams:
            st_.wait_event(e)

    def join():
        for st_ in streams:
            ej = torch.cuda.Event()
            ej.record(st_)
            torch.cuda.current_stream().wait_event(ej)

    sampler = ClockSampler(local)
    sampler.start()
    # ---- per-launch durations (roofline per k): one sequential pass, default grid, NOT part of `value`
    per_k = {k: [] for k in mine}
    for rep in range(3):
        for k in mine:
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            B.check(lib.ttm_objgrad_ir_launch(tm._plans[k], Xp, ld, n, stream))
            eb.record()
            torch.cuda.synchronize()
            if rep > 0:
                per_k[k].append(ea.elapsed_time(eb) * 1e-3)
    # ---- value: inputs resident in HBM, device time only
    B.check(lib.ttm_ctx_set_blocks_per_sm(tm._ctx, args.bps))
    for _ in range(args.warmup):
        e0 = torch.cuda.Event()
        e0.record()
        fork(e0)
        step_concurrent()
        join()
    barrier()
    sampler.active = True
    sampler.t_on = time.perf_counter()
    t_steps = []
    wall0 = time.perf_counter()
    for s in range(args.steps):
        flush.fill_(float(s))                       # L2 flush between timed iterations (outside the event pair)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fork(e0)
        step_concurrent()
        join()
        e1.record()
        torch.cuda.synchronize()
        t_steps.append(e0.elapsed_time(e1) * 1e-3)
    barrier()
    wall_value = time.perf_counter() - wall0
    t_local = float(sum(t_steps))
    # read before the e2e leg below reuses the plans
    outputs = step_outputs(tm, mine, coefs, world, dist, torch) if args.dump_outputs else None

    # ---- e2e: through the public class API with host coefficient vectors in, host (J, grad) out
    rng = np.random.default_rng(1)

    import concurrent.futures
    import threading
    tls = threading.local()
    pool = concurrent.futures.ThreadPoolExecutor(max_workers=NSTREAMS)

    def eval_one(args_):
        k, s = args_
        if not hasattr(tls, 'stream'):
            # a new host thread starts on device 0: without this, the workers of every rank but 0 created their stream
            # there and all their launches fell back to the default stream of the rank's own GPU (serialised: the e2e
            # figure of N >= 2 ranks read 13 % low)
            torch.cuda.set_device(local)
            tls.stream = torch.cuda.Stream(device=local)
        with torch.cuda.stream(tls.stream):
            c = coefs[k] + 1e-6 * (s + 1)           # new point every step: no memoised result is reused
            div = len(non[k])
            f = tm.objective_function(c, k, div)
            g = tm.objective_function_jacobian(c, k, div)
        return f + g[0]

    def run_e2e(steps):
        """Public class API from two host threads (what optimize() does): host coefficients in, host (J, grad) out.
        The evaluations of all steps form one queue (no barrier between steps: the 64 evaluations are independent and
        so are the steps); every evaluation is a complete host -> device -> host round trip."""
        return sum(pool.map(eval_one, [(k, s) for s in steps for k in mine]))

    run_e2e([-s - 1 for s in range(args.warmup)])
    barrier()
    w0 = time.perf_counter()
    run_e2e(list(range(args.steps)))
    torch.cuda.synchronize()
    t_e2e_local = time.perf_counter() - w0
    pool.shutdown()
    B.check(lib.ttm_ctx_set_blocks_per_sm(tm._ctx, 0))
    barrier()
    sampler.active = False
    sampler.t_off = time.perf_counter()

    fp64_peak_tflops = tm.fp64_peak_tflops() if rank == 0 else 0.0

    # ---- end-to-end fit of the north-star map: optimize() of all 64 components at N = 1M, Q = 100 (components sharded
    # over the ranks, one all-gather of the coefficients), wall clock, max over ranks
    fit = None
    if not args.no_fit:
        barrier()
        t_f = time.perf_counter()
        tm.optimize()
        torch.cuda.synchronize()
        t_fit_local = time.perf_counter() - t_f
        gmax = 0.0
        for k in mine[:2] + mine[-1:]:
            c = np.concatenate((tm.coeffs_nonmon[k], tm.coeffs_mon[k]))
            gmax = max(gmax, float(np.max(np.abs(tm.objective_function_jacobian(c, k, len(tm.coeffs_nonmon[k]))))))
        tf = torch.tensor([t_fit_local, gmax], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(tf, op=dist.ReduceOp.MAX)
        fit = {'optimize_wall_s': float(tf[0]), 'max_abs_gradient_at_solution': float(tf[1]),
               'fit_s_rank0': tm._last_timing['fit_s'], 'gather_s_rank0': tm._last_timing['gather_s'],
               'components_rank0': tm._last_timing['components'], 'gram_setup_s': gram_setup_s,
               'fit_threads': tm.fit_threads,
               'evaluations_rank0': int(sum(tm._fit_info[k]['nfev'] for k in mine)),
               'slowest_component_rank0': max(({'k': k, **tm._fit_info[k]} for k in mine), key=lambda r: r['seconds'])}
        if world > 1:
            fit['coefficients_identical_across_ranks'] = coefficients_identical_across_ranks(tm, dist, torch)
    sampler.stop()
    multi = multi_gpu_check(rank, world, dist, torch) if world > 1 else None

    tt = torch.tensor([t_local, t_e2e_local], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_max, t_e2e = float(tt[0]), float(tt[1])

    inv = None
    if not args.no_inverse:
        del tm, flush
        torch.cuda.empty_cache()
        inv = inverse_metric(rank, world, dist, torch, with_cpu=not args.no_cpu)
    ext = None
    if not args.no_extras and rank == 0 and world == 1:
        try:
            ext = extras(torch, with_cpu=not args.no_cpu)
        except Exception as e:                                  # noqa: BLE001  (extras never take the headline down)
            ext = {'error': repr(e)}

    if rank == 0:
        value = D * args.steps / t_max
        e2e_value = D * args.steps / t_e2e
        # dominant kernel = the fused objgrad kernel (every launch of the timed region is one)
        kt = {k: float(np.mean(v)) for k, v in per_k.items()}
        fl = sum(flops_per_eval(k, n) for k in mine)
        by = sum(bytes_per_eval(k, n) for k in mine)
        t_kernels = t_local / args.steps            # the step is 64 launches of this one kernel (2 streams)
        t_seq = sum(kt.values())
        # FP64 peak: the tracked measurement of tools/pipe_probe.cu on this pool (profiles/fp64_peaks_r2.json, written
        # once with its clock record); the live probe of this run is reported beside it
        peaks_fp64 = {}
        try:
            peaks_fp64 = json.load(open(os.path.join(ROOT, 'profiles', 'fp64_peaks_r2.json')))
        except Exception:
            pass
        fp64_peak = float(peaks_fp64.get('dfma_tflops', fp64_peak_tflops))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        hbm_peak = peaks.get('hbm_gbs', 6650.0)
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic_r2.json')))
        except Exception:
            pass
        fl18 = sum(flops_per_eval(k, n, c_exp=14) for k in mine)
        flx = sum(flops_executed(k, n) for k in mine)
        achieved = fl / t_kernels / 1e12
        per_launch_traffic = traffic.get('per_launch_avg_bytes') if (n == N_FULL and world == 1) else None
        roofline = {
            'bound': 'fp64', 'achieved': achieved, 'peak': fp64_peak, 'unit': 'TFLOP/s', 'frac': achieved / fp64_peak,
            'traffic': per_launch_traffic,
            'traffic_source': traffic.get('source'),
            'peak_source': 'profiles/fp64_peaks_r2.json: tools/pipe_probe.cu dependent-free DFMA chains, %s MHz '
                           '(MEASURED_PEAKS.json has no FP64 figure); DMMA peak %s TFLOP/s' % (
                               peaks_fp64.get('clock_rate_mhz'), peaks_fp64.get('dmma_m8n8k4_tflops')),
            'peak_live_probe': fp64_peak_tflops,
            # the same time against two other flop counts (DESIGN.md section 4): the survey formula re-frozen for the
            # shipped exp (c_exp = 14 instead of the library's 30), and the flops the shipped SASS executes
            'achieved_refrozen': fl18 / t_kernels / 1e12, 'frac_refrozen': fl18 / t_kernels / 1e12 / fp64_peak,
            'achieved_executed': flx / t_kernels / 1e12, 'frac_executed': flx / t_kernels / 1e12 / fp64_peak,
            'ncu_pipe_fp64_active_pct': traffic.get('pipe_fp64_active_pct'),
            'flops_per_launch_avg': fl / len(mine), 'bytes_per_launch_avg': by / len(mine),
            'launch_ms_avg': t_kernels / len(mine) * 1e3,
            'launch_ms_avg_sequential': t_seq / len(mine) * 1e3,
            'how': 'achieved = algorithmic flops of the step (SURVEY 8(d), frozen c_exp = 30) / CUDA-event step time '
                   '(launches overlap on %d streams); per_k = isolated sequential launches with the default grid' % NSTREAMS,
            'hbm': {'achieved_gbs': by / t_kernels / 1e9, 'peak_gbs': hbm_peak, 'frac': by / t_kernels / 1e9 / hbm_peak,
                    'peak_source': 'MEASURED_PEAKS.json' if 'hbm_gbs' in peaks else 'fallback'},
            'per_k': {str(k): {'ms': kt[k] * 1e3, 'tflops': flops_per_eval(k, n) / kt[k] / 1e12,
                               'frac': flops_per_eval(k, n) / kt[k] / 1e12 / fp64_peak,
                               'tflops_refrozen': flops_per_eval(k, n, c_exp=14) / kt[k] / 1e12,
                               'tflops_executed': flops_executed(k, n) / kt[k] / 1e12,
                               'evals_per_s': 1.0 / kt[k]} for k in (0, 31, 63) if k in kt},
        }
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': t_max / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': 'C4: synthetic D=64 integrated-rectifier map, order-3 Hermite functions, Q=%d, N=%d' % (Q, n),
                       'components': D, 'samples': n, 'quadrature_order': Q, 'parallelism': 'components sharded over %d GPU(s)' % world,
                       'l2': 'flushed between timed steps (512 MB write); the sample matrix itself is %d MB' % (8 * n * D >> 20),
                       'issue': '64 independent evaluations per step on %d CUDA stream(s), %d resident block(s) per SM per launch; '
                                'Gram matrix of the ensemble precomputed once (%.3f s, not in the timed region)' % (
                                    NSTREAMS, args.bps, gram_setup_s)},
            'e2e': {'value': e2e_value, 'unit': UNIT,
                    'h2d_bytes_per_step': int(sum(8 * len(coefs[k]) for k in range(D))),
                    'd2h_bytes_per_step': int(sum(8 * (1 + len(coefs[k])) for k in range(D))),
                    'api': 'transport_map.objective_function + objective_function_jacobian per component (host numpy in/out), '
                           'called from %d host threads like optimize()' % NSTREAMS},
            'gpu_launches': D * args.steps,
            'roofline': roofline,
            'clocks': sampler.summary(),
            'wall_s_value_region': wall_value,
        }
        if fit is not None:
            line['fit'] = fit
            line['optimize_wall_s'] = fit['optimize_wall_s']
        if multi is not None:
            line['multi_gpu_check'] = multi
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            ks = [0, 31, 63]
            n_cpu = 20000
            v, per = cpu_port(n_cpu, ks, 1)
            # parity leg: the GPU map on the same rows and coefficients against the oracle values just computed
            tg = transport_map(X=synthetic_samples(n_cpu, D, seed=0), monotone=mon, nonmonotone=non,
                               polynomial_type='hermite function', monotonicity='integrated rectifier',
                               quadrature_input={'order': Q}, verbose=False)
            worst = 0.0
            for k in ks:
                fo, go = _CPU_VALUES[k]
                fg = tg.objective_function(coefs[k], k, len(non[k]))
                gg = tg.objective_function_jacobian(coefs[k], k, len(non[k]))
                worst = max(worst, abs(fg - fo) / max(1.0, abs(fo)), float(np.max(np.abs(gg - go) / np.maximum(1.0, np.abs(go)))))
            del tg
            line['parity'] = {'objgrad_max_rel': worst,
                              'objgrad_sample': 'J and grad J of k=0,31,63 on the CPU leg\'s %d rows, GPU (tile kernel, Gram mode) vs oracle' % n_cpu}
            line['cpu_baseline'] = {
                'value': v, 'unit': UNIT, 'cores': 1, 'kind': 'port',
                'sample': 'components k=0,31,63 of the same C4 map on %d samples (single process, BLAS threads = %s), '
                          'evals/s scaled linearly to N=1M; host has %d cores' % (n_cpu, os.environ.get('OPENBLAS_NUM_THREADS'), cores)}
        if ext is not None:
            line['other_configs'] = ext
        if inv is not None:
            line['inverse_map'] = inv
            if 'parity_max_abs' in inv:
                line.setdefault('parity', {})['inverse_max_abs'] = inv['parity_max_abs']
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--n', type=int, default=N_FULL, help='samples (default: the metric point, 1M)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-inverse', action='store_true', help='skip the secondary inverse_map metric (config C5)')
    ap.add_argument('--no-extras', action='store_true', help='skip the C1/C2/C3 small-configuration figures')
    ap.add_argument('--no-fit', action='store_true', help='skip the end-to-end optimize() of the C4 map')
    ap.add_argument('--streams', type=int, default=2, help='CUDA streams the evaluations of a step are issued on')
    ap.add_argument('--bps', type=int, default=2, help='resident blocks per SM of one launch (x streams = blocks per SM)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed to DIR as float64 .npy files: '
                         'objective.npy (J_k, k = 0..63) and gradient.npy (grad J_k in component order)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU run')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
