"""bench.py --dump-outputs: what it writes after the timed steps is what objective_function /
objective_function_jacobian return for the benchmark's map, samples and coefficients (here at a small N)."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from cases import synthetic_samples, c4_terms
from harness import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_outputs_are_what_the_public_api_returns(tmp_path):
    import bench
    from transport_map import transport_map
    n = 8192
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--n', str(n), '--steps', '2', '--warmup', '1', '--no-cpu',
           '--no-inverse', '--no-extras', '--no-fit', '--dump-outputs', str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])['steps'] == 2
    J, grad = np.load(tmp_path / 'objective.npy'), np.load(tmp_path / 'gradient.npy')
    mon, non = c4_terms(bench.D)
    coefs = bench.coefficients(mon, non)
    off = np.cumsum([0] + [len(c) for c in coefs])
    assert J.dtype == grad.dtype == np.float64 and J.shape == (bench.D,) and grad.shape == (off[-1],)
    tm = transport_map(X=synthetic_samples(n, bench.D, seed=0), monotone=mon, nonmonotone=non,
                       polynomial_type='hermite function', monotonicity='integrated rectifier',
                       quadrature_input={'order': bench.Q}, verbose=False)
    for k in range(bench.D):
        div = len(non[k])
        assert rel_err(J[k], tm.objective_function(coefs[k], k, div)) <= 1e-12, k
        assert rel_err(grad[off[k]:off[k + 1]], tm.objective_function_jacobian(coefs[k], k, div)) <= 1e-12, k
