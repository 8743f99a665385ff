"""Coefficient persistence in the reference examples' pickle format (example_01.py:215-231) and the chronicle layout
(tm.py:4703-4711, :4943-4950).  Host logic only: runs without a GPU."""

import importlib.util
import os
import pickle

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
spec = importlib.util.spec_from_file_location(
    'ttt_persistence', os.path.join(HERE, '..', 'triangular-transport-toolbox_b200', 'persistence.py'))
P = importlib.util.module_from_spec(spec)
spec.loader.exec_module(P)

# the coefficients of the reference's Example 01 pickle (dict_coeffs_order=10.p), per component [nonmonotone | monotone]
EX01_KNOWN_ANSWER = os.path.join(HERE, 'golden', 'ex01_known_answer.npz')


class FakeMap:
    def __init__(self, sizes):
        rng = np.random.default_rng(0)
        self.D = len(sizes)
        self.coeffs_mon = [rng.standard_normal(m) for m, _ in sizes]
        self.coeffs_nonmon = [rng.standard_normal(n) for _, n in sizes]
        self.monotone = [[[k]] * m for k, (m, _) in enumerate(sizes)]
        self.nonmonotone = [[[]] * n for _, n in sizes]


def test_round_trip_in_the_examples_format(tmp_path):
    tm = FakeMap([(3, 1), (4, 7)])
    path = tmp_path / 'dict_coeffs.p'
    P.save_coefficients(tm, path)
    d = pickle.load(open(path, 'rb'))                       # what example_01.py:226 does
    assert sorted(d) == ['coeffs_mon', 'coeffs_nonmon']
    other = FakeMap([(3, 1), (4, 7)])
    for k in range(2):
        other.coeffs_mon[k] *= 0
    P.load_coefficients(other, path)
    for k in range(2):
        assert np.array_equal(other.coeffs_mon[k], tm.coeffs_mon[k])
        assert np.array_equal(other.coeffs_nonmon[k], tm.coeffs_nonmon[k])


def test_shape_mismatch_is_an_error(tmp_path):
    path = tmp_path / 'c.p'
    P.save_coefficients(FakeMap([(3, 1), (4, 7)]), path)
    with pytest.raises(ValueError):
        P.load_coefficients(FakeMap([(3, 1)]), path)
    with pytest.raises(ValueError):
        P.load_coefficients(FakeMap([(3, 1), (5, 7)]), path)


def test_reads_the_pickle_shipped_with_example_01(tmp_path):
    """Example 01's shipped coefficients, pickled the way example_01.py:215-224 writes them."""
    ka = np.load(EX01_KNOWN_ANSWER)
    d = {'coeffs_mon': [], 'coeffs_nonmon': []}
    for k in range(2):
        c, div = ka['full_coeffs_%d' % k], int(ka['full_div_%d' % k])
        d['coeffs_nonmon'].append(c[:div])
        d['coeffs_mon'].append(c[div:])
    path = tmp_path / 'dict_coeffs_order=10.p'
    with open(path, 'wb') as f:
        pickle.dump(d, f)
    tm = FakeMap([(len(m), len(n)) for m, n in zip(d['coeffs_mon'], d['coeffs_nonmon'])])
    P.load_coefficients(tm, path)
    assert tm.D == 2 and len(tm.coeffs_mon[1]) == 55 and len(tm.coeffs_nonmon[1]) == 11
    for k in range(2):
        assert np.array_equal(tm.coeffs_mon[k], d['coeffs_mon'][k])
        assert np.array_equal(tm.coeffs_nonmon[k], d['coeffs_nonmon'][k])


def test_chronicle_layout(tmp_path):
    tm = FakeMap([(3, 1), (4, 7)])
    c = P.Chronicle()
    c.record(tm, 1, nit=12, nfev=15)
    c.record(tm, 1, nit=3, nfev=4)
    c.record(tm, 0)
    assert sorted(c) == [0, 1] and sorted(c[1]) == [0, 1]
    assert set(c[1][0]) >= {'monotone', 'nonmonotone', 'coeffs_nonmon', 'coeffs_mon', 'nit'}
    path = tmp_path / 'dictionary_adaptation_chronicle.p'
    c.save(path)
    back = pickle.load(open(path, 'rb'))                    # a plain dict, like tm.py:4948-4950 writes
    assert type(back) is dict and back[1][1]['nit'] == 3
    assert np.array_equal(P.Chronicle.load(path)[0][0]['coeffs_mon'], tm.coeffs_mon[0])
