"""The tile kernel's exp of a product (csrc/ttm_exp.cuh, exp_prod_v) restated in numpy and checked on the CPU: its error
bound for |a b| <= 40, and that the folded high words insert the binary exponent with one integer multiply-add,
reproducing tab64 * 2^n bit for bit."""
import os
import re

import numpy as np
import pytest

from test_exp_constants import CSRC, macros, table

MAGIC = 6755399441055744.0


def two_prod(a, b):
    """a * b = p + e exactly (Dekker), so that fma(a, b, c) can be restated without an FMA."""
    p = a * b
    split = 134217729.0
    ah = a * split; ah = ah - (ah - a); al = a - ah
    bh = b * split; bh = bh - (bh - b); bl = b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def product_coefficients(variant):
    """The rescaled coefficients PK_C1..PK_C(DEG) as ttm_exp.cuh defines them (constexpr products of the macros of the
    variant, evaluated left to right like C++), highest degree first."""
    m = macros(variant)
    text = open(os.path.join(CSRC, 'ttm_exp.cuh')).read()
    out = {}
    deg = 4 if variant == 64 else 5
    for i, expr in re.findall(r'constexpr double PK_C(\d) = ([^;]+);', text):
        if int(i) > deg:                        # PK_C5 exists for the degree-5 variant only
            continue
        v = 1.0
        for name in expr.split('*'):
            v = v * m[name.strip()[len('TTM_E32_'):]]
        out[int(i)] = v
    return [out[i] for i in range(deg, 0, -1)]


@pytest.mark.parametrize('variant', [64, 32])
def test_product_coefficients_are_the_polynomial_rescaled_by_powers_of_c(variant):
    m = macros(variant)
    C = m['C']
    q = [1.0, m['Q0'], m['Q1'], m['Q2']] + ([m['Q3']] if variant == 32 else [])
    want = [C ** i * q[i - 1] for i in range(len(q), 0, -1)]
    assert np.allclose(product_coefficients(variant), want, rtol=1e-15, atol=0)


def exp_prod(a, b, variant):
    """exp(a b) the way exp_prod_v computes it from bK = b K; returns the polynomial, the exponent word and u."""
    m = macros(variant)
    E = variant
    coef = product_coefficients(variant)
    bK = b * m['K']
    p, e = two_prod(a, bK)
    nf = np.round(p + e)                        # = fma(a, bK, MAGIC) - MAGIC (round to nearest even, like the add)
    u = (p - nf) + e                            # fma(a, bK, -nf): p - nf is exact
    q = np.full_like(u, coef[0])
    for cf in coef[1:]:
        q = q * u + cf
    q = q * u + 1.0
    c = nf.astype(np.int64) + 1021 * E          # low word of t (in range: no clamp)
    return q, c, u


@pytest.mark.parametrize('variant,bound', [(64, 1.5e-14), (32, 1e-14)])
def test_product_form_stays_within_the_stated_error(variant, bound):
    rng = np.random.default_rng(3)
    E = variant
    x = np.concatenate((np.linspace(-40.0, 40.0, 200001), rng.uniform(-1e-3, 1e-3, 20001)))
    b = np.exp(rng.uniform(np.log(0.05), np.log(20.0), x.size)) * rng.choice([-1.0, 1.0], x.size)
    a = x / b
    q, c, u = exp_prod(a, b, variant)
    assert np.max(np.abs(u)) <= 0.5 + 1e-9
    tab = table(E)
    got = q * np.ldexp(tab[c % E], c // E)      # table entries carry 2^-1021; c // E = n + 1021
    ref = np.exp(a.astype(np.longdouble) * b.astype(np.longdouble))
    err = float(np.max(np.abs((got.astype(np.longdouble) - ref) / ref)))
    assert err <= bound, err


def test_folded_table_reproduces_the_scaled_table_bit_for_bit():
    E = 64
    tab = table(E)
    bits = tab.view(np.uint64)
    lo = (bits & np.uint64(0xffffffff)).astype(np.uint32)
    hi = (bits >> np.uint64(32)).astype(np.uint32)
    folded = (hi.astype(np.int64) - (np.arange(E, dtype=np.int64) << 14)).astype(np.uint32)
    c = np.arange(0, 2044 * E + E, dtype=np.int64)            # every clamped exponent word (TOP = 2044 E + 63)
    j = c & (E - 1)
    whi = ((c * (1 << 14) + folded[j].astype(np.int64)) & 0xffffffff).astype(np.uint64)
    word = ((whi << np.uint64(32)) | lo[j].astype(np.uint64)).view(np.float64)
    expect = np.ldexp(tab[j], c // E)
    assert np.array_equal(word.view(np.uint64), expect.view(np.uint64))
    # scaling the table word before the product gives the product scaled after it (both normal: exact)
    rng = np.random.default_rng(5)
    p = rng.uniform(np.exp(-np.log(2) / 128), np.exp(np.log(2) / 128), c.size)
    after = np.ldexp(p * tab[j], c // E)
    assert np.array_equal((p * word).view(np.uint64), after.view(np.uint64))
