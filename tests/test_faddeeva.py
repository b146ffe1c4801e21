"""The in-kernel Faddeeva algorithm (Weideman N=36, csrc/beamfields.cuh::wofz_multi_q1), restated
in NumPy from the generated coefficient table, against scipy.special.wofz -- the function
the reference calls (xline/mathlibs.py:11-13).  scipy's wofz is itself off by up to 2.3e-14 of |w|
near the real axis, so the bounds here measure the difference of the two float64 evaluations;
the series alone is within 1e-14 of |w| of a 34-digit w (tests/test_beamfield_reference.py)."""
import os
import re

import numpy as np
from scipy.special import wofz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _table():
    txt = open(os.path.join(ROOT, "xline_b200", "csrc", "faddeeva_coeffs.inc")).read()
    L = float(re.search(r"XLB_WEID_L (\S+)", txt).group(1))
    body = txt.split("XLB_WEID_COEFFS")[1]
    coeffs = [float(t) for t in re.findall(r"[-+]?\d\.\d+e[-+]\d+|[-+]?\d+\.\d+", body)]
    return L, np.array(coeffs)


def weideman(z, synthetic_division=True):
    """The kernel's evaluation: p(Z) has real coefficients, so it is divided by the real quadratic
    X^2 - r X + s with the roots Z, conj(Z) (r = 2 Re Z, s = |Z|^2; two real FMAs per coefficient)
    and p(Z) = alpha Z + beta from the remainder.  synthetic_division=False: the complex Horner the
    first version of the kernel ran (four real FMAs per coefficient), kept as a cross-check."""
    L, a = _table()
    inv = 1.0 / (L - 1j * z)
    Z = (L + 1j * z) * inv
    if synthetic_division:
        r, s = 2 * Z.real, Z.real ** 2 + Z.imag ** 2
        b2 = np.zeros_like(r) + a[0]
        b1 = a[1] + r * b2
        for c in a[2:-1]:
            b2, b1 = b1, c + (r * b1 - s * b2)
        p = b1 * Z + (a[-1] - s * b2)
    else:
        p = np.zeros_like(Z) + a[0]
        for c in a[1:]:
            p = p * Z + c
    return 2 * p * inv * inv + inv / np.sqrt(np.pi)


def test_table_matches_generator():
    import importlib.util

    spec = importlib.util.spec_from_file_location("gen", os.path.join(ROOT, "scripts", "gen_faddeeva_coeffs.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    L, a = gen.coefficients()
    L2, a2 = _table()
    assert len(a2) == 36 and L == L2 and np.array_equal(a, a2)


def test_weideman_matches_wofz_in_first_quadrant():
    rng = np.random.default_rng(0)
    r = 10 ** rng.uniform(-8, 6, 200_000)
    th = rng.uniform(0, np.pi / 2, 200_000)
    z = np.concatenate([
        r * np.exp(1j * th),
        rng.uniform(0, 8, 100_000) + 1j * rng.uniform(0, 8, 100_000),
        rng.uniform(0, 30, 50_000) + 1j * 10 ** rng.uniform(-12, -1, 50_000),
        1j * 10 ** rng.uniform(-8, 3, 10_000), 10 ** rng.uniform(-8, 1.5, 10_000) + 0j,
        np.array([0j, 1e-300 + 1e-300j]),
    ])
    z = np.concatenate([z, 10 ** rng.uniform(-12, -2, 50_000) + 1j * rng.uniform(0, 4, 50_000),
                        10 ** rng.uniform(-12, -2, 50_000) + 1j * 10 ** rng.uniform(-12, -2, 50_000)])
    ref = wofz(z)
    for form in (True, False):  # the synthetic division is as accurate as the complex Horner
        err = np.abs(weideman(z, form) - ref) / np.abs(ref)
        assert err.max() < 5e-14, (form, err.max(), z[err.argmax()])


def test_accuracy_against_series_length():
    """Why N = 36: the difference from scipy's wofz falls by ~30x per four terms down to the
    floor of the two float64 evaluations (3.6e-14 of |w|, most of it scipy's: the series itself is
    within 7.6e-15 of a 34-digit w), reached at N = 36; longer series buy
    nothing, shorter ones are visibly worse."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("gen", os.path.join(ROOT, "scripts", "gen_faddeeva_coeffs.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    rng = np.random.default_rng(5)
    z = np.concatenate([rng.uniform(0, 8, 100_000) + 1j * rng.uniform(0, 8, 100_000),
                        10 ** rng.uniform(-8, 6, 100_000) * np.exp(1j * rng.uniform(0, np.pi / 2, 100_000))])
    ref = wofz(z)
    worst = {}
    for n in (28, 32, 36, 40, 44):
        L, a = gen.coefficients(n)
        inv = 1.0 / (L - 1j * z)
        Z = (L + 1j * z) * inv
        p = np.zeros_like(Z) + a[0]
        for c in a[1:]:
            p = p * Z + c
        worst[n] = (np.abs(2 * p * inv * inv + inv / np.sqrt(np.pi) - ref) / np.abs(ref)).max()
    assert worst[28] > 5e-12 and worst[32] > 1e-13
    assert worst[36] < 5e-14 and worst[40] < 5e-14 and worst[44] < 5e-14
    assert worst[36] < 1.5 * worst[44]
