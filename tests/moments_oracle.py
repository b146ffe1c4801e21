"""Exact reference for the beam moments (``xline_b200.moments``, ``csrc/moments.cu``): the counting
rule, the 27 sums of a store in exact rational arithmetic, and the centring / emittance arithmetic
on the (hi, lo) pairs with ``fractions.Fraction``."""
import math
from fractions import Fraction

import numpy as np

COORDS = ("x", "px", "y", "py", "zeta", "delta")
PAIRS = tuple((u, None) for u in range(6)) + tuple((u, v) for u in range(6) for v in range(u, 6))
WORDS = 56
# AccurateDWPlusDW: relative error <= 3 u^2 / (1 - 4 u) per addition, u = 2^-53
DD_ADD_REL = Fraction(3, 2 ** 106) / (1 - Fraction(4, 2 ** 53))


def counted(cols, state):
    """(mask of the particles that count, number of alive particles with a non-finite coordinate)."""
    alive = np.asarray(state) == 1
    finite = np.ones(len(alive), dtype=bool)
    for k in COORDS:
        finite &= np.isfinite(np.asarray(cols[k], dtype=np.float64))
    return alive & finite, int((alive & ~finite).sum())


def _scaled_ints(values):
    """Exact integers ``m`` and one shift ``L`` with ``value == m / 2**L`` for every value."""
    ratios = [float(v).as_integer_ratio() for v in values]
    L = max((d.bit_length() - 1 for _, d in ratios), default=0)
    return [nu << (L - (d.bit_length() - 1)) for nu, d in ratios], L


def exact_store(cols, state):
    """``dict(n, n_nonfinite, sums, abs_sums)``: the 27 sums of a store and the sums of the
    absolute values of their terms, exact (``Fraction``)."""
    ok, n_bad = counted(cols, state)
    ints, shifts = [], []
    for k in COORDS:
        m, L = _scaled_ints(np.asarray(cols[k], dtype=np.float64)[ok])
        ints.append(m)
        shifts.append(L)
    sums, abs_sums = [], []
    for u, v in PAIRS:
        if v is None:
            s = sum(ints[u])
            a = sum(abs(t) for t in ints[u])
            den = 2 ** shifts[u]
        else:
            terms = [a * b for a, b in zip(ints[u], ints[v])]
            s = sum(terms)
            a = sum(abs(t) for t in terms)
            den = 2 ** (shifts[u] + shifts[v])
        sums.append(Fraction(s, den))
        abs_sums.append(Fraction(a, den))
    return dict(n=int(ok.sum()), n_nonfinite=n_bad, sums=sums, abs_sums=abs_sums)


def store_errors(words, exact):
    """``|hi + lo - exact| / Σ|terms|`` of every pair of a store (0 where Σ|terms| == 0), as
    Fractions; also checks the two counts."""
    words = [float(w) for w in words]
    assert words[0] == exact["n"] and words[1] == exact["n_nonfinite"], (words[:2], exact["n"], exact["n_nonfinite"])
    out = []
    for q in range(len(PAIRS)):
        got = Fraction(words[2 + 2 * q]) + Fraction(words[3 + 2 * q])
        err = abs(got - exact["sums"][q])
        a = exact["abs_sums"][q]
        out.append(err / a if a else (Fraction(0) if err == 0 else Fraction(10 ** 9)))
    return out


def bound(n):
    """The accuracy contract of a reduction over n slots: 3·2^-106 per level, ceil(log2 n) levels."""
    return DD_ADD_REL * max(1, math.ceil(math.log2(max(n, 1))))


def pair_values(words):
    """The 27 exact values hi + lo of a store."""
    return [Fraction(float(words[2 + 2 * q])) + Fraction(float(words[3 + 2 * q])) for q in range(len(PAIRS))]


def centred(words):
    """Exact mean [6] and covariance [6][6] (Fractions) from the pairs of a store:
    Σu / n and (Σu·v - Σu·Σv / n) / n."""
    n = Fraction(float(words[0]))
    s = pair_values(words)
    mean = [s[u] / n for u in range(6)]
    cov = [[None] * 6 for _ in range(6)]
    for q, (u, v) in enumerate(PAIRS):
        if v is None:
            continue
        c = (s[q] - s[u] * s[v] / n) / n
        cov[u][v] = cov[v][u] = c
    return mean, cov


def ulps(got, exact):
    """Distance of the float ``got`` from the exact value, in ulps of the exact value."""
    exact = Fraction(exact)
    if exact == 0:
        return 0.0 if got == 0 else math.inf
    ulp = math.ulp(float(exact))
    return float(abs(Fraction(float(got)) - exact) / Fraction(ulp))


def emittance_from_cov(c, k):
    """sqrt(det) of the 2 x 2 block (k, k + 1) of float covariances ``c``: the determinant exact,
    then the float square root of the determinant rounded once."""
    a, b, d = Fraction(float(c[k][k])), Fraction(float(c[k][k + 1])), Fraction(float(c[k + 1][k + 1]))
    return math.sqrt(float(a * d - b * b))
