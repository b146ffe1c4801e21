"""Generates xline_b200/csrc/synrad_table.inc: the inverse CDF of the synchrotron photon-number
spectrum, which the radiation kernel samples photon energies from (include/xline_b200.h,
XLB_T_MULTIPOLE_RAD; DESIGN.md §4.9).

With x = u / u_c (photon energy over the critical energy) the number spectrum is

    dN/dx  ∝  S(x) = ∫ₓ^∞ K_{5/3}(t) dt,      ∫₀^∞ S(x) dx = 5π/3,

so F(x) = (3/(5π)) ∫₀ˣ S.  Integrating by parts, F(x) = (3/(5π)) [x S(x) + ∫₀ˣ t K_{5/3}(t) dt] and
1 - F(x) = (3/(5π)) ∫ₓ^∞ (t - x) K_{5/3}(t) dt: single integrals of scipy.special.kv / kve with no
cancellation, evaluated with scipy.integrate.quad in log t (small x) or on [x, ∞) scaled by e^x.

The table is x = F⁻¹(U) in two parts, each a polynomial of degree DEG per segment in the local
coordinate s ∈ [-1, 1] of the segment (Horner, highest power first):
  * U < U_SPLIT: w(U) = x^(1/3) on N_LO segments uniform in U.  Near 0, F ∝ x^(1/3) + O(x), so w is
    an analytic function of U there and x = w³ ∝ U³;
  * U >= U_SPLIT: x(t), t = -ln(1 - U), on N_HI segments of width DT from T0 = -ln(1 - U_SPLIT).
    In the tail x ≈ t.  The segments reach t = 38, past the largest t the kernel's uniforms take
    (U <= 1 - 2^-54, t <= 37.43).
Evaluation takes + - × and, in the upper part, one log: the GPU and NumPy agree to rounding.
The polynomials interpolate F⁻¹ at the DEG + 1 Chebyshev points of every segment; `check()`
reports the largest relative error in x on a dense grid and the moments <x> and <x²>.
"""
import math
import os
import sys

import numpy as np
from scipy.integrate import quad
from scipy.optimize import brentq
from scipy.special import kv, kve

U_SPLIT = 0.75
N_LO = 64
N_HI = 74
DEG = 9
T0 = -math.log(1.0 - U_SPLIT)
DT = (38.0 - T0) / N_HI
NORM = 3.0 / (5.0 * math.pi)
MEAN_X = 8.0 / (15.0 * math.sqrt(3.0))
MEAN_X2 = 11.0 / 27.0


def _S(x):
    """∫ₓ^∞ K_{5/3}."""
    if x < 1.0:
        v, _ = quad(lambda u: kv(5.0 / 3.0, math.exp(u)) * math.exp(u), math.log(x), math.log(1.0),
                    epsabs=0.0, epsrel=1e-13, limit=400)
        return v + _S(1.0)
    v, _ = quad(lambda s: kve(5.0 / 3.0, x + s) * math.exp(-s), 0.0, np.inf, epsabs=0.0, epsrel=1e-13, limit=400)
    return v * math.exp(-x)


def cdf(x):
    """F(x), for x small to moderate (no cancellation when F is not close to 1)."""
    lo = math.log(x)
    v, _ = quad(lambda u: kv(5.0 / 3.0, math.exp(u)) * math.exp(2.0 * u), lo - 140.0, lo,
                epsabs=0.0, epsrel=1e-13, limit=400)
    return NORM * (x * _S(x) + v)


def log_sf(x):
    """ln(1 - F(x)) = ln((3/(5π)) ∫ₓ^∞ (t - x) K_{5/3}(t) dt)."""
    v, _ = quad(lambda s: s * kve(5.0 / 3.0, x + s) * math.exp(-s), 0.0, np.inf, epsabs=0.0, epsrel=1e-13,
                limit=400)
    return math.log(NORM * v) - x


def inverse(U):
    """x with F(x) = U, by Newton's method (F' = (3/(5π)) S)."""
    if U < U_SPLIT:
        # on w = x^(1/3), where F is nearly linear: F ~ (27/10π) Γ(5/3) 2^(2/3) w near 0
        w0 = U / (NORM * 4.5 * math.gamma(5.0 / 3.0) * 2.0 ** (2.0 / 3.0))
        w = brentq(lambda v: cdf(v ** 3) - U, 0.5 * w0, max(1.5 * w0, 1e-300) if U < 1e-3 else 1.0,
                   xtol=1e-300, rtol=1e-15, maxiter=200)
        return w ** 3
    return inverse_t(-math.log1p(-U))


def inverse_t(t):
    """x with 1 - F(x) = e^-t, by Newton's method on ln(1 - F)."""
    x = max(t - 0.5 * math.log(max(t, 1.0)), 0.05)
    for _ in range(60):
        g = log_sf(x) + t
        dg = -NORM * _S(x) / math.exp(log_sf(x))
        dx = g / dg
        x -= dx
        if abs(dx) <= 1e-15 * abs(x):
            break
    return x


def _cheb_nodes(n):
    return np.cos(np.pi * (np.arange(n) + 0.5) / n)


def _fit(fun, n_seg, a, h):
    """Per segment [a + i h, a + (i+1) h]: coefficients (highest power first) of the polynomial in
    s ∈ [-1, 1] that interpolates fun at the Chebyshev points."""
    nodes = _cheb_nodes(DEG + 1)
    out = np.zeros((n_seg, DEG + 1))
    for i in range(n_seg):
        z = a + (i + 0.5 * (nodes + 1.0)) * h
        vals = np.array([fun(v) for v in z])
        out[i] = np.polyfit(nodes, vals, DEG)
    return out


def build():
    lo = _fit(lambda U: inverse(U) ** (1.0 / 3.0), N_LO, 0.0, U_SPLIT / N_LO)
    hi = _fit(inverse_t, N_HI, T0, DT)
    return lo, hi


def evaluate(U, lo, hi):
    """x = F⁻¹(U) from the table (NumPy form of the kernel's synrad_x)."""
    U = np.asarray(U, dtype=np.float64)
    x = np.empty_like(U)
    m = U < U_SPLIT
    s = U[m] * (N_LO / U_SPLIT)
    i = np.minimum(s.astype(np.int64), N_LO - 1)
    s = 2.0 * (s - i) - 1.0
    w = np.zeros_like(s)
    for k in range(DEG + 1):
        w = w * s + lo[i, k]
    x[m] = w * w * w
    t = -np.log(1.0 - U[~m])
    s = (t - T0) * (1.0 / DT)
    i = np.clip(s.astype(np.int64), 0, N_HI - 1)
    s = 2.0 * (s - i) - 1.0
    v = np.zeros_like(s)
    for k in range(DEG + 1):
        v = v * s + hi[i, k]
    x[~m] = v
    return x


def moments(lo, hi):
    """<x> and <x²> of the table: Gauss-Legendre per segment, in U below U_SPLIT, in t (dU = e^-t dt)
    above; the table's x is a polynomial per segment, so this is exact to rounding."""
    g, wg = np.polynomial.legendre.leggauss(40)
    m1 = m2 = 0.0
    h = U_SPLIT / N_LO
    for i in range(N_LO):
        U = (i + 0.5 * (g + 1.0)) * h
        x = evaluate(U, lo, hi)
        m1 += 0.5 * h * np.sum(wg * x)
        m2 += 0.5 * h * np.sum(wg * x * x)
    for i in range(N_HI):
        t = T0 + (i + 0.5 * (g + 1.0)) * DT
        s = np.full_like(t, 0.0) + g
        v = np.zeros_like(s)
        for k in range(DEG + 1):
            v = v * s + hi[i, k]
        wt = np.exp(-t) * 0.5 * DT * wg
        m1 += np.sum(wt * v)
        m2 += np.sum(wt * v * v)
    # U beyond t = 38: probability e^-38, x < 40
    return m1, m2


def parse_inc(path):
    """(lo, hi) arrays from the generated include file."""
    txt = open(path).read()
    vals = []
    for name in ("xlb_synrad_lo", "xlb_synrad_hi"):
        body = txt.split(name)[1].split("{", 1)[1].split("};", 1)[0]
        vals.append(np.array([float(v) for v in body.replace("{", " ").replace("}", " ").split(",") if v.strip()]))
    return vals[0].reshape(N_LO, DEG + 1), vals[1].reshape(N_HI, DEG + 1)


def check(lo, hi, n=400):
    """Largest relative error of the table against `inverse` on points between the interpolation
    nodes, over U in (1e-9, 1 - 1e-15]."""
    U = np.concatenate([np.geomspace(1e-9, 0.05, n // 4), np.linspace(0.05, U_SPLIT, n // 4, endpoint=False),
                        1.0 - np.geomspace(1.0 - U_SPLIT, 1e-15, n // 2)])
    ref = np.array([inverse(u) for u in U])
    return float(np.max(np.abs(evaluate(U, lo, hi) - ref) / ref))


INC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "xline_b200", "csrc", "synrad_table.inc")


def _rows(a):
    return ",\n".join("    {" + ", ".join(repr(float(v)) for v in row) + "}" for row in a)


if __name__ == "__main__":
    lo, hi = build()
    m1, m2 = moments(lo, hi)
    with open(INC, "w") as fh:
        fh.write("// generated by scripts/gen_synrad_table.py -- inverse CDF of the synchrotron photon-number\n")
        fh.write("// spectrum, x = u/u_c = F^-1(U); see the script for the layout.  <x> = %.15f, <x^2> = %.15f\n"
                 % (m1, m2))
        fh.write("#define XLB_SYNRAD_U_SPLIT %r\n" % U_SPLIT)
        fh.write("#define XLB_SYNRAD_N_LO %d\n" % N_LO)
        fh.write("#define XLB_SYNRAD_LO_SCALE %r\n" % (N_LO / U_SPLIT))
        fh.write("#define XLB_SYNRAD_N_HI %d\n" % N_HI)
        fh.write("#define XLB_SYNRAD_DEG %d\n" % DEG)
        fh.write("#define XLB_SYNRAD_T0 %r\n" % T0)
        fh.write("#define XLB_SYNRAD_INV_DT %r\n" % (1.0 / DT))
        fh.write("static __constant__ double xlb_synrad_lo[%d][%d] = {\n%s};\n" % (N_LO, DEG + 1, _rows(lo)))
        fh.write("static __constant__ double xlb_synrad_hi[%d][%d] = {\n%s};\n" % (N_HI, DEG + 1, _rows(hi)))
    print("wrote", os.path.normpath(INC))
    print("<x> = %.15f (exact %.15f), <x^2> = %.15f (exact %.15f)" % (m1, MEAN_X, m2, MEAN_X2))
    if "--check" in sys.argv:
        print("max relative error in x:", check(lo, hi))
