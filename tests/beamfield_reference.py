"""34-digit reference for the beam-field kicks (BeamBeam4D, SCCoasting, SCQGaussProfile,
SCInterpolatedProfile) and their derivatives, CPU only.

Each function evaluates the *reference's formula* (xline/be_beamfields/gaussian_fields.py,
spacecharge.py, qgauss.py, beambeam.py; restated in oracle/xline_oracle.py) in mpmath at
``mp.dps = 34`` on the exact float64 inputs: the same operation, not the physical field.  So the
round field keeps the reference's linearised branch for r^2 < 1e-20, and the round/elliptic,
Gaussian/q-Gaussian and interval choices are made in float64 exactly as the packer
(``lattice._gauss_field_block``) and the reference make them.

Every value comes with an error *scale*: the sum of the magnitudes of the terms the formula
adds, through which a relative perturbation of order eps of the inputs or of the intermediate
results propagates.  Errors of a float64 evaluation are judged against that scale, not against
the value itself, so that the formula's own cancellation (near the origin, in the small-axis
component near the big axis, in w'(z) = -2 z w(z) + 2i/sqrt(pi) far out) is not counted against
the evaluation.
"""
import math
from fractions import Fraction

import mpmath as M
import numpy as np
from scipy.constants import e as QE
from scipy.constants import epsilon_0

M.mp.dps = 34
mpf, mpc = M.mpf, M.mpc

A = 1 / (2 * M.pi * mpf(epsilon_0))  # 1/(2 pi eps0): the field of a unit line charge is A/r
SQRT_PI = M.sqrt(M.pi)
TWO_OVER_SQRT_PI = 2 / SQRT_PI
EPS = 2.0 ** -52


def wofz(z):
    """Faddeeva w(z) = exp(-z^2) erfc(-iz) (scipy.special.wofz, xline/mathlibs.py:11-13).  The
    phase of exp(-z^2) needs |z|^2 more digits of z^2 than the result has: the evaluation runs at
    2 log10|z| + 5 digits more than the working precision (on 50 points of the far field this
    takes the agreement with the integral representation from 24 to > 30 digits)."""
    z = mpc(z)
    extra = 5 + (2 * int(M.log10(abs(z))) if abs(z) > 1 else 0)
    with M.extradps(extra):
        w = M.exp(-z * z) * M.erfc(-1j * z)
    return +w


def dwofz(z, w=None):
    """w'(z) = -2 z w(z) + 2i/sqrt(pi)."""
    z = mpc(z)
    w = wofz(z) if w is None else w
    return -2 * z * w + 2j / SQRT_PI


# ----------------------------------------------------------------------------- fields
def _sgn(v):
    return -1 if v < 0 else 1  # -0.0 is not < 0: the reference keeps the first-quadrant sign


def field_ellip(x, y, sx, sy, jac=False):
    """gaussian_fields.py:29-99 for one point: (Ex, Ey, T) with T = |factBE| (|w(z1)| + e |w(z2)|);
    with ``jac`` also ((dEx/dx, dEx/dy, dEy/dx, dEy/dy), Tjac), Tjac the magnitudes of the terms
    of the derivative.  A = 1/(2 pi eps0) is part of every value."""
    if sx == sy:
        raise ZeroDivisionError("float division by zero")
    wide = sx > sy
    big, small = (mpf(sx), mpf(sy)) if wide else (mpf(sy), mpf(sx))
    u, v = (mpf(abs(x)), mpf(abs(y))) if wide else (mpf(abs(y)), mpf(abs(x)))
    S = M.sqrt(2 * (big * big - small * small))
    fact = A * SQRT_PI / S  # = 1/(2 eps0 sqrt(pi) S)
    z1 = mpc(u, v) / S
    z2 = mpc(small / big * u, big / small * v) / S
    w1, w2 = wofz(z1), wofz(z2)
    e = M.exp(-u * u / (2 * big * big) - v * v / (2 * small * small))
    F = w1 - e * w2
    f_big, f_small = fact * F.imag, fact * F.real
    T = fact * (abs(w1) + e * abs(w2))
    ex, ey = (f_big, f_small) if wide else (f_small, f_big)
    sxs, sys_ = _sgn(x), _sgn(y)
    if not jac:
        return sxs * ex, sys_ * ey, T
    d1, d2 = dwofz(z1, w1), dwofz(z2, w2)
    deu, dev = -u / (big * big) * e, -v / (small * small) * e
    Fu = d1 / S - e * (small / big) / S * d2 - w2 * deu
    Fv = 1j * d1 / S - e * 1j * (big / small) / S * d2 - w2 * dev
    sxy = sxs * sys_
    if wide:  # Ex = sgn(x) fact Im F(|x|, |y|), Ey = sgn(y) fact Re F
        J = (fact * Fu.imag, sxy * fact * Fv.imag, sxy * fact * Fu.real, fact * Fv.real)
    else:     # u = |y|, v = |x|: Ex = sgn(x) fact Re F, Ey = sgn(y) fact Im F
        J = (fact * Fv.real, sxy * fact * Fu.real, sxy * fact * Fv.imag, fact * Fu.imag)
    ratio = big / small
    Tjac = fact * ((2 * abs(z1 * w1) + TWO_OVER_SQRT_PI) / S
                   + e * ratio / S * (2 * abs(z2 * w2) + TWO_OVER_SQRT_PI)
                   + abs(w2) * (abs(deu) + abs(dev)))
    return sxs * ex, sys_ * ey, T, J, Tjac


def field_round(x, y, sigma, jac=False):
    """gaussian_fields.py:5-21: E = temp (x, y), temp = A (1 - exp(-r^2/(2 sigma^2))) / r^2, or the
    reference's linearised temp = sqrt(r^2) A / sigma where r^2 < 1e-20 (decided on the float64
    r^2, as the reference and the kernels decide it).  T = |E| (1 + exp(-q)) / (1 - exp(-q)) on the
    full branch (the two terms of 1 - exp(-q)), |E| on the linearised one.  With ``jac`` the
    derivative of the full branch, judged on a scale of the order of |J| (the kernel's derivative
    takes 1 - exp(-q) from expm1, which does not cancel); on the linearised branch the physical
    A/(2 sigma^2) of the
    field at the origin, which is what the tangent kernel returns there (the linearised branch
    itself has no derivative at 0)."""
    X, Y, sg = mpf(x), mpf(y), mpf(sigma)
    r2 = X * X + Y * Y
    if float(x) * float(x) + float(y) * float(y) < 1e-20:
        temp = M.sqrt(r2) * A / sg
        T = abs(temp) * M.sqrt(r2)
        J = (A / (2 * sg * sg), mpf(0), mpf(0), A / (2 * sg * sg))
        Tjac = A / (2 * sg * sg)
    else:
        q = r2 / (2 * sg * sg)
        eq = M.exp(-q)
        temp = (1 - eq) * A / r2
        T = A * (1 + eq) / M.sqrt(r2)
        dtemp = A * (eq / (2 * sg * sg) - (1 - eq) / r2) / r2
        J = (temp + 2 * X * X * dtemp, 2 * X * Y * dtemp, 2 * X * Y * dtemp, temp + 2 * Y * Y * dtemp)
        # the derivative's term scale is that of the form the tangent kernel evaluates, with
        # om = 1 - exp(-q) taken from expm1 (no cancellation): temp = A om / r2 and
        # 2 x^2 dtemp, |dtemp| <= A (exp(-q) / (2 sigma^2) + om / r2) / r2 -- of the order of |J|
        om = -M.expm1(-q)
        Tjac = A * (3 * om / r2 + eq / (sg * sg))
    if not jac:
        return temp * X, temp * Y, T
    return temp * X, temp * Y, T, J, Tjac


def is_round(sx, sy, min_sigma_diff):
    """gaussian_fields.py:115 / lattice._gauss_field_block, in float64."""
    return abs(float(sx) - float(sy)) < min_sigma_diff


def field(x, y, sx, sy, min_sigma_diff, jac=False):
    """gaussian_fields.py:107-121 for scalar sigmas (skip_Gs)."""
    if is_round(sx, sy, min_sigma_diff):
        return field_round(x, y, 0.5 * (float(sx) + float(sy)), jac)
    return field_ellip(x, y, sx, sy, jac)


_FIELD_CACHE = {}


def fields(x, y, sx, sy, min_sigma_diff, jac=False):
    """``field`` over arrays, as float64 arrays: Ex, Ey, T (and J [n, 4], Tjac with ``jac``).  The
    reference depends on |x|, |y| and the signs only, so each first-quadrant point is evaluated
    once; results are cached per (point, sigmas, branch)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    rnd = is_round(sx, sy, min_sigma_diff)
    n = len(x)
    Ex, Ey, T = np.empty(n), np.empty(n), np.empty(n)
    J, Tj = np.empty((n, 4)), np.empty(n)
    for k in range(n):
        key = (abs(float(x[k])), abs(float(y[k])), float(sx), float(sy), rnd, jac)
        hit = _FIELD_CACHE.get(key)
        if hit is None:
            r = field(key[0], key[1], sx, sy, min_sigma_diff, jac)
            hit = tuple(float(t) for t in r[:3])
            if jac:
                hit = hit + (tuple(float(t) for t in r[3]), float(r[4]))
            _FIELD_CACHE[key] = hit
        sxs, sys_ = _sgn(x[k]), _sgn(y[k])
        Ex[k], Ey[k], T[k] = sxs * hit[0], sys_ * hit[1], hit[2]
        if jac:
            jxx, jxy, jyx, jyy = hit[3]
            J[k] = (jxx, sxs * sys_ * jxy, sxs * sys_ * jyx, jyy)
            Tj[k] = hit[4]
    if jac:
        return Ex, Ey, T, J, Tj
    return Ex, Ey, T


# ----------------------------------------------------------------------------- line densities
def qgauss_cq(q, eps=1e-6):
    """qgauss.py:5-21 in mpmath (branches chosen in float64)."""
    cq = SQRT_PI
    Q = mpf(q)
    if q >= 1 + eps:
        cq *= M.gamma((3 - Q) / (2 * Q - 2)) / (M.sqrt(Q - 1) * M.gamma(1 / (Q - 1)))
    elif q <= 1 - eps:
        cq *= 2 * M.gamma(1 / (1 - Q)) / ((3 - Q) * M.sqrt(1 - Q) * M.gamma((3 - Q) / (2 - 2 * Q)))
    return cq


def qgauss(zeta, rvv, q, bunchlength_rms, eps=1e-6):
    """spacecharge.py:80-104 / qgauss.py:27-37,67-75 at sigma = zeta / rvv:
    (lambda, dlambda/dzeta, scale, scale of the derivative).  The scale is |lambda| (1 + 2 arg) for the Gaussian (exp is
    conditioned by its argument, and arg carries the rounding of zeta/rvv twice); for q != 1 it is
    |p| c u^(p-1) (1 + 2 arg |1-q|) + |lambda| (1 + |p ln u|) with p = 1/(1-q), u = 1 - arg (1-q)
    floored at the rounding of its own evaluation (so that a float64 u just inside the support
    edge where the exact one is just outside is within scale)."""
    sb = 1 / (M.sqrt(2) * mpf(bunchlength_rms))
    c = sb / qgauss_cq(q)
    sg = mpf(zeta) / mpf(rvv)
    arg = sb * sb * sg * sg
    darg = 2 * sb * sb * sg / mpf(rvv)
    if not abs(1 - q) > eps:
        lam = c * M.exp(-arg)
        return lam, -lam * darg, abs(lam) * (1 + 2 * arg), abs(lam * darg) * (3 + 2 * arg)
    p = 1 / (1 - mpf(q))
    up = 1 - arg * (1 - mpf(q))
    if up > 0:
        lam = c * up ** p
        dlam = -lam * p * (1 - mpf(q)) * darg / up
        tail = abs(lam) * (1 + abs(p * M.log(up)))
    else:
        lam, dlam, tail = mpf(0), mpf(0), mpf(0)
    om = abs(1 - mpf(q))
    ueff = max(up, 0) + EPS * (1 + 2 * arg * om)
    scale = abs(p) * c * ueff ** (p - 1) * (1 + 2 * arg * om) + tail
    dscale = abs(p) * c * om * abs(darg) * (abs(p - 1) * om * ueff ** (p - 2) * (1 + 2 * arg * om)
                                            + ueff ** (p - 1) * (3 + abs(p * M.log(ueff))))
    return lam, dlam, scale, dscale


def knots(z0, dz, n):
    """The abscissae the reference interpolates on (spacecharge.py:150: np.linspace)."""
    return np.linspace(z0, z0 + dz * (n - 1), n)


def _kernel_interval(zeta, z0, dz, n):
    """The interval the kernels (and the tangent kernel's derivative) take: floor((z - z0)/dz) in
    float64, clamped to [0, n-2].  At a knot the derivative is one-sided; this is the side."""
    i = int(math.floor((zeta - z0) / dz))
    return min(max(i, 0), n - 2)


def interp_linear(zeta, z0, dz, prof):
    """numpy.interp(zeta, knots, prof) exactly (clamped outside), with the kernel's one-sided
    derivative (0 outside [z0, last knot]), the scale |f_j| + |f_j+1| + |slope| (|z| + |x_j| + dz)
    and the derivative's 2 |slope|."""
    prof = np.asarray(prof, dtype=np.float64)
    n = len(prof)
    xk = knots(z0, dz, n)
    Z = mpf(zeta)
    i = _kernel_interval(zeta, z0, dz, n)
    dlam = mpf(0)
    last = float(Fraction(n - 1) * Fraction(dz) + Fraction(z0))  # the kernels form z0 + (n-1) dz in one FMA
    if not (zeta <= z0 or zeta >= last):
        dlam = (mpf(prof[i + 1]) - mpf(prof[i])) / mpf(dz)
    if zeta <= xk[0]:
        return mpf(prof[0]), dlam, abs(mpf(prof[0])), 2 * abs(dlam)
    if zeta >= xk[-1]:
        return mpf(prof[-1]), dlam, abs(mpf(prof[-1])), 2 * abs(dlam)
    j = int(np.searchsorted(xk, zeta, side="right")) - 1
    slope = (mpf(prof[j + 1]) - mpf(prof[j])) / (mpf(xk[j + 1]) - mpf(xk[j]))
    lam = mpf(prof[j]) + slope * (Z - mpf(xk[j]))
    scale = abs(mpf(prof[j])) + abs(mpf(prof[j + 1])) + abs(slope) * (abs(Z) + abs(mpf(xk[j])) + abs(mpf(dz)))
    return lam, dlam, scale, 2 * abs(dlam)


def interp_cubic(zeta, z0, dz, prof):
    """scipy CubicSpline(knots, prof)(zeta) from its own piecewise coefficients (end polynomials
    outside), exactly; the derivative of the piece the kernel selects; the scale is the sum of
    the magnitudes of the polynomial's terms plus |dlambda/dz| (|z| + |x_i|), and the same for the
    derivative."""
    from scipy.interpolate import CubicSpline

    prof = np.asarray(prof, dtype=np.float64)
    n = len(prof)
    xk = knots(z0, dz, n)
    c = CubicSpline(xk, prof).c
    Z = mpf(zeta)

    def piece(i):
        t = Z - mpf(xk[i])
        terms = [mpf(c[k, i]) * t ** (3 - k) for k in range(4)]
        dterms = [mpf(c[k, i]) * (3 - k) * t ** (2 - k) for k in range(3)]
        d2 = 6 * mpf(c[0, i]) * t + 2 * mpf(c[1, i])
        shift = abs(Z) + abs(mpf(xk[i]))
        return (sum(terms), sum(dterms), sum(abs(tt) for tt in terms) + abs(sum(dterms)) * shift,
                sum(abs(tt) for tt in dterms) + abs(d2) * shift)

    j = min(max(int(np.searchsorted(xk, zeta, side="right")) - 1, 0), n - 2)  # PPoly's interval
    lam, _, scale, _ = piece(j)
    _, dlam, _, dscale = piece(_kernel_interval(zeta, z0, dz, n))
    return lam, dlam, scale, dscale


# ----------------------------------------------------------------------------- kick prefactors
def bb4d_fact(chi, charge_ratio, q0, beta0, rvv, p0c, charge, beta_r):
    """beambeam.py:53-79: chi charge qe (charge_ratio q0) qe (1 + beta beta_r) /
    (p0c qe (beta + beta_r)), beta = beta0 / rvv (p0c in eV)."""
    beta = mpf(beta0) / mpf(rvv)
    br = mpf(beta_r)
    return (mpf(chi) * mpf(charge) * mpf(QE) * mpf(charge_ratio) * mpf(q0) * (1 + beta * br)
            / (mpf(p0c) * (beta + br)))


def sc_fact(chi, charge_ratio, q0, beta0, p0c, number_of_particles, length, circumference=1.0):
    """spacecharge.py:26-52, 80-104, 137-177 without the line density: chi charge_ratio N qe L /
    circumference * q0^2 (1 - beta0^2) / (p0c beta0) (p0c in eV)."""
    b0 = mpf(beta0)
    return (mpf(chi) * mpf(charge_ratio) * mpf(number_of_particles) * mpf(QE) * mpf(length)
            / mpf(circumference) * mpf(q0) ** 2 * (1 - b0 * b0) / (mpf(p0c) * b0))


# ----------------------------------------------------------------------------- point sets
RADII = np.logspace(-8, 3, 45)  # r / sigma per axis
ANGLES = np.array([0.0, 1e-6, 1e-3, 0.1, 0.3, 0.6, np.pi / 4, 0.9, 1.1, 1.4, 1.57, np.pi / 2 - 1e-6, np.pi / 2])


def points(sx, sy, radii=RADII, angles=ANGLES):
    """Structured transverse points for sigmas (sx, sy): x = rho sx cos(theta), y = rho sy sin(theta)
    over ``radii`` x ``angles`` (theta = 0 and pi/2 exactly on the axes), in all four quadrants,
    the axes with both signs of zero, and the origin with all four."""
    rho, th = np.meshgrid(radii, angles, indexing="ij")
    x = (rho * sx * np.cos(th)).ravel()
    y = (rho * sy * np.sin(th)).ravel()
    x[np.isclose(th.ravel(), np.pi / 2, rtol=0, atol=1e-15)] = 0.0
    y[th.ravel() == 0.0] = 0.0
    xs, ys = [], []
    for a in (1.0, -1.0):
        for b in (1.0, -1.0):
            xs.append(a * x)  # a zero coordinate takes the sign of a or b: +0.0 and -0.0
            ys.append(b * y)
    xs.append(np.array([0.0, -0.0, 0.0, -0.0]))
    ys.append(np.array([0.0, 0.0, -0.0, -0.0]))
    return np.concatenate(xs), np.concatenate(ys)
