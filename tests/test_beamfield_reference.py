"""The 34-digit beam-field reference (tests/beamfield_reference.py) against an independent
statement of the same field, and what it says about the float64 evaluations: the NumPy
restatement of the kernel's Faddeeva series, scipy.special.wofz and the oracle's field_gauss."""
import numpy as np
import mpmath as M
from scipy.special import wofz as scipy_wofz

from oracle import xline_oracle as xo
from tests import beamfield_reference as R
from tests.test_faddeeva import weideman


def _field_integral(x, y, sx, sy):
    """E of a 2-D Gaussian of unit line charge from its integral representation,
    Ex = A x int_0^inf exp(-x^2/(a+q) - y^2/(b+q)) / ((a+q)^(3/2) (b+q)^(1/2)) dq, a = 2 sx^2,
    b = 2 sy^2, A = 1/(2 pi eps0) (Ey with the powers swapped); at 40 digits, the quadrature
    split where the integrand changes scale."""
    with M.workdps(40):
        X, Y, a, b = M.mpf(x), M.mpf(y), 2 * M.mpf(sx) ** 2, 2 * M.mpf(sy) ** 2

        def g(q, px, py):
            return M.exp(-X * X / (a + q) - Y * Y / (b + q)) / ((a + q) ** px * (b + q) ** py)

        pts = [M.mpf(0)] + sorted({a, b, X * X + Y * Y}) + [M.inf]
        ex = R.A * X * M.quad(lambda q: g(q, 1.5, 0.5), pts)
        ey = R.A * Y * M.quad(lambda q: g(q, 0.5, 1.5), pts)
        return ex, ey


def _integral_points():
    out = []
    for sx, sy in ((1e-3, 0.6e-3), (1e-3, 1e-6), (1e-3, 1e-3 + 2e-10), (1e-3, 1e-3 * 1.01)):
        for s1, s2 in ((sx, sy), (sy, sx)):  # both orientations
            for rho, th in ((1e-6, 0.4), (0.5, 1.2), (3.0, 0.05), (1e3, 0.8), (2.0, 1.5), (30.0, 0.3)):
                out.append((rho * s1 * np.cos(th), rho * s2 * np.sin(th), s1, s2))
    return out[:50]


def test_bassetti_erskine_matches_the_integral_representation():
    """Near the origin, far field, flat 1e-3, near-round, both orientations: >= 25 digits of |E|."""
    worst = 0.0
    for x, y, sx, sy in _integral_points():
        ex, ey, _ = R.field_ellip(x, y, sx, sy)
        ix, iy = _field_integral(x, y, sx, sy)
        err = float(M.sqrt((ex - ix) ** 2 + (ey - iy) ** 2) / M.sqrt(ix * ix + iy * iy))
        worst = max(worst, err)
        assert err < 1e-25, (x, y, sx, sy, err)
    print("Bassetti-Erskine vs integral: %.1e of |E| at worst" % worst)


def test_round_field_limit_and_branches():
    """The round field is the integral with sx = sy; the linearised branch below r^2 = 1e-20 is the
    reference's, not the physical limit."""
    for x, y in ((3e-4, -1e-4), (2e-2, 5e-3), (1e-9, 2e-9)):
        ex, ey, T = R.field_round(x, y, 1e-3)  # 1 - exp(-q) cancels near the origin: judged on T
        ix, iy = _field_integral(x, y, 1e-3, 1e-3)
        assert abs(ex - ix) <= 1e-25 * T and abs(ey - iy) <= 1e-25 * T
    ex, ey, _ = R.field_round(3e-11, 4e-11, 1e-3)
    X, Y = M.mpf(3e-11), M.mpf(4e-11)
    assert ex == M.sqrt(X * X + Y * Y) * R.A / M.mpf(1e-3) * X  # r A / sigma x, ...
    assert ex < 1e-12 * R.A * X / (2 * M.mpf(1e-3) ** 2)  # ... far below the physical A x / (2 sigma^2)
    assert R.is_round(1e-3, 1e-3 + 0.5e-10, 1e-10) and not R.is_round(1e-3, 1e-3 + 2e-10, 1e-10)


def _faddeeva_points():
    """The families of test_faddeeva.test_weideman_matches_wofz_in_first_quadrant, 6 000 points."""
    rng = np.random.default_rng(0)
    r = 10 ** rng.uniform(-8, 6, 1500)
    th = rng.uniform(0, np.pi / 2, 1500)
    return np.concatenate([
        r * np.exp(1j * th),
        rng.uniform(0, 8, 1000) + 1j * rng.uniform(0, 8, 1000),
        rng.uniform(0, 30, 1000) + 1j * 10 ** rng.uniform(-12, -1, 1000),
        1j * 10 ** rng.uniform(-8, 3, 300), 10 ** rng.uniform(-8, 1.5, 300) + 0j,
        np.array([0j, 1e-300 + 1e-300j]),
        10 ** rng.uniform(-12, -2, 950) + 1j * rng.uniform(0, 4, 950),
        10 ** rng.uniform(-12, -2, 948) + 1j * 10 ** rng.uniform(-12, -2, 948),
    ])


_W = {}


def _w_reference():
    if not _W:
        z = _faddeeva_points()
        _W["z"] = z
        _W["w"] = np.array([complex(R.wofz(M.mpc(v.real, v.imag))) for v in z])
        # |w| is never below 1/(sqrt(pi) |z|) here, so the complex rounding of the 34-digit value
        # to float64 costs 1e-16 of |w| at most
    return _W["z"], _W["w"]


def test_weideman_series_against_34_digits():
    """The NumPy restatement of the kernel's series is within 1e-14 of |w| (7.6e-15 measured);
    scipy.special.wofz on the same points is off by up to 2.3e-14 of |w| near the real axis, so the
    5e-14 of test_faddeeva measures scipy at least as much as the series."""
    z, ref = _w_reference()
    for form in (True, False):
        err = np.abs(weideman(z, form) - ref) / np.abs(ref)
        assert err.max() < 1e-14, (form, err.max(), z[err.argmax()])
    sc = np.abs(scipy_wofz(z) - ref) / np.abs(ref)
    series = np.abs(weideman(z) - ref) / np.abs(ref)
    print("max err of |w|: series %.2e, scipy.special.wofz %.2e" % (series.max(), sc.max()))
    assert sc.max() < 5e-14


ORACLE_SIGMAS = ((1e-3, 1e-3 / 1.6), (1e-3 / 10, 1e-3), (1e-3, 1e-6), (1e-3 + 2e-10, 1e-3), (1e-3, 1e-3))
ORACLE_TOL = 3e-14  # of T (measured 1.0e-14)


def test_oracle_field_against_the_reference():
    """The float64 oracle (scipy.special.wofz, NumPy exp) is within ORACLE_TOL of the field scale T
    of the reference on the structured point sets; the number is the float64 baseline the GPU
    kernels are compared with in test_gpu_beamfield_accuracy."""
    worst = 0.0
    for sx, sy in ORACLE_SIGMAS:
        x, y = R.points(sx, sy, radii=R.RADII[::2])
        ex, ey, T = R.fields(x, y, sx, sy, 1e-10)
        ox, oy = xo.field_gauss(x, y, sx, sy, 1e-10, True)
        z = T == 0  # the origin of the round field: both exactly 0
        assert np.all(ox[z] == 0) and np.all(oy[z] == 0) and np.all(ex[z] == 0)
        err = max(np.max(np.abs(ox - ex)[~z] / T[~z]), np.max(np.abs(oy - ey)[~z] / T[~z]))
        worst = max(worst, err)
        assert err < ORACLE_TOL, (sx, sy, err)
    print("oracle field_gauss: %.2e of T at worst" % worst)


def test_line_densities():
    """q-Gaussian switch and support, interpolation semantics (numpy.interp, CubicSpline)."""
    from scipy.interpolate import CubicSpline

    # q = 1 +- 1e-7 is the Gaussian (|1 - q| <= 1e-6), 1 +- 2e-6 is not
    g = R.qgauss(0.3, 1.0, 1.0, 0.5)[0]
    assert R.qgauss(0.3, 1.0, 1 + 1e-7, 0.5)[0] == g
    assert abs(R.qgauss(0.3, 1.0, 1 + 2e-6, 0.5)[0] / g - 1) < 1e-5
    assert R.qgauss(0.3, 1.0, 1 + 2e-6, 0.5)[0] != g
    # compact support for q < 1, and zeta / rvv
    assert R.qgauss(10.0, 1.0, 0.7, 0.5)[0] == 0 and R.qgauss(10.0, 1.0, 0.7, 0.5)[1] == 0
    assert R.qgauss(0.6, 2.0, 1.0, 0.5)[0] == R.qgauss(0.3, 1.0, 1.0, 0.5)[0]
    assert abs(float(R.qgauss(0.3, 1.0, 0.7, 0.5)[0]) - xo.qgauss_eval(0.3, 0.7, 1 / (np.sqrt(2) * 0.5),
                                                                       xo.qgauss_cq(0.7))) < 1e-14
    # the oracle's pieces at and off the knots
    prof = np.array([0.0, 1.0, 3.0, 2.5, 0.5, 0.2])
    z0, dz = -0.25, 0.1
    xk = R.knots(z0, dz, len(prof))
    cs = CubicSpline(xk, prof)
    for z in list(xk) + [np.nextafter(v, np.inf) for v in xk] + [np.nextafter(v, -np.inf) for v in xk] + [
            z0 - 1.0, xk[-1] + 0.7, -0.123]:
        lam, _, sc, _ = R.interp_linear(z, z0, dz, prof)
        assert abs(float(lam) - np.interp(z, xk, prof)) <= 4e-16 * float(sc), z
        lam, _, sc, _ = R.interp_cubic(z, z0, dz, prof)
        assert abs(float(lam) - float(cs(z))) <= 1e-15 * float(sc), z
    assert R.interp_linear(z0 - 1, z0, dz, prof)[1] == 0 and R.interp_linear(xk[-1], z0, dz, prof)[1] == 0


def test_qgauss_next_to_the_switch_is_refused_like_the_reference():
    """Just outside |1 - q| <= 1e-6 the normalisation Gamma(1/|1-q|) overflows: cq = inf/inf is NaN
    and both the reference (qgauss_eval's assert abs(cq) > 0) and the packer refuse the lens."""
    import pytest

    import xline_b200 as xl
    from xline_b200.lattice import pack_line

    for q in (1 + 2e-6, 1 - 2e-6):
        with np.errstate(all="ignore"):
            assert np.isnan(xo.qgauss_cq(q))
        el = xl.SCQGaussProfile(number_of_particles=1e11, bunchlength_rms=0.2, sigma_x=1e-3, sigma_y=6e-4,
                                length=1.0, q_parameter=q)
        with pytest.raises(AssertionError):
            pack_line([el], strict=False)
        o = xo.OracleParticles(1, p0c=1e9, mass0=9.38e8, x=np.array([1e-3]), zeta=np.array([0.1]))
        with pytest.raises(AssertionError):
            xo.line_track(xl.Line([el]).to_specs(), o)
