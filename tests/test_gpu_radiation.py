"""Synchrotron radiation on the GPU (track_kernel_radiation): against the oracle per element and over
100 turns, energy loss per turn against the radiation integrals, damping times, the quantum
equilibrium, photon statistics, bitwise determinism and the refusals (include/xline_b200.h,
DESIGN.md §4.9)."""
import math

import numpy as np
import pytest
import torch

import xline_b200 as xl
from tests import radiation_oracle as RO
from xline_b200 import configs, lattice, optics

pytestmark = pytest.mark.gpu

ELECTRON = configs.ELECTRON_MASS_EV
P0C = 6e9
COORDS = ("x", "px", "y", "py", "zeta", "delta")
# The photon count inverts a Poisson CDF: where the uniform falls within a few ulp of a partial sum,
# exp(-nbar) (one ulp between CUDA and NumPy) can move k by one.  A particle whose oracle draws came
# that close is exempt from the coordinate comparison, as the NAFF tests exempt near-tied peaks.
TIE = 1e-12


def _ring(n_cells=8, theta=0.02, sextupoles=True, aperture=True):
    """A short 6 GeV ring of radiating bends (with a gradient) and quadrupoles, (skew) sextupoles, an
    aperture and a cavity that replaces the loss.  The ring need not close: theta = 0.02 (rho = 75 m)
    keeps the loss well inside the bucket."""
    els = []
    for c in range(n_cells):
        for sgn in (1.0, -1.0):
            els += [xl.Multipole(knl=[0.0, sgn * 0.35], ksl=[0.0, 0.0], length=0.3), xl.DriftExact(length=1.0)]
            if sextupoles:
                els += [xl.Multipole(knl=[0.0, 0.0, sgn * 2.0], ksl=[0.0, 0.0, 0.3])]
            els += [xl.Drift(length=0.5), xl.Multipole(knl=[theta, 0.01], ksl=[0.0, 0.0], hxl=theta, length=1.5),
                    xl.DriftExact(length=1.0)]
    u0 = optics.radiation_integrals(xl.Line(els), P0C, ELECTRON)["U0"]
    els += ([xl.LimitEllipse(a=0.02, b=0.01)] if aperture else []) + [_cavity(u0, 3 * u0)]
    return els


def _cavity(u0, volts):
    """A 500 MHz cavity whose synchronous phase (above transition) replaces the loss u0 at zeta ~ 0."""
    return xl.Cavity(voltage=volts, frequency=5e8, lag=180.0 - math.degrees(math.asin(u0 / volts)))


def _beam(n, rng, scale=1.0):
    return dict(x=rng.normal(0, 3e-4 * scale, n), px=rng.normal(0, 3e-5 * scale, n), y=rng.normal(0, 2e-4 * scale, n),
                py=rng.normal(0, 2e-5 * scale, n), zeta=rng.normal(0, 2e-3 * scale, n),
                delta=rng.normal(0, 1e-3 * scale, n))


def _line(els, mode, seed=0):
    line = xl.Line(els)
    line.radiation = mode
    line.radiation_seed = seed
    return line


def _track(line, cols, num_turns=1, **kw):
    p = xl.Particles(p0c=P0C, mass0=ELECTRON, device="cuda", **cols)
    line.track(p, num_turns=num_turns, **kw)
    torch.cuda.synchronize()
    return p.to_numpy()


def _tied(log, n):
    tied = np.zeros(n, dtype=bool)
    for e in log:
        if "margin" in e:
            tied[e["pid"][e["margin"] < TIE]] = True
    return tied


def _compare(got, want, tied, tol=1e-12):
    ok = ~tied
    np.testing.assert_array_equal(got["state"][ok], want["state"][ok])
    for k in COORDS:  # error relative to the beam's r.m.s. of the coordinate (as smoke() measures it)
        a, b = got[k][ok], want[k][ok]
        err = np.max(np.abs(a - b)) / max(np.sqrt(np.mean(b ** 2)), 1e-300)
        assert err < tol, (k, err)


@pytest.mark.parametrize("mode", RO.MODES)
def test_each_element_against_oracle(mode):
    rng = np.random.default_rng(1)
    cols = _beam(2048, rng, 3.0)
    for i, el in enumerate(_ring(1)):
        line = _line([el], mode, seed=5)
        got = _track(line, cols)
        log = []
        want = RO.run_oracle(lattice.element_specs([el]), cols, P0C, ELECTRON, radiation=mode, seed=5, log=log)
        _compare(got, want, _tied(log, 2048))


@pytest.mark.parametrize("mode", RO.MODES)
def test_short_ring_100_turns_against_oracle(mode):
    rng = np.random.default_rng(2)
    n = 256
    cols = _beam(n, rng)
    line = _line(_ring(), mode, seed=123)
    got = _track(line, cols, num_turns=100)
    log = []
    want = RO.run_oracle(line.to_specs(), cols, P0C, ELECTRON, num_turns=100, radiation=mode, seed=123, log=log)
    tied = _tied(log, n)
    assert tied.sum() <= 2, tied.sum()
    _compare(got, want, tied, tol=1e-11)
    if mode == "quantum":
        photons = sum(int(e["k"].sum()) for e in log)
        assert photons > 100 * n  # the comparison covered photon emission, not just empty halves


def _energy(delta):
    E0 = math.hypot(P0C, ELECTRON)
    P = (1 + np.asarray(delta)) * P0C
    return np.sqrt(P * P + ELECTRON ** 2) - E0


@pytest.mark.parametrize("name", ["petra_like", "petra4"])
def test_energy_loss_per_turn_matches_u0(name):
    if name == "petra_like":
        line, _, p0c, m0 = configs.config_petra_like(n=1)
    else:
        line, _, p0c, m0 = configs.config_petra4(n=1)
    for el in line.elements:
        if isinstance(el, (xl.Cavity, xl.RFMultipole)):
            el.voltage = 0.0
    line.radiation = "mean"
    r = optics.radiation_integrals(line, p0c, m0)
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=np.zeros(1))
    line.track(p, num_turns=1)
    dE = -float(_energy(p.to_numpy()["delta"])[0])
    # the loss changes delta by U0/E over the turn, and the loss scales as (1+delta)^2 (plus the
    # dispersion orbit it drives): agreement to O(U0/E)
    assert abs(dE / r["U0"] - 1) < 3 * r["U0"] / r["energy"], (dE, r["U0"])


def _damping_ring():
    """The test ring with theta = 0.2 (rho = 7.5 m: U0 ~ 8 MeV, tau_x ~ 2000 turns),
    uncoupled and linear (no sextupoles, no aperture), so that the integrals' plane-by-plane damping
    applies.  (``config_petra_like(n_cells=24)``, the other 6 GeV option, does not keep an
    off-momentum particle: its 96 m cells have ~9 m of dispersion under sextupoles made for 120 cells.)"""
    return xl.Line(_ring(theta=0.2, sextupoles=False, aperture=False)), P0C, ELECTRON


def _planes(m, tw):
    """Betatron emittances with the dispersion taken out (D, D' at the start of the line), and the
    longitudinal emittance, from the covariance of every store."""
    c = m.cov.cpu().numpy()
    d, dp = tw["dx"][0], tw["dpx"][0]
    t = np.eye(6)
    t[0, 5], t[1, 5] = -d, -dp
    c = np.einsum("ij,sjk,lk->sil", t, c, t)

    def em(a, b):
        return np.sqrt(np.maximum(c[:, a, a] * c[:, b, b] - c[:, a, b] ** 2, 0))

    return em(0, 1), em(2, 3), em(4, 5), np.sqrt(c[:, 5, 5])


def test_damping_times_match_radiation_integrals():
    """Mean mode: a small beam's emittances decay as exp(-2 t / tau).  The fit runs over 1.5 tau_x
    of the damping ring; tolerance 5 %: the integrals are first order in the
    amplitudes and in delta, the beam's 1e-4 relative energy spread and the synchronous-phase
    offset change the rates at the per-cent level."""
    line, p0c, m0 = _damping_ring()
    line.radiation = "mean"
    r = optics.radiation_integrals(line, p0c, m0)
    tw = optics.twiss(line)
    rng = np.random.default_rng(4)
    n = 512
    cols = dict(x=rng.normal(0, 1e-5, n), px=rng.normal(0, 1e-7, n), y=rng.normal(0, 1e-5, n),
                py=rng.normal(0, 1e-7, n), zeta=rng.normal(0, 1e-4, n), delta=rng.normal(0, 1e-5, n))
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)
    turns = int(1.5 * r["tau_x"])
    m = xl.BeamMoments(num_stores=turns // 50 + 1, start=0, skip=50)
    line.track(p, num_turns=turns, moments=m)
    t = m.turn.numpy().astype(float)
    ex, ey, ez, _ = _planes(m, tw)
    # after the start-up transient (the beam settles on the damped orbit); the longitudinal fit stops
    # at 2 tau_z: by then eps_z has shrunk e^4-fold and the zeta the slower betatron motion drives
    # through the bends (hxl x) starts to dominate it
    fits = {}
    for name, e, win in (("tau_x", ex, t >= 500), ("tau_y", ey, t >= 500),
                         ("tau_z", ez, (t >= 100) & (t <= 2 * r["tau_z"]))):
        slope = np.polyfit(t[win], np.log(e[win]), 1)[0]
        fits[name] = -2.0 / slope
    print("damping fits", fits, {k: r[k] for k in fits})
    for k in fits:
        assert abs(fits[k] / r[k] - 1) < 0.05, (k, fits[k], r[k])


def test_quantum_equilibrium_matches_radiation_integrals():
    """4096 particles from zero emittance, 5 tau_x in quantum mode.  Each store estimates eps_x and
    sigma_delta^2 with a statistical error of sqrt(2/N) = 2.2 %; averaging the stores of the last
    1.5 tau_x (about 3 independent values of eps_x, correlation time tau_x/2; 9 of sigma_delta^2)
    leaves ~1.3 % and ~0.8 % (sigma_delta: half of that).  Tolerance: 4 sigma plus 3 % for the
    thin-lens integrals' first-order treatment of H and of the dispersion orbit."""
    line, p0c, m0 = _damping_ring()
    line.radiation = "quantum"
    line.radiation_seed = 2024
    r = optics.radiation_integrals(line, p0c, m0)
    tw = optics.twiss(line)
    n = 4096
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=np.zeros(n), particle_id=np.arange(n))
    turns = int(5 * r["tau_x"])
    m = xl.BeamMoments(num_stores=turns // 100 + 1, start=0, skip=100)
    line.track(p, num_turns=turns, moments=m)
    t = m.turn.numpy().astype(float)
    ex, _, _, sd = _planes(m, tw)
    last = t >= turns - 1.5 * r["tau_x"]
    ex_eq, sd_eq = float(np.mean(ex[last])), float(np.sqrt(np.mean(sd[last] ** 2)))
    print("equilibrium eps_x %.4g (integrals %.4g), sigma_delta %.4g (integrals %.4g)"
          % (ex_eq, r["eps_x"], sd_eq, r["sigma_delta"]))
    assert abs(ex_eq / r["eps_x"] - 1) < 4 * 0.013 + 0.03
    assert abs(sd_eq / r["sigma_delta"] - 1) < 4 * 0.004 + 0.03


def test_photon_statistics_per_element():
    """1e6 particles through one bend: the mean and variance of the energy lost equal
    2 nbar <u> and 2 nbar <u^2> (two halves; nbar does not depend on delta to first order and u_c
    moves by 2 delta ~ 1e-6) within 5 sigma."""
    L, theta, n = 0.4, 0.02, 1_000_000
    el = xl.Multipole(knl=[theta], ksl=[0.0], hxl=theta, length=L)
    got = _track(_line([el], "quantum", seed=77), dict(x=np.zeros(n)))
    dE = -_energy(got["delta"])
    E0 = math.hypot(P0C, ELECTRON)
    m = math.sqrt((E0 - P0C) * (E0 + P0C))
    g = E0 / m
    kap = theta / L
    nbar = 5 / (2 * math.sqrt(3)) * RO.ALPHA * g * kap * L / 2
    uc = 1.5 * RO.HBAR_C * g ** 3 * kap
    mu, var = 2 * nbar * uc * 8 / (15 * math.sqrt(3)), 2 * nbar * uc ** 2 * 11 / 27
    m4 = np.mean((dE - dE.mean()) ** 4)
    assert abs(dE.mean() - mu) < 5 * math.sqrt(var / n)
    assert abs(dE.var() - var) < 5 * math.sqrt((m4 - var ** 2) / n)


def test_bitwise_determinism():
    rng = np.random.default_rng(6)
    n = 3000
    cols = _beam(n, rng)
    cols["x"] = cols["x"] * 50.0  # a heavy-loss beam: the aperture removes many, compaction runs
    cols["particle_id"] = np.arange(n) * 7 + 3
    line = _line(_ring(), "quantum", seed=99)
    ref = _track(line, cols, num_turns=40)
    assert 0.05 * n < (ref["state"] == 0).sum() < 0.95 * n
    for kw in (dict(particles_per_thread=1), dict(particles_per_thread=2), dict(particles_per_thread=3),
               dict(particles_per_thread=4), dict(particles_per_thread=1, threads_per_block=256),
               dict(turns_per_launch=3), dict(turns_per_launch=7, compact_threshold=1e-6),
               dict(turns_per_item=1), dict(turns_per_item=-1)):
        got = _track(line, cols, num_turns=40, **kw)
        for k in COORDS + ("state", "at_turn", "at_element"):
            np.testing.assert_array_equal(got[k], ref[k], err_msg=str((kw, k)))
    # T1 then T2 turns
    p = xl.Particles(p0c=P0C, mass0=ELECTRON, device="cuda", **cols)
    line.track(p, num_turns=15)
    line.track(p, num_turns=25)
    split = p.to_numpy()
    for k in COORDS + ("state", "at_turn"):
        np.testing.assert_array_equal(split[k], ref[k])
    # one particle alone, with its id, against the same particle in the batch
    j = int(np.flatnonzero(ref["state"] == 1)[0])
    alone = _track(line, {k: v[j:j + 1] for k, v in cols.items()}, num_turns=40)
    for k in COORDS:
        assert alone[k][0] == ref[k][j]
    # another seed, other draws
    other = _track(_line(_ring(), "quantum", seed=100), cols, num_turns=40)
    assert not np.array_equal(other["delta"], ref["delta"])


def test_elem_by_elem_uses_the_same_draws():
    rng = np.random.default_rng(8)
    cols = _beam(64, rng)
    line = _line(_ring(2), "quantum", seed=31)
    ref = _track(line, cols)
    p = xl.Particles(p0c=P0C, mass0=ELECTRON, device="cuda", **cols)
    line.track_elem_by_elem(p, start=False)
    got = p.to_numpy()
    for k in COORDS:
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-12, atol=1e-18)
    tr = line.trace_elem_by_elem(xl.Particles(p0c=P0C, mass0=ELECTRON, device="cuda", **cols))
    for f, k in enumerate(COORDS):
        np.testing.assert_allclose(tr[-1, f].cpu().numpy(), ref[k], rtol=1e-12, atol=1e-18)


def test_polygon_apertures_ride_on_the_radiation_twin():
    rng = np.random.default_rng(9)
    cols = _beam(1024, rng, 20.0)
    els = _ring(2)
    rect = els + [xl.LimitRect(min_x=-3e-3, max_x=3e-3, min_y=-2e-3, max_y=2e-3)]
    poly = els + [xl.LimitPolygon(x_vertices=[-3e-3, 3e-3, 3e-3, -3e-3], y_vertices=[-2e-3, -2e-3, 2e-3, 2e-3])]
    a = _line(rect, "quantum", seed=4)
    b = _line(poly, "quantum", seed=4)
    b.polygon_apertures = True
    ra, rb = _track(a, cols, num_turns=5), _track(b, cols, num_turns=5)
    assert b.pack().flags & lattice.F_POLYGONS and b.pack().flags & lattice.F_RADIATION
    on_edge = (np.abs(np.abs(ra["x"]) - 3e-3) < 1e-15) | (np.abs(np.abs(ra["y"]) - 2e-3) < 1e-15)
    assert not on_edge.any()
    for k in COORDS + ("state",):
        np.testing.assert_array_equal(ra[k], rb[k])


def test_refusals():
    line = _line(_ring(1), "mean")
    cols = dict(x=np.zeros(4))
    with pytest.raises(ValueError, match="radiation"):
        _track(line, cols, strict=True)
    with pytest.raises(ValueError, match="one species"):
        _track(line, dict(x=np.zeros(4), chi=np.array([1.0, 0.5, 1.0, 1.0])))
    with pytest.raises(Exception, match="one species"):  # the C ABI's own check
        _track(line, cols, _general_kernels=True)
    p = xl.Particles(p0c=P0C, mass0=ELECTRON, device="cuda", x=np.zeros(4))
    with pytest.raises(ValueError, match="radiation"):
        line.track_tangent(p, xl.TangentMap(4, device="cuda"))
    with pytest.raises(ValueError, match="radiation"):
        xl.closed_orbit(line, p)
    # without radiation the same line tracks
    line.radiation = None
    _track(line, cols)
