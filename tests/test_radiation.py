"""Synchrotron radiation without a GPU: the random stream, the photon-energy table, the packed
record, the oracle's map against closed forms, the packed-format interpreter against the oracle,
the radiation integrals and the refusals (include/xline_b200.h, DESIGN.md §4.9)."""
import ctypes as C
import math
import re

import numpy as np
import pytest

import xline_b200 as xl
from tests import packed_interpreter as PI
from tests import radiation_oracle as RO
from xline_b200 import lattice, optics

ELECTRON = 0.51099895e6
P0C = 6e9
HEADER = open(RO.ROOT + "/include/xline_b200.h").read()


def _hdefine(name):
    return int(re.search(r"#define %s \(?([0-9]+)" % name, HEADER).group(1).replace("u", ""), 0)


# ---------------------------------------------------------------- random stream
@pytest.mark.parametrize("ctr,key,out", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, out):
    r = RO.philox(*[np.array([v]) for v in ctr], *key)
    assert " ".join("%08x" % int(w[0]) for w in r) == out


def test_counter_and_uniform_layout():
    seed, pid, turn, elem = 0x0123456789abcdef, (5 << 32) | 7, 11, 1234
    r = RO.philox([pid & 0xffffffff], [pid >> 32], [turn], [(elem << 8) | (1 << 7) | 3], seed & 0xffffffff, seed >> 32)
    u2j, u2j1 = RO.uniforms(seed, [pid], [turn], elem, 1, 3)
    w0 = (int(r[1][0]) << 32) | int(r[0][0])
    w1 = (int(r[3][0]) << 32) | int(r[2][0])
    assert u2j[0] == ((w0 >> 11) + 0.5) * 2.0 ** -53 and u2j1[0] == ((w1 >> 11) + 0.5) * 2.0 ** -53
    # extremes stay inside (0, 1)
    assert RO.u01([0], [0])[0] == 2.0 ** -54 and RO.u01([0xffffffff], [0xffffffff])[0] == 1 - 2.0 ** -54
    # the half and the call index change the draw
    assert RO.uniforms(seed, [pid], [turn], elem, 0, 3)[0][0] != u2j[0]
    assert RO.uniforms(seed, [pid], [turn], elem, 1, 2)[0][0] != u2j[0]


# ---------------------------------------------------------------- photon-energy table
def test_table_against_scipy_inverse_cdf():
    U = np.concatenate([np.geomspace(1e-9, 0.7, 12), 0.75 + np.linspace(0, 0.2, 5), 1 - np.geomspace(0.04, 1e-15, 12)])
    ref = np.array([RO.GEN.inverse(u) for u in U])
    assert np.max(np.abs(RO.synrad_x(U) - ref) / ref) < 1e-6


def test_table_moments():
    m1, m2 = RO.GEN.moments(RO.LO, RO.HI)
    assert abs(m1 - 8 / (15 * math.sqrt(3))) < 1e-6 and abs(m2 - 11 / 27) < 1e-6
    # the spectrum's normalisation and the photon rate per unit bend angle
    from scipy.integrate import quad
    from scipy.special import kv

    total, _ = quad(lambda x: RO.GEN._S(x), 0, 60, limit=400, points=[1e-6, 1e-3, 1])
    assert abs(total - 5 * math.pi / 3) < 1e-8
    assert abs(5 / (2 * math.sqrt(3)) - 1.443375673) < 1e-9
    assert kv(5 / 3, 1.0) > 0


def test_table_header_constants_match_script():
    txt = open(RO.ROOT + "/xline_b200/csrc/synrad_table.inc").read()
    for name, val in (("N_LO", RO.GEN.N_LO), ("N_HI", RO.GEN.N_HI), ("DEG", RO.GEN.DEG)):
        assert int(re.search(r"XLB_SYNRAD_%s (\d+)" % name, txt).group(1)) == val


# ---------------------------------------------------------------- the record
def test_header_constants():
    assert "XLB_T_MULTIPOLE_RAD = 20" in HEADER and "XLB_T__COUNT = 21" in HEADER
    assert _hdefine("XLB_F_RADIATION") == lattice.F_RADIATION == 32
    assert _hdefine("XLB_RAD_MEAN") == lattice.RADIATION_MODES["mean"]
    assert _hdefine("XLB_RAD_QUANTUM") == lattice.RADIATION_MODES["quantum"]
    assert "#define XLB_ABI_VERSION 4" in HEADER


@pytest.mark.parametrize("curved", [False, True])
def test_record_layout_and_constants(curved):
    from scipy.constants import alpha, c, e, epsilon_0, hbar

    mp = xl.Multipole(knl=[0.01, 0.2], ksl=[0.0, 0.0], hxl=0.01 if curved else 0.0, length=0.5)
    pk = lattice.pack_line([mp, xl.Drift(length=1.0)], radiation="quantum", radiation_seed=(1 << 63) + 5)
    w = pk.words
    f = w.view(np.float64)
    assert pk.flags & lattice.F_RADIATION and pk.record_counts[20] == 1
    assert int(w[0]) & 0xff == 20 and (int(w[0]) >> 8) & 0xff == 1
    assert int(w[1]) == 2 and f[2] == 0.5 and f[3] == 2.0
    assert f[4] == e / (4 * math.pi * epsilon_0) and f[5] == hbar * c / e and f[6] == alpha
    assert int(w[7]) == (1 << 63) + 5
    plain = lattice.pack_line([mp], fuse=False)
    size = (int(plain.words[0]) >> 16) & 0x3fff
    np.testing.assert_array_equal(w[8: 8 + 2 * size], plain.words[: 2 * size])
    assert (int(w[0]) >> 16) & 0x3fff == 4 + size
    assert _validate(pk) == 0


def _validate(pk, **override):
    lat = pk.c_lattice()
    for k, v in override.items():
        setattr(lat, k, v)
    return xl._cabi.lib().xlb_lattice_validate(C.byref(lat))


def test_validator_errors():
    mp = xl.Multipole(knl=[0.01], hxl=0.01, length=0.5)
    pk = lattice.pack_line([mp, xl.Drift(length=1.0)], radiation="mean")
    assert _validate(pk, flags=pk.flags & ~lattice.F_RADIATION) == -3
    assert _validate(pk, flags=pk.flags | lattice.F_BEAMFIELDS) == -3
    assert _validate(pk, n_elements=(1 << 24) + 1) == -3
    for word, bad in ((1, 3), (2, np.float64(0.0).view(np.uint64)), (4, np.float64(np.inf).view(np.uint64))):
        w = pk.words.copy()
        w[word] = bad
        bad_pk = lattice.PackedLattice(w, pk.chunk_words, pk.n_chunks, pk.n_elements, pk.flags,
                                       dict(layout=[], words=0), pk.record_counts)
        assert _validate(bad_pk) == -3


def test_radiating_multipoles_stay_out_of_blocks():
    els = [xl.Multipole(knl=[0.0, 0.1], length=0.3), xl.LimitEllipse(a=0.01, b=0.01), xl.Drift(length=1.0),
           xl.Multipole(knl=[0.0, 0.1]), xl.LimitRect(min_x=-0.1, max_x=0.1, min_y=-0.1, max_y=0.1),
           xl.Drift(length=1.0), xl.Multipole(knl=[0.0, -0.1]), xl.Multipole(knl=[0.01], hxl=0.01, length=0.4),
           xl.Drift(length=1.0)]
    off = lattice.pack_line(els)
    on = lattice.pack_line(els, radiation="mean")
    assert 20 not in off.record_counts
    assert on.record_counts[20] == 2
    # the zero-length multipole still fuses with its aperture and drift; the one before the second
    # radiating multipole cannot merge with it
    assert sum(v for k, v in on.record_counts.items() if k & 0xe0 == 0x80) == 2
    assert on.record_counts[lattice.T_LIMIT_ELLIPSE] == 1
    assert on.flags & lattice.F_LOW_ORDER


# ---------------------------------------------------------------- the map
def test_mean_mode_bend_closed_form():
    L, theta = 0.4, 0.01
    spec = [("Multipole", dict(knl=[theta], ksl=[0.0], hxl=theta, hyl=0.0, length=L))]
    cols = dict(x=np.zeros(1), px=np.zeros(1), y=np.zeros(1), py=np.zeros(1), zeta=np.zeros(1), delta=np.zeros(1))
    out = RO.run_oracle(spec, cols, P0C, ELECTRON, radiation="mean")
    E0 = math.hypot(P0C, ELECTRON)
    m = math.sqrt((E0 - P0C) * (E0 + P0C))  # the rest energy as the map takes it (include/xline_b200.h)
    assert abs(m / ELECTRON - 1) < 1e-7
    g, b = E0 / m, P0C / E0
    dE1 = (2 / 3) * RO.K_E * b ** 3 * g ** 4 * (theta / L) ** 2 * L / 2
    # exit half with the new delta: kappa scales as 1/(1+delta), gamma^4 beta^3 with the energy
    p = xl.Particles(p0c=P0C, mass0=ELECTRON, device="cpu", delta=[0.0])
    p.add_to_energy(-dE1)
    d1 = float(p.delta[0])
    P1 = (1 + d1) * P0C
    E1 = math.hypot(P1, ELECTRON)
    E1 = math.sqrt(P1 * P1 + m * m)
    dE2 = (2 / 3) * RO.K_E * (P1 / E1) ** 3 * (E1 / m) ** 4 * (theta / L / (1 + d1)) ** 2 * L / 2
    p.add_to_energy(-dE2)
    assert abs(out["delta"][0] - float(p.delta[0])) < 1e-15 * abs(out["delta"][0]) * 10
    # px: the bend's own kick hxl*delta at the intermediate delta, scaled by the exit half
    assert abs(out["px"][0] - theta * d1 * (1 + float(p.delta[0])) / (1 + d1)) < 1e-18


def _random_line(rng, n=30):
    els = []
    for _ in range(n):
        kind = rng.integers(6)
        if kind == 0:
            th = rng.uniform(0.002, 0.02)
            els.append(xl.Multipole(knl=[th, rng.normal(0, 0.05)], ksl=[0.0, 0.0], hxl=th, length=rng.uniform(0.2, 1)))
        elif kind == 1:
            els.append(xl.Multipole(knl=[0.0, rng.normal(0, 0.2), rng.normal(0, 2)], ksl=[0.0, 0.0, rng.normal(0, 0.5)],
                                    length=rng.uniform(0.1, 0.5)))
        elif kind == 2:
            els.append(xl.Multipole(knl=[0.0, rng.normal(0, 0.1)]))
        elif kind == 3:
            els.append(xl.DriftExact(length=rng.uniform(0.1, 2)))
        elif kind == 4:
            els.append(xl.Drift(length=rng.uniform(0.1, 2)))
        else:
            els.append(xl.LimitEllipse(a=0.004, b=0.003))
    els.append(xl.Cavity(voltage=3e7, frequency=5e8, lag=175.0))
    return els


@pytest.mark.parametrize("mode", RO.MODES)
def test_interpreter_against_oracle_on_random_lines(mode):
    rng = np.random.default_rng(3 if mode == "mean" else 4)
    for trial in range(3):
        els = _random_line(rng)
        n = 64
        cols = dict(x=rng.normal(0, 1e-3, n), px=rng.normal(0, 1e-4, n), y=rng.normal(0, 1e-3, n),
                    py=rng.normal(0, 1e-4, n), zeta=rng.normal(0, 1e-3, n), delta=rng.normal(0, 1e-3, n))
        pk = lattice.pack_line(els, radiation=mode, radiation_seed=trial + 17, merge=False)
        got = PI.track(pk, cols, P0C, ELECTRON, num_turns=3)
        want = RO.run_oracle(lattice.element_specs(els), cols, P0C, ELECTRON, num_turns=3, radiation=mode,
                             seed=trial + 17)
        np.testing.assert_array_equal(got["state"], want["state"])
        for k in ("x", "px", "y", "py", "zeta", "delta"):
            np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-15)


def test_quantum_mean_matches_mean_mode():
    """The expected quantum loss of one half is (2/3) K_e gamma^4 kappa^2 l_h: with many draws it
    agrees with the mean mode's up to beta^3 and statistics."""
    L, theta, n = 0.4, 0.02, 200_000
    spec = [("Multipole", dict(knl=[theta], ksl=[0.0], hxl=theta, hyl=0.0, length=L))]
    cols = dict(delta=np.zeros(n))
    q = RO.run_oracle(spec, cols, P0C, ELECTRON, radiation="quantum", seed=9)
    m = RO.run_oracle(spec, dict(delta=np.zeros(1)), P0C, ELECTRON, radiation="mean")
    mean, err = np.mean(q["delta"]), np.std(q["delta"]) / math.sqrt(n)
    assert abs(mean - m["delta"][0]) < 5 * err


# ---------------------------------------------------------------- radiation integrals
def test_radiation_integrals_isomagnetic_ring():
    n, rho = 64, 25.0
    theta = 2 * math.pi / n
    L = rho * theta
    k1 = 0.6
    els = []
    for i in range(n):
        els += [xl.Multipole(knl=[0.0, k1 if i % 2 else -k1]), xl.Drift(length=1.0),
                xl.Multipole(knl=[theta], hxl=theta, length=L), xl.Drift(length=1.0)]
    r = optics.radiation_integrals(xl.Line(els), P0C, ELECTRON)
    assert abs(r["I2"] - 2 * math.pi / rho) < 1e-12 * r["I2"]
    assert abs(r["I3"] - 2 * math.pi / rho ** 2) < 1e-12 * r["I3"]
    E0 = math.hypot(P0C, ELECTRON)
    assert abs(r["U0"] - (2 / 3) * RO.K_E * (P0C / E0) ** 3 * (E0 / ELECTRON) ** 4 * 2 * math.pi / rho) < 1e-9 * r["U0"]
    assert abs(r["Jx"] + r["Jy"] + r["Jz"] - 4) < 1e-12
    # C_gamma: U0 = 88.46e-6 m/GeV^3 E^4 / rho
    assert abs(r["U0"] / (8.846e-5 * 6.0 ** 4 / rho * 1e9) - 1) < 1e-3


# ---------------------------------------------------------------- refusals
def test_refusals_at_pack_time():
    mp = xl.Multipole(knl=[0.01], hxl=0.01, length=0.5)
    with pytest.raises(ValueError, match="radiation"):
        lattice.pack_line([mp], strict=True, radiation="mean")
    with pytest.raises(ValueError, match="radiation"):
        lattice.pack_line([mp], radiation="classical")
    with pytest.raises(ValueError, match="radiation_seed"):
        lattice.pack_line([mp], radiation="mean", radiation_seed=-1)
    bb = xl.BeamBeam4D(charge=1e10, sigma_x=1e-3, sigma_y=2e-3, beta_r=1.0, x_bb=0, y_bb=0, d_px=0, d_py=0)
    with pytest.raises(ValueError, match="radiation"):
        lattice.pack_line([mp, bb], radiation="mean")


def test_line_options_stamp_the_pack_cache():
    line = xl.Line([xl.Multipole(knl=[0.01], hxl=0.01, length=0.5), xl.Drift(length=1.0)])
    a = line.pack()
    line.radiation = "mean"
    b = line.pack()
    line.radiation_seed = 3
    c = line.pack()
    assert 20 not in a.record_counts and b.record_counts[20] == 1
    assert c is not b and int(c.words[7]) == 3
    assert line.algorithmic_ops_per_turn() > lattice.algorithmic_ops(line.elements)


def test_tangent_refuses_radiation():
    line = xl.Line([xl.Multipole(knl=[0.01], hxl=0.01, length=0.5), xl.Drift(length=1.0)])
    line.radiation = "mean"
    p = xl.Particles(p0c=P0C, mass0=ELECTRON, device="cpu", x=[0.0])
    with pytest.raises(ValueError, match="radiation"):
        xl.closed_orbit(line, p)
