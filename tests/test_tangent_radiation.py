"""Radiation in the tangent map without a GPU: the NumPy statement of the radiating record's Jacobian
and diffusion (tests/tangent_radiation_oracle.py) against Richardson-extrapolated central differences
of the packed interpreter's map, V_h against the photon statistics of the committed table, the
header and the refusals that need no device."""
import math
import os
import re

import numpy as np
import pytest

import xline_b200 as xl
from tests import radiation_oracle as RO
from tests import tangent_oracle as TO
from tests import tangent_radiation_oracle as TRO
from xline_b200 import _cabi, configs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ELECTRON = configs.ELECTRON_MASS_EV
P0C = 6e9
Z = np.array([1.2e-3, -2.1e-4, -0.7e-3, 1.3e-4, 0.05, 1.7e-4])

CASES = [
    ("straight_skew_sextupole", xl.Multipole(knl=[0.0, 0.35, 2.0], ksl=[0.0, 0.05, 0.3], length=0.3), Z),
    ("curved_gradient", xl.Multipole(knl=[0.02, 0.01], ksl=[0.0, 0.0], hxl=0.02, length=1.5), Z),
    ("curved_skew_hyl", xl.Multipole(knl=[0.03, 0.2, 1.0], ksl=[1e-3, -0.05], hxl=0.03, hyl=1e-3, length=1.2), Z),
    ("curved_negative_k0l", xl.Multipole(knl=[-0.02, 0.1], ksl=[0.0, 0.0], hxl=-0.02, length=0.8), Z),
    ("quadrupole_on_axis", xl.Multipole(knl=[0.0, 0.35], ksl=[0.0, 0.0], length=0.3),
     np.array([0.0, -2.1e-4, 0.0, 1.3e-4, 0.05, 1.7e-4])),
]


def _boosted(el, boost):
    """The element's radiating packing with K_e and alpha multiplied by ``boost``: the radiation terms of
    J then stand out of its radiation-free part, so the differences test them, not just the kick."""
    packed = TO.pack_one(el, radiation="mean")
    f64 = packed.words.view(np.float64)
    f64[4] *= boost
    f64[6] *= boost
    return packed


@pytest.mark.parametrize("boost", [1.0, 1e5])
@pytest.mark.parametrize("case", CASES, ids=lambda c: c[0])
def test_oracle_jacobian_matches_finite_differences(case, boost):
    name, el, z = case
    packed = _boosted(el, boost)
    _, J, _, _, alive = TO.track(packed, z, P0C, ELECTRON)
    assert alive
    fd = TO.fd_jacobian(packed, z, P0C, ELECTRON)
    scale = np.maximum(np.max(np.abs(J), axis=0), 1e-300)
    err = np.max(np.abs(J - fd) / scale)
    assert err <= 1e-8, (name, err, J, fd)
    # the radiation part itself, against the differences of the map without radiation
    if boost > 1 and name != "quadrupole_on_axis":
        bare = TO.pack_one(el, radiation="mean")
        bare.words.view(np.float64)[4] = 0.0
        J0 = TO.track(bare, z, P0C, ELECTRON)[1]
        rad = J - J0
        assert np.max(np.abs(rad)) > 1e-4 * np.max(np.abs(J))
        fd0 = TO.fd_jacobian(bare, z, P0C, ELECTRON)
        err = np.max(np.abs(rad - (fd - fd0))) / np.max(np.abs(rad))
        assert err <= 1e-6, (name, err)


def test_on_axis_quadrupole_radiates_nothing():
    el = CASES[-1][1]
    z = CASES[-1][2]
    packed = TO.pack_one(el, radiation="mean")
    zz, J, S, lost, alive = TO.track(packed, z, P0C, ELECTRON)
    assert lost == 0.0 and not S.any()


@pytest.mark.parametrize("case", CASES[:4], ids=lambda c: c[0])
def test_diffusion_matches_difference_jacobians_and_vh(case):
    """D of one record = V_1 (J_2 K g_1)(J_2 K g_1)^T + V_2 g_2 g_2^T, rebuilt from central differences:
    g_h = dz_after/dW of a half is the difference of the map under a shift of the half's loss, taken
    here by a shift of K_e in that half alone (W is proportional to K_e)."""
    name, el, z = case
    packed = TO.pack_one(el, radiation="mean")
    words = np.ascontiguousarray(packed.words)
    b = TO.Particle(z, P0C, ELECTRON).beam
    J, D, lost, zout = TRO.rad_record(words, 0, z, b)
    f64 = words.view(np.float64)
    rec = (f64[2], f64[3], f64[4], f64[5], f64[6])
    # the two halves' losses and V_h from the record constants
    m2 = (b.energy0 - b.p0c) * (b.energy0 + b.p0c)
    gam0 = math.sqrt((1 + z[5]) ** 2 * P0C ** 2 + m2) / math.sqrt(m2)
    P = RO.field_kick(_P(z), dict(knl=list(el.knl), ksl=list(el.ksl)))
    fl = math.hypot(float(P[0][0]), float(P[1][0]))
    lh = 0.5 * (rec[0] + float(el.hxl) * z[0] - float(el.hyl) * z[2])
    kap = fl / rec[0] / (1 + z[5])
    v1 = (5 / (2 * math.sqrt(3))) * rec[4] * gam0 * kap * lh * (11 / 27) * (1.5 * rec[3] * gam0 ** 3 * kap) ** 2
    # differences: the map with an extra energy change eps in half h only
    g = []
    for half in (0, 1):
        def out(eps):
            return _map_with_kick(words, z, b, half, eps)
        h = 1e-6 * b.energy0  # a step of 1e-6 in delta: delta carries an absolute rounding of ~1e-16
        g.append((4 * (out(h / 2) - out(-h / 2)) / h - (out(h) - out(-h)) / (2 * h)) / 3)
    # the exit half's V_h at the state after the first half and the kick
    _, V1, _, _, z1 = TRO._half(b, z, rec, fl, lh, (0.0, 0.0), float(el.hxl), float(el.hyl))
    assert abs(V1 / v1 - 1) < 1e-12
    _, z2 = TRO._kick(words, 8, z1, b)
    _, V2, _, _, _ = TRO._half(b, z2, rec, fl, lh, (0.0, 0.0), float(el.hxl), float(el.hyl))
    Dfd = V1 * np.outer(g[0], g[0]) + V2 * np.outer(g[1], g[1])
    err = np.max(np.abs(D - Dfd)) / np.max(np.abs(D))
    assert err < 1e-8, (name, err)
    assert np.allclose(D, D.T, rtol=0, atol=1e-12 * np.max(np.abs(D)))


def _P(z):
    import types

    return types.SimpleNamespace(x=np.array([z[0]]), y=np.array([z[2]]))


def _map_with_kick(words, z, b, half, eps):
    """The record's map (the oracle's own state arithmetic) with the loss of half ``half`` changed by
    ``eps`` eV."""
    f64 = words.view(np.float64)
    rec = (f64[2], f64[3], f64[4], f64[5], f64[6])
    aux = (int(words[0]) >> 8) & 0xFF
    sub = 8
    tag = int(words[sub]) & 0xFF
    at = sub + 2 if tag == 4 else sub + 6
    pairs = f64[at: at + 2 * (aux + 1)].reshape(aux + 1, 2)
    hxl, hyl = (0.0, 0.0) if tag == 4 else (f64[sub + 1], f64[sub + 2])
    c = pairs[:, 0] + 1j * pairs[:, 1]
    P = sum(c[m] * complex(z[0], z[2]) ** (aux - m) for m in range(aux + 1))
    fl = abs(P)
    lh = 0.5 * (rec[0] + hxl * z[0] - hyl * z[2])

    def shifted_half(zz, extra):
        _, _, _, dE, _ = TRO._half(b, zz, rec, fl, lh, (0.0, 0.0), hxl, hyl)
        # the same half with the loss dE + extra: an energy change through the oracle's bookkeeping
        d = zz[5]
        rvv, ptaub0 = TRO._energy(b, d)
        ptau = (ptaub0 + (dE + extra) / b.energy0) / b.beta0
        dn = math.sqrt(ptau ** 2 + 2 * ptau / b.beta0 + 1) - 1
        rvvn = (1 + dn) / (1 + ptau * b.beta0)
        f = (1 + dn) / (1 + d)
        out = zz.copy()
        out[5], out[4], out[1], out[3] = dn, zz[4] * rvvn / rvv, zz[1] * f, zz[3] * f
        return out

    z1 = shifted_half(z, eps if half == 0 else 0.0)
    _, z2 = TRO._kick(words, sub, z1, b)
    return shifted_half(z2, eps if half == 1 else 0.0)


def test_vh_matches_the_photon_statistics_of_the_table():
    """V_h = nbar <x^2> u_c^2 is the variance of a compound Poisson sum: the table's second moment
    (midpoint rule in U over 2^20 cells, the tail past 1 - 2^-20 added from the cell average) equals
    the 11/27 the envelope uses."""
    n = 1 << 20
    u = (np.arange(n) + 0.5) / n
    x2 = float(np.mean(RO.synrad_x(u) ** 2))
    assert abs(x2 / TRO.X2_MEAN - 1) < 2e-3, x2
    # and the mean, for scale: 8/(15 sqrt 3)
    assert abs(float(np.mean(RO.synrad_x(u))) / (8 / (15 * math.sqrt(3))) - 1) < 1e-4


def test_oracle_record_matches_the_interpreter_state():
    for name, el, z in CASES:
        packed = TO.pack_one(el, radiation="mean")
        words = np.ascontiguousarray(packed.words)
        zout = TRO.rad_record(words, 0, z, TO.Particle(z, P0C, ELECTRON).beam)[3]
        ref, alive = TO.element_map(words, 0, z, P0C, ELECTRON)
        assert alive
        np.testing.assert_allclose(zout, ref, rtol=1e-13, atol=1e-19, err_msg=name)


def test_header_declares_the_new_entry_points():
    hdr = open(os.path.join(ROOT, "include", "xline_b200.h")).read()
    for name in ("xlb_track_tangent_radiation_device", "xlb_track_envelope_device"):
        assert re.search(r"int %s\(" % name, hdr), name
        assert name in _cabi.EXPORTS
    assert _cabi.ABI_VERSION == 4


def test_envelope_container():
    env = xl.Envelope(3, device="cpu")
    assert env.cov.shape == (3, 6, 6) and not env.cov.any()
    assert env.energy_loss.shape == (3,) and not env.energy_loss.any()
    assert len(env) == 3


def test_refusals_without_gpu():
    line = xl.Line([xl.Multipole(knl=[0.02], hxl=0.02, length=1.0), xl.Drift(length=1.0)])
    line.radiation = "mean"
    p = xl.Particles(p0c=P0C, mass0=ELECTRON, x=np.zeros(1))
    if p.x.device.type != "cuda":
        with pytest.raises(RuntimeError, match="CUDA"):
            line.track_envelope(p, xl.Envelope(1, device="cpu"))
    with pytest.raises(ValueError, match="4d"):
        xl.closed_orbit(line, p, mode="4d", radiation=True)
    # the default mode is 6d on a radiating line, which needs an RF voltage
    with pytest.raises(ValueError, match="6d closed orbit needs an RF"):
        xl.closed_orbit(line, p, radiation=True)
    with pytest.raises(ValueError, match="RF"):
        xl.radiation_equilibrium(line, p)
    line.radiation = None
    with pytest.raises(ValueError, match="does not radiate"):
        xl.radiation_equilibrium(line, p)
