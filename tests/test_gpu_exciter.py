"""Exciter on the GPU: the sample every particle reads against the oracle, exciter lines against the
oracle in every kernel family that carries the case, bitwise determinism, and the physics of an AC
dipole and of quadrupole ripple."""
import math

import numpy as np
import pytest
import torch
from scipy.constants import c as clight

import xline_b200 as xl
from tests import exciter_oracle as EO
from tests import helpers as H
from xline_b200 import configs

pytestmark = pytest.mark.gpu

COLUMNS = H.COORDS + ("rpp", "rvv", "s", "state", "at_element", "at_turn")
P0C, M0 = 450e9, 938.27208816e6


def _beta0(p0c=P0C, m0=M0):
    return p0c / math.sqrt(p0c * p0c + m0 * m0)


def _track(line, cols, num_turns=1, p0c=P0C, m0=M0, **kw):
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)
    line.track(p, num_turns=num_turns, **kw)
    torch.cuda.synchronize()
    return p.to_numpy()


def _bitwise(a, b, keys=COLUMNS):
    for k in keys:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k]), equal_nan=True), k


def _like_oracle(got, ref, tol):
    for k in ("state", "at_element", "at_turn"):
        assert np.array_equal(got[k], ref[k]), k
    for k in H.COORDS:
        assert H.scaled_err(got[k], ref[k]) <= tol, (k, H.scaled_err(got[k], ref[k]))


# ---------------------------------------------------------------- 1. the sample index, particle by particle
@pytest.mark.parametrize("ppt", [1, 2, 3, 4])
@pytest.mark.parametrize("h", [1.0, 3.0, 35640.0])
def test_each_particle_reads_the_oracles_sample(h, ppt):
    """Samples 2^0 .. 2^39 and knl = [k0]: px after the element is -k0 * s exactly, so it names the sample.
    zeta spread over several samples (and at half-sample boundaries, one ulp either side), turns before
    start_turn and past the last sample, NaN and infinite zeta."""
    frev = 11245.5
    ex = xl.Exciter(knl=[1e-6], samples=[2.0 ** k for k in range(40)], sampling_frequency=h * frev, frev=frev,
                    start_turn=5)
    rng = np.random.default_rng(int(h) + ppt)
    n = 8191
    beta0 = _beta0()
    at_turn = rng.integers(0, 60, n) if h == 1.0 else rng.integers(0, 8, n)
    a, b = h, h * frev / clight
    k = rng.integers(-3, 43, n).astype(np.float64)
    zeta = ((at_turn - 5) * a - (k - 0.5)) * beta0 / b
    zeta[: n // 3] = np.nextafter(zeta[: n // 3], rng.choice([-np.inf, np.inf], n // 3))
    zeta[n // 3: 2 * n // 3] += rng.uniform(-0.5, 0.5, 2 * n // 3 - n // 3) * beta0 / b
    zeta[:6] = [np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-310]
    cols = dict(zeta=zeta, at_turn=at_turn, x=rng.normal(0, 1e-3, n), y=rng.normal(0, 1e-3, n))
    got = _track(xl.Line([ex]), cols, 1, particles_per_thread=ppt)
    idx = EO.sample_index(ex.to_dict(), at_turn, zeta, beta0)
    want_s = EO.sample_values(ex.to_dict(), idx)
    assert np.array_equal(-got["px"] / 1e-6, want_s)
    assert np.all(got["py"] == 0.0)
    assert (idx < 0).sum() > 100 and len(np.unique(idx)) > 20
    assert np.array_equal(got["at_turn"], at_turn + 1)
    ref = EO.run_oracle(xl.Line([ex]).to_specs(), cols, P0C, M0)
    _like_oracle(got, ref, 0.0)


def test_higher_order_kick_agrees_with_the_oracle():
    ex = xl.Exciter(knl=[1e-5, 2e-3, -0.4, 30.0], ksl=[0, 1e-3, 0.2], samples=np.linspace(-1, 1, 9),
                    sampling_frequency=2 * 11245.5, frev=11245.5)
    rng = np.random.default_rng(3)
    n = 4099
    cols = dict(x=rng.normal(0, 2e-3, n), y=rng.normal(0, 2e-3, n), px=rng.normal(0, 1e-5, n),
                py=rng.normal(0, 1e-5, n), zeta=rng.uniform(-5e4, 5e4, n), at_turn=rng.integers(0, 6, n))
    got = _track(xl.Line([ex]), cols)
    ref = EO.run_oracle(xl.Line([ex]).to_specs(), cols, P0C, M0)
    for k in ("px", "py"):
        assert H.floor_rel_err(got[k], ref[k]) <= 1e-12, k


# ---------------------------------------------------------------- 2. lines
def _ac(frev, n, q, amp=1e-6, order=0, plane="x"):
    s = amp * np.cos(2 * np.pi * q * np.arange(n))
    knl, ksl = ([0.0] * order + [1.0], [0.0]) if plane == "x" else ([0.0], [1.0])
    return xl.Exciter(knl=knl, ksl=ksl, samples=s, sampling_frequency=frev, frev=frev)


def _with_exciters(line, every, make):
    els, names = [], []
    for i, (el, nm) in enumerate(zip(line.elements, line.element_names)):
        els.append(el)
        names.append(nm)
        if i % every == every // 2:
            els.append(make(i))
            names.append("exc%d" % i)
    return xl.Line(els, names)


def _frev(line, p0c=P0C, m0=M0):
    return _beta0(p0c, m0) * clight / line.get_length()


def test_fodo_with_exciters_200_turns():
    line, cols, p0c, m0 = configs.config_fodo(1000)
    f = _frev(line, p0c, m0)
    rng = np.random.default_rng(11)
    ln = _with_exciters(line, max(2, len(line.elements) // 4),
                        lambda i: xl.Exciter(knl=[rng.normal(0, 1e-5), rng.normal(0, 1e-3)], ksl=[0, 1e-4],
                                             samples=rng.normal(0, 1, 150), sampling_frequency=f * 2.5, frev=f,
                                             start_turn=int(rng.integers(0, 40))))
    assert ln.pack().record_counts.get(0x40, 0) >= 3
    got = _track(ln, cols, 200, p0c, m0)
    ref = EO.run_oracle(ln.to_specs(), cols, p0c, m0, num_turns=200)
    _like_oracle(got, ref, 1e-10)


@pytest.mark.parametrize("config", ["c2", "c3_no_6d", "c5"])
def test_exciter_lines_in_the_lhc_and_beam_field_families(config):
    """LHC with apertures (thin-lens family), LHC with the 4D lenses of C3 (beam-field family) and the
    PS Booster with space charge, each with exciters at several positions, against the oracle."""
    n = 1000
    if config == "c2":
        line, cols, p0c, m0 = configs.config_lhc(n)
        turns = 3
    elif config == "c3_no_6d":
        full, cols, p0c, m0 = configs.config_lhc_beambeam(n)
        keep = [i for i, e in enumerate(full.elements) if type(e).__name__ != "BeamBeam6D"]
        line = xl.Line([full.elements[i] for i in keep], [full.element_names[i] for i in keep])
        turns = 3
    else:
        line, cols, p0c, m0 = configs.config_psb(n)
        turns = 20
    f = _frev(line, p0c, m0)
    rng = np.random.default_rng(len(config))
    ln = _with_exciters(line, max(2, len(line.elements) // 5),
                        lambda i: xl.Exciter(knl=[rng.normal(0, 1e-7), rng.normal(0, 1e-5)], ksl=[1e-8],
                                             samples=rng.normal(0, 1, 64), sampling_frequency=f, frev=f))
    got = _track(ln, cols, turns, p0c, m0)
    ref = EO.run_oracle(ln.to_specs(), cols, p0c, m0, num_turns=turns)
    _like_oracle(got, ref, 3e-11 * turns)


def test_radiating_ring_with_an_exciter_runs_the_radiation_twin():
    line, _, p0c, m0 = configs.config_petra_like(1)
    f = _frev(line, p0c, m0)
    ln = xl.Line(list(line.elements) + [_ac(f, 64, 0.27, amp=1e-5)], list(line.element_names) + ["ac"])
    ln.radiation = "mean"
    rng = np.random.default_rng(8)
    n = 500
    cols = dict(x=rng.normal(0, 2e-5, n), px=rng.normal(0, 2e-6, n), y=rng.normal(0, 1e-5, n),
                py=rng.normal(0, 1e-6, n), zeta=rng.normal(0, 1e-3, n), delta=rng.normal(0, 1e-4, n))
    got = _track(ln, cols, 5, p0c, m0)
    alive = got["state"] == 1
    assert alive.all()
    ref = EO.run_oracle(ln.to_specs(), cols, p0c, m0, num_turns=5, radiation="mean")
    _like_oracle(got, ref, 1e-10)
    off = xl.Line(list(line.elements), list(line.element_names))
    off.radiation = "mean"
    assert np.max(np.abs(_track(off, cols, 5, p0c, m0)["px"] - got["px"])[alive]) > 1e-7


def test_element_by_element_paths():
    line, cols, p0c, m0 = configs.config_fodo(300)
    f = _frev(line, p0c, m0)
    ln = _with_exciters(line, 3, lambda i: xl.Exciter(knl=[1e-6, 1e-4], samples=[1.0, -2.0, 0.5],
                                                       sampling_frequency=f, frev=f))
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)
    tr = ln.trace_elem_by_elem(p).cpu().numpy()
    p2 = xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)
    outs = ln.track_elem_by_elem(p2)
    ref = EO.run_oracle(ln.to_specs(), cols, p0c, m0)
    for f, k in enumerate(H.COORDS):
        assert H.scaled_err(tr[-1, f], ref[k]) <= 1e-12, k
        assert H.scaled_err(outs[-1].to_numpy()[k], ref[k]) <= 1e-12, k
    assert np.all(outs[-1].to_numpy()["at_turn"] == 0)  # el.track never counts turns


# ---------------------------------------------------------------- 3. determinism
def _det_case():
    line, cols, p0c, m0 = configs.config_fodo(20000)
    f = _frev(line, p0c, m0)
    rng = np.random.default_rng(5)
    ln = _with_exciters(line, 4, lambda i: xl.Exciter(knl=[rng.normal(0, 1e-5), 1e-3], samples=rng.normal(0, 1, 97),
                                                       sampling_frequency=f * 1.5, frev=f, start_turn=2))
    ln.append_element(xl.LimitEllipse(a=2.5e-3, b=2.5e-3), "aperture")  # losses: compaction has work to do
    return ln, cols, p0c, m0


def test_results_do_not_depend_on_the_launch_shape_or_the_batch():
    """Bit for bit; s is left out: its sum follows the launches (include/xline_b200.h, path length)."""
    ln, cols, p0c, m0 = _det_case()
    keys = tuple(k for k in COLUMNS if k != "s")
    base = _track(ln, cols, 24, p0c, m0)
    assert 0 < (base["state"] == 0).sum() < len(base["x"])
    for kw in (dict(particles_per_thread=1), dict(particles_per_thread=2, threads_per_block=256),
               dict(particles_per_thread=3), dict(particles_per_thread=4), dict(turns_per_launch=5),
               dict(turns_per_launch=1, compact_threshold=1e-6), dict(turns_per_item=3),
               dict(turns_per_item=-1)):
        _bitwise(_track(ln, cols, 24, p0c, m0, **kw), base, keys)
    sub = slice(5000, 7001)
    part = _track(ln, {k: np.asarray(v)[sub] for k, v in cols.items()}, 24, p0c, m0)
    _bitwise(part, {k: v[sub] for k, v in base.items()}, keys)
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)
    ln.track(p, num_turns=9)
    ln.track(p, num_turns=15)
    _bitwise(p.to_numpy(), base, keys)


# ---------------------------------------------------------------- 4. physics
def _fodo_tunes(line, p0c, m0):
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=[0.0])
    co = xl.closed_orbit(line, p, mode="4d")
    m = co.matrix
    qx = math.acos(0.5 * (m[0, 0] + m[1, 1])) / (2 * math.pi)
    if m[0, 1] < 0:
        qx = 1 - qx
    return qx, m


def test_ac_dipole_drives_at_its_tune_with_the_steady_state_amplitude():
    base, _, p0c, m0 = configs.config_fodo(1)
    qx, M = _fodo_tunes(base, p0c, m0)
    qd = qx + 0.01
    ramp, flat = 2000, 3000
    n = ramp + flat
    k0 = 1e-7
    env = np.minimum(np.arange(n) / ramp, 1.0)
    env = 0.5 - 0.5 * np.cos(np.pi * env)  # smooth ramp, then held
    f = _frev(base, p0c, m0)
    ex = xl.Exciter(knl=[k0], samples=env * np.cos(2 * np.pi * qd * np.arange(n)), sampling_frequency=f, frev=f)
    mon = xl.BeamMonitor(num_stores=2048, start=ramp + 500, skip=1, min_particle_id=0, max_particle_id=0)
    line = xl.Line([mon] + list(base.elements) + [ex])
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=[0.0], px=[0.0], zeta=[0.0])
    line.track(p, num_turns=ramp + 500 + 2048)
    assert int(p.state[0]) == 1
    res = xl.monitor_tunes(mon)
    assert abs(float(res["qx"][0, 0]) - qd) <= 1e-6, (float(res["qx"][0, 0]), qd)
    # exact steady state of z_(n+1) = M z_n + b cos(2 pi qd n), the kick at the end of the turn
    b = np.zeros(6)
    b[1] = -k0
    z = np.linalg.solve(np.exp(2j * np.pi * qd) * np.eye(6) - M, b)
    x = mon.data["x"][:, 0].cpu().numpy()
    amp = math.sqrt(2 * np.mean(x * x))
    assert abs(amp / abs(z[0]) - 1) <= 0.02, (amp, abs(z[0]))


def test_quadrupole_ripple_gives_sidebands_at_the_ripple_frequency():
    base, _, p0c, m0 = configs.config_fodo(1)
    qx, _ = _fodo_tunes(base, p0c, m0)
    fr = 0.0371  # ripple frequency / frev
    n = 4096
    f = _frev(base, p0c, m0)
    ripple = xl.Exciter(knl=[0.0, 2e-3], samples=np.sin(2 * np.pi * fr * np.arange(n)), sampling_frequency=f, frev=f)
    mon = xl.BeamMonitor(num_stores=n, start=0, skip=1, min_particle_id=0, max_particle_id=0)
    line = xl.Line([mon] + list(base.elements) + [ripple])
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=[1e-4])
    line.track(p, num_turns=n)
    x = mon.data["x"][:, 0].cpu().numpy()
    q0, _ = xl.naff(torch.tensor(x[:, None], device="cuda"))
    q0 = float(q0[0])
    assert abs(q0 - qx) < 1e-3
    t = np.arange(n)
    basis = np.stack([np.cos(2 * np.pi * q0 * t), np.sin(2 * np.pi * q0 * t)], axis=1)
    resid = x - basis @ np.linalg.lstsq(basis, x, rcond=None)[0]
    q1, a1 = xl.naff(torch.tensor(resid[:, None], device="cuda"))
    q1 = float(q1[0])
    assert min(abs(q1 - (q0 + fr)), abs(q1 - (q0 - fr))) < 2e-4, (q0, q1, fr)
    assert float(a1[0]) > 1e-3 * float(np.max(np.abs(x)))
    # without the ripple there is no such line
    plain = xl.Line([mon] + list(base.elements))
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=[1e-4])
    plain.track(p, num_turns=n)
    y = mon.data["x"][:, 0].cpu().numpy()
    r2 = y - basis @ np.linalg.lstsq(basis, y, rcond=None)[0]
    hann = 1 - np.cos(2 * np.pi * t / n)

    def line_at(r, q):
        return abs(np.sum(hann * r * np.exp(-2j * np.pi * q * t))) / np.sum(hann)

    assert line_at(r2, q1) < 0.02 * line_at(resid, q1)
