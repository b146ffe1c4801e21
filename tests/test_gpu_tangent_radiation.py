"""Radiation in the tangent map on the GPU (tangent_kernel_radiation, envelope_kernel; DESIGN.md
§4.10): Jacobians and envelopes against the NumPy oracle, coordinates against ``Line.track``, the
damped closed orbit against long mean-mode tracking, damping times, partition numbers and the
equilibrium against the radiation integrals and quantum tracking, bitwise reproducibility, the
refusals and the ptxas properties of both twins."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

import xline_b200 as xl
from tests import tangent_oracle as TO
from tests.test_gpu_radiation import _damping_ring, _planes, _ring
from xline_b200 import build, configs, lattice, optics, tangent

pytestmark = pytest.mark.gpu

ELECTRON = configs.ELECTRON_MASS_EV
P0C = 6e9
COORDS = ("x", "px", "y", "py", "zeta", "delta")
Z0 = np.array([[4e-4, -3e-5, -2e-4, 2e-5, 1e-3, 5e-4], [-6e-4, 4e-5, 3e-4, -1e-5, -2e-3, -8e-4],
               [1e-4, 1e-5, 1e-4, 1e-5, 0.0, 1e-4]])


def _particles(z, **kw):
    z = np.atleast_2d(z)
    return xl.Particles(p0c=P0C, mass0=ELECTRON, device="cuda", **{k: z[:, i].copy() for i, k in enumerate(COORDS)},
                        **kw)


def _line(els, mode="mean"):
    line = xl.Line(els)
    line.radiation = mode
    return line


def _z(p):
    d = p.to_numpy()
    return np.stack([d[k] for k in COORDS], axis=1)


def _jac_err(J, ref):
    scale = np.maximum(np.max(np.abs(ref), axis=0), 1e-300)
    return float(np.max(np.abs(J - ref) / scale))


def _spd(rng, scale):
    a = rng.normal(size=(6, 6)) * scale[:, None]
    return a @ a.T + np.diag(scale ** 2)


@pytest.mark.parametrize("which", ["elements", "turn"])
def test_jacobian_against_oracle_and_coordinates_against_track(which):
    els = _ring(1)
    lines = [[el] for el in els] if which == "elements" else [els]
    worst_j = worst_z = 0.0
    for part in lines:
        line = _line(part)
        p = _particles(Z0)
        t = xl.TangentMap(len(Z0), device="cuda")
        line.track_tangent(p, t, radiation=True)
        q = _particles(Z0)
        line.track(q)
        got, ref = _z(p), _z(q)
        scale = np.maximum(np.sqrt(np.mean(ref ** 2, axis=0)), 1e-30)
        worst_z = max(worst_z, float(np.max(np.abs(got - ref) / scale)))
        packed, _ = line._tangent_lattice(torch.device("cuda", torch.cuda.current_device()), radiation=True)
        for i, z in enumerate(Z0):
            zz, J, _, _, alive = TO.track(packed, z, P0C, ELECTRON)
            assert alive
            worst_j = max(worst_j, _jac_err(t.matrix()[i].cpu().numpy(), J))
    print("tangent with radiation (%s): J vs oracle %.3g, z vs Line.track %.3g" % (which, worst_j, worst_z))
    # measured on a B200: 1.2e-15 and 0 (the coordinates are bit for bit those of Line.track)
    assert worst_j < 2.5e-15
    assert worst_z < 1e-15


def test_envelope_without_radiation_is_j_sigma_jt():
    rng = np.random.default_rng(11)
    line = xl.Line(_ring(2))
    n = 5
    z = Z0[rng.integers(0, 3, n)] * rng.uniform(0.5, 1.5, (n, 1))
    s0 = np.stack([_spd(rng, np.array([1e-4, 1e-5, 1e-4, 1e-5, 1e-3, 1e-4])) for _ in range(n)])
    env = xl.Envelope(n, device="cuda")
    env.cov.copy_(torch.from_numpy(s0))
    p = _particles(z)
    line.track_envelope(p, env, num_turns=3)
    q = _particles(z)
    t = xl.TangentMap(n, device="cuda")
    line.track_tangent(q, t, num_turns=3)
    J = t.matrix().cpu().numpy()
    want = np.einsum("nij,njk,nlk->nil", J, s0, J)
    got = env.cov.cpu().numpy()
    err = np.max(np.abs(got - want)) / np.max(np.abs(want))
    print("envelope without radiation vs J S0 J^T: %.3g" % err)
    assert err < 2e-15  # measured 9.1e-16
    assert np.array_equal(got, np.transpose(got, (0, 2, 1)))
    assert not env.energy_loss.any()
    for k in COORDS:
        assert torch.equal(getattr(p, k), getattr(q, k))


def test_envelope_on_the_radiating_ring_against_oracle():
    rng = np.random.default_rng(12)
    line = _line(_ring(1))
    s0 = _spd(rng, np.array([1e-4, 1e-5, 1e-4, 1e-5, 1e-3, 1e-4]))
    env = xl.Envelope(len(Z0), device="cuda")
    env.cov.copy_(torch.from_numpy(np.stack([s0] * len(Z0))))
    line.track_envelope(_particles(Z0), env)
    packed, _ = line._tangent_lattice(torch.device("cuda", torch.cuda.current_device()), radiation=True)
    worst_s = worst_d = worst_u = 0.0
    for i, z in enumerate(Z0):
        _, J, S, lost, _ = TO.track(packed, z, P0C, ELECTRON, cov=s0)
        got = env.cov[i].cpu().numpy()
        worst_s = max(worst_s, float(np.max(np.abs(got - S)) / np.max(np.abs(S))))
        worst_u = max(worst_u, abs(float(env.energy_loss[i]) / lost - 1))
    # the diffusion alone, from Sigma = 0
    env0 = xl.Envelope(len(Z0), device="cuda")
    line.track_envelope(_particles(Z0), env0)
    for i, z in enumerate(Z0):
        D = TO.track(packed, z, P0C, ELECTRON)[2]
        worst_d = max(worst_d, float(np.max(np.abs(env0.cov[i].cpu().numpy() - D)) / np.max(np.abs(D))))
    print("envelope vs oracle: Sigma %.3g, D %.3g, energy loss %.3g" % (worst_s, worst_d, worst_u))
    # measured on a B200: 2.2e-15, 7.1e-16, 2.2e-16
    assert worst_s < 5e-15 and worst_d < 1.5e-15 and worst_u < 5e-16


def _equilibrium(line, p0c, m0):
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=np.zeros(1))
    return xl.radiation_equilibrium(line, p)


def test_damping_ring_equilibrium():
    """The damped orbit, damping times, partition numbers and equilibrium of the damping ring against the
    radiation integrals, against the oracle and against long mean-mode tracking.  The oracle's check is
    on its analytic one-turn Jacobian (the eigenvalues of M), not on one-turn differences of the tracked
    map: such differences are unreliable for tau_z (delta steps of 1e-10 and 1e-8 give damping times
    16x apart on C4), while the oracle's per-record Jacobians are themselves checked against
    Richardson-extrapolated differences record by record in tests/test_tangent_radiation.py."""
    line, p0c, m0 = _damping_ring()
    line.radiation = "mean"
    r = optics.radiation_integrals(line, p0c, m0)
    eq = _equilibrium(line, p0c, m0)
    tau_int = np.array([r["tau_x"], r["tau_y"], r["tau_z"]])
    robinson = float(eq.partition.sum())
    print("damping ring: orbit %s, %d iterations; tau %s (integrals %s); J %s (sum %.6f); U %.6g (U0 %.6g); "
          "eps %s; sigma_delta %.5g (integrals %.5g), eps_x integrals %.5g"
          % (eq.orbit.tolist(), eq.iterations, eq.damping_times.tolist(), tau_int.tolist(), eq.partition.tolist(),
             robinson, eq.energy_loss, r["U0"], eq.emittances.tolist(), eq.sigma_delta, r["sigma_delta"], r["eps_x"]))
    assert eq.iterations < 30
    # measured on a B200: tau 0.99 %, 6.1e-5, 0.25 % from the integrals (first order in the orbit and
    # uncoupled: the 6.5e-4 delta of the damped orbit moves tau_x); Robinson's sum 4 + 3.4e-5
    rel = np.abs(eq.damping_times / tau_int - 1)
    assert rel[0] < 0.02 and rel[1] < 1.2e-4 and rel[2] < 5e-3, rel
    assert abs(robinson - 4) < 7e-5
    # the oracle's one-turn matrix on the GPU's orbit: the same eigenvalues
    packed, _ = line._tangent_lattice(torch.device("cuda", torch.cuda.current_device()), radiation=True)
    zz, J, D, U, alive = TO.track(packed, eq.orbit, p0c, m0)
    assert alive
    assert np.max(np.abs(zz - eq.orbit)) < 1e-12
    lam, _ = tangent._symplectic_modes(J)
    tau_o = np.sort(-1 / np.log(np.abs(lam)))
    print("damping times vs the oracle's one-turn matrix: %.3g" % np.max(np.abs(np.sort(eq.damping_times) / tau_o - 1)))
    assert np.max(np.abs(np.sort(eq.damping_times) / tau_o - 1)) < 1.5e-11  # measured 6.0e-12
    assert np.max(np.abs(D - eq.diffusion)) < 1e-10 * np.max(np.abs(D))
    # emittance and energy spread against the integrals
    # measured on a B200: 1.9 % and 1.2 % above the integrals
    assert abs(eq.emittances[0] / r["eps_x"] - 1) < 0.04, (eq.emittances[0], r["eps_x"])
    assert abs(eq.sigma_delta / r["sigma_delta"] - 1) < 0.024, (eq.sigma_delta, r["sigma_delta"])
    # the orbit a mean-mode particle settles on after 15 tau_x: the offset decays as e^-15 = 3e-7
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", x=[1e-4], delta=[1e-4])
    turns = int(15 * eq.damping_times.max())
    line.track(p, num_turns=turns)
    z = _z(p)[0]
    err = np.abs(z - eq.orbit)
    # the start's offset from the orbit in the modes of M: every mode has decayed by e^-15 or more, so
    # coordinate i is off by at most e^-15 sum_k |a_k v_k,i + conj(a_k v_k,i)| (twice that allowed)
    lam, V = tangent._symplectic_modes(eq.matrix)
    a = np.linalg.solve(V, np.array([1e-4, 0, 0, 0, 0, 1e-4]) - eq.orbit)
    amp = sum(2 * np.abs(V[:, 2 * k] * a[2 * k]) for k in range(3))
    bound = 2 * math.exp(-15) * amp + 1e-12
    print("orbit after %d turns of tracking - damped orbit: %s (bound %s)" % (turns, err.tolist(), bound.tolist()))
    assert np.all(err < bound), (err, bound)


def test_damping_ring_equilibrium_against_quantum_tracking():
    """4096 particles from zero emittance over 5 tau_x in quantum mode (as the radiation tests run it):
    the envelope's eps_x and sigma_delta within 4 sigma of that run's statistics plus 1 %."""
    line, p0c, m0 = _damping_ring()
    line.radiation = "quantum"
    line.radiation_seed = 2024
    eq = _equilibrium(line, p0c, m0)
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
    print("quantum tracking eps_x %.5g sigma_delta %.5g; envelope eps_x %.5g sigma_delta %.5g"
          % (ex_eq, sd_eq, eq.emittances[0], eq.sigma_delta))
    assert abs(eq.emittances[0] / ex_eq - 1) < 4 * 0.013 + 0.01
    assert abs(eq.sigma_delta / sd_eq - 1) < 4 * 0.004 + 0.01


def test_petra4_equilibrium():
    line, _, p0c, m0 = configs.config_petra4(n=1)
    line.radiation = "mean"
    r = optics.radiation_integrals(line, p0c, m0)
    eq = _equilibrium(line, p0c, m0)
    tau_int = np.array([r["tau_x"], r["tau_y"], r["tau_z"]])
    print("PETRA IV: orbit %s, %d iterations; tau %s (integrals %s); sum J %.6f; eps %s (eps_x integrals %.4g); "
          "sigma_delta %.4g (integrals %.4g)"
          % (eq.orbit.tolist(), eq.iterations, eq.damping_times.tolist(), tau_int.tolist(), eq.partition.sum(),
             eq.emittances.tolist(), r["eps_x"], eq.sigma_delta, r["sigma_delta"]))
    assert eq.iterations < 30
    # measured on a B200: 8.1e-7 and 4 + 1.8e-6
    assert np.max(np.abs(eq.damping_times / tau_int - 1)) < 2e-6
    assert abs(eq.partition.sum() - 4) < 4e-6


@pytest.mark.parametrize("twin", ["tangent", "envelope"])
def test_bitwise_reproducibility(twin):
    rng = np.random.default_rng(13)
    n = 300
    line = _line(_ring(2))
    z = np.stack([rng.normal(0, s, n) for s in (3e-3, 3e-4, 2e-3, 2e-4, 2e-3, 1e-3)], axis=1)
    z[:, 0] *= np.where(rng.uniform(size=n) < 0.2, 8.0, 1.0)  # some particles hit the aperture

    def run(zz, turns_list, threads=0):
        p = _particles(zz)
        if twin == "tangent":
            c = xl.TangentMap(len(zz), device="cuda")
            for tt in turns_list:
                line.track_tangent(p, c, num_turns=tt, threads_per_block=threads, radiation=True)
            out = [c.jacobian, c.log2_scale, c.fli]
        else:
            c = xl.Envelope(len(zz), device="cuda")
            for tt in turns_list:
                line.track_envelope(p, c, num_turns=tt, threads_per_block=threads)
            out = [c.cov, c.energy_loss]
        d = p.to_numpy()
        return [o.cpu().numpy() for o in out] + [d[k] for k in COORDS + ("state", "at_turn", "at_element")]

    ref = run(z, [20])
    assert 0 < (ref[-3] == 0).sum() < n
    for got in (run(z, [20], threads=256), run(z, [20], threads=32), run(z, [7, 13])):
        for a, b in zip(got, ref):
            np.testing.assert_array_equal(a, b)
    perm = rng.permutation(n)
    got = run(z[perm], [20])
    for a, b in zip(got, ref):
        np.testing.assert_array_equal(a, b[perm])
    j = int(np.flatnonzero(ref[-3] == 1)[0])
    alone = run(z[j:j + 1], [20])
    for a, b in zip(alone, ref):
        np.testing.assert_array_equal(a[0], b[j])


def test_radiation_true_without_radiation_is_the_existing_path():
    """On a line without radiation: ``radiation=True`` takes the existing path, and the radiation twin
    itself, run on the same lattice (no radiating records), gives the existing kernel's results bit for
    bit (include/xline_b200.h)."""
    line = xl.Line(_ring(2))
    z = np.concatenate([Z0, Z0[:1] * 40.0])  # the last particle is lost at the aperture

    def twin(lib, lat, cp, opts, stream, t):
        return lib.xlb_track_tangent_radiation_device(
            C.byref(lat), C.byref(cp), C.byref(opts), C.c_void_p(t.jacobian.data_ptr()),
            C.c_void_p(t.log2_scale.data_ptr()), C.c_void_p(t.fli.data_ptr()), stream)

    out = []
    for how in ("existing", "radiation=True", "twin"):
        p = _particles(z)
        t = xl.TangentMap(len(z), device="cuda")
        if how == "twin":
            tangent._launch(line, p, 5, 0, False, lambda *a: twin(*a, t))
        else:
            line.track_tangent(p, t, num_turns=5, radiation=how != "existing")
        d = p.to_numpy()
        out.append([t.jacobian.cpu().numpy(), t.log2_scale.cpu().numpy(), t.fli.cpu().numpy()]
                   + [d[k] for k in COORDS + ("state", "at_turn", "at_element")])
    assert out[0][-3][-1] == 0 and (out[0][-3][:-1] == 1).all()
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert np.array_equal(a, b)


def test_refusals():
    line = _line(_ring(1), "quantum")
    p = _particles(Z0)
    t = xl.TangentMap(len(Z0), device="cuda")
    with pytest.raises(ValueError, match="radiation"):
        line.track_tangent(p, t)
    with pytest.raises(ValueError, match="quantum"):
        line.track_tangent(p, t, radiation=True)
    with pytest.raises(ValueError, match="radiation"):
        xl.closed_orbit(line, p)
    line.radiation = "mean"
    with pytest.raises(ValueError, match="radiation"):
        line.track_tangent(p, t)
    with pytest.raises(ValueError, match="4d"):
        xl.closed_orbit(line, p, mode="4d", radiation=True)
    with pytest.raises(ValueError, match="one species"):
        q = _particles(Z0, chi=np.array([1.0, 0.5, 1.0]))
        line.track_tangent(q, xl.TangentMap(3, device="cuda"), radiation=True)
    # the C entry point refuses a quantum-mode record, naming the element
    els = _ring(1)
    packed = lattice.pack_line(els, strict=False, fuse=False, merge=False, split_lenses=False, drop_noops=False,
                               radiation="quantum")
    words = torch.from_numpy(packed.words.view(np.int64)).to("cuda")
    line._tangent_lattice = lambda dev, radiation=False: (packed, words)
    first = next(i for i, el in enumerate(els) if lattice.radiates(el, "quantum"))
    with pytest.raises(ValueError, match="element %d radiates in quantum mode" % first):
        tangent._tangent_call(line, p, t, 1, 0, True)
    with pytest.raises(ValueError, match="element %d radiates in quantum mode" % first):
        tangent.track_envelope(line, p, xl.Envelope(3, device="cuda"))
    # the tangent entry point without radiation still refuses the radiating lattice
    with pytest.raises(ValueError, match="radiating multipoles are not in the tangent map"):
        tangent._tangent_call(line, p, t, 1, 0, False)


def test_ptxas_both_twins():
    txt = build.ptxas_report().get("tangent")
    assert txt, "no ptxas report for the tangent unit"
    for k in ("24tangent_kernel_radiation", "15envelope_kernel"):
        m = re.search(r"Function properties for _ZN3xlb7tangent%s\S*\n\s*(\d+) bytes stack frame, "
                      r"(\d+) bytes spill stores, (\d+) bytes spill loads" % k, txt)
        assert m and m.groups() == ("0", "0", "0"), (k, txt)
    assert os.path.exists(os.path.join(build.OBJ, "tangent.o"))
