"""Tangent map on the GPU (Line.track_tangent, xl.closed_orbit): Jacobians against the NumPy
tangent oracle and against central differences of Line.track itself, the tracked orbit against
Line.track, linear optics, symplecticity, the FLI, closed orbits, determinism, refusals and the
kernel's build artefacts."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

import xline_b200 as xl
from tests import tangent_oracle as TO
from xline_b200 import _cabi, configs, optics

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
COORDS = TO.COORDS


def _beam(cols, p0c, m0):
    return xl.Particles(p0c=p0c, mass0=m0, device=DEV, **{k: np.asarray(v, dtype=float) for k, v in cols.items()})


def _z_cols(z):
    z = np.atleast_2d(np.asarray(z, dtype=float))
    return {k: z[:, i] for i, k in enumerate(COORDS)}


def _tangent(line, z, p0c, m0, turns=1):
    p = _beam(_z_cols(z), p0c, m0)
    t = xl.TangentMap(len(p), DEV)
    line.track_tangent(p, t, num_turns=turns)
    torch.cuda.synchronize()
    return p, t


def _coords(p):
    return np.stack([getattr(p, k).cpu().numpy() for k in COORDS], axis=1)


@pytest.mark.parametrize("case", TO.element_cases(), ids=lambda c: c[0])
def test_element_jacobian_matches_oracle_and_track(case):
    name, el, p0c, z = case
    line = xl.Line([el])
    p, t = _tangent(line, z, p0c, TO.MASS0)
    J = t.matrix()[0].cpu().numpy()
    ref = TO.oracle_jacobian(el, z, p0c)
    scale = np.maximum(np.max(np.abs(ref), axis=0), 1e-300)
    assert np.max(np.abs(J - ref) / scale) <= 1e-11, (name, J, ref)
    q = _beam(_z_cols(z), p0c, TO.MASS0)
    xl.Line([el]).track(q)
    a, b = _coords(p)[0], _coords(q)[0]
    assert np.all(np.abs(a - b) <= 1e-12 * np.maximum(np.abs(b), 1e-3 * np.abs(b).max())), (name, a, b)


def _lattice(name):
    if name == "fodo":
        line, cols, p0c, m0 = configs.config_fodo(1)
    elif name == "lhc":
        line, cols, p0c, m0 = configs.config_lhc(1, apertures=False)
    elif name == "petra4":
        line, cols, p0c, m0 = configs.config_petra4(1)
    elif name == "psb":
        line, cols, p0c, m0 = configs.config_psb(1, n_sc=16)
    else:  # C3 without its 6D lenses
        line, cols, p0c, m0 = configs.config_lhc_beambeam(1)
        line = xl.Line([e for e in line.elements if not isinstance(e, xl.BeamBeam6D)],
                       [n for e, n in zip(line.elements, line.element_names) if not isinstance(e, xl.BeamBeam6D)])
    return line, p0c, m0


def _fd_of_track(line, z, p0c, m0, h):
    """Richardson-extrapolated central differences of one turn of Line.track (steps h, h/2)."""
    zs = [z]
    for c in range(6):
        for s in (h[c], -h[c], h[c] / 2, -h[c] / 2):
            zz = z.copy()
            zz[c] += s
            zs.append(zz)
    p = _beam(_z_cols(np.array(zs)), p0c, m0)
    line.track(p)
    out = _coords(p)
    fd = np.zeros((6, 6))
    for c in range(6):
        a, b, a2, b2 = out[1 + 4 * c: 5 + 4 * c]
        d1, d2 = (a - b) / (2 * h[c]), (a2 - b2) / h[c]
        fd[:, c] = (4 * d2 - d1) / 3
    return fd


@pytest.mark.parametrize("name", ["fodo", "lhc", "petra4", "psb", "c3_no_bb6d"])
def test_one_turn_jacobian_matches_differences_of_track(name):
    line, p0c, m0 = _lattice(name)
    z = np.array([2e-4, 3e-6, -1.5e-4, -2e-6, 1e-3, 1e-4])
    p, t = _tangent(line, z, p0c, m0)
    J = t.matrix()[0].cpu().numpy()
    # The difference quotients of Line.track carry two errors: the rounding of ~1e4 records (the
    # tracked coordinates differ by ~1e-16 relative per record, amplified by the optics, divided by
    # the step) and the truncation of the Richardson formula (~(h / aperture)^4).  Two step sets a
    # decade apart bracket the optimum; the best one is compared, all are printed.  Measured on a B200:
    # 1.7e-9 (FODO), 4.2e-7 (LHC), 1.4e-6 (PETRA IV: exact drifts and strong sextupoles), 1.1e-7
    # (PSB), 1.7e-7 (C3 without 6D lenses) -- against 4e-15 for the NumPy oracle of the same map.
    scale = np.maximum(np.max(np.abs(J), axis=0), 1e-300)
    errs = []
    for f in (1.0, 3.0, 10.0):
        fd = _fd_of_track(line, z, p0c, m0, f * np.array([1e-6, 1e-8, 1e-6, 1e-8, 1e-5, 1e-6]))
        errs.append(np.max(np.abs(J - fd) / scale))
    print(name, "max column-relative |J - FD| = %.3g (steps h), %.3g (3 h), %.3g (10 h)" % tuple(errs))
    assert min(errs) <= 3e-6, (name, errs)


def test_lattice_jacobian_matches_oracle_on_fodo_and_psb():
    for name in ("fodo", "psb"):
        line, p0c, m0 = _lattice(name)
        z = np.array([2e-4, 3e-6, -1.5e-4, -2e-6, 1e-3, 1e-4])
        p, t = _tangent(line, z, p0c, m0)
        J = t.matrix()[0].cpu().numpy()
        packed, _ = line._tangent_lattice(DEV)
        zz, ref, _, _, alive = TO.track(packed, z, p0c, m0)
        assert alive
        scale = np.maximum(np.max(np.abs(ref), axis=0), 1e-300)
        err = np.max(np.abs(J - ref) / scale)
        print(name, "max column-relative |J - oracle| = %.3g" % err)
        assert err <= 1e-10, (name, err)


def test_same_orbit_as_track_on_c2():
    n, turns = 20_000, 100
    line, cols, p0c, m0 = configs.config_lhc(n)
    p = _beam(cols, p0c, m0)
    q = _beam(cols, p0c, m0)
    t = xl.TangentMap(n, DEV)
    line.track_tangent(p, t, num_turns=1)
    line.track(q, num_turns=1)
    a, b = _coords(p), _coords(q)
    alive = (q.state.cpu().numpy() == 1) & (p.state.cpu().numpy() == 1)
    # relative to max(|value|, the coordinate's rms over the beam): a coordinate that happens to pass
    # near zero keeps the absolute rounding of the turn.  The two kernels round differently (fused
    # block records against one record per element); 2.6e4 records x 2^-53 bounds the drift at 3e-12
    rms = np.sqrt(np.mean(b[alive] ** 2, axis=0))
    worst = np.max(np.abs(a - b)[alive] / np.maximum(np.abs(b[alive]), rms))
    print("C2, one turn: max |track_tangent - track| / max(|track|, rms) = %.3g" % worst)
    assert worst <= 3e-12
    line.track_tangent(p, t, num_turns=turns - 1)
    line.track(q, num_turns=turns - 1)
    sp, sq = p.to_numpy(), q.to_numpy()
    diff = (sp["state"] != sq["state"]) | (sp["at_element"] != sq["at_element"]) | (sp["at_turn"] != sq["at_turn"])
    # a particle may only change its fate when it grazes an aperture: the two kernels round
    # differently (fused against element-by-element records, ~1e-16 per element), which over 100
    # turns moves an orbit by far less than 1e-9 m; allow the particles lost within that margin
    print("C2, 100 turns: %d of %d particles with another fate" % (int(diff.sum()), n))
    assert int(diff.sum()) <= max(2, n // 5000)
    assert int(sq["state"].sum()) < n  # the beam does hit the apertures


@pytest.mark.parametrize("name", ["fodo", "lhc"])
def test_origin_matches_linear_optics(name):
    line, p0c, m0 = _lattice(name)
    if name == "lhc":
        # optics.py is the linear model: quadrupoles, bends, edges, rotations.  At the origin of the
        # full LHC the particle follows the crossing bumps through the sextupoles and octupoles, and
        # their feed-down is in J (as in the tracked map) but not in optics; the cavities change
        # delta.  Compare on the same lattice with multipoles cut at order 1 and the RF off.
        els = []
        for el in line.elements:
            if isinstance(el, xl.Multipole):
                el = xl.Multipole(knl=list(el.knl)[:2], ksl=list(el.ksl)[:2], hxl=el.hxl, hyl=el.hyl,
                                  length=el.length)
            elif isinstance(el, (xl.Cavity, xl.RFMultipole)):
                continue
            els.append(el)
        line = xl.Line(els)
    p, t = _tangent(line, np.zeros(6), p0c, m0)
    J = t.matrix()[0].cpu().numpy()
    m = optics.one_turn_matrix(line)
    # FODO: the full (x, px, y, py) x (x, px, y, py, delta) block.  LHC: the 4x4 block -- its origin is
    # not on the closed orbit (crossing bumps), and the delta column of the tracked map carries the
    # -px L / (1 + delta)^2 terms of that orbit in every drift, which the linear model leaves out.
    cols = [0, 1, 2, 3, 5] if name == "fodo" else [0, 1, 2, 3]
    got = J[np.ix_([0, 1, 2, 3], cols)]
    ref = m[:4][:, [0, 1, 2, 3, 4][: len(cols)]]
    assert np.allclose(got, ref, rtol=0, atol=1e-10 * np.abs(m).max()), (got, ref)
    co = xl.closed_orbit(line, p, mode="4d")

    def eigen_tunes(m4):
        return np.sort([a for a in np.angle(np.linalg.eigvals(m4)) / (2 * math.pi) if a > 0])

    q = eigen_tunes(co.matrix[:4, :4])
    if name == "fodo":
        tw = optics.twiss(line)
        ref = np.sort([tw["qx"] % 1.0, tw["qy"] % 1.0])
    else:
        # the LHC's skew quadrupoles and rotations couple the planes; optics.twiss reads the diagonal
        # blocks only (uncoupled lattices), so the reference is the eigen-tunes of its one-turn matrix
        ref = eigen_tunes(optics.one_turn_matrix(line)[:4, :4])
    print(name, "eigen-tunes of the closed-orbit matrix", q, "reference", ref)
    assert np.max(np.abs(q - ref)) < 1e-9, (name, q, ref)


def test_symplectic_transverse_block():
    line, p0c, m0 = _lattice("lhc")
    for el in line.elements:
        if isinstance(el, (xl.Cavity, xl.RFMultipole)):
            el.voltage = 0.0
    S = np.kron(np.eye(2), np.array([[0.0, 1.0], [-1.0, 0.0]]))
    z = np.array([[1e-4, 0, 1e-4, 0, 0, 0], [1.5e-3, 0, 1.2e-3, 0, 0, 2e-4], [5e-3, 0, 4e-3, 0, 0, 0]])
    p, t = _tangent(line, z, p0c, m0, turns=10)
    worst = 0.0
    for k in range(len(z)):
        if int(p.state[k]) != 1:
            continue
        J4 = t.matrix()[k].cpu().numpy()[:4, :4]
        worst = max(worst, np.max(np.abs(J4.T @ S @ J4 - S)) / max(1.0, np.max(np.abs(J4)) ** 2))
    print("LHC, 10 turns: max |J4^T S J4 - S| / max(1, |J4|^2) = %.3g" % worst)
    assert worst < 1e-11


def test_fli_separates_survivors_from_late_losses():
    line, cols, p0c, m0 = configs.config_lhc(1)
    n = 1024
    amp = np.linspace(5e-5, 8e-4, n)  # the C2 beam's core sigma is 1e-4 m: 0.5 to 8 sigma
    z = np.zeros((n, 6))
    z[:, 0], z[:, 2] = amp, 0.7 * amp
    p, t = _tangent(line, z, p0c, m0, turns=1000)
    fli = t.fli.cpu().numpy()
    alive_1k = p.state.cpu().numpy() == 1
    q = _beam(_z_cols(z), p0c, m0)
    line.track(q, num_turns=10_000)
    survive = q.state.cpu().numpy() == 1
    late = alive_1k & ~survive
    print("FLI at 1000 turns: %d survivors of 1e4 turns (median %.3g, max %.3g), %d lost between 1e3 and 1e4 "
          "turns (median %.3g, min %.3g)" % (survive.sum(), np.median(fli[survive]) if survive.any() else float("nan"),
                                            fli[survive].max() if survive.any() else float("nan"), late.sum(),
                                            np.median(fli[late]) if late.any() else float("nan"),
                                            fli[late].min() if late.any() else float("nan")))
    if not late.any() or not survive.any():
        pytest.skip("the scan has no particle lost between 1e3 and 1e4 turns")
    assert np.median(fli[late]) > np.median(fli[survive])


def test_closed_orbit_4d_with_kick_errors_and_offsets():
    line, p0c, m0 = _lattice("fodo")
    name = [n for e, n in zip(line.elements, line.element_names) if isinstance(e, xl.Multipole)][0]
    line._add_multipole_error_to(name, knl=[2e-5], ksl=[-1e-5])
    line._add_offset_error_to(name, dx=3e-4, dy=-2e-4)
    p = _beam(_z_cols(np.zeros(6)), p0c, m0)
    co = xl.closed_orbit(line, p, mode="4d")
    # thin lenses of order <= 1 plus dipole kicks: the transverse map is affine, M(z) = A z + b
    A = optics.one_turn_matrix(line)[:4, :4]
    q = _beam(_z_cols(np.zeros(6)), p0c, m0)
    line.track(q)
    b = _coords(q)[0, :4]
    ref = np.linalg.solve(np.eye(4) - A, b)
    assert np.max(np.abs(co.z[:4] - ref)) <= 1e-12 * np.max(np.abs(ref)), (co.z, ref)
    assert co.residual / max(1.0, np.max(np.abs(co.z[:4])) / 1e-3) <= 1e-14
    assert co.iterations <= 5


def test_closed_orbit_6d_psb():
    line, p0c, m0 = _lattice("psb")
    p = _beam(_z_cols(np.zeros(6)), p0c, m0)
    co = xl.closed_orbit(line, p, guess=[0, 0, 0, 0, 0.3, 2e-4])
    assert co.residual <= 1e-14, co
    q = _beam(_z_cols(co.z), p0c, m0)
    line.track(q, num_turns=100)
    drift = np.max(np.abs(_coords(q)[0] - co.z))
    print("PSB 6d closed orbit", co.z, "iterations", co.iterations, "drift over 100 turns %.3g" % drift)
    assert drift <= 1e-12
    ev = np.linalg.eigvals(co.matrix)
    assert np.allclose(np.abs(ev), 1.0, atol=1e-8)


def test_closed_orbit_errors():
    p = _beam(_z_cols(np.zeros(6)), 1e9, TO.MASS0)
    with pytest.raises(ValueError, match="singular"):
        xl.closed_orbit(xl.Line([xl.Drift(length=1.0)]), p, guess=[1e-3, 1e-4, 0, 0, 0, 0], mode="4d")
    line = xl.Line([xl.Multipole(knl=[0, 0.1]), xl.Drift(length=1.0),
                    xl.LimitRect(min_x=-1e-3, max_x=1e-3, min_y=-1e-3, max_y=1e-3)])
    with pytest.raises(ValueError, match="lost"):
        xl.closed_orbit(line, p, guess=[5e-3, 0, 0, 0, 0, 0], mode="4d")


def _run(line, z, p0c, m0, turns, perm=None, threads=0):
    p = _beam(_z_cols(z), p0c, m0)
    t = xl.TangentMap(len(p), DEV)
    line.track_tangent(p, t, num_turns=turns, threads_per_block=threads)
    return p.to_numpy(), t.jacobian.cpu().numpy(), t.log2_scale.cpu().numpy(), t.fli.cpu().numpy()


def test_bitwise_independent_of_batch_and_order_and_split():
    line, cols, p0c, m0 = configs.config_lhc(100_003)
    z = np.stack([cols[k] for k in COORDS], axis=1)
    big = _run(line, z, p0c, m0, 3)
    for n in (1, 37):
        small = _run(line, z[:n], p0c, m0, 3, threads=64)
        for a, b in zip(small[1:], big[1:]):
            assert np.array_equal(a, b[:n])
        for k in COORDS:
            assert np.array_equal(small[0][k], big[0][k][:n])
    perm = np.random.default_rng(5).permutation(len(z))[:5000]
    shuf = _run(line, z[perm], p0c, m0, 3)
    assert np.array_equal(shuf[1], big[1][perm]) and np.array_equal(shuf[3], big[3][perm])
    # T1 + T2 == T1 then T2
    p = _beam(_z_cols(z[:4096]), p0c, m0)
    t = xl.TangentMap(len(p), DEV)
    line.track_tangent(p, t, num_turns=1)
    line.track_tangent(p, t, num_turns=2)
    assert np.array_equal(t.jacobian.cpu().numpy(), big[1][:4096])
    assert np.array_equal(t.fli.cpu().numpy(), big[3][:4096])
    assert np.array_equal(p.to_numpy()["x"], big[0]["x"][:4096])


def test_overflow_guard_is_exact():
    # origin of a cell that is unstable in x (trace 3): the particle stays at the fixed point while
    # ||J|| grows by 2.6 per turn and crosses 2^512 after ~370 turns
    line = xl.Line([xl.Multipole(knl=[0.0, -1.0]), xl.Drift(length=1.0)])
    turns = 1200
    p = _beam(_z_cols(np.zeros(6)), 1e9, TO.MASS0)
    a = xl.TangentMap(1, DEV)
    line.track_tangent(p, a, num_turns=turns)
    q = _beam(_z_cols(np.zeros(6)), 1e9, TO.MASS0)
    b = xl.TangentMap(1, DEV)
    b.jacobian *= 2.0 ** -300  # the same map, rescaled at other turns
    b.log2_scale += 300
    line.track_tangent(q, b, num_turns=turns)
    sa, sb = int(a.log2_scale[0]), int(b.log2_scale[0])
    assert sa > 1000 and sb > 1000
    ja = torch.ldexp(a.jacobian, torch.tensor(float(sa - sb), device=DEV)).cpu().numpy()
    assert np.array_equal(ja, b.jacobian.cpu().numpy())
    assert abs(float(a.fli[0]) - float(b.fli[0])) < 1e-12 * float(a.fli[0])
    assert abs(float(a.lyapunov(turns)[0]) - math.log((3 + math.sqrt(5)) / 2)) < 1e-2


def test_refusals():
    line, cols, p0c, m0 = configs.config_lhc_beambeam(4)
    p = _beam(cols, p0c, m0)
    with pytest.raises(ValueError, match="BeamBeam6D"):
        line.track_tangent(p, xl.TangentMap(4, DEV))
    with pytest.raises(ValueError):
        line.track_tangent(p, xl.TangentMap(5, DEV))
    # a trace and a fused packing through the C entry point
    fodo, p0c, m0 = _lattice("fodo")
    q = _beam(_z_cols(np.zeros((2, 6))), p0c, m0)
    t = xl.TangentMap(2, DEV)
    from xline_b200.line import _c_particles

    cp, _ = _c_particles(q)
    L = _cabi.lib()
    packed, words = fodo._tangent_lattice(DEV)
    lat = packed.c_lattice(words.data_ptr())
    opts = _cabi.TrackOptions()
    opts.num_turns = 1
    trace = torch.zeros(len(fodo) * 6 * 2, dtype=torch.float64, device=DEV)
    opts.trace, opts.trace_particles = trace.data_ptr(), 2
    args = (C.c_void_p(t.jacobian.data_ptr()), C.c_void_p(t.log2_scale.data_ptr()), C.c_void_p(t.fli.data_ptr()), None)
    assert L.xlb_track_tangent_device(C.byref(lat), C.byref(cp), C.byref(opts), *args) == -1
    opts.trace, opts.trace_particles = None, 0
    opts.threads_per_block = 48
    assert L.xlb_track_tangent_device(C.byref(lat), C.byref(cp), C.byref(opts), *args) == -1
    opts.threads_per_block = 0
    fused, fwords = fodo._device_lattice(torch.device(DEV), False)
    flat = fused.c_lattice(fwords.data_ptr())
    if any(int(k) >= 0x80 for k in fused.record_counts):
        assert L.xlb_track_tangent_device(C.byref(flat), C.byref(cp), C.byref(opts), *args) == -1
    assert L.xlb_track_tangent_device(C.byref(lat), C.byref(cp), C.byref(opts), *args) == 0


def test_kernel_has_no_local_memory_and_no_stack():
    from xline_b200 import build

    txt = build.ptxas_report().get("tangent")
    assert txt, "no ptxas report for the tangent unit"
    m = re.search(r"Function properties for _ZN3xlb7tangent14tangent_kernel\S*\n\s*(\d+) bytes stack frame, "
                  r"(\d+) bytes spill stores, (\d+) bytes spill loads", txt)
    assert m and m.groups() == ("0", "0", "0"), txt
    obj = os.path.join(build.OBJ, "tangent.o")
    import subprocess

    res = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True)
    if res.returncode == 0:
        body = res.stdout
        assert "tangent_kernel" in body
        assert not re.search(r"\b(LDL|STL)\b", body)
