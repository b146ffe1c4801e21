"""Linear lattice functions of a thin-lens ``Line`` (host-side setup, not on the hot path).

The reference obtains beam sizes for its space-charge elements from a MAD-X ``twiss`` table
(``tests/test_madx_import.py:19-33`` sets up 120 kicks from ``betx bety dx`` at the kick
positions); MAD-X does not exist here, so this module derives the same quantities from the
line itself: the first-order map of every element about the reference orbit, written down
from the element definitions (``xline/elements.py``: Drift :48-56, Multipole :120-156,
DipoleEdge :538-548, SRotation :379-390), acting on ``(x, px, y, py, delta)`` with ``delta``
constant.  Everything else (apertures, monitors, cavities, space-charge and beam-beam
lenses) is the identity for this purpose.  Uncoupled lattices only: skew terms are carried in
the matrices, but ``twiss`` reads the two 2x2 diagonal blocks.

The GPU tracker is the check on this code, not the other way round
(``tests/test_gpu_parity.py::test_optics_tunes_match_tracking``).
"""
import math

import numpy as np

from . import elements as E


def element_matrix(el):
    """5x5 first-order map on ``(x, px, y, py, delta)`` or ``None`` for the identity."""
    if isinstance(el, (E.Drift, E.DriftExact)):
        if el.length == 0:
            return None
        m = np.eye(5)
        m[0, 1] = m[2, 3] = el.length
        return m
    if isinstance(el, E.Multipole):
        knl = list(el.knl) + [0.0, 0.0]
        ksl = list(el.ksl) + [0.0, 0.0]
        m = np.eye(5)
        # px -= k1l x - k1sl y ; py += k1l y + k1sl x   (Horner at first order, chi = 1)
        m[1, 0] -= knl[1]
        m[1, 2] += ksl[1]
        m[3, 2] += knl[1]
        m[3, 0] += ksl[1]
        hxl, hyl, length = float(el.hxl), float(el.hyl), float(el.length)
        if hxl or hyl:  # curvature terms: px += hxl delta - k0l hxl x / L ; py -= hyl delta - k0sl hyl y / L
            m[1, 4] += hxl
            m[3, 4] -= hyl
            if length > 0:
                m[1, 0] -= knl[0] * hxl / length
                m[3, 2] += ksl[0] * hyl / length
        return None if np.array_equal(m, np.eye(5)) else m
    if isinstance(el, E.DipoleEdge):
        corr = 2 * el.h * el.hgap * el.fint
        m = np.eye(5)
        m[1, 0] = el.h * math.tan(el.e1)
        m[3, 2] = -el.h * math.tan(el.e1 - corr / math.cos(el.e1) * (1 + math.sin(el.e1) ** 2))
        return m
    if isinstance(el, E.SRotation):
        c, s = math.cos(math.radians(el.angle)), math.sin(math.radians(el.angle))
        m = np.eye(5)
        m[0, 0] = m[1, 1] = m[2, 2] = m[3, 3] = c
        m[0, 2] = m[1, 3] = s
        m[2, 0] = m[3, 1] = -s
        return m
    return None


def one_turn_matrix(line):
    m = np.eye(5)
    for el in line.elements:
        e = element_matrix(el)
        if e is not None:
            m = e @ m
    return m


def _plane(m2):
    cosmu = 0.5 * (m2[0, 0] + m2[1, 1])
    if abs(cosmu) >= 1:
        raise ValueError("unstable linear optics (|cos mu| = %.6g)" % abs(cosmu))
    sinmu = math.copysign(math.sqrt(1 - cosmu * cosmu), m2[0, 1])
    beta = m2[0, 1] / sinmu
    alpha = (m2[0, 0] - m2[1, 1]) / (2 * sinmu)
    mu = math.atan2(sinmu, cosmu) % (2 * math.pi)
    return beta, alpha, mu / (2 * math.pi)


def twiss(line):
    """Periodic lattice functions at the ENTRY of every element.

    Returns a dict of arrays of length ``len(line) + 1`` (last entry = end of line):
    ``s betx alfx mux bety alfy muy dx dpx dy dpy`` plus scalars ``qx qy`` (full tunes from the
    accumulated phase advance), ``length`` and ``alfa_c`` (momentum compaction: the thin bends
    lengthen the path by ``hxl x - hyl y``, xline/elements.py:151)."""
    m = one_turn_matrix(line)
    betx, alfx, _ = _plane(m[0:2, 0:2])
    bety, alfy, _ = _plane(m[2:4, 2:4])
    disp = np.linalg.solve(np.eye(4) - m[:4, :4], m[:4, 4])
    n = len(line.elements)
    out = {k: np.zeros(n + 1) for k in ("s", "betx", "alfx", "mux", "bety", "alfy", "muy", "dx", "dpx", "dy", "dpy")}
    bx = np.array([[betx, -alfx], [-alfx, (1 + alfx * alfx) / betx]])
    by = np.array([[bety, -alfy], [-alfy, (1 + alfy * alfy) / bety]])
    d = np.append(disp, 1.0)
    s = mux = muy = path = 0.0

    def store(i):
        out["s"][i], out["mux"][i], out["muy"][i] = s, mux, muy
        out["betx"][i], out["alfx"][i] = bx[0, 0], -bx[0, 1]
        out["bety"][i], out["alfy"][i] = by[0, 0], -by[0, 1]
        out["dx"][i], out["dpx"][i], out["dy"][i], out["dpy"][i] = d[:4]

    for i, el in enumerate(line.elements):
        store(i)
        if isinstance(el, E.Multipole) and (el.hxl or el.hyl):
            path += el.hxl * d[0] - el.hyl * d[2]
        e = element_matrix(el)
        if e is not None:
            ex, ey = e[0:2, 0:2], e[2:4, 2:4]
            # phase advance of a 2x2 block: tan(dmu) = m12 / (m11 beta - m12 alpha)
            mux += math.atan2(ex[0, 1], ex[0, 0] * bx[0, 0] + ex[0, 1] * bx[0, 1]) / (2 * math.pi)
            muy += math.atan2(ey[0, 1], ey[0, 0] * by[0, 0] + ey[0, 1] * by[0, 1]) / (2 * math.pi)
            bx = ex @ bx @ ex.T
            by = ey @ by @ ey.T
            d = e @ d
        if isinstance(el, (E.Drift, E.DriftExact)):
            s += el.length
    store(n)
    out["qx"], out["qy"], out["length"] = mux, muy, s
    out["alfa_c"] = path / s if s > 0 else 0.0
    return out


def match_tunes(build_line, knobs, qx, qy, tol=1e-10, max_iter=20, step=1e-5):
    """Two-knob Newton iteration on the full tunes -- what the ``MATCH ... lmdif`` block of
    ``tests/psb/psb_fb_lhc.madx:46-52`` does with ``kqf`` / ``kqd``.  ``build_line(k0, k1)``
    returns the line for the knob values; returns the matched knobs."""
    k = np.array(knobs, dtype=float)

    def tunes(kk):
        tw = twiss(build_line(kk[0], kk[1]))
        return np.array([tw["qx"], tw["qy"]])

    target = np.array([qx, qy])
    for _ in range(max_iter):
        q0 = tunes(k)
        if np.max(np.abs(q0 - target)) < tol:
            break
        jac = np.empty((2, 2))
        for j in range(2):
            kp = k.copy()
            kp[j] += step
            jac[:, j] = (tunes(kp) - q0) / step
        k = k + np.linalg.solve(jac, target - q0)
    else:
        raise ValueError("tune matching did not converge")
    return float(k[0]), float(k[1])


def radiation_integrals(line, p0c, mass0, q0=1.0):
    """Synchrotron radiation integrals of the thin-lens map that ``Line.radiation`` tracks
    (include/xline_b200.h, DESIGN.md §4.9), from ``twiss``: what to expect of energy loss, damping
    and the equilibrium beam.  Energies in eV, ``p0c`` and ``mass0`` too.

    Per radiating multipole i (a Multipole of length L_i > 0), with k_i = k0l_i / L_i (curvature of
    the design orbit; kappa_i = |k_i|), h_i = hxl_i / L_i, and D (dispersion), H = gamma D^2 +
    2 alpha D D' + beta D'^2 (horizontal) at the element -- the mean of its entrance and exit values,
    as the two radiating halves sit on either side of the kick:
      I2 = sum kappa^2 L,  I3 = sum kappa^3 L,  I4 = sum D (h kappa^2 L + 2 k k1l),  I5 = sum H kappa^3 L.
    I4 follows from the map to first order in x = D delta: the path length of a half grows by
    hxl x / 2 and kappa^2 by 2 k k1l x / L^2 (for k0l >= 0, k = kappa: the textbook form).  I1 =
    sum D hxl over all curved multipoles (the momentum compaction times the length).  Then, with
    C_gamma-free constants K_e = e^2/(4 pi eps0) and hbar c in eV m:
      U0 = (2/3) q0^2 K_e beta^3 gamma^4 I2  (the mean mode's loss per turn on the design orbit);
      J_x = 1 - I4/I2, J_y = 1, J_z = 2 + I4/I2;  tau_u = 2 E / (J_u U0) turns;
      eps_x = C_q gamma^2 I5 / (J_x I2),  sigma_delta^2 = C_q gamma^2 I3 / (J_z I2),
      C_q = 55 hbar c / (32 sqrt(3) m)  (from <x^2> = 11/27 and the photon rate of the quantum mode).
    Returns a dict of those (``I1`` .. ``I5``, ``U0``, ``Jx Jy Jz``, ``tau_x tau_y tau_z``,
    ``eps_x``, ``sigma_delta``, ``gamma``, ``energy``)."""
    from .lattice import radiation_constants

    ke, hbarc, _ = radiation_constants()
    tw = twiss(line)
    energy = math.sqrt(p0c * p0c + mass0 * mass0)
    gamma, beta = energy / mass0, p0c / energy
    i1 = i2 = i3 = i4 = i5 = 0.0

    def curly_h(k):
        b, a, d, dp = tw["betx"][k], tw["alfx"][k], tw["dx"][k], tw["dpx"][k]
        return ((1 + a * a) / b) * d * d + 2 * a * d * dp + b * dp * dp

    for i, el in enumerate(line.elements):
        if isinstance(el, E.Multipole) and (el.hxl or el.hyl):
            i1 += el.hxl * tw["dx"][i]
        if not (isinstance(el, E.Multipole) and float(el.length) > 0):
            continue
        length = float(el.length)
        knl = list(el.knl) + [0.0, 0.0]
        k = knl[0] / length
        kap = abs(k)
        h = float(el.hxl) / length
        d = tw["dx"][i]
        i2 += kap * kap * length
        i3 += kap ** 3 * length
        i4 += d * (h * kap * kap * length + 2 * k * knl[1])
        i5 += 0.5 * (curly_h(i) + curly_h(i + 1)) * kap ** 3 * length
    u0 = (2.0 / 3.0) * q0 * q0 * ke * beta ** 3 * gamma ** 4 * i2
    jx, jy, jz = 1 - i4 / i2, 1.0, 2 + i4 / i2
    cq = 55.0 * hbarc / (32.0 * math.sqrt(3.0) * mass0)
    return dict(I1=i1, I2=i2, I3=i3, I4=i4, I5=i5, U0=u0, Jx=jx, Jy=jy, Jz=jz,
                tau_x=2 * energy / (jx * u0), tau_y=2 * energy / (jy * u0), tau_z=2 * energy / (jz * u0),
                eps_x=cq * gamma ** 2 * i5 / (jx * i2), sigma_delta=math.sqrt(cq * gamma ** 2 * i3 / (jz * i2)),
                gamma=gamma, energy=energy)
