"""TEST INFRASTRUCTURE -- a NumPy statement of the tangent recursion of include/xline_b200.h
("Tangent map"): one particle walked through the element-by-element packing of a line (fast
encoding, ``Line._tangent_lattice``), the coordinates advanced with the maps of
``tests/packed_interpreter.py`` and ``J <- M(z before) . J`` with each element's 6x6 Jacobian M
written out densely from the element definitions.  Everything but BeamBeam6D.  A mean-mode
MULTIPOLE_RAD record's Jacobian and diffusion come from ``tests/tangent_radiation_oracle.py``,
and the walk carries the envelope Sigma <- M Sigma M^T + D along with J.
"""
import math
import types

import numpy as np
from scipy.special import wofz

from tests import packed_interpreter as PI

X, PX, Y, PY, ZETA, DELTA = range(6)
COORDS = ("x", "px", "y", "py", "zeta", "delta")


class Particle:
    """One particle with the energy bookkeeping of the packed interpreter."""

    def __init__(self, z, p0c, mass0, q0=1.0, chi=1.0):
        beam = PI._Beam({k: [float(v)] for k, v in zip(COORDS, z)}, p0c, mass0, q0)
        self.beam = beam
        self.p = PI._Live(beam)
        self.p.chi = np.array([float(chi)])

    def z(self):
        return np.array([float(getattr(self.p, k)[0]) for k in COORDS])


def _rv1(beta0, delta, rvv):
    E = (1.0 + delta) / rvv
    return (1.0 - beta0 ** 2) / E ** 3


def _energy_jac(b, d, rvv, zeta, W, g):
    """dz_new/dz of add_to_energy(W) with dW/d(x, y, zeta, delta) = g (the kick rows aside)."""
    E = (1.0 + d) / rvv
    P1 = E + W / b.energy0
    ptau = (P1 - 1.0) / b.beta0
    opdn = math.sqrt(ptau * ptau + 2 * ptau / b.beta0 + 1)
    rvvn = opdn / P1
    dd_dP = P1 / (b.beta0 ** 2 * opdn)
    drvv_dP = dd_dP / P1 - opdn / P1 ** 2
    gP = np.zeros(6)
    gP[[X, Y, ZETA, DELTA]] = np.asarray(g) / b.energy0
    gP[DELTA] += b.beta0 ** 2 * (1 + d) / E
    M = np.eye(6)
    M[DELTA] = dd_dP * gP
    M[ZETA] = zeta / rvv * drvv_dP * gP
    M[ZETA, ZETA] += rvvn / rvv
    M[ZETA, DELTA] -= zeta / rvv * (rvvn / rvv) * _rv1(b.beta0, d, rvv)
    return M


def _field_jac(f64, i64, w, x, y):
    """(Ex, Ey, [[dEx/dx, dEx/dy], [dEy/dx, dEy/dy]]) of the fast field block at word w."""
    sx, sy, kind, A = f64[w], f64[w + 1], int(i64[w + 2]), f64[w + 4]
    if kind == 0:
        sig = 0.5 * (sx + sy)
        r2 = x * x + y * y
        if r2 < 1e-20:
            t = math.sqrt(r2) * A / sig
            return t * x, t * y, np.eye(2) * A / (2 * sig * sig)
        om = -math.expm1(-0.5 * r2 / sig ** 2)
        t = om * A / r2
        dt = A * ((1 - om) * 0.5 / sig ** 2 - om / r2) / r2
        return t * x, t * y, np.array([[t + 2 * x * x * dt, 2 * x * y * dt], [2 * x * y * dt, t + 2 * y * y * dt]])
    inv_s, fact, r_sb, r_bs, hb, hs = (f64[w + k] for k in range(6, 12))
    wide = kind == 1
    u, v = (abs(x), abs(y)) if wide else (abs(y), abs(x))
    z1 = complex(u * inv_s, v * inv_s)
    z2 = complex(r_sb * u * inv_s, r_bs * v * inv_s)
    w1, w2 = wofz(z1), wofz(z2)
    d1 = -2 * z1 * w1 + 2j / math.sqrt(math.pi)
    d2 = -2 * z2 * w2 + 2j / math.sqrt(math.pi)
    e = math.exp(-(u * u * hb + v * v * hs))
    F = w1 - e * w2
    Fu = d1 * inv_s - e * d2 * r_sb * inv_s + w2 * 2 * u * hb * e
    Fv = 1j * d1 * inv_s - e * 1j * d2 * r_bs * inv_s + w2 * 2 * v * hs * e
    sxy = -1.0 if (x < 0) != (y < 0) else 1.0
    sgx, sgy = (-1.0 if x < 0 else 1.0), (-1.0 if y < 0 else 1.0)
    if wide:
        Ex, Ey = sgx * fact * F.imag, sgy * fact * F.real
        D = fact * np.array([[Fu.imag, sxy * Fv.imag], [sxy * Fu.real, Fv.real]])
    else:
        Ex, Ey = sgx * fact * F.real, sgy * fact * F.imag
        D = fact * np.array([[Fv.real, sxy * Fu.real], [sxy * Fv.imag, Fu.imag]])
    return Ex, Ey, D


def _drift_jac(b, s, L, exact):
    d, px, py, rvv = s[DELTA], s[PX], s[PY], s[7]
    M = np.eye(6)
    rv1 = _rv1(b.beta0, d, rvv)
    if not exact:
        rpp = s[6]
        xp, yp = px * rpp, py * rpp
        M[X, PX], M[X, DELTA] = rpp * L, -xp * rpp * L
        M[Y, PY], M[Y, DELTA] = rpp * L, -yp * rpp * L
        M[ZETA, PX], M[ZETA, PY] = -L * xp * rpp, -L * yp * rpp
        M[ZETA, DELTA] = L * (rv1 + (xp * xp + yp * yp) * rpp)
        return M
    opd = 1 + d
    pz = math.sqrt(opd * opd - px * px - py * py)
    lpzi, g = L / pz, L / pz ** 3
    dl = g * np.array([0, px, 0, py, 0, -opd])  # gradient of lpzi
    M[X] += px * dl
    M[X, PX] += lpzi
    M[Y] += py * dl
    M[Y, PY] += lpzi
    M[ZETA] += -opd * dl
    M[ZETA, DELTA] += L * rv1 - lpzi
    return M


def element_jacobian(words, w, s, b, chi=1.0, qr=1.0):
    """M = dz_after/dz_before of the record at word ``w`` for the state ``s`` =
    (x, px, y, py, zeta, delta, rpp, rvv); ``b`` the beam constants (beta0, energy0, p0c, q0)."""
    f64, i64 = words.view(np.float64), words.view(np.int64)
    hdr = int(words[w])
    tag, aux = hdr & 0xFF, (hdr >> 8) & 0xFF
    p0 = f64[w + 1]
    x, px, y, py, zeta, d, rpp, rvv = s
    M = np.eye(6)
    if tag in (PI.T_DRIFT, PI.T_DRIFT_EXACT):
        return _drift_jac(b, s, p0, tag == PI.T_DRIFT_EXACT)
    if tag in (PI.T_MULTIPOLE, PI.T_MULTIPOLE_CURVED):
        at = w + 2 if tag == PI.T_MULTIPOLE else w + 6
        pairs = f64[at: at + 2 * (aux + 1)].reshape(aux + 1, 2)
        c = pairs[:, 0] + 1j * pairs[:, 1]  # c[m] = coefficient of z^(aux - m)
        z = complex(x, y)
        dP = sum(c[m] * (aux - m) * z ** (aux - m - 1) for m in range(aux))
        M[PX, X], M[PX, Y] = -chi * dP.real, chi * dP.imag
        M[PY, X], M[PY, Y] = chi * dP.imag, chi * dP.real
        if tag == PI.T_MULTIPOLE_CURVED:
            hxl, hyl, inv_len = p0, f64[w + 2], f64[w + 4]
            M[PX, X] -= chi * pairs[aux, 0] * hxl * inv_len
            M[PY, Y] += chi * pairs[aux, 1] * hyl * inv_len
            M[PX, DELTA], M[PY, DELTA] = hxl, -hyl
            M[ZETA, X], M[ZETA, Y] = -chi * hxl, chi * hyl
        return M
    if tag in (PI.T_CAVITY, PI.T_SAWTOOTH_CAVITY):
        k, lag = f64[w + 2], f64[w + 3]
        phase = lag - k * (zeta / rvv / b.beta0)
        C = qr * b.q0 * p0
        if tag == PI.T_CAVITY:
            wv, dw = math.sin(phase), math.cos(phase)
        else:
            wv, dw = (phase + math.pi) % (2 * math.pi) - math.pi, 1.0
        rv1 = _rv1(b.beta0, d, rvv)
        g = [0.0, 0.0, C * dw * (-k / (rvv * b.beta0)), C * dw * k * zeta * rv1 / (rvv * rvv * b.beta0)]
        return _energy_jac(b, d, rvv, zeta, C * wv, g)
    if tag == PI.T_RFMULTIPOLE:
        k, lag = f64[w + 2], f64[w + 3]
        ktau = k * (zeta / rvv / b.beta0)
        z = complex(x, y)
        Q1 = B0 = A1 = 0j
        dptr = 0.0
        for ii in range(aux + 1):
            kn, ks, pn, ps = f64[w + 4 + 4 * ii: w + 8 + 4 * ii]
            A = math.cos(pn - ktau) * kn + 1j * math.cos(ps - ktau) * ks
            B = math.sin(pn - ktau) * kn + 1j * math.sin(ps - ktau) * ks
            Zi, Zm, Zp = z ** ii / math.factorial(ii), (z ** (ii - 1) / math.factorial(ii - 1) if ii else 0), \
                z ** (ii + 1) / math.factorial(ii + 1)
            Q1 += A * Zm
            B0 += B * Zi
            A1 += A * Zp
            dptr += (B * Zp).real
        rv1 = _rv1(b.beta0, d, rvv)
        kz, kd = k / (rvv * b.beta0), -k * zeta * rv1 / (rvv * rvv * b.beta0)
        C = qr * b.q0
        W = C * (p0 * math.sin(lag - ktau) - b.p0c * k * dptr)
        dWk = C * (-p0 * math.cos(lag - ktau) + b.p0c * k * A1.real)
        M = _energy_jac(b, d, rvv, zeta, W, [-C * b.p0c * k * B0.real, C * b.p0c * k * B0.imag, dWk * kz, dWk * kd])
        M[PX, [X, Y, ZETA, DELTA]] += [-chi * Q1.real, chi * Q1.imag, -chi * B0.real * kz, -chi * B0.real * kd]
        M[PY, [X, Y, ZETA, DELTA]] += [chi * Q1.imag, chi * Q1.real, chi * B0.imag * kz, chi * B0.imag * kd]
        return M
    if tag == PI.T_SROTATION:
        cz, sz = p0, f64[w + 2]
        R = np.array([[cz, sz], [-sz, cz]])
        M[np.ix_([X, Y], [X, Y])] = R
        M[np.ix_([PX, PY], [PX, PY])] = R
        return M
    if tag == PI.T_DIPOLE_EDGE:
        M[PX, X], M[PY, Y] = p0, f64[w + 2]
        return M
    if tag in (PI.T_BEAMBEAM4D, PI.T_SPACECHARGE):
        xo, yo = f64[w + 2], f64[w + 3]
        Ex, Ey, D = _field_jac(f64, i64, w + 4, x - xo, y - yo)
        t = w + 2 * (2 + 6)
        fz = fd = 0.0
        if tag == PI.T_BEAMBEAM4D:
            beta_r, cq = f64[t + 2], f64[t + 3]
            beta = b.beta0 / rvv
            K = chi * cq * qr * b.q0 / b.p0c
            f = K * (1 + beta * beta_r) / (beta + beta_r)
            fd = K * (beta_r ** 2 - 1) / (beta + beta_r) ** 2 * (-b.beta0 * _rv1(b.beta0, d, rvv) / rvv ** 2)
        else:
            base, p1 = f64[t], f64[t + 1]
            g = chi * qr * b.q0 ** 2 * (1 - b.beta0 ** 2) / (b.p0c * b.beta0) * base
            kind = aux & 0xF
            lam, dlz, dld = 1.0, 0.0, 0.0
            if kind == 1:
                sg = zeta / rvv
                arg = p1 * sg * sg
                if int(i64[t + 6]):
                    lam = f64[t + 2] * math.exp(-arg)
                    dla = -lam
                else:
                    up = max(1.0 - arg * f64[t + 3], 0.0)
                    lam = f64[t + 2] * up ** f64[t + 4]
                    dla = -f64[t + 3] * f64[t + 4] * f64[t + 2] * up ** (f64[t + 4] - 1) if up > 0 else 0.0
                dlz = dla * 2 * p1 * sg / rvv
                dld = dla * 2 * p1 * sg * (-zeta * _rv1(b.beta0, d, rvv) / rvv ** 2)
            elif kind in (2, 3):
                z0, dz, n = p1, f64[t + 2], int(i64[t + 4])
                i = min(max(int(math.floor((zeta - z0) / dz)), 0), n - 2)
                if kind == 2:
                    prof = f64[t + 6: t + 6 + n]
                    if z0 < zeta < z0 + (n - 1) * dz:
                        dlz = (prof[i + 1] - prof[i]) / dz
                        lam = dlz * (zeta - (z0 + i * dz)) + prof[i]
                    else:
                        lam = prof[0] if zeta <= z0 else prof[n - 1]
                else:
                    xk = f64[t + 6: t + 6 + n]
                    c = f64[t + 6 + n: t + 6 + n + 4 * (n - 1)]
                    m, tt = n - 1, zeta - xk[i]
                    lam = ((c[i] * tt + c[m + i]) * tt + c[2 * m + i]) * tt + c[3 * m + i]
                    dlz = (3 * c[i] * tt + 2 * c[m + i]) * tt + c[2 * m + i]
            f, fz, fd = g * lam, g * dlz, g * dld
        M[PX, [X, Y]] += f * D[0]
        M[PY, [X, Y]] += f * D[1]
        M[PX, [ZETA, DELTA]] += Ex * np.array([fz, fd])
        M[PY, [ZETA, DELTA]] += Ey * np.array([fz, fd])
        return M
    return M  # XYSHIFT, LIMIT_*, MONITOR: the identity


def element_map(words, w, z, p0c, mass0, q0=1.0):
    """z after the record at word ``w`` (packed interpreter), and whether the particle survived: the
    interpreter runs a one-record copy of the lattice, closed by END_TURN."""
    size = (int(words[w]) >> 16) & 0x3FFF
    rec = np.zeros(2 * size + 2, dtype=np.uint64)
    rec[: 2 * size] = words[w: w + 2 * size]
    f64, i64 = rec.view(np.float64), rec.view(np.int64)
    hdr = int(rec[0])
    # a one-record pass starts at s = 0: the s_here word, if any, holds 0.0 and END_TURN the advance
    s_at, adv = PI._path_length_words(hdr & 0xFF, (hdr >> 8) & 0xFF, 0, f64, i64)
    if s_at is not None:
        f64[s_at] = 0.0
    rec[2 * size] = np.uint64(PI.T_END_TURN)
    f64[2 * size + 1] = adv
    packed = types.SimpleNamespace(words=rec, chunk_words=len(rec), n_chunks=1, strict=False, segments=None)
    part = Particle(z, p0c, mass0, q0)
    out = PI.track(packed, {k: getattr(part.p, k) for k in COORDS}, p0c, mass0, 1)
    return np.array([out[k][0] for k in COORDS]), bool(out["state"][0] == 1)


def track(packed, z, p0c, mass0, q0=1.0, num_turns=1, cov=None):
    """(z, J, Sigma, energy lost, alive) of one particle after ``num_turns`` turns of ``packed``
    (element-by-element packing, fast encoding, mean-mode radiating records included); Sigma starts
    at ``cov`` (default 0).  Tagging records it cannot follow raises."""
    from tests import tangent_radiation_oracle as TRO

    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
    z = np.array(z, dtype=np.float64)
    J = np.eye(6)
    S = np.zeros((6, 6)) if cov is None else np.array(cov, dtype=np.float64)
    lost = 0.0
    b = Particle(z, p0c, mass0, q0).beam
    for _ in range(num_turns):
        for ch in range(packed.n_chunks):
            w = ch * packed.chunk_words
            end = False
            while True:
                hdr = int(words[w])
                tag, size = hdr & 0xFF, (hdr >> 16) & 0x3FFF
                if tag == PI.T_END_CHUNK:
                    break
                if tag == PI.T_END_TURN:
                    end = True
                    break
                if tag == PI.T_MULTIPOLE_RAD:
                    M, D, e, _ = TRO.rad_record(words, w, z, b)
                    lost += e
                else:
                    part = Particle(z, p0c, mass0, q0)
                    s = [float(getattr(part.p, k)[0]) for k in COORDS + ("rpp", "rvv")]
                    M, D = element_jacobian(words, w, s, b), 0.0
                J = M @ J
                S = M @ S @ M.T + D
                z, alive = element_map(words, w, z, p0c, mass0, q0)
                if not alive:
                    return z, J, S, lost, False
                w += 2 * size
            if end:
                break
    return z, J, S, lost, True


P0C, MASS0 = 6.5e12, 938.27208816e6  # LHC protons: beta0 close to 1
P0C_LOW = 1.2e9                        # a slow beam (PS Booster-like): rvv visibly depends on delta


def element_cases():
    """(name, element, p0c, z) for every element type the tangent kernel covers, at a point where
    every term of its Jacobian is active."""
    import xline_b200 as xl

    prof = np.exp(-np.linspace(-3, 3, 41) ** 2 / 2)
    z = np.array([1.2e-3, -2.1e-4, -0.7e-3, 1.3e-4, 0.05, 1.7e-4])
    zb = np.array([0.9e-3, -2.1e-4, -1.6e-3, 1.3e-4, 0.0513, 1.7e-4])  # beam fields: |x| < |y|, zeta off the grid
    sc = dict(number_of_particles=2e11, sigma_x=1.3e-3, sigma_y=0.8e-3, length=1.5, x_co=1e-4, y_co=-2e-4)
    return [
        ("drift", xl.Drift(length=2.3), P0C_LOW, z),
        ("drift_exact", xl.DriftExact(length=2.3), P0C_LOW, z),
        ("multipole", xl.Multipole(knl=[1e-4, 0.02, -0.5, 30.0], ksl=[2e-5, -0.01, 0.3, 5.0]), P0C, z),
        ("multipole_curved", xl.Multipole(knl=[3e-3, 0.02, 0.4], ksl=[1e-4, 0.01], hxl=3e-3, hyl=2e-4, length=1.2),
         P0C, z),
        ("cavity", xl.Cavity(voltage=5e6, frequency=4e8, lag=30.0), P0C_LOW, z),
        ("sawtooth_cavity", xl.SawtoothCavity(voltage=5e6, frequency=4e8, lag=30.0), P0C_LOW, z),
        ("rfmultipole", xl.RFMultipole(voltage=2e6, frequency=4e8, lag=20.0, knl=[1e-3, 0.02, 0.7],
                                       ksl=[2e-4, -0.03, 0.2], pn=[10.0, 40.0, -30.0], ps=[5.0, -20.0, 60.0]),
         P0C_LOW, z),
        ("xyshift", xl.XYShift(dx=1e-4, dy=-3e-4), P0C, z),
        ("srotation", xl.SRotation(angle=17.0), P0C, z),
        ("dipole_edge", xl.DipoleEdge(h=0.05, e1=0.1, hgap=0.03, fint=0.5), P0C, z),
        ("beambeam4d_round", xl.BeamBeam4D(charge=1.1e11, sigma_x=1.6e-3, sigma_y=1.6e-3, beta_r=1.0,
                                           x_bb=1e-4, y_bb=2e-4, d_px=1e-7, d_py=-1e-7), P0C_LOW, zb),
        ("beambeam4d_wide", xl.BeamBeam4D(charge=1.1e11, sigma_x=1.6e-3, sigma_y=0.9e-3, beta_r=0.8,
                                          x_bb=1e-4, y_bb=2e-4), P0C_LOW, zb),
        ("beambeam4d_tall", xl.BeamBeam4D(charge=1.1e11, sigma_x=0.9e-3, sigma_y=1.6e-3, beta_r=0.8,
                                          x_bb=1e-4, y_bb=2e-4), P0C_LOW, zb),
        ("sc_coasting", xl.SCCoasting(circumference=157.0, **sc), P0C_LOW, zb),
        ("sc_qgauss_gauss", xl.SCQGaussProfile(bunchlength_rms=0.2, q_parameter=1.0, **sc), P0C_LOW, zb),
        ("sc_qgauss_q", xl.SCQGaussProfile(bunchlength_rms=0.2, q_parameter=1.2, **sc), P0C_LOW, zb),
        ("sc_interp_linear", xl.SCInterpolatedProfile(line_density_profile=prof, dz=0.025, z0=-0.5, method=0, **sc),
         P0C_LOW, zb),
        ("sc_interp_cubic", xl.SCInterpolatedProfile(line_density_profile=prof, dz=0.025, z0=-0.5, method=1, **sc),
         P0C_LOW, zb),
        ("limit_rect", xl.LimitRect(min_x=-0.01, max_x=0.01, min_y=-0.01, max_y=0.01), P0C, z),
        ("limit_ellipse", xl.LimitEllipse(a=0.02, b=0.01), P0C, z),
        ("limit_rect_ellipse", xl.LimitRectEllipse(max_x=0.02, max_y=0.01, a=0.03, b=0.02), P0C, z),
    ]


def pack_one(element, radiation=None):
    """The element-by-element packing ``Line.track_tangent`` uses, of a one-element line
    (``radiation="mean"``: that of ``Line.track_tangent(..., radiation=True)``)."""
    from xline_b200.lattice import pack_line

    return pack_line([element], strict=False, fuse=False, merge=False, split_lenses=False, drop_noops=False,
                     radiation=radiation)


def fd_jacobian(packed, z, p0c, mass0=MASS0, rel=1e-3, w=0):
    """Central differences of the packed interpreter's map of the record at word ``w``,
    Richardson-extrapolated (h, h/2)."""
    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
    # delta steps are the largest: rvv and rpp are recomputed from delta with an error of ~1e-16 each
    scale = np.array([1e-3, 1e-4, 1e-3, 1e-4, 1e-2, 1e-3])
    out = np.zeros((6, 6))
    for c in range(6):
        h = rel * scale[c]

        def d(hh):
            zp, zm = z.copy(), z.copy()
            zp[c] += hh
            zm[c] -= hh
            return (element_map(words, w, zp, p0c, mass0)[0] - element_map(words, w, zm, p0c, mass0)[0]) / (2 * hh)

        out[:, c] = (4 * d(h / 2) - d(h)) / 3
    return out


def oracle_jacobian(element, z, p0c):
    packed = pack_one(element)
    zz, J, _, _, alive = track(packed, z, p0c, MASS0)
    assert alive
    return J
