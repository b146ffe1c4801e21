"""TEST INFRASTRUCTURE -- a NumPy statement of the tangent map and the envelope of lines with
mean-mode radiating multipoles (include/xline_b200.h, xlb_track_tangent_radiation_device and
xlb_track_envelope_device; DESIGN.md §4.10).

One particle is walked through the element-by-element packing with radiation
(``Line._tangent_lattice(..., radiation=True)``): the coordinates advance with
``tests/radiation_interpreter.py`` (the packed maps), every other record's Jacobian comes from
``tests/tangent_oracle.py``, and a MULTIPOLE_RAD record's Jacobian is written out densely here as
half . kick . half, each half the chain of add_to_energy and the scaling of px, py.  The envelope
adds, per radiating half, V_h g g^T with V_h = nbar (11/27) u_c^2 and g = dz_after/dW.
"""
import math
import types

import numpy as np

from tests import packed_interpreter as PI
from tests import radiation_interpreter as RI
from tests import tangent_oracle as TO

X, PX, Y, PY, ZETA, DELTA = range(6)
COORDS = TO.COORDS
T_MULTIPOLE_RAD = RI.T_MULTIPOLE_RAD
X2_MEAN = 11.0 / 27.0  # <x^2> of the photon-number spectrum (x = photon energy / u_c)


class Beam:
    def __init__(self, p0c, mass0, q0=1.0):
        self.p0c, self.mass0, self.q0 = float(p0c), float(mass0), float(q0)
        self.energy0 = math.sqrt(self.p0c ** 2 + self.mass0 ** 2)
        self.beta0 = self.p0c / self.energy0


def _energy(b, d):
    """(rvv, ptaub0) of delta (the bookkeeping of the packed interpreter)."""
    db0 = d * b.beta0
    ptaub0 = math.sqrt(db0 ** 2 + 2 * db0 * b.beta0 + 1) - 1
    return (1 + d) / (1 + ptaub0), ptaub0


def _half(b, z, rec, fl, lh, f2, hxl, hyl):
    """One mean-mode radiating half at the state ``z``: (M = dz_after/dz_before, V_h, g, dE, z_after).
    ``f2`` = the gradient of fl^2 over (x, y)."""
    length, inv_len, ke, hbarc, alpha = rec
    d = z[DELTA]
    rvv, ptaub0 = _energy(b, d)
    m2 = (b.energy0 - b.p0c) * (b.energy0 + b.p0c)
    opd = 1 + d
    P = opd * b.p0c
    E = math.sqrt(P * P + m2)
    gamma = E / math.sqrt(m2)
    beta = P / E
    kappa = fl * inv_len / opd
    q2 = b.q0 ** 2
    if kappa == 0.0:
        return np.eye(6), 0.0, np.zeros(6), 0.0, z.copy()
    dE = -(2.0 / 3.0) * q2 * ke * beta ** 3 * gamma ** 4 * kappa ** 2 * lh
    A = -(2.0 / 3.0) * q2 * ke * beta ** 3 * gamma ** 4 * (inv_len / opd) ** 2
    gW = np.array([A * (f2[0] * lh + fl * fl * 0.5 * hxl), A * (f2[1] * lh - fl * fl * 0.5 * hyl), 0.0,
                   dE * (1 / opd + P * b.p0c / E ** 2)])
    M = TO._energy_jac(b, d, rvv, z[ZETA], dE, gW)
    # new state (add_to_energy, then px, py scaled)
    ptau = (ptaub0 + dE / b.energy0) / b.beta0
    dn = math.sqrt(ptau ** 2 + 2 * ptau / b.beta0 + 1) - 1
    rvvn = (1 + dn) / (1 + ptau * b.beta0)
    f = (1 + dn) / opd
    zn = z.copy()
    zn[DELTA], zn[ZETA] = dn, z[ZETA] * rvvn / rvv
    zn[PX], zn[PY] = z[PX] * f, z[PY] * f
    # px' = px (1+delta')/(1+delta)
    Mf = np.eye(6)
    for r in (PX, PY):
        Mf[r] = 0.0
        Mf[r, r] = f
        Mf[r] += z[r] / opd * M[DELTA]
        Mf[r, DELTA] -= z[r] * f / opd
    for r in (ZETA, DELTA):
        Mf[r] = M[r]
    # g = dz_after / dW at fixed z_before
    E1 = opd / rvv
    P1 = E1 + dE / b.energy0
    opdn = math.sqrt(((P1 - 1) / b.beta0) ** 2 + 2 * (P1 - 1) / b.beta0 ** 2 + 1)
    dd_dP = P1 / (b.beta0 ** 2 * opdn)
    drvv_dP = dd_dP / P1 - opdn / P1 ** 2
    gd = dd_dP / b.energy0
    g = np.array([0.0, z[PX] / opd * gd, 0.0, z[PY] / opd * gd, z[ZETA] / rvv * drvv_dP / b.energy0, gd])
    nbar = (5.0 / (2.0 * math.sqrt(3.0))) * q2 * alpha * gamma * kappa * lh
    uc = 1.5 * hbarc * gamma ** 3 * kappa
    return Mf, nbar * X2_MEAN * uc * uc, g, dE, zn


def _kick(words, w_sub, z, b):
    """The embedded multipole record at word ``w_sub``: (M, z_after)."""
    f64 = words.view(np.float64)
    hdr = int(words[w_sub])
    tag, aux = hdr & 0xFF, (hdr >> 8) & 0xFF
    rvv, _ = _energy(b, z[DELTA])
    s = list(z) + [1 / (1 + z[DELTA]), rvv]
    M = TO.element_jacobian(words, w_sub, s, b)
    at = w_sub + 2 if tag == PI.T_MULTIPOLE else w_sub + 6
    pairs = f64[at: at + 2 * (aux + 1)].reshape(aux + 1, 2)
    c = pairs[:, 0] + 1j * pairs[:, 1]
    P = sum(c[m] * complex(z[X], z[Y]) ** (aux - m) for m in range(aux + 1))
    zn = z.copy()
    zn[PX] -= P.real
    zn[PY] += P.imag
    if tag == PI.T_MULTIPOLE_CURVED:
        hxl, hyl, inv_len = f64[w_sub + 1], f64[w_sub + 2], f64[w_sub + 4]
        zn[PX] += hxl + hxl * z[DELTA] - pairs[aux, 0] * hxl * z[X] * inv_len
        zn[PY] -= hyl + hyl * z[DELTA] - pairs[aux, 1] * hyl * z[Y] * inv_len
        zn[ZETA] -= hxl * z[X] - hyl * z[Y]
    return M, zn


def rad_record(words, w, z, b):
    """A mean-mode MULTIPOLE_RAD record at word ``w`` for the state ``z``: (J, D, energy lost, z_after)
    with D the diffusion the record adds at its exit."""
    f64 = words.view(np.float64)
    hdr = int(words[w])
    aux = (hdr >> 8) & 0xFF
    rec = (f64[w + 2], f64[w + 3], f64[w + 4], f64[w + 5], f64[w + 6])
    sub = w + 8
    tag = int(words[sub]) & 0xFF
    if tag == PI.T_MULTIPOLE:
        pairs, hxl, hyl = f64[sub + 2: sub + 2 + 2 * (aux + 1)].reshape(aux + 1, 2), 0.0, 0.0
    else:
        pairs, hxl, hyl = f64[sub + 6: sub + 6 + 2 * (aux + 1)].reshape(aux + 1, 2), f64[sub + 1], f64[sub + 2]
    c = pairs[:, 0] + 1j * pairs[:, 1]
    zc = complex(z[X], z[Y])
    P = sum(c[m] * zc ** (aux - m) for m in range(aux + 1))
    dP = sum(c[m] * (aux - m) * zc ** (aux - m - 1) for m in range(aux))
    fl = abs(P)
    f2 = (2 * (P.real * dP.real + P.imag * dP.imag), 2 * (P.imag * dP.real - P.real * dP.imag))
    lh = 0.5 * (rec[0] + hxl * z[X] - hyl * z[Y])
    M1, V1, g1, e1, z1 = _half(b, z, rec, fl, lh, f2, hxl, hyl)
    K, z2 = _kick(words, sub, z1, b)
    M2, V2, g2, e2, z3 = _half(b, z2, rec, fl, lh, f2, hxl, hyl)
    T = M2 @ K
    D = V1 * np.outer(T @ g1, T @ g1) + V2 * np.outer(g2, g2)
    return M2 @ K @ M1, D, -(e1 + e2), z3


def _one_record(words, w, size):
    rec = np.zeros(2 * size + 2, dtype=np.uint64)
    rec[: 2 * size] = words[w: w + 2 * size]
    f64 = rec.view(np.float64)
    tag = int(rec[0]) & 0xFF
    f64[2 * size + 1] = f64[1] if tag in (PI.T_DRIFT, PI.T_DRIFT_EXACT) else 0.0  # END_TURN
    if tag in (PI.T_LIMIT_RECT, PI.T_LIMIT_ELLIPSE):
        f64[5] = 0.0
    return types.SimpleNamespace(words=rec, chunk_words=len(rec), n_chunks=1, strict=False, segments=None)


def element_map(words, w, z, p0c, mass0):
    """z after the record at word ``w`` (radiation interpreter), and whether the particle survived."""
    size = (int(words[w]) >> 16) & 0x3FFF
    out = RI.track(_one_record(words, w, size), {k: [float(v)] for k, v in zip(COORDS, z)}, p0c, mass0, 1)
    return np.array([out[k][0] for k in COORDS]), bool(out["state"][0] == 1)


def track(packed, z, p0c, mass0, num_turns=1, cov=None):
    """(z, J, Sigma, energy lost, alive) of one particle after ``num_turns`` turns of ``packed``
    (element-by-element packing with mean-mode radiating records); Sigma starts at ``cov``
    (default 0)."""
    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
    z = np.array(z, dtype=np.float64)
    J = np.eye(6)
    S = np.zeros((6, 6)) if cov is None else np.array(cov, dtype=np.float64)
    b = Beam(p0c, mass0)
    lost = 0.0
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
                if tag == T_MULTIPOLE_RAD:
                    M, D, e, _ = rad_record(words, w, z, b)
                    lost += e
                else:
                    rvv, _ = _energy(b, z[DELTA])
                    M = TO.element_jacobian(words, w, list(z) + [1 / (1 + z[DELTA]), rvv], b)
                    D = 0.0
                J = M @ J
                S = M @ S @ M.T + D
                z, alive = element_map(words, w, z, p0c, mass0)
                if not alive:
                    return z, J, S, lost, False
                w += 2 * size
            if end:
                break
    return z, J, S, lost, True


def pack_one(element):
    """The packing ``Line.track_tangent(..., radiation=True)`` uses, of a one-element line."""
    from xline_b200.lattice import pack_line

    return pack_line([element], strict=False, fuse=False, merge=False, split_lenses=False, drop_noops=False,
                     radiation="mean")


def fd_jacobian(packed, z, p0c, mass0, rel=1e-3, w=0):
    """Central differences of the radiation interpreter's map of the record at word ``w``,
    Richardson-extrapolated (h, h/2)."""
    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
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
