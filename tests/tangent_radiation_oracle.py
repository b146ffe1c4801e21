"""TEST INFRASTRUCTURE -- a NumPy statement of the Jacobian and the diffusion of a mean-mode
MULTIPOLE_RAD record (include/xline_b200.h, xlb_track_tangent_radiation_device and
xlb_track_envelope_device; DESIGN.md §4.10), for the walk of ``tests/tangent_oracle.py``.

The record's Jacobian is written out densely as half . kick . half, each half the chain of
add_to_energy and the scaling of px, py.  The envelope adds, per radiating half, V_h g g^T with
V_h = nbar (11/27) u_c^2 and g = dz_after/dW.  ``b`` is the beam of ``tangent_oracle.Particle``.
"""
import math

import numpy as np

from tests import packed_interpreter as PI
from tests import tangent_oracle as TO

X, PX, Y, PY, ZETA, DELTA = range(6)
X2_MEAN = 11.0 / 27.0  # <x^2> of the photon-number spectrum (x = photon energy / u_c)


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
