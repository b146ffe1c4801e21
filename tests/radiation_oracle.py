"""TEST INFRASTRUCTURE -- the CPU oracle of synchrotron radiation in thin multipoles, and a
``Line.track`` loop over the oracle's element maps (``oracle/xline_oracle.py``) that includes it.

The reference tracks without radiation, so this restates the project's own definition
(include/xline_b200.h, XLB_T_MULTIPOLE_RAD; DESIGN.md §4.9) from the element fields: a NumPy
Philox4x32-10, the photon-energy table of ``xline_b200/csrc/synrad_table.inc`` evaluated as
``scripts/gen_synrad_table.py`` describes it, and the two radiating halves around the oracle's own
multipole map.  Nothing is shared with the product package.
"""
import importlib.util
import math
import os

import numpy as np
from scipy.constants import alpha as ALPHA
from scipy.constants import c as CLIGHT
from scipy.constants import e as QE
from scipy.constants import epsilon_0, hbar

from oracle import xline_oracle as xo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K_E = QE / (4.0 * math.pi * epsilon_0)  # eV m
HBAR_C = hbar * CLIGHT / QE             # eV m
MODES = ("mean", "quantum")


def _gen():
    spec = importlib.util.spec_from_file_location("gen_synrad_table", os.path.join(ROOT, "scripts", "gen_synrad_table.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


GEN = _gen()
LO, HI = GEN.parse_inc(os.path.join(ROOT, "xline_b200", "csrc", "synrad_table.inc"))

# ---------------------------------------------------------------- Philox4x32-10
M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counters (arrays of uint32 values) under the key (k0, k1): four uint64 arrays
    holding the 32-bit output words r0..r3."""
    c = [np.asarray(v, dtype=np.uint64) & MASK for v in (c0, c1, c2, c3)]
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c[0]
        p1 = M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1),
             p0 & MASK]
        k0 = (k0 + W0) & 0xFFFFFFFF
        k1 = (k1 + W1) & 0xFFFFFFFF
    return c


def u01(lo, hi):
    """((w >> 11) + 0.5) 2^-53 of w = hi 2^32 + lo."""
    w = (np.asarray(hi, dtype=np.uint64) << np.uint64(32)) | np.asarray(lo, dtype=np.uint64)
    return ((w >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def uniforms(seed, pid, turn, elem, half, j):
    """Uniforms 2j and 2j+1 of a half (arrays over particles)."""
    pid = np.asarray(pid, dtype=np.int64).astype(np.uint64)
    turn = np.asarray(turn, dtype=np.int64).astype(np.uint64)
    c3 = (np.uint64(int(elem)) << np.uint64(8)) | np.uint64(int(half) << 7) | np.uint64(int(j))
    r = philox(pid & MASK, pid >> np.uint64(32), turn & MASK, np.broadcast_to(c3, pid.shape), seed & 0xFFFFFFFF,
               seed >> 32)
    return u01(r[0], r[1]), u01(r[2], r[3])


def synrad_x(U):
    """x = F^-1(U) from the committed table."""
    return GEN.evaluate(U, LO, HI)


def poisson_count(u0, nbar):
    """Smallest i with u0 <= C_i (C_0 = p_0 = exp(-nbar), p_i = p_(i-1) nbar / i), capped at 255;
    also returns the margin min |u0 - C_i| over the steps taken (for the near-tie exemption)."""
    p = np.exp(-nbar)
    cdf = p.copy()
    k = np.zeros(len(u0), dtype=np.int64)
    margin = np.abs(u0 - cdf)
    live = u0 > cdf
    while live.any():
        k = np.where(live & (k < 255), k + 1, k)
        p = np.where(live, p * nbar / np.maximum(k, 1), p)
        cdf = np.where(live, cdf + p, cdf)
        margin = np.where(live, np.minimum(margin, np.abs(u0 - cdf)), margin)
        live = live & (u0 > cdf) & (k < 255)
    return k, margin


# ---------------------------------------------------------------- the map
def field_kick(p, f):
    """(dpx_f, dpy_f): the Horner polynomial of knl/ksl at (x, y), k0l included (xline/elements.py:128-134)."""
    knl_in, ksl_in = f.get("knl", [0]), f.get("ksl", [0])
    order = max(len(knl_in), len(ksl_in)) - 1
    knl, ksl = xo._padded(knl_in, order + 1), xo._padded(ksl_in, order + 1)
    dpx, dpy = knl[order] + 0 * p.x, ksl[order] + 0 * p.x
    for ii in range(order, 0, -1):
        zre = (dpx * p.x - dpy * p.y) / ii
        zim = (dpx * p.y + dpy * p.x) / ii
        dpx, dpy = knl[ii - 1] + zre, ksl[ii - 1] + zim
    return dpx, dpy


def radiate_half(p, fl, lh, length, mode, seed, elem, half, log=None, consts=(K_E, HBAR_C, ALPHA)):
    """One half: the energy loss and its application (include/xline_b200.h).  ``consts``: (K_e, hbar c,
    alpha); ``p`` needs the oracle particles' columns, particle_id, at_turn and add_to_energy."""
    ke, hbarc, alpha = consts
    m2 = (p.energy0 - p.p0c) * (p.energy0 + p.p0c)
    opd = 1.0 + p.delta
    P = opd * p.p0c
    E = np.sqrt(P * P + m2)
    gamma = E / math.sqrt(m2)
    kappa = fl * (1.0 / length) / opd
    q2 = p.q0 * p.q0
    if mode == "mean":
        beta = P / E
        dE = -(2.0 / 3.0) * q2 * ke * (beta * beta * beta) * (gamma * gamma * gamma * gamma) * (kappa * kappa) * lh
        act = kappa != 0.0
        k = None
    else:
        u0, u1 = uniforms(seed, p.particle_id, p.at_turn, elem, half, 0)
        nbar = (5.0 / (2.0 * math.sqrt(3.0))) * q2 * alpha * gamma * kappa * lh
        k, margin = poisson_count(u0, nbar)
        sx = np.zeros(len(p.x))
        cur = (u0, u1)
        for m in range(1, int(k.max(initial=0)) + 1):
            if m % 2 == 0:
                cur = uniforms(seed, p.particle_id, p.at_turn, elem, half, m >> 1)
            sx = np.where(k >= m, sx + synrad_x(cur[1] if m & 1 else cur[0]), sx)
        dE = -(sx * (1.5 * hbarc * (gamma * gamma * gamma) * kappa))
        act = k > 0
        if log is not None:
            log.append(dict(elem=elem, half=half, pid=p.particle_id.copy(), turn=p.at_turn.copy(), k=k.copy(),
                            margin=margin, nbar=nbar, dE=dE.copy()))
    if mode == "mean" and log is not None:
        log.append(dict(elem=elem, half=half, pid=p.particle_id.copy(), turn=p.at_turn.copy(), dE=dE.copy()))
    old = dict(delta=p.delta.copy(), rpp=p.rpp.copy(), rvv=p.rvv.copy(), zeta=p.zeta.copy())
    p.add_to_energy(np.where(act, dE, 0.0))
    for key, v in old.items():
        setattr(p, key, np.where(act, getattr(p, key), v))
    fac = (1.0 + p.delta) / opd
    p.px = np.where(act, p.px * fac, p.px)
    p.py = np.where(act, p.py * fac, p.py)


def track_multipole_rad(p, f, mode, seed, elem, log=None):
    length = float(f.get("length", 0.0))
    hxl, hyl = float(f.get("hxl", 0.0)), float(f.get("hyl", 0.0))
    dpx, dpy = field_kick(p, f)
    fl = np.sqrt(dpx * dpx + dpy * dpy)
    lh = 0.5 * (length + hxl * p.x - hyl * p.y)
    radiate_half(p, fl, lh, length, mode, seed, elem, 0, log)
    xo.track_multipole(p, f)
    radiate_half(p, fl, lh, length, mode, seed, elem, 1, log)


def radiates(name, f):
    return name == "Multipole" and float(f.get("length", 0.0)) > 0


def line_track(specs, p, num_turns=1, radiation="mean", seed=0, log=None, element_offset=0, count_turns=True):
    """``xline_oracle.line_track`` (no monitors) with radiating multipoles."""
    for _ in range(num_turns):
        if len(p) == 0:
            break
        for iel, (name, f) in enumerate(specs):
            if name == "BeamMonitor":
                continue
            if radiation is not None and radiates(name, f):
                track_multipole_rad(p, f, radiation, seed, iel + element_offset, log)
                continue
            rec = xo.TRACKERS[name](p, f)
            if rec is not None:
                rec["at_element"][:] = iel + element_offset
                rec["state"][:] = 0
                if len(p) == 0:
                    break
        if count_turns:
            p.at_turn = p.at_turn + 1
    return p


def run_oracle(specs, cols, p0c, mass0, num_turns=1, radiation="mean", seed=0, log=None, q0=1.0):
    """Full-length result columns by particle id (``tests/helpers.run_oracle`` with radiation)."""
    n = len(next(iter(cols.values())))
    p = xo.OracleParticles(n, p0c=p0c, mass0=mass0, q0=q0, **cols)
    line_track(specs, p, num_turns=num_turns, radiation=radiation, seed=seed, log=log)
    return xo.gather_full(p, n)
