"""Packs a list of elements into the flat device lattice buffer of
``include/xline_b200.h`` (element type tags + fp64 parameters, cut into TMA-sized chunks).

Everything that depends only on element fields is evaluated here, once, on the host:
``2*pi*f/c`` and ``lag*pi/180`` of cavities (``xline/elements.py:241-243``), ``cos/sin`` of
``SRotation`` (``:380-382``), the ``DipoleEdge`` matrix entries (``:542-546``), the
Bassetti-Erskine prefactors (``be_beamfields/gaussian_fields.py:49-50``), the whole of
``BB6D_init`` (``be_beamfields/BB6Ddata.py:192-304``, which the reference redoes on every
``track`` call).  Physical constants come from ``scipy.constants`` at run time, as in the
reference (``xline/elements.py:2-5``) -- the kernel hard-codes none.

Two encodings (see the header): ``strict=False`` folds ``1/i!`` into the multipole
coefficients and reciprocals into aperture/curvature terms (FMA-friendly, the performance
path); ``strict=True`` keeps raw reference parameters for the strict kernel.
"""
import math

import numpy as np
from scipy.constants import c as clight
from scipy.constants import e as qe
from scipy.constants import epsilon_0
from scipy.constants import alpha as fine_structure
from scipy.constants import hbar

from . import elements as E

T_END_TURN, T_END_CHUNK, T_DRIFT, T_DRIFT_EXACT, T_MULTIPOLE, T_MULTIPOLE_CURVED = range(6)
T_CAVITY, T_RFMULTIPOLE, T_XYSHIFT, T_SROTATION, T_DIPOLE_EDGE = range(6, 11)
T_LIMIT_RECT, T_LIMIT_ELLIPSE, T_LIMIT_RECT_ELLIPSE, T_MONITOR, T_SAWTOOTH_CAVITY = range(11, 16)
T_BEAMBEAM4D, T_SPACECHARGE, T_BEAMBEAM6D, T_LIMIT_POLYGON, T_MULTIPOLE_RAD = 16, 17, 18, 19, 20
T_EXCITER = 0x40  # outside the contiguous single-element tags 0..20 (include/xline_b200.h)

F_STRICT = 1
F_BEAMFIELDS = 2
F_BB6D = 4
F_LOW_ORDER = 8  # every multipole-family record has order <= LOW_ORDER_MAX (straight-line Horner kernels)
F_POLYGONS = 16  # the lattice holds LIMIT_POLYGON records (only the kernels that carry the case run it)
F_RADIATION = 32  # the lattice holds MULTIPOLE_RAD records (only the kernels that carry the case run it)
F_EXCITER = 64  # the lattice holds EXCITER records and their data region after the chunks
RADIATION_MODES = {"mean": 1, "quantum": 2}
RAD_MAX_ELEMENTS = 1 << 24
LOW_ORDER_MAX = 3

DEFAULT_CHUNK_WORDS = 2048  # 16 KiB per TMA bulk copy, 3 in flight per CTA
MONITOR_FIELDS = ("x", "px", "y", "py", "zeta", "delta", "at_turn")

_FACT = [math.factorial(i) for i in range(64)]
MAX_ORDER = len(_FACT) - 1  # the highest multipole order the packer has coefficients for
EXCITER_MAX_SAMPLES = (1 << 31) - 1  # per Exciter (16 GiB of waveform): offsets and indices stay exact


def _f2u(x):
    return np.array([x], dtype=np.float64).view(np.uint64)[0]


def _i2u(i):
    return np.array([i], dtype=np.int64).view(np.uint64)[0]


AUX_DRIFT, AUX_DRIFT_EXACT = 0x10, 0x20  # aux bits of the LIMIT_* and SPACECHARGE records: fused drift
HDR_HX_ONLY = 1 << 31  # header flag: curved block record with hyl == 0 (fast encoding)
HDR_HAS_A1 = 1 << 30   # header flag: merged block with an aperture between its two kicks


def _hdr(tag, aux, idx, size_pairs=1, flags=0):
    assert 0 <= tag < 256 and 0 <= aux < 256 and 0 <= idx < (1 << 31)
    assert 1 <= size_pairs < (1 << 14), "record too large for the 14-bit size field"
    assert flags & ~(HDR_HX_ONLY | HDR_HAS_A1) == 0
    return np.uint64(tag | (aux << 8) | (size_pairs << 16) | flags | (idx << 32))


class _Rec:
    """One record under construction: header word + fp64/int64 words, padded to pairs."""

    def __init__(self, tag, aux, idx, first=0.0):
        self.tag, self.aux, self.idx = tag, aux, idx
        self.w = [np.uint64(0), _f2u(first)]
        self.flags = 0         # header flag bits (HDR_HX_ONLY)
        self.drift_len = 0.0   # by how much the record advances s
        self.drift_before = 0.0  # part of it that comes BEFORE the point a particle can be lost at
        self.s_word = None     # index of the word that receives the path length up to the record

    def path_length_here(self):
        """Reserve the next word for the path length from the start of the pass to this record
        (filled in by pack_line): what a particle lost here has travelled."""
        self.s_word = len(self.w)
        self.w.append(_f2u(0.0))
        return self

    def f(self, *vals):
        self.w.extend(_f2u(float(v)) for v in vals)
        return self

    def i(self, *vals):
        self.w.extend(_i2u(int(v)) for v in vals)
        return self

    def words(self):
        if len(self.w) & 1:
            self.w.append(np.uint64(0))
        self.w[0] = _hdr(self.tag, self.aux, self.idx, len(self.w) // 2, self.flags)
        return self.w


def _pad(seq, size):
    a = np.array(seq, dtype=np.float64).reshape(-1)
    if len(a) < size:
        a = np.concatenate([a, np.zeros(size - len(a))])
    return a


FIELD_BLOCK_PAIRS = {True: 3, False: 6}  # strict / fast encoding


def _gauss_field_block(rec, sigma_x, sigma_y, min_sigma_diff, strict):
    """The pairs describing a frozen 2-D Gaussian of fixed sigmas
    (be_beamfields/gaussian_fields.py:107-121, 5-21, 29-99): ``[sx, sy][kind, 0][A, 0]`` and,
    in the fast encoding, three more pairs with everything Bassetti-Erskine needs that depends
    on the sigmas only -- ``[1/S, A sqrt(pi)/S][small/big, big/small][1/(2 big^2), 1/(2 small^2)]``
    -- so that the kernel spends no square root and no division on them per particle."""
    inv2pieps0 = 1.0 / (2.0 * math.pi * epsilon_0)
    if abs(sigma_x - sigma_y) < min_sigma_diff:
        rec.f(sigma_x, sigma_y).i(0, 0).f(inv2pieps0, 0.0)
        if not strict:
            rec.f(0.0, 0.0).f(0.0, 0.0).f(0.0, 0.0)
        return
    if sigma_x == sigma_y:
        # gaussian_fields.py:91-92 -> 1.0/0.0 (tests/test_beamfields.py:86-98)
        raise ZeroDivisionError("float division by zero")
    rec.f(sigma_x, sigma_y).i(1 if sigma_x > sigma_y else 2, 0).f(inv2pieps0, 0.0)
    if not strict:
        big, small = max(sigma_x, sigma_y), min(sigma_x, sigma_y)
        S = math.sqrt(2.0 * (big * big - small * small))
        inv_s = 1.0 / S
        rec.f(inv_s, inv2pieps0 * 1.772453850905516 * inv_s)
        rec.f(small / big, big / small)
        rec.f(1.0 / (2.0 * big * big), 1.0 / (2.0 * small * small))


def _pack_beambeam4d(el, idx, strict):
    """be_beamfields/beambeam.py:45-82: min_sigma_diff hard-coded to 1e-10 (:63)."""
    rec = _Rec(T_BEAMBEAM4D, 0, idx)
    rec.f(el.x_bb, el.y_bb)
    _gauss_field_block(rec, float(el.sigma_x), float(el.sigma_y), 1e-10, strict)
    rec.f(el.d_px, el.d_py)
    rec.f(el.beta_r, float(el.charge) * qe)
    return rec


def _qgauss_cq(q, eps=1e-6):
    """be_beamfields/qgauss.py:5-21."""
    from scipy.special import gamma as tgamma

    assert q < 3
    cq = math.sqrt(math.pi)
    if q >= (1 + eps):
        cq *= tgamma((3 - q) / (2 * q - 2))
        cq /= math.sqrt((q - 1)) * tgamma(1 / (q - 1))
    elif q <= (1 - eps):
        cq *= 2 * tgamma(1 / (1 - q))
        cq /= (3 - q) * math.sqrt(1 - q) * tgamma((3 - q) / (2 - 2 * q))
    return cq


def _pack_spacecharge(el, idx, strict):
    """be_beamfields/spacecharge.py:26-52, 80-104, 137-177."""
    name = type(el).__name__
    if name == "SCCoasting":
        kind = 0
    elif name == "SCQGaussProfile":
        kind = 1
    else:
        kind = {0: 2, 1: 3}.get(int(el.method), 0)
    rec = _Rec(T_SPACECHARGE, kind, idx)
    rec.f(el.x_co, el.y_co)
    _gauss_field_block(rec, float(el.sigma_x), float(el.sigma_y), float(el.min_sigma_diff), strict)
    base = float(el.number_of_particles) * qe * float(el.length)
    if name == "SCCoasting":
        rec.f(base / float(el.circumference), 0.0)
    elif name == "SCQGaussProfile":
        q = float(el.q_parameter)
        assert q < 3
        assert el.bunchlength_rms > 0
        sqrt_beta = 1 / (math.sqrt(2) * float(el.bunchlength_rms))
        cq = _qgauss_cq(q)
        assert abs(cq) > 0
        gauss = not (abs(1 - q) > 1e-6)
        rec.f(base, sqrt_beta * sqrt_beta)
        rec.f(sqrt_beta / cq, 1.0 - q)
        rec.f(0.0 if gauss else 1.0 / (1.0 - q), 0.0).i(1 if gauss else 0, 0)
    else:
        prof = np.asarray(el.line_density_profile, dtype=np.float64)
        n = len(prof)
        if kind == 0:  # method not in (0, 1): ld_factor = 1 (spacecharge.py:173)
            rec.f(base, 0.0)
        else:
            rec.f(base, float(el.z0)).f(float(el.dz), 0.0).i(n, 0)
            if kind == 2:
                rec.f(*prof)
            else:
                from scipy.interpolate import CubicSpline

                absc = np.linspace(el.z0, el.z0 + el.dz * (n - 1), n)
                cs = CubicSpline(absc, prof)
                # per interval: c3, c2, c1, c0 of (z - x_i) and the knot x_i
                rec.f(*absc)
                for k in range(4):
                    rec.f(*cs.c[k])
    return rec


def _boost_scalar(x, px, y, py, sigma, delta, pb):
    """be_beamfields/boost.py:6-49 for Python floats."""
    sphi, cphi, tphi, salpha, calpha = pb
    h = delta + 1.0 - math.sqrt((1.0 + delta) * (1.0 + delta) - px * px - py * py)
    px_st = px / cphi - h * calpha * tphi / cphi
    py_st = py / cphi - h * salpha * tphi / cphi
    delta_st = delta - px * calpha * tphi - py * salpha * tphi + h * tphi * tphi
    pz_st = math.sqrt((1.0 + delta_st) * (1.0 + delta_st) - px_st * px_st - py_st * py_st)
    hx_st = px_st / pz_st
    hy_st = py_st / pz_st
    hsigma_st = 1.0 - (delta_st + 1) / pz_st
    L11 = 1.0 + hx_st * calpha * sphi
    L12 = hx_st * salpha * sphi
    L13 = calpha * tphi
    L21 = hy_st * calpha * sphi
    L22 = 1.0 + hy_st * salpha * sphi
    L23 = salpha * tphi
    L31 = hsigma_st * calpha * sphi
    L32 = hsigma_st * salpha * sphi
    L33 = 1.0 / cphi
    return (
        L11 * x + L12 * y + L13 * sigma,
        L21 * x + L22 * y + L23 * sigma,
        L31 * x + L32 * y + L33 * sigma,
    )


def _pack_beambeam6d(el, idx):
    """be_beamfields/beambeam.py:219-283 + BB6Ddata.py:192-304 (BB6D_init hoisted here)."""
    z = np.atleast_1d(np.asarray(el.zeta_slices, dtype=np.float64))
    npart = np.atleast_1d(np.asarray(el.charge_slices, dtype=np.float64))
    assert len(z) == len(npart)
    order = np.argsort(z)[::-1]  # head of the strong beam first (BB6Ddata.py:250-252)
    z, npart = np.take(z, order), np.take(npart, order)
    phi, alpha = float(el.phi), float(el.alpha)
    pb = (math.sin(phi), math.cos(phi), math.tan(phi), math.sin(alpha), math.cos(alpha))
    cphi = pb[1]
    rec = _Rec(T_BEAMBEAM6D, 0, idx, float(len(z)))
    rec.f(pb[0], pb[1]).f(pb[2], pb[3]).f(pb[4], 0.0)
    # boosted Sigma matrix (BB6Ddata.py:62-75)
    rec.f(el.sigma_11, el.sigma_12 / cphi)
    rec.f(el.sigma_13, el.sigma_14 / cphi)
    rec.f(el.sigma_22 / cphi / cphi, el.sigma_23 / cphi)
    rec.f(el.sigma_24 / cphi / cphi, el.sigma_33)
    rec.f(el.sigma_34 / cphi, el.sigma_44 / cphi / cphi)
    rec.f(el.min_sigma_diff, el.threshold_singular)
    rec.f(el.x_co, el.px_co).f(el.y_co, el.py_co).f(el.zeta_co, el.delta_co)
    rec.f(el.x_bb_co, el.y_bb_co)
    rec.f(el.d_x, el.d_px).f(el.d_y, el.d_py).f(el.d_zeta, el.d_delta)
    rec.f(qe, 1.0 / (2.0 * math.pi * epsilon_0))
    for zi, ni in zip(z, npart):
        xs, ys, ss = _boost_scalar(0.0, 0.0, 0.0, 0.0, float(zi), 0.0, pb)
        rec.f(ni, xs).f(ys, ss)
    return rec


def _is_noop(el, name):
    if name in ("Drift", "DriftExact"):
        return el.length == 0
    if name == "Multipole":
        return (not np.any(np.asarray(el.knl, dtype=float)) and
                not np.any(np.asarray(el.ksl, dtype=float)) and el.hxl == 0 and el.hyl == 0)
    if name == "XYShift":
        return el.dx == 0 and el.dy == 0
    if name == "SRotation":
        return el.angle == 0
    if name in ("BeamBeam4D", "BeamBeam6D", "SCCoasting", "SCQGaussProfile", "SCInterpolatedProfile"):
        return not el.enabled  # `if self.enabled:` beambeam.py:46,220; spacecharge.py:27,81,138
    return False


def polygon_edges(x_vertices, y_vertices):
    """The edges a LIMIT_POLYGON record stores, ``[(y_lo, y_hi, x_lo, slope), ...]`` in vertex
    order (include/xline_b200.h): every edge V_k -> V_(k+1) mod n that is not horizontal, from
    its lower end, with ``slope = (x_hi - x_lo) / (y_hi - y_lo)`` rounded once here.  Raises
    ``ValueError`` for a polygon the predicate is not defined for."""
    xv = [float(v) for v in x_vertices]
    yv = [float(v) for v in y_vertices]
    if len(xv) != len(yv) or len(xv) < 3:
        raise ValueError("LimitPolygon needs x_vertices and y_vertices of the same length >= 3 "
                         "(got %d and %d)" % (len(xv), len(yv)))
    if not all(math.isfinite(v) for v in xv + yv):
        raise ValueError("LimitPolygon has a non-finite vertex")
    edges = []
    n = len(xv)
    for k in range(n):
        x0, y0, x1, y1 = xv[k], yv[k], xv[(k + 1) % n], yv[(k + 1) % n]
        if y0 == y1:
            continue  # horizontal: never crossed
        if y1 < y0:
            x0, y0, x1, y1 = x1, y1, x0, y0
        slope = (x1 - x0) / (y1 - y0)
        if not math.isfinite(slope):
            raise ValueError("LimitPolygon edge %d has a non-finite slope" % k)
        edges.append((y0, y1, x0, slope))
    if not edges:
        raise ValueError("LimitPolygon has no edge that is not horizontal")
    return edges


def _pack_limit_polygon(el, idx):
    """XLB_T_LIMIT_POLYGON: [hdr,n_edges][s_here,drift_length] then [y_lo,y_hi][x_lo,slope] per
    stored edge; the same words in both encodings."""
    edges = polygon_edges(el.x_vertices, el.y_vertices)
    rec = _Rec(T_LIMIT_POLYGON, 0, idx)
    rec.w[1] = _i2u(len(edges))
    rec.path_length_here().f(0.0)  # word 3: the length of a fused drift (pack_line)
    for y_lo, y_hi, x_lo, slope in edges:
        rec.f(y_lo, y_hi).f(x_lo, slope)
    return rec


def radiation_constants():
    """(K_e = e^2/(4 pi eps0), hbar c) in eV m and the fine-structure constant, from scipy.constants."""
    return qe / (4.0 * math.pi * epsilon_0), hbar * clight / qe, fine_structure


def check_radiation(radiation, radiation_seed):
    """The radiation options: None, "mean" or "quantum", and a seed in [0, 2^64)."""
    if radiation is not None and radiation not in RADIATION_MODES:
        raise ValueError("radiation must be None, 'mean' or 'quantum' (got %r)" % (radiation,))
    if not (isinstance(radiation_seed, (int, np.integer)) and 0 <= int(radiation_seed) < (1 << 64)):
        raise ValueError("radiation_seed must be an integer in [0, 2^64) (got %r)" % (radiation_seed,))


def radiates(el, radiation):
    """Does ``el`` radiate when the line is tracked with ``radiation``: a Multipole with length > 0."""
    return radiation is not None and type(el).__name__ == "Multipole" and float(el.length) > 0


def _pack_multipole_rad(el, idx, radiation, seed):
    """XLB_T_MULTIPOLE_RAD: [hdr,mode][L,1/L][K_e,hbar_c][alpha,seed] then the element's own
    (fast-encoding) MULTIPOLE / MULTIPOLE_CURVED record, header word included."""
    plain = _pack_element(el, idx, False, None)
    length = float(el.length)
    ke, hbarc, alpha = radiation_constants()
    rec = _Rec(T_MULTIPOLE_RAD, plain.aux, idx)
    rec.w[1] = _i2u(RADIATION_MODES[radiation])
    rec.f(length, 1.0 / length).f(ke, hbarc).f(alpha)
    rec.w.append(np.uint64(int(seed)))
    rec.w.extend(plain.words())
    return rec


def _finite_floats(values, what):
    a = np.array(values, dtype=np.float64).reshape(-1)
    if not np.all(np.isfinite(a)):
        raise ValueError("Exciter has a non-finite %s" % what)
    return a


def _pack_exciter(el, idx, data):
    """XLB_T_EXCITER: [hdr,A][B,start_turn][n_samples,data_offset] then (kn_i,ks_i) i=order..0, with
    A = sampling_frequency/frev, B = sampling_frequency/c.  The samples are appended to ``data`` (the
    data region); ``data_offset`` is relative to the region here and made absolute by pack_line."""
    fs, frev = float(el.sampling_frequency), float(el.frev)
    if not (math.isfinite(fs) and fs > 0 and math.isfinite(frev) and frev > 0):
        raise ValueError("Exciter needs finite sampling_frequency > 0 and frev > 0 (got %r, %r)"
                         % (el.sampling_frequency, el.frev))
    if isinstance(el.start_turn, bool) or not isinstance(el.start_turn, (int, np.integer)) or \
            not -(1 << 62) <= int(el.start_turn) < (1 << 62):
        raise ValueError("Exciter.start_turn must be an integer (got %r)" % (el.start_turn,))
    if len(el.samples) > EXCITER_MAX_SAMPLES:
        raise ValueError("Exciter has %d samples, more than the %d a record can address"
                         % (len(el.samples), EXCITER_MAX_SAMPLES))
    samples = _finite_floats(el.samples, "sample")
    order = el.order
    if order > MAX_ORDER:
        raise ValueError("Exciter of order %d: the highest order is %d" % (order, MAX_ORDER))
    knl = _pad(_finite_floats(el.knl, "knl"), order + 1)
    ksl = _pad(_finite_floats(el.ksl, "ksl"), order + 1)
    rec = _Rec(T_EXCITER, order, idx, fs / frev)
    rec.f(fs / clight).i(int(el.start_turn), len(samples), sum(len(d) for d in data))
    for i in range(order, -1, -1):
        rec.f(knl[i] / _FACT[i], ksl[i] / _FACT[i])
    data.append(samples)
    return rec


def _pack_element(el, idx, strict, monitors, polygons=False, data=None):
    name = type(el).__name__
    if name == "Drift":
        rec = _Rec(T_DRIFT, 0, idx, el.length)
        rec.drift_len = float(el.length)
        return rec
    if name == "DriftExact":
        rec = _Rec(T_DRIFT_EXACT, 0, idx, el.length)
        rec.drift_len = float(el.length)
        return rec
    if name == "Multipole":
        order = el.order
        knl, ksl = _pad(el.knl, order + 1), _pad(el.ksl, order + 1)
        curved = (el.hxl != 0 or el.hyl != 0)
        if curved:
            rec = _Rec(T_MULTIPOLE_CURVED, order, idx, el.hxl)
            rec.f(el.hyl, el.length)
            rec.f(1.0 / el.length if el.length > 0 else 0.0, 0.0)
        else:
            rec = _Rec(T_MULTIPOLE, order, idx)
        for i in range(order, -1, -1):
            if strict:
                rec.f(knl[i], ksl[i])
            else:
                rec.f(knl[i] / _FACT[i], ksl[i] / _FACT[i])
        return rec
    if name in ("Cavity", "SawtoothCavity"):
        tag = T_CAVITY if name == "Cavity" else T_SAWTOOTH_CAVITY
        k = 2 * np.pi * el.frequency / clight
        return _Rec(tag, 0, idx, el.voltage).f(k, el.lag * np.pi / 180)
    if name == "RFMultipole":
        order = el.order
        deg2rad = np.pi / 180
        k = 2 * np.pi * el.frequency / clight
        rec = _Rec(T_RFMULTIPOLE, order, idx, el.voltage).f(k, el.lag * deg2rad)
        knl, ksl = _pad(el.knl, order + 1), _pad(el.ksl, order + 1)
        pn, ps = _pad(el.pn, order + 1) * deg2rad, _pad(el.ps, order + 1) * deg2rad
        for i in range(order + 1):
            rec.f(knl[i], ksl[i]).f(pn[i], ps[i])
        return rec
    if name == "XYShift":
        return _Rec(T_XYSHIFT, 0, idx, el.dx).f(el.dy, 0.0)
    if name == "SRotation":
        deg2rad = np.pi / 180
        return _Rec(T_SROTATION, 0, idx, np.cos(el.angle * deg2rad)).f(np.sin(el.angle * deg2rad), 0.0)
    if name == "DipoleEdge":
        corr = 2 * el.h * el.hgap * el.fint
        r21 = el.h * np.tan(el.e1)
        r43 = -el.h * np.tan(el.e1 - corr / np.cos(el.e1) * (1 + np.sin(el.e1) ** 2))
        return _Rec(T_DIPOLE_EDGE, 0, idx, r21).f(r43, 0.0)
    if name == "LimitRect":
        sym = (not strict) and el.min_x == -el.max_x and el.min_y == -el.max_y
        return _Rec(T_LIMIT_RECT, 1 if sym else 0, idx, el.min_x).f(el.max_x, el.min_y).f(el.max_y).path_length_here()
    if name == "LimitEllipse":
        a2, b2 = el.a * el.a, el.b * el.b
        return _Rec(T_LIMIT_ELLIPSE, 0, idx, a2).f(b2, 1.0 / a2).f(1.0 / b2).path_length_here()
    if name == "LimitRectEllipse":
        a2, b2 = el.a * el.a, el.b * el.b
        return _Rec(T_LIMIT_RECT_ELLIPSE, 0, idx, el.max_x).f(el.max_y, a2).f(b2, 1.0 / a2).f(1.0 / b2).path_length_here()
    if name == "BeamMonitor":
        assert el.is_turn_ordered  # xline/elements.py:504
        nn = el.max_particle_id - el.min_particle_id + 1 if el.max_particle_id >= el.min_particle_id else 0
        off = monitors["words"]
        slot = dict(element_index=idx, offset=off, num_stores=int(el.num_stores), nn=int(nn))
        monitors["layout"].append(slot)
        monitors["words"] += len(MONITOR_FIELDS) * max(int(el.num_stores), 0) * max(int(nn), 0)
        rec = _Rec(T_MONITOR, len(monitors["layout"]) - 1, idx)
        rec.i(el.start, max(int(el.skip), 1)).i(el.num_stores, el.min_particle_id)
        rec.i(el.max_particle_id, 1 if el.is_rolling else 0).i(off, 0)
        return rec
    if name == "BeamBeam4D":
        return _pack_beambeam4d(el, idx, strict)
    if name in ("SCCoasting", "SCQGaussProfile", "SCInterpolatedProfile"):
        return _pack_spacecharge(el, idx, strict)
    if name == "BeamBeam6D":
        return _pack_beambeam6d(el, idx)
    if name == "Exciter":
        if strict:
            raise ValueError("Exciter: the strict encoding has no exciter records (track with strict=False)")
        return _pack_exciter(el, idx, data)
    if name == "LimitPolygon":
        if polygons:
            return _pack_limit_polygon(el, idx)
        # the reference's LimitPolygon.track raises (xline/elements.py:483); tracking one is opt-in
        raise NotImplementedError("LimitPolygon apertures are tracked only on request: set "
                                  "Line.polygon_apertures = True (pack_line(..., polygons=True))")
    raise ValueError("element type %s is not supported by the B200 tracking kernel" % name)


class PackedLattice:
    """Result of :func:`pack_line`: ``words`` (uint64 numpy array, chunked) + metadata."""

    def __init__(self, words, chunk_words, n_chunks, n_elements, flags, monitors, counts, segments=None):
        # int32 [n_segments, 3] = first_chunk, n_chunks, kind (xlb_lattice_t::segments) or None
        self.segments = None if segments is None else np.ascontiguousarray(segments, dtype=np.int32)
        self.words = words
        self.chunk_words = chunk_words
        self.n_chunks = n_chunks
        self.n_elements = n_elements
        self.flags = flags
        self.monitor_layout = monitors["layout"]
        self.monitor_words = monitors["words"]
        self.record_counts = counts  # tag -> number of records actually packed

    @property
    def strict(self):
        return bool(self.flags & F_STRICT)

    # ---- on-disk form of the packed lattice (SURVEY.md §8f-3): the chunked words plus the
    # header fields of xlb_lattice_t; reload with PackedLattice.load and hand to the C ABI
    def save(self, path):
        np.savez_compressed(
            path, words=self.words, chunk_words=self.chunk_words, n_chunks=self.n_chunks,
            n_elements=self.n_elements, flags=self.flags, monitor_words=self.monitor_words,
            monitor_layout=np.array([[m["element_index"], m["offset"], m["num_stores"], m["nn"]]
                                     for m in self.monitor_layout], dtype=np.int64).reshape(-1, 4),
            record_tags=np.array(sorted(self.record_counts), dtype=np.int64),
            record_counts=np.array([self.record_counts[k] for k in sorted(self.record_counts)], dtype=np.int64),
            segments=(np.zeros((0, 3), dtype=np.int32) if self.segments is None else self.segments))

    @classmethod
    def load(cls, path):
        d = np.load(path)
        layout = [dict(element_index=int(r[0]), offset=int(r[1]), num_stores=int(r[2]), nn=int(r[3]))
                  for r in d["monitor_layout"]]
        counts = {int(k): int(v) for k, v in zip(d["record_tags"], d["record_counts"])}
        return cls(np.ascontiguousarray(d["words"], dtype=np.uint64), int(d["chunk_words"]), int(d["n_chunks"]),
                   int(d["n_elements"]), int(d["flags"]), dict(layout=layout, words=int(d["monitor_words"])), counts,
                   d["segments"] if "segments" in d and len(d["segments"]) else None)

    def c_lattice(self, words_ptr=None):
        """The ``xlb_lattice_t`` for these words (``words_ptr``: a device copy; default the
        host array).  The segment table stays host memory owned by this object."""
        from . import _cabi

        lat = _cabi.Lattice(self.words.ctypes.data if words_ptr is None else words_ptr, self.words.size,
                            self.chunk_words, self.n_chunks, self.n_elements, self.flags)
        if self.segments is not None:
            lat.n_segments = int(self.segments.shape[0])
            lat.segments = self.segments.ctypes.data
        return lat

    @property
    def nbytes(self):
        return int(self.words.nbytes)


T_THIN_BLOCK = 0x80  # tag family: | aperture kind (bits 0-1) | curved << 2 | drift << 3 | exact << 4
AP_NONE, AP_RECT_SYM, AP_RECT, AP_ELLIPSE = 0, 1, 2, 3
TB_CURVED, TB_DRIFT, TB_DRIFT_EXACT = 4, 8, 16


def _pack_thin_block(mp, idx, aper, drift, strict):
    """Fused record of the XLB_T_THIN_BLOCK family: the multipole's kick, then the aperture
    test, then the drift -- the same maps in the same order as the separate elements."""
    order = mp.order
    knl, ksl = _pad(mp.knl, order + 1), _pad(mp.ksl, order + 1)
    tag = T_THIN_BLOCK
    aper_idx = 0
    curved = mp.hxl != 0 or mp.hyl != 0
    if curved:
        tag |= TB_CURVED
    lim = None
    if aper is not None:
        aper_idx, ap = aper
        if type(ap).__name__ == "LimitRect":
            sym = (not strict) and ap.min_x == -ap.max_x and ap.min_y == -ap.max_y
            tag |= AP_RECT_SYM if sym else AP_RECT
            lim = (ap.min_x, ap.max_x, ap.min_y, ap.max_y)
        else:
            tag |= AP_ELLIPSE
            a2, b2 = ap.a * ap.a, ap.b * ap.b
            lim = (a2, b2, 1.0 / a2, 1.0 / b2)
    if drift is not None:
        tag |= TB_DRIFT
        if type(drift[1]).__name__ == "DriftExact":
            tag |= TB_DRIFT_EXACT
    rec = _Rec(tag, order, idx, drift[1].length if drift is not None else 0.0)
    rec.drift_len = float(drift[1].length) if drift is not None else 0.0
    if curved and mp.hyl == 0 and not strict:
        rec.flags |= HDR_HX_ONLY
    rec.i(aper_idx).path_length_here()
    for i in range(order, -1, -1):
        if strict:
            rec.f(knl[i], ksl[i])
        else:
            rec.f(knl[i] / _FACT[i], ksl[i] / _FACT[i])
    if curved:
        rec.f(mp.hxl, mp.hyl).f(mp.length, 1.0 / mp.length if mp.length > 0 else 0.0)
    if lim is not None:
        rec.f(*lim)
    return rec


T_MERGED_BLOCK = 0xA0  # thin-block bits | 0x20: two co-located multipoles as one (fast only)
T_EDGE_BLOCK = 0xC0    # dipole edge -> drift
MERGE_MAX_K1_ORDER = 4


def _pack_merged_block(k1, idx1, a1, k2, idx2, a2, drift):
    """XLB_T_MERGED_BLOCK: [K1][A1 ellipse?][K2][A2?][drift?] with the two thin kicks summed
    into one coefficient set (fast encoding only; see include/xline_b200.h)."""
    order = max(k1.order, k2.order)
    kn = _pad(k1.knl, order + 1) + _pad(k2.knl, order + 1)
    ks = _pad(k1.ksl, order + 1) + _pad(k2.ksl, order + 1)
    tag = T_MERGED_BLOCK
    curved = k2.hxl != 0 or k2.hyl != 0
    if curved:
        tag |= TB_CURVED
    lim2 = None
    a2_idx = 0
    if a2 is not None:
        a2_idx, ap = a2
        if type(ap).__name__ == "LimitRect":
            sym = ap.min_x == -ap.max_x and ap.min_y == -ap.max_y
            tag |= AP_RECT_SYM if sym else AP_RECT
            lim2 = (ap.min_x, ap.max_x, ap.min_y, ap.max_y)
        else:
            tag |= AP_ELLIPSE
            aa, bb = ap.a * ap.a, ap.b * ap.b
            lim2 = (aa, bb, 1.0 / aa, 1.0 / bb)
    if drift is not None:
        tag |= TB_DRIFT
        if type(drift[1]).__name__ == "DriftExact":
            tag |= TB_DRIFT_EXACT
    rec = _Rec(tag, order, idx2, drift[1].length if drift is not None else 0.0)
    rec.drift_len = float(drift[1].length) if drift is not None else 0.0
    if curved and k2.hyl == 0:
        rec.flags |= HDR_HX_ONLY
    a1_idx = a1[0] if a1 is not None else 0
    if a1 is not None:
        rec.flags |= HDR_HAS_A1
    rec.i(a1_idx | (a2_idx << 32), k1.order | ((1 if a1 is not None else 0) << 8))
    for i in range(order, -1, -1):
        rec.f(kn[i] / _FACT[i], ks[i] / _FACT[i])
    if curved:
        rec.f(k2.hxl, k2.hyl).f(k2.length, 1.0 / k2.length if k2.length > 0 else 0.0)
        rec.f(_pad(k2.knl, 1)[0], _pad(k2.ksl, 1)[0])
    if a1 is not None:
        aa, bb = a1[1].a * a1[1].a, a1[1].b * a1[1].b
        rec.f(aa, bb, 1.0 / aa, 1.0 / bb)
    if lim2 is not None:
        rec.f(*lim2)
    k1n, k1s = _pad(k1.knl, k1.order + 1), _pad(k1.ksl, k1.order + 1)
    for i in range(k1.order, -1, -1):
        rec.f(k1n[i] / _FACT[i], k1s[i] / _FACT[i])
    return rec.path_length_here()


def _try_merge(live, pos, radiation=None):
    """Match [K1 straight, low order][LimitEllipse?][K2][LimitRect|LimitEllipse?][Drift?]
    starting at live[pos]; returns (record, new_pos) or None.  Radiating multipoles do not merge."""
    def kind(i):
        return type(live[i][1]).__name__ if i < len(live) else None

    idx1, k1 = live[pos]
    if k1.hxl != 0 or k1.hyl != 0 or k1.order > MERGE_MAX_K1_ORDER:
        return None
    i = pos + 1
    a1 = None
    if kind(i) == "LimitEllipse":
        a1 = live[i]
        i += 1
    if kind(i) != "Multipole" or radiates(live[i][1], radiation):
        return None
    idx2, k2 = live[i]
    i += 1
    a2 = None
    if kind(i) in ("LimitRect", "LimitEllipse"):
        a2 = live[i]
        i += 1
    drift = None
    if kind(i) in ("Drift", "DriftExact"):
        drift = live[i]
        i += 1
    return _pack_merged_block(k1, idx1, a1, k2, idx2, a2, drift), i


SEG_MAIN, SEG_BB6D = 0, 1


def pack_line(elements, strict=False, chunk_words=DEFAULT_CHUNK_WORDS, drop_noops=True, fuse=True,
              merge=True, split_lenses=True, hx_only=True, polygons=False, radiation=None, radiation_seed=0):
    """Pack ``elements`` (the ``Line.elements`` list).  ``element_index`` in every record
    is the position in that list, so ``at_element`` matches the reference's indexing even
    though exact no-ops (zero-length drifts, all-zero multipoles, disabled lenses) are not
    emitted.

    ``split_lenses`` (fast encoding only): every BeamBeam6D record gets a chunk of its own
    and the lattice becomes a sequence of segments -- tracking-kernel segments separated by
    6D-lens segments (``xlb_lattice_t::segments``) -- so that the tracking kernels need not
    carry the register-hungry 6D lens.

    ``hx_only`` (fast encoding only): flag curved block records whose ``hyl`` is exactly zero with
    ``XLB_HDR_HX_ONLY`` so that the kernel leaves the ``hyl`` terms out (same bits, fewer
    instructions); ``False`` packs them for the general formula (the tests compare the two).

    ``polygons``: pack ``LimitPolygon`` apertures as XLB_T_LIMIT_POLYGON records (the project's
    own definition, see include/xline_b200.h).  ``False``, the default, refuses them with
    ``NotImplementedError`` like the reference's ``LimitPolygon.track``.

    ``Exciter`` elements pack as XLB_T_EXCITER records, their samples into a data region after the
    chunks (``words`` holds ``chunk_words * n_chunks`` words, then the samples); fast encoding only
    (``ValueError`` for ``strict=True``), and such a line keeps its BeamBeam6D lenses in the tracking
    kernel (no ``split_lenses``): a segment's kernel could not address the data region.

    ``radiation`` (None, "mean" or "quantum") and ``radiation_seed``: synchrotron radiation in every
    Multipole of length > 0, packed as XLB_T_MULTIPOLE_RAD records that never enter a block
    (include/xline_b200.h, DESIGN.md §4.9).  Fast encoding, one-species thin-lens lattices only:
    ``ValueError`` for ``strict=True``, beam-field elements, or more than 2^24 elements."""
    assert chunk_words % 2 == 0 and chunk_words >= 16
    check_radiation(radiation, radiation_seed)
    if radiation is not None:
        if strict:
            raise ValueError("radiation: the strict encoding has no radiating multipoles (set radiation=None)")
        if len(elements) > RAD_MAX_ELEMENTS:
            raise ValueError("radiation: lines of more than 2^24 elements are not supported")
    monitors = dict(layout=[], words=0)
    data = []  # the exciters' samples, in record order: the data region
    recs = []
    flags = F_STRICT if strict else 0
    counts = {}
    live = [(idx, el) for idx, el in enumerate(elements)
            if not (drop_noops and _is_noop(el, type(el).__name__))]
    pos = 0
    while pos < len(live):
        idx, el = live[pos]
        pos += 1
        name = type(el).__name__
        if fuse and name == "DipoleEdge" and pos < len(live) and \
                type(live[pos][1]).__name__ in ("Drift", "DriftExact"):
            # dipole edge -> drift in one record
            d = live[pos][1]
            pos += 1
            plain = _pack_element(el, idx, strict, monitors)
            rec = _Rec(T_EDGE_BLOCK | TB_DRIFT | (TB_DRIFT_EXACT if type(d).__name__ == "DriftExact" else 0),
                       0, idx, d.length)
            rec.w.extend([plain.w[1], plain.w[2]])  # r21, r43 as evaluated for the plain record
            rec.drift_len = float(d.length)
            counts[rec.tag] = counts.get(rec.tag, 0) + 1
            recs.append((rec.tag, rec.words(), rec.s_word, rec.drift_len, rec.drift_before))
            continue
        nxt = type(live[pos][1]).__name__ if pos < len(live) else None
        if fuse and name in ("LimitRect", "LimitEllipse", "LimitRectEllipse", "LimitPolygon") and \
                nxt in ("Drift", "DriftExact"):
            # aperture -> drift in one record (aux bit 4; the drift length in a pair of its own,
            # in word 3 of a polygon record)
            d = live[pos][1]
            pos += 1
            rec = _pack_element(el, idx, strict, monitors, polygons)
            rec.aux |= AUX_DRIFT | (AUX_DRIFT_EXACT if nxt == "DriftExact" else 0)
            if rec.tag == T_LIMIT_POLYGON:
                rec.w[3] = _f2u(float(d.length))
            else:
                rec.f(d.length, 0.0)
            rec.drift_len = float(d.length)
            counts[rec.tag] = counts.get(rec.tag, 0) + 1
            recs.append((rec.tag, rec.words(), rec.s_word, rec.drift_len, rec.drift_before))
            continue
        if fuse and name in ("SCCoasting", "SCQGaussProfile", "SCInterpolatedProfile") and nxt in ("Drift", "DriftExact"):
            # space-charge kick -> drift in one record (aux bit 4; the drift length in word 1)
            d = live[pos][1]
            pos += 1
            rec = _pack_element(el, idx, strict, monitors)
            rec.aux |= AUX_DRIFT | (AUX_DRIFT_EXACT if nxt == "DriftExact" else 0)
            rec.w[1] = _f2u(float(d.length))
            rec.drift_len = float(d.length)
            counts[rec.tag] = counts.get(rec.tag, 0) + 1
            recs.append((rec.tag, rec.words(), rec.s_word, rec.drift_len, rec.drift_before))
            continue
        rad = radiates(el, radiation)
        merged = (_try_merge(live, pos - 1, radiation) if (fuse and merge and not strict and name == "Multipole"
                                                            and not rad) else None)
        if rad:
            rec = _pack_multipole_rad(el, idx, radiation, radiation_seed)
        elif merged is not None:
            # two co-located thin multipoles (apertures in between allowed): one summed kick
            rec, pos = merged
        elif fuse and name == "Multipole":
            # peephole: thin multipole -> [LimitRect | LimitEllipse] -> [Drift] in one record
            aper = drift = None
            if pos < len(live) and type(live[pos][1]).__name__ in ("LimitRect", "LimitEllipse"):
                aper = live[pos]
                pos += 1
            if pos < len(live) and type(live[pos][1]).__name__ in ("Drift", "DriftExact"):
                drift = live[pos]
                pos += 1
            rec = _pack_thin_block(el, idx, aper, drift, strict)
        else:
            rec = _pack_element(el, idx, strict, monitors, polygons, data)
        tag = rec.tag
        counts[tag] = counts.get(tag, 0) + 1
        if not hx_only:
            rec.flags &= ~HDR_HX_ONLY
        recs.append((tag, rec.words(), rec.s_word, rec.drift_len, rec.drift_before))
    exciters = any(r[0] == T_EXCITER for r in recs)
    split = bool(split_lenses) and not strict and not exciters and any(r[0] == T_BEAMBEAM6D for r in recs)
    for tag, _, _, _, _ in recs:
        if tag == T_BEAMBEAM6D:
            flags |= F_BB6D
        if tag in (T_BEAMBEAM4D, T_SPACECHARGE) or (tag == T_BEAMBEAM6D and not split):
            flags |= F_BEAMFIELDS
        if tag == T_LIMIT_POLYGON:
            flags |= F_POLYGONS
        if tag == T_MULTIPOLE_RAD:
            flags |= F_RADIATION
        if tag == T_EXCITER:
            flags |= F_EXCITER
    if (flags & F_RADIATION) and (flags & (F_BEAMFIELDS | F_BB6D)):
        raise ValueError("radiation: lines with beam-beam or space-charge elements are not supported "
                         "(set radiation=None)")
    horner_orders = [(int(r[0]) >> 8) & 0xFF for tag, r, _, _, _ in recs
                     if tag in (T_MULTIPOLE, T_MULTIPOLE_CURVED, T_MULTIPOLE_RAD, T_EXCITER)
                     or (tag & 0xC0) == T_THIN_BLOCK]
    if all(o <= LOW_ORDER_MAX for o in horner_orders):
        flags |= F_LOW_ORDER
    biggest = max([len(r[1]) for r in recs] + [0])
    while biggest + 2 > chunk_words:
        chunk_words *= 2
    if chunk_words * 8 > 96 * 1024:
        raise ValueError("an element record (%d words) exceeds the 96 KiB chunk limit" % biggest)
    chunks = []    # (words, is last chunk of its segment)
    segments = []  # [first_chunk, n_chunks, kind]

    # Path length: `s` advances by the drift lengths only (xline/elements.py:56,72).  The fast
    # kernels do not add them up particle by particle: every END_TURN record carries the length
    # of the pass (segment) it closes, and every record a particle can be lost at carries the
    # length from the start of the pass up to itself (see include/xline_b200.h).
    def close_segment(cur, first, kind, length):
        cur += [_hdr(T_END_TURN, 0, 0), _f2u(length)]
        chunks.append((cur, True))
        segments.append([first, len(chunks) - first, kind])

    cur, first, s_pass = [], 0, 0.0
    exciter_words = []  # (chunk, word in the chunk) of every exciter's data_offset
    for tag, r, s_word, drift_len, drift_before in recs:
        if split and tag == T_BEAMBEAM6D:
            if cur or len(chunks) > first:  # a tracking segment precedes the lens
                close_segment(cur, first, SEG_MAIN, s_pass)
            close_segment(list(r), len(chunks), SEG_BB6D, 0.0)
            cur, first, s_pass = [], len(chunks), 0.0
            continue
        if len(cur) + len(r) + 2 > chunk_words:
            cur += [_hdr(T_END_CHUNK, 0, 0), np.uint64(0)]
            chunks.append((cur, False))
            cur = []
        if s_word is not None:
            r = list(r)
            r[s_word] = _f2u(s_pass + drift_before)
        if tag == T_EXCITER:
            exciter_words.append((len(chunks), len(cur) + 5))
        cur = cur + r
        s_pass = s_pass + drift_len
    close_segment(cur, first, SEG_MAIN, s_pass)  # the closing tracking segment (may be empty) counts the turn
    region = len(chunks) * chunk_words
    words = np.zeros(region + sum(len(d) for d in data), dtype=np.uint64)
    for i, (ch, last) in enumerate(chunks):
        words[i * chunk_words: i * chunk_words + len(ch)] = np.array(ch, dtype=np.uint64)
        # fill the tail with END_CHUNK/END_TURN so a stray read can never run away
        tail = _hdr(T_END_TURN if last else T_END_CHUNK, 0, 0)
        words[i * chunk_words + len(ch): (i + 1) * chunk_words: 2] = tail
    for ci, w in exciter_words:  # data_offset: from the start of the data region to an absolute word index
        words[ci * chunk_words + w] += np.uint64(region)
    if data:
        words[region:] = np.concatenate(data).view(np.uint64)
    seg = np.array(segments, dtype=np.int32).reshape(-1, 3) if split else None
    return PackedLattice(words, chunk_words, len(chunks), len(elements), flags, monitors, counts, seg)


def element_specs(elements):
    """Neutral ``(type_name, {field: value})`` description of a line -- what the tests hand
    to the CPU oracle (the oracle shares no code with this package)."""
    out = []
    for el in elements:
        d = el.to_dict(keepextra=True)
        d.pop("__class__")
        d.pop("data", None)
        out.append((type(el).__name__, d))
    return out


RAD_OPS = {"mean": 74, "quantum": 82}  # per radiating multipole, photon sampling not counted
EXCITER_OPS = 8  # per Exciter on top of its multipole: the sample index (6) and the two scalings by it


def algorithmic_ops(elements, radiation=None):
    """FP64 operations per particle-turn by the SURVEY.md §8(a)/(d) convention (every
    + - * / and **2 counts 1, each sqrt/sin/cos/exp 1, a wofz call taken as 100).  With
    ``radiation``, every radiating multipole adds ``RAD_OPS[radiation]``: the field magnitude and
    path length (8), and per half the particle's gamma, beta, kappa (9), the energy loss (mean: 9;
    quantum: n̄, exp, the first Poisson step: 13), add_to_energy (13) and the px, py scaling (3).
    The data-dependent rest of the quantum mode (further Poisson steps, ~23 per photon) is not
    counted.  An Exciter counts as a straight multipole of its order plus ``EXCITER_OPS``."""
    WOFZ = 100
    total = 0
    for el in elements:
        name = type(el).__name__
        if radiates(el, radiation):
            total += RAD_OPS[radiation]
        if name == "Drift":
            total += 15
        elif name == "DriftExact":
            total += 18
        elif name == "Multipole":
            total += 10 * el.order + 4 + (19 if (el.hxl != 0 or el.hyl != 0) else 0)
        elif name == "Exciter":
            total += 10 * el.order + 4 + EXCITER_OPS
        elif name in ("Cavity", "SawtoothCavity"):
            total += 33
        elif name == "RFMultipole":
            total += 32 * (el.order + 1) + 38
        elif name == "SRotation":
            total += 12
        elif name == "XYShift":
            total += 2
        elif name == "DipoleEdge":
            total += 4
        elif name == "LimitRect":
            total += 4
        elif name == "LimitEllipse":
            total += 6
        elif name == "LimitRectEllipse":
            total += 10
        elif name == "LimitPolygon":  # per stored edge: two compares (y slab), sub, mul, add, compare
            yv = list(el.y_vertices)
            total += 6 * sum(1 for k in range(len(yv)) if yv[k] != yv[(k + 1) % len(yv)])
        elif name in ("BeamBeam4D", "SCCoasting", "SCQGaussProfile", "SCInterpolatedProfile"):
            if el.enabled:
                msd = 1e-10 if name == "BeamBeam4D" else el.min_sigma_diff
                rnd = abs(el.sigma_x - el.sigma_y) < msd
                total += 35 + (15 if rnd else 31 + 2 * WOFZ)
        elif name == "BeamBeam6D":
            if el.enabled:
                ns = len(np.atleast_1d(el.charge_slices))
                total += 200 + ns * (230 + 2 * WOFZ + 8)
    return total
