"""TEST INFRASTRUCTURE -- a NumPy interpreter of the packed lattice format.

Walks the 8-byte words produced by ``xline_b200.lattice.pack_line`` exactly as
``include/xline_b200.h`` documents them (chunks, record headers, the thin / merged / edge block
families, both encodings) and applies the element maps with plain NumPy arithmetic.  It exists
so that the packer and the format can be checked on a machine without a GPU
(``tests/test_packed_format.py``): a lattice packed in the *strict* encoding and interpreted
here must reproduce the oracle bit for bit (NumPy has no FMA contraction, and the strict
encoding keeps the reference's operation order), the *fast* encoding to rounding.

Everything but the BeamBeam6D record (covered by the GPU parity tests); the Faddeeva function of
the Gaussian-field records is scipy's, and a MULTIPOLE_RAD record radiates through
``tests/radiation_oracle.py`` with the mode, constants and seed it reads from the record.  Nothing
in the product imports this file.
"""
import numpy as np

from tests import radiation_oracle as RO

T_END_TURN, T_END_CHUNK, T_DRIFT, T_DRIFT_EXACT, T_MULTIPOLE, T_MULTIPOLE_CURVED = range(6)
T_CAVITY, T_RFMULTIPOLE, T_XYSHIFT, T_SROTATION, T_DIPOLE_EDGE = range(6, 11)
T_LIMIT_RECT, T_LIMIT_ELLIPSE, T_LIMIT_RECT_ELLIPSE, T_MONITOR, T_SAWTOOTH_CAVITY = range(11, 16)
T_BEAMBEAM4D, T_SPACECHARGE, T_BEAMBEAM6D, T_LIMIT_POLYGON, T_MULTIPOLE_RAD = 16, 17, 18, 19, 20
AP_NONE, AP_RECT_SYM, AP_RECT, AP_ELLIPSE = range(4)
COORDS = ("x", "px", "y", "py", "zeta", "delta", "rpp", "rvv")


class _Beam:
    """Fixed-length arrays with a state flag, like the device side: lost particles stay where
    they were lost (``state = 0``, ``at_element``, ``at_turn`` set)."""

    def __init__(self, cols, p0c, mass0, q0=1.0):
        n = len(cols["x"])
        self.n = n
        self.q0, self.p0c, self.mass0 = float(q0), float(p0c), float(mass0)
        self.energy0 = float(np.sqrt(self.p0c * self.p0c + self.mass0 * self.mass0))
        self.beta0 = self.p0c / self.energy0
        for k in ("x", "px", "y", "py", "zeta"):
            setattr(self, k, np.array(cols.get(k, np.zeros(n)), dtype=np.float64))
        self.chi = np.ones(n)
        self.charge_ratio = np.ones(n)
        d = np.array(cols.get("delta", np.zeros(n)), dtype=np.float64)
        db0 = d * self.beta0
        ptaub0 = np.sqrt(db0 ** 2 + 2 * db0 * self.beta0 + 1) - 1
        self.delta = d
        self.rvv = (1 + d) / (1 + ptaub0)
        self.rpp = 1 / (1 + d)
        self.state = np.ones(n, dtype=np.int64)
        self.at_element = np.zeros(n, dtype=np.int64)
        self.at_turn = np.zeros(n, dtype=np.int64)
        self.particle_id = np.arange(n, dtype=np.int64)

    def result(self):
        return {k: getattr(self, k).copy() for k in COORDS + ("state", "at_element", "at_turn")}


class _Live:
    """The alive particles of a beam as working copies; ``commit`` writes them back, ``lose``
    freezes a subset as it is now."""

    def __init__(self, beam):
        self.beam = beam
        self.idx = np.flatnonzero(beam.state == 1)
        for k in COORDS + ("chi", "charge_ratio"):
            setattr(self, k, getattr(beam, k)[self.idx].copy())

    def __len__(self):
        return len(self.idx)

    def commit(self):
        for k in COORDS:
            getattr(self.beam, k)[self.idx] = getattr(self, k)

    def lose(self, lost, elem_idx, turn, override=None):
        """``lost``: boolean over the live set.  ``override``: {name: array over the live set}
        of values the lost particles are frozen with instead of the current ones."""
        if not lost.any():
            return
        gone = self.idx[lost]
        for k in COORDS:
            src = override[k] if override and k in override else getattr(self, k)
            getattr(self.beam, k)[gone] = src[lost]
        self.beam.state[gone] = 0
        self.beam.at_element[gone] = elem_idx
        self.beam.at_turn[gone] = turn
        keep = ~lost
        self.idx = self.idx[keep]
        for k in COORDS + ("chi", "charge_ratio"):
            setattr(self, k, getattr(self, k)[keep])


def _add_to_energy(p, beam, energy):  # Pyparticles.add_to_energy as restated in the oracle
    b0 = beam.beta0
    old_rvv = p.rvv
    db0 = p.delta * b0
    ptaub0 = np.sqrt(db0 ** 2 + 2 * db0 * b0 + 1) - 1
    ptaub0 = ptaub0 + energy / beam.energy0
    ptau = ptaub0 / b0
    p.delta = np.sqrt(ptau ** 2 + 2 * ptau / b0 + 1) - 1
    opd = 1 + p.delta
    p.rvv = opd / (1 + ptaub0)
    p.rpp = 1 / opd
    p.zeta = p.zeta * (p.rvv / old_rvv)


def _drift(p, L):
    xp = p.px * p.rpp
    yp = p.py * p.rpp
    p.x = p.x + xp * L
    p.y = p.y + yp * L
    p.zeta = p.zeta + L * (p.rvv - (1 + (xp ** 2 + yp ** 2) / 2))


def _drift_exact(p, L):
    opd = 1 + p.delta
    lpzi = L / np.sqrt(opd ** 2 - p.px ** 2 - p.py ** 2)
    p.x = p.x + p.px * lpzi
    p.y = p.y + p.py * lpzi
    p.zeta = p.zeta + (p.rvv * L - opd * lpzi)


def _closing_drift(p, tag, L):
    if tag & 8:
        if tag & 16:
            _drift_exact(p, L)
        else:
            _drift(p, L)


def _horner(p, pairs, order, strict):
    """pairs[m] = (kn, ks)[order - m]; strict: raw knl/ksl and the division by ii at every
    step; fast: coefficients already divided by i!."""
    dpx = pairs[0, 0]
    dpy = pairs[0, 1]
    for ii in range(order, 0, -1):
        k = pairs[order - ii + 1]
        zre = dpx * p.x - dpy * p.y
        zim = dpx * p.y + dpy * p.x
        if strict:
            zre = zre / ii
            zim = zim / ii
        dpx = k[0] + zre
        dpy = k[1] + zim
    one = np.ones_like(p.x)
    return dpx * one, dpy * one  # arrays also for order 0 (x * 1.0 is exact)


def _kick(p, dpx, dpy, curved, strict, k0=None):
    """Returns (new px, new py, new zeta) of a thin multipole (elements.py:135-156).
    ``curved`` = (hxl, hyl, length, 1/length) or None; ``k0`` = (knl[0], ksl[0]) used by the
    curvature terms."""
    ddx = -p.chi * dpx
    ddy = p.chi * dpy
    zeta = p.zeta
    if curved is not None:
        hxl, hyl, length, inv_length = curved
        b1l = p.chi * k0[0]
        a1l = p.chi * k0[1]
        hxlx = hxl * p.x
        hyly = hyl * p.y
        if strict:
            if length > 0:
                hxx = hxlx / length
                hyy = hyly / length
            else:
                hxx = 0
                hyy = 0
        else:
            hxx = hxlx * inv_length
            hyy = hyly * inv_length
        ddx = ddx + (hxl + hxl * p.delta - b1l * hxx)
        ddy = ddy - (hyl + hyl * p.delta - a1l * hyy)
        zeta = p.zeta - p.chi * (hxlx - hyly)
    return p.px + ddx, p.py + ddy, zeta


def _multipole(p, f64, w, tag, aux, strict):
    """The MULTIPOLE / MULTIPOLE_CURVED record at word ``w``: the kick applied to ``p``."""
    if tag == T_MULTIPOLE:
        pairs = f64[w + 2: w + 2 + 2 * (aux + 1)].reshape(aux + 1, 2)
        curved = None
    else:
        pairs = f64[w + 6: w + 6 + 2 * (aux + 1)].reshape(aux + 1, 2)
        curved = (f64[w + 1], f64[w + 2], f64[w + 3], f64[w + 4])
    dpx, dpy = _horner(p, pairs, aux, strict)
    p.px, p.py, p.zeta = _kick(p, dpx, dpy, curved, strict, k0=pairs[aux])


class _Rad:
    """The live particles as the radiation oracle's map sees them."""

    def __init__(self, live, beam):
        self.live, self.beam = live, beam
        self.q0, self.p0c, self.energy0 = beam.q0, beam.p0c, beam.energy0
        self.particle_id = beam.particle_id[live.idx]
        self.at_turn = beam.at_turn[live.idx]

    def __getattr__(self, k):
        return getattr(self.live, k)

    def __setattr__(self, k, v):
        if k in COORDS:
            setattr(self.live, k, v)
        else:
            object.__setattr__(self, k, v)

    def add_to_energy(self, energy):
        _add_to_energy(self.live, self.beam, energy)


def _multipole_rad(p, beam, words, f64, i64, w, aux, elem, strict):
    """The MULTIPOLE_RAD record at word ``w``: radiate, the embedded multipole, radiate."""
    mode = {1: "mean", 2: "quantum"}[int(i64[w + 1])]
    length = f64[w + 2]
    consts = (f64[w + 4], f64[w + 5], f64[w + 6])
    seed = int(words[w + 7])
    sub = w + 8
    tag = int(words[sub]) & 0xFF
    if tag == T_MULTIPOLE:
        pairs = f64[sub + 2: sub + 2 + 2 * (aux + 1)].reshape(aux + 1, 2)
        hxl = hyl = 0.0
    else:
        pairs = f64[sub + 6: sub + 6 + 2 * (aux + 1)].reshape(aux + 1, 2)
        hxl, hyl = f64[sub + 1], f64[sub + 2]
    dpx, dpy = _horner(p, pairs, aux, strict)
    fl = np.sqrt(dpx * dpx + dpy * dpy)
    lh = 0.5 * (length + hxl * p.x - hyl * p.y)
    RO.radiate_half(_Rad(p, beam), fl, lh, length, mode, seed, elem, 0, consts=consts)
    _multipole(p, f64, sub, tag, aux, strict)
    RO.radiate_half(_Rad(p, beam), fl, lh, length, mode, seed, elem, 1, consts=consts)


def _inside(kind, x, y, lim, strict):
    if kind == AP_RECT_SYM:
        return (np.abs(x) <= lim[1]) & (np.abs(y) <= lim[3])
    if kind == AP_RECT:
        return (x >= lim[0]) & (x <= lim[1]) & (y >= lim[2]) & (y <= lim[3])
    if strict:
        return x * x / lim[0] + y * y / lim[1] <= 1.0
    return x * x * lim[2] + y * y * lim[3] <= 1.0


def polygon_inside(f64, i64, w, x, y):
    """LIMIT_POLYGON at word ``w``: [hdr,n_edges][s_here,drift] then [y_lo,y_hi][x_lo,slope] per edge."""
    n_edges = int(i64[w + 1])
    odd = np.zeros(len(x), dtype=bool)
    for y_lo, y_hi, x_lo, slope in f64[w + 4: w + 4 + 4 * n_edges].reshape(-1, 4):
        assert y_lo < y_hi
        with np.errstate(invalid="ignore"):  # inf * 0 for an infinite y at a vertical edge
            odd ^= (y >= y_lo) & (y < y_hi) & (x < x_lo + (y - y_lo) * slope)
    return odd


def _gauss_field(f64, i64, w, x, y, strict):
    """Field block at word ``w``: [sx,sy][i64 kind,0][A,0] and, in the fast encoding,
    [1/S, A sqrt(pi)/S][small/big, big/small][1/(2 big^2), 1/(2 small^2)]
    (gaussian_fields.py:5-21 round, :29-99 Bassetti-Erskine).  Returns Ex, Ey and the number of
    pairs the block occupies."""
    from scipy.special import wofz

    sx, sy = f64[w], f64[w + 1]
    kind = int(i64[w + 2])
    A = f64[w + 4]
    npairs = 3 if strict else 6
    if kind == 0:
        sigma = 0.5 * (sx + sy)
        r2 = x * x + y * y
        with np.errstate(all="ignore"):
            temp = np.where(r2 < 1e-20, np.sqrt(r2) * A / sigma,
                            (1.0 - np.exp(-0.5 * r2 / (sigma * sigma))) * A / np.where(r2 > 0, r2, 1.0))
        return temp * x, temp * y, npairs
    wide = kind == 1
    u, v = (np.abs(x), np.abs(y)) if wide else (np.abs(y), np.abs(x))  # along big, along small
    if strict:
        big, small = (sx, sy) if wide else (sy, sx)
        S = np.sqrt(2.0 * (big * big - small * small))
        fact = A * 1.772453850905516 / S
        w1 = wofz((u + 1j * v) / S)
        w2 = wofz((small / big * u + 1j * (big / small * v)) / S)
        e = np.exp(-u * u / (2.0 * big * big) - v * v / (2.0 * small * small))
    else:
        inv_s, fact = f64[w + 6], f64[w + 7]
        r_sb, r_bs = f64[w + 8], f64[w + 9]
        h_big, h_small = f64[w + 10], f64[w + 11]
        us, vs = u * inv_s, v * inv_s
        w1 = wofz(us + 1j * vs)
        w2 = wofz(r_sb * us + 1j * (r_bs * vs))
        e = np.exp(-(u * u * h_big + v * v * h_small))
    f_im = fact * (w1.imag - w2.imag * e)  # field along the big axis
    f_re = fact * (w1.real - w2.real * e)  # field along the small axis
    ex, ey = (f_im, f_re) if wide else (f_re, f_im)
    return np.where(x < 0, -ex, ex), np.where(y < 0, -ey, ey), npairs


def _path_length_words(tag, aux, w, f64, i64):
    """-> (index of the record's s_here word or None, by how much the record advances s)."""
    if tag in (T_DRIFT, T_DRIFT_EXACT):
        return None, f64[w + 1]
    if tag in (T_LIMIT_RECT, T_LIMIT_ELLIPSE):
        return w + 5, (f64[w + 6] if aux & 0x10 else 0.0)
    if tag == T_LIMIT_RECT_ELLIPSE:
        return w + 7, (f64[w + 8] if aux & 0x10 else 0.0)
    if tag == T_LIMIT_POLYGON:
        return w + 2, (f64[w + 3] if aux & 0x10 else 0.0)
    if tag == T_SPACECHARGE:
        return None, (f64[w + 1] if aux & 0x10 else 0.0)
    if (tag & 0xC0) == 0xC0:  # dipole edge -> [drift]
        return None, (f64[w + 1] if tag & 8 else 0.0)
    if (tag & 0xC0) == 0x80:
        adv = f64[w + 1] if tag & 8 else 0.0
        if not tag & 0x20:
            return w + 3, adv
        info = int(i64[w + 3])
        k1_order, has_a1 = info & 0xFF, (info >> 8) & 1
        t = 2 + aux + 1 + (3 if tag & 4 else 0) + (2 if has_a1 else 0) + (2 if tag & 3 else 0)
        return w + 2 * (t + k1_order + 1), adv
    return None, 0.0


def track(packed, cols, p0c, mass0, num_turns=1, monitor=None):
    """Interpret ``packed`` (a PackedLattice without segments) for ``num_turns`` turns.
    ``monitor``: fp64 array of ``packed.monitor_words`` words (NaN-filled by the caller), the
    BeamMonitor storage of include/xline_b200.h: per monitor [7 fields][num_stores][n_ids]."""
    assert packed.segments is None
    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
    f64 = words.view(np.float64)
    i64 = words.view(np.int64)
    strict = packed.strict
    beam = _Beam(cols, p0c, mass0)
    cw = packed.chunk_words
    for turn in range(num_turns):
        p = _Live(beam)
        done = False
        s_pass = 0.0  # drift lengths since the start of the pass, summed in record order
        for ch in range(packed.n_chunks):
            if done:
                break
            w = ch * cw
            while True:
                hdr = int(words[w])
                tag, aux, size, elem = hdr & 0xFF, (hdr >> 8) & 0xFF, (hdr >> 16) & 0x3FFF, hdr >> 32
                hx_only = bool((hdr >> 31) & 1)  # XLB_HDR_HX_ONLY
                assert w % 2 == 0 and w + 2 * size <= (ch + 1) * cw, "record straddles a chunk"
                p0 = f64[w + 1]
                pair = lambda m, _w=w: f64[_w + 2 * m: _w + 2 * m + 2]  # noqa: E731
                nxt = w + 2 * size
                if tag == T_END_CHUNK:
                    break
                if tag == T_END_TURN:
                    assert p0 == s_pass, "END_TURN must carry the length of the pass"
                    done = True
                    break
                # the path-length bookkeeping of the format (include/xline_b200.h, "Path length")
                s_at, adv = _path_length_words(tag, aux, w, f64, i64)
                if s_at is not None:
                    assert f64[s_at] == s_pass, "s_here of record at word %d" % w
                if hx_only:
                    assert (tag & 0xC4) == 0x84 and not strict
                    assert f64[w + 2 * (2 + aux + 1) + 1] == 0.0, "XLB_HDR_HX_ONLY needs hyl == 0"
                s_pass = s_pass + adv
                if len(p) == 0:
                    w = nxt
                    continue
                if (tag & 0xC0) == 0x80:  # thin (0x80) or merged (0xA0) block
                    merged = bool(tag & 0x20)
                    assert not (merged and strict)
                    order = aux
                    pairs = f64[w + 4: w + 4 + 2 * (order + 1)].reshape(order + 1, 2)
                    t = 2 + order + 1  # pair index of what follows the coefficients
                    dpx, dpy = _horner(p, pairs, order, strict)
                    ap = tag & 3
                    if not merged:
                        curved = None
                        if tag & 4:
                            curved = (pair(t)[0], pair(t)[1], pair(t + 1)[0], pair(t + 1)[1])
                            t += 2
                        p.px, p.py, p.zeta = _kick(p, dpx, dpy, curved, strict, k0=pairs[order])
                        if ap != AP_NONE:
                            lim = np.concatenate([pair(t), pair(t + 1)])
                            p.lose(~_inside(ap, p.x, p.y, lim, strict), int(i64[w + 2]), turn)
                    else:
                        idxs, info = int(i64[w + 2]), int(i64[w + 3])
                        a1_idx, a2_idx = idxs & 0xFFFFFFFF, idxs >> 32
                        k1_order, has_a1 = info & 0xFF, (info >> 8) & 1
                        assert has_a1 == (hdr >> 30) & 1, "XLB_HDR_HAS_A1 must mirror the record"
                        curved = k0 = None
                        if tag & 4:
                            curved = (pair(t)[0], pair(t)[1], pair(t + 1)[0], pair(t + 1)[1])
                            k0 = pair(t + 2)
                            t += 3
                        npx, npy, nzeta = _kick(p, dpx, dpy, curved, False, k0=k0)
                        if has_a1:  # lost at A1: frozen with K1's kick only
                            lim = np.concatenate([pair(t), pair(t + 1)])
                            t += 2
                            lost = ~_inside(AP_ELLIPSE, p.x, p.y, lim, False)
                            if lost.any():
                                k1_pairs_at = t + (2 if ap != AP_NONE else 0)
                                k1 = f64[w + 2 * k1_pairs_at: w + 2 * (k1_pairs_at + k1_order + 1)].reshape(-1, 2)
                                kx, ky = _horner(p, k1, k1_order, False)
                                frozen = dict(px=p.px + (-p.chi * kx), py=p.py + p.chi * ky)
                                keep = ~lost
                                p.lose(lost, a1_idx, turn, override=frozen)
                                npx, npy, nzeta = npx[keep], npy[keep], nzeta[keep]
                        p.px, p.py, p.zeta = npx, npy, nzeta
                        if ap != AP_NONE:
                            lim = np.concatenate([pair(t), pair(t + 1)])
                            p.lose(~_inside(ap, p.x, p.y, lim, False), a2_idx, turn)
                    _closing_drift(p, tag, p0)
                elif (tag & 0xC0) == 0xC0:  # dipole edge -> [drift]
                    e = pair(1)
                    p.px = p.px + e[0] * p.x
                    p.py = p.py + e[1] * p.y
                    _closing_drift(p, tag, p0)
                elif tag == T_DRIFT:
                    _drift(p, p0)
                elif tag == T_DRIFT_EXACT:
                    _drift_exact(p, p0)
                elif tag in (T_MULTIPOLE, T_MULTIPOLE_CURVED):
                    _multipole(p, f64, w, tag, aux, strict)
                elif tag == T_MULTIPOLE_RAD:
                    _multipole_rad(p, beam, words, f64, i64, w, aux, elem, strict)
                elif tag in (T_CAVITY, T_SAWTOOTH_CAVITY):
                    k, lag = pair(1)
                    tau = p.zeta / p.rvv / beam.beta0
                    phase = lag - k * tau
                    if tag == T_CAVITY:
                        wave = np.sin(phase)
                    else:
                        wave = (phase + np.pi) % (2 * np.pi) - np.pi
                    _add_to_energy(p, beam, p.charge_ratio * beam.q0 * p0 * wave)
                elif tag == T_XYSHIFT:
                    p.x = p.x - p0
                    p.y = p.y - pair(1)[0]
                elif tag == T_SROTATION:
                    cz, sz = p0, pair(1)[0]
                    xn = cz * p.x + sz * p.y
                    yn = -sz * p.x + cz * p.y
                    p.x, p.y = xn, yn
                    xn = cz * p.px + sz * p.py
                    yn = -sz * p.px + cz * p.py
                    p.px, p.py = xn, yn
                elif tag == T_DIPOLE_EDGE:
                    p.px = p.px + p0 * p.x
                    p.py = p.py + pair(1)[0] * p.y
                elif tag == T_LIMIT_RECT:
                    lim = np.array([p0, pair(1)[0], pair(1)[1], pair(2)[0]])
                    p.lose(~_inside(AP_RECT_SYM if aux & 1 else AP_RECT, p.x, p.y, lim, strict), elem, turn)
                    if aux & 0x10:  # the drift that follows the aperture
                        (_drift_exact if aux & 0x20 else _drift)(p, pair(3)[0])
                elif tag == T_LIMIT_ELLIPSE:
                    lim = np.array([p0, pair(1)[0], pair(1)[1], pair(2)[0]])
                    p.lose(~_inside(AP_ELLIPSE, p.x, p.y, lim, strict), elem, turn)
                    if aux & 0x10:
                        (_drift_exact if aux & 0x20 else _drift)(p, pair(3)[0])
                elif tag == T_LIMIT_RECT_ELLIPSE:
                    mx, my = p0, pair(1)[0]
                    lim = np.array([pair(1)[1], pair(2)[0], pair(2)[1], pair(3)[0]])
                    inside = ((p.x >= -mx) & (p.x <= mx) & (p.y >= -my) & (p.y <= my)
                              & _inside(AP_ELLIPSE, p.x, p.y, lim, strict))
                    p.lose(~inside, elem, turn)
                    if aux & 0x10:
                        (_drift_exact if aux & 0x20 else _drift)(p, pair(4)[0])
                elif tag == T_LIMIT_POLYGON:
                    p.lose(~polygon_inside(f64, i64, w, p.x, p.y), elem, turn)
                    if aux & 0x10:
                        (_drift_exact if aux & 0x20 else _drift)(p, f64[w + 3])
                elif tag == T_RFMULTIPOLE:  # [hdr,V][k,lag] then per order [knl,ksl][pn,ps]
                    k, lag = pair(1)
                    ktau = k * (p.zeta / p.rvv / beam.beta0)
                    dpx = dpy = dptr = 0
                    zre, zim = 1, 0
                    for ii in range(aux + 1):
                        kn, ks = pair(2 + 2 * ii)
                        pn, ps = pair(3 + 2 * ii)
                        cn, sn = np.cos(pn - ktau), np.sin(pn - ktau)
                        cs, ss = np.cos(ps - ktau), np.sin(ps - ktau)
                        dpx = dpx + (cn * kn * zre - cs * ks * zim)
                        dpy = dpy + (cs * ks * zre + cn * kn * zim)
                        zret = (zre * p.x - zim * p.y) / (ii + 1)
                        zim = (zim * p.x + zre * p.y) / (ii + 1)
                        zre = zret
                        dptr = dptr + (sn * (kn * zre) - ss * (ks * zim))
                    p.px = p.px + -p.chi * dpx
                    p.py = p.py + p.chi * dpy
                    dv0 = p0 * np.sin(lag - ktau)
                    _add_to_energy(p, beam, p.charge_ratio * beam.q0 * (dv0 - beam.p0c * k * dptr))
                elif tag == T_MONITOR:  # [hdr,0][start,skip][num_stores,min_id][max_id,rolling][offset,0]
                    start, skip, num_stores, min_id = (int(v) for v in i64[w + 2: w + 6])
                    max_id, rolling, off = (int(v) for v in i64[w + 6: w + 9])
                    nn = max_id - min_id + 1
                    if monitor is not None and nn > 0 and num_stores > 0 and turn >= start \
                            and (turn - start) % skip == 0:
                        st = (turn - start) // skip
                        if st >= num_stores and rolling:
                            st %= num_stores
                        if st < num_stores:
                            pid = beam.particle_id[p.idx]
                            sel = (pid >= min_id) & (pid <= max_id)
                            plane = num_stores * nn
                            o = off + st * nn + (pid[sel] - min_id)
                            for f, name in enumerate(("x", "px", "y", "py", "zeta", "delta")):
                                monitor[o + f * plane] = getattr(p, name)[sel]
                            monitor[o + 6 * plane] = float(turn)
                elif tag == T_BEAMBEAM4D:  # [hdr,0][x_bb,y_bb] field [d_px,d_py][beta_r, charge*qe]
                    ex, ey, nf = _gauss_field(f64, i64, w + 4, p.x - pair(1)[0], p.y - pair(1)[1], strict)
                    d, bc = pair(2 + nf), pair(3 + nf)
                    beta = beam.beta0 / p.rvv  # sic, beambeam.py:55
                    fact = p.chi * bc[1] * (p.charge_ratio * beam.q0) * (1.0 + beta * bc[0]) / (beam.p0c * (beta + bc[0]))
                    p.px = p.px + (fact * ex - d[0])
                    p.py = p.py + (fact * ey - d[1])
                elif tag == T_SPACECHARGE:  # [hdr,0][x_co,y_co] field [base, p1] ...; aux = profile kind
                    ex, ey, nf = _gauss_field(f64, i64, w + 4, p.x - pair(1)[0], p.y - pair(1)[1], strict)
                    t = w + 2 * (2 + nf)  # first word after the field block
                    base, p1 = f64[t], f64[t + 1]
                    common = beam.q0 * beam.q0 * (1.0 - beam.beta0 * beam.beta0) / (beam.p0c * beam.beta0) * base
                    kind = aux & 0xF
                    lam = 1.0
                    if kind == 1:  # q-Gaussian in zeta / rvv: [sqrt_beta/cq, 1-q][1/(1-q), 0][i64 gauss, 0]
                        arg = p1 * (p.zeta / p.rvv) ** 2
                        if int(i64[t + 6]):
                            lam = f64[t + 2] * np.exp(-arg)
                        else:
                            up = np.maximum(1.0 + (-arg) * f64[t + 3], 0.0)
                            lam = f64[t + 2] * up ** f64[t + 4]
                    elif kind in (2, 3):  # [base,z0][dz,0][i64 n,0] then the profile / the spline
                        z0, dz, npts = p1, f64[t + 2], int(i64[t + 4])
                        i = np.clip(np.floor((p.zeta - z0) / dz).astype(np.int64), 0, npts - 2)
                        if kind == 2:
                            prof = f64[t + 6: t + 6 + npts]
                            xi = z0 + i * dz
                            lam = (prof[i + 1] - prof[i]) / dz * (p.zeta - xi) + prof[i]
                            lam = np.where(p.zeta <= z0, prof[0], lam)
                            lam = np.where(p.zeta >= z0 + (npts - 1) * dz, prof[npts - 1], lam)
                        else:
                            xk = f64[t + 6: t + 6 + npts]
                            c = f64[t + 6 + npts: t + 6 + npts + 4 * (npts - 1)]
                            m = npts - 1
                            dt = p.zeta - xk[i]
                            lam = ((c[i] * dt + c[m + i]) * dt + c[2 * m + i]) * dt + c[3 * m + i]
                    fact = p.chi * p.charge_ratio * common * lam
                    p.px = p.px + fact * ex
                    p.py = p.py + fact * ey
                    if aux & 0x10:  # the drift that follows the kick
                        (_drift_exact if aux & 0x20 else _drift)(p, p0)
                else:
                    raise NotImplementedError("tag 0x%02x is outside the interpreter's scope" % tag)
                w = nxt
        assert done, "lattice without END_TURN"
        p.commit()
        beam.at_turn[p.idx] += 1
    return beam.result()
