"""TEST INFRASTRUCTURE -- a NumPy interpreter of packed lattices that hold MULTIPOLE_RAD records.

Walks the words of ``xline_b200.lattice.pack_line(..., radiation=...)`` as include/xline_b200.h
documents them, with the element maps and bookkeeping of ``tests/packed_interpreter.py`` and
``tests/polygon_interpreter.py`` (whose helpers it uses), for the record kinds the radiation tests
pack: thin blocks, drifts, straight and curved multipoles, cavities, the LIMIT_* apertures and
MULTIPOLE_RAD, whose mode, constants and seed it reads from the record.  Any other record raises.
Fast encoding: to rounding against ``tests/radiation_oracle.py``.
"""
import numpy as np

from tests import packed_interpreter as PI
from tests import polygon_interpreter as PY
from tests import radiation_oracle as RO

T_MULTIPOLE_RAD = 20
T_MULTIPOLE_CURVED = 5
T_CAVITY = 6


class _Rad:
    """The live particles as the oracle's radiation map sees them."""

    def __init__(self, live, beam):
        self.live, self.beam = live, beam
        self.q0, self.p0c, self.energy0 = beam.q0, beam.p0c, beam.energy0
        self.particle_id = beam.particle_id[live.idx]
        self.at_turn = beam.at_turn[live.idx]

    def __getattr__(self, k):
        return getattr(self.live, k)

    def __setattr__(self, k, v):
        if k in PI.COORDS:
            setattr(self.live, k, v)
        else:
            object.__setattr__(self, k, v)

    def add_to_energy(self, energy):
        PI._add_to_energy(self.live, self.beam, energy)


def _multipole(p, f64, w, tag, aux):
    """The MULTIPOLE / MULTIPOLE_CURVED record at word ``w`` (fast encoding)."""
    if tag == PI.T_MULTIPOLE:
        pairs = f64[w + 2: w + 2 + 2 * (aux + 1)].reshape(aux + 1, 2)
        curved = None
    else:
        pairs = f64[w + 6: w + 6 + 2 * (aux + 1)].reshape(aux + 1, 2)
        curved = (f64[w + 1], f64[w + 2], f64[w + 3], f64[w + 4])
    dpx, dpy = PI._horner(p, pairs, aux, False)
    p.px, p.py, p.zeta = PI._kick(p, dpx, dpy, curved, False, k0=pairs[aux])
    return dpx, dpy, curved


def _multipole_rad(p, beam, words, f64, i64, w, aux, elem, elem_off):
    mode = {1: "mean", 2: "quantum"}[int(i64[w + 1])]
    length = f64[w + 2]
    consts = (f64[w + 4], f64[w + 5], f64[w + 6])
    seed = int(words[w + 7])
    sub = w + 8
    tag = int(words[sub]) & 0xFF
    if tag == PI.T_MULTIPOLE:
        pairs = f64[sub + 2: sub + 2 + 2 * (aux + 1)].reshape(aux + 1, 2)
        hxl = hyl = 0.0
    else:
        pairs = f64[sub + 6: sub + 6 + 2 * (aux + 1)].reshape(aux + 1, 2)
        hxl, hyl = f64[sub + 1], f64[sub + 2]
    dpx, dpy = PI._horner(p, pairs, aux, False)
    fl = np.sqrt(dpx * dpx + dpy * dpy)
    lh = 0.5 * (length + hxl * p.x - hyl * p.y)
    RO.radiate_half(_Rad(p, beam), fl, lh, length, mode, seed, elem + elem_off, 0, consts=consts)
    _multipole(p, f64, sub, tag, aux)
    RO.radiate_half(_Rad(p, beam), fl, lh, length, mode, seed, elem + elem_off, 1, consts=consts)


def track(packed, cols, p0c, mass0, num_turns=1):
    """Interpret ``packed`` (fast encoding, no segments, no monitors) for ``num_turns`` turns."""
    assert packed.segments is None and not packed.strict
    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
    f64, i64 = words.view(np.float64), words.view(np.int64)
    beam = PI._Beam(cols, p0c, mass0)
    cw = packed.chunk_words
    for turn in range(num_turns):
        p = PI._Live(beam)
        done = False
        for ch in range(packed.n_chunks):
            if done:
                break
            w = ch * cw
            while True:
                hdr = int(words[w])
                tag, aux, size, elem = hdr & 0xFF, (hdr >> 8) & 0xFF, (hdr >> 16) & 0x3FFF, hdr >> 32
                p0 = f64[w + 1]
                pair = lambda m, _w=w: f64[_w + 2 * m: _w + 2 * m + 2]  # noqa: E731
                nxt = w + 2 * size
                if tag == PI.T_END_CHUNK:
                    break
                if tag == PI.T_END_TURN:
                    done = True
                    break
                if len(p) == 0:
                    w = nxt
                    continue
                if (tag & 0xE0) == 0x80:  # thin block: kick -> [aperture] -> [drift]
                    order = aux
                    pairs = f64[w + 4: w + 4 + 2 * (order + 1)].reshape(order + 1, 2)
                    t = 2 + order + 1
                    dpx, dpy = PI._horner(p, pairs, order, False)
                    curved = None
                    if tag & 4:
                        curved = (pair(t)[0], pair(t)[1], pair(t + 1)[0], pair(t + 1)[1])
                        t += 2
                    p.px, p.py, p.zeta = PI._kick(p, dpx, dpy, curved, False, k0=pairs[order])
                    if tag & 3:
                        lim = np.concatenate([pair(t), pair(t + 1)])
                        p.lose(~PI._inside(tag & 3, p.x, p.y, lim, False), int(i64[w + 2]), turn)
                    PI._closing_drift(p, tag, p0)
                elif tag == T_MULTIPOLE_RAD:
                    p.commit()
                    _multipole_rad(p, beam, words, f64, i64, w, aux, elem, 0)
                elif tag in (PI.T_MULTIPOLE, T_MULTIPOLE_CURVED):
                    _multipole(p, f64, w, tag, aux)
                elif tag == PI.T_DRIFT:
                    PI._drift(p, p0)
                elif tag == PI.T_DRIFT_EXACT:
                    PI._drift_exact(p, p0)
                elif tag == T_CAVITY:
                    k, lag = pair(1)
                    tau = p.zeta / p.rvv / beam.beta0
                    PI._add_to_energy(p, beam, beam.q0 * p0 * np.sin(lag - k * tau))
                elif tag in (PI.T_LIMIT_RECT, PI.T_LIMIT_ELLIPSE):
                    lim = np.array([p0, pair(1)[0], pair(1)[1], pair(2)[0]])
                    kind = PI.AP_ELLIPSE if tag == PI.T_LIMIT_ELLIPSE else (PI.AP_RECT_SYM if aux & 1 else PI.AP_RECT)
                    p.lose(~PI._inside(kind, p.x, p.y, lim, False), elem, turn)
                    PY._fused_drift(p, aux, pair(3)[0])
                else:
                    raise NotImplementedError("tag 0x%02x is outside this interpreter's scope" % tag)
                w = nxt
        assert done, "lattice without END_TURN"
        p.commit()
        beam.at_turn[p.idx] += 1
    return beam.result()
